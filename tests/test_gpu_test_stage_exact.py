"""The test stage at gene-set size against exact references (tests/exact_ref.py): substitution counts, sequence
frequencies, K6 gene and element mode, the window denominators, K5 gene tabulation, the scale-factor sums and the
27 result rows of the fused burden test.  Bounds are in units of u = 2^-53 and hold for nonnegative data; each check
prints its worst observed error, which records the device's margins.

Everything is seeded.  No genome is built: K6 only sees window counts, so they are drawn at random, with runs of
all-zero windows standing in for assembly gaps, over the 10 kb windows of a 3.1 Gb hg19-like genome."""
import math

import numpy as np
import pytest
import torch

import exact_ref as X

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
WINDOW = 10_000
N_RANDOM_GENES = 20_000
U = X.U
SUB = np.arange(192) // 3


def _t(a, dt):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dtype=dt)


def _np(t):
    return t.cpu().numpy()


def _check(name, err_u, bound_u):
    """err_u, bound_u: per-element error and bound in units of u."""
    err_u, bound_u = np.broadcast_arrays(np.asarray(err_u, dtype=np.float64), np.asarray(bound_u, dtype=np.float64))
    ratio = np.where(err_u == 0, 0.0, err_u / bound_u)
    i = int(np.argmax(ratio)) if ratio.size else 0
    worst = float(err_u.ravel()[np.argmax(err_u)]) if err_u.size else 0.0
    print("\n%-40s worst %.3g u, worst error / bound %.3g" % (name, worst, ratio.ravel()[i] if ratio.size else 0.0))
    assert np.all(err_u <= bound_u), "%s: %d values over the bound, first at %d (%.3g u > %.3g u)" % (
        name, int((err_u > bound_u).sum()), int(np.flatnonzero(err_u > bound_u)[0]),
        err_u.ravel()[np.flatnonzero(err_u > bound_u)[0]], bound_u.ravel()[np.flatnonzero(err_u > bound_u)[0]])


def _same(a, b):
    """Bit-identical up to the NaN payload."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


# ---------------------------------------------------------------- fixture

def _edge_genes(rng, n_win_chrom0, zero_run):
    """Constructed genes on chromosome 0: (strand, [(start, inclusive end), ...]) each."""
    genes = []
    w = 1000                                                 # window number of the next gene, 200 windows apart

    def base(k, off=100):
        return k * WINDOW + off
    for offset in (0, 31):
        for span in (1, 31, 32, 33, 64, 65):
            blocks = []
            if offset:
                blocks.append((base(w), base(w, 900)))       # anchor: the span starts 31 windows after it
            a = w + offset
            blocks.append((base(a), base(a + span - 1, 5000)))
            genes.append(blocks)
            w += 200
    # 32 set windows of one word, hit by single-window blocks in scrambled order
    genes.append([(base(w + k), base(w + k, 300)) for k in rng.permutation(32)])
    w += 200
    # unsorted, overlapping and duplicated blocks
    genes.append([(base(w + 5), base(w + 7)), (base(w + 1), base(w + 3)), (base(w + 2), base(w + 6)),
                  (base(w + 1), base(w + 3)), (base(w + 40), base(w + 41))])
    w += 200
    # inclusive end on a multiple of the window: window w + 3 is not overlapped
    genes.append([(base(w, 10), (w + 3) * WINDOW)])
    w += 200
    # zero-length block on a window boundary: no window
    genes.append([(base(w, 5), base(w, 500)), ((w + 7) * WINDOW, (w + 7) * WINDOW)])
    w += 200
    # every window zero-count: D = 0, P = NaN
    genes.append([(base(zero_run + 1), base(zero_run + 2, 5000))])
    assert w < n_win_chrom0 - 200
    return [(1 if i % 2 == 0 else -1, b) for i, b in enumerate(genes)]


@pytest.fixture(scope="module")
def fx():
    from digdriver_b200 import genome as G, kernels, pipeline
    rng = np.random.default_rng(2024)
    lengths = G.hg19_like_lengths(3_100_000_000)
    wins = G.tile_windows(np.arange(len(lengths)), lengths, WINDOW)
    n_win = len(wins)
    off, wmap = kernels.build_window_map(wins[:, 0], wins[:, 1], WINDOW, len(lengths))
    counts = rng.integers(0, 400, (n_win, 64), dtype=np.int32)
    for s in rng.integers(0, n_win - 8, 2000):              # N runs of 1-6 windows
        counts[s:s + rng.integers(1, 7)] = 0
    zero_run = 22_000                                       # chromosome 0: rows == window numbers
    counts[zero_run:zero_run + 5] = 0
    y_pred, std, y_true, flag = pipeline.synth_region_params(n_win, 2025)
    chrom, strand, ptr, bs, be = pipeline.synth_genes(N_RANDOM_GENES, lengths, WINDOW, 2026)
    edges = _edge_genes(rng, int(off[1] - off[0]), zero_run)
    e_bs = [s for _, b in edges for s, _ in b]
    e_be = [e for _, b in edges for _, e in b]
    e_ptr = ptr[-1] + np.cumsum([0] + [len(b) for _, b in edges])
    chrom = np.concatenate([chrom, np.zeros(len(edges), dtype=np.int32)])
    strand = np.concatenate([strand, np.array([s for s, _ in edges], dtype=np.int8)])
    ptr = np.concatenate([ptr, e_ptr[1:]])
    bs, be = np.concatenate([bs, e_bs]).astype(np.int64), np.concatenate([be, e_be]).astype(np.int64)
    E = len(chrom)
    edge = np.arange(N_RANDOM_GENES, E)
    L = rng.integers(0, 60, (E, 192, 4)).astype(np.float64)
    # one zero per gene and column: a gene whose windows are all zero-count gets P = sum (d / 0) L = NaN, which the
    # scale sums skip as pandas does (an all-positive column would give inf and zero every gene's scale factor)
    for c in range(4):
        L[np.arange(E), rng.integers(0, 192, E), c] = 0.0
    d_pr = np.exp(rng.uniform(np.log(1e-9), np.log(1e-3), 192))
    assert len(np.unique(d_pr)) == 192
    dev = dict(counts=_t(counts, torch.int32), y_pred=_t(y_pred, torch.float64), std=_t(std, torch.float64),
               y_true=_t(y_true, torch.float64), flag=_t(flag, torch.uint8), d_pr=_t(d_pr, torch.float64),
               L=_t(L, torch.float64))
    args = (chrom, strand, ptr, bs, be, WINDOW, off, wmap)
    out = kernels.element_transfer(*args, dev["counts"], dev["y_pred"], dev["std"], dev["y_true"], dev["flag"],
                                   dev["d_pr"], L_elt=dev["L"], device=DEV)
    ref = X.gene_transfer_ref(*args, counts, y_pred, std, y_true, flag, d_pr, L=L)
    return dict(args=args, counts=counts, y_pred=y_pred, std=std, y_true=y_true, flag=flag, d_pr=d_pr, L=L, dev=dev,
                out=out, ref=ref, E=E, edge=edge, n_win=n_win, rng=rng)


def _check_transfer(name, o, ref, rows=slice(None)):
    nw = ref["N_WIN"][rows]
    for k in ("R_SIZE", "ELT_SIZE", "N_WIN"):
        assert np.array_equal(_np(o[k])[rows], ref[k][rows]), "%s %s" % (name, k)
    assert np.array_equal(_np(o["R_OBS"])[0][rows], ref["R_OBS"][rows]), name + " R_OBS"
    assert np.array_equal(_np(o["FLAG"])[0][rows].astype(bool), ref["FLAG"][rows]), name + " FLAG"
    _check(name + " MU", X._rel_err_u(_np(o["MU"])[0][rows], ref["MU"][rows]), nw + 1)
    _check(name + " SIGMA", X._rel_err_u(_np(o["SIGMA"])[0][rows], ref["SIGMA"][rows]), nw / 2 + 2)
    P, Pr = _np(o["P"])[0][rows], ref["P"][rows]
    fin = np.isfinite(Pr)
    assert _same(P[~fin], Pr[~fin]), name + " P where the denominator is 0"
    _check(name + " P", X._rel_err_u(P[fin], Pr[fin]), 32)


def test_gene_transfer_exact(fx):
    """K6 gene mode on 20 000 synthetic genes and the constructed edge genes."""
    ref = fx["ref"]
    assert np.isnan(ref["P"][fx["E"] - 1]).all() and ref["N_WIN"][fx["E"] - 1] == 2
    assert ref["N_WIN"].max() >= 65 and (ref["N_WIN"] == 32).any()
    _check_transfer("K6 gene mode", fx["out"], ref)


def test_element_transfer_exact_on_edge_genes(fx):
    """K6 element mode (block counts, n_col = 1) on the constructed genes."""
    from digdriver_b200 import kernels
    chrom, strand, ptr, bs, be, window, off, wmap = fx["args"]
    edge = fx["edge"]
    p0 = ptr[edge[0]]
    eptr = ptr[edge[0]:] - p0
    ebs, ebe = bs[p0:], be[p0:]
    bc = fx["rng"].integers(0, 400, (len(ebs), 64), dtype=np.int32)
    args = (chrom[edge], strand[edge], eptr, ebs, ebe, window, off, wmap)
    d = fx["dev"]
    out = kernels.element_transfer(*args, d["counts"], d["y_pred"], d["std"], d["y_true"], d["flag"], d["d_pr"],
                                   blk_counts=bc, device=DEV)
    ref = X.gene_transfer_ref(*args, fx["counts"], fx["y_pred"], fx["std"], fx["y_true"], fx["flag"], fx["d_pr"],
                              blk_counts=bc)
    _check_transfer("K6 element mode", out, ref)


def test_gene_transfer_generic_column_path(fx):
    """The per-column path (L not 16-byte aligned, or n_col != 4) sums in the same order as the paired-load path."""
    from digdriver_b200 import kernels
    d, E = fx["dev"], fx["E"]
    P4 = _np(fx["out"]["P"])[0]

    def run(L):
        return _np(kernels.element_transfer(*fx["args"], d["counts"], d["y_pred"], d["std"], d["y_true"], d["flag"],
                                            d["d_pr"], L_elt=L, device=DEV)["P"])[0]
    buf = torch.empty(E * 192 * 4 + 1, dtype=torch.float64, device=DEV)
    buf[1:].copy_(d["L"].reshape(-1))
    Lu = buf[1:].view(E, 192, 4)
    assert Lu.data_ptr() % 16 == 8
    assert _same(run(Lu), P4)
    for n_col in (1, 2, 3):
        assert _same(run(d["L"][:, :, :n_col].contiguous()), P4[:, :n_col]), n_col
    P5 = run(torch.cat([d["L"], d["L"][:, :, :1]], dim=2))
    assert _same(P5[:, :4], P4) and _same(P5[:, 4], P4[:, 0])


def test_window_denominators_exact(fx):
    from digdriver_b200 import _lib
    d, n = fx["dev"], fx["n_win"]
    dp, dm = (torch.empty(n, dtype=torch.float64, device=DEV) for _ in range(2))
    _lib.call("dig_window_denominators", d["counts"].data_ptr(), d["d_pr"].data_ptr(), n, dp.data_ptr(), dm.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    got_p, got_m = _np(dp), _np(dm)
    counts, rc = fx["counts"], X.revcomp64()
    want_p, want_m = np.empty(n), np.empty(n)
    for i in range(0, n, 1 << 16):
        c = counts[i:i + (1 << 16)]
        want_p[i:i + len(c)] = X.exact_dot_int(fx["d_pr"], c[:, SUB])
        want_m[i:i + len(c)] = X.exact_dot_int(fx["d_pr"], c[:, rc][:, SUB])
    zero = ~counts.any(axis=1)
    assert zero.sum() > 1000
    assert np.all(got_p[zero] == 0) and np.all(got_m[zero] == 0)
    _check("window denominators +", X._rel_err_u(got_p, want_p), 16)
    _check("window denominators -", X._rel_err_u(got_m, want_m), 16)


# ---------------------------------------------------------------- sequence model

def test_substitution_counts_and_sequence_freq():
    from digdriver_b200 import kernels
    rng = np.random.default_rng(11)
    n = 1_000_000
    ctx = rng.integers(0, 64, n).astype(np.int32)
    ctx[rng.random(n) < 0.1] = -1
    alt = rng.integers(0, 4, n).astype(np.uint8)
    alt[rng.random(n) < 0.05] = 255
    alt[rng.random(n) < 0.01] = rng.integers(4, 255, 1).astype(np.uint8)[0]
    ref = (ctx >> 2) & 3
    same = rng.random(n) < 0.05
    alt[same] = ref[same]                                    # ALT == REF rows are not substitutions
    keep = (ctx >= 0) & (alt <= 3) & (alt != ref)
    a = alt.astype(np.int64)
    want = np.bincount((3 * ctx + a - (a > ref))[keep], minlength=192)
    got = kernels.substitution_counts(_t(ctx, torch.int32), alt)
    assert np.array_equal(_np(got), want)
    # FREQ = COUNT / S_genome[ctx]; context 5 has no genome occurrence (0 / 0 = NaN, x / 0 = inf)
    tot = rng.integers(10 ** 6, 10 ** 9, 64)
    tot[5] = 0
    cnt = want.copy()
    cnt[15], cnt[16] = 0, 7
    freq = _np(kernels.sequence_freq(_t(cnt, torch.int64), _t(tot, torch.int64)))
    with np.errstate(divide="ignore", invalid="ignore"):
        wf = cnt.astype(np.float64) / np.repeat(tot.astype(np.float64), 3)
    assert np.isnan(wf[15]) and np.isinf(wf[16])
    assert _same(freq, wf)


# ---------------------------------------------------------------- observed counts

def _mutation_mix(rng, n, n_gene, n_sample=2500):
    """The benchmark's mix: 30 % coding SNVs, 7 % indels (half of them in genes), the rest non-coding; Zipf samples;
    plus rows naming genes outside the table."""
    gene = np.full(n, -1, dtype=np.int32)
    cls = np.full(n, 255, dtype=np.uint8)
    n_cds, n_ind = int(0.30 * n), int(0.07 * n)
    gene[:n_cds] = rng.integers(0, n_gene, n_cds)
    cls[:n_cds] = rng.choice(4, size=n_cds, p=[0.23, 0.68, 0.04, 0.05])
    gene[n_cds:n_cds + n_ind // 2] = rng.integers(0, n_gene, n_ind // 2)
    cls[n_cds:n_cds + n_ind // 2] = 4
    far = rng.choice(n, 2000, replace=False)
    gene[far] = rng.integers(n_gene, n_gene + 50, 2000)
    cls[far] = rng.integers(0, 5, 2000)
    w = 1.0 / np.arange(1, n_sample + 1)
    sample = rng.choice(n_sample, size=n, p=w / w.sum()).astype(np.int32)
    perm = rng.permutation(n)
    return gene[perm], sample[perm], cls[perm]


def test_tabulate_genes_exact():
    from digdriver_b200 import kernels
    rng = np.random.default_rng(12)
    n_gene = 20_000
    gene, sample, cls = _mutation_mix(rng, 1_000_000, n_gene)
    capped = None
    for cap in (None, 3):
        obs, nsamp = kernels.tabulate_genes(gene, sample, cls, n_gene, 3 * 10 ** 9 if cap is None else cap, device=DEV)
        wo, wn = X.tabulate_genes_ref(gene, sample, cls, n_gene, cap)
        assert np.array_equal(_np(obs), wo), cap
        assert np.array_equal(_np(nsamp), wn), cap
        if cap is None:
            capped = wo
    assert not np.array_equal(capped, wo)                   # the cap binds somewhere


def test_tabulate_genes_table_overflow_raises():
    """2 000 distinct (gene, sample) keys cannot fit a 1024-slot table: status 1, which the wrapper turns into an
    error."""
    from digdriver_b200 import _lib, kernels
    n = 2000
    mg, ms = _t(np.arange(n), torch.int32), _t(np.zeros(n), torch.int32)
    mc = _t(np.zeros(n), torch.uint8)
    cap = 1024
    keys = torch.empty(cap, dtype=torch.int64, device=DEV)
    cnt = torch.empty((cap, 5), dtype=torch.int32, device=DEV)
    obs = torch.empty((n, 5), dtype=torch.int64, device=DEV)
    nsamp = torch.empty((n, 7), dtype=torch.int64, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    _lib.call("dig_tabulate_genes", mg.data_ptr(), ms.data_ptr(), mc.data_ptr(), n, keys.data_ptr(), cnt.data_ptr(),
              cap, 2 ** 62, n, obs.data_ptr(), nsamp.data_ptr(), status.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    assert int(status.item()) == 1
    with pytest.raises(_lib.DigError, match="overflow"):
        kernels._check_status(status, "dig_tabulate_genes")


# ---------------------------------------------------------------- scale-factor sums

def _scale_terms(mu, sigma, P, pi_indel):
    """The kernel's terms, elementwise as it forms them."""
    with np.errstate(all="ignore"):
        t0 = mu * P[:, 0]
        t1 = pi_indel * ((mu * mu) / (sigma * sigma)) * ((sigma * sigma) / mu)
    return t0, t1


def _check_scale_sums(name, got, mu, sigma, P, pi_indel, obs, cgc, tp53):
    n = len(mu)
    t0, t1 = _scale_terms(mu, sigma, P, pi_indel)
    k0 = ~np.isnan(t0)
    if 0 <= tp53 < n:
        k0[tp53] = False
    non = np.ones(n, dtype=bool) if cgc is None else ~cgc
    k1 = non & ~np.isnan(t1)
    bound = math.ceil(n / 8192) + 18
    errs = []
    for i, (t, k) in enumerate(((t0, k0), (t1, k1))):
        s = math.fsum(t[k])
        if math.isinf(s):                                    # an infinite term: pandas' sum is inf
            assert got[i] == s, "%s sums[%d]: %r, want %r" % (name, i, got[i], s)
            errs.append(0.0)
            continue
        err = abs(got[i] - s) / (U * math.fsum(np.abs(t[k]))) if k.any() else abs(got[i]) / U
        assert err <= bound, "%s sums[%d]: %.3g u > %d u" % (name, i, err, bound)
        errs.append(err)
    assert got[2] == float(obs[non, 4].sum()), name
    return errs[0]


def test_gene_scale_sums_exact_sweep():
    """Every rank, stride and unroll remainder of the one-cluster reduction: n across the 1024-gene block ranges and
    the 8192-gene strides, TP53 in several ranks, three CGC masks, NaN rows in every rank's range."""
    from digdriver_b200 import kernels
    rng = np.random.default_rng(13)
    nmax = 100_000
    mu = rng.gamma(2.0, 20.0, nmax) + 0.05
    sigma = mu * rng.uniform(0.01, 1.5, nmax)
    P = rng.uniform(1e-6, 1e-2, (nmax, 4))
    pi = rng.uniform(1e-6, 1e-2, nmax)
    obs = rng.integers(0, 40, (nmax, 5)).astype(np.int64)
    g = np.arange(nmax)
    P[g % 1024 == 3, 0] = np.nan                             # NaN rows in every rank's range, every stride
    pi[g % 1024 == 700] = np.nan
    dmu, dsg, dP, dpi, dobs = (_t(x, dt) for x, dt in ((mu, torch.float64), (sigma, torch.float64),
                                                         (P, torch.float64), (pi, torch.float64), (obs, torch.int64)))
    worst = 0.0
    for n in (1, 300, 1023, 1024, 1025, 7168, 7169, 8191, 8192, 8193, 32767, 32768, 32769, 100_000):
        masks = {"none": None, "5%": rng.random(n) < 0.05, "all": np.ones(n, dtype=bool)}
        for tp53 in sorted({-1, 0, 7 * 1024 + 5 if n > 7 * 1024 + 5 else n // 2, n - 1}):
            for mname, cgc in masks.items():
                s = _np(kernels.gene_scale_sums(dmu[:n], dsg[:n], dP[:n], dpi[:n], dobs[:n], cgc, tp53))
                e = _check_scale_sums("n=%d tp53=%d cgc=%s" % (n, tp53, mname), s, mu[:n], sigma[:n], P[:n],
                                      pi[:n], obs[:n], cgc, tp53)
                worst = max(worst, e)
    print("\ngene_scale_sums sweep: worst sums[0] error %.3g u * sum|t|" % worst)
    # one infinite Pi_INDEL (a gene with no countable window context): pandas' sum is inf
    pi2 = pi[:20_000].copy()
    pi2[12_345] = np.inf
    s = _np(kernels.gene_scale_sums(dmu[:20_000], dsg[:20_000], dP[:20_000], _t(pi2, torch.float64), dobs[:20_000]))
    assert s[1] == np.inf
    _check_scale_sums("inf Pi_INDEL", s, mu[:20_000], sigma[:20_000], P[:20_000], pi2, obs[:20_000], None, -1)


# ---------------------------------------------------------------- the burden test on the fixture's K6 output

@pytest.fixture(scope="module")
def stage(fx):
    from digdriver_b200 import kernels
    out, ref, E = fx["out"], fx["ref"], fx["E"]
    rng = np.random.default_rng(14)
    gene, sample, cls = _mutation_mix(rng, 1_000_000, E)
    obs, nsamp = kernels.tabulate_genes(gene, sample, cls, E, device=DEV)
    mu, sigma, P = out["MU"][0].contiguous(), out["SIGMA"][0].contiguous(), out["P"][0].contiguous()
    pi = kernels.size_ratio(out["ELT_SIZE"], out["R_SIZE"])
    with np.errstate(divide="ignore"):
        assert _same(_np(pi), ref["ELT_SIZE"].astype(np.float64) / ref["R_SIZE"].astype(np.float64))
    # genes without countable window context (Pi_INDEL = inf) in the CGC set, so the indel scale factor stays finite
    cgc = (rng.random(E) < 0.05) | (ref["R_SIZE"] == 0)
    tp53 = 12_345
    sums = kernels.gene_scale_sums(mu, sigma, P, pi, obs, cgc, tp53)
    h = dict(mu=_np(mu), sigma=_np(sigma), P=_np(P), pi=_np(pi), obs=_np(obs), nsamp=_np(nsamp), sums=_np(sums))
    e = _check_scale_sums("K6 output, 20 000 genes", h["sums"], h["mu"], h["sigma"], h["P"], h["pi"], h["obs"], cgc,
                          tp53)
    print("\ngene_scale_sums on the K6 output: sums[0] error %.3g u * sum|t|" % e)
    assert np.all(np.isfinite(h["sums"]) & (h["sums"] > 0))          # cj and t_indel are not degenerate
    return dict(dev=(mu, sigma, P, pi, obs, nsamp), sums=sums, h=h, n_syn=float(h["obs"][:, 0].sum()))


def _burden_rows_ref(h, cj, t_indel):
    """Rows 0-5, 18 and 21-26 in the kernel's operation order."""
    m, s, P, pi = h["mu"], h["sigma"], h["P"], h["pi"]
    with np.errstate(all="ignore"):
        alpha = (m * m) / (s * s)
        theta0 = (s * s) / m
        theta = theta0 * cj
        theta_i = theta0 * t_indel
        p_trunc = P[:, 2] + P[:, 3]
        p_nonsyn = P[:, 1] + p_trunc
        pis = [P[:, 0], P[:, 1], P[:, 2], P[:, 3], p_trunc, p_nonsyn]
        rows = {c: (alpha * theta) * pis[c] for c in range(6)}
        rows[18] = (alpha * theta_i) * pi
    rows.update({21: alpha, 22: theta, 23: theta_i, 24: pi, 25: p_trunc, 26: p_nonsyn})
    return rows, alpha, theta, theta_i, pis


@pytest.mark.parametrize("path", ["scale_factor", "n_syn", "sums3"])
def test_gene_burden_test_routing(stage, path):
    """Every row of dig_gene_burden_test from its inputs: the arithmetic rows bit-exact to numpy, the 13 p-values
    bit-identical to dig_nb_burden_test fed the reference's (k, ALPHA, THETA, Pi), the Fisher row to
    dig_fisher_combine2.  cj comes from scale_factor, from n_syn / sums[0], or from sums[3] / sums[0] (n_syn=None)."""
    from digdriver_b200 import kernels
    h, sums = stage["h"], stage["sums"]
    n_syn = stage["n_syn"]
    if path == "scale_factor":
        out = kernels.gene_burden_test(*stage["dev"], sums, 0.0, scale_factor=1.3)
        cj = 1.3
    elif path == "n_syn":
        out = kernels.gene_burden_test(*stage["dev"], sums, n_syn)
        cj = n_syn / h["sums"][0]
    else:
        s4 = torch.cat([sums, torch.tensor([n_syn], dtype=torch.float64, device=DEV)])
        out = kernels.gene_burden_test(*stage["dev"], s4, None)
        cj = n_syn / h["sums"][0]
    out = _np(out)
    t_indel = h["sums"][2] / h["sums"][1]
    rows, alpha, theta, theta_i, pis = _burden_rows_ref(h, cj, t_indel)
    for r, want in rows.items():
        assert _same(out[r], want), "row %d (%s)" % (r, kernels.GENE_OUT_ROWS[r])
    o, ns = h["obs"].astype(np.float64), h["nsamp"].astype(np.float64)
    ks = [o[:, 0], o[:, 1], o[:, 2], o[:, 3], o[:, 2] + o[:, 3], o[:, 1] + (o[:, 2] + o[:, 3])]
    ks += [ns[:, c] for c in range(6)] + [o[:, 4]]
    pi_all = pis + pis + [h["pi"]]
    th_all = [theta] * 12 + [theta_i]
    E = len(alpha)
    _, pv = kernels.nb_burden_test(np.concatenate(ks), np.tile(alpha, 13), np.concatenate(th_all),
                                   np.concatenate(pi_all), DEV, want_exp=False)
    pv = _np(pv).reshape(13, E)
    for t in range(13):
        r = 6 + t if t < 12 else 19
        assert _same(out[r], pv[t]), "row %d (%s)" % (r, kernels.GENE_OUT_ROWS[r])
    assert _same(out[20], _np(kernels.fisher_combine2(out[10], out[19], DEV)))
    assert (h["obs"][:, 3] > 0).any() and (h["nsamp"][:, 6] > 0).any()
