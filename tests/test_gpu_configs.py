"""GPU parity tests for the other BASELINE.json configurations at reduced-but-realistic size:
config 3 (site-level test), config 4 (noncoding elements on 10 kb and 1 Mb maps) and config 5 (many
cohorts per launch).  Full outputs are checked on a random subset against the CPU oracle and in full through
size-independent properties (permutation invariance, strand symmetry, batch == single launches)."""
import numpy as np
import pandas as pd
import pytest
import torch

from conftest import assert_pvals_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def world(oracle):
    """A 3-chromosome, 60 Mb synthetic genome with 10 kb and 1 Mb maps."""
    from digdriver_b200 import kernels
    from digdriver_b200.genome import DeviceGenome, tile_windows
    lengths = np.array([30_000_001, 20_000_500, 10_123_456], dtype=np.int64)
    dg = DeviceGenome.synthetic(["chr1", "chr2", "chr3"], lengths, seed=44, device=DEV)
    rng = np.random.default_rng(5)
    maps = {}
    for W in (10_000, 1_000_000):
        wins = tile_windows([1, 2, 3], lengths, W)                      # chromosome NUMBERS
        c64, _ = kernels.count_contexts(dg, wins[:, 0] - 1, wins[:, 1], wins[:, 2], 1, 1)
        n = len(wins)
        yp = rng.gamma(2.0, 10.0 * W / 1e4, n)
        maps[W] = dict(wins=wins, c64=c64, c64h=c64.cpu().numpy().astype(np.int64), y_pred=yp,
                       std=yp * rng.uniform(0.05, 0.5, n), y_true=rng.poisson(yp).astype(np.float64),
                       flag=rng.random(n) < 0.1,
                       index={(int(c), int(s)): i for i, (c, s, e) in enumerate(wins)})
        maps[W]["off"], maps[W]["wmap"] = kernels.build_window_map(wins[:, 0], wins[:, 1], W, 4)
    d_pr = np.exp(rng.normal(np.log(1e-6), 1.0, 192))
    return dict(dg=dg, lengths=lengths, maps=maps, d_pr=d_pr, rng=rng)


def _elements(rng, lengths, n, window):
    """Regulatory-element-like BED12 intervals: 1-3 blocks of 200-2000 bp, both strands, some across windows."""
    chrom = rng.integers(1, 4, n)
    nb = rng.integers(1, 4, n)
    ptr = np.concatenate([[0], np.cumsum(nb)])
    owner = np.repeat(np.arange(n), nb)
    usable = (lengths[chrom - 1] - 1) // window * window
    g0 = (rng.random(n) * (usable - 12_000)).astype(np.int64) + 100
    g0[::7] = (g0[::7] // window) * window + window - 300                # straddle a window boundary
    size = rng.integers(200, 2001, ptr[-1])
    gap = rng.integers(0, 1500, ptr[-1])
    step = size + gap
    cs = np.cumsum(step) - step
    rel = cs - cs[ptr[:-1]][owner]
    bs = g0[owner] + rel
    be = np.minimum(bs + size, usable[owner] - 1)
    bs = np.minimum(bs, be - 1)
    strand = np.where(rng.random(n) < 0.5, -1, 1).astype(np.int8)
    return chrom, strand, ptr, bs, be, owner


def test_config4_noncoding_elements_two_maps(world, oracle):
    from digdriver_b200 import kernels, pipeline
    rng, dg, lengths = world["rng"], world["dg"], world["lengths"]
    E = 100_000
    chrom, strand, ptr, bs, be, owner = _elements(rng, lengths, E, 1_000_000)
    bc, _ = kernels.count_contexts(dg, chrom[owner] - 1, bs, be, 1, 1, strand=strand[owner])       # K4
    seq = None
    sub = rng.choice(E, 250, replace=False)
    for W in (10_000, 1_000_000):
        m = world["maps"][W]
        out = kernels.element_transfer(chrom, strand, ptr, bs, be, W, m["off"], m["wmap"], m["c64"], m["y_pred"],
                                       m["std"], m["y_true"], m["flag"], world["d_pr"], blk_counts=bc, device=DEV)
        o = {k: v.cpu().numpy() for k, v in out.items()}
        # ---- oracle on a random subset
        if seq is None:
            seq = np.full(dg.n_bases, ord("N"), dtype=np.uint8)
            for off_, n_ in zip(dg.chrom_off, lengths):
                seq[off_:off_ + n_] = oracle.synth_genome(int(off_), int(n_), 44)
        sp = np.concatenate([[0], np.cumsum(np.diff(ptr)[sub])])
        sel = np.concatenate([np.arange(ptr[i], ptr[i + 1]) for i in sub])
        c64s, _ = oracle.count_regions(seq, dg.chrom_off, lengths, chrom[owner][sel] - 1, bs[sel], be[sel], 1, 1,
                                       strand=strand[owner][sel])
        assert np.array_equal(c64s, bc.cpu().numpy()[sel])
        Ls = np.zeros((len(sub), 192))
        np.add.at(Ls, np.repeat(np.arange(len(sub)), np.diff(sp)), np.repeat(c64s, 3, axis=1))
        want = oracle.element_transfer(chrom[sub], strand[sub], sp, bs[sel], be[sel], Ls, W, m["index"], m["c64h"],
                                       m["y_pred"], m["std"], m["y_true"], m["flag"], world["d_pr"])
        np.testing.assert_allclose(o["MU"][0][sub], want["MU"], rtol=1e-12)
        np.testing.assert_allclose(o["SIGMA"][0][sub], want["SIGMA"], rtol=1e-12)
        np.testing.assert_allclose(o["P"][0][sub, 0], want["P_SUM"], rtol=1e-9)
        assert np.array_equal(o["R_SIZE"][sub], want["R_SIZE"]) and np.array_equal(o["ELT_SIZE"][sub], want["ELT_SIZE"])
        assert np.array_equal(o["N_WIN"][sub], want["N_WIN"]) and np.array_equal(o["FLAG"][0][sub].astype(bool), want["FLAG"])
        # ---- full-size properties
        assert np.all(o["ELT_SIZE"] <= (be - bs)[ptr[:-1]] * 0 + np.add.reduceat(be - bs, ptr[:-1]))
        perm = rng.permutation(E)                                         # element order must not matter
        pptr = np.concatenate([[0], np.cumsum(np.diff(ptr)[perm])])
        psel = np.concatenate([np.arange(ptr[i], ptr[i + 1]) for i in perm[:2000]])
        out2 = kernels.element_transfer(chrom[perm[:2000]], strand[perm[:2000]], pptr[:2001], bs[psel], be[psel], W,
                                        m["off"], m["wmap"], m["c64"], m["y_pred"], m["std"], m["y_true"], m["flag"],
                                        world["d_pr"], blk_counts=bc[torch.from_numpy(psel).to(DEV)], device=DEV)
        # (elements inside an N run have no valid context: 0/0 = NaN, as in the reference)
        assert np.array_equal(out2["P"].cpu().numpy()[0, :, 0], o["P"][0][perm[:2000], 0], equal_nan=True)
        assert np.array_equal(out2["MU"].cpu().numpy()[0], o["MU"][0][perm[:2000]])
    # ---- observed counts + test at scale: 1M SNVs / indels against the 100k elements
    M = 1_000_000
    mchrom = rng.integers(1, 4, M)
    mpos = (rng.random(M) * (lengths[mchrom - 1] - 50)).astype(np.int64)
    hot = rng.choice(len(bs), M // 4)                                     # a quarter land inside blocks
    mchrom[: M // 4] = chrom[owner][hot]
    mpos[: M // 4] = bs[hot] + (rng.random(M // 4) * (be - bs)[hot]).astype(np.int64)
    is_indel = rng.random(M) < 0.08
    mend = mpos + np.where(is_indel, rng.integers(1, 20, M), 1)
    sample = (rng.zipf(1.3, M) % 300).astype(np.int32)
    key = lambda c, p: (c.astype(np.int64) << 32) | p
    obs, stot = kernels.tabulate_elements(key(chrom[owner], bs), key(chrom[owner], be), owner, key(mchrom, mpos),
                                          key(mchrom, mend), sample, is_indel, E, 300, device=DEV)
    obs = obs.cpu().numpy()
    assert int(stot.sum()) == int(obs[:, 1].sum() + obs[:, 2].sum())    # checksum of checksums
    mut = pd.DataFrame({"CHROM": mchrom, "START": mpos, "END": mend, "REF": "A", "ALT": "C",
                        "SAMPLE": sample, "ANNOT": np.where(is_indel, "INDEL", "Noncoding")})
    near = np.zeros(M, dtype=bool)                                        # oracle on the mutations near the subset
    blocks = pd.DataFrame({"CHROM": chrom[owner][sel], "START": bs[sel], "END": be[sel], "ELT": owner[sel]})
    for c in (1, 2, 3):
        b = blocks[blocks.CHROM == c]
        if len(b):
            mm = mchrom == c
            near |= mm & (mpos < b.END.max()) & (mend > b.START.min())
    # every block of a subset element belongs to the subset, so counts restricted to those elements are complete
    want_tab, _ = oracle.tabulate_mutations_in_element(mut[near].reset_index(drop=True), blocks, drop_duplicates=False)
    got = pd.DataFrame(obs[sub], index=sub, columns=["OBS_SAMPLES", "OBS_SNV", "OBS_INDEL"])
    got = got[got.OBS_SAMPLES > 0].sort_index()
    assert list(got.index) == list(want_tab.index)
    assert np.array_equal(got.values, want_tab[["OBS_SAMPLES", "OBS_SNV", "OBS_INDEL"]].values.astype(np.int64))
    res = pipeline.element_burden_test(out, torch.from_numpy(obs).to(DEV), 0.8, 0.3)
    a, t = oracle.normal_params_to_gamma(o["MU"][0][sub], o["SIGMA"][0][sub])
    e_, p_ = oracle.burden_test(obs[sub, 1].astype(float), a, t * 0.8, o["P"][0][sub, 0])
    np.testing.assert_allclose(res["EXP_SNV"].cpu().numpy()[sub], e_, rtol=1e-12)
    assert_pvals_close(res["PVAL_SNV_BURDEN"].cpu().numpy()[sub], p_)
    _, pi_ = oracle.burden_test(obs[sub, 2].astype(float), a, t * 0.3, o["ELT_SIZE"][sub] / o["R_SIZE"][sub])
    assert_pvals_close(res["PVAL_INDEL_BURDEN"].cpu().numpy()[sub], pi_)
    assert_pvals_close(res["PVAL_MUT_BURDEN"].cpu().numpy()[sub], oracle.fisher2(p_, pi_))


def test_strand_symmetry_property(world):
    """With a strand-symmetric sequence model (d_pr[j] == d_pr[revcomp(j)]) an element and its reverse-strand
    copy must get the same P_SUM: checks the revcomp permutation of region counts against K4's strand handling."""
    from digdriver_b200 import kernels
    rng, dg, lengths = world["rng"], world["dg"], world["lengths"]
    names = np.array(__import__("oracle.dig_oracle", fromlist=["x"]).substitution_names())
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    rc = lambda s: "".join(comp[c] for c in reversed(s))
    pos = {n: i for i, n in enumerate(names)}
    partner = np.array([pos[rc(n.split(">")[0]) + ">" + rc(n.split(">")[1])] for n in names])
    d = np.exp(rng.normal(np.log(1e-6), 1.0, 192))
    d_sym = 0.5 * (d + d[partner])
    E = 5000
    chrom, strand, ptr, bs, be, owner = _elements(rng, lengths, E, 10_000)
    m = world["maps"][10_000]
    res = []
    for sgn in (1, -1):
        st = np.full(E, sgn, dtype=np.int8)
        bc, _ = kernels.count_contexts(dg, chrom[owner] - 1, bs, be, 1, 1, strand=st[owner])
        out = kernels.element_transfer(chrom, st, ptr, bs, be, 10_000, m["off"], m["wmap"], m["c64"], m["y_pred"],
                                       m["std"], m["y_true"], m["flag"], d_sym, blk_counts=bc, device=DEV)
        res.append(out["P"].cpu().numpy()[0, :, 0])
    np.testing.assert_allclose(res[0], res[1], rtol=1e-12)


def test_config5_many_cohorts_one_launch(world):
    """37 cohorts (own region parameters and sequence model each) in one K6 launch == 37 single launches."""
    from digdriver_b200 import kernels
    rng, lengths = world["rng"], world["lengths"]
    m = world["maps"][10_000]
    nW = len(m["wins"])
    C, E = 37, 3000
    chrom, strand, ptr, bs, be, owner = _elements(rng, lengths, E, 10_000)
    L = rng.integers(0, 40, (E, 192, 4)).astype(np.float64)
    yp = rng.gamma(2.0, 10.0, (C, nW))
    sd = yp * rng.uniform(0.05, 0.5, (C, nW))
    yt = rng.poisson(yp).astype(np.float64)
    fl = rng.random((C, nW)) < 0.1
    dpr = np.exp(rng.normal(np.log(1e-6), 1.0, (C, 192)))
    args = (chrom, strand, ptr, bs, be - 1, 10_000, m["off"], m["wmap"], m["c64"])
    batch = kernels.element_transfer(*args, yp, sd, yt, fl, dpr, L_elt=L, device=DEV)
    b = {k: v.cpu().numpy() for k, v in batch.items()}
    for ci in (0, 17, 36):
        one = kernels.element_transfer(*args, yp[ci], sd[ci], yt[ci], fl[ci], dpr[ci], L_elt=L, device=DEV)
        for k in ("MU", "SIGMA", "R_OBS", "FLAG", "P"):
            assert np.array_equal(one[k].cpu().numpy()[0], b[k][ci], equal_nan=(k == "P")), (k, ci)
        assert np.array_equal(one["R_SIZE"].cpu().numpy(), b["R_SIZE"])
    with pytest.raises(Exception):
        kernels.element_transfer(*args, np.ones((65, nW)), np.ones((65, nW)), np.ones((65, nW)),
                                 np.zeros((65, nW)), np.ones((65, 192)), L_elt=L, device=DEV)


def test_config3_site_sets(world, oracle, tmp_path):
    """Site-level test: per site-set L from the sites' own substitutions (strand-flipped), windows from the sites'
    intervals, exact-match observed counts, SNV-only p-values -- array level vs the oracle, then through files."""
    from digdriver_b200 import storage
    from digdriver_b200.data_tools import mutation_tools as mt
    from digdriver_b200.driver_model import transfer_tools as tt
    from digdriver_b200.sequence_model import genic_driver_tools as gd
    rng, dg, lengths = world["rng"], world["dg"], world["lengths"]
    m = world["maps"][10_000]
    wins = m["wins"]
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2], "Y_TRUE": m["y_true"],
                       "Y_PRED": m["y_pred"], "STD": m["std"], "FLAG": m["flag"]},
                      index=["chr%d:%d-%d" % tuple(r) for r in wins])
    rm = gd.RegionModel(rp)
    names = oracle.substitution_names()
    S, n_sets = 60_000, 150
    set_id = rng.integers(0, n_sets, S)
    set_chrom = rng.integers(1, 4, n_sets)
    set_strand = np.where(rng.random(n_sets) < 0.5, "-", "+")
    centre = (rng.random(n_sets) * (lengths[set_chrom - 1] - 300_000)).astype(np.int64) + 100_000
    pos = centre[set_id] + rng.integers(-40_000, 40_000, S)
    sub = rng.integers(0, 192, S)
    ctx = np.array([names[j].split(">")[0] for j in sub])
    alt = np.array([names[j].split(">")[1][1] for j in sub])
    sites = pd.DataFrame({"CHROM": set_chrom[set_id], "START": pos, "END": pos + 1, "REF": [c[1] for c in ctx],
                          "ALT": alt, "SAMPLE": ["SET%03d" % i for i in set_id], "GENE": "G", "ANNOT": "Missense",
                          "MUT_TYPE": [c[1] + ">" + a for c, a in zip(ctx, alt)], "CONTEXT": ctx,
                          "STRAND": set_strand[set_id]})
    sites.loc[::501, "CONTEXT"] = "nan"
    got = gd.sites_model_arrays(sites, rm, m["c64"], world["d_pr"]).set_index("ELT")
    # oracle: L by hand, blocks = the sites' intervals
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    rc = lambda s: "".join(comp[c] for c in reversed(s))
    npos = {n: i for i, n in enumerate(names)}
    order = np.argsort(sites.SAMPLE.values, kind="stable")
    ss = sites.iloc[order]
    elts, eid = np.unique(ss.SAMPLE.values, return_inverse=True)
    L = np.zeros((len(elts), 192))
    for e, mt_, cx, sd in zip(eid, ss.MUT_TYPE, ss.CONTEXT, ss.STRAND):
        if "nan" in cx:
            continue
        name = cx + ">" + cx[0] + mt_[2] + cx[2]
        if sd == "-":
            name = rc(cx) + ">" + rc(cx[0] + mt_[2] + cx[2])
        L[e, npos[name]] += 1
    first = np.concatenate([[0], np.flatnonzero(np.diff(eid)) + 1])
    ptr = np.concatenate([first, [len(ss)]])
    want = oracle.element_transfer(ss.CHROM.values[first], np.where(ss.STRAND.values[first] == "-", -1, 1), ptr,
                                   ss.START.values, ss.END.values, L, 10_000, m["index"], m["c64h"], m["y_pred"],
                                   m["std"], m["y_true"], m["flag"], world["d_pr"])
    assert list(got.index) == list(elts)
    np.testing.assert_allclose(got.P_SUM.values, want["P_SUM"], rtol=1e-9)
    np.testing.assert_allclose(got.MU.values, want["MU"], rtol=1e-12)
    assert np.array_equal(got.ELT_SIZE.values, want["ELT_SIZE"]) and np.array_equal(got.R_SIZE.values, want["R_SIZE"])
    # ---- through files: run_sites_region_model
    f_sites, f_mut, f_pre = tmp_path / "sites.tsv", tmp_path / "mut.tsv", str(tmp_path / "pre")
    sites_f = sites[sites.CONTEXT != "nan"]
    sites_f.to_csv(f_sites, sep="\t", header=False, index=False)
    hit = sites_f.sample(4000, random_state=1, replace=True)
    mut = hit.drop(columns=["STRAND"]).copy()
    mut["SAMPLE"] = ["P%02d" % s for s in rng.zipf(1.4, len(mut)) % 30]
    miss = mut.iloc[:500].copy()
    miss["START"] += 3
    miss["END"] += 3
    mut = pd.concat([mut, miss])
    mut.to_csv(f_mut, sep="\t", header=False, index=False)
    st = storage.Store(f_pre, "w")
    st.write_table("SITES", got.reset_index())
    df = tt.run_sites_region_model(str(f_mut), str(f_sites), f_pre, "SITES", scale_factor=1.7, scale_by_expectation=False)
    on = ["CHROM", "START", "END", "REF", "ALT", "GENE", "ANNOT", "MUT_TYPE", "CONTEXT"]
    mm = mt.read_mutation_file(str(f_mut)).merge(mt.read_mutation_file(str(f_sites)).rename(columns={"SAMPLE": "ELT"}), on=on)
    cnt = mm.groupby("ELT").agg(OBS_SAMPLES=("SAMPLE", lambda x: len(set(x))), OBS_SNV=("CHROM", "size"))
    cnt = cnt.reindex(df.index).fillna(0)
    assert np.array_equal(df.OBS_SNV.values, cnt.OBS_SNV.values) and np.array_equal(df.OBS_SAMPLES.values, cnt.OBS_SAMPLES.values)
    a, t = oracle.normal_params_to_gamma(df.MU.values, df.SIGMA.values)
    e_, p_ = oracle.burden_test(cnt.OBS_SNV.values, a, t * 1.7, df.Pi_SUM.values)
    np.testing.assert_allclose(df.EXP_SNV.values, e_, rtol=1e-12)
    assert_pvals_close(df.PVAL_SNV_BURDEN.values, p_)


def test_config3_per_site_test_30m_sites(world, oracle):
    """BASELINE config 3 at scale: 30 M sites, each its own one-site site set.  (1) a random subset is bit-identical to
    the same sites pushed through K6 as one-site elements (one-hot L) and within tolerance of the oracle's
    element_transfer + burden_test; (2) size-independent properties over all 30 M: the result of a site depends only
    on (window, strand, substitution, k) -- permuting the sites permutes the outputs -- and P * denom == d_pr[sub]."""
    from digdriver_b200 import kernels
    from digdriver_b200.sequence_model import genic_driver_tools as gd
    rng, lengths = np.random.default_rng(33), world["lengths"]
    m = world["maps"][10_000]
    wins, d_pr, cj = m["wins"], world["d_pr"], 1.37
    n = 30_000_000
    chrom = rng.integers(1, 4, n).astype(np.int32)
    usable = ((lengths - 1) // 10_000 * 10_000)[chrom - 1]
    start = (rng.random(n) * (usable - 1)).astype(np.int64)
    sub = rng.integers(0, 192, n).astype(np.uint8)
    strand = np.where(rng.random(n) < 0.5, -1, 1).astype(np.int8)
    k = rng.poisson(0.05, n).astype(np.float64)
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    dev = torch.device(DEV)
    args_d = [torch.from_numpy(a).to(dev) for a in (chrom, start, sub, k, strand)]
    for rep in range(2):                                     # the second call re-uses the allocator's blocks
        torch.cuda.synchronize()
        t0.record()
        out = kernels.site_test(args_d[0], args_d[1], args_d[2], args_d[3], 10_000, m["off"], m["wmap"], m["c64"],
                                m["y_pred"], m["std"], d_pr, cj=cj, site_strand=args_d[4], device=dev)
        t1.record()
        torch.cuda.synchronize()
    print("per-site test: %d sites in %.2f ms -> %.2f G sites/s" % (n, t0.elapsed_time(t1), n / t0.elapsed_time(t1) / 1e6))
    P, EXP, PV = (out[x].cpu().numpy() for x in ("P", "EXP", "PVAL"))
    assert not np.isnan(PV).any()
    # (2a) P * denom == d_pr[sub] up to one rounding
    row = np.array([m["index"][(int(c), int(s) // 10_000 * 10_000)] for c, s in zip(chrom[:200_000], start[:200_000])])
    den = np.where(strand[:200_000] < 0, out["DENOM_MINUS"].cpu().numpy()[row], out["DENOM_PLUS"].cpu().numpy()[row])
    fin = den > 0                                            # windows that are all N have denom 0 (P = inf, as in the reference)
    assert fin.mean() > 0.9 and np.all(np.isinf(P[:200_000][~fin]))
    np.testing.assert_allclose((P[:200_000] * den)[fin], d_pr[sub[:200_000]][fin], rtol=1e-15)
    # (2b) permutation invariance over all sites
    perm = torch.randperm(n, device=dev)
    out2 = kernels.site_test(args_d[0][perm], args_d[1][perm], args_d[2][perm], args_d[3][perm], 10_000, m["off"],
                             m["wmap"], m["c64"], m["y_pred"], m["std"], d_pr, cj=cj, site_strand=args_d[4][perm],
                             device=dev)
    assert torch.equal(out2["PVAL"], out["PVAL"][perm]) and torch.equal(out2["EXP"], out["EXP"][perm])
    # (1) subset through K6 as one-site elements, and through the oracle
    sel = rng.choice(np.flatnonzero(np.isfinite(P[:5_000_000])), 3000, replace=False)
    rp = pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2], "Y_TRUE": m["y_true"],
                       "Y_PRED": m["y_pred"], "STD": m["std"], "FLAG": m["flag"]})
    L = np.zeros((len(sel), 192))
    L[np.arange(len(sel)), sub[sel]] = 1.0
    res = gd.transfer_elements(gd.RegionModel(rp), m["c64"], d_pr, chrom[sel], strand[sel], np.arange(len(sel) + 1),
                               start[sel], start[sel] + 1, L_elt=L.reshape(len(sel), 192, 1))
    assert np.array_equal(res["P"][:, 0], P[sel]), np.abs(res["P"][:, 0] / P[sel] - 1).max()
    want = oracle.element_transfer(chrom[sel], strand[sel], np.arange(len(sel) + 1), start[sel], start[sel] + 1, L,
                                   10_000, m["index"], m["c64h"], m["y_pred"], m["std"], m["y_true"], m["flag"], d_pr)
    np.testing.assert_allclose(P[sel], want["P_SUM"], rtol=1e-9)
    a, t = oracle.normal_params_to_gamma(want["MU"], want["SIGMA"])
    e_, p_ = oracle.burden_test(k[sel], a, t * cj, want["P_SUM"])
    np.testing.assert_allclose(EXP[sel], e_, rtol=1e-9)
    assert_pvals_close(PV[sel], p_)
    # a site outside every window raises like the reference's KeyError
    with pytest.raises(KeyError):
        kernels.site_test([3], [int(lengths[2]) + 50_000], [5], [0.0], 10_000, m["off"], m["wmap"], m["c64"], m["y_pred"],
                          m["std"], d_pr, device=dev)


def test_config2_parity_sample_at_full_size(oracle):
    """BASELINE config 2 AT SIZE (3.1 Gb, 310 k windows, 1 M SNVs, 20 k genes): ~500 windows drawn uniformly over
    the whole genome -- chromosomes whose global offset exceeds 2^31 included --, the SNVs inside them and ~200 genes
    are recomputed by the CPU oracle from regenerated slices of the synthetic genome (oracle/parity_sample.py) and
    compared with the full GPU run: count rows and mutation contexts bit-exact, pretrain columns to 1e-9, the 13 NB
    p-values and the Fisher combination to 1e-6 in log10.  The same check runs inside bench.py after the timed
    region (`parity_sample` in its JSON line)."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    dev = torch.device(DEV)
    dg, ascii_d, d = bench.build_workload(3.1e9, seed=1, device=dev)
    del ascii_d
    di = bench.DeviceInputs(d, dev)
    res = bench.hot_path_step(dg, di, d, None)
    torch.cuda.synchronize()
    out = bench.parity_sample(dg, d, di, res, seed=1, n_windows=500, n_genes=200)
    assert out["ok"], out
    # every synthetic gene holds countable context, so every result is finite: one gene with R_SIZE = 0 (Pi_INDEL = inf)
    # would zero the indel scale factor, and with it EXP_INDEL, of all genes
    for k, v in res.items():
        assert not v.is_floating_point() or bool(torch.isfinite(v).all()), k
    assert float(res["EXP_INDEL"].min()) > 0
    assert out["windows"] == 500 and out["genes"] == 200
    assert out["windows_beyond_2^31"] > 50, out           # ~30 % of hg19 lies beyond 2^31
    assert out["mutations"] > 500 and out["p_values"] > 500, out
    # the lane-bank kernel and the per-warp kernel agree on every row of the full table (a checksum of checksums)
    from digdriver_b200 import kernels, _lib
    c5 = torch.empty_like(di.counts5)
    c3 = torch.empty_like(di.counts3)
    kernels.count_contexts_fused53(dg, di.win_chrom, di.win_start, di.win_end, out5=c5, out3=c3, variant=_lib.SCAN_HEX)
    assert torch.equal(c5, di.counts5) and torch.equal(c3, di.counts3)
    assert int(di.counts5.sum(dim=1).max()) <= bench.WINDOW
    # EVERY window of the 3.1 Gb genome (309 990 x 1088 bins) and the genome-wide totals against the C oracle, one
    # chromosome at a time: the synthetic genome is regenerated on the host from the global position alone
    import time
    from oracle import parity_sample as ps
    t0 = time.time()
    allw = ps.check_all_windows(d["lengths"], dg.chrom_off, 1, d["wins"], lambda a, b: di.counts5[a:b].cpu().numpy(),
                                lambda a, b: di.counts3[a:b].cpu().numpy(), di.totals5.cpu().numpy(), di.totals3.cpu().numpy())
    assert allw["ok"] and allw["windows"] == len(d["wins"]), allw
    print("full-size parity: %d windows x (1024 + 64) bins and both totals equal the C oracle bit for bit (%.1f s of host work)"
          % (allw["windows"], time.time() - t0))
