"""Exact host references for the test stage and the per-position test (numpy and math.fsum only).

A float64 kernel result is judged against the correctly rounded value of the same real-number expression, so a
bound in units of u = 2^-53 measures the kernel's own rounding and nothing else:

- exact_dot(a, B): the correctly rounded sum_j a_j B_ij of every row, from exact product splits and math.fsum.
- exact_dot_int(a, R): the same for an integer matrix R, exact in int64 limbs (fast enough for every window).
- warp_dot_model(a, B): the summation order of the warp kernels (K6, dig_window_denominators) in numpy.
- gene_transfer_ref(...): K6 gene / element mode with every sum exact.
- tabulate_genes_ref(...): K5 gene mode from np.unique.
- position_layout_ref, kmer_keys_ref, position_norm_ref, position_model_ref, position_obs_ref: K8's centres and bins,
  k-mer keys, exact normaliser, arithmetic in the kernel's order, and observed counts and positions.
"""
import math

import numpy as np

from oracle.dig_oracle import ideal_overlaps

U = 2.0 ** -53
_SPLIT = 134217729.0                      # 2^27 + 1: Veltkamp's splitter for 53-bit significands


def _split(x):
    c = _SPLIT * x
    hi = c - (c - x)
    return hi, x - hi


def two_prod(a, b):
    """p, e with p = fl(a b) and p + e == a b exactly (Dekker's TwoProduct, no FMA needed).  Exact while every nonzero
    factor and product lies between 1e-290 and 1e290 in magnitude: the splits then neither overflow nor underflow."""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact_dot(a, B):
    """Correctly rounded sum_j a[j] * B[i, j] of every row i of B (float64 [n_row]); domain as two_prod."""
    a = np.asarray(a, dtype=np.float64)
    B = np.atleast_2d(np.asarray(B, dtype=np.float64))
    p, e = two_prod(a[None, :], B)
    parts = np.concatenate([p, e], axis=1)
    return np.array([math.fsum(row) for row in parts])


_LIMB = 21                                # |R| < 2^31 times a 21-bit limb stays below 2^52 per product
_COLS = 2048                             # columns per int64 matrix product: 2048 * 2^31 * 2^21 = 2^63


def exact_dot_int(a, R):
    """Correctly rounded sum_j a[j] * R[i, j] for an integer matrix R (|R| < 2^31, any number of columns) and finite a
    whose result is a normal float64.  Every a_j is an integer multiple of 2^e0 (e0 = the smallest exponent of its
    last significand bit), so the sum is 2^e0 times an integer, formed exactly from int64 products of 21-bit limbs
    over blocks of at most 2048 columns and combined as Python integers."""
    a = np.asarray(a, dtype=np.float64)
    R = np.atleast_2d(np.asarray(R))
    assert R.dtype.kind in "iu" and R.shape[1] == a.size
    R = R.astype(np.int64)
    assert R.size == 0 or np.abs(R).max() < 2 ** 31
    assert np.all(np.isfinite(a))
    nz = a != 0
    if not nz.any():
        return np.zeros(R.shape[0])
    f, ex = np.frexp(a)                                      # a = f 2^ex, 0.5 <= |f| < 1
    m = (f * 2.0 ** 53).astype(np.int64)                     # exact: a = m 2^(ex - 53)
    e0 = int((ex - 53)[nz].min())
    M = [int(mj) << int(xj - 53 - e0) if mj else 0 for mj, xj in zip(m, ex)]   # a_j = M_j 2^e0, Python ints
    n_limb = max(abs(v).bit_length() for v in M) // _LIMB + 1
    mask = (1 << _LIMB) - 1
    total = np.zeros(R.shape[0], dtype=object)
    for k in range(n_limb):
        # signed limbs: M_j = sum_k sign_j limb_jk 2^(21 k)
        limb = np.array([(1 if v >= 0 else -1) * ((abs(v) >> (_LIMB * k)) & mask) for v in M], dtype=np.int64)
        if not limb.any():
            continue
        for c0 in range(0, a.size, _COLS):
            s = R[:, c0:c0 + _COLS] @ limb[c0:c0 + _COLS]    # |s| < 2048 * 2^52: exact in int64
            total = total + (s.astype(object) << (_LIMB * k))
    # Python's int / int is correctly rounded
    if e0 >= 0:
        return np.array([float(t << e0) for t in total])
    den = 1 << -e0
    return np.array([t / den for t in total])


def butterfly(x):
    """The xor-shuffle warp sum over the last axis (32 lanes), offsets 16, 8, 4, 2, 1: every lane ends with the same
    value; lane 0's is returned."""
    x = np.array(x, dtype=np.float64)
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        x = x + x[..., lanes ^ o]
    return x[..., 0]


def warp_dot_model(a, B, lanes=32):
    """sum_j a[j] B[i, j] (a [192], or [n_row, 192] for per-row weights) over 192 terms in the warp kernels' order:
    lane l holds terms l + 32 t, sums them serially over t, then the lanes combine through the xor butterfly.  Every
    product is rounded here; the kernels may fuse it into the addition (one rounding fewer), so the model is never more
    accurate than the device.
    lanes < 32 drops the terms of lanes >= `lanes` (a model of a broken kernel for the tests of the bounds)."""
    a = np.asarray(a, dtype=np.float64)
    B = np.atleast_2d(np.asarray(B, dtype=np.float64))
    acc = np.zeros((B.shape[0], 32))
    for t in range(B.shape[1] // 32):
        acc = acc + a[..., 32 * t:32 * t + 32] * B[:, 32 * t:32 * t + 32]
    acc[:, lanes:] = 0.0
    return butterfly(acc)


def revcomp64():
    """rc[c] = index of the reverse complement of trinucleotide c (2-bit codes, first base most significant)."""
    c = np.arange(64)
    b0, b1, b2 = (c >> 4) & 3, (c >> 2) & 3, c & 3
    return ((3 - b2) << 4) | ((3 - b1) << 2) | (3 - b0)


def _rel_err_u(got, want):
    """|got - want| / |want| in units of u (0 where both are equal, inf where want is 0 and got is not)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.abs(got - want) / np.abs(want) / U
    r[got == want] = 0.0
    return r


def gene_windows(chrom, blk_ptr, blk_start, blk_end, window, win_map_off, win_map):
    """Rows of the windows each element overlaps (ideal_overlaps of its blocks, ascending), as (owner, row) arrays."""
    owner, rows = [], []
    for e in range(len(chrom)):
        a, b = blk_ptr[e], blk_ptr[e + 1]
        wins = ideal_overlaps(blk_start[a:b], blk_end[a:b], window)
        wn = np.asarray(wins, dtype=np.int64) // window
        r = win_map[win_map_off[chrom[e]] + wn]
        assert np.all(r >= 0) and np.all(wn < win_map_off[chrom[e] + 1] - win_map_off[chrom[e]])
        owner.append(np.full(len(r), e, dtype=np.int64))
        rows.append(r.astype(np.int64))
    return np.concatenate(owner), np.concatenate(rows)


def gene_transfer_ref(chrom, strand, blk_ptr, blk_start, blk_end, window, win_map_off, win_map, win_counts,
                      y_pred, std, y_true, flag, d_pr, L=None, blk_counts=None):
    """K6 with every sum exact.  MU, R_OBS: one correctly rounded sum each; SIGMA = sqrt of the correctly rounded sum
    of the squares as the kernel forms them (std * std, rounded); R_SIZE, N_WIN, FLAG, ELT_SIZE exact integers;
    D = sum_j d_pr[j] R[j / 3] (R reverse-complemented for minus-strand elements) and N_c = sum_j d_pr[j] L[j, c] exact,
    P_c = N_c / D, one rounding.  Where D = 0 P is what the reference's (d_pr / 0 * L).sum() gives (NaN or inf).
    L [E, 192, n_col] (gene mode) or blk_counts [n_blk, 64] (element mode: L[j] = the summed block counts of j / 3)."""
    E = len(chrom)
    owner, rows = gene_windows(chrom, blk_ptr, blk_start, blk_end, window, win_map_off, win_map)
    cnt = np.bincount(owner, minlength=E)
    R64 = np.zeros((E, 64), dtype=np.int64)
    np.add.at(R64, owner, win_counts[rows].astype(np.int64))
    minus = np.asarray(strand) < 0
    R64[minus] = R64[minus][:, revcomp64()]
    sq = std * std
    out = {"N_WIN": cnt, "R_SIZE": R64.sum(axis=1), "MU": np.zeros(E), "SIGMA": np.zeros(E), "R_OBS": np.zeros(E),
           "FLAG": np.zeros(E, dtype=bool)}
    starts = np.concatenate([[0], np.cumsum(cnt)])
    for e in range(E):
        r = rows[starts[e]:starts[e + 1]]
        out["MU"][e] = math.fsum(y_pred[r])
        out["SIGMA"][e] = math.sqrt(math.fsum(sq[r]))
        out["R_OBS"][e] = math.fsum(y_true[r])
        out["FLAG"][e] = bool(np.any(flag[r]))
    sub = np.arange(192) // 3
    bown = np.repeat(np.arange(E), np.diff(blk_ptr))
    if blk_counts is not None:
        L64 = np.zeros((E, 64), dtype=np.int64)
        np.add.at(L64, bown, np.asarray(blk_counts, dtype=np.int64))
        L = L64[:, sub][:, :, None].astype(np.float64)
        out["ELT_SIZE"] = L64.sum(axis=1)
    else:
        L = np.asarray(L, dtype=np.float64)
        out["ELT_SIZE"] = np.zeros(E, dtype=np.int64)
        np.add.at(out["ELT_SIZE"], bown, np.asarray(blk_end, dtype=np.int64) - np.asarray(blk_start) + 1)
    D = exact_dot(d_pr, R64[:, sub].astype(np.float64))
    N = np.stack([exact_dot(d_pr, L[:, :, c]) for c in range(L.shape[2])], axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        P = N / D[:, None]
        zero = D == 0
        if zero.any():
            P[zero] = ((d_pr / 0.0)[None, :, None] * L[zero]).sum(axis=1)
    out["D"], out["N"], out["P"] = D, N, P
    return out


def tabulate_genes_ref(gene, sample, cls, n_gene, cap=None):
    """K5 gene mode: per (gene, sample) the class counts (SYN, MIS, NONS, SPL, INDEL), each capped at `cap`, summed per
    gene (obs [n_gene, 5]); nsamp [n_gene, 7] counts the samples with a SYN / MIS / NONS / SPL / TRUNC (NONS or SPL) /
    NONSYN (MIS, NONS or SPL) / INDEL mutation.  Rows with gene < 0 or class > 4 are ignored; genes >= n_gene are
    tabulated but not reported."""
    gene, sample, cls = (np.asarray(x, dtype=np.int64) for x in (gene, sample, cls))
    keep = (gene >= 0) & (cls <= 4)
    g, s, c = gene[keep], sample[keep], cls[keep]
    keys, inv = np.unique(g * (1 << 32) + s, return_inverse=True)
    tab = np.zeros((len(keys), 5), dtype=np.int64)
    np.add.at(tab, (inv.ravel(), c), 1)
    kg = keys >> 32
    mine = kg < n_gene
    kg, tab = kg[mine], tab[mine]
    capped = tab if cap is None else np.minimum(tab, cap)
    obs = np.zeros((n_gene, 5), dtype=np.int64)
    np.add.at(obs, kg, capped)
    has = tab > 0
    flags = np.stack([has[:, 0], has[:, 1], has[:, 2], has[:, 3], has[:, 2] | has[:, 3],
                      has[:, 1] | has[:, 2] | has[:, 3], has[:, 4]], axis=1)
    nsamp = np.zeros((n_gene, 7), dtype=np.int64)
    np.add.at(nsamp, kg, flags.astype(np.int64))
    return obs, nsamp


# ---------------------------------------------------------------- K8: the per-position / per-bin hotspot test

def position_layout_ref(chrom_len, reg_chrom, reg_start, reg_end, n_up, n_down, binsize):
    """Per region: its first centre (chromosome coordinate), its number of positions and its number of bins, and the
    CSR bin_ptr [n_reg + 1].  The rules of fetch_sequence (sequence_tools.py:21-29) and count_sequence_context
    (:65-78): START == 0 becomes n_up; the fetched string is [START - n_up, END + n_down), which faidx clips at the
    chromosome end (empty when it starts at or past the end); its centres are the bases with n_up bases before and
    n_down after them inside the string."""
    n = len(reg_chrom)
    first, n_pos = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
    for r in range(n):
        L = int(chrom_len[int(reg_chrom[r])])
        start, end = int(reg_start[r]), int(reg_end[r])
        if start == 0:
            start = n_up
        assert start >= n_up, "0 < START < n_up: the reference raises"
        f0, f1 = start - n_up, end + n_down
        f0, f1 = min(f0, L), min(f1, L)
        first[r] = f0 + n_up
        n_pos[r] = max(f1 - f0 - n_up - n_down, 0)
    n_bin = (n_pos + binsize - 1) // binsize
    return first, n_pos, n_bin, np.concatenate([[0], np.cumsum(n_bin)]).astype(np.int64)


_CODE = np.full(256, -1, dtype=np.int64)
for _i, _b in enumerate(b"ACGT"):
    _CODE[_b] = _i
    _CODE[_b | 0x20] = _i                    # the synthetic genome is half lower case: the reference upper-cases it


def kmer_keys_ref(ascii, off, centres, n_up, n_down):
    """(key, valid) of the k-mer [c - n_up, c + n_down] of every centre c: key = its base-4 index with the first
    base most significant (mk_context_sequences order), valid = all of its bases are one of ACGTacgt.
    ascii[i] is the base at coordinate off + i."""
    ascii = np.asarray(ascii, dtype=np.uint8)
    idx = np.asarray(centres, dtype=np.int64) - off - n_up
    key = np.zeros(idx.shape, dtype=np.int64)
    valid = np.ones(idx.shape, dtype=bool)
    for j in range(n_up + n_down + 1):
        c = _CODE[ascii[idx + j]]
        valid &= c >= 0
        key = key * 4 + np.maximum(c, 0)
    return key, valid


def position_norm_ref(s_prob, key, valid, region, n_reg):
    """The exact normaliser of every region: the correctly rounded sum_k counts[r, k] s_prob[k], with the context
    counts tabulated from the reference keys (region[i] = region of position i).  Returns (norm, counts)."""
    K = len(s_prob)
    counts = np.bincount(region[valid] * K + key[valid], minlength=n_reg * K).reshape(n_reg, K)
    return exact_dot_int(s_prob, counts), counts


def position_model_ref(s_prob, key, valid, n_pos, norm, mu, sigma, binsize):
    """K8's arithmetic in the kernel's order, for regions whose positions are concatenated in key / valid (n_pos
    each): q = s_prob[key] / norm (0 for an invalid k-mer), pt = q summed position by position over each bin (the last
    bin padded with +0.0), exp = pt mu, alpha = (mu mu) / (sigma sigma), theta = (sigma sigma) / mu and
    p = 1 / (pt theta + 1), every operation rounded once.  Given the kernel's own norm this is bit-identical to it.
    Returns dict(pt, exp, alpha, p) per bin (alpha repeated over the region's bins)."""
    n_pos = np.asarray(n_pos, dtype=np.int64)
    n_bin = (n_pos + binsize - 1) // binsize
    reg = np.repeat(np.arange(len(n_pos)), n_pos)
    within = np.arange(len(reg)) - np.repeat(np.cumsum(n_pos) - n_pos, n_pos)
    bin_of = np.repeat(np.cumsum(n_bin) - n_bin, n_pos) + within // binsize
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(valid, np.asarray(s_prob)[key], 0.0) / np.asarray(norm)[reg]
    Q = np.zeros(int(n_bin.sum()) * binsize)
    Q[bin_of * binsize + within % binsize] = q
    Q = Q.reshape(-1, binsize)
    pt = np.zeros(Q.shape[0])
    for j in range(binsize):
        pt = pt + Q[:, j]
    m, s = np.repeat(np.asarray(mu, dtype=np.float64), n_bin), np.repeat(np.asarray(sigma, dtype=np.float64), n_bin)
    with np.errstate(divide="ignore", invalid="ignore"):
        theta = (s * s) / m
        return dict(pt=pt, exp=pt * m, alpha=(m * m) / (s * s), p=1.0 / (pt * theta + 1.0), q=q, bin_of=bin_of)


def position_obs_ref(mut_chrom, mut_start, reg_chrom, first, n_pos, bin_ptr, binsize):
    """obs per bin (mutation rows whose (chromosome, START) is a position of the bin, duplicates counted) and pos per
    bin (the mean of its positions, first + b binsize + (n_in_bin - 1) / 2, exact in float64)."""
    keys, cnt = np.unique((np.asarray(mut_chrom, dtype=np.int64) << 32) | np.asarray(mut_start, dtype=np.int64),
                          return_counts=True)
    rc = np.asarray(reg_chrom, dtype=np.int64)
    lo = np.searchsorted(keys, (rc << 32) | first)
    hi = np.searchsorted(keys, (rc << 32) | (first + n_pos))
    nh = hi - lo
    reg = np.repeat(np.arange(len(rc)), nh)
    k = np.repeat(lo, nh) + np.arange(int(nh.sum())) - np.repeat(np.cumsum(nh) - nh, nh)
    obs = np.zeros(int(bin_ptr[-1]), dtype=np.int64)
    np.add.at(obs, bin_ptr[reg] + ((keys[k] & 0xFFFFFFFF) - first[reg]) // binsize, cnt[k])
    n_bin = np.diff(bin_ptr)
    reg_b = np.repeat(np.arange(len(rc)), n_bin)
    b = np.arange(int(bin_ptr[-1])) - bin_ptr[reg_b]
    n_in = np.minimum(binsize, n_pos[reg_b] - b * binsize)
    pos = (first[reg_b] + b * binsize).astype(np.float64) + 0.5 * (n_in - 1).astype(np.float64)
    return obs, pos
