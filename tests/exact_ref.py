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
- cds_engine(...): the gene annotation and codon rules over a whole gene set, vectorised; from it cds_table_ref (K9a),
  annotate_ref (K9b), codon_records_ref (K9c), snv_codons_ref (K9d); codon_transfer_ref (K10) from the codon records.
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


def int_limbs(a, limb=_LIMB):
    """Integer form of finite float64 a: a_j = sum_k limbs[k, j] 2^(limb k) 2^e0 exactly, with signed limbs of `limb`
    bits (int64 [n_limb, len(a)]).  Returns (limbs, e0)."""
    a = np.asarray(a, dtype=np.float64)
    assert np.all(np.isfinite(a))
    nz = a != 0
    if not nz.any():
        return np.zeros((1, a.size), np.int64), 0
    f, ex = np.frexp(a)                                      # a = f 2^ex, 0.5 <= |f| < 1
    m = (f * 2.0 ** 53).astype(np.int64)                     # exact: a = m 2^(ex - 53)
    e0 = int((ex - 53)[nz].min())
    M = [int(mj) << int(xj - 53 - e0) if mj else 0 for mj, xj in zip(m, ex)]   # a_j = M_j 2^e0, Python ints
    n_limb = max(abs(v).bit_length() for v in M) // limb + 1
    mask = (1 << limb) - 1
    limbs = np.array([[(1 if v >= 0 else -1) * ((abs(v) >> (limb * k)) & mask) for v in M] for k in range(n_limb)],
                     dtype=np.int64)
    return limbs, e0


def limbs_to_float(S, e0, limb=_LIMB):
    """Correctly rounded float64 of sum_k S[:, k] 2^(limb k) 2^e0 (S [n, n_limb] of integers, int64 or Python ints),
    through Python integers: Python's int / int is correctly rounded."""
    S = np.atleast_2d(np.asarray(S))
    total = np.zeros(S.shape[0], dtype=object)
    for k in range(S.shape[1]):
        total = total + (S[:, k].astype(object) << (limb * k))
    if e0 >= 0:
        return np.array([float(t << e0) for t in total], dtype=np.float64)
    return (total / (1 << -e0)).astype(np.float64)


def exact_dot_int(a, R):
    """Correctly rounded sum_j a[j] * R[i, j] for an integer matrix R (|R| < 2^31, any number of columns) and finite a
    whose result is a normal float64.  Every a_j is an integer multiple of 2^e0 (int_limbs), so the sum is 2^e0 times
    an integer, formed exactly from int64 products of 21-bit limbs over blocks of at most 2048 columns and combined as
    Python integers (limbs_to_float)."""
    a = np.asarray(a, dtype=np.float64)
    R = np.atleast_2d(np.asarray(R))
    assert R.dtype.kind in "iu" and R.shape[1] == a.size
    R = R.astype(np.int64)
    assert R.size == 0 or np.abs(R).max() < 2 ** 31
    limbs, e0 = int_limbs(a)
    S = np.zeros((R.shape[0], len(limbs)), dtype=object)
    for k, limb in enumerate(limbs):
        if not limb.any():
            continue
        for c0 in range(0, a.size, _COLS):
            s = R[:, c0:c0 + _COLS] @ limb[c0:c0 + _COLS]    # |s| < 2048 * 2^52: exact in int64
            S[:, k] = S[:, k] + s.astype(object)
    return limbs_to_float(S, e0)


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


# ---------------------------------------------------------------- K9a-K9d, K10: gene annotation and the codon test
#
# One vectorised engine restates the annotation rules of csrc/cdsannot.cu and the codon rules of csrc/codon.cu
# (DESIGN.md section 5) for a whole gene set: transcripts are the genes' inclusive blocks, reversed on minus-strand
# genes; bases come from the caller's reader (host bytes of each gene's span plus one base either side); amino acids
# from NCBI table 1 with the consequence rules of oracle/cds_annot.py; essential-splice positions from
# oracle/cds_annot.splice_positions, gene by gene.  Every output is an integer or a float64 sum in a stated order.

_NO = 255                                  # no site / no hit / a codon with an N
_ACGT = "ACGT"


def _codon_tables():
    """aa[c] (ASCII) of the 64 codons in ACGT index order (first base most significant), and the consequence code
    cons[c_ref, c_alt]: 0 Synonymous, 1 Missense, 2 Nonsense, 5 Stop_loss (the DIG_CDS_* codes)."""
    from oracle import cds_annot as O
    names = [a + b + c for a in _ACGT for b in _ACGT for c in _ACGT]
    aa = np.array([ord(O.CODON_TABLE[n]) for n in names], dtype=np.uint8)
    stop = aa == ord("*")
    cons = np.where(stop[None, :], 2, np.where(stop[:, None], 5, 1)).astype(np.uint8)
    cons[aa[:, None] == aa[None, :]] = 0
    return aa, cons


_AA64, _CONS64 = _codon_tables()
_BASE_CODE = np.full(256, 4, dtype=np.uint8)
for _i, _b in enumerate(b"ACGT"):
    _BASE_CODE[_b] = _BASE_CODE[_b | 0x20] = _i


def _gene_dict(strand, ptr, bs, be, e):
    return {"strand": int(strand[e]), "blocks": list(zip(bs[ptr[e]:ptr[e + 1]].tolist(), be[ptr[e]:ptr[e + 1]].tolist()))}


def cds_engine(read, chrom_len, genes, donor=(1, 2, 5), acceptor=(1, 2), chunk=2000):
    """The annotation and codon rules over every gene.  read(c, lo, n) returns the n bytes of chromosome c (genome
    index) from position lo; genes = (chrom, strand, ptr, blk_start, blk_end) with inclusive, strictly ascending blocks.
    Returns a dict: T [E] (CDS length), PTR [E+1] (floor(T / 3) codons per gene), per codon POS [n, 3], CC [n] (codon
    code 16 b0 + 4 b1 + b2 of the transcript bases, 255 with an N), BIN / CLASS [n, 9], REF_AA [n], N_SITES [n]; per
    gene L [E, 192, 4] (int64) and FLAGS [E]; SPLICE_KEY (sorted gene << 32 | position of every essential-splice
    position).  Genes are processed `chunk` at a time, so only that many spans are in memory at once."""
    from oracle import cds_annot as O
    chrom, strand, ptr, bs, be = (np.asarray(x) for x in genes)
    ptr, bs, be = ptr.astype(np.int64), bs.astype(np.int64), be.astype(np.int64)
    chrom_len = np.asarray(chrom_len, dtype=np.int64)
    E = len(chrom)
    blen = be - bs + 1
    owner = np.repeat(np.arange(E), np.diff(ptr))
    T = np.bincount(owner, weights=blen, minlength=E).astype(np.int64)
    nc = T // 3
    cptr = np.concatenate([[0], np.cumsum(nc)]).astype(np.int64)
    n = int(cptr[-1])
    out = {"T": T, "PTR": cptr, "POS": np.zeros((n, 3), np.int64), "CC": np.zeros(n, np.uint8),
           "BIN": np.full((n, 9), _NO, np.uint8), "CLASS": np.full((n, 9), _NO, np.uint8),
           "REF_AA": np.zeros(n, np.uint8), "N_SITES": np.zeros(n, np.uint8),
           "L": np.zeros((E, 192, 4), np.int64), "FLAGS": np.zeros(E, np.int32)}
    rc = revcomp64()
    splice_keys = []
    for g0 in range(0, E, chunk):
        g1 = min(g0 + chunk, E)
        ge = np.arange(g0, g1)
        Lc = chrom_len[chrom[ge]]
        lo = np.maximum(bs[ptr[ge]] - 1, 0)
        hi = np.minimum(be[ptr[ge + 1] - 1] + 2, Lc)
        code = _BASE_CODE[np.concatenate([np.asarray(read(int(chrom[e]), int(a), int(b - a)), dtype=np.uint8)
                                          for e, a, b in zip(ge, lo, hi)])]
        boff = np.concatenate([[0], np.cumsum(hi - lo)])[:-1] - lo        # buffer index of (gene, p) = boff + p
        # CDS bases in genomic order, then their transcript index
        b0, b1 = ptr[g0], ptr[g1]
        bl = blen[b0:b1]
        nb = int(bl.sum())
        blk = np.repeat(np.arange(b0, b1), bl)
        gpos = bs[blk] + np.arange(nb) - np.repeat(np.cumsum(bl) - bl, bl)
        gown = owner[blk]
        loc = gown - g0
        Tg = T[ge]
        tstart = np.concatenate([[0], np.cumsum(Tg)])[:-1]
        i_in_gene = np.arange(nb) - tstart[loc]
        minus_b = strand[gown] < 0
        tx = tstart[loc] + np.where(minus_b, Tg[loc] - 1 - i_in_gene, i_in_gene)
        # transcript-ordered base, context and position
        idx = boff[loc] + gpos
        Lb = chrom_len[chrom[gown]]
        has_ctx = (gpos >= 1) & (gpos + 1 < Lb)
        i0, i2 = np.where(has_ctx, idx - 1, idx), np.where(has_ctx, idx + 1, idx)
        t3 = np.stack([code[i0], code[idx], code[i2]], axis=1).astype(np.int64)
        ok = has_ctx & (t3 < 4).all(axis=1)
        ctx_g = 16 * t3[:, 0] + 4 * t3[:, 1] + t3[:, 2]
        ctx = np.where(ok, np.where(minus_b, rc[np.where(ok, ctx_g, 0)], ctx_g), -1)
        base = t3[:, 1]
        tb = np.where(base < 4, np.where(minus_b, 3 - base, base), 4)
        TB, CTX, TPOS = (np.empty(nb, np.int64) for _ in range(3))
        TB[tx], CTX[tx], TPOS[tx] = tb, ctx, gpos
        # codons
        ncg = nc[ge]
        cown = np.repeat(np.arange(g1 - g0), ncg)
        k = np.arange(int(ncg.sum())) - np.repeat(np.cumsum(ncg) - ncg, ncg)
        ti = tstart[cown][:, None] + 3 * k[:, None] + np.arange(3)[None, :]
        cb, cx = TB[ti], CTX[ti]
        has_n = (cb >= 4).any(axis=1)
        cc = np.where(has_n, 0, 16 * cb[:, 0] + 4 * cb[:, 1] + cb[:, 2])
        sl = slice(int(cptr[g0]), int(cptr[g1]))
        out["POS"][sl] = TPOS[ti]
        out["CC"][sl] = np.where(has_n, _NO, cc)
        out["REF_AA"][sl] = np.where(has_n, 0, _AA64[cc])
        bins = np.full((len(k), 9), _NO, np.int64)
        clss = np.full((len(k), 9), _NO, np.int64)
        Lg = np.zeros((g1 - g0) * 768, np.int64)
        for j in range(3):
            shift = 2 * (2 - j)
            for r in range(3):
                a = r + (r >= cb[:, j])
                new = (cc & ~(3 << shift)) | (a << shift)
                cls = _CONS64[cc, new].astype(np.int64)
                live = ~has_n & (cx[:, j] >= 0)
                b = 3 * cx[:, j] + r
                inL = live & (cls != 5)
                Lg += np.bincount(cown[inL] * 768 + b[inL] * 4 + cls[inL], minlength=len(Lg))
                site = live & ((cls == 1) | (cls == 2))
                bins[site, 3 * j + r] = b[site]
                clss[site, 3 * j + r] = cls[site]
        out["BIN"][sl], out["CLASS"][sl] = bins, clss
        out["N_SITES"][sl] = (bins != _NO).sum(axis=1)
        # flags: the trailing partial codon counts for the N flag but not for the stop flag
        flags = np.where(Tg % 3 != 0, 1, 0)
        nown = np.repeat(np.arange(g1 - g0), Tg)
        flags |= np.where(np.bincount(nown[TB >= 4], minlength=g1 - g0) > 0, 2, 0)
        stop = ~has_n & (_AA64[cc] == ord("*")) & (k < ncg[cown] - 1)
        flags |= np.where(np.bincount(cown[stop], minlength=g1 - g0) > 0, 4, 0)
        out["FLAGS"][g0:g1] = flags
        # essential-splice positions, gene by gene from the plain-Python rule
        se, sp = [], []
        for e in ge:
            q = O.splice_positions(_gene_dict(strand, ptr, bs, be, e), donor, acceptor)
            se += [e] * len(q)
            sp += q
        se, sp = np.asarray(se, np.int64), np.asarray(sp, np.int64)
        splice_keys.append((se << 32) | sp)
        sl_loc = se - g0
        si = boff[sl_loc] + sp
        sLc = chrom_len[chrom[se]]
        sok = (sp >= 1) & (sp + 1 < sLc)
        s3 = np.stack([code[np.where(sok, si - 1, si)], code[si], code[np.where(sok, si + 1, si)]], axis=1).astype(np.int64)
        sok &= (s3 < 4).all(axis=1)
        sctx = 16 * s3[:, 0] + 4 * s3[:, 1] + s3[:, 2]
        sctx = np.where(strand[se] < 0, rc[sctx & 63], sctx)
        for r in range(3):
            Lg += np.bincount(sl_loc[sok] * 768 + (3 * sctx[sok] + r) * 4 + 3, minlength=len(Lg))
        out["L"][g0:g1] = Lg.reshape(-1, 192, 4)
    out["SPLICE_KEY"] = np.sort(np.concatenate(splice_keys)) if splice_keys else np.zeros(0, np.int64)
    return out


def cds_table_ref(eng):
    """K9a: L [E, 192, 4] (Synonymous, Missense, Nonsense, Essential_Splice) as float64, and the flags."""
    return eng["L"].astype(np.float64), eng["FLAGS"]


def codon_records_ref(eng):
    """K9c: PTR, POS [n, 3], BIN / CLASS [n, 9], REF_AA, N_SITES."""
    return {k: eng[k] for k in ("PTR", "POS", "BIN", "CLASS", "REF_AA", "N_SITES")}


def _transcript_index(genes, T, e, p):
    """Transcript index of position p in gene e (arrays), -1 where p is not a CDS base of that gene."""
    chrom, strand, ptr, bs, be = genes
    ptr, bs, be = (np.asarray(x, dtype=np.int64) for x in (ptr, bs, be))
    e, p = np.asarray(e, dtype=np.int64), np.asarray(p, dtype=np.int64)
    owner = np.repeat(np.arange(len(ptr) - 1, dtype=np.int64), np.diff(ptr))
    blen = be - bs + 1
    before = np.concatenate([[0], np.cumsum(blen)])[:-1] - np.concatenate([[0], np.cumsum(T)])[:-1][owner]
    b = np.searchsorted((owner << 32) | bs, (e << 32) | p, side="right") - 1
    bc = np.clip(b, 0, max(len(bs) - 1, 0))
    hit = (b >= ptr[e]) & (b < ptr[e + 1]) & (p <= be[bc]) & (p >= bs[bc])
    i = before[bc] + p - bs[bc]
    t = np.where(np.asarray(strand)[e] < 0, T[e] - 1 - i, i)
    return np.where(hit, t, -1)


def _codon_of(eng, genes, e, p):
    """(codon index or -1, phase j, transcript base of p or 4) of position p in gene e."""
    t = _transcript_index(genes, eng["T"], e, p)
    k = np.where(t >= 0, t // 3, 0)
    ok = (t >= 0) & (k < np.diff(eng["PTR"])[e])
    ci = np.where(ok, eng["PTR"][e] + k, -1)
    cc = np.where(ok, eng["CC"][np.maximum(ci, 0)], _NO).astype(np.int64)
    j = np.where(ok, t - 3 * k, 0)
    tb = np.where(cc != _NO, (cc >> (2 * (2 - j))) & 3, 4)
    return np.where(cc != _NO, ci, -1), j, tb, cc


def annotate_ref(eng, genes, pair_gene, pos, alt):
    """K9b: class of the SNV (genomic ALT 0..3, anything else none) at pos in gene pair_gene: the coding consequence
    of a countable coding site (complete codon free of N), else 3 at an essential-splice position, else 255."""
    strand = np.asarray(genes[1])
    e, p, alt = (np.asarray(x, dtype=np.int64) for x in (pair_gene, pos, alt))
    ci, j, tb, cc = _codon_of(eng, genes, e, p)
    a = np.where(strand[e] < 0, 3 - alt, alt)
    coding = (ci >= 0) & (alt < 4) & (a != tb)
    shift = 2 * (2 - j)
    new = (np.where(cc == _NO, 0, cc) & ~(3 << shift)) | (np.clip(a, 0, 3) << shift)
    cls = np.where(coding, _CONS64[np.where(cc == _NO, 0, cc), new], _NO)
    key = (e << 32) | p
    sk = eng["SPLICE_KEY"]
    at = np.searchsorted(sk, key)
    splice = (at < len(sk)) & (sk[np.minimum(at, max(len(sk) - 1, 0))] == key) if len(sk) else np.zeros(len(e), bool)
    incds = _transcript_index(genes, eng["T"], e, p) >= 0
    cls = np.where(~incds & splice & (alt < 4), 3, cls)
    return cls.astype(np.uint8)


def snv_codons_ref(eng, genes, pair_gene, pos, ref, alt):
    """K9d: (codon, slot) of the SNV (genomic REF / ALT codes) at pos in gene pair_gene: a site only when REF and ALT
    are bases, differ, REF equals the genome's base and the slot holds a bin; (-1, 255) otherwise."""
    strand = np.asarray(genes[1])
    e, p, ref, alt = (np.asarray(x, dtype=np.int64) for x in (pair_gene, pos, ref, alt))
    ci, j, tb, _ = _codon_of(eng, genes, e, p)
    minus = strand[e] < 0
    rt, at = np.where(minus, 3 - ref, ref), np.where(minus, 3 - alt, alt)
    ok = (ci >= 0) & (ref < 4) & (alt < 4) & (ref != alt) & (rt == tb)
    slot = 3 * j + np.where(at > tb, at - 1, at)
    slot = np.where(ok, slot, 0)
    ok &= eng["BIN"][np.maximum(ci, 0), slot] != _NO
    return np.where(ok, ci, -1), np.where(ok, slot, _NO).astype(np.uint8)


def window_rows(win_map_off, win_map, chrom_num, wn):
    """Row of window number wn of chromosome number chrom_num in the dense window map, -1 where absent."""
    off = np.asarray(win_map_off, dtype=np.int64)
    c, wn = np.asarray(chrom_num, dtype=np.int64), np.asarray(wn, dtype=np.int64)
    inr = (c >= 0) & (c < len(off) - 1) & (wn >= 0)
    cc = np.where(inr, c, 0)
    inr &= wn < off[cc + 1] - off[cc]
    return np.where(inr, np.asarray(win_map)[np.where(inr, off[cc] + wn, 0)], -1).astype(np.int64)


def codon_transfer_ref(rec, gene_chrom_num, gene_strand, window, win_map_off, win_map, win_counts, y_pred, std, y_true,
                       flag, d_pr, denom_plus=None, denom_minus=None, exact=True):
    """K10 per codon from its window set: the sorted distinct floor(p / window) of the bases that carry a site, each
    looked up in the window map of the gene's chromosome NUMBER.  Exact: N_WIN (windows found), R_SIZE (their 64
    counts summed), FLAG (OR), MISSING (a window of the set is absent).  Sequential float64 sums from 0.0 in ascending
    window order: MU, SIGMA = sqrt(sum fl(s s)), R_OBS; PI_NUM = sum of d_pr[bin] in slot order.  PI_SUM (with the
    given per-window denominators, by strand) = fl(PI_NUM / their sequential sum): the kernel's order.  PI_SUM_EXACT =
    fl(sum d_pr[bin]) / fl(sum_j d_pr[j] R[j / 3]) with both sums correctly rounded and R the strand-ordered sum of the
    window counts -- nonc_model's P_SUM for a one-codon site set.  Codons without sites are all zero; MU, SIGMA,
    PI_SUM and PI_SUM_EXACT are NaN for a codon with a missing window.  exact=False skips PI_SUM_EXACT."""
    ptr, pos, bins = rec["PTR"], rec["POS"], rec["BIN"].astype(np.int64)
    n = len(bins)
    gene = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    minus = np.asarray(gene_strand)[gene] < 0
    cnum = np.asarray(gene_chrom_num, dtype=np.int64)[gene]
    has = (bins != _NO).reshape(n, 3, 3).any(axis=2)
    tested = has.any(axis=1)
    BIG = np.iinfo(np.int64).max
    w = np.sort(np.where(has, pos // window, BIG), axis=1)
    valid = w != BIG
    valid[:, 1:] &= w[:, 1:] != w[:, :-1]
    rows = np.where(valid, window_rows(win_map_off, win_map, cnum[:, None], np.where(valid, w, 0)), -1)
    present = valid & (rows >= 0)
    missing = (valid & (rows < 0)).any(axis=1)
    y_pred, std, y_true = (np.asarray(x, dtype=np.float64) for x in (y_pred, std, y_true))
    flag = np.asarray(flag).astype(bool)
    counts = np.asarray(win_counts, dtype=np.int64)
    rsum = counts.sum(axis=1)
    mu, var, ro = np.zeros(n), np.zeros(n), np.zeros(n)
    den = np.zeros(n)
    fl = np.zeros(n, bool)
    rsize = np.zeros(n, np.int64)
    for u in range(3):
        m, r = present[:, u], np.maximum(rows[:, u], 0)
        mu = np.where(m, mu + y_pred[r], mu)
        var = np.where(m, var + std[r] * std[r], var)
        ro = np.where(m, ro + y_true[r], ro)
        fl |= m & flag[r]
        rsize += np.where(m, rsum[r], 0)
        if denom_plus is not None:
            den = np.where(m, den + np.where(minus, denom_minus[r], denom_plus[r]), den)
    dp = np.concatenate([np.asarray(d_pr, dtype=np.float64), [0.0]])
    b9 = np.where(bins == _NO, 192, bins)
    num = np.zeros(n)
    for s in range(9):
        num = num + dp[b9[:, s]]
    nw = present.sum(axis=1)
    out = {"N_WIN": nw, "R_SIZE": rsize, "FLAG": fl, "MISSING": missing & tested, "R_OBS": ro, "PI_NUM": num}
    nan = np.full(n, np.nan)
    with np.errstate(divide="ignore", invalid="ignore"):
        out["MU"] = np.where(missing, nan, mu)
        out["SIGMA"] = np.where(missing, nan, np.sqrt(var))
        if denom_plus is not None:
            out["PI_SUM"] = np.where(missing, nan, np.where(nw > 0, num / den, 0.0))
    if not exact:
        return out
    # nonc_model's P_SUM: exact numerator and denominator, each rounded once, one division
    limbs, e0 = int_limbs(dp[:192])
    limbs193 = np.concatenate([limbs, np.zeros((len(limbs), 1), np.int64)], axis=1)
    S_num = np.stack([limbs193[k][b9].sum(axis=1) for k in range(len(limbs))], axis=1)
    g64 = limbs.reshape(len(limbs), 64, 3).sum(axis=2)               # sum_r limb[3 c + r]: R[j / 3] groups by c
    rc = revcomp64()
    Wp = np.stack([counts @ g64[k] for k in range(len(limbs))], axis=1)
    Wm = np.stack([counts @ g64[k][rc] for k in range(len(limbs))], axis=1)
    S_den = np.zeros((n, len(limbs)), np.int64)
    for u in range(3):
        m, r = present[:, u], np.maximum(rows[:, u], 0)
        S_den += np.where(m[:, None], np.where(minus[:, None], Wm[r], Wp[r]), 0)
    sel = np.flatnonzero(tested & ~missing)
    exact = np.zeros(n)
    if len(sel):
        with np.errstate(divide="ignore", invalid="ignore"):
            exact[sel] = limbs_to_float(S_num[sel], e0) / limbs_to_float(S_den[sel], e0)
    out["PI_SUM_EXACT"] = np.where(missing, nan, exact)
    return out
