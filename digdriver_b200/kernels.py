"""Tensor-level wrappers over the C ABI (include/dig_b200.h).

PyTorch is used only to own device memory and streams; every computation below is one of
the hand-written sm_100a kernels in csrc/, reached through ctypes with raw device pointers.
"""
import numpy as np
import torch

from . import _lib


def _stream(device, stream=None):
    st = stream if stream is not None else torch.cuda.current_stream(device)
    return st.cuda_stream


def _dev(x, dtype, device):
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype).contiguous()
    return torch.from_numpy(np.ascontiguousarray(x)).to(device=device, dtype=dtype)


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _tile_hint(reg_start, reg_end, tile_window):
    """Window size to pass as dig_scan_opts.tile_window: the caller's, or, for HOST arrays, the common length of the
    regions (it is only a hint: the kernel verifies it per group of windows on the device)."""
    if tile_window is not None:
        return int(tile_window)
    if isinstance(reg_start, torch.Tensor) or isinstance(reg_end, torch.Tensor):
        return 0
    s, e = np.asarray(reg_start), np.asarray(reg_end)
    if s.size == 0:
        return 0
    w = int(e.flat[0]) - int(s.flat[0])
    return w if w > 0 and bool(np.all(e - s == w)) else 0


def _scan_opts(dev, n_reg, variant, totals_limit_kb, workspace, tile_window=0, peer_rows=None, mc_rows=None, genome=None):
    """dig_scan_opts for one scan call: the device scratch the lane-bank kernel needs (caller-owned, sized by
    dig_scan_workspace_bytes) plus the A/B knobs.  peer_rows: device addresses (ints) of the trinucleotide row block in
    every rank's peer-mapped buffer (fused all-gather), mc_rows its multicast alias.  genome: its per-128-base N summary
    (DeviceGenome.nsum, None = none) goes with the call.
    Returns (struct, byref, workspace tensor to keep alive)."""
    import ctypes
    if workspace is None and n_reg > 0:
        nbytes = int(_lib.load().dig_scan_workspace_bytes(int(n_reg)))
        workspace = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    opts = _lib.ScanOpts(workspace.data_ptr() if workspace is not None else None,
                         workspace.numel() if workspace is not None else 0, int(variant), int(totals_limit_kb),
                         int(tile_window))
    if peer_rows:
        assert len(peer_rows) <= 8, "at most 8 peers"
        opts.n_peer_counts3 = len(peer_rows)
        for i, a in enumerate(peer_rows):
            opts.peer_counts3_d[i] = int(a)
        opts.mc_counts3_d = int(mc_rows) if mc_rows else None
    if genome is not None and getattr(genome, "nsum", None) is not None:
        # the summary lives in the mask's allocation, nsum_offset words after it
        assert genome.nsum.data_ptr() == genome.nmask.data_ptr() + 4 * genome.nsum_offset
        opts.nsum_offset_words = genome.nsum_offset
    return opts, ctypes.byref(opts), workspace


def peer_broadcast(src, dst_addrs, stream=None):
    """Copy the bytes of `src` (a contiguous device tensor, 16-byte aligned, a multiple of 16 bytes) to each device
    address in dst_addrs (peer-mapped buffers)."""
    import ctypes
    dev = src.device
    arr = (ctypes.c_void_p * len(dst_addrs))(*[int(a) for a in dst_addrs])
    with torch.cuda.device(dev):
        _lib.call("dig_peer_broadcast", src.data_ptr(), src.numel() * src.element_size(), arr, len(dst_addrs), _stream(dev, stream))


def scan_workspace(genome_or_device, n_reg):
    """Scratch tensor for count_contexts / count_contexts_fused53 (reuse it across calls on one stream)."""
    dev = getattr(genome_or_device, "device", genome_or_device)
    return torch.empty(int(_lib.load().dig_scan_workspace_bytes(int(n_reg))), dtype=torch.uint8, device=dev)


def count_contexts(genome, reg_chrom, reg_start, reg_end, n_up=1, n_down=1, strand=None,
                   want_totals=False, out=None, totals=None, stream=None, variant=_lib.SCAN_AUTO,
                   totals_limit_kb=0, workspace=None, tile_window=None, peer_rows=None, mc_rows=None):
    """K2/K4: per-region context histogram.

    genome: DeviceGenome.  reg_chrom: chromosome indices into the genome (int32).
    Returns (counts int32 [n, K] on device, totals int64 [K] on device or None)."""
    dev = genome.device
    rc = _dev(reg_chrom, torch.int32, dev)
    rs = _dev(reg_start, torch.int64, dev)
    re = _dev(reg_end, torch.int64, dev)
    st = _dev(strand, torch.int8, dev) if strand is not None else None
    n = rc.numel()
    K = 4 ** (n_up + n_down + 1)
    if out is None:
        out = torch.empty((n, K), dtype=torch.int32, device=dev)
    if want_totals and totals is None:
        totals = torch.zeros(K, dtype=torch.int64, device=dev)
    lane_bank = ((n_up, n_down) in ((2, 2), (1, 1)) and st is None and variant == _lib.SCAN_AUTO
                 and getattr(genome, "nsum", None) is not None)
    opts, opts_ref, workspace = _scan_opts(dev, n if lane_bank else 0, variant, totals_limit_kb,
                                           workspace if lane_bank else None,
                                           _tile_hint(reg_start, reg_end, tile_window) if lane_bank else 0,
                                           peer_rows, mc_rows, genome)
    with torch.cuda.device(dev):
        _lib.call("dig_count_contexts", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), rc.data_ptr(), rs.data_ptr(),
                  re.data_ptr(), _ptr(st), n, int(n_up), int(n_down), out.data_ptr(), _ptr(totals), opts_ref,
                  _stream(dev, stream))
    if lane_bank and n > 0:
        _lib.launch_count += 1          # lane-bank kernel + the per-warp kernel over its redo list
    return out, totals


def count_contexts_fused53(genome, reg_chrom, reg_start, reg_end, want_totals=False, out5=None, out3=None,
                           totals5=None, totals3=None, stream=None, variant=_lib.SCAN_AUTO, totals_limit_kb=0,
                           workspace=None, tile_window=None, peer_rows=None, mc_rows=None):
    """K2 fused: pentanucleotide and trinucleotide tables (+ totals) of the same regions in one pass.
    Returns (counts5 [n,1024], counts3 [n,64], totals5, totals3)."""
    dev = genome.device
    rc = _dev(reg_chrom, torch.int32, dev)
    rs = _dev(reg_start, torch.int64, dev)
    re = _dev(reg_end, torch.int64, dev)
    n = rc.numel()
    if out5 is None:
        out5 = torch.empty((n, 1024), dtype=torch.int32, device=dev)
    if out3 is None:
        out3 = torch.empty((n, 64), dtype=torch.int32, device=dev)
    if want_totals and totals5 is None:
        totals5 = torch.zeros(1024, dtype=torch.int64, device=dev)
        totals3 = torch.zeros(64, dtype=torch.int64, device=dev)
    lane_bank = variant == _lib.SCAN_AUTO and getattr(genome, "nsum", None) is not None
    opts, opts_ref, workspace = _scan_opts(dev, n if lane_bank else 0, variant, totals_limit_kb,
                                           workspace if lane_bank else None,
                                           _tile_hint(reg_start, reg_end, tile_window) if lane_bank else 0,
                                           peer_rows, mc_rows, genome)
    with torch.cuda.device(dev):
        _lib.call("dig_count_contexts_fused53", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), rc.data_ptr(), rs.data_ptr(),
                  re.data_ptr(), n, out5.data_ptr(), out3.data_ptr(), _ptr(totals5), _ptr(totals3), opts_ref,
                  _stream(dev, stream))
    if lane_bank and n > 0:
        _lib.launch_count += 1
    return out5, out3, totals5, totals3


def mutation_contexts(genome, mut_chrom, mut_start, mut_ref, n_up=1, n_down=1, stream=None):
    """K3: context index per mutation row (-1 = dropped by the reference).  Rows grouped by chromosome."""
    dev = genome.device
    mc = _dev(mut_chrom, torch.int32, dev)
    ms = _dev(mut_start, torch.int64, dev)
    mr = _dev(mut_ref, torch.uint8, dev)
    out = torch.empty(mc.numel(), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_mutation_contexts", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), mc.data_ptr(), ms.data_ptr(),
                  mr.data_ptr(), mc.numel(), int(n_up), int(n_down), out.data_ptr(), _stream(dev, stream))
    return out


def nb_pvalue_greater_midp(k, alpha, p, device="cuda:0", stream=None):
    """K7: 0.5 * nbinom.pmf(k, alpha, p) + betainc(k + 1, alpha, 1 - p) in FP64 on the GPU."""
    dev = torch.device(device)
    kd, ad, pd_ = (_dev(x, torch.float64, dev) for x in (k, alpha, p))
    out = torch.empty_like(kd)
    with torch.cuda.device(dev):
        _lib.call("dig_nb_pvalue_greater_midp", kd.data_ptr(), ad.data_ptr(), pd_.data_ptr(), kd.numel(),
                  out.data_ptr(), _stream(dev, stream))
    return out


def nb_burden_test(k, alpha, theta, pi, device="cuda:0", want_exp=True, stream=None):
    """K7 fused: EXP = ALPHA*THETA*Pi and the mid-p p-value with p = 1/(THETA*Pi+1)."""
    dev = torch.device(device)
    kd, ad, td, fd = (_dev(x, torch.float64, dev) for x in (k, alpha, theta, pi))
    pval = torch.empty_like(kd)
    exp = torch.empty_like(kd) if want_exp else None
    with torch.cuda.device(dev):
        _lib.call("dig_nb_burden_test", kd.data_ptr(), ad.data_ptr(), td.data_ptr(), fd.data_ptr(), kd.numel(),
                  _ptr(exp), pval.data_ptr(), _stream(dev, stream))
    return exp, pval


def fisher_combine2(p1, p2, device="cuda:0", stream=None):
    dev = torch.device(device)
    a, b = _dev(p1, torch.float64, dev), _dev(p2, torch.float64, dev)
    out = torch.empty_like(a)
    with torch.cuda.device(dev):
        _lib.call("dig_fisher_combine2", a.data_ptr(), b.data_ptr(), a.numel(), out.data_ptr(), _stream(dev, stream))
    return out


def _table_capacity(n_pairs):
    """Hash-table slots for up to n_pairs distinct keys: the rule lives in the library (dig_tabulate_capacity)."""
    return int(_lib.load().dig_tabulate_capacity(int(n_pairs)))


def _check_status(status, what, sink=None):
    """Raises for a non-zero device status word.  Reading it is a host synchronisation; callers on a
    stream-ordered hot path pass a list as `sink` and call check_deferred(sink) once at the end instead."""
    if sink is not None:
        sink.append((status, what))
        return
    code = int(status.item())
    if code == 1:
        raise _lib.DigError("%s: hash table overflow" % what)
    if code == 2:
        raise KeyError("%s: an element overlaps a window that is not in region_params "
                       "(the reference raises KeyError on the same input)" % what)
    if code == 3:
        raise _lib.DigError("%s: element window span exceeds the shared-memory bitmap" % what)
    if code != 0:
        raise _lib.DigError("%s: status %d" % (what, code))


def check_deferred(sink):
    """Checks (and clears) the device status words collected through a `status_sink` list."""
    pending, sink[:] = list(sink), []
    for status, what in pending:
        _check_status(status, what)


def tabulate_elements(blk_kstart, blk_kend, blk_elt, mut_kstart, mut_kend, mut_sample, mut_isindel,
                      n_elt, n_sample, max_muts_per_sample=10 ** 9, max_per_elt_per_sample=3 * 10 ** 9,
                      device="cuda:0", stream=None, sample_rows_mode=False, return_table=False, max_hits=None,
                      status_sink=None):
    """K5: (OBS_SAMPLES, OBS_SNV, OBS_INDEL) per element and the per-sample totals used for the
    hypermutator black-list.  Blocks need not be sorted.  Returns (obs int64 [n_elt,3], sample_tot [n_sample]).

    max_hits: an upper bound of the number of (mutation, element) pairs; with it the table is sized without
    reading the device-side hit count (no host synchronisation; an overflow still sets the status word)."""
    dev = torch.device(device)
    bks = np.asarray(blk_kstart, dtype=np.int64)
    order = np.argsort(bks, kind="stable")
    bks = bks[order]
    bke = np.asarray(blk_kend, dtype=np.int64)[order]
    belt = np.asarray(blk_elt, dtype=np.int32)[order]
    pmax = np.maximum.accumulate(bke) if len(bke) else bke
    t = {k: _dev(v, dt, dev) for k, v, dt in (
        ("bks", bks, torch.int64), ("bke", bke, torch.int64), ("pmax", pmax, torch.int64), ("belt", belt, torch.int32),
        ("mks", mut_kstart, torch.int64), ("mke", mut_kend, torch.int64), ("ms", mut_sample, torch.int32),
        ("mi", mut_isindel, torch.uint8))}
    n_blk, n_mut = len(bks), t["mks"].numel()
    sptr = _stream(dev, stream)
    with torch.cuda.device(dev):
        if max_hits is None:
            n_hits = torch.zeros(1, dtype=torch.int64, device=dev)
            _lib.call("dig_count_hits", t["bks"].data_ptr(), t["bke"].data_ptr(), t["pmax"].data_ptr(),
                      t["belt"].data_ptr(), n_blk, t["mks"].data_ptr(), t["mke"].data_ptr(), n_mut, n_hits.data_ptr(), sptr)
            max_hits = int(n_hits.item())
        cap = _table_capacity(max_hits)
        keys = torch.empty(cap, dtype=torch.int64, device=dev)
        snv = torch.empty(cap, dtype=torch.int32, device=dev)
        ind = torch.empty(cap, dtype=torch.int32, device=dev)
        sample_tot = torch.empty(max(n_sample, 1), dtype=torch.int64, device=dev)
        obs = torch.empty((max(n_elt, 1), 3), dtype=torch.int64, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.call("dig_tabulate_elements", t["bks"].data_ptr(), t["bke"].data_ptr(), t["pmax"].data_ptr(),
                  t["belt"].data_ptr(), n_blk, t["mks"].data_ptr(), t["mke"].data_ptr(), t["ms"].data_ptr(),
                  t["mi"].data_ptr(), n_mut, keys.data_ptr(), snv.data_ptr(), ind.data_ptr(), cap, n_sample,
                  sample_tot.data_ptr(), int(min(max_muts_per_sample, 2 ** 62)),
                  int(min(max_per_elt_per_sample, 2 ** 62)), n_elt, obs.data_ptr(), status.data_ptr(),
                  int(bool(sample_rows_mode)), sptr)
        _check_status(status, "dig_tabulate_elements", status_sink)
    if return_table:
        # the (element, sample) hash table itself: key = (element << 32 | sample) + 1, 0 = empty slot
        return obs[:n_elt], sample_tot[:n_sample], (keys, snv, ind)
    return obs[:n_elt], sample_tot[:n_sample]


def tabulate_genes(mut_gene, mut_sample, mut_class, n_gene, max_per_gene_per_sample=3 * 10 ** 9,
                   device="cuda:0", stream=None, status_sink=None):
    """K5 (genes): obs int64 [n_gene,5] (SYN, MIS, NONS, SPL, INDEL) and nsamp int64 [n_gene,7]
    (SYN, MIS, NONS, SPL, TRUNC, NONSYN, INDEL)."""
    dev = torch.device(device)
    mg, ms, mc = _dev(mut_gene, torch.int32, dev), _dev(mut_sample, torch.int32, dev), _dev(mut_class, torch.uint8, dev)
    n_mut = mg.numel()
    cap = _table_capacity(n_mut)
    with torch.cuda.device(dev):
        keys = torch.empty(cap, dtype=torch.int64, device=dev)
        cnt = torch.empty((cap, 5), dtype=torch.int32, device=dev)
        obs = torch.empty((max(n_gene, 1), 5), dtype=torch.int64, device=dev)
        nsamp = torch.empty((max(n_gene, 1), 7), dtype=torch.int64, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.call("dig_tabulate_genes", mg.data_ptr(), ms.data_ptr(), mc.data_ptr(), n_mut, keys.data_ptr(),
                  cnt.data_ptr(), cap, int(min(max_per_gene_per_sample, 2 ** 62)), n_gene, obs.data_ptr(),
                  nsamp.data_ptr(), status.data_ptr(), _stream(dev, stream))
        _check_status(status, "dig_tabulate_genes", status_sink)
    return obs[:n_gene], nsamp[:n_gene]


def element_transfer(elt_chrom, elt_strand, blk_ptr, blk_start, blk_end, window, win_map_off, win_map,
                     win_counts, y_pred, std, y_true, flag, d_pr, blk_counts=None, L_elt=None,
                     device="cuda:0", stream=None, max_span=None, status_sink=None):
    """K6.  Region-parameter arrays are [n_cohort, n_win] (1-D inputs are taken as one cohort), d_pr is
    [n_cohort, 192].  Returns a dict of device tensors (MU, SIGMA, R_OBS, FLAG: [n_cohort, n_elt];
    R_SIZE, ELT_SIZE, N_WIN: [n_elt]; P: [n_cohort, n_elt, n_col])."""
    dev = torch.device(device)
    ec, es = _dev(elt_chrom, torch.int32, dev), _dev(elt_strand, torch.int8, dev)
    bp, bs, be = (_dev(x, torch.int64, dev) for x in (blk_ptr, blk_start, blk_end))
    wmo, wm = _dev(win_map_off, torch.int64, dev), _dev(win_map, torch.int32, dev)
    wc = _dev(win_counts, torch.int32, dev)
    yp, sd, yt = (_dev(x, torch.float64, dev).reshape(-1, wc.shape[0]) for x in (y_pred, std, y_true))
    fl = _dev(np.asarray(flag).astype(np.uint8) if not isinstance(flag, torch.Tensor) else flag.to(torch.uint8),
              torch.uint8, dev).reshape(-1, wc.shape[0])
    dp = _dev(d_pr, torch.float64, dev).reshape(-1, 192)
    n_cohort = dp.shape[0]
    assert yp.shape[0] == n_cohort and sd.shape[0] == n_cohort and yt.shape[0] == n_cohort and fl.shape[0] == n_cohort
    n_elt = ec.numel()
    n_win = wc.shape[0]
    if blk_counts is not None:
        bc, Le, n_col = _dev(blk_counts, torch.int32, dev), None, 1
    else:
        Le = _dev(L_elt, torch.float64, dev)
        Le = Le.reshape(n_elt, 192, -1)
        bc, n_col = None, Le.shape[2]
    if max_span is None:
        max_span = element_max_span(bp, bs, be, window)
    out = {
        "MU": torch.empty((n_cohort, n_elt), dtype=torch.float64, device=dev),
        "SIGMA": torch.empty((n_cohort, n_elt), dtype=torch.float64, device=dev),
        "R_OBS": torch.empty((n_cohort, n_elt), dtype=torch.float64, device=dev),
        "FLAG": torch.empty((n_cohort, n_elt), dtype=torch.uint8, device=dev),
        "R_SIZE": torch.empty(n_elt, dtype=torch.int64, device=dev),
        "ELT_SIZE": torch.empty(n_elt, dtype=torch.int64, device=dev),
        "P": torch.empty((n_cohort, n_elt, n_col), dtype=torch.float64, device=dev),
        "N_WIN": torch.empty(n_elt, dtype=torch.int32, device=dev),
    }
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_element_transfer", ec.data_ptr(), es.data_ptr(), bp.data_ptr(), bs.data_ptr(), be.data_ptr(),
                  n_elt, int(window), int(wmo.numel()) - 1, wmo.data_ptr(), wm.data_ptr(), wc.data_ptr(), yp.data_ptr(),
                  sd.data_ptr(), yt.data_ptr(), fl.data_ptr(), n_win, n_cohort, dp.data_ptr(), _ptr(bc), _ptr(Le), n_col, max_span,
                  out["MU"].data_ptr(), out["SIGMA"].data_ptr(), out["R_OBS"].data_ptr(), out["FLAG"].data_ptr(),
                  out["R_SIZE"].data_ptr(), out["ELT_SIZE"].data_ptr(), out["P"].data_ptr(),
                  out["N_WIN"].data_ptr(), status.data_ptr(), _stream(dev, stream))
        _check_status(status, "dig_element_transfer", status_sink)
    return out


def element_max_span(blk_ptr, blk_start, blk_end, window):
    """Widest window span (in windows) of any element: sizes K6's shared-memory bitmap.  Host-side; cache it
    when the same annotation is used repeatedly."""
    def host(x):
        return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    bp_h, bs_h, be_h = host(blk_ptr).astype(np.int64), host(blk_start).astype(np.int64), host(blk_end).astype(np.int64)
    n_elt = len(bp_h) - 1
    max_span = 1
    if n_elt > 0 and len(bs_h):
        lo = np.floor_divide(bs_h, window)
        hi = -np.floor_divide(-be_h, window)
        owner = np.repeat(np.arange(n_elt), np.diff(bp_h))
        wmin = np.full(n_elt, np.iinfo(np.int64).max)
        wmax = np.full(n_elt, np.iinfo(np.int64).min)
        np.minimum.at(wmin, owner, lo)
        np.maximum.at(wmax, owner, hi)
        has = wmax > wmin
        if has.any():
            max_span = int((wmax[has] - wmin[has]).max())
    return max_span


def build_window_map(win_chrom_idx, win_start, window, n_chrom):
    """Dense (chromosome, window number) -> row map for K6.  Returns (win_map_off int64 [n_chrom+1],
    win_map int32)."""
    wc = np.asarray(win_chrom_idx, dtype=np.int64)
    wn = np.asarray(win_start, dtype=np.int64) // int(window)
    per = np.zeros(n_chrom, dtype=np.int64)
    if len(wc):
        np.maximum.at(per, wc, wn + 1)
    off = np.zeros(n_chrom + 1, dtype=np.int64)
    off[1:] = np.cumsum(per)
    wmap = np.full(int(off[-1]), -1, dtype=np.int32)
    wmap[off[wc] + wn] = np.arange(len(wc), dtype=np.int32)
    return off, wmap


def substitution_counts(ctx, alt, n_up=1, n_down=1, stream=None, out=None):
    """Histogram of substitutions in sorted 'CTX>CTX2' order: int64 [3K] on the device of ``ctx`` (overwrites `out`)."""
    dev = ctx.device
    al = _dev(alt, torch.uint8, dev)
    if out is None:
        out = torch.empty(3 * 4 ** (n_up + n_down + 1), dtype=torch.int64, device=dev)
    assert out.dtype == torch.int64 and out.is_contiguous() and out.numel() == 3 * 4 ** (n_up + n_down + 1)
    with torch.cuda.device(dev):
        _lib.call("dig_substitution_counts", ctx.data_ptr(), al.data_ptr(), ctx.numel(), int(n_up), int(n_down),
                  out.data_ptr(), _stream(dev, stream))
    return out


def sequence_freq(subst_counts, ctx_totals, stream=None):
    """FREQ of every substitution = COUNT / S_genome[context] (float64 [3K], sorted substitution order)."""
    dev = subst_counts.device
    n_ctx = ctx_totals.numel()
    out = torch.empty(3 * n_ctx, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_sequence_freq", subst_counts.data_ptr(), ctx_totals.data_ptr(), n_ctx, out.data_ptr(),
                  _stream(dev, stream))
    return out


GENE_OUT_ROWS = (["EXP_" + c for c in ("SYN", "MIS", "NONS", "SPL", "TRUNC", "NONSYN")] +
                 ["PVAL_%s_BURDEN" % c for c in ("SYN", "MIS", "NONS", "SPL", "TRUNC", "NONSYN")] +
                 ["PVAL_%s_BURDEN_SAMPLE" % c for c in ("SYN", "MIS", "NONS", "SPL", "TRUNC", "NONSYN")] +
                 ["EXP_INDEL", "PVAL_INDEL_BURDEN", "PVAL_MUT_BURDEN", "ALPHA", "THETA", "THETA_INDEL", "Pi_INDEL",
                  "Pi_TRUNC", "Pi_NONSYN"])


def size_ratio(num, den, stream=None):
    """float64 num / den of two int64 device tensors in one launch (Pi_INDEL = ELT_SIZE / R_SIZE,
    genic_driver_tools.py:158-159)."""
    dev = num.device
    assert num.dtype == torch.int64 and den.dtype == torch.int64 and num.is_contiguous() and den.is_contiguous()
    assert num.numel() == den.numel()
    out = torch.empty(num.shape, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_size_ratio", num.data_ptr(), den.data_ptr(), num.numel(), out.data_ptr(), _stream(dev, stream))
    return out


def gene_scale_sums(mu, sigma, P, pi_indel, obs, cgc_mask=None, tp53=-1, stream=None):
    """[sum_{g != TP53} MU*Pi_SYN, sum_{non-CGC} Pi_INDEL*ALPHA*THETA, sum_{non-CGC} OBS_INDEL] on the device."""
    dev = mu.device
    sums = torch.empty(3, dtype=torch.float64, device=dev)
    cg = _dev(cgc_mask, torch.uint8, dev) if cgc_mask is not None else None
    with torch.cuda.device(dev):
        _lib.call("dig_gene_scale_sums", mu.data_ptr(), sigma.data_ptr(), P.data_ptr(), pi_indel.data_ptr(),
                  obs.data_ptr(), _ptr(cg), int(tp53), mu.numel(), sums.data_ptr(), _stream(dev, stream))
    return sums


def gene_burden_test(mu, sigma, P, pi_indel, obs, nsamp, sums, n_syn, scale_factor=None, stream=None):
    """All 13 NB tests + Fisher per gene in one launch pair.  Returns float64 [27, E] (rows: GENE_OUT_ROWS).
    n_syn=None: the synonymous count is sums[3] on the device (multi-GPU path, no host read), so without a
    scale_factor sums must hold four values; gene_scale_sums returns three, and the caller appends the count."""
    need = 4 if n_syn is None and scale_factor is None else 3
    if sums.numel() < need:
        raise ValueError("gene_burden_test: sums has %d values, the kernel reads %d (n_syn=None takes the synonymous "
                         "count from sums[3])" % (sums.numel(), need))
    dev = mu.device
    E = mu.numel()
    out = torch.empty((len(GENE_OUT_ROWS), E), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_gene_burden_test", mu.data_ptr(), sigma.data_ptr(), P.data_ptr(), pi_indel.data_ptr(),
                  obs.data_ptr(), nsamp.data_ptr(), E, sums.data_ptr(), float("nan") if n_syn is None else float(n_syn),
                  float("nan") if scale_factor is None else float(scale_factor), out.data_ptr(), _stream(dev, stream))
    return out


def site_counts(site_elt, site_sub, n_elt, n_sub=192, device="cuda:0", stream=None):
    """L[elt, sub] = number of sites per (site-set, substitution): int64 [n_elt, n_sub] on the device."""
    dev = torch.device(device)
    se, ss = _dev(site_elt, torch.int32, dev), _dev(site_sub, torch.int32, dev)
    out = torch.empty((max(n_elt, 1), n_sub), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_site_counts", se.data_ptr(), ss.data_ptr(), se.numel(), n_elt, n_sub, out.data_ptr(),
                  _stream(dev, stream))
    return out[:n_elt]


def nb_pvalue_exact(k, alpha, p, device="cuda:0", stream=None):
    """K8 scalar form: nb_model.nb_pvalue_exact(k, alpha, p) (nb_model.py:298-314) element-wise in FP64 on the GPU."""
    dev = torch.device(device)
    kk, aa, pp = (_dev(x, torch.float64, dev).contiguous() for x in (k, alpha, p))
    out = torch.empty_like(kk)
    with torch.cuda.device(dev):
        _lib.call("dig_nb_pvalue_exact", kk.data_ptr(), aa.data_ptr(), pp.data_ptr(), kk.numel(), out.data_ptr(),
                  _stream(dev, stream))
    return out


def position_bins(genome, reg_chrom, reg_start, reg_end, n_up, n_down, binsize):
    """Host-side bin layout of K8: positions per region (the centres the scan walks, quirks a1-i/ii included)
    and the CSR bin_ptr [n_reg + 1]."""
    rc = np.asarray(reg_chrom, dtype=np.int64)
    rs = np.asarray(reg_start, dtype=np.int64).copy()
    re = np.asarray(reg_end, dtype=np.int64)
    L = np.asarray(genome.chrom_len, dtype=np.int64)[rc]
    rs[rs < n_up] = n_up                                     # START == 0 -> n_up (sequence_tools.py:25-26)
    first = np.minimum(rs, L)
    last = np.minimum(re + n_down, L) - n_down               # faidx clips at the chromosome end
    n_pos = np.maximum(last - first, 0)
    n_bin = -(-n_pos // binsize)
    ptr = np.zeros(len(rc) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(n_bin)
    return first, n_pos, ptr


def position_test(genome, reg_chrom, reg_start, reg_end, mu, sigma, s_prob, mut_chrom, mut_start, n_up=2, n_down=2,
                  binsize=1, normed=True, want=("pt", "exp", "pos"), stream=None):
    """K8: apply_nb_to_region / nb_model (nb_model.py:126-235) for a list of regions.  s_prob is the [K] table of
    per-context probabilities in k-mer index order; (mut_chrom, mut_start) are the mutation rows (chromosome index
    into the genome, 0-based START).  Returns a dict of device tensors over all bins (regions concatenated):
    pval, obs and, if wanted, pt / exp / pos, plus the host arrays bin_ptr and n_pos."""
    dev = genome.device
    rc = _dev(reg_chrom, torch.int32, dev)
    rs = _dev(reg_start, torch.int64, dev)
    re = _dev(reg_end, torch.int64, dev)
    n_reg = rc.numel()
    K = 4 ** (n_up + n_down + 1)
    sp = _dev(s_prob, torch.float64, dev).contiguous()
    assert sp.numel() == K, "s_prob must have 4^(n_up+n_down+1) entries"
    mu_d, sg_d = _dev(mu, torch.float64, dev).contiguous(), _dev(sigma, torch.float64, dev).contiguous()
    assert mu_d.numel() == n_reg and sg_d.numel() == n_reg
    host = lambda x: x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    first, n_pos, ptr = position_bins(genome, host(reg_chrom), host(reg_start), host(reg_end), n_up, n_down, binsize)
    n_bin = int(ptr[-1])
    ptr_d = torch.from_numpy(ptr).to(dev)
    mk = (host(mut_chrom).astype(np.int64) << 32) | host(mut_start).astype(np.int64)
    mk_d = torch.from_numpy(np.sort(mk)).to(dev)
    sptr = _stream(dev, stream)
    out = {"bin_ptr": ptr, "n_pos": n_pos, "first": first}
    with torch.cuda.device(dev):
        norm = None
        if normed:
            counts, _ = count_contexts(genome, rc, rs, re, n_up, n_down, stream=stream)
            norm = torch.empty(n_reg, dtype=torch.float64, device=dev)
            _lib.call("dig_region_prob_norm", counts.data_ptr(), sp.data_ptr(), n_reg, K, norm.data_ptr(), sptr)
            out["norm"] = norm
        obs = torch.empty(max(n_bin, 1), dtype=torch.int32, device=dev)
        _lib.call("dig_position_obs", mk_d.data_ptr(), mk_d.numel(), genome.chrom_off_d.data_ptr(),
                  genome.chrom_len_d.data_ptr(), rc.data_ptr(), rs.data_ptr(), re.data_ptr(), n_reg, int(n_up),
                  int(n_down), int(binsize), ptr_d.data_ptr(), n_bin, obs.data_ptr(), sptr)
        pval = torch.empty(max(n_bin, 1), dtype=torch.float64, device=dev)
        extra = {k: (torch.empty(max(n_bin, 1), dtype=torch.float64, device=dev) if k in want else None)
                 for k in ("pt", "exp", "pos")}
        _lib.call("dig_position_test", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), rc.data_ptr(), rs.data_ptr(),
                  re.data_ptr(), n_reg, int(n_up), int(n_down), sp.data_ptr(), _ptr(norm), mu_d.data_ptr(),
                  sg_d.data_ptr(), int(binsize), ptr_d.data_ptr(), obs.data_ptr(), pval.data_ptr(),
                  _ptr(extra["pt"]), _ptr(extra["exp"]), _ptr(extra["pos"]), sptr)
    out["pval"], out["obs"] = pval[:n_bin], obs[:n_bin]
    for k, v in extra.items():
        if v is not None:
            out[k] = v[:n_bin]
    return out


DNDS_CLASSES = ("SYN", "MIS", "NONS", "SPL", "TRUNC", "NONSYN")
DNDS_OUT_ROWS = (["EXP_%s" % c for c in DNDS_CLASSES] + ["T_SYN", "MRFOLD"] + ["EXP_%s_ML" % c for c in DNDS_CLASSES] +
                 ["PVAL_%s_BURDEN_DNDS" % c for c in DNDS_CLASSES] +
                 ["PVAL_SYN_SEL_NB", "PVAL_MIS_SEL_NB", "PVAL_TRUNC_SEL_NB", "PVAL_NONSYN_SEL_NB"])


def gene_dnds_sel(alpha, theta, pi6, obs6, device="cuda:0", stream=None):
    """Secondary gene tests in one launch: float64 [24, E] with rows DNDS_OUT_ROWS (include/dig_b200.h)."""
    dev = torch.device(device)
    a, t = _dev(alpha, torch.float64, dev).contiguous(), _dev(theta, torch.float64, dev).contiguous()
    p6, o6 = _dev(pi6, torch.float64, dev).contiguous(), _dev(obs6, torch.float64, dev).contiguous()
    E = a.numel()
    assert p6.shape == (E, 6) and o6.shape == (E, 6)
    out = torch.empty((len(DNDS_OUT_ROWS), E), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_gene_dnds_sel", a.data_ptr(), t.data_ptr(), p6.data_ptr(), o6.data_ptr(), E, out.data_ptr(),
                  _stream(dev, stream))
    return out


def selection_coefficient(obs, exp, alpha=None, theta=None, pi=None, device="cuda:0", stream=None):
    """SEL = (OBS + 1e-16) / (EXP + 1e-16) and (when alpha/theta/pi are given) its LLR p-value."""
    dev = torch.device(device)
    o, e = _dev(obs, torch.float64, dev).contiguous(), _dev(exp, torch.float64, dev).contiguous()
    want_p = alpha is not None
    a, t, p = ((_dev(x, torch.float64, dev).contiguous() for x in (alpha, theta, pi)) if want_p else (None, None, None))
    sel = torch.empty_like(o)
    pval = torch.empty_like(o) if want_p else None
    with torch.cuda.device(dev):
        _lib.call("dig_selection_coefficient", o.data_ptr(), e.data_ptr(), _ptr(a), _ptr(t), _ptr(p), o.numel(),
                  sel.data_ptr(), _ptr(pval), _stream(dev, stream))
    return sel, pval


def site_test(site_chrom, site_start, site_sub, site_k, window, win_map_off, win_map, win_counts, y_pred, std, d_pr,
              cj=1.0, site_strand=None, device="cuda:0", want=("P", "EXP"), stream=None, status_sink=None):
    """Per-site burden test (config 3): P, EXP and PVAL for every site as a one-site site set.  site_chrom indexes
    win_map_off like dig_element_transfer's elt_chrom; site_sub is the substitution index 0..191 (already flipped for
    minus-strand sites); win_counts int32 [n_win, 64]; y_pred / std [n_win].  Returns a dict of device tensors."""
    dev = torch.device(device)
    sc, ss = _dev(site_chrom, torch.int32, dev), _dev(site_start, torch.int64, dev)
    sb, sk = _dev(site_sub, torch.uint8, dev), _dev(site_k, torch.float64, dev)
    st = _dev(site_strand, torch.int8, dev) if site_strand is not None else None
    wmo, wm = _dev(win_map_off, torch.int64, dev), _dev(win_map, torch.int32, dev)
    wc = _dev(win_counts, torch.int32, dev).contiguous()
    yp, sd = _dev(y_pred, torch.float64, dev).contiguous(), _dev(std, torch.float64, dev).contiguous()
    dp = _dev(d_pr, torch.float64, dev).contiguous()
    n_win, n = wc.shape[0], sc.numel()
    den_p = torch.empty(n_win, dtype=torch.float64, device=dev)
    den_m = torch.empty(n_win, dtype=torch.float64, device=dev)
    out = {"PVAL": torch.empty(n, dtype=torch.float64, device=dev)}
    for k in ("P", "EXP"):
        out[k] = torch.empty(n, dtype=torch.float64, device=dev) if k in want else None
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    sptr = _stream(dev, stream)
    with torch.cuda.device(dev):
        _lib.call("dig_window_denominators", wc.data_ptr(), dp.data_ptr(), n_win, den_p.data_ptr(), den_m.data_ptr(), sptr)
        _lib.call("dig_site_test", sc.data_ptr(), ss.data_ptr(), sb.data_ptr(), _ptr(st), sk.data_ptr(), n, int(window),
                  int(wmo.numel()) - 1, wmo.data_ptr(), wm.data_ptr(), yp.data_ptr(), sd.data_ptr(), den_p.data_ptr(), den_m.data_ptr(),
                  dp.data_ptr(), float(cj), _ptr(out["P"]), _ptr(out["EXP"]), out["PVAL"].data_ptr(),
                  status.data_ptr(), sptr)
        _check_status(status, "dig_site_test", status_sink)
    out["DENOM_PLUS"], out["DENOM_MINUS"] = den_p, den_m
    return {k: v for k, v in out.items() if v is not None}


NB_MODES = {"greater": 0, "greater_midp": 1, "less": 2, "less_midp": 3, "exact": 4, "midp": 5}


def nb_pvalue_variant(mode, k, alpha, p, mu=None, device="cuda:0", stream=None):
    """The other tail conventions of nb_model.py (:243-337) element-wise in FP64 on the GPU; mode is a key of
    NB_MODES.  mu (optional array) is the expectation override of nb_pvalue_exact / nb_pvalue_midp."""
    dev = torch.device(device)
    kk, aa, pp = (_dev(x, torch.float64, dev).contiguous() for x in (k, alpha, p))
    mm = _dev(mu, torch.float64, dev).contiguous() if mu is not None else None
    out = torch.empty_like(kk)
    with torch.cuda.device(dev):
        _lib.call("dig_nb_pvalue_variant", NB_MODES[mode], kk.data_ptr(), aa.data_ptr(), pp.data_ptr(), _ptr(mm),
                  kk.numel(), out.data_ptr(), _stream(dev, stream))
    return out


LL_KINDS = {"nb": 0, "pois": 1, "gamma": 2}


def loglik(kind, x, a, b=None, device="cuda:0", stream=None):
    """_ll_nb(k, alpha, theta) / _ll_pois(k, lam) / _ll_gamma(lam, alpha, theta) (transfer_tools.py:1254-1262)."""
    dev = torch.device(device)
    xx, aa = _dev(x, torch.float64, dev).contiguous(), _dev(a, torch.float64, dev).contiguous()
    bb = _dev(b, torch.float64, dev).contiguous() if b is not None else None
    out = torch.empty_like(xx)
    with torch.cuda.device(dev):
        _lib.call("dig_loglik", LL_KINDS[kind], xx.data_ptr(), aa.data_ptr(), _ptr(bb), xx.numel(), out.data_ptr(),
                  _stream(dev, stream))
    return out


def gene_llr_test(model, alpha, theta, pi3, obs3, mrfold, t_syn=None, device="cuda:0", stream=None):
    """_llr_test_nb (model "nb"; SYN, MIS, TRUNC) / _llr_test_gamma_poiss (model "gamma_poisson"; SYN, MIS, NONS) for
    every row: float64 [4, n] = p_syn, p_mis, p_third, p_nonsyn."""
    dev = torch.device(device)
    a, t, m = (_dev(x, torch.float64, dev).contiguous() for x in (alpha, theta, mrfold))
    p3, o3 = _dev(pi3, torch.float64, dev).contiguous(), _dev(obs3, torch.float64, dev).contiguous()
    ts = _dev(t_syn, torch.float64, dev).contiguous() if t_syn is not None else None
    n = a.numel()
    assert p3.shape == (n, 3) and o3.shape == (n, 3)
    out = torch.empty((4, n), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_gene_llr_test", {"nb": 0, "gamma_poisson": 1}[model], a.data_ptr(), t.data_ptr(), p3.data_ptr(),
                  o3.data_ptr(), m.data_ptr(), _ptr(ts), n, out.data_ptr(), _stream(dev, stream))
    return out


def overlap_pairs(blk_kstart, blk_kend, mut_kstart, mut_kend, device="cuda:0", stream=None):
    """Overlap join (`bedtools intersect -wa -wb`): int64 arrays (pair_mut, pair_blk) on the host, one entry per
    overlapping (mutation, block) pair, grouped by mutation in input order; block indices refer to the caller's
    (unsorted) block order."""
    dev = torch.device(device)
    bks = np.asarray(blk_kstart, dtype=np.int64)
    order = np.argsort(bks, kind="stable")
    bks = bks[order]
    bke = np.asarray(blk_kend, dtype=np.int64)[order]
    pmax = np.maximum.accumulate(bke) if len(bke) else bke
    b0, b1, b2 = (_dev(x, torch.int64, dev) for x in (bks, bke, pmax))
    m0, m1 = _dev(mut_kstart, torch.int64, dev), _dev(mut_kend, torch.int64, dev)
    n_blk, n_mut = len(bks), m0.numel()
    sptr = _stream(dev, stream)
    off = torch.zeros(n_mut + 1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        cnt = torch.zeros(max(n_mut, 1), dtype=torch.int64, device=dev)
        _lib.call("dig_overlap_count", _ptr(b0), _ptr(b1), _ptr(b2), n_blk, m0.data_ptr(), m1.data_ptr(), n_mut,
                  cnt.data_ptr(), sptr)
        off[1:] = torch.cumsum(cnt[:n_mut], 0)
        total = int(off[-1].item()) if n_mut else 0
        pm = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        pb = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        if total:
            _lib.call("dig_overlap_fill", b0.data_ptr(), b1.data_ptr(), b2.data_ptr(), n_blk, m0.data_ptr(),
                      m1.data_ptr(), n_mut, off.data_ptr(), pm.data_ptr(), pb.data_ptr(), sptr)
    return pm[:total].cpu().numpy(), order[pb[:total].cpu().numpy()]


def overlap_counts(blk_kstart, blk_kend, mut_kstart, mut_kend, device="cuda:0", stream=None):
    """Number of blocks each mutation overlaps (dig_overlap_count): int64 host array [n_mut]."""
    dev = torch.device(device)
    bks = np.asarray(blk_kstart, dtype=np.int64)
    order = np.argsort(bks, kind="stable")
    bks = bks[order]
    bke = np.asarray(blk_kend, dtype=np.int64)[order]
    pmax = np.maximum.accumulate(bke) if len(bke) else bke
    b0, b1, b2 = (_dev(x, torch.int64, dev) for x in (bks, bke, pmax))
    m0, m1 = _dev(mut_kstart, torch.int64, dev), _dev(mut_kend, torch.int64, dev)
    n_mut = m0.numel()
    cnt = torch.zeros(max(n_mut, 1), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_overlap_count", _ptr(b0), _ptr(b1), _ptr(b2), len(bks), m0.data_ptr(), m1.data_ptr(), n_mut,
                  cnt.data_ptr(), _stream(dev, stream))
    return cnt[:n_mut].cpu().numpy()


def element_region_counts(elt_chrom, elt_strand, blk_ptr, blk_start, blk_end, window, win_map_off, win_map, win_counts,
                          device="cuda:0", stream=None, status_sink=None):
    """The `region_counts` intermediate of preprocess_nonc / preprocess_sites: int64 [n_elt, 64] sums of the window
    trinucleotide counts over each element's overlapped windows (reverse-complemented for minus-strand elements) and
    the number of windows per element."""
    dev = torch.device(device)
    ec, es = _dev(elt_chrom, torch.int32, dev), _dev(elt_strand, torch.int8, dev)
    bp, bs, be = (_dev(x, torch.int64, dev) for x in (blk_ptr, blk_start, blk_end))
    wmo, wm = _dev(win_map_off, torch.int64, dev), _dev(win_map, torch.int32, dev)
    wc = _dev(win_counts, torch.int32, dev).contiguous()
    n_elt = ec.numel()
    rc = torch.empty((max(n_elt, 1), 64), dtype=torch.int64, device=dev)
    nw = torch.empty(max(n_elt, 1), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_element_region_counts", ec.data_ptr(), es.data_ptr(), bp.data_ptr(), bs.data_ptr(), be.data_ptr(),
                  n_elt, int(window), int(wmo.numel()) - 1, wmo.data_ptr(), wm.data_ptr(), wc.data_ptr(), wc.shape[0],
                  element_max_span(bp, bs, be, window), rc.data_ptr(), nw.data_ptr(), status.data_ptr(),
                  _stream(dev, stream))
        _check_status(status, "dig_element_region_counts", status_sink)
    return rc[:n_elt], nw[:n_elt]


def element_psum(L, region_counts, d_pr, device="cuda:0", stream=None, want_denom=False):
    """P_SUM from persisted L_counts / region_counts [n_elt, 192] (dig_element_psum)."""
    dev = torch.device(device)
    Ld = _dev(L, torch.float64, dev).contiguous().reshape(-1, 192)
    Rd = _dev(region_counts, torch.int64, dev).contiguous().reshape(-1, 192)
    dp = _dev(d_pr, torch.float64, dev).contiguous()
    n = Ld.shape[0]
    assert Rd.shape[0] == n and dp.numel() == 192
    p = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
    den = torch.empty(max(n, 1), dtype=torch.float64, device=dev) if want_denom else None
    with torch.cuda.device(dev):
        _lib.call("dig_element_psum", Ld.data_ptr(), Rd.data_ptr(), dp.data_ptr(), n, p.data_ptr(), _ptr(den),
                  _stream(dev, stream))
    return (p[:n], den[:n]) if want_denom else p[:n]


# ---------------------------------------------------------------------------------------------
# K9: gene annotation from a CDS gene set (csrc/cdsannot.cu)
# ---------------------------------------------------------------------------------------------

CDS_CLASS_NAMES = {0: "Synonymous", 1: "Missense", 2: "Nonsense", 3: "Essential_Splice", 5: "Stop_loss"}
CDS_NO_HIT = 255


def _splice_offsets(donor, acceptor):
    """ctypes int32 arrays (host) of the donor / acceptor intron offsets."""
    import ctypes
    d, a = [int(x) for x in donor], [int(x) for x in acceptor]
    return (ctypes.c_int32 * max(len(d), 1))(*d), len(d), (ctypes.c_int32 * max(len(a), 1))(*a), len(a)


def _check_cds_status(status, what):
    code = int(status.item())
    if code:
        why = [m for bit, m in ((1, "a gene has more than 2048 CDS blocks"),
                                (2, "a gene's chromosome or block lies outside the genome"),
                                (4, "a gene's blocks are not strictly ascending"),
                                (8, "the codon numbering does not fit the CDS lengths")) if code & bit]
        raise _lib.DigError("%s: %s" % (what, "; ".join(why)))


def cds_substitution_table(genome, gene_chrom, gene_strand, blk_ptr, blk_start, blk_end, donor=(1, 2, 5),
                           acceptor=(1, 2), stream=None):
    """K9a: per-gene substitution table of the CDS.  Blocks are inclusive [start, end] chromosome coordinates,
    ascending within each gene; gene_chrom indexes the genome.  Returns (L float64 [E, 192, 4] = silent, missense,
    nonsense, essential splice; flags int32 [E]) on the device."""
    dev = genome.device
    gc, gs = _dev(gene_chrom, torch.int32, dev), _dev(gene_strand, torch.int8, dev)
    bp, bs, be = (_dev(x, torch.int64, dev) for x in (blk_ptr, blk_start, blk_end))
    E = gc.numel()
    L = torch.empty((max(E, 1), 192, 4), dtype=torch.float64, device=dev)
    flags = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    d, nd, a, na = _splice_offsets(donor, acceptor)
    with torch.cuda.device(dev):
        _lib.call("dig_cds_substitution_table", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), len(genome.chrom_len), gc.data_ptr(),
                  gs.data_ptr(), bp.data_ptr(), bs.data_ptr(), be.data_ptr(), E, d, nd, a, na, L.data_ptr(),
                  flags.data_ptr(), status.data_ptr(), _stream(dev, stream))
        _check_cds_status(status, "dig_cds_substitution_table")
    return L[:E], flags[:E]


def annotate_snvs(genome, gene_chrom, gene_strand, blk_ptr, blk_start, blk_end, mut_chrom, mut_pos, mut_alt,
                  donor=(1, 2, 5), acceptor=(1, 2), stream=None):
    """K9b: coding class of SNVs in every gene that holds them.  mut_chrom indexes the genome, mut_pos is the 0-based
    position, mut_alt 0..3 (A/C/G/T).  The SNVs are joined (dig_overlap_count / dig_overlap_fill) against the CDS blocks
    widened by the largest splice offset, the (mutation, gene) pairs de-duplicated, then classified.  Returns device
    tensors (pair_mut int64, pair_gene int32, cls uint8), sorted by mutation, then gene; cls is a DIG_CDS_* code
    (CDS_CLASS_NAMES, CDS_NO_HIT for a pair that is neither a countable coding site nor a splice position)."""
    dev = genome.device
    gc, gs = _dev(gene_chrom, torch.int32, dev), _dev(gene_strand, torch.int8, dev)
    bp, bs, be = (_dev(x, torch.int64, dev) for x in (blk_ptr, blk_start, blk_end))
    mp, ma = _dev(mut_pos, torch.int64, dev), _dev(mut_alt, torch.uint8, dev)
    E = gc.numel()
    pad = max([int(x) for x in donor] + [int(x) for x in acceptor] + [0])
    pair_mut, pair_gene = _snv_gene_pairs(dev, gc, bp, bs, be, mut_chrom, mp, pad, stream)
    if pair_mut.numel() == 0:
        return pair_mut, pair_gene, torch.zeros(0, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        cls = torch.empty(pair_mut.numel(), dtype=torch.uint8, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        d, nd, a, na = _splice_offsets(donor, acceptor)
        _lib.call("dig_annotate_snvs", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), len(genome.chrom_len), gc.data_ptr(),
                  gs.data_ptr(), bp.data_ptr(), bs.data_ptr(), be.data_ptr(), E, d, nd, a, na, mp.data_ptr(),
                  ma.data_ptr(), pair_mut.data_ptr(), pair_gene.data_ptr(), pair_mut.numel(), cls.data_ptr(),
                  status.data_ptr(), _stream(dev, stream))
        _check_cds_status(status, "dig_annotate_snvs")
    return pair_mut, pair_gene, cls


def _snv_gene_pairs(dev, gc, bp, bs, be, mut_chrom, mp, pad, stream):
    """(mutation, gene) pairs of SNVs against the CDS blocks widened by `pad` bases (dig_overlap_count /
    dig_overlap_fill), one per pair, sorted by mutation, then gene.  Device tensors (pair_mut int64, pair_gene int32)."""
    mc = _dev(mut_chrom, torch.int64, dev)
    E, n_mut = gc.numel(), mp.numel()
    owner = torch.repeat_interleave(torch.arange(E, dtype=torch.int64, device=dev), bp[1:] - bp[:-1])
    kc = gc.to(torch.int64)[owner] << 32
    ks, order = torch.sort(kc | torch.clamp(bs - pad, min=0), stable=True)
    ke = (kc | (be + 1 + pad))[order]
    pmax = torch.cummax(ke, 0).values if ke.numel() else ke
    owner = owner[order]
    mks = (mc << 32) | mp
    mke = mks + 1
    sptr = _stream(dev, stream)
    empty = (torch.zeros(0, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    if n_mut == 0 or ks.numel() == 0:
        return empty
    with torch.cuda.device(dev):
        cnt = torch.empty(n_mut, dtype=torch.int64, device=dev)
        _lib.call("dig_overlap_count", ks.data_ptr(), ke.data_ptr(), pmax.data_ptr(), ks.numel(), mks.data_ptr(),
                  mke.data_ptr(), n_mut, cnt.data_ptr(), sptr)
        off = torch.zeros(n_mut + 1, dtype=torch.int64, device=dev)
        off[1:] = torch.cumsum(cnt, 0)
        total = int(off[-1].item())
        if total == 0:
            return empty
        pm = torch.empty(total, dtype=torch.int64, device=dev)
        pb = torch.empty(total, dtype=torch.int64, device=dev)
        _lib.call("dig_overlap_fill", ks.data_ptr(), ke.data_ptr(), pmax.data_ptr(), ks.numel(), mks.data_ptr(),
                  mke.data_ptr(), n_mut, off.data_ptr(), pm.data_ptr(), pb.data_ptr(), sptr)
        # blocks of one gene may all reach the same SNV: one pair per (mutation, gene), in (mutation, gene) order
        key = torch.unique(pm * E + owner[pb])
        pair_mut = torch.div(key, E, rounding_mode="floor")
        pair_gene = (key - pair_mut * E).to(torch.int32)
    return pair_mut, pair_gene


# ---------------------------------------------------------------------------------------------
# K9c / K10 / K9d: codon-level driver test (csrc/codon.cu)
# ---------------------------------------------------------------------------------------------

CODON_NO_SITE = 255


def codon_ptr(blk_ptr, blk_start, blk_end, device):
    """int64 [E + 1] device tensor numbering floor(CDS length / 3) codons per gene (the codon_ptr of dig_codon_*)."""
    bp, bs, be = (_dev(x, torch.int64, device) for x in (blk_ptr, blk_start, blk_end))
    E = bp.numel() - 1
    owner = torch.repeat_interleave(torch.arange(E, dtype=torch.int64, device=device), bp[1:] - bp[:-1])
    T = torch.zeros(E, dtype=torch.int64, device=device).index_add_(0, owner, be - bs + 1)
    ptr = torch.zeros(E + 1, dtype=torch.int64, device=device)
    ptr[1:] = torch.cumsum(torch.div(T, 3, rounding_mode="floor"), 0)
    return ptr


def codon_sites(genome, gene_chrom, gene_strand, blk_ptr, blk_start, blk_end, stream=None):
    """K9c: the 9-slot site record of every complete codon of every gene (dig_codon_sites).  Returns a dict of device
    tensors: PTR int64 [E+1], POS int64 [n, 3], BIN uint8 [n, 9], CLASS uint8 [n, 9], REF_AA uint8 [n] (ASCII),
    N_SITES uint8 [n]."""
    dev = genome.device
    gc, gs = _dev(gene_chrom, torch.int32, dev), _dev(gene_strand, torch.int8, dev)
    bp, bs, be = (_dev(x, torch.int64, dev) for x in (blk_ptr, blk_start, blk_end))
    E = gc.numel()
    ptr = codon_ptr(bp, bs, be, dev)
    n = int(ptr[-1].item())
    out = {"PTR": ptr, "POS": torch.empty((n, 3), dtype=torch.int64, device=dev),
           "BIN": torch.empty((n, 9), dtype=torch.uint8, device=dev),
           "CLASS": torch.empty((n, 9), dtype=torch.uint8, device=dev),
           "REF_AA": torch.empty(n, dtype=torch.uint8, device=dev), "N_SITES": torch.empty(n, dtype=torch.uint8, device=dev)}
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.call("dig_codon_sites", genome.packed2.data_ptr(), genome.nmask.data_ptr(), genome.n_bases,
                  genome.chrom_off_d.data_ptr(), genome.chrom_len_d.data_ptr(), len(genome.chrom_len), gc.data_ptr(),
                  gs.data_ptr(), bp.data_ptr(), bs.data_ptr(), be.data_ptr(), E, ptr.data_ptr(), n,
                  out["POS"].data_ptr(), out["BIN"].data_ptr(), out["CLASS"].data_ptr(), out["REF_AA"].data_ptr(),
                  out["N_SITES"].data_ptr(), status.data_ptr(), _stream(dev, stream))
        _check_cds_status(status, "dig_codon_sites")
    return out


def codon_transfer(sites, gene_chrom_num, gene_strand, window, win_map_off, win_map, win_counts, y_pred, std, y_true,
                   flag, d_pr, device, stream=None):
    """K10 (after dig_window_denominators): MU, SIGMA, R_OBS, FLAG, R_SIZE, PI_NUM, PI_SUM, N_WIN per codon of
    `sites` (codon_sites output) over the windows of its site-carrying bases.  gene_chrom_num holds chromosome NUMBERS
    (they index win_map_off).  The device status word is returned as STATUS: 2 = a site-carrying base lies in a window
    missing from the window map (the reference's KeyError); those codons have NaN MU, so the caller can name them."""
    dev = torch.device(device)
    gc, gs = _dev(gene_chrom_num, torch.int32, dev), _dev(gene_strand, torch.int8, dev)
    wmo, wm = _dev(win_map_off, torch.int64, dev), _dev(win_map, torch.int32, dev)
    wc = _dev(win_counts, torch.int32, dev).contiguous()
    yp, sd, yt = (_dev(x, torch.float64, dev).contiguous() for x in (y_pred, std, y_true))
    fl = _dev(np.asarray(flag).astype(np.uint8) if not isinstance(flag, torch.Tensor) else flag.to(torch.uint8),
              torch.uint8, dev)
    dp = _dev(d_pr, torch.float64, dev).contiguous()
    ptr, pos, bins, ns = sites["PTR"], sites["POS"], sites["BIN"], sites["N_SITES"]
    n, n_win = ns.numel(), wc.shape[0]
    f64 = lambda: torch.empty(n, dtype=torch.float64, device=dev)
    out = {"MU": f64(), "SIGMA": f64(), "R_OBS": f64(), "FLAG": torch.empty(n, dtype=torch.uint8, device=dev),
           "R_SIZE": torch.empty(n, dtype=torch.int64, device=dev), "PI_NUM": f64(), "PI_SUM": f64(),
           "N_WIN": torch.empty(n, dtype=torch.int32, device=dev)}
    den_p = torch.empty(max(n_win, 1), dtype=torch.float64, device=dev)
    den_m = torch.empty(max(n_win, 1), dtype=torch.float64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    sptr = _stream(dev, stream)
    with torch.cuda.device(dev):
        _lib.call("dig_window_denominators", wc.data_ptr(), dp.data_ptr(), n_win, den_p.data_ptr(), den_m.data_ptr(), sptr)
        _lib.call("dig_codon_transfer", ptr.data_ptr(), gc.data_ptr(), gs.data_ptr(), gc.numel(), pos.data_ptr(),
                  bins.data_ptr(), ns.data_ptr(), n, int(window), int(wmo.numel()) - 1, wmo.data_ptr(), wm.data_ptr(),
                  wc.data_ptr(), yp.data_ptr(), sd.data_ptr(), yt.data_ptr(), fl.data_ptr(), den_p.data_ptr(),
                  den_m.data_ptr(), dp.data_ptr(), out["MU"].data_ptr(), out["SIGMA"].data_ptr(), out["R_OBS"].data_ptr(),
                  out["FLAG"].data_ptr(), out["R_SIZE"].data_ptr(), out["PI_NUM"].data_ptr(), out["PI_SUM"].data_ptr(),
                  out["N_WIN"].data_ptr(), status.data_ptr(), sptr)
    out["STATUS"] = status
    return out


def snv_codons(genome, gene_chrom, gene_strand, blk_ptr, blk_start, blk_end, sites, mut_chrom, mut_pos, mut_ref,
               mut_alt, stream=None):
    """K9d: SNVs (mut_chrom indexes the genome, 0-based mut_pos, mut_ref / mut_alt 0..3 as written) joined against the
    CDS blocks; per (mutation, gene) pair the codon whose site it is and the slot, -1 / CODON_NO_SITE otherwise.
    Returns device tensors (pair_mut int64, pair_gene int32, codon int64, slot uint8)."""
    dev = genome.device
    gc, gs = _dev(gene_chrom, torch.int32, dev), _dev(gene_strand, torch.int8, dev)
    bp, bs, be = (_dev(x, torch.int64, dev) for x in (blk_ptr, blk_start, blk_end))
    mp = _dev(mut_pos, torch.int64, dev)
    mr, ma = _dev(mut_ref, torch.uint8, dev), _dev(mut_alt, torch.uint8, dev)
    pair_mut, pair_gene = _snv_gene_pairs(dev, gc, bp, bs, be, mut_chrom, mp, 0, stream)
    n = pair_mut.numel()
    codon = torch.empty(n, dtype=torch.int64, device=dev)
    slot = torch.empty(n, dtype=torch.uint8, device=dev)
    if n:
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.call("dig_snv_codons", gs.data_ptr(), bp.data_ptr(), bs.data_ptr(), be.data_ptr(),
                      sites["PTR"].data_ptr(), gc.numel(), sites["POS"].data_ptr(), sites["BIN"].data_ptr(),
                      mp.data_ptr(), mr.data_ptr(), ma.data_ptr(), pair_mut.data_ptr(), pair_gene.data_ptr(), n,
                      codon.data_ptr(), slot.data_ptr(), status.data_ptr(), _stream(dev, stream))
            _check_cds_status(status, "dig_snv_codons")
    return pair_mut, pair_gene, codon, slot
