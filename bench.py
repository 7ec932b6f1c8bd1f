#!/usr/bin/env python
"""bench.py -- the reference's headline workload on B200, measured as the driver contract asks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--bases G] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): synthetic hg19-sized genome (3.1 Gb, 22 chromosomes, ~3 % N,
50 % lower case), 10 kb windows (310 k), pentanucleotide AND trinucleotide context maps with genome
totals, sequence model from 1 M SNVs, 20 k-gene CDS pretrain + observed counts + NB burden test
(13 p-values + Fisher per gene).  One "step" = one pass of that whole path.

  value  : genome bases scanned per second over the whole step, inputs resident in HBM;
  e2e    : the same step through the package's host-buffer API (digdriver_b200.host_pipeline.HostScan): packed
           genome (the .dig2bit cache; `cold` = ASCII), mutations and gene tables start in pinned host memory,
           uint16 count tables and p-values end in host memory (copies inside the timing);
  roofline: the dominant kernel (pentanucleotide scan), algorithmic bytes / its CUDA-event time,
           against the measured HBM peak in MEASURED_PEAKS.json;
  cpu_baseline / --impl reference: the reference's own algorithm (pure-Python per-base loop under
           multiprocessing.Pool, SciPy p-values) timed on this box's host cores on a bounded sample.

Multi-GPU (torchrun, one rank per GPU), default --scaling strong: ONE 3.1 Gb genome; the windows are cut into N
range slices, a rank scans its slice, ONE all_gather_into_tensor carries the trinucleotide rows and the partial genome
totals, genes go to the rank that holds their first block (StrongShard).  --scaling weak keeps round 1's "one genome
per rank" run for comparison.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WINDOW = 10_000
N_GENES = 20_000
N_MUT = 1_000_000
N_SAMPLES = 200
B_PER_BASE_K1024 = 0.25 + 0.125 + 4.0 * 1024 / WINDOW      # SURVEY.md 8d: 0.7846 B/base
B_PER_BASE_FUSED = 0.25 + 0.125 + 4.0 * (1024 + 64) / WINDOW  # both tables written by one pass: 0.8102
B_PER_BASE_K64 = 0.25 + 0.125 + 4.0 * 64 / WINDOW
SCAN_DRAM_TRAFFIC = 2.4683e9      # dram read + write bytes of one fused scan launch at 3.1 Gb (ncu --set full, profiles/)


_JSON_OUT = None


def emit_json(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=30, help="timed steps of each timed leg")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bases", type=float, default=3.1e9, help="genome size per GPU (debug override)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-sample", action="store_true")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="strong scaling: trinucleotide rows stored into all ranks' symmetric buffers by the scan kernel "
                         "(fused, falls back to nccl when symmetric memory is unavailable) or one NCCL all-gather")
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"],
                    help="N > 1: strong = ONE 3.1 Gb genome range-sharded over the ranks (default), weak = one genome per rank")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="single process only: after the timed steps, write what the last one computed to DIR/<name>.npy")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
# host placement
# ------------------------------------------------------------------------------------------------

def bind_to_gpu_numa_node(local_rank):
    """Best effort: run this rank (and therefore first-touch its pinned host buffers) on the CPUs of the NUMA node its
    GPU hangs off, so that the e2e leg's host<->device copies of eight ranks do not all cross the socket interconnect.
    Returns a short description for the JSON line; never raises."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return "numa node unknown for %s" % bdf
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no allowed cpu on numa node %d" % node
        os.sched_setaffinity(0, cpus)
        return "gpu %s -> numa node %d (%d cpus)" % (bdf, node, len(cpus))
    except Exception as exc:
        return "not bound: %r" % (exc,)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []          # (host time of arrival, csv line)
        self.t_begin = None
        self.t_end = None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for (t_arr, ln) in self.lines:
            if self.t_begin is not None and not (self.t_begin <= t_arr <= (self.t_end or t_arr) + 0.06):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload construction
# ------------------------------------------------------------------------------------------------

def build_workload(total_bases, seed, device):
    """All inputs of one rank's shard: device genome (+ASCII copy for the e2e leg), windows, region
    parameters, genes with L, mutations.  Returns a dict of HOST arrays plus the device genome."""
    import torch
    from digdriver_b200 import genome as G, kernels, pipeline
    lengths = G.hg19_like_lengths(int(total_bases))
    names = ["chr%d" % (i + 1) for i in range(len(lengths))]
    dg, ascii_d = G.DeviceGenome.synthetic(names, lengths, seed=seed, device=device, return_ascii=True)
    wins = G.tile_windows(np.arange(len(lengths)), lengths, WINDOW)
    n_win = len(wins)
    y_pred, std, y_true, flag = pipeline.synth_region_params(n_win, seed + 100)
    g_chrom, g_strand, g_ptr, g_bs, g_be = pipeline.synth_genes(N_GENES, lengths, WINDOW, seed + 200)
    owner = np.repeat(np.arange(N_GENES), np.diff(g_ptr))
    # L from the CDS content itself (K4, strand-aware; half-open block ends = inclusive end + 1)
    cds_counts = lambda: kernels.count_contexts(dg, g_chrom[owner], g_bs, g_be + 1, 1, 1,
                                                strand=g_strand[owner])[0].cpu().numpy()
    bc = cds_counts()
    # A gene drawn inside one of the genome's N runs (10-51 kb) has no countable context, in its CDS or in its windows:
    # R_SIZE = 0 makes its Pi_INDEL infinite, and the reference's sum over genes then zeroes the indel scale factor of
    # every gene.  Real CDS never lie in assembly gaps, so such a gene is moved 64 kb along its chromosome (further in
    # than the longest N run) until its CDS holds a countable context.
    lim = np.maximum((lengths - 1) // WINDOW * WINDOW - 1, 0) - 1          # last CDS position synth_genes allows
    for _ in range(16):
        empty = np.flatnonzero(np.add.reduceat(bc.sum(axis=1), g_ptr[:-1]) == 0)
        if len(empty) == 0:
            break
        for g in empty:
            a, b = g_ptr[g], g_ptr[g + 1]
            shift = 1 << 16 if g_be[a:b].max() + (1 << 16) <= lim[g_chrom[g]] else -(1 << 16)
            g_bs[a:b] += shift
            g_be[a:b] += shift
        assert g_bs.min() >= 5, "a gene was moved off the start of its chromosome"
        bc = cds_counts()
    else:
        raise RuntimeError("synthetic genes without countable context remain after 16 moves")
    L = pipeline.synth_gene_L(bc, g_ptr, seed + 300)
    # mutations: 30 % coding SNVs, 63 % non-coding SNVs, 7 % indels; Zipf-weighted samples
    rng = np.random.default_rng(seed + 400)
    n_cds = int(0.30 * N_MUT)
    n_ind = int(0.07 * N_MUT)
    n_nc = N_MUT - n_cds - n_ind
    bsize = (g_be - g_bs + 1).astype(np.float64)
    bidx = rng.choice(len(g_bs), size=n_cds + n_ind // 2, p=bsize / bsize.sum())
    cds_pos = g_bs[bidx] + (rng.random(len(bidx)) * bsize[bidx]).astype(np.int64)
    cds_chrom = g_chrom[owner[bidx]]
    cds_gene = owner[bidx].astype(np.int32)
    nc_n = n_nc + (n_ind - n_ind // 2)
    nc_chrom = rng.choice(len(lengths), size=nc_n, p=lengths / lengths.sum()).astype(np.int32)
    nc_pos = (rng.random(nc_n) * (lengths[nc_chrom] - 10)).astype(np.int64) + 5
    chrom = np.concatenate([cds_chrom, nc_chrom]).astype(np.int32)
    pos = np.concatenate([cds_pos, nc_pos])
    gene = np.concatenate([cds_gene, np.full(nc_n, -1, dtype=np.int32)])
    is_indel = np.zeros(len(pos), dtype=bool)
    is_indel[n_cds:n_cds + n_ind // 2] = True
    is_indel[len(cds_pos) + n_nc:] = True
    cls = np.full(len(pos), 255, dtype=np.uint8)
    cls[:n_cds] = rng.choice(4, size=n_cds, p=[0.23, 0.68, 0.04, 0.05]).astype(np.uint8)
    cls[is_indel & (gene >= 0)] = 4
    w = 1.0 / np.arange(1, N_SAMPLES + 1)
    sample = rng.choice(N_SAMPLES, size=len(pos), p=w / w.sum()).astype(np.int32)
    order = np.lexsort((pos, chrom))
    chrom, pos, gene, is_indel, cls, sample = (a[order] for a in (chrom, pos, gene, is_indel, cls, sample))
    # REF = the genome base (device gather on the ASCII copy; setup only), ALT = another base
    gpos = torch.from_numpy(dg.chrom_off[chrom] + pos).to(device)
    up = (ascii_d[gpos] & 0xDF).cpu().numpy()
    ref = np.full(len(pos), 255, dtype=np.uint8)
    for code, ch in enumerate(b"ACGT"):
        ref[up == ch] = code
    ref[is_indel] = 255
    alt = ((ref.astype(np.int64) + 1 + rng.integers(0, 3, len(pos))) % 4).astype(np.uint8)
    alt[ref > 3] = 255
    d = dict(lengths=lengths, names=names, wins=wins, y_pred=y_pred, std=std, y_true=y_true, flag=flag,
             g_chrom=g_chrom, g_strand=g_strand, g_ptr=g_ptr, g_bs=g_bs, g_be=g_be, L=L,
             m_chrom=chrom, m_pos=pos, m_ref=ref, m_alt=alt, m_gene=gene, m_cls=cls, m_sample=sample,
             n_syn=int(((cls == 0) & (gene >= 0)).sum()))
    return dg, ascii_d, d


class DeviceInputs:
    """Device-resident copies of one shard's inputs (the `value` leg starts from these)."""

    def __init__(self, d, device):
        import torch
        from digdriver_b200 import kernels
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(device=device, dtype=dt)
        self.win_chrom = t(d["wins"][:, 0], torch.int32)
        self.win_start = t(d["wins"][:, 1], torch.int64)
        self.win_end = t(d["wins"][:, 2], torch.int64)
        self.y_pred, self.std, self.y_true = (t(d[k], torch.float64) for k in ("y_pred", "std", "y_true"))
        self.flag = t(d["flag"].astype(np.uint8), torch.uint8)
        off, wmap = kernels.build_window_map(d["wins"][:, 0], d["wins"][:, 1], WINDOW, len(d["lengths"]))
        self.wmap_off, self.wmap = t(off, torch.int64), t(wmap, torch.int32)
        self.g_chrom, self.g_strand = t(d["g_chrom"], torch.int32), t(d["g_strand"], torch.int8)
        self.g_ptr, self.g_bs, self.g_be = (t(d[k], torch.int64) for k in ("g_ptr", "g_bs", "g_be"))
        self.L = t(d["L"], torch.float64)
        self.m_chrom, self.m_pos = t(d["m_chrom"], torch.int32), t(d["m_pos"], torch.int64)
        self.m_ref, self.m_alt = t(d["m_ref"], torch.uint8), t(d["m_alt"], torch.uint8)
        self.m_gene, self.m_sample = t(d["m_gene"], torch.int32), t(d["m_sample"], torch.int32)
        self.m_cls = t(d["m_cls"], torch.uint8)
        n_win = len(d["wins"])
        self.max_span = kernels.element_max_span(d["g_ptr"], d["g_bs"], d["g_be"], WINDOW)
        self.counts5 = torch.empty((n_win, 1024), dtype=torch.int32, device=device)
        self.counts3 = torch.empty((n_win, 64), dtype=torch.int32, device=device)
        self.totals53 = torch.zeros(1024 + 64, dtype=torch.int64, device=device)
        self.totals5, self.totals3 = self.totals53[:1024], self.totals53[1024:]
        self.side_stream = torch.cuda.Stream(device)


def scan_stage(dg, di, ev=None, lo=0, hi=None, zero=True):
    """Context maps + genome totals (K2) for windows [lo, hi): pentanucleotide and trinucleotide tables in one
    fused pass (dig_count_contexts_fused53).  Range-sharded runs (StrongShard) scan only the rank's slice, straight
    into the rank's block of the buffer that is all-gathered afterwards."""
    from digdriver_b200 import kernels
    shard = getattr(di, "shard", None)
    if shard is not None:
        lo, hi = shard.lo, shard.hi
        out5, out3, tot5, tot3 = di.counts5[lo:hi], shard.rows[: hi - lo], shard.tot5, shard.tot3
    else:
        hi = di.win_chrom.numel() if hi is None else hi
        out5, out3, tot5, tot3 = di.counts5[lo:hi], di.counts3[lo:hi], di.totals5, di.totals3
    if zero:
        # both totals are adjacent views of one buffer: one fill kernel in front of the scan instead of two
        both = getattr(shard if shard is not None else di, "totals53", None)
        if both is not None:
            both.zero_()
        else:
            tot5.zero_()
            tot3.zero_()
    if shard is not None:
        shard.mutation_contexts(dg)                      # 125 k - 500 k SNVs per rank: a few microseconds, outside the scan's events
    if ev is not None:
        ev[0].record()
    if getattr(di, "scan_ws", None) is None or di.scan_ws_n < hi - lo:
        di.scan_ws, di.scan_ws_n = kernels.scan_workspace(dg, hi - lo), hi - lo
    fused = shard is not None and shard.fused
    if hi > lo:
        kernels.count_contexts_fused53(dg, di.win_chrom[lo:hi], di.win_start[lo:hi], di.win_end[lo:hi],
                                       out5=out5, out3=out3, totals5=tot5, totals3=tot3, workspace=di.scan_ws,
                                       tile_window=WINDOW, peer_rows=shard.peer_rows if fused else None,
                                       mc_rows=shard.mc_rows if fused else None)
    if ev is not None:
        ev[1].record()
    if shard is not None:
        if fused:
            shard.finish_fused_exchange()
        shard.table_ready = fused


class StrongShard:
    """ONE genome over all ranks (BASELINE north_star: "the 3.1 Gb genome is sharded by range over 8 GPUs").

    Windows are cut into `world` contiguous slices of equal base count (sharding.partition_windows); a rank scans
    only its slice.  Its trinucleotide rows and its partial genome totals are exchanged by ONE all_gather_into_tensor
    (sharding.GatheredTable: the element stage reads the gathered buffer in place through a remapped window map);
    the pentanucleotide rows stay range-sharded (their consumer is the host).  Genes belong to the rank whose slice
    holds their first block (sharding.partition_elements) and are resolved against the gathered table, so a gene
    that straddles a cut needs nothing else.  Mutation contexts (K3): every rank handles the mutations inside its own
    range, BEFORE the exchange, and the 192 partial substitution counts ride in the tail of its block next to the partial
    genome totals, so the sequence model costs no collective of its own; observed counts (K5) only for the rank's genes.
    Further exchanges: all-reduce of the five scale-factor sums, all-gather of the result rows."""

    def __init__(self, d, di, coll, device, fused_exchange=True):
        import torch
        from digdriver_b200 import kernels, sharding
        wins = d["wins"]
        self.world, self.rank = coll.world, coll.rank
        parts = sharding.partition_windows(wins[:, 1], wins[:, 2], self.world)
        self.table = sharding.GatheredTable(parts)
        self.lo, self.hi = parts[self.rank]
        gt = self.table
        # The exchange buffer lives in symmetric (peer-mapped) memory when the platform offers it: the scan kernel then
        # stores every trinucleotide row straight into all ranks' copies (NVSwitch multicast store, or one store per peer),
        # the 10 KB of partial totals and substitution counts follow with dig_peer_broadcast, and a device barrier replaces the collective.
        self.fused, self.fused_note, self.symm = False, "disabled (--exchange nccl)", None
        n_words = self.world * gt.block_rows * 64
        if fused_exchange:
            try:
                import torch.distributed as dist
                import torch.distributed._symmetric_memory as symm
                buf = symm.empty(n_words, dtype=torch.int32, device=device)
                self.symm = symm.rendezvous(buf, dist.group.WORLD)
                buf.zero_()
                self.gathered = buf.view(self.world, gt.block_rows, 64)
                blk = gt.block_rows * 64 * 4
                self.peer_rows = [int(self.symm.buffer_ptrs[p_]) + self.rank * blk for p_ in range(self.world)]
                self.peer_tail = [a + gt.m * 64 * 4 for a in self.peer_rows if a != self.peer_rows[self.rank]]
                mc = int(getattr(self.symm, "multicast_ptr", 0) or 0)
                self.mc_rows = mc + self.rank * blk if mc and os.environ.get("DIG_NO_MULTICAST", "") == "" else 0
                self.fused = True
                self.fused_note = "symmetric memory, %s" % ("multimem stores through the NVSwitch multicast alias" if self.mc_rows
                                                            else "one store per peer over NVLink")
            except Exception as exc:      # report, never hide: the NCCL all-gather is the fallback
                self.fused, self.fused_note = False, "symmetric memory unavailable: %r" % (exc,)
        if not self.fused:
            self.gathered = torch.zeros((self.world, gt.block_rows, 64), dtype=torch.int32, device=device)
        # this rank's block, in place: the scan writes its rows and totals where the other ranks expect them
        self.local = self.gathered[self.rank]
        self.table_ready = False
        self.rows, self.tot5, self.tot3, self.sub = gt.local_views(self.local)
        self.totals53 = self.local[gt.m:].view(torch.int64).reshape(-1)[:1024 + 64]      # tot5 | tot3, adjacent in the tail
        off, wmap = gt.window_map(wins[:, 0], wins[:, 1], WINDOW, len(d["lengths"]))
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(device=device, dtype=dt)
        self.wmap_off, self.wmap = t(off, torch.int64), t(wmap, torch.int32)
        row_of = gt.row_of_window(len(wins))
        self.row_of = t(row_of, torch.int64)
        n_rows = self.world * gt.block_rows

        def relay(x, dt):                  # region parameters in the row order of the gathered buffer
            out = torch.zeros(n_rows, dtype=dt, device=device)
            out[self.row_of] = x.to(dt)
            return out
        self.y_pred_g, self.std_g, self.y_true_g = (relay(x, torch.float64) for x in (di.y_pred, di.std, di.y_true))
        self.flag_g = relay(di.flag, torch.uint8)
        # genes of this rank
        g_ptr = d["g_ptr"]
        owner = sharding.partition_elements(d["g_chrom"], d["g_bs"][g_ptr[:-1]], wins[:, 0], wins[:, 1], wins[:, 2], parts)
        assert (owner >= 0).all(), "a gene starts outside every window"
        self.gene_ids = np.flatnonzero(owner == self.rank)
        self.genes_per_rank = [int((owner == r).sum()) for r in range(self.world)]
        nb = np.diff(g_ptr)[self.gene_ids]
        ptr = np.zeros(len(self.gene_ids) + 1, dtype=np.int64)
        ptr[1:] = np.cumsum(nb)
        bsel = np.concatenate([np.arange(g_ptr[g], g_ptr[g + 1]) for g in self.gene_ids]) if len(self.gene_ids) else \
            np.zeros(0, dtype=np.int64)
        self.g_chrom, self.g_strand = t(d["g_chrom"][self.gene_ids], torch.int32), t(d["g_strand"][self.gene_ids], torch.int8)
        self.g_ptr, self.g_bs, self.g_be = t(ptr, torch.int64), t(d["g_bs"][bsel], torch.int64), t(d["g_be"][bsel], torch.int64)
        self.L = t(d["L"][self.gene_ids], torch.float64)
        self.n_genes = len(self.gene_ids)
        self.max_span = kernels.element_max_span(ptr, d["g_bs"][bsel], d["g_be"][bsel], WINDOW)
        # mutations of this rank's genes, with local gene ids (K5)
        local_id = np.full(N_GENES, -1, dtype=np.int64)
        local_id[self.gene_ids] = np.arange(self.n_genes)
        mg = d["m_gene"]
        mine = (mg >= 0) & (local_id[np.clip(mg, 0, N_GENES - 1)] >= 0)
        self.m_gene = t(local_id[mg[mine]], torch.int32)
        self.m_sample, self.m_cls = t(d["m_sample"][mine], torch.int32), t(d["m_cls"][mine], torch.uint8)
        self.n_syn = int(((d["m_cls"][mine] == 0)).sum())
        self.exchange_bytes = int(self.gathered.numel() * 4)
        # mutation contexts (K3) of the mutations inside this rank's range; their 192 substitution counts travel in the
        # tail of the rank's block, next to the partial genome totals.  A mutation belongs to the rank whose slice starts
        # at or before it: the untiled tail of a chromosome goes with the chromosome's last window.
        first_key = lambda r: (int(wins[parts[r][0], 0]) << 40) | int(wins[parts[r][0], 1])
        lo_key = first_key(self.rank) if self.rank > 0 else -1
        nxt = [r for r in range(self.rank + 1, self.world) if parts[r][1] > parts[r][0]]
        hi_key = first_key(nxt[0]) if nxt else np.iinfo(np.int64).max
        mk = (d["m_chrom"].astype(np.int64) << 40) | d["m_pos"]
        self.k3_idx = np.flatnonzero((mk >= lo_key) & (mk < hi_key))
        self.k3_host = tuple(np.ascontiguousarray(d[k][self.k3_idx]) for k in ("m_chrom", "m_pos", "m_ref", "m_alt"))
        self.k3 = (t(self.k3_host[0], torch.int32), t(self.k3_host[1], torch.int64), t(self.k3_host[2], torch.uint8),
                   t(self.k3_host[3], torch.uint8))
        self.ctx_own = None

    def all_gather_table(self):
        """NCCL exchange (in place: this rank's block already sits at its offset of the output)."""
        import torch.distributed as dist
        dist.all_gather_into_tensor(self.gathered.view(-1, 64), self.local)

    def mutation_contexts(self, dg, k3=None):
        """K3 + substitution histogram of the rank's own mutations, written into the tail of its block (before the
        exchange; it needs the genome only, not the scan)."""
        from digdriver_b200 import kernels
        mc, mp, mr, ma = k3 if k3 is not None else self.k3
        self.ctx_own = kernels.mutation_contexts(dg, mc, mp, mr, 1, 1)
        kernels.substitution_counts(self.ctx_own, ma, 1, 1, out=self.sub)

    def finish_fused_exchange(self):
        """After a scan that stored its rows into every rank's buffer: send the partial totals after them and meet the
        other ranks (device-side barrier on the current stream; no host synchronisation)."""
        from digdriver_b200 import kernels
        if self.peer_tail:
            kernels.peer_broadcast(self.local[self.table.m:], self.peer_tail)
        self.symm.barrier(channel=0)

    def totals(self):
        return self.table.summed_totals(self.gathered)


def test_stage(dg, di, d, dist_ctx, sink=None):
    """Sequence model (K3), gene pretrain (K6), observed counts (K5), burden test (K7).  With `sink` the device
    status words are collected instead of read (no host synchronisation inside the stage)."""
    import torch
    from digdriver_b200 import kernels, pipeline
    dev = dg.device
    # the observed counts (K5) depend on nothing else in the stage: they run on a second stream next to the
    # K3 -> sequence model -> K6 chain (both are latency-bound and leave most SMs idle); inside the CUDA graph
    # this becomes two parallel branches
    main = torch.cuda.current_stream(dev)
    side = di.side_stream
    shard = getattr(di, "shard", None)
    if shard is not None:
        return strong_test_stage(dg, di, d, dist_ctx, shard, sink)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        obs, nsamp = kernels.tabulate_genes(di.m_gene, di.m_sample, di.m_cls, N_GENES, device=dev, status_sink=sink)
    ctx = kernels.mutation_contexts(dg, di.m_chrom, di.m_pos, di.m_ref, 1, 1)
    sub = kernels.substitution_counts(ctx, di.m_alt, 1, 1)
    if dist_ctx is not None:
        # genome-wide totals and substitution counts are cohort-wide quantities: all-reduce across shards
        buf = torch.cat([di.totals5, di.totals3, sub])
        dist_ctx.all_reduce_sum(buf)
        tot3, sub = buf[1024:1088], buf[1088:]
    else:
        tot3 = di.totals3
    d_pr = kernels.sequence_freq(sub.contiguous(), tot3.contiguous())
    pre = kernels.element_transfer(di.g_chrom, di.g_strand, di.g_ptr, di.g_bs, di.g_be, WINDOW, di.wmap_off,
                                   di.wmap, di.counts3, di.y_pred, di.std, di.y_true, di.flag, d_pr,
                                   L_elt=di.L, device=dev, max_span=di.max_span, status_sink=sink)
    main.wait_stream(side)
    if not torch.cuda.is_current_stream_capturing():
        obs.record_stream(main)          # allocated on the side stream, consumed on the main one
        nsamp.record_stream(main)
    res = pipeline.gene_burden_test(pre, obs, nsamp, d["n_syn"], collectives=dist_ctx)
    res["D_PR"], res["CTX"] = d_pr, ctx                  # for the parity sample (outside the timed region)
    return res


def strong_test_stage(dg, di, d, dist_ctx, shard, sink):
    """The test stage of a range-sharded run: (table exchange,) then this rank's genes (see StrongShard).  The mutation
    contexts were computed before the exchange (StrongShard.mutation_contexts): their counts arrive in the block tails."""
    import torch
    from digdriver_b200 import kernels, pipeline
    dev = dg.device
    main = torch.cuda.current_stream(dev)
    side = di.side_stream
    side.wait_stream(main)
    with torch.cuda.stream(side):
        # does not depend on the exchange: observed counts of the rank's genes
        obs, nsamp = kernels.tabulate_genes(shard.m_gene, shard.m_sample, shard.m_cls, max(shard.n_genes, 1), device=dev,
                                            status_sink=sink)
    if not shard.table_ready:
        shard.all_gather_table()                         # THE exchange: trinucleotide rows + partial totals + substitution counts
    tot = shard.totals()
    main.wait_stream(side)
    if not torch.cuda.is_current_stream_capturing():
        for t in (obs, nsamp):
            t.record_stream(main)
    d_pr = kernels.sequence_freq(tot[1088:1280].contiguous(), tot[1024:1088].contiguous())
    pre = kernels.element_transfer(shard.g_chrom, shard.g_strand, shard.g_ptr, shard.g_bs, shard.g_be, WINDOW,
                                   shard.wmap_off, shard.wmap, shard.gathered.view(-1, 64), shard.y_pred_g, shard.std_g,
                                   shard.y_true_g, shard.flag_g, d_pr, L_elt=shard.L, device=dev,
                                   max_span=shard.max_span, status_sink=sink)
    res = pipeline.gene_burden_test(pre, obs, nsamp, shard.n_syn, collectives=dist_ctx)
    res["D_PR"], res["CTX"], res["TOTALS"] = d_pr, shard.ctx_own, tot
    return res


def hot_path_step(dg, di, d, dist_ctx, ev=None):
    """One pass of the whole path on device-resident inputs.  Returns the per-gene result dict."""
    scan_stage(dg, di, ev)
    return test_stage(dg, di, d, dist_ctx)


def gather_results(coll, t):
    """Per-gene results of every shard on rank 0 (the reference's pd.concat of chunk results)."""
    return coll.gather_rows(t.unsqueeze(1), sizes=[N_GENES] * coll.world)


def result_columns():
    from digdriver_b200 import pipeline
    return ["PVAL_%s_BURDEN" % c for c in pipeline.GENE_CLASSES] + ["PVAL_%s_BURDEN_SAMPLE" % c for c in pipeline.GENE_CLASSES] + \
           ["PVAL_INDEL_BURDEN", "PVAL_MUT_BURDEN"]


def gather_strong_results(coll, shard, res):
    """The 14 p-value columns of every rank's genes on every rank: one all_gather_into_tensor of padded row blocks
    (rows are in owner-rank order; StrongShard.gene_ids maps them back to the annotation's order)."""
    import torch
    from digdriver_b200 import sharding
    cols = [res[c] for c in result_columns()]
    # stacked straight into a block of the common (longest rank's) size: no separate padding copy before the collective
    pad = torch.empty((max(shard.genes_per_rank), len(cols)), dtype=cols[0].dtype, device=cols[0].device)
    torch.stack(cols, dim=1, out=pad[: cols[0].numel()])
    return sharding.all_gather_rows(coll, pad, shard.genes_per_rank)


class GraphedStep:
    """The step as it is launched in production: the scan kernel, then ONE CUDA-graph launch holding the whole
    test stage (15 small kernels + the NCCL exchanges when sharded), so the step is not bound by launch gaps.
    Falls back to eager launches if capture is not possible (reported in the JSON line)."""

    def __init__(self, dg, di, d, dist_ctx, device):
        import torch
        from digdriver_b200 import kernels
        self.dg, self.di, self.d, self.dist_ctx = dg, di, d, dist_ctx
        self.graph, self.res, self.gathered, self.sink = None, None, None, []
        self.error = None
        try:
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                for _ in range(2):
                    self._stage()
            torch.cuda.current_stream(device).wait_stream(side)
            torch.cuda.synchronize(device)
            kernels.check_deferred(self.sink)
            g = torch.cuda.CUDAGraph()
            from digdriver_b200 import _lib
            n0 = _lib.launch_count
            with torch.cuda.graph(g):
                self._stage()
            self.launches_per_step = 1 + (_lib.launch_count - n0)      # the scan + the captured kernels
            self.graph = g
        except Exception as exc:          # report, never hide
            self.error = repr(exc)[:200]
            self.graph = None
            self.sink = []
            torch.cuda.synchronize(device)

    def _stage(self):
        self.res = test_stage(self.dg, self.di, self.d, self.dist_ctx, sink=self.sink)
        shard = getattr(self.di, "shard", None)
        if shard is not None:
            self.gathered = gather_strong_results(self.dist_ctx, shard, self.res)
        elif self.dist_ctx is not None:
            self.gathered = gather_results(self.dist_ctx, self.res["PVAL_MUT_BURDEN"])

    def step(self, ev=None):
        scan_stage(self.dg, self.di, ev)
        if self.graph is not None:
            self.graph.replay()
        else:
            self._stage()
        return self.res

    def check(self):
        """Reads the device status words of the stage (one host synchronisation, outside the timed region)."""
        from digdriver_b200 import kernels
        kernels.check_deferred(self.sink)


def parity_sample(dg, d, di, res, seed, n_windows=500, n_genes=200):
    """Post-timing self-check at full size: ~500 windows drawn over the whole 3.1 Gb genome (chromosomes beyond 2^31 in
    global coordinates included), the SNVs inside them and ~200 genes are recomputed by the CPU oracle from
    regenerated slices of the synthetic genome and compared with this run's results (oracle/parity_sample.py)."""
    import torch
    from oracle import parity_sample as ps
    dev = dg.device
    shard = getattr(di, "shard", None)
    rows = lambda t: (lambda idx: t[torch.from_numpy(np.asarray(idx)).to(dev)].cpu().numpy())
    cols = ["MU", "SIGMA", "Pi_SYN", "Pi_MIS", "Pi_NONS", "Pi_SPL", "Pi_TRUNC", "Pi_NONSYN", "ALPHA", "THETA", "OBS_SYN",
            "OBS_MIS", "OBS_NONS", "OBS_SPL", "PVAL_INDEL_BURDEN", "PVAL_MUT_BURDEN"] + ["PVAL_%s_BURDEN" % c for c in ps.CLASSES]
    if shard is None:
        # (N independent genomes, --scaling weak: the scale factors are cohort-wide, so the synonymous count the kernel
        # used is the all-reduced one that rides in SUMS[3])
        got = {"counts5": rows(di.counts5), "counts3": rows(di.counts3),
               "n_syn": float(res["SUMS"][3].item()) if res["SUMS"].numel() > 3 else d["n_syn"]}
        for k in cols:
            got[k] = res[k].cpu().numpy()
        pools = {}
    else:
        # range-sharded run: pentanucleotide rows of the rank's own windows; trinucleotide rows are read from the
        # all-gathered buffer (so windows scanned by OTHER ranks are checked too); per-gene columns of the rank's genes
        tab = shard.gathered.view(-1, 64)
        got = {"counts5": rows(di.counts5),
               "counts3": lambda idx: tab[shard.row_of[torch.from_numpy(np.asarray(idx)).to(dev)]].cpu().numpy(),
               "n_syn": float(res["SUMS"][3].item())}         # the all-reduced synonymous count the kernel used
        for k in cols:
            full = np.full(N_GENES, np.nan)
            full[shard.gene_ids] = res[k].cpu().numpy()
            got[k] = full
        pools = {"win_pool": np.arange(shard.lo, shard.hi), "gene_pool": shard.gene_ids}
    if shard is None:
        ctx_all = res["CTX"].cpu().numpy()
    else:
        ctx_all = np.full(len(d["m_pos"]), -2, dtype=np.int32)           # the mutations inside this rank's range
        ctx_all[shard.k3_idx] = res["CTX"].cpu().numpy()
    got.update({"ctx": ctx_all, "d_pr": res["D_PR"].cpu().numpy(), "sums": res["SUMS"].cpu().numpy()})
    out = ps.check_sample(d["lengths"], dg.chrom_off, seed, WINDOW, d, got, n_windows=n_windows, n_genes=n_genes, **pools)
    # EVERY window this rank scanned (all 309 990 on one GPU), both tables, against the C oracle; the totals when the rank
    # holds the whole genome
    a0, b0 = (0, len(d["wins"])) if shard is None else (shard.lo, shard.hi)
    c3rows = (lambda a, b: di.counts3[a:b].cpu().numpy()) if shard is None else \
        (lambda a, b: got["counts3"](np.arange(a, b)))
    allw = ps.check_all_windows(d["lengths"], dg.chrom_off, seed, d["wins"], lambda a, b: di.counts5[a:b].cpu().numpy(),
                                c3rows, di.totals5.cpu().numpy() if shard is None else None,
                                di.totals3.cpu().numpy() if shard is None else None, lo=a0, hi=b0)
    out["all_windows_checked"] = allw["windows"]
    if not allw["ok"]:
        out["ok"] = False
        out["detail"] += "; all windows: " + allw["detail"]
    if shard is not None:
        # rows of windows scanned by the OTHER ranks, as they arrived through the exchange
        other = np.setdiff1d(np.arange(len(d["wins"])), pools["win_pool"])
        if len(other):
            idx = np.sort(np.random.default_rng(1).choice(other, size=min(100, len(other)), replace=False))
            _, c3, _ = ps.window_rows(d["lengths"], dg.chrom_off, seed, d["wins"], idx)
            same = bool(np.array_equal(np.asarray(got["counts3"](idx), dtype=np.int64), c3))
            out["gathered_rows_checked"] = int(len(idx))
            if not same:
                out["ok"] = False
                out["detail"] += "; all-gathered trinucleotide rows differ"
    return out


DUMP_WINDOWS = 8192          # count-table rows written by --dump-outputs (the whole pentanucleotide table is 1.27 GB)
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, di, res):
    """What the last timed step computed, as out_dir/<name>.npy, for comparing two builds output for output: the rows
    of both count tables for a fixed, seeded sample of DUMP_WINDOWS windows (their indices in sample_windows), the
    genome totals, and every array of the test stage's result (per-gene columns, scale-factor sums, sequence model,
    mutation contexts).  Integer arrays whose values float32 holds exactly (the counts, the contexts) are written as
    float32, all others as float64."""
    import torch
    n_win = di.win_chrom.numel()
    rows = np.sort(np.random.default_rng(0).choice(n_win, size=min(DUMP_WINDOWS, n_win), replace=False))
    idx = torch.from_numpy(rows).to(di.counts5.device)
    arrays = {"sample_windows": rows, "counts5_sample": di.counts5[idx], "counts3_sample": di.counts3[idx],
              "totals5": di.totals5, "totals3": di.totals3}
    arrays.update(res)
    out = {}
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        exact32 = a.dtype.kind in "iub" and (a.size == 0 or int(np.abs(a).max()) < 1 << 24)
        out[name] = a.astype(np.float32 if exact32 else np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# FP64 side of the test stage at the sizes where it binds (BASELINE configs 5 and 3), outside the step's timing
# ------------------------------------------------------------------------------------------------

# FP64-pipe instructions per thread, from the ncu pass of tools/probe_fp64.py (profiles/r02_fp64_peak.txt):
# sm__inst_executed_pipe_fp64.sum x 32 / number of threads
FP64_INSTR_PER_PVALUE = 404151555 * 32 / 9_620_000          # dig_nb_burden_test, config-5 distribution of (k, alpha, p)
FP64_INSTR_PER_SITE = 539514614 * 32 / 30_000_000           # dig_site_test, config 3 (Poisson(0.05) observed counts)
FP64_PEAK_FALLBACK = 1.707e13                               # DFMA thread-instructions/s measured by tools/micro_dfma.cu


def fp64_extras(dg, di, device):
    """Timings of the two kernels of the test stage that are FP64-bound at scale: 37 cohorts x 20 k genes x 13 tests
    (config 5) through ONE launch of the burden-test kernel, and 30 M one-site site sets (config 3).  `fp64_frac` =
    FP64-pipe instructions (static count per item from the committed ncu pass) / time / measured DFMA peak."""
    import torch
    from digdriver_b200 import kernels
    peak = FP64_PEAK_FALLBACK
    exe = os.path.join(ROOT, "tools", "micro_dfma")
    src = "tools/micro_dfma.cu on an earlier box of this pool (profiles/r02_fp64_peak.txt)"
    if os.path.exists(exe):
        try:
            out = subprocess.run([exe], stdout=subprocess.PIPE, text=True, timeout=60).stdout
            for ln in out.splitlines():
                if ln.startswith("fp64_peak_dfma_per_s"):
                    peak, src = float(ln.split()[1]), "tools/micro_dfma measured in this run"
        except Exception:
            pass

    def best_ms(fn, n=3):
        fn()
        torch.cuda.synchronize(device)
        ts = []
        for _ in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize(device)
            ts.append(a.elapsed_time(b))
        return min(ts)

    g = torch.Generator(device=device)
    g.manual_seed(7)
    n5 = 37 * N_GENES * 13
    mu = torch._standard_gamma(torch.full((n5,), 2.0, dtype=torch.float64, device=device)) * 20.0
    sigma = mu * (0.05 + 0.45 * torch.rand(n5, dtype=torch.float64, device=device, generator=g))
    alpha, theta = mu ** 2 / sigma ** 2, sigma ** 2 / mu
    pi = 1e-4 + (0.05 - 1e-4) * torch.rand(n5, dtype=torch.float64, device=device, generator=g)
    k = torch.poisson(mu * pi)
    ms5 = best_ms(lambda: kernels.nb_burden_test(k, alpha, theta, pi, device))
    del mu, sigma, alpha, theta, pi, k
    n3 = 30_000_000
    n_win = di.win_chrom.numel()
    w = torch.randint(0, n_win, (n3,), device=device, generator=g)
    chrom = di.win_chrom[w]
    start = di.win_start[w] + torch.randint(0, WINDOW, (n3,), device=device, generator=g)
    sub = torch.randint(0, 192, (n3,), device=device, generator=g).to(torch.uint8)
    kk = torch.poisson(torch.full((n3,), 0.05, dtype=torch.float64, device=device))
    d_pr = torch.exp(torch.randn(192, dtype=torch.float64, device=device, generator=g) - 13.8)
    ms3 = best_ms(lambda: kernels.site_test(chrom, start, sub, kk, WINDOW, di.wmap_off, di.wmap, di.counts3, di.y_pred, di.std,
                                            d_pr, cj=1.37, device=device, want=()), n=2)
    return {"fp64_peak_thread_instr_per_s": peak, "fp64_peak_source": src,
            "config5_burden_test": {"p_values": n5, "ms": ms5, "p_values_per_s": n5 / ms5 * 1e3,
                                    "fp64_frac": n5 * FP64_INSTR_PER_PVALUE / (ms5 * 1e-3) / peak},
            "config3_site_test": {"sites": n3, "ms": ms3, "sites_per_s": n3 / ms3 * 1e3,
                                  "fp64_frac": n3 * FP64_INSTR_PER_SITE / (ms3 * 1e-3) / peak}}


# ------------------------------------------------------------------------------------------------
# e2e leg: host buffers in, host buffers out
# ------------------------------------------------------------------------------------------------

class HostPath:
    """The step through the host-buffer API of the package: digdriver_b200.host_pipeline.HostScan (pinned host genome
    -> per-chromosome H2D / pack / fused scan / uint16 narrowing / D2H on three streams) followed by the test stage on
    mutation and gene tables that also start in pinned host memory; p-values and totals end in host memory.

    source = "packed": the packed-genome cache (2-bit bases + run-length N mask, 0.25 B/base) that get_device_genome /
    countGenomeContext keep next to the FASTA -- what every run after the first uploads;
    source = "ascii": the cold path, the FASTA's bytes (1 B/base) packed on the device."""

    def __init__(self, host_genome, d, di, device, shard=None):
        import torch
        from digdriver_b200 import host_pipeline
        self.device, self.d, self.shard = device, d, shard
        wins = d["wins"]
        if shard is not None:
            wins = wins[shard.lo:shard.hi]
        self.scan = host_pipeline.HostScan(host_genome, wins, device, tile_window=WINDOW,
                                           upload_all=shard is None)
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        if shard is None:
            self.host_in = {k: pin(d[k]) for k in ("y_pred", "std", "y_true", "g_chrom", "g_strand", "g_ptr", "g_bs",
                                                    "g_be", "L", "m_chrom", "m_pos", "m_ref", "m_alt", "m_gene",
                                                    "m_cls", "m_sample")}
            self.host_in["flag"] = pin(d["flag"].astype(np.uint8))
            n_out = N_GENES
        else:
            # range-sharded: this rank's genes and their mutations, the mutations inside its window slice (K3), and
            # the region parameters of all windows (2.5 MB each; K6 may touch a neighbour's windows)
            cpu = lambda t: t.cpu()
            self.host_in = {"y_pred_g": cpu(shard.y_pred_g).pin_memory(), "std_g": cpu(shard.std_g).pin_memory(),
                            "y_true_g": cpu(shard.y_true_g).pin_memory(), "flag_g": cpu(shard.flag_g).pin_memory(),
                            "g_chrom": cpu(shard.g_chrom).pin_memory(), "g_strand": cpu(shard.g_strand).pin_memory(),
                            "g_ptr": cpu(shard.g_ptr).pin_memory(), "g_bs": cpu(shard.g_bs).pin_memory(),
                            "g_be": cpu(shard.g_be).pin_memory(), "L": cpu(shard.L).pin_memory(),
                            "m_gene": cpu(shard.m_gene).pin_memory(), "m_sample": cpu(shard.m_sample).pin_memory(),
                            "m_cls": cpu(shard.m_cls).pin_memory(),
                            "k3_chrom": pin(shard.k3_host[0].astype(np.int32)), "k3_pos": pin(shard.k3_host[1]),
                            "k3_ref": pin(shard.k3_host[2]), "k3_alt": pin(shard.k3_host[3])}
            n_out = max(shard.n_genes, 1)
        self.host_out = torch.empty((n_out, 14), dtype=torch.float64, pin_memory=True)
        self.table_stream = torch.cuda.Stream(device)
        self.h2d_bytes = self.scan.h2d_bytes + sum(v.numel() * v.element_size() for v in self.host_in.values())
        self.d2h_bytes = self.scan.d2h_bytes + self.host_out.numel() * 8
        self.launches = 0

    def step(self, di):
        import copy
        import torch
        from digdriver_b200 import _lib, kernels
        dev, d, hs, shard = self.device, self.d, self.scan, self.shard
        n0 = _lib.launch_count
        main = torch.cuda.current_stream(dev)
        self.table_stream.wait_stream(main)
        with torch.cuda.stream(self.table_stream):          # small tables ride next to the genome
            t = {k: v.to(dev, non_blocking=True) for k, v in self.host_in.items()}
            ev_tables = torch.cuda.Event()
            ev_tables.record(self.table_stream)
        hs.run(sync=False)
        main.wait_event(ev_tables)
        di2 = copy.copy(di)
        sink = []
        if shard is None:
            for k in ("y_pred", "std", "y_true", "flag", "g_chrom", "g_strand", "g_ptr", "g_bs", "g_be", "L", "m_chrom",
                      "m_pos", "m_ref", "m_alt", "m_gene", "m_cls", "m_sample"):
                setattr(di2, k, t[k])
            di2.counts3, di2.totals5, di2.totals3 = hs.counts3, hs.totals, hs.totals3
            res = test_stage(hs.genome, di2, d, None, sink=sink)
        else:
            sh = copy.copy(shard)
            for k in ("y_pred_g", "std_g", "y_true_g", "flag_g", "g_chrom", "g_strand", "g_ptr", "g_bs", "g_be", "L",
                      "m_gene", "m_sample", "m_cls"):
                setattr(sh, k, t[k])
            sh.table_ready = False                            # the host path's rows are exchanged with NCCL
            n_loc = shard.hi - shard.lo
            sh.rows[:n_loc].copy_(hs.counts3)                 # into this rank's block of the exchange buffer
            sh.tot5.copy_(hs.totals)
            sh.tot3.copy_(hs.totals3)
            # only the chromosomes of the rank's slice are resident: it handles the mutations inside its range
            sh.mutation_contexts(hs.genome, (t["k3_chrom"], t["k3_pos"], t["k3_ref"], t["k3_alt"]))
            di2.shard = sh
            from digdriver_b200.sharding import Collectives
            res = test_stage(hs.genome, di2, d, Collectives(), sink=sink)
        self.host_out.copy_(torch.stack([res[c] for c in result_columns()], dim=1), non_blocking=True)
        torch.cuda.synchronize(dev)
        hs.finish()
        kernels.check_deferred(sink)
        self.launches = _lib.launch_count - n0
        return self.host_out


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own algorithm on the host cores
# ------------------------------------------------------------------------------------------------

def _py_mutation_contexts(seq, pos, ref, n_up=1, n_down=1):
    """The reference's per-mutation loop (mutation_contexts_by_chrom, sequence_tools.py:130-178) on an in-memory
    chromosome string: fetch + upper per row, REF check, N check, same-START reuse."""
    out, prev_start, prev = [], None, None
    for st, r in zip(pos, ref):
        if st == prev_start and prev is not None:
            out.append(prev)
            continue
        s5 = seq[st - n_up:st + n_down + 1].upper()
        if len(s5) != n_up + n_down + 1 or s5[n_up] != r:
            prev_start, prev = st, None
            continue
        ctx = "" if "N" in s5 else s5
        out.append(ctx)
        prev_start, prev = st, ctx
    return out


def reference_sample_step(n_proc, windows_per_proc, genes_sample, seed, pool=None):
    """One bounded sample of the same workload with the reference's algorithm, all five stages of BASELINE.md section 3:
      scan      per-base pure-Python context counting under multiprocessing.Pool (sequence_tools.py:65-128), BOTH sizes;
      contexts  the per-mutation loop of mutation_contexts_by_chrom (sequence_tools.py:130-178);
      observed  the pandas group-bys of mutations_per_gene + distinct-sample counts (mutation_tools.py:329-361,
                transfer_tools.py:235-265) on the FULL coding-mutation table;
      transfer  the per-gene loop of genic_model / DIG_onthefly (genic_driver_tools.py:86-168, :275-283);
      test      SciPy burden tests (transfer_tools.py:394-456, :484-592, :709-729) for `genes_sample` genes.
    Pool start-up is not timed.  Returns a dict of (seconds, units) per stage."""
    import pandas as pd
    from oracle import dig_oracle
    n_win = n_proc * windows_per_proc
    L = n_win * WINDOW + 10
    seq = dig_oracle.synth_genome(0, L, seed).tobytes().decode()
    starts = np.arange(n_win) * WINDOW
    chroms = ["chr1"] * n_win
    jobs_all = []
    for (u, d) in ((2, 2), (1, 1)):
        # each worker receives only its own windows' sequence (the reference re-opens the FASTA per worker)
        for p in range(n_proc):
            a, b = p * windows_per_proc, (p + 1) * windows_per_proc
            lo = max(int(starts[a]) - u, 0)
            sub = {"chr1": seq[lo:int(starts[b - 1]) + WINDOW + d]}
            st = starts[a:b] - lo
            st[st == 0] = u                     # the reference's START == 0 -> n_up rule happens upstream
            jobs_all.append((sub, chroms[a:b], st, starts[a:b] - lo + WINDOW, u, d))
    t0 = time.perf_counter()
    if pool is not None:
        pool.map(dig_oracle._py_chunk, jobs_all, chunksize=1)
    else:
        for j in jobs_all:
            dig_oracle._py_chunk(j)
    out = {"scan": (time.perf_counter() - t0, n_win * WINDOW)}
    rng = np.random.default_rng(seed)
    # ---- mutation contexts: 30 k SNVs on the first 20 Mb of the sample
    n_mc = 30_000
    span = min(L - 10, 20_000_000)
    pos = np.sort(rng.integers(5, span, n_mc))
    up = seq[:span + 5].upper()
    ref = [up[p_] for p_ in pos]
    t0 = time.perf_counter()
    _py_mutation_contexts(seq, pos.tolist(), ref)
    out["contexts"] = (time.perf_counter() - t0, n_mc)
    # ---- observed counts: the full coding table (335 k rows), pandas as in the reference
    n_cds = int(0.30 * N_MUT) + int(0.07 * N_MUT) // 2
    w = 1.0 / np.arange(1, N_SAMPLES + 1)
    annots = np.array(["Synonymous", "Missense", "Nonsense", "Essential_Splice", "INDEL"])
    df = pd.DataFrame({"GENE": rng.integers(0, N_GENES, n_cds), "SAMPLE": rng.choice(N_SAMPLES, size=n_cds, p=w / w.sum()),
                       "ANNOT": annots[rng.choice(5, size=n_cds, p=[0.21, 0.61, 0.04, 0.04, 0.10])]})
    t0 = time.perf_counter()
    dig_oracle.gene_observed_counts(df)
    out["observed"] = (time.perf_counter() - t0, n_cds)
    # ---- gene transfer: 400 genes of ~10 exons against a 2 000-window map
    n_g, n_w = 400, 2000
    nblk = np.minimum(1 + rng.geometric(1 / 8.7, n_g), 300)
    ptr = np.concatenate([[0], np.cumsum(nblk)])
    owner = np.repeat(np.arange(n_g), nblk)
    g0 = rng.integers(10, (n_w - 60) * WINDOW, n_g)
    rel = np.concatenate([np.arange(k) for k in nblk]) * 1630
    bs = g0[owner] + rel
    be = bs + 130
    counts64 = rng.integers(50, 400, (n_w, 64))
    yp = rng.gamma(2.0, 10.0, n_w)
    index = {(0, i * WINDOW): i for i in range(n_w)}
    Lg = rng.integers(0, 40, (n_g, 192, 4)).astype(np.float64)
    d_pr = np.exp(rng.normal(np.log(1e-6), 1.0, 192))
    t0 = time.perf_counter()
    dig_oracle.gene_transfer(np.zeros(n_g, dtype=np.int64), np.where(rng.random(n_g) < 0.5, -1, 1), ptr, bs, be, Lg, WINDOW,
                             index, counts64, yp, yp * 0.2, yp, np.zeros(n_w, dtype=bool), d_pr)
    out["transfer"] = (time.perf_counter() - t0, n_g)
    # ---- the test
    E = genes_sample
    mu = rng.gamma(2.0, 20.0, E)
    sigma = mu * rng.uniform(0.05, 0.5, E)
    alpha, theta = dig_oracle.normal_params_to_gamma(mu, sigma)
    t0 = time.perf_counter()
    for _ in range(13):
        pi = rng.uniform(1e-4, 0.05, E)
        k = rng.poisson(mu * pi).astype(np.float64)
        dig_oracle.burden_test(k, alpha, theta, pi)
    dig_oracle.fisher2(rng.uniform(0, 1, E), rng.uniform(0, 1, E))
    out["test"] = (time.perf_counter() - t0, E)
    return out


def reference_value(total_bases, n_proc, seed, pool, windows_per_proc):
    """bases/s of the whole step, every stage EXTRAPOLATED linearly from its bounded sample to the workload's size."""
    st = reference_sample_step(n_proc, windows_per_proc, N_GENES, seed, pool)
    n_snv = N_MUT - int(0.07 * N_MUT)
    full = {"scan": total_bases, "contexts": n_snv, "observed": st["observed"][1], "transfer": N_GENES, "test": N_GENES}
    secs = {k: st[k][0] * (full[k] / st[k][1]) for k in st}
    return total_bases / sum(secs.values()), st, secs


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm on this box's host cores (no GPU, no torch)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    n_proc = max(1, min((os.cpu_count() or 2) - 2, 64))
    n_steps = args.warmup + args.steps
    # about 3 s of pool work per step (1000 windows = 10 Mb per worker and context size)
    wpp = 1000
    pool = mp.Pool(n_proc) if n_proc > 1 else None
    vals, sample = [], ""
    stages = None
    for i in range(n_steps):
        v, st, secs = reference_value(args.bases, n_proc, 1000 + i, pool, wpp)
        if i >= args.warmup:
            vals.append(v)
        nb = st["scan"][1]
        sample = ("EXTRAPOLATED from bounded samples, stage by stage: scan %d x 10 kb windows (%.1f Mb) for K=1024 and K=64, "
                  "pure-Python per-base loop under multiprocessing.Pool(%d): %.2f s; mutation contexts of %d SNVs "
                  "(per-row Python loop, 1 process): %.3f s; observed counts of %d coding mutations (pandas, full size): "
                  "%.3f s; gene transfer of %d genes (per-gene loop): %.3f s; 13 SciPy NB tests + Fisher on %d genes "
                  "(full size): %.3f s; each scaled linearly to %.3g bases / %d SNVs / %d genes"
                  % (nb // WINDOW, nb / 1e6, n_proc, st["scan"][0], st["contexts"][1], st["contexts"][0],
                     st["observed"][1], st["observed"][0], st["transfer"][1], st["transfer"][0], N_GENES, st["test"][0],
                     args.bases, N_MUT - int(0.07 * N_MUT), N_GENES))
        stages = {k: round(v_, 3) for k, v_ in secs.items()}
    if pool is not None:
        pool.close()
    v = float(np.median(vals))
    line = {"impl": "reference", "metric": "genome_bases_scanned_per_s", "value": v, "unit": "bases/s",
            "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup,
            "ms_per_step": args.bases / v * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8 bases -> int64 counts; f64 p-values", "data": "synthetic",
            "config": workload_config(args.bases, args.gpus, True),
            "cpu_baseline": {"value": v, "unit": "bases/s", "cores": n_proc, "kind": "port", "sample": sample,
                             "extrapolated": True, "full_size_seconds_by_stage": stages},
            "e2e": {"value": v, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_json(line)


def workload_config(bases, n_gpus, strong=True):
    return {"workload": "synthetic hg19-sized genome (%.3g bases %s, 22 chromosomes), 10 kb windows, "
                        "pentanucleotide + trinucleotide context maps with genome totals, sequence model from "
                        "1M SNVs, 20k-gene CDS pretrain + observed counts + NB burden test (13 p-values + Fisher "
                        "per gene)" % (bases, "in total" if strong else "per GPU"),
            "window": WINDOW, "genes": N_GENES, "snvs": N_MUT, "samples": N_SAMPLES,
            "parallelism": ("ONE genome range-sharded over %d GPU(s)" if strong else "one genome per GPU x%d") % n_gpus,
            "l2_policy": "inputs (1.16 GB packed genome) and outputs (1.35 GB count tables) exceed the 126 MB L2"}


# ------------------------------------------------------------------------------------------------
# main
# ------------------------------------------------------------------------------------------------

def main():
    args = parse_args()
    # Only the JSON line may appear on stdout: library banners (NCCL prints its version to stdout under torchrun)
    # and the prints of helper code are sent to stderr for the whole run.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from digdriver_b200 import _lib, host_pipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a single-process run; it is not supported under torchrun")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    placement = bind_to_gpu_numa_node(local_rank) if world > 1 else "single process, not bound"
    dist_ctx = None
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
        from digdriver_b200.sharding import Collectives
        dist_ctx = Collectives()
    strong = world > 1 and args.scaling in ("auto", "strong")

    clocks = ClockSampler(local_rank)
    clocks.start()                       # nvidia-smi takes a while to start: launch it before the set-up
    # strong: every rank builds the SAME workload (the generator is a pure function of the position) and keeps the
    # whole packed genome resident (1.16 GB), but scans only its slice; weak: one genome per rank
    seed = 1 if strong else 1 + rank
    dg, ascii_d, d = build_workload(args.bases, seed=seed, device=device)
    di = DeviceInputs(d, device)
    if strong:
        di.shard = StrongShard(d, di, dist_ctx, device, fused_exchange=args.exchange == "fused")
        n_local = float((d["wins"][di.shard.lo:di.shard.hi, 2] - d["wins"][di.shard.lo:di.shard.hi, 1]).sum())
        n_total = float((d["wins"][:, 2] - d["wins"][:, 1]).sum())
        n_genes_total = N_GENES
    else:
        n_local = float((d["wins"][:, 2] - d["wins"][:, 1]).sum())
        n_total = n_local * world
        n_genes_total = N_GENES * world

    def barrier():
        torch.cuda.synchronize(device)
        if dist_ctx is not None:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- value leg: inputs resident in HBM
    clocks.mark_begin()                  # samples kept: warm-up + timed region + e2e leg (all under load)
    res_eager = hot_path_step(dg, di, d, dist_ctx)       # eager pass: status words checked, reference result
    eager_p = res_eager["PVAL_MUT_BURDEN"].clone()
    stepper = GraphedStep(dg, di, d, dist_ctx, device)
    for _ in range(max(args.warmup, 3)):
        res = stepper.step()
    barrier()
    assert torch.equal(torch.nan_to_num(res["PVAL_MUT_BURDEN"], nan=-1.0), torch.nan_to_num(eager_p, nan=-1.0)), \
        "graph replay and eager step disagree"
    ev_all = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = _lib.launch_count
    barrier()
    start.record()
    for i in range(args.steps):
        res = stepper.step(ev=ev_all[i])
    end.record()
    barrier()
    stepper.check()
    launches = _lib.launch_count - launches0
    if stepper.graph is not None:
        # kernels replayed from the graph do not pass through _lib.call: count them from the capture pass
        launches = args.steps * stepper.launches_per_step
    elapsed_ms = start.elapsed_time(end)
    k5_ms = float(np.mean([a.elapsed_time(b) for a, b in ev_all]))
    k5_local_ms = k5_ms
    if dist_ctx is not None:
        t = torch.tensor([elapsed_ms, k5_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, k5_ms = float(t[0]), float(t[1])
    ms_per_step = elapsed_ms / args.steps
    value = n_total / (ms_per_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, di, res)

    # ---- the all-gathered result rows (range-sharded runs): every rank's block, as it arrived on EVERY rank, against the
    #      rows that rank computed (bitwise, NaN = NaN); outside the timed region
    gathered_ok = None
    shard_ = getattr(di, "shard", None)
    if shard_ is not None and dist_ctx is not None and stepper.gathered is not None:
        mine = torch.stack([res[c] for c in result_columns()], dim=1).contiguous().cpu().numpy()
        blocks = [None] * world
        dist.all_gather_object(blocks, mine)
        got_all = stepper.gathered.cpu().numpy()
        want_all = np.concatenate(blocks, axis=0)
        flag = torch.tensor([int(got_all.shape == want_all.shape and np.array_equal(got_all.view(np.int64), want_all.view(np.int64)))],
                            dtype=torch.int64, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gathered_ok = bool(int(flag[0]))

    # ---- parity at full size, outside every timed region (rank 0; the oracle regenerates the slices it needs)
    parity = None
    if rank == 0 and not args.no_parity_sample:
        try:
            parity = parity_sample(dg, d, di, res, seed=seed)
        except Exception as exc:      # report, never hide
            parity = {"ok": False, "detail": "parity sample failed to run: %r" % (exc,)}
        if gathered_ok is not None:
            parity["gathered_result_rows_ok"] = gathered_ok
            if not gathered_ok:
                parity["ok"] = False
                parity["detail"] = parity.get("detail", "") + "; all-gathered result rows differ from the ranks' own rows"

    # ---- e2e leg: host buffers in and out, through digdriver_b200.host_pipeline
    e2e = None
    if not args.no_e2e:
        shard = getattr(di, "shard", None)

        def timed(hp, n):
            for _ in range(2):
                hp.step(di)
            barrier()
            t0 = time.perf_counter()
            for _ in range(n):
                hp.step(di)
            barrier()
            sec = (time.perf_counter() - t0) / n
            if dist_ctx is not None:
                tt = torch.tensor([sec], dtype=torch.float64, device=device)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                sec = float(tt[0])
            return sec

        def totals_over_ranks(*vals):
            tt = torch.tensor(vals, dtype=torch.float64, device=device)
            if dist_ctx is not None:
                dist.all_reduce(tt, op=dist.ReduceOp.SUM)
            return [int(v) for v in tt.tolist()]

        # (1) the steady state: the packed-genome cache as the source (every run after the first one)
        hg_packed = host_pipeline.HostGenome.from_device(dg)
        hp = HostPath(hg_packed, d, di, device, shard=shard)
        e2e_s = timed(hp, args.steps)
        h2d, d2h = totals_over_ranks(hp.h2d_bytes, hp.d2h_bytes)
        e2e = {"value": n_total / e2e_s, "unit": "bases/s", "ms_per_step": e2e_s * 1e3,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "gpu_launches_per_step": hp.launches,
               "api": "digdriver_b200.host_pipeline.HostScan + test stage: pinned host packed genome (the .dig2bit cache "
                      "of get_device_genome / countGenomeContext: 2-bit bases + run-length N mask, 0.25 B/base) + mutation "
                      "/ gene tables in; uint16 count tables, totals and 14 p-value columns out; bytes are summed over ranks"}
        # host-side check of what arrived (outside the timing): totals of the host copy == device totals of the value leg
        if rank == 0 and shard is None:
            same = bool(torch.equal(hp.scan.host_totals, torch.cat([di.totals5, di.totals3]).cpu()))
            row_ok = bool(np.array_equal(hp.scan.host_counts[:64].numpy().astype(np.int64), di.counts5[:64].cpu().numpy()))
            e2e["host_results_match_value_leg"] = same and row_ok
        del hp, hg_packed
        # (2) the cold path: ASCII in (first run on a new FASTA), packed on the device
        hg_ascii = host_pipeline.HostGenome.from_device(dg, ascii_d)
        del ascii_d
        hp = HostPath(hg_ascii, d, di, device, shard=shard)
        cold_s = timed(hp, args.steps)
        h2d, d2h = totals_over_ranks(hp.h2d_bytes, hp.d2h_bytes)
        e2e["cold"] = {"value": n_total / cold_s, "ms_per_step": cold_s * 1e3, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "source": "pinned host ASCII genome (1 B/base), K1 pack on the device"}
        del hp, hg_ascii

    fp64 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            fp64 = fp64_extras(dg, di, device)
        except Exception as exc:      # report, never hide
            fp64 = {"error": repr(exc)[:200]}

    clocks.mark_end()
    clock_info = clocks.stop()

    # ---- roofline of the dominant kernel
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, which = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, which = 6650.0, "fallback (B200_PROFILING.md)"
    # the scan of THIS rank's windows against its own launch time (rank 0's)
    achieved = n_local * B_PER_BASE_FUSED / (k5_local_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "scan_lb_kernel<TRI, TOT> (lane-bank scan: pentanucleotide K=1024 through "
                                          "hexamer pairs + trinucleotide K=64 window tables and genome totals in one pass; "
                                          "followed by scan_hex_kernel over its redo list, empty here)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of one launch at the default size, from the committed
                # ncu --set full capture (profiles/r02_scan_lb_summary.txt)
                "traffic": SCAN_DRAM_TRAFFIC if abs(args.bases - 3.1e9) < 1 and not strong else None,
                "algorithmic_bytes": n_local * B_PER_BASE_FUSED,
                "peak_source": which, "kernel_ms": k5_local_ms,
                "algorithmic_bytes_per_base": B_PER_BASE_FUSED,
                "note": "HBM is the roofline the contract asks for; the kernel alternates an integer-ALU-bound counting "
                        "phase with a shared-memory-bound write-out phase (DESIGN.md section 4)",
                "share_of_step": k5_local_ms / ms_per_step}

    def finish():
        """Leave without tearing NCCL down: destroy_process_group() after a CUDA graph that holds NCCL kernels was
        captured can block for ever (seen at N=2), and the process is exiting anyway."""
        sys.stdout.flush()
        sys.stderr.flush()
        if dist_ctx is not None:
            stepper.graph = None
            torch.cuda.synchronize(device)
            dist.barrier()
            torch.cuda.synchronize(device)
            os._exit(0)

    if rank != 0:
        finish()
        return

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the reference's algorithm
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        # run in a fresh process (no CUDA context to fork) through the same code as --impl reference
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3",
                              "--warmup", "1", "--bases", str(args.bases)], stdout=subprocess.PIPE, text=True)
        try:
            cpu_baseline = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as exc:      # report, never hide
            cpu_baseline = {"error": "reference arm failed: %r" % (exc,)}

    line = {"metric": "genome_bases_scanned_per_s", "value": value, "unit": "bases/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong" if strong or world == 1 else "weak", "vs_baseline": None,
            "dtype": "u8 bases -> int32 counts; f64 p-values", "data": "synthetic",
            "config": workload_config(args.bases, world, strong or world == 1),
            "elements_tested_per_s": n_genes_total / (ms_per_step * 1e-3),
            "cuda_graph": {"test_stage_captured": stepper.graph is not None, "error": stepper.error},
            "host_placement": placement,
            "clocks": clock_info, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
            "cpu_baseline": cpu_baseline, "parity_sample": parity, "test_stage_fp64": fp64}
    if strong:
        sh = di.shard
        how = ("trinucleotide rows stored into every rank's buffer BY THE SCAN KERNEL (%s), partial totals by one "
               "dig_peer_broadcast, one device barrier" % sh.fused_note) if sh.fused else \
              ("1 all_gather_into_tensor of %.1f MB (trinucleotide rows + partial totals) [%s]" % (sh.exchange_bytes / 1e6, sh.fused_note))
        line["sharding"] = {"windows_per_rank": [b - a for a, b in sh.table.parts], "genes_per_rank": sh.genes_per_rank,
                            "exchange": how + "; then 1 all_reduce of 4 doubles and 1 all_gather_into_tensor of the result "
                                              "rows inside the CUDA graph",
                            "scan_kernel_ms_max_over_ranks": k5_ms}
    emit_json(line)
    finish()


if __name__ == "__main__":
    main()
