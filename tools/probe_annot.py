"""Device timing of the gene annotation entry points (K9, csrc/cdsannot.cu) at hg19 size, with CUDA events.

    python tools/probe_annot.py [--genes 20000] [--snvs 1000000] [--coding 0.3]

Workload: the 3.1 Gb synthetic genome (22 hg19-proportioned autosomes), pipeline.synth_genes genes (about 30 Mb of
CDS), SNVs of which the given fraction sits on CDS bases and the rest anywhere in the genome.  Prints the card name and
power limit first.  Timed: dig_cds_substitution_table (the whole gene set), dig_annotate_snvs alone on the (mutation,
gene) pairs of the join, and kernels.annotate_snvs end to end (join, pair de-duplication, classification; it reads
the pair count back to the host once).
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from digdriver_b200 import _lib, genome as G, kernels, pipeline  # noqa: E402


def timed(fn, n=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), float(np.median(ts)), max(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genes", type=int, default=20_000)
    ap.add_argument("--snvs", type=int, default=1_000_000)
    ap.add_argument("--coding", type=float, default=0.3)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    print("device: %s | %s" % (torch.cuda.get_device_name(0), q))
    lengths = G.hg19_like_lengths()
    g = G.DeviceGenome.synthetic(["chr%d" % i for i in range(1, 23)], lengths, seed=5, device="cuda:0")
    chrom, strand, ptr, bs, be = pipeline.synth_genes(args.genes, lengths, 10_000, seed=9)
    ok = np.array([np.all(bs[ptr[e] + 1:ptr[e + 1]] > be[ptr[e]:ptr[e + 1] - 1]) for e in range(len(chrom))])
    keep = np.flatnonzero(ok)
    take = np.concatenate([np.arange(ptr[i], ptr[i + 1]) for i in keep])
    ptr = np.concatenate([[0], np.cumsum(np.diff(ptr)[keep])]).astype(np.int64)
    chrom, strand, bs, be = chrom[keep], strand[keep], bs[take], be[take]
    E, cds = len(chrom), int((be - bs + 1).sum())
    print("genes %d (of %d drawn; %d with overlapping blocks left out), blocks %d, CDS %.1f Mb"
          % (E, args.genes, args.genes - E, len(bs), cds / 1e6))
    dev = g.device
    gc, gs = torch.from_numpy(chrom.astype(np.int32)).to(dev), torch.from_numpy(strand.astype(np.int8)).to(dev)
    bp, b0, b1 = (torch.from_numpy(x.astype(np.int64)).to(dev) for x in (ptr, bs, be))
    L = torch.empty((E, 192, 4), dtype=torch.float64, device=dev)
    flags = torch.empty(E, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    d, nd, a, na = kernels._splice_offsets((1, 2, 5), (1, 2))
    st = torch.cuda.current_stream().cuda_stream
    nchr = len(lengths)

    def table():
        _lib.call("dig_cds_substitution_table", g.packed2.data_ptr(), g.nmask.data_ptr(), g.n_bases,
                  g.chrom_off_d.data_ptr(), g.chrom_len_d.data_ptr(), nchr, gc.data_ptr(), gs.data_ptr(), bp.data_ptr(),
                  b0.data_ptr(), b1.data_ptr(), E, d, nd, a, na, L.data_ptr(), flags.data_ptr(), status.data_ptr(), st)

    best, med, worst = timed(table)
    assert int(status.item()) == 0
    n_sites = 9.0 * cds
    print("dig_cds_substitution_table: best %.3f ms, median %.3f ms, max %.3f ms over 20 runs -> %.2f G substitutions/s; "
          "flagged genes %d" % (best, med, worst, n_sites / best / 1e6, int((flags != 0).sum())))
    rng = np.random.default_rng(3)
    n_cod = int(args.snvs * args.coding)
    blk = rng.choice(len(bs), n_cod, p=(be - bs + 1) / cds)
    owner = np.repeat(np.arange(E), np.diff(ptr))
    mc = np.concatenate([chrom[owner[blk]], rng.choice(nchr, args.snvs - n_cod, p=lengths / lengths.sum())]).astype(np.int64)
    mp = np.concatenate([bs[blk] + (rng.random(n_cod) * (be[blk] - bs[blk] + 1)).astype(np.int64),
                         (rng.random(args.snvs - n_cod) * lengths[mc[n_cod:]]).astype(np.int64)])
    ma = rng.integers(0, 4, args.snvs).astype(np.uint8)
    mc_d, mp_d, ma_d = (torch.from_numpy(x).to(dev) for x in (mc, mp, ma))
    pm, pg, cls = kernels.annotate_snvs(g, gc, gs, bp, b0, b1, mc_d, mp_d, ma_d)
    n_pair = pm.numel()
    out = torch.empty(n_pair, dtype=torch.uint8, device=dev)

    def annot():
        _lib.call("dig_annotate_snvs", g.packed2.data_ptr(), g.nmask.data_ptr(), g.n_bases, g.chrom_off_d.data_ptr(),
                  g.chrom_len_d.data_ptr(), nchr, gc.data_ptr(), gs.data_ptr(), bp.data_ptr(), b0.data_ptr(),
                  b1.data_ptr(), E, d, nd, a, na, mp_d.data_ptr(), ma_d.data_ptr(), pm.data_ptr(), pg.data_ptr(),
                  n_pair, out.data_ptr(), status.data_ptr(), st)

    best, med, worst = timed(annot)
    c = cls.cpu().numpy()
    print("dig_annotate_snvs: %d SNVs (%.0f%% on CDS) -> %d (mutation, gene) pairs, %d with a class; best %.3f ms, "
          "median %.3f ms, max %.3f ms over 20 runs" % (args.snvs, 100 * args.coding, n_pair, int((c != 255).sum()),
                                                        best, med, worst))
    best, med, worst = timed(lambda: kernels.annotate_snvs(g, gc, gs, bp, b0, b1, mc_d, mp_d, ma_d), n=10)
    print("kernels.annotate_snvs (join + de-duplication + classification): best %.3f ms, median %.3f ms, max %.3f ms "
          "over 10 runs" % (best, med, worst))


if __name__ == "__main__":
    main()
