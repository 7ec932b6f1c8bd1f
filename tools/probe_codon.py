"""Device timing of the codon-test entry points (K9c / K10 / K9d, csrc/codon.cu) at hg19 size, with CUDA events.

    python tools/probe_codon.py [--genes 20000] [--snvs 1000000]

Workload: the 3.1 Gb synthetic genome (22 hg19-proportioned autosomes), pipeline.synth_genes genes (about 32 Mb of
CDS), 10 kb windows with random region parameters, and a cohort of which 70 % of rows are codon sites.  Prints the card
name and power limit first.  Timed (warm, 20 runs): dig_codon_sites on the whole gene set, dig_window_denominators +
dig_codon_transfer, dig_snv_codons alone on the join's pairs, dig_nb_burden_test on every tested codon; then
codon_model_arrays end to end on in-memory inputs (enumeration, transfer, join, string checks, K5, K7, q-values and the
results table; 20 runs).  run_codon_model is that plus reading its files; the cohort file, the largest of them, is
timed on its own (read_mutation_file, 20 runs), the FASTA is parsed once per process and cached.
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402

from digdriver_b200 import _lib, genome as G, kernels, pipeline  # noqa: E402
from digdriver_b200.data_tools import mutation_tools  # noqa: E402
from digdriver_b200.driver_model import codon_tools  # noqa: E402
from digdriver_b200.sequence_model.genic_driver_tools import RegionModel  # noqa: E402


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


class Genes:
    def __init__(self, chrom, strand, ptr, bs, be):
        self.chrom, self.strand = chrom.astype(np.int64) + 1, strand.astype(np.int8)
        self.ptr, self.start, self.end = ptr, bs, be
        self.names = np.array(["G%d" % e for e in range(len(chrom))])

    def __len__(self):
        return len(self.names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genes", type=int, default=20_000)
    ap.add_argument("--snvs", type=int, default=1_000_000)
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
    gs = Genes(chrom, strand, ptr, bs, be)
    E, cds = len(chrom), int((be - bs + 1).sum())
    dev = g.device
    wins = G.tile_windows(list(range(1, 23)), lengths, 10_000)
    rng = np.random.default_rng(3)
    n = len(wins)
    rm = RegionModel(pd.DataFrame({"CHROM": wins[:, 0], "START": wins[:, 1], "END": wins[:, 2],
                                   "Y_TRUE": rng.poisson(20, n), "Y_PRED": rng.gamma(2.0, 10.0, n),
                                   "STD": rng.uniform(0.5, 5.0, n), "FLAG": rng.random(n) < 0.1}))
    wc, _ = kernels.count_contexts(g, g.chrom_indices(wins[:, 0]), wins[:, 1], wins[:, 2], 1, 1)
    d_pr = rng.uniform(1e-9, 1e-7, 192)
    cs = codon_tools.enumerate_codons(g, gs)
    n_codon = cs["N_SITES"].numel()
    tested = torch.nonzero(cs["N_SITES"]).squeeze(1)
    n_sites = int(cs["N_SITES"].sum(dtype=torch.int64).item())
    print("genes %d, CDS %.1f Mb, codons %d, tested %d, sites %d, windows %d"
          % (E, cds / 1e6, n_codon, tested.numel(), n_sites, n))
    st = torch.cuda.current_stream().cuda_stream
    gcd = torch.from_numpy(g.chrom_indices(gs.chrom)).to(dev)
    gsd = torch.from_numpy(gs.strand).to(dev)
    bp, b0, b1 = (torch.from_numpy(x.astype(np.int64)).to(dev) for x in (ptr, bs, be))
    status = torch.zeros(1, dtype=torch.int32, device=dev)

    def sites():
        _lib.call("dig_codon_sites", g.packed2.data_ptr(), g.nmask.data_ptr(), g.n_bases, g.chrom_off_d.data_ptr(),
                  g.chrom_len_d.data_ptr(), len(lengths), gcd.data_ptr(), gsd.data_ptr(), bp.data_ptr(), b0.data_ptr(),
                  b1.data_ptr(), E, cs["PTR"].data_ptr(), n_codon, cs["POS"].data_ptr(), cs["BIN"].data_ptr(),
                  cs["CLASS"].data_ptr(), cs["REF_AA"].data_ptr(), cs["N_SITES"].data_ptr(), status.data_ptr(), st)

    best, med, worst = timed(sites)
    assert int(status.item()) == 0
    print("dig_codon_sites: best %.3f ms, median %.3f ms, max %.3f ms over 20 runs -> %.1f M codons/s"
          % (best, med, worst, n_codon / best / 1e3))
    best, med, worst = timed(lambda: kernels.codon_transfer(cs, gs.chrom, gs.strand, rm.window, rm.win_map_off,
                                                            rm.win_map, wc, rm.y_pred, rm.std, rm.y_true, rm.flag, d_pr,
                                                            dev))
    print("kernels.codon_transfer (dig_window_denominators + dig_codon_transfer, inputs already on the device "
          "except the region model): best %.3f ms, median %.3f ms, max %.3f ms over 20 runs" % (best, med, worst))
    tr = kernels.codon_transfer(cs, gs.chrom, gs.strand, rm.window, rm.win_map_off, rm.win_map, wc, rm.y_pred, rm.std,
                                rm.y_true, rm.flag, d_pr, dev)
    wm0, wm1 = torch.from_numpy(rm.win_map_off).to(dev), torch.from_numpy(rm.win_map).to(dev)
    yp, sd, yt = (torch.from_numpy(x).to(dev) for x in (rm.y_pred, rm.std, rm.y_true))
    fl = torch.from_numpy(rm.flag.astype(np.uint8)).to(dev)
    wcd = wc.to(torch.int32).contiguous()
    dp = torch.from_numpy(d_pr).to(dev)
    den_p = torch.empty(n, dtype=torch.float64, device=dev)
    den_m = torch.empty(n, dtype=torch.float64, device=dev)
    gnum = torch.from_numpy(gs.chrom.astype(np.int32)).to(dev)
    _lib.call("dig_window_denominators", wcd.data_ptr(), dp.data_ptr(), n, den_p.data_ptr(), den_m.data_ptr(), st)

    def transfer():
        _lib.call("dig_codon_transfer", cs["PTR"].data_ptr(), gnum.data_ptr(), gsd.data_ptr(), E, cs["POS"].data_ptr(),
                  cs["BIN"].data_ptr(), cs["N_SITES"].data_ptr(), n_codon, rm.window, wm0.numel() - 1, wm0.data_ptr(),
                  wm1.data_ptr(), wcd.data_ptr(), yp.data_ptr(), sd.data_ptr(), yt.data_ptr(), fl.data_ptr(),
                  den_p.data_ptr(), den_m.data_ptr(), dp.data_ptr(), tr["MU"].data_ptr(), tr["SIGMA"].data_ptr(),
                  tr["R_OBS"].data_ptr(), tr["FLAG"].data_ptr(), tr["R_SIZE"].data_ptr(), tr["PI_NUM"].data_ptr(),
                  tr["PI_SUM"].data_ptr(), tr["N_WIN"].data_ptr(), status.data_ptr(), st)

    best, med, worst = timed(transfer)
    assert int(status.item()) == 0
    print("dig_codon_transfer alone: best %.3f ms, median %.3f ms, max %.3f ms over 20 runs -> %.1f M codons/s"
          % (best, med, worst, n_codon / best / 1e3))
    # cohort: site rows; the last 30 % relabelled Synonymous, so that they match no site
    bins, cls, pos = cs["BIN"].cpu().numpy(), cs["CLASS"].cpu().numpy(), cs["POS"].cpu().numpy()
    cptr = cs["PTR"].cpu().numpy()
    ci, sl = np.nonzero(bins != 255)
    pick = rng.integers(0, len(ci), args.snvs)
    ci, sl = ci[pick], sl[pick]
    gene = np.searchsorted(cptr, ci, side="right") - 1
    ref, alt, ctx = codon_tools._site_bases(bins[ci, sl], gs.strand[gene] < 0)
    p = pos[ci, sl // 3]
    REF, ALT = codon_tools._ACGT[ref], codon_tools._ACGT[alt]
    df_mut = pd.DataFrame({"CHROM": gs.chrom[gene], "START": p, "END": p + 1, "REF": REF, "ALT": ALT,
                           "SAMPLE": np.char.add("S", (np.arange(len(p)) % 500).astype(str)), "GENE": gs.names[gene],
                           "ANNOT": codon_tools.CLASS_NAMES[cls[ci, sl]], "MUT_TYPE": REF + ">" + ALT,
                           "CONTEXT": codon_tools._TRI[ctx]})
    df_mut.loc[np.arange(len(df_mut)) >= int(0.7 * len(df_mut)), "ANNOT"] = "Synonymous"
    mchrom = torch.from_numpy(g.chrom_indices(gs.chrom[gene]).astype(np.int64)).to(dev)
    pm, pg = kernels._snv_gene_pairs(dev, gcd, bp, b0, b1, mchrom, torch.from_numpy(p).to(dev), 0, None)
    mr, ma = torch.from_numpy(ref.astype(np.uint8)).to(dev), torch.from_numpy(alt.astype(np.uint8)).to(dev)
    mp = torch.from_numpy(p).to(dev)
    n_pair = pm.numel()
    co = torch.empty(n_pair, dtype=torch.int64, device=dev)
    so = torch.empty(n_pair, dtype=torch.uint8, device=dev)

    def snv():
        _lib.call("dig_snv_codons", gsd.data_ptr(), bp.data_ptr(), b0.data_ptr(), b1.data_ptr(), cs["PTR"].data_ptr(),
                  E, cs["POS"].data_ptr(), cs["BIN"].data_ptr(), mp.data_ptr(), mr.data_ptr(), ma.data_ptr(),
                  pm.data_ptr(), pg.data_ptr(), n_pair, co.data_ptr(), so.data_ptr(), status.data_ptr(), st)

    best, med, worst = timed(snv)
    print("dig_snv_codons: %d SNVs -> %d (mutation, gene) pairs, %d on a site; best %.3f ms, median %.3f ms, "
          "max %.3f ms over 20 runs" % (args.snvs, n_pair, int((co >= 0).sum()), best, med, worst))
    k = torch.ones(tested.numel(), dtype=torch.float64, device=dev)
    mu, sg, pi = tr["MU"][tested], tr["SIGMA"][tested], tr["PI_SUM"][tested]
    alpha, theta = mu * mu / (sg * sg), sg * sg / mu
    best, med, worst = timed(lambda: kernels.nb_burden_test(k, alpha, theta, pi, dev))
    print("dig_nb_burden_test on %d tested codons (EXP + p-value): best %.3f ms, median %.3f ms, max %.3f ms over "
          "20 runs" % (tested.numel(), best, med, worst))
    del tr
    ts = []
    for _ in range(21):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res, n_tested = codon_tools.codon_model_arrays(g, gs, rm, wc, d_pr, df_mut, 1.0)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    print("codon_model_arrays end to end on in-memory inputs (%d tested codons, %d rows with OBS_SNV >= 1, OBS_SNV "
          "total %d): best %.2f s, median %.2f s over 20 runs after one warm-up (wall clock; no file is read)"
          % (n_tested, len(res), int(res.OBS_SNV.sum()), min(ts[1:]), float(np.median(ts[1:]))))
    # the host file I/O run_codon_model adds: it reads the cohort file twice (scale factor, observed counts)
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "cohort.tsv")
        df_mut.to_csv(f, sep="\t", header=False, index=False)
        ts = []
        for _ in range(20):
            t0 = time.perf_counter()
            mutation_tools.read_mutation_file(f, drop_duplicates=False)
            ts.append(time.perf_counter() - t0)
    print("read_mutation_file of the %d-row cohort (10 columns): best %.2f s, median %.2f s over 20 runs; "
          "run_codon_model reads it twice, so file I/O adds about %.1f s to the line above"
          % (len(df_mut), min(ts), float(np.median(ts)), 2 * float(np.median(ts))))


if __name__ == "__main__":
    main()
