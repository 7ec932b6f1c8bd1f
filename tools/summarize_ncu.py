"""Turn ncu outputs into the small text summaries committed under profiles/.

  python tools/summarize_ncu.py launches gpurun_out/launches.csv  > profiles/rNN_launches.txt
  python tools/summarize_ncu.py kernel   gpurun_out/prof.ncu-rep   > profiles/rNN_kernel.txt
"""
import collections
import csv
import subprocess
import sys

KEYS = [
    "gpu__time_duration.sum", "sm__cycles_elapsed.avg", "launch__grid_size", "launch__block_size",
    "launch__registers_per_thread", "launch__occupancy_limit_registers", "launch__occupancy_limit_shared_mem",
    "sm__warps_active.avg.pct_of_peak_sustained_active", "dram__bytes_read.sum", "dram__bytes_write.sum",
    "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
    "smsp__inst_executed.sum", "smsp__issue_active.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active",
    "l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed",
    "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum", "l1tex__data_pipe_lsu_wavefronts_mem_shared_op_atom.sum",
    "smsp__inst_executed_op_shared_atom.sum", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum",
    "lts__t_bytes.sum",
]


def launches(path):
    lines = [l for l in open(path) if not l.startswith("==")]
    rows = list(csv.DictReader(lines))
    names = [(r["Kernel Name"], float(r["Metric Value"].replace(",", ""))) for r in rows]
    if any("scan_lb_kernel" in n for n, _ in names):
        is_scan = lambda n: "scan_lb_kernel" in n       # noqa: E731  (its redo pass, scan_hex_kernel, belongs to the same step)
    else:
        is_scan = lambda n: "scan_sym_kernel<2" in n or "scan_hex_kernel" in n   # noqa: E731
    big = max([v for n, v in names if is_scan(n)] or [0.0])
    # a step = one whole-genome scan (the per-chromosome scans of the e2e leg are much shorter) and what follows it,
    # up to the next scan or pack launch; the last COMPLETE one is reported (-c may cut the run anywhere)
    marks = [i for i, (n, v) in enumerate(names) if is_scan(n) and v >= 0.5 * big]
    step = names
    for m in reversed(marks):
        end = next((j for j in range(m + 1, len(names)) if is_scan(names[j][0]) or "pack_kernel" in names[j][0]), None)
        if end is not None or m == marks[-1]:
            step = names[m:end]
            if end is not None:
                break
    tot = sum(v for _, v in step)
    agg = collections.OrderedDict()
    for n, v in step:
        k = n.split("(")[0][-70:]
        agg.setdefault(k, [0, 0.0])
        agg[k][0] += 1
        agg[k][1] += v
    print("# last step of the run: %d launches, %.1f us of kernel time (ncu serialised, cold cache: compare SHARES)" %
          (len(step), tot / 1e3))
    for k, (c, v) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print("%9.1f us %5.1f%%  x%-3d %s" % (v / 1e3, 100 * v / tot, c, k))


def kernel(path):
    out = subprocess.run(["ncu", "-i", path, "--page", "raw", "--csv"], stdout=subprocess.PIPE, text=True).stdout
    rows = list(csv.reader(out.splitlines()))
    hdr, units = rows[0], rows[1]
    for r in rows[2:]:
        d = dict(zip(hdr, r))
        print("== %s" % d["Kernel Name"][:120])
        for k in KEYS:
            if k in d:
                print("   %-72s %s %s" % (k, d[k], units[hdr.index(k)]))
        st = {k: float(v.replace(",", "")) for k, v in d.items()
              if k.startswith("smsp__average_warps_issue_stalled") and k.endswith("_per_issue_active.ratio")}
        print("   top stall reasons (warps stalled per issue-active cycle):")
        for k, v in sorted(st.items(), key=lambda kv: -kv[1])[:6]:
            print("      %-60s %.2f" % (k.replace("smsp__average_warps_issue_stalled_", "").replace("_per_issue_active.ratio", ""), v))


if __name__ == "__main__":
    {"launches": launches, "kernel": kernel}[sys.argv[1]](sys.argv[2])
