"""The constructed edge set of the codon tests (tests/test_gpu_codon_exact.py on a 3.1 Gb genome, tests/test_exact_ref.py
on the 3.3 Mb genome of the small fixtures): genes placed where the annotation and codon kernels can go wrong.  Plain
numpy, no device."""
import numpy as np


def n_runs(seq, offset=0):
    """(start, end) of every N run (end exclusive) of a stretch of a chromosome that starts at position offset."""
    isn = np.concatenate([[False], (np.asarray(seq) | 0x20) == ord("n"), [False]])
    d = np.diff(isn.astype(np.int8))
    return list(zip((np.flatnonzero(d == 1) + offset).tolist(), (np.flatnonzero(d == -1) + offset).tolist()))


def edge_gene_set(lengths, runs, window, small=False):
    """Constructed genes (chrom index, strand, ptr, blk_start, blk_end), window-aligned where it matters:
    codons over two and three blocks (1- and 2-bp exons) on both strands and their opposite-strand twins; genes of
    1-bp exons one window apart (every codon over three windows, about half of them with a site on all three bases:
    >= 100 such codons on the minus strand); 3-bp exons straddling a window edge every other window (a lone third base
    in the next window or the previous one, often without a site); exons next to and across N runs (runs[c] = N runs known on chromosome c); genes on the first and
    last base of chromosomes; a gene of exactly 2048 blocks and one of > 40 000 codons."""
    lengths = np.asarray(lengths, dtype=np.int64)
    genes = []
    cursor = {c: 60_000 for c in range(len(lengths))}

    def alloc(size, order):
        for c in order:
            x = -(-cursor[c] // window) * window + window
            if x + size + 60_000 < lengths[c]:
                cursor[c] = x + size + window
                return c, x
        raise AssertionError("no room for %d bases" % size)
    order = list(range(len(lengths))) if small else [1, 2, 3, 4, 5]
    # codons over two and three blocks, both strands, and an opposite-strand twin shifted by one base
    for shape in ([(0, 10), (20, 20), (30, 31), (40, 61)], [(0, 3), (10, 10), (15, 15), (20, 21), (30, 30), (40, 52)],
                  [(0, 1), (9, 9), (12, 12), (20, 20), (25, 26), (33, 80)]):
        c, x = alloc(200, order)
        for strand in (1, -1):
            genes.append((c, strand, [(x + s, x + t) for s, t in shape]))
        genes.append((c, -1, [(x + s + 1, x + t + 1) for s, t in shape]))
    # 1-bp exons one window apart: minus (300 codons, about half with a site on every base) and plus
    for strand, nb in ((-1, 60 if small else 900), (1, 30 if small else 99)):
        c, x = alloc(nb * window, order)
        genes.append((c, strand, [(x + i * window + 1000 + (37 * i) % 8000,) * 2 for i in range(nb)]))
    # 3-bp exons straddling a window edge every other window: plus [kW-2, kW] (lone third base after the edge),
    # minus [kW-1, kW+1] (lone third transcript base before it)
    for strand, shape in ((1, (-2, 0)), (-1, (-1, 1))):
        nb = 20 if small else 200
        c, x = alloc(2 * nb * window + window, order)
        genes.append((c, strand, [(x + 2 * k * window + shape[0], x + 2 * k * window + shape[1]) for k in range(1, nb + 1)]))
    # N runs: an exon ending just before a run, one starting just after it, one across its start
    for c, rr in sorted(runs.items()) if isinstance(runs, dict) else enumerate(runs):
        for ns, ne in [r for r in rr if r[0] > 2000 and r[1] + 2000 < lengths[c]][:2]:
            for strand in (1, -1):
                genes.append((c, strand, [(ns - 400, ns - 351), (ns - 100, ns - 1)]))
                genes.append((c, strand, [(ne, ne + 60), (ne + 100, ne + 131)]))
                genes.append((c, strand, [(ns - 300, ns - 250), (ns - 40, ns + 4), (ne + 5, ne + 30)]))
    # the first and last base of chromosomes
    for c in range(len(lengths)) if small else range(0, len(lengths), 3):
        L = int(lengths[c])
        genes += [(c, 1, [(0, 40), (50, 80)]), (c, -1, [(0, 0), (5, 50)]),
                  (c, -1, [(L - 60, L - 30), (L - 20, L - 1)]), (c, 1, [(L - 61, L - 61), (L - 55, L - 1)])]
    # exactly 2048 blocks (40 960 codons), and > 40 000 codons in ten blocks
    c, x = alloc(2048 * 100, order)
    genes.append((c, 1, [(x + 100 * i, x + 100 * i + 59) for i in range(2048)]))
    c, x = alloc(10 * 12_103, order)
    genes.append((c, -1, [(x + 12_103 * i, x + 12_103 * i + 12_002) for i in range(10)]))
    chrom = np.array([g[0] for g in genes], dtype=np.int32)
    strand = np.array([g[1] for g in genes], dtype=np.int8)
    ptr = np.concatenate([[0], np.cumsum([len(g[2]) for g in genes])]).astype(np.int64)
    bs = np.array([b[0] for g in genes for b in g[2]], dtype=np.int64)
    be = np.array([b[1] for g in genes for b in g[2]], dtype=np.int64)
    return chrom, strand, ptr, bs, be
