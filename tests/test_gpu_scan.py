"""GPU parity tests for K1 (pack), K2 (window scan) and K4 (strand-aware block counts).
Everything goes through the C ABI (digdriver_b200.kernels -> libdigb200.so) and is compared
bit-exactly with the golden vectors of the unmodified reference and with the CPU oracle."""
import numpy as np
import pytest
import torch

from conftest import golden, golden_genome

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def gold_dev_genome(dev):
    from digdriver_b200.genome import Genome, DeviceGenome
    z = golden("scan")
    g = Genome(["chr1", "chr2"], [z["seq_chr1"], z["seq_chr2"]])
    return DeviceGenome.from_genome(g, dev)


def test_pack_matches_layout_definition(dev, oracle):
    from digdriver_b200.genome import DeviceGenome
    rng = np.random.default_rng(5)
    for n in (1, 15, 16, 17, 31, 32, 33, 1000, 4097, 100003):
        seq = rng.choice(np.frombuffer(b"ACGTacgtNnRYx-", dtype=np.uint8), size=n)
        for shift in (0, 3):                 # aligned and unaligned device pointers
            buf = torch.zeros(n + shift, dtype=torch.uint8, device=dev)
            buf[shift:] = torch.from_numpy(seq).to(dev)
            p2, nm, n_other = DeviceGenome.pack_ascii(buf[shift:])
            want_p2, want_nm = oracle.pack_genome(seq)
            got_p2 = p2.cpu().numpy().view(np.uint32)
            got_nm = nm.cpu().numpy().view(np.uint32)
            assert np.array_equal(got_p2[:len(want_p2)], want_p2), n
            assert np.all(got_p2[len(want_p2):] == 0)
            assert np.array_equal(got_nm[:len(want_nm)], want_nm), n
            assert int(n_other.item()) == int(np.isin(seq, np.frombuffer(b"RYx-", dtype=np.uint8)).sum())


def test_synth_genome_matches_oracle(dev, oracle):
    from digdriver_b200 import _lib
    for g0, n, seed, frac in ((0, 70001, 3, 16), (1 << 20, 1 << 21, 9, 16), (12345, 5000, 1, 0)):
        buf = torch.empty(n, dtype=torch.uint8, device=dev)
        _lib.call("dig_synth_genome", buf.data_ptr(), g0, n, seed, frac, torch.cuda.current_stream(dev).cuda_stream)
        want = oracle.synth_genome(g0, n, seed, frac)
        assert np.array_equal(buf.cpu().numpy(), want)
    assert 0.01 < (oracle.synth_genome(0, 1 << 22, 3) == ord("N")).mean() < 0.06


@pytest.mark.parametrize("u,d", [(1, 1), (2, 2), (0, 0), (1, 2), (2, 0)])
def test_scan_golden_bit_exact(gold_dev_genome, u, d):
    from digdriver_b200 import kernels
    z = golden("scan")
    w = z["windows"][z["rows_%d_%d" % (u, d)]]
    counts, totals = kernels.count_contexts(gold_dev_genome, w[:, 0] - 1, w[:, 1], w[:, 2], u, d, want_totals=True)
    got = counts.cpu().numpy().astype(np.int64)
    want = z["counts_%d_%d" % (u, d)]
    assert np.array_equal(got, want)
    assert np.array_equal(totals.cpu().numpy(), want.sum(axis=0))


def test_block_counts_strand_golden(gold_dev_genome):
    from digdriver_b200 import kernels
    z = golden("scan")
    counts, _ = kernels.count_contexts(gold_dev_genome, z["blk_chrom"] - 1, z["blk_start"], z["blk_end"], 1, 1,
                                       strand=z["blk_strand"])
    got = np.repeat(counts.cpu().numpy(), 3, axis=1).astype(np.float64)
    assert np.array_equal(got, z["blk_L192"])


@pytest.mark.parametrize("u,d", [(1, 1), (2, 2), (0, 0), (2, 1), (0, 3), (3, 2)])
def test_scan_random_regions_vs_oracle(dev, oracle, u, d):
    """Ragged, empty, chromosome-edge and both-strand regions against the C oracle."""
    from digdriver_b200 import kernels
    from digdriver_b200.genome import Genome, DeviceGenome
    rng = np.random.default_rng(100 + 10 * u + d)
    lens = [70001, 33, 5, 40000]
    seqs = []
    for L in lens:
        s = rng.choice(np.frombuffer(b"ACGTacgt", dtype=np.uint8), size=L)
        for _ in range(max(1, L // 9000)):
            a = int(rng.integers(0, L))
            s[a:a + int(rng.integers(1, 300))] = ord("N")
        seqs.append(s)
    g = Genome(["chr%d" % (i + 1) for i in range(len(lens))], seqs)
    dg = DeviceGenome.from_genome(g, dev)
    n = 600
    chrom = rng.integers(0, len(lens), n)
    L = np.array(lens)[chrom]
    start = (rng.random(n) * (L + 5)).astype(np.int64)
    ln = np.where(rng.random(n) < 0.2, rng.integers(0, 4, n), rng.integers(0, 9000, n))
    end = start + ln
    start[::17] = 0
    start = np.where((start > 0) & (start < u), u, start)      # the reference raises inside pysam there
    end = np.maximum(end, start)
    strand = np.where(rng.random(n) < 0.5, -1, 1).astype(np.int8)
    seq = np.full(dg.n_bases, ord("N"), dtype=np.uint8)
    for o, s in zip(dg.chrom_off, seqs):
        seq[o:o + len(s)] = s
    for st in (None, strand):
        counts, totals = kernels.count_contexts(dg, chrom, start, end, u, d, strand=st, want_totals=True)
        want, _ = oracle.count_regions(seq, dg.chrom_off, dg.chrom_len, chrom, start, end, u, d, strand=st)
        got = counts.cpu().numpy().astype(np.int64)
        bad = np.flatnonzero((got != want).any(axis=1))
        assert bad.size == 0, "regions %s differ (first: chrom %d %d-%d)" % (
            bad[:5], chrom[bad[0]], start[bad[0]], end[bad[0]])
        assert np.array_equal(totals.cpu().numpy(), want.sum(axis=0))


def test_scan_chr22_sized_vs_oracle(dev, oracle):
    """BASELINE config 1 scale: 51 Mb synthetic chromosome, 10 kb windows, both context sizes."""
    from digdriver_b200 import kernels
    from digdriver_b200.genome import DeviceGenome, tile_windows
    lengths = np.array([51_000_000], dtype=np.int64)
    dg = DeviceGenome.synthetic(["chr22"], lengths, seed=22, device=dev)
    wins = tile_windows([0], lengths, 10_000)
    assert len(wins) == 5099
    seq = oracle.synth_genome(0, int(lengths[0]), 22)
    for (u, d) in ((1, 1), (2, 2)):
        counts, totals = kernels.count_contexts(dg, wins[:, 0], wins[:, 1], wins[:, 2], u, d, want_totals=True)
        want, n_other = oracle.count_regions(seq, dg.chrom_off, lengths, wins[:, 0], wins[:, 1], wins[:, 2], u, d)
        assert n_other == 0
        assert np.array_equal(counts.cpu().numpy().astype(np.int64), want)
        assert np.array_equal(totals.cpu().numpy(), want.sum(axis=0))


@pytest.mark.parametrize("u", [0, 1, 2])
def test_scan_large_windows_totals_overflow_guard(dev, oracle, u):
    """1 Mb windows, and the guard that moves a CTA from int32 shared-memory totals to global
    uint64 atomics (forced here by lowering its threshold through the test hook)."""
    import ctypes
    from digdriver_b200 import kernels, _lib
    from digdriver_b200.genome import DeviceGenome, tile_windows
    lengths = np.array([9_000_001], dtype=np.int64)
    dg = DeviceGenome.synthetic(["chr1"], lengths, seed=4, device=dev, n_frac16=0)
    wins = np.concatenate([tile_windows([0], lengths, 1_000_000)] * 40)      # 320 regions > one wave of warps
    seq = oracle.synth_genome(0, int(lengths[0]), 4, 0)
    want, _ = oracle.count_regions(seq, dg.chrom_off, lengths, wins[:, 0], wins[:, 1], wins[:, 2], u, u)
    for limit in (0, 1500):                          # 0 = the library default
        # AUTO sends the 1 Mb regions of a (2,2) scan through the lane-bank kernel's redo list (regions > 32 kb)
        for variant in ((_lib.SCAN_AUTO, _lib.SCAN_HEX, _lib.SCAN_PER_BASE) if u == 2 else (_lib.SCAN_AUTO,)):
            counts, totals = kernels.count_contexts(dg, wins[:, 0], wins[:, 1], wins[:, 2], u, u, want_totals=True,
                                                    totals_limit_kb=limit, variant=variant)
            assert np.array_equal(counts.cpu().numpy().astype(np.int64), want), (limit, variant)
            assert np.array_equal(totals.cpu().numpy(), want.sum(axis=0)), (limit, variant)


def test_fused_penta_tri_scan_matches_two_scans(dev, oracle, gold_dev_genome):
    """dig_count_contexts_fused53: one pass giving both tables must equal the two separate scans bit for bit
    (golden windows incl. START == 0 / chromosome-end / tiny windows, random ragged regions with N runs,
    and a 51 Mb chromosome)."""
    from digdriver_b200 import kernels
    from digdriver_b200.genome import Genome, DeviceGenome, tile_windows
    z = golden("scan")
    w = z["windows"][z["rows_2_2"]]
    c5, c3, t5, t3 = kernels.count_contexts_fused53(gold_dev_genome, w[:, 0] - 1, w[:, 1], w[:, 2], want_totals=True)
    assert np.array_equal(c5.cpu().numpy(), z["counts_2_2"])
    rows3 = {tuple(r): i for i, r in enumerate(z["windows"][z["rows_1_1"]])}
    want3 = z["counts_1_1"][[rows3[tuple(r)] for r in w]]
    assert np.array_equal(c3.cpu().numpy(), want3)
    assert np.array_equal(t5.cpu().numpy(), z["counts_2_2"].sum(axis=0)) and np.array_equal(t3.cpu().numpy(), want3.sum(axis=0))
    # random regions on a genome with many short N runs and N exactly two bases from valid centres
    rng = np.random.default_rng(99)
    lens = [50_001, 64, 7, 33_000]
    seqs = []
    for L in lens:
        s = rng.choice(np.frombuffer(b"ACGTacgt", dtype=np.uint8), size=L)
        for _ in range(max(1, L // 400)):
            a = int(rng.integers(0, L))
            s[a:a + int(rng.integers(1, 4))] = ord("N")
        seqs.append(s)
    dg = DeviceGenome.from_genome(Genome(["c%d" % i for i in range(len(lens))], seqs), dev)
    n = 800
    chrom = rng.integers(0, len(lens), n)
    Lc = np.array(lens)[chrom]
    start = (rng.random(n) * (Lc + 3)).astype(np.int64)
    end = start + np.where(rng.random(n) < 0.3, rng.integers(0, 5, n), rng.integers(0, 4000, n))
    start[::13] = 0
    start = np.where((start > 0) & (start < 2), 2, start)
    end = np.maximum(end, start)
    c5, c3, t5, t3 = kernels.count_contexts_fused53(dg, chrom, start, end, want_totals=True)
    w5, _ = kernels.count_contexts(dg, chrom, start, end, 2, 2)
    w3, _ = kernels.count_contexts(dg, chrom, start, end, 1, 1)
    assert np.array_equal(c5.cpu().numpy(), w5.cpu().numpy())
    bad = np.flatnonzero((c3.cpu().numpy() != w3.cpu().numpy()).any(axis=1))
    assert bad.size == 0, (bad[:5], chrom[bad[:5]], start[bad[:5]], end[bad[:5]])
    assert np.array_equal(t3.cpu().numpy(), w3.cpu().numpy().astype(np.int64).sum(axis=0))
    # chr22-sized
    lengths = np.array([51_000_000], dtype=np.int64)
    dg = DeviceGenome.synthetic(["chr22"], lengths, seed=22, device=dev)
    wins = tile_windows([0], lengths, 10_000)
    c5, c3, t5, t3 = kernels.count_contexts_fused53(dg, wins[:, 0], wins[:, 1], wins[:, 2], want_totals=True)
    seq = oracle.synth_genome(0, int(lengths[0]), 22)
    want5, _ = oracle.count_regions(seq, dg.chrom_off, lengths, wins[:, 0], wins[:, 1], wins[:, 2], 2, 2)
    want3, _ = oracle.count_regions(seq, dg.chrom_off, lengths, wins[:, 0], wins[:, 1], wins[:, 2], 1, 1)
    assert np.array_equal(c5.cpu().numpy(), want5) and np.array_equal(c3.cpu().numpy(), want3)
    assert np.array_equal(t5.cpu().numpy(), want5.sum(axis=0)) and np.array_equal(t3.cpu().numpy(), want3.sum(axis=0))


def test_hexamer_pair_scan_adversarial_and_rejected_variants(dev, oracle):
    """scan_hex.cu counts pentanucleotides through hexamer pairs at even positions; this drives the parts
    that differ from the per-base kernels: pairs with a single valid centre (N every few bases, odd
    region boundaries, odd chromosome ends), 16-bit packed counters on homopolymers longer than one
    flush interval (98 304 bases), regions shorter than one pair, and the register totals.  The retired variants
    (variant 2, the per-base kernel of the fused scan) are rejected with DIG_ERR_ARG."""
    import ctypes
    from digdriver_b200 import kernels, _lib
    from digdriver_b200.genome import Genome, DeviceGenome
    rng = np.random.default_rng(2024)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    period6 = np.tile(np.frombuffer(b"AAAAAN", dtype=np.uint8), 5000)           # one valid 5-mer per 6 bases
    period7 = np.tile(np.frombuffer(b"ACGTACN", dtype=np.uint8), 4001)
    homo = np.full(300_007, ord("A"), dtype=np.uint8)                            # 3 flush intervals of one hexamer
    homo[150_000] = ord("N")
    mixed = rng.choice(acgt, size=250_003)
    mixed[rng.integers(0, mixed.size, 4000)] = ord("N")                          # isolated N: singles everywhere
    seqs = [period6, period7, homo, mixed, rng.choice(acgt, size=7)]
    dg = DeviceGenome.from_genome(Genome(["c%d" % i for i in range(len(seqs))], seqs), dev)
    lens = np.array([len(s) for s in seqs])
    n = 400
    chrom = rng.integers(0, len(seqs), n)
    start = (rng.random(n) * lens[chrom]).astype(np.int64)
    ln = np.where(rng.random(n) < 0.25, rng.integers(0, 8, n), rng.integers(0, 40_000, n))
    end = start + ln
    # whole chromosomes (multi-chunk regions), odd and even starts
    chrom = np.concatenate([chrom, np.arange(len(seqs)), [2, 2, 3, 3]])
    start = np.concatenate([start, np.zeros(len(seqs), dtype=np.int64), [1, 2, 3, 100_001]])
    end = np.concatenate([end, lens, [300_007, 300_006, 250_003, 250_002]])
    start = np.where((start > 0) & (start < 2), 2, start)
    end = np.maximum(end, start)
    seq = np.full(dg.n_bases, ord("N"), dtype=np.uint8)
    for o, s in zip(dg.chrom_off, seqs):
        seq[o:o + len(s)] = s
    want5, _ = oracle.count_regions(seq, dg.chrom_off, dg.chrom_len, chrom, start, end, 2, 2)
    want3, _ = oracle.count_regions(seq, dg.chrom_off, dg.chrom_len, chrom, start, end, 1, 1)
    # lane-bank kernel (+ its redo list: the homopolymer overflows 8-bit fields, long regions exceed its chunk
    # limit) and the per-warp hexamer kernel
    for variant in (_lib.SCAN_AUTO, _lib.SCAN_HEX):
        for limit in (0, 64):                        # 64 kb: the register totals spill to global many times
            kw = dict(variant=variant, totals_limit_kb=limit)
            c5, c3, t5, t3 = kernels.count_contexts_fused53(dg, chrom, start, end, want_totals=True, **kw)
            bad = np.flatnonzero((c5.cpu().numpy() != want5).any(axis=1))
            assert bad.size == 0, (variant, bad[:5], chrom[bad[:5]], start[bad[:5]], end[bad[:5]])
            bad = np.flatnonzero((c3.cpu().numpy() != want3).any(axis=1))
            assert bad.size == 0, (variant, bad[:5], chrom[bad[:5]], start[bad[:5]], end[bad[:5]])
            assert np.array_equal(t5.cpu().numpy(), want5.sum(axis=0)), variant
            assert np.array_equal(t3.cpu().numpy(), want3.sum(axis=0)), variant
            p5, pt = kernels.count_contexts(dg, chrom, start, end, 2, 2, want_totals=True, **kw)
            assert np.array_equal(p5.cpu().numpy(), want5) and np.array_equal(pt.cpu().numpy(), want5.sum(axis=0))
            q5, _ = kernels.count_contexts(dg, chrom, start, end, 2, 2, **kw)
            assert np.array_equal(q5.cpu().numpy(), want5)
    # the per-base kernels stay available and agree; the fused scan has none, and 2 names no variant
    p5, _ = kernels.count_contexts(dg, chrom, start, end, 2, 2, variant=_lib.SCAN_PER_BASE)
    assert np.array_equal(p5.cpu().numpy(), want5)
    for variant in (_lib.SCAN_PER_BASE, 2):
        with pytest.raises(_lib.DigError):
            kernels.count_contexts_fused53(dg, chrom, start, end, variant=variant)
    with pytest.raises(_lib.DigError):
        kernels.count_contexts(dg, chrom, start, end, 2, 2, variant=2)
    # trinucleotide-only lane-bank kernel (4-mer pairs): it takes over from 64 regions per SM, so the same adversarial
    # set is repeated (and shuffled, so that every batch of 32 mixes chromosomes, lengths and parities); whole
    # chromosomes of 300 kb run through ~150 chunks per lane while their batch neighbours have one
    reps = 64 * 160 // len(chrom) + 1
    order = np.random.default_rng(7).permutation(reps * len(chrom))
    big_c, big_s, big_e = (np.tile(a, reps)[order] for a in (chrom, start, end))
    want_big = np.tile(want3, (reps, 1))[order]
    for limit in (0, 64):
        k3, kt = kernels.count_contexts(dg, big_c, big_s, big_e, 1, 1, want_totals=True, totals_limit_kb=limit)
        bad = np.flatnonzero((k3.cpu().numpy() != want_big).any(axis=1))
        assert bad.size == 0, (limit, bad[:5], big_c[bad[:5]], big_s[bad[:5]], big_e[bad[:5]])
        assert np.array_equal(kt.cpu().numpy(), want_big.astype(np.int64).sum(axis=0)), limit
    k3b, _ = kernels.count_contexts(dg, big_c, big_s, big_e, 1, 1, variant=_lib.SCAN_PER_BASE)
    assert np.array_equal(k3b.cpu().numpy(), want_big)
    # the same shuffled set through the FUSED lane-bank kernel, four times over: every CTA then works through several
    # consecutive batches whose chunk counts differ (0 to 16 chunks, long regions on the redo list), which is what the
    # four-slot staging ring (slot kq % 4, the fourth slot aliased onto the slice buffers, one fill parity per slot) and
    # its hand-offs across batch boundaries have to survive; twice, with and without register-total spills
    reps5 = 4 * reps
    order5 = np.random.default_rng(11).permutation(reps5 * len(chrom))
    f_c, f_s, f_e = (np.tile(a, reps5)[order5] for a in (chrom, start, end))
    want_f5, want_f3 = np.tile(want5, (reps5, 1))[order5], np.tile(want3, (reps5, 1))[order5]
    for limit in (0, 64):
        c5, c3, t5, t3 = kernels.count_contexts_fused53(dg, f_c, f_s, f_e, want_totals=True, totals_limit_kb=limit)
        bad = np.flatnonzero((c5.cpu().numpy() != want_f5).any(axis=1))
        assert bad.size == 0, (limit, bad[:5], f_c[bad[:5]], f_s[bad[:5]], f_e[bad[:5]])
        bad = np.flatnonzero((c3.cpu().numpy() != want_f3).any(axis=1))
        assert bad.size == 0, (limit, bad[:5], f_c[bad[:5]], f_s[bad[:5]], f_e[bad[:5]])
        assert np.array_equal(t5.cpu().numpy(), want_f5.astype(np.int64).sum(axis=0)), limit
        assert np.array_equal(t3.cpu().numpy(), want_f3.astype(np.int64).sum(axis=0)), limit
        p5, _ = kernels.count_contexts(dg, f_c, f_s, f_e, 2, 2, totals_limit_kb=limit)       # K = 1024 alone (TRI = 0)
        assert np.array_equal(p5.cpu().numpy(), want_f5), limit


def test_empty_inputs_through_the_c_abi(dev):
    """Zero regions / mutations / elements / p-values: every entry point returns cleanly with empty (or zeroed)
    outputs instead of launching an empty grid or touching a null pointer."""
    from digdriver_b200 import kernels
    from digdriver_b200.genome import Genome, DeviceGenome
    dg = DeviceGenome.from_genome(Genome(["chr1"], [np.frombuffer(b"ACGTNACGTACGTTTGACA" * 20, dtype=np.uint8)]), dev)
    e32, e64 = np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.int64)
    for (u, d) in ((1, 1), (2, 2), (0, 3)):
        c, t = kernels.count_contexts(dg, e32, e64, e64, u, d, want_totals=True)
        assert c.shape == (0, 4 ** (u + d + 1)) and int(t.sum()) == 0
    c5, c3, t5, t3 = kernels.count_contexts_fused53(dg, e32, e64, e64, want_totals=True)
    assert c5.shape == (0, 1024) and c3.shape == (0, 64) and int(t5.sum()) == 0 and int(t3.sum()) == 0
    # regions that contain no centre at all (length 0, beyond the chromosome end) give zero rows
    c5, c3, _, _ = kernels.count_contexts_fused53(dg, [0, 0, 0], [5, 380, 1000], [5, 380, 2000])
    assert int(c5.sum()) == 0 and int(c3.sum()) == 0
    assert kernels.mutation_contexts(dg, e32, e64, np.zeros(0, dtype=np.uint8), 1, 1).numel() == 0
    assert int(kernels.substitution_counts(torch.zeros(0, dtype=torch.int32, device=dev), np.zeros(0, dtype=np.uint8), 1, 1).sum()) == 0
    f = np.zeros(0)
    assert kernels.nb_pvalue_greater_midp(f, f, f, dev).numel() == 0
    assert kernels.nb_pvalue_exact(f, f, f, dev).numel() == 0
    exp, pv = kernels.nb_burden_test(f, f, f, f, dev)
    assert exp.numel() == 0 and pv.numel() == 0
    obs, nsamp = kernels.tabulate_genes(e32, e32, np.zeros(0, dtype=np.uint8), 7, device=dev)
    assert obs.shape == (7, 5) and int(obs.sum()) == 0 and int(nsamp.sum()) == 0
    obs, stot = kernels.tabulate_elements(np.array([10], dtype=np.int64), np.array([20], dtype=np.int64), [0], e64, e64,
                                          e32, np.zeros(0, dtype=np.uint8), 1, 3, device=dev)
    assert obs.shape == (1, 3) and int(obs.sum()) == 0 and int(stot.sum()) == 0
    out = kernels.position_test(dg, e32, e64, e64, f, f, np.ones(1024), e32, e64, 2, 2, 1)
    assert out["pval"].numel() == 0 and out["obs"].numel() == 0
    out = kernels.position_test(dg, [0], [0], [40], [3.0], [1.0], np.ones(64), e32, e64, 1, 1, 7)
    assert out["pval"].numel() == 6 and int(out["obs"].sum()) == 0           # 39 positions in bins of 7
    assert kernels.gene_dnds_sel(f, f, np.zeros((0, 6)), np.zeros((0, 6)), dev).shape == (24, 0)


def test_fused_exchange_stores_rows_into_every_peer_buffer(dev):
    """dig_scan_opts.peer_counts3_d (the all-gather fused into the scan for range-sharded runs): with peers given the
    trinucleotide rows go to the same offsets of EVERY peer buffer instead of the local pointer -- here the "peers" are
    two more buffers of this GPU, which exercises the per-peer store path of both lane-bank kernels (the multicast
    path needs NVSwitch symmetric memory and is covered by bench.py's parity sample under torchrun) -- and
    dig_peer_broadcast copies the totals block after them."""
    from digdriver_b200 import kernels
    from digdriver_b200.genome import DeviceGenome, tile_windows
    lengths = np.array([1_500_000, 700_001], dtype=np.int64)
    dg = DeviceGenome.synthetic(["a", "b"], lengths, seed=21, device=dev)
    base = tile_windows(np.arange(2), lengths, 10_000)
    wins = np.concatenate([base] * (64 * 160 // len(base) + 1))          # enough regions for the trinucleotide-only kernel
    n = len(wins)
    want5, want3, _, _ = kernels.count_contexts_fused53(dg, wins[:, 0], wins[:, 1], wins[:, 2])
    bufs = [torch.full((n, 64), -7, dtype=torch.int32, device=dev) for _ in range(3)]
    local = torch.full((n, 64), -7, dtype=torch.int32, device=dev)
    got5, _, _, _ = kernels.count_contexts_fused53(dg, wins[:, 0], wins[:, 1], wins[:, 2], out3=local,
                                                   peer_rows=[b.data_ptr() for b in bufs])
    torch.cuda.synchronize()
    assert torch.equal(got5, want5)
    assert all(torch.equal(b, want3) for b in bufs)
    assert bool((local == -7).all())                                      # the local pointer is not written in this mode
    for b in bufs:
        b.fill_(-7)
    kernels.count_contexts(dg, wins[:, 0], wins[:, 1], wins[:, 2], 1, 1, out=local, peer_rows=[b.data_ptr() for b in bufs[:2]])
    torch.cuda.synchronize()
    assert torch.equal(bufs[0], want3) and torch.equal(bufs[1], want3) and bool((bufs[2] == -7).all())
    # too few regions for the lane-bank kernel: the request must be refused, not silently ignored
    from digdriver_b200._lib import DigError
    with pytest.raises(DigError):
        kernels.count_contexts(dg, base[:, 0], base[:, 1], base[:, 2], 1, 1, peer_rows=[bufs[0].data_ptr()])
    src = torch.arange(4096, dtype=torch.int32, device=dev)
    dst = [torch.zeros(4096, dtype=torch.int32, device=dev) for _ in range(3)]
    kernels.peer_broadcast(src[16:2064], [d[16:2064].data_ptr() for d in dst])
    torch.cuda.synchronize()
    for d in dst:
        assert torch.equal(d[16:2064], src[16:2064]) and int(d[:16].sum()) == 0 and int(d[2064:].sum()) == 0
