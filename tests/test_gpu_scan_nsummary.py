"""The per-128-base N summary (dig_nmask_summary) and the lane-bank scan that stages bases only when it has one.

The summary is checked against a NumPy definition; the lane-bank scan, which runs only with the summary, against the
same call without it (nsum_offset_words = 0: the per-warp kernels run) and against the CPU oracle, on N layouts chosen to
hit every case of the span-state rule: N runs starting and ending at every offset mod 128, single N in the four halo
bases of the next block, windows inside N runs, N lead-ins, chromosome ends."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _nsum_ref(words):
    """Two bits per block of four mask words: bit 0 = any N, bit 1 = all N; missing tail words count as N."""
    w = np.asarray(words, dtype=np.uint32)
    nb = (len(w) + 3) // 4
    pad = np.full(nb * 4, 0xFFFFFFFF, dtype=np.uint32)
    pad[:len(w)] = w
    blk = pad.reshape(nb, 4)
    st = (blk != 0).any(axis=1).astype(np.uint64) | ((blk == 0xFFFFFFFF).all(axis=1).astype(np.uint64) << 1)
    return st


def _unpack_nsum(nsum, nb):
    v = nsum.cpu().numpy().view(np.uint32).astype(np.uint64)
    j = np.arange(nb)
    return (v[j >> 4] >> (2 * (j & 15)).astype(np.uint64)) & 3


def test_nmask_summary_matches_numpy():
    from digdriver_b200 import _lib
    rng = np.random.default_rng(3)
    st = torch.cuda.current_stream().cuda_stream
    for n_words in (1, 4, 5, 63, 64, 65, 127, 1000, 4099, 50_000):
        kinds = rng.integers(0, 4, n_words)
        w = np.where(kinds == 0, 0, np.where(kinds == 1, 0xFFFFFFFF, np.where(kinds == 2, 1 << rng.integers(0, 32, n_words),
                                                                               rng.integers(0, 1 << 32, n_words))))
        # long clean / all-N stretches, so that whole blocks are clean or all N
        for _ in range(max(1, n_words // 40)):
            a = int(rng.integers(0, n_words))
            w[a:a + int(rng.integers(1, 40))] = rng.choice([0, 0xFFFFFFFF])
        w = w.astype(np.uint32)
        nm = torch.from_numpy(w.view(np.int32).copy()).cuda()
        nb = (n_words + 3) // 4
        nsum = torch.full(((nb + 15) // 16,), -1, dtype=torch.int32, device="cuda")
        _lib.call("dig_nmask_summary", nm.data_ptr(), 0, n_words, nsum.data_ptr(), st)
        assert np.array_equal(_unpack_nsum(nsum, nb), _nsum_ref(w)), n_words
        # rebuild of a sub-range (word0 a multiple of 4, any length): only its blocks change
        for word0 in (0, 4, 60, 64, 68):
            if word0 >= n_words:
                continue
            cnt = int(rng.integers(1, n_words - word0 + 1))
            w2 = w.copy()
            w2[word0:word0 + cnt] = rng.integers(0, 1 << 32, cnt, dtype=np.uint64).astype(np.uint32) * (rng.random(cnt) < 0.3)
            nm.copy_(torch.from_numpy(w2.view(np.int32).copy()))
            before = _unpack_nsum(nsum, nb)
            _lib.call("dig_nmask_summary", nm.data_ptr(), word0, cnt, nsum.data_ptr(), st)
            got = _unpack_nsum(nsum, nb)
            b0, b1 = word0 // 4, (word0 + cnt + 3) // 4
            want = before.copy()
            want[b0:b1] = _nsum_ref(w2[word0:word0 + cnt])
            assert np.array_equal(got, want), (n_words, word0, cnt)
            w = w2
        # blocks of the last summary word past the mask keep their all-N bits
        tail = nsum.cpu().numpy().view(np.uint32)[-1]
        if nb % 16:
            assert tail >> (2 * (nb % 16)) == 0xFFFFFFFF >> (2 * (nb % 16))
    with pytest.raises(_lib.DigError):
        _lib.call("dig_nmask_summary", nm.data_ptr(), 2, 8, nsum.data_ptr(), st)


def _adversarial_genome(lengths, W, seed):
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = [acgt[rng.integers(0, 4, int(n))] for n in lengths]
    s0 = seqs[0]
    # N runs starting at every offset mod 128 and ending at every offset mod 128, one per window region
    for o in range(128):
        o2 = (37 * o + 11) % 128
        start = 4096 + o * 3000 + (o * 128) % 2048 // 128 * 128 + o
        ln = 128 * int(rng.integers(0, 4)) + (o2 - o) % 128 + 1
        s0[start:start + ln] = ord("N")
    # single N in the first four bases of a block (the halo of the span before it), and at the span's last bases
    for j, t in enumerate((0, 1, 2, 3, 127, 126, 4, 5) * 16):
        p = 400_000 + 2_000 * j + 128 * (j % 7) + t
        if p < len(s0):
            s0[p] = ord("N")
    # N just before window starts (lead-ins), one and a few bases long
    for i in range(10, 40):
        s0[i * W - 1 - (i % 5): i * W] = ord("N")
    s1 = seqs[1]
    s1[:300] = ord("N")                                  # chromosome start in N
    s1[50_000:50_000 + 3 * W + 777] = ord("N")           # windows fully inside an N run
    s1[200_003:251_000] = ord("N")
    seqs[2][-5000:] = ord("N")                           # chromosome end in N
    seqs[2][100_000:100_000 + 2 * W] = ord("N")
    s1[-3:] = ord("N")
    return seqs


@pytest.fixture(scope="module")
def adv(oracle):
    from digdriver_b200.genome import DeviceGenome, Genome, tile_windows
    lengths = np.array([17_000_123, 13_500_077, 9_800_001], dtype=np.int64)
    W = 4096
    seqs = _adversarial_genome(lengths, W, 17)
    g = Genome(["chr1", "chr2", "chr3"], seqs)
    dg = DeviceGenome.from_genome(g, "cuda:0")
    seq = np.full(dg.n_bases, ord("N"), dtype=np.uint8)
    for o, s in zip(dg.chrom_off, seqs):
        seq[int(o):int(o) + len(s)] = s
    wins = tile_windows(np.arange(3), lengths, W)
    rng = np.random.default_rng(5)
    n = 12_000
    c = rng.integers(0, 3, n)
    st = (rng.random(n) * lengths[c]).astype(np.int64)
    st[:50] = 0                                          # START == 0
    en = st + rng.integers(1, 6000, n)
    en[50:100] = lengths[c[50:100]] + 7                  # past the chromosome end
    st[100:150] = np.maximum(lengths[c[100:150]] - rng.integers(1, 300, 50), 2)
    en[100:150] = lengths[c[100:150]]
    st = np.where((st > 0) & (st < 2), 2, st)
    return dg, seq, wins, (c, st, en)


def _both(dg, fn):
    """fn() with the genome's summary (lane-bank kernel) and without it (per-warp kernels)."""
    nsum = dg.nsum
    try:
        with_sum = fn()
        dg.nsum = None
        without = fn()
    finally:
        dg.nsum = nsum
    return with_sum, without


def test_summary_marks_the_layout(adv):
    dg, seq, _, _ = adv
    nb = dg.n_bases // 128
    blk = (seq[:nb * 128].reshape(nb, 128) == ord("N"))
    want = blk.any(axis=1).astype(np.uint64) | (blk.all(axis=1).astype(np.uint64) << 1)
    got = _unpack_nsum(dg.nsum, nb)
    assert np.array_equal(got, want)
    assert (got == 1).sum() > 300 and (got == 3).sum() > 300 and (got == 0).sum() > nb // 2


@pytest.mark.parametrize("which", ["tiled", "ragged"])
def test_fused_scan_with_summary_matches_mask_staging_and_oracle(adv, oracle, which):
    from digdriver_b200 import kernels
    dg, seq, wins, rag = adv
    c, s, e = (wins[:, 0], wins[:, 1], wins[:, 2]) if which == "tiled" else rag
    (a5, a3, at5, at3), (b5, b3, bt5, bt3) = _both(
        dg, lambda: tuple(t.cpu().numpy() for t in kernels.count_contexts_fused53(dg, c, s, e, want_totals=True)))
    assert np.array_equal(a5, b5) and np.array_equal(a3, b3)
    assert np.array_equal(at5, bt5) and np.array_equal(at3, bt3)
    want5, _ = oracle.count_regions(seq, dg.chrom_off, dg.chrom_len, c, s, e, 2, 2)
    want3, _ = oracle.count_regions(seq, dg.chrom_off, dg.chrom_len, c, s, e, 1, 1)
    assert np.array_equal(a5, want5) and np.array_equal(a3, want3)
    assert np.array_equal(at5, want5.sum(axis=0)) and np.array_equal(at3, want3.sum(axis=0))


@pytest.mark.parametrize("which", ["tiled", "ragged"])
def test_tri_scan_with_summary_matches_mask_staging_and_oracle(adv, oracle, which):
    from digdriver_b200 import _lib, kernels
    dg, seq, wins, rag = adv
    c, s, e = (wins[:, 0], wins[:, 1], wins[:, 2]) if which == "tiled" else rag
    assert len(c) >= 64 * int(_lib.load().dig_device_sm_count())      # the trinucleotide lane-bank kernel's threshold
    (a, at), (b, bt) = _both(dg, lambda: tuple(t.cpu().numpy() for t in kernels.count_contexts(dg, c, s, e, 1, 1,
                                                                                              want_totals=True)))
    assert np.array_equal(a, b) and np.array_equal(at, bt)
    want, _ = oracle.count_regions(seq, dg.chrom_off, dg.chrom_len, c, s, e, 1, 1)
    assert np.array_equal(a, want) and np.array_equal(at, want.sum(axis=0))


def test_penta_scan_with_summary_matches_mask_staging(adv):
    from digdriver_b200 import kernels
    dg, _, wins, _ = adv
    (a, at), (b, bt) = _both(dg, lambda: tuple(t.cpu().numpy() for t in kernels.count_contexts(
        dg, wins[:, 0], wins[:, 1], wins[:, 2], 2, 2, want_totals=True)))
    assert np.array_equal(a, b) and np.array_equal(at, bt)


def test_host_scan_rebuilds_the_summary_per_chromosome(oracle):
    """HostScan rewrites the mask chromosome by chromosome (copy, runs or pack); each chromosome's summary must follow."""
    from digdriver_b200 import host_pipeline as hp, kernels
    from digdriver_b200.genome import DeviceGenome, Genome, tile_windows
    lengths = np.array([310_000, 250_001, 180_077], dtype=np.int64)
    W = 10_000
    seqs = _adversarial_genome(lengths, W, 23)
    seqs[0][120_000:170_000] = ord("N")                  # every chromosome has its own layout
    seqs[2][:70_000] = ord("N")
    g = Genome(["chr1", "chr2", "chr3"], seqs)
    wins = tile_windows(np.arange(3), lengths, W)
    dg = DeviceGenome.from_genome(g, "cuda:0")
    want5, want3, wt5, wt3 = (t.cpu().numpy() for t in
                              kernels.count_contexts_fused53(dg, wins[:, 0], wins[:, 1], wins[:, 2], want_totals=True))
    hg = hp.HostGenome.from_genome(g)                                   # ASCII: packed on the device per chromosome
    hs = hp.HostScan(hg, wins, "cuda:0").run()
    assert torch.equal(hs.genome.nsum, dg.nsum)
    hg2 = hp.HostGenome.from_device(hs.genome)                          # packed, N mask as runs
    perm = np.concatenate([np.flatnonzero(wins[:, 0] == 2), np.flatnonzero(wins[:, 0] == 0),
                           np.flatnonzero(wins[:, 0] == 1)])
    for h, order in ((hs, np.arange(len(wins))), (hp.HostScan(hg2, wins, "cuda:0").run(), np.arange(len(wins))),
                     (hp.HostScan(hg2, wins[perm], "cuda:0").run(), perm)):
        assert np.array_equal(h.host_counts.numpy().astype(np.int64), want5[order])
        assert np.array_equal(h.host_counts3.numpy().astype(np.int64), want3[order])
        assert np.array_equal(h.host_totals.numpy(), np.concatenate([wt5, wt3]))
    seq = np.full(dg.n_bases, ord("N"), dtype=np.uint8)
    for o, s in zip(dg.chrom_off, seqs):
        seq[int(o):int(o) + len(s)] = s
    oc, _ = oracle.count_regions(seq, dg.chrom_off, lengths, wins[:, 0], wins[:, 1], wins[:, 2], 2, 2)
    assert np.array_equal(want5, oc)
