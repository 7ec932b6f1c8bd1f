"""countGenomeContext from HOST memory to HOST memory (reference scripts/DigPreprocess.py:19-73).

The reference reads the FASTA window by window in a multiprocessing.Pool (sequence_tools.py:96-128) and gathers the
rows with pd.concat.  Here the genome sits in pinned host memory -- as ASCII, or as the packed cache written next to
the FASTA (2-bit bases + the N mask in run-length form, 0.25 B/base: a quarter of the bytes over PCIe) -- and goes through
the device once,
chromosome by chromosome, on three streams:

    copy stream :  H2D of chromosome c+1
    main stream :  K1 pack (ASCII sources only) -> K2 fused scan of chromosome c's windows -> narrow to uint16
    out stream  :  D2H of the count rows of chromosome c-1

The device genome stays resident for the stages that follow (mutation contexts, element transfer).  Count rows are
shipped as uint16 whenever every region is shorter than 65536 bases (a region holds at most its length in centres, so
no count can exceed it); the narrowing kernel double-checks and the int32 rows are shipped instead if it objects.

PackedGenomeCache: `<fasta>.dig2bit/` holds the packed bases and the mask runs keyed on the FASTA's path, size and mtime, so
that a second run neither parses nor packs nor uploads ASCII.
"""
import json
import os

import numpy as np
import torch

from . import _lib, kernels
from .genome import DeviceGenome, Genome, _layout, alloc_nmask

CACHE_VERSION = 2


def mask_runs_of(nmask_words, chrom_off, n_bases):
    """Run-length form of the N mask: int64 [n, 3] rows (first word, number of words, 32-bit word value) over the non-zero
    words, split at chromosome boundaries so that a chromosome's runs can be written on their own.  A genome has a few
    hundred to a few thousand N runs (hg19: 3 % of the bases), so this replaces 1/3 of the packed bytes by ~100 KB."""
    w = np.ascontiguousarray(nmask_words).view(np.uint32).reshape(-1)
    idx = np.flatnonzero(w)
    if idx.size == 0:
        return np.zeros((0, 3), dtype=np.int64)
    val = w[idx]
    bounds = (np.asarray(chrom_off, dtype=np.int64) // 32)                # first mask word of every chromosome
    chrom_of = np.searchsorted(bounds, idx, side="right")
    brk = np.ones(idx.size, dtype=bool)
    brk[1:] = (idx[1:] != idx[:-1] + 1) | (val[1:] != val[:-1]) | (chrom_of[1:] != chrom_of[:-1])
    first = np.flatnonzero(brk)
    count = np.diff(np.append(first, idx.size))
    return np.stack([idx[first].astype(np.int64), count.astype(np.int64), val[first].astype(np.int64)], axis=1)



def _pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype, pin_memory=True)


class HostGenome:
    """A genome in pinned host memory in the device layout (chromosomes concatenated, each starting at a multiple of
    128 bases): either `ascii` (uint8 [n_bases], padding = 'N') or `packed2` + `nmask` (int32 words)."""

    def __init__(self, names, chrom_len, ascii=None, packed2=None, nmask=None, n_other=0, mask_runs=None):
        self.names = list(names)
        self.chrom_len = np.asarray(chrom_len, dtype=np.int64)
        self.chrom_off, self.n_bases = _layout(self.chrom_len)
        self.ascii, self.packed2, self.nmask = ascii, packed2, nmask
        # packed sources carry the N mask as words (nmask) or in run-length form (mask_runs, pinned int64 [n, 3])
        self.mask_runs = mask_runs
        self.n_other = int(n_other)
        assert (ascii is not None) != (packed2 is not None and (nmask is not None or mask_runs is not None)), \
            "either ASCII or packed arrays (with the N mask as words or as runs)"

    @property
    def is_packed(self):
        return self.packed2 is not None

    @property
    def nbytes(self):
        if self.is_packed:
            mask = self.nmask.numel() * 4 if self.nmask is not None else self.mask_runs.numel() * 8
            return self.packed2.numel() * 4 + mask
        return self.ascii.numel()

    @classmethod
    def from_genome(cls, genome):
        """Pinned ASCII copy of a host Genome (FASTA contents)."""
        lengths = genome.lengths
        off, total = _layout(lengths)
        buf = _pinned((max(total, 1),), torch.uint8)
        view = buf.numpy()
        view[:] = ord("N")
        for o, s in zip(off, genome.seqs):
            view[int(o):int(o) + len(s)] = s
        return cls(genome.names, lengths, ascii=buf[:total])

    @classmethod
    def from_device(cls, dg, ascii_d=None, rle_mask=True):
        """Pinned copy of a DeviceGenome: the packed bases + the N mask in run-length form (rle_mask=False: as words), or
        (ascii_d given) the ASCII it was packed from."""
        if ascii_d is not None:
            buf = _pinned((ascii_d.numel(),), torch.uint8)
            buf.copy_(ascii_d)
            return cls(dg.names, dg.chrom_len, ascii=buf, n_other=dg.n_other)
        p2 = _pinned((dg.packed2.numel(),), torch.int32)
        p2.copy_(dg.packed2)
        if not rle_mask:
            nm = _pinned((dg.nmask.numel(),), torch.int32)
            nm.copy_(dg.nmask)
            return cls(dg.names, dg.chrom_len, packed2=p2, nmask=nm, n_other=dg.n_other)
        runs = mask_runs_of(dg.nmask.cpu().numpy(), dg.chrom_off, dg.n_bases)
        return cls(dg.names, dg.chrom_len, packed2=p2, mask_runs=torch.from_numpy(runs).pin_memory(), n_other=dg.n_other)


# ------------------------------------------------------------------------------------------------
# packed-genome cache next to the FASTA
# ------------------------------------------------------------------------------------------------

class PackedGenomeCache:
    """`<fasta>.dig2bit/{meta.json, packed2.bin, nmask_runs.npy}`; valid while the FASTA's size and mtime are unchanged."""

    @staticmethod
    def cache_dir(fasta_path, cache_dir=None):
        return cache_dir or (os.path.abspath(str(fasta_path)) + ".dig2bit")

    @staticmethod
    def _key(fasta_path):
        st = os.stat(fasta_path)
        return {"path": os.path.abspath(str(fasta_path)), "size": int(st.st_size), "mtime_ns": int(st.st_mtime_ns),
                "version": CACHE_VERSION}

    @classmethod
    def load(cls, fasta_path, cache_dir=None):
        """HostGenome (packed, pinned) if a valid cache exists, else None."""
        d = cls.cache_dir(fasta_path, cache_dir)
        meta_p = os.path.join(d, "meta.json")
        if not os.path.exists(meta_p):
            return None
        try:
            meta = json.load(open(meta_p))
            if meta.get("key") != cls._key(fasta_path):
                return None
            n2 = int(meta["packed2_words"])
            p2 = _pinned((n2,), torch.int32)
            path = os.path.join(d, "packed2.bin")
            if os.path.getsize(path) != 4 * n2:
                return None
            with open(path, "rb") as f:
                got = f.readinto(memoryview(p2.numpy()).cast("B"))
            if got != 4 * n2:
                return None
            runs = np.load(os.path.join(d, "nmask_runs.npy"))
            if runs.ndim != 2 or runs.shape[1] != 3 or runs.shape[0] != int(meta["n_mask_runs"]):
                return None
            return HostGenome(meta["names"], meta["chrom_len"], packed2=p2,
                              mask_runs=torch.from_numpy(np.ascontiguousarray(runs, dtype=np.int64)).pin_memory(),
                              n_other=meta["n_other"])
        except (OSError, ValueError, KeyError):
            return None

    @classmethod
    def store(cls, fasta_path, dg, cache_dir=None):
        """Write the packed arrays of `dg` (packed from this FASTA).  Best effort: a read-only directory is not an error."""
        d = cls.cache_dir(fasta_path, cache_dir)
        try:
            os.makedirs(d, exist_ok=True)
            p2 = dg.packed2.cpu().numpy()
            runs = mask_runs_of(dg.nmask.cpu().numpy(), dg.chrom_off, dg.n_bases)
            p2.tofile(os.path.join(d, "packed2.bin"))
            np.save(os.path.join(d, "nmask_runs.npy"), runs)
            meta = {"key": cls._key(fasta_path), "names": list(dg.names), "chrom_len": [int(x) for x in dg.chrom_len],
                    "n_other": int(dg.n_other), "packed2_words": int(p2.size), "n_mask_runs": int(runs.shape[0])}
            tmp = os.path.join(d, "meta.json.tmp")
            json.dump(meta, open(tmp, "w"))
            os.replace(tmp, os.path.join(d, "meta.json"))          # the meta file appears last: a torn cache is invalid
            return d
        except OSError:
            return None


def host_genome_from_fasta(fasta_path, use_cache=True, cache_dir=None):
    """(HostGenome, from_cache): the packed cache when valid, else the parsed FASTA as pinned ASCII."""
    if use_cache:
        hg = PackedGenomeCache.load(fasta_path, cache_dir)
        if hg is not None:
            return hg, True
    return HostGenome.from_genome(Genome.from_fasta(fasta_path)), False


# ------------------------------------------------------------------------------------------------
# the pipelined scan
# ------------------------------------------------------------------------------------------------

class HostScan:
    """Pipelined host -> device -> host context scan of a fixed window list.

    windows: int64 [Nw, 3] (chromosome index, start, end), grouped by chromosome in ascending order.
    tables : "penta+tri" (fused pentanucleotide + trinucleotide scan), or an (n_up, n_down) pair.
    All device and pinned buffers are allocated once; run() can be called repeatedly (bench.py's e2e leg)."""

    def __init__(self, host_genome, windows, device, tables="penta+tri", narrow="auto", tile_window=None,
                 upload_all=True):
        self.hg = host_genome
        self.device = torch.device(device)
        dev = self.device
        w = np.ascontiguousarray(windows, dtype=np.int64)
        assert w.ndim == 2 and w.shape[1] == 3
        self.windows = w
        self.n_win = len(w)
        self.fused = tables == "penta+tri"
        self.n_up, self.n_down = (2, 2) if self.fused else (int(tables[0]), int(tables[1]))
        self.K = 4 ** (self.n_up + self.n_down + 1)
        n_chrom = len(host_genome.names)
        # chromosomes are processed in the order their windows appear (one run of rows each); the rest afterwards
        cuts = np.flatnonzero(np.diff(w[:, 0])) + 1 if len(w) else np.zeros(0, dtype=np.int64)
        los = np.concatenate([[0], cuts]).astype(np.int64) if len(w) else np.zeros(0, dtype=np.int64)
        his = np.concatenate([cuts, [len(w)]]).astype(np.int64) if len(w) else np.zeros(0, dtype=np.int64)
        run_chrom = w[los, 0] if len(w) else np.zeros(0, dtype=np.int64)
        if len(set(run_chrom.tolist())) != len(run_chrom):
            raise ValueError("windows must be grouped by chromosome")
        if len(w) and (w[:, 0].min() < 0 or w[:, 0].max() >= n_chrom):
            raise KeyError("window on a chromosome that is not in the genome")
        # upload_all=False: chromosomes without windows stay on the host (a range-sharded rank needs only its own)
        self.order = [(int(c), int(a), int(b)) for c, a, b in zip(run_chrom, los, his)] + \
                     ([(c, 0, 0) for c in range(n_chrom) if c not in set(run_chrom.tolist())] if upload_all else [])
        self.wlo, self.whi = los, his
        longest = int((w[:, 2] - w[:, 1]).max()) if len(w) else 0
        self.narrow = (longest < 65536) if narrow == "auto" else bool(narrow)
        if self.K < 8:
            self.narrow = False                # rows shorter than 16 bytes: nothing to gain, and row slices lose alignment
        if tile_window is None and len(w):
            tw = int(w[0, 2] - w[0, 1])
            tile_window = tw if tw > 0 and bool(np.all(w[:, 2] - w[:, 1] == tw)) else 0
        self.tile_window = int(tile_window or 0)
        hg = host_genome
        n = hg.n_bases
        lib = _lib.load()
        # device: the packed genome (kept), the ASCII landing buffer (ASCII sources), the count tables
        self.packed2 = torch.empty(max(int(lib.dig_packed_words(n)), 2), dtype=torch.int32, device=dev)
        self.nmask = alloc_nmask(max(int(lib.dig_nmask_words(n)), 1), dev)       # with room for its N summary
        self.n_other_d = torch.zeros(1, dtype=torch.int64, device=dev)
        self.dev_ascii = None if hg.is_packed else torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
        self.runs_d, self.run_lo = None, None
        if hg.is_packed and hg.nmask is None:
            # run-length mask: the (small) run table goes up once per pass, each chromosome's share is expanded on the
            # device right before its scan (dig_nmask_fill_runs)
            runs = hg.mask_runs.numpy()
            self.runs_d = torch.empty((max(len(runs), 1), 3), dtype=torch.int64, device=dev)
            word_off = np.append(hg.chrom_off // 32, (n + 31) // 32)
            self.run_lo = np.searchsorted(runs[:, 0], word_off, side="left") if len(runs) else np.zeros(len(word_off), dtype=np.int64)
            self.word_off = word_off
        self.genome = DeviceGenome(hg.names, hg.chrom_len, hg.chrom_off, n, self.packed2, self.nmask, hg.n_other, dev,
                                   build_nsum=False)
        self.win_chrom = torch.from_numpy(w[:, 0].astype(np.int32)).to(dev)
        self.win_start = torch.from_numpy(np.ascontiguousarray(w[:, 1])).to(dev)
        self.win_end = torch.from_numpy(np.ascontiguousarray(w[:, 2])).to(dev)
        self.counts = torch.empty((self.n_win, self.K), dtype=torch.int32, device=dev)
        self.counts3 = torch.empty((self.n_win, 64), dtype=torch.int32, device=dev) if self.fused else None
        self.totals = torch.zeros(self.K, dtype=torch.int64, device=dev)
        self.totals3 = torch.zeros(64, dtype=torch.int64, device=dev) if self.fused else None
        biggest = int((his - los).max()) if len(los) else 0
        self.workspace = kernels.scan_workspace(dev, max(biggest, 1))
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        out_dt = torch.uint16 if self.narrow else torch.int32
        if self.narrow:
            self.narrow_d = torch.empty((self.n_win, self.K), dtype=torch.uint16, device=dev)
            self.narrow3_d = torch.empty((self.n_win, 64), dtype=torch.uint16, device=dev) if self.fused else None
        # host: results
        self.host_counts = _pinned((self.n_win, self.K), out_dt)
        self.host_counts3 = _pinned((self.n_win, 64), out_dt) if self.fused else None
        self.host_totals = _pinned((self.K + (64 if self.fused else 0),), torch.int64)
        self.host_status = _pinned((1,), torch.int32)
        self.copy_stream = torch.cuda.Stream(dev)
        self.out_stream = torch.cuda.Stream(dev)
        per_base = (0.375 if hg.nmask is not None else 0.25) if hg.is_packed else 1.0
        ends = np.append(hg.chrom_off[1:], hg.n_bases) if n_chrom else np.zeros(0, dtype=np.int64)
        self.h2d_bytes = int(sum(int(ends[c] - hg.chrom_off[c]) for c, _, _ in self.order) * per_base) + \
            (int(hg.mask_runs.numel()) * 8 if hg.is_packed and hg.nmask is None else 0)
        per = 2 if self.narrow else 4
        self.d2h_bytes = self.n_win * (self.K + (64 if self.fused else 0)) * per + self.host_totals.numel() * 8 + 4
        self.launches_per_run = 0

    # -- one chromosome ---------------------------------------------------------------------------
    def _upload(self, c):
        hg = self.hg
        a = int(hg.chrom_off[c])
        b = int(hg.chrom_off[c + 1]) if c + 1 < len(hg.chrom_off) else hg.n_bases
        if b <= a:
            return
        if hg.is_packed:
            self.packed2[a // 16:b // 16].copy_(hg.packed2[a // 16:b // 16], non_blocking=True)
            if hg.nmask is not None:
                self.nmask[a // 32:b // 32].copy_(hg.nmask[a // 32:b // 32], non_blocking=True)
        else:
            self.dev_ascii[a:b].copy_(hg.ascii[a:b], non_blocking=True)

    def _pack(self, c, stream):
        hg = self.hg
        a = int(hg.chrom_off[c])
        b = int(hg.chrom_off[c + 1]) if c + 1 < len(hg.chrom_off) else hg.n_bases
        if b <= a:
            return
        if hg.is_packed and self.runs_d is not None:
            lo, hi = int(self.run_lo[c]), int(self.run_lo[c + 1])
            _lib.call("dig_nmask_fill_runs", self.runs_d.data_ptr() + lo * 24, hi - lo, self.nmask.data_ptr(),
                      int(self.word_off[c]), int(self.word_off[c + 1] - self.word_off[c]), stream.cuda_stream)
        elif not hg.is_packed:
            _lib.call("dig_pack_genome", self.dev_ascii.data_ptr() + a, b - a, self.packed2.data_ptr() + a // 16 * 4,
                      self.nmask.data_ptr() + a // 32 * 4, self.n_other_d.data_ptr(), stream.cuda_stream)
        # this chromosome's mask words were just rewritten (copy, runs or pack): its part of the N summary follows them
        self.genome.rebuild_nsum(a // 32, (b + 31) // 32 - a // 32, stream)

    def _scan(self, lo, hi, stream):
        g = self.genome
        if self.fused:
            kernels.count_contexts_fused53(g, self.win_chrom[lo:hi], self.win_start[lo:hi], self.win_end[lo:hi],
                                           out5=self.counts[lo:hi], out3=self.counts3[lo:hi], totals5=self.totals,
                                           totals3=self.totals3, stream=stream, workspace=self.workspace,
                                           tile_window=self.tile_window)
        else:
            kernels.count_contexts(g, self.win_chrom[lo:hi], self.win_start[lo:hi], self.win_end[lo:hi], self.n_up,
                                   self.n_down, out=self.counts[lo:hi], totals=self.totals, stream=stream,
                                   workspace=self.workspace, tile_window=self.tile_window)
        if self.narrow:
            for src, dst in ((self.counts, self.narrow_d), (self.counts3, self.narrow3_d if self.fused else None)):
                if src is not None and dst is not None:
                    _lib.call("dig_narrow_counts_u16", src[lo:hi].data_ptr(), (hi - lo) * src.shape[1],
                              dst[lo:hi].data_ptr(), self.status.data_ptr(), stream.cuda_stream)

    def _download(self, lo, hi):
        src, src3 = (self.narrow_d, self.narrow3_d) if self.narrow else (self.counts, self.counts3)
        self.host_counts[lo:hi].copy_(src[lo:hi], non_blocking=True)
        if self.fused:
            self.host_counts3[lo:hi].copy_(src3[lo:hi], non_blocking=True)

    def run(self, sync=True):
        """One pass.  Returns self (results in host_counts / host_counts3 / host_totals once synchronised).
        With sync=False the caller must synchronise the device before reading the host buffers (and then call
        finish())."""
        dev = self.device
        n0 = _lib.launch_count
        main = torch.cuda.current_stream(dev)
        cs, os_ = self.copy_stream, self.out_stream
        cs.wait_stream(main)
        os_.wait_stream(main)
        self.totals.zero_()
        if self.fused:
            self.totals3.zero_()
        self.status.zero_()
        if not self.hg.is_packed:
            self.n_other_d.zero_()
        with torch.cuda.device(dev):
            if self.runs_d is not None and self.hg.mask_runs.numel():
                with torch.cuda.stream(cs):
                    self.runs_d[: self.hg.mask_runs.shape[0]].copy_(self.hg.mask_runs, non_blocking=True)
            for c, lo, hi in self.order:
                with torch.cuda.stream(cs):
                    self._upload(c)
                    e_in = torch.cuda.Event()
                    e_in.record(cs)
                main.wait_event(e_in)
                self._pack(c, main)
                if hi > lo:
                    self._scan(lo, hi, main)
                    e_scan = torch.cuda.Event()
                    e_scan.record(main)
                    with torch.cuda.stream(os_):
                        os_.wait_event(e_scan)
                        self._download(lo, hi)
            tot = torch.cat([self.totals, self.totals3]) if self.fused else self.totals
            self.host_totals.copy_(tot, non_blocking=True)
            self.host_status.copy_(self.status, non_blocking=True)
            main.wait_stream(os_)
        self.launches_per_run = _lib.launch_count - n0
        if sync:
            torch.cuda.synchronize(dev)
            self.finish()
        return self

    def finish(self):
        """After the device has been synchronised: act on the narrowing verdict, pick up n_other."""
        if not self.hg.is_packed:
            self.genome.n_other = int(self.n_other_d.item())
        if self.narrow and int(self.host_status[0]) != 0:
            # a count did not fit 16 bits (regions >= 65536 bases slipped through a forced narrow=True): ship int32
            self.host_counts = self.counts.cpu()
            if self.fused:
                self.host_counts3 = self.counts3.cpu()
            self.narrow = False
        return self


def count_contexts_from_fasta(fasta_path, chrom_idx, starts, ends, n_up, n_down, device="cuda:0", use_cache=True,
                              cache_dir=None, also_tri=False):
    """countGenomeContext's data path for a FASTA file: packed cache (or parse + pack), pipelined scan, host results.
    Returns (counts [Nw, K] numpy (uint16 or int32), totals int64 [K], DeviceGenome, extras dict)."""
    hg, hit = host_genome_from_fasta(fasta_path, use_cache, cache_dir)
    w = np.stack([np.asarray(chrom_idx, dtype=np.int64), np.asarray(starts, dtype=np.int64),
                  np.asarray(ends, dtype=np.int64)], axis=1)
    fused = also_tri and n_up == 2 and n_down == 2
    hs = HostScan(hg, w, device, tables="penta+tri" if fused else (n_up, n_down))
    hs.run()
    if use_cache and not hit:
        PackedGenomeCache.store(fasta_path, hs.genome, cache_dir)
    extras = {"cache_hit": hit, "h2d_bytes": hs.h2d_bytes, "d2h_bytes": hs.d2h_bytes}
    K = hs.K
    if fused:
        extras["counts3"] = hs.host_counts3.numpy()
        extras["totals3"] = hs.host_totals[K:].numpy().copy()
    return hs.host_counts.numpy(), hs.host_totals[:K].numpy().copy(), hs.genome, extras
