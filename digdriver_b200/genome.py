"""Genome containers: host ASCII chromosomes and the device-resident 2-bit packed genome.

The reference reads the genome through ``pysam.FastaFile`` one window at a time
(DIGDriver/sequence_model/sequence_tools.py:21-29, :84); here the whole genome is packed once
into HBM (0.375 B/base: 2-bit bases + N bitmask) and every kernel works on that.
"""

import numpy as np
import torch

from . import _lib

ALIGN = 128  # chromosome offsets are multiples of 128 bases (32 B of packed bases, 16 B of mask)


class Genome:
    """Host-side genome: chromosome names (as in the FASTA, e.g. 'chr1') and uint8 ASCII arrays."""

    def __init__(self, names, seqs):
        self.names = list(names)
        self.seqs = [np.ascontiguousarray(s, dtype=np.uint8) for s in seqs]
        self._index = {n: i for i, n in enumerate(self.names)}

    @classmethod
    def from_dict(cls, d):
        names, seqs = [], []
        for k, v in d.items():
            names.append(k)
            seqs.append(np.frombuffer(v.encode(), dtype=np.uint8) if isinstance(v, str) else v)
        return cls(names, seqs)

    @classmethod
    def from_fasta(cls, path):
        """Minimal FASTA reader (plain text or .gz); sequence names are the first word of each header."""
        import gzip
        opener = gzip.open if str(path).endswith(".gz") else open
        with opener(path, "rb") as f:
            data = np.frombuffer(f.read(), dtype=np.uint8)
        nl = np.flatnonzero(data == 10)
        line_starts = np.concatenate(([0], nl + 1))
        line_starts = line_starts[line_starts < len(data)]
        hdr_lines = line_starts[data[line_starts] == ord(">")]
        names, seqs = [], []
        for i, h in enumerate(hdr_lines):
            h_end = nl[np.searchsorted(nl, h)] if len(nl) and np.searchsorted(nl, h) < len(nl) else len(data)
            name = data[h + 1:h_end].tobytes().decode().split()[0] if h_end > h + 1 else ""
            body_end = hdr_lines[i + 1] if i + 1 < len(hdr_lines) else len(data)
            body = data[h_end + 1:body_end]
            body = body[(body != 10) & (body != 13)]
            names.append(name)
            seqs.append(body)
        return cls(names, seqs)

    def index(self, name):
        return self._index[name]

    def __contains__(self, name):
        return name in self._index

    @property
    def lengths(self):
        return np.array([len(s) for s in self.seqs], dtype=np.int64)

    def fetch(self, name, start=None, end=None):
        s = self.seqs[self._index[name]]
        return (s if start is None else s[start:end]).tobytes().decode()


def nsum_layout(n_mask_words):
    """(offset in words, number of words) of the per-128-base N summary that follows a mask of n_mask_words words in
    the same allocation (dig_scan_opts.nsum_offset_words)."""
    return (n_mask_words + 3) // 4 * 4, max(((n_mask_words + 3) // 4 + 15) // 16, 1)


def alloc_nmask(n_mask_words, device):
    """An int32 N mask of n_mask_words words with room for its N summary behind it (summary blocks read as all N)."""
    off, nsw = nsum_layout(n_mask_words)
    buf = torch.empty(off + nsw, dtype=torch.int32, device=device)
    buf[off:].fill_(-1)
    return buf[:n_mask_words]


def _layout(lengths):
    lengths = np.asarray(lengths, dtype=np.int64)
    padded = (lengths + ALIGN - 1) // ALIGN * ALIGN
    off = np.zeros(len(lengths), dtype=np.int64)
    if len(lengths) > 1:
        off[1:] = np.cumsum(padded)[:-1]
    total = int(padded.sum())
    return off, total


class DeviceGenome:
    """2-bit packed genome + N mask in HBM, with per-chromosome offsets (global coordinates).

    ``nsum`` is the per-128-base N summary of ``nmask`` (dig_nmask_summary, 2 bits per block), stored ``nsum_offset``
    words behind the mask in the same allocation (alloc_nmask; a mask without that room is copied into such a buffer):
    the lane-bank scan reads it instead of staging the mask.  It is built here from ``nmask``; whoever rewrites words of
    ``nmask`` afterwards calls ``rebuild_nsum`` over the same words (build_nsum=False: the mask is filled later)."""

    def __init__(self, names, chrom_len, chrom_off, n_bases, packed2, nmask, n_other, device, build_nsum=True):
        self.names = list(names)
        self._index = {n: i for i, n in enumerate(self.names)}
        self.chrom_len = np.asarray(chrom_len, dtype=np.int64)
        self.chrom_off = np.asarray(chrom_off, dtype=np.int64)
        self.n_bases = int(n_bases)
        self.packed2 = packed2
        self.nsum_offset, nsw = nsum_layout(nmask.numel())
        if not nmask.is_contiguous() or nmask.untyped_storage().nbytes() < (nmask.storage_offset() + self.nsum_offset + nsw) * 4:
            m = alloc_nmask(nmask.numel(), nmask.device)
            m.copy_(nmask)
            nmask = m
        self.nmask = nmask
        self.nsum = nmask.as_strided((nsw,), (1,), nmask.storage_offset() + self.nsum_offset)
        self.n_other = int(n_other)
        self.device = device
        self.chrom_len_d = torch.from_numpy(self.chrom_len).to(device)
        self.chrom_off_d = torch.from_numpy(self.chrom_off).to(device)
        if build_nsum:
            self.rebuild_nsum(0, nmask.numel())

    def rebuild_nsum(self, word0, n_words, stream=None):
        """Rebuild the summary of mask words [word0, word0 + n_words) (word0 a multiple of 4) on `stream`."""
        st = stream if stream is not None else torch.cuda.current_stream(self.nmask.device)
        with torch.cuda.device(self.nmask.device):
            _lib.call("dig_nmask_summary", self.nmask.data_ptr(), int(word0), int(n_words), self.nsum.data_ptr(),
                      st.cuda_stream)

    def index(self, name):
        return self._index[name]

    def __contains__(self, name):
        return name in self._index

    def chrom_indices(self, chroms, prefix="chr"):
        """Map reference-style chromosome labels (ints or strings, with or without 'chr') to indices."""
        out = np.empty(len(chroms), dtype=np.int32)
        cache = {}
        for i, c in enumerate(chroms):
            k = c if not isinstance(c, (np.generic,)) else c.item()
            if k not in cache:
                s = str(k)
                if s in self._index:
                    cache[k] = self._index[s]
                elif prefix + s in self._index:
                    cache[k] = self._index[prefix + s]
                else:
                    raise KeyError("chromosome %r not in genome" % (c,))
            out[i] = cache[k]
        return out

    @staticmethod
    def pack_ascii(ascii_d, stream=None):
        """Run K1 on a device uint8 tensor; returns (packed2, nmask, n_other)."""
        lib = _lib.load()
        n = ascii_d.numel()
        dev = ascii_d.device
        packed2 = torch.empty(max(int(lib.dig_packed_words(n)), 2), dtype=torch.int32, device=dev)
        nmask = alloc_nmask(max(int(lib.dig_nmask_words(n)), 1), dev)
        n_other = torch.zeros(1, dtype=torch.int64, device=dev)
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        with torch.cuda.device(dev):
            _lib.call("dig_pack_genome", ascii_d.data_ptr(), n, packed2.data_ptr(), nmask.data_ptr(),
                      n_other.data_ptr(), st.cuda_stream)
        return packed2, nmask, n_other

    @classmethod
    def from_genome(cls, genome, device="cuda:0"):
        device = torch.device(device)
        lengths = genome.lengths
        off, total = _layout(lengths)
        ascii_d = torch.full((max(total, 1),), ord("N"), dtype=torch.uint8, device=device)
        for o, s in zip(off, genome.seqs):
            if len(s):
                ascii_d[int(o):int(o) + len(s)].copy_(torch.from_numpy(s), non_blocking=False)
        packed2, nmask, n_other = cls.pack_ascii(ascii_d[:total])
        n_other = int(n_other.item())
        del ascii_d
        return cls(genome.names, lengths, off, total, packed2, nmask, n_other, device)

    @classmethod
    def synthetic(cls, names, lengths, seed, device="cuda:0", n_frac16=16, return_ascii=False):
        """Generate the synthetic genome of BASELINE.json's configs directly in HBM.

        Chromosome c occupies global positions [off[c], off[c]+len[c]) of the generator's
        coordinate space, so oracle.synth_genome(off[c], len[c], seed) reproduces it on the CPU."""
        device = torch.device(device)
        lengths = np.asarray(lengths, dtype=np.int64)
        off, total = _layout(lengths)
        ascii_d = torch.full((max(total, 1),), ord("N"), dtype=torch.uint8, device=device)
        st = torch.cuda.current_stream(device)
        with torch.cuda.device(device):
            for o, n in zip(off, lengths):
                _lib.call("dig_synth_genome", ascii_d.data_ptr() + int(o), int(o), int(n), int(seed),
                          int(n_frac16), st.cuda_stream)
        packed2, nmask, n_other = cls.pack_ascii(ascii_d[:total])
        g = cls(names, lengths, off, total, packed2, nmask, int(n_other.item()), device)
        if return_ascii:
            return g, ascii_d[:total]
        return g


def hg19_like_lengths(total=3_100_000_000):
    """22 autosome-like chromosome lengths (hg19 proportions) summing to ``total``."""
    hg19 = np.array([249250621, 243199373, 198022430, 191154276, 180915260, 171115067, 159138663, 146364022,
                     141213431, 135534747, 135006516, 133851895, 115169878, 107349540, 102531392, 90354753,
                     81195210, 78077248, 59128983, 63025520, 48129895, 51304566], dtype=np.float64)
    ln = np.floor(hg19 / hg19.sum() * total).astype(np.int64)
    ln[0] += total - ln.sum()
    return ln


def tile_windows(chrom_labels, lengths, window):
    """Window tiling of the reference's data extractor: from 0 in steps of ``window`` while
    i + window < chrom_len (scripts/DataExtractor.py:70-77).  Returns int64 [Nw, 3]."""
    rows = []
    for c, L in zip(chrom_labels, lengths):
        n = max(0, (int(L) - 1) // window) if L > window else 0
        starts = np.arange(n, dtype=np.int64) * window
        rows.append(np.stack([np.full(n, c, dtype=np.int64), starts, starts + window], axis=1))
    return np.concatenate(rows, axis=0) if rows else np.zeros((0, 3), dtype=np.int64)
