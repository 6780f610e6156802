"""Seeded synthetic BAM/FASTA data (include/bamqc_synth.h) and the SURVEY.md section 8(d) data sets."""
import ctypes
from dataclasses import dataclass, field

import numpy as np

from . import _lib

GRCH38 = [  # chr1..22, X, Y lengths (cfg 2/3 geometry)
    248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422,
    135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167,
    46709983, 50818468, 156040895, 57227415]
GRCH38_NAMES = ["chr%d" % i for i in range(1, 23)] + ["chrX", "chrY"]


@dataclass
class Genome:
    names: list
    lengths: list
    packed: list  # numpy uint8 arrays, 2-bit packed
    seed: int = 0

    @staticmethod
    def make(seed, names, lengths):
        lib = _lib.load_synth()
        packed = []
        for i, n in enumerate(lengths):
            a = np.zeros((n + 31) // 32 * 8 + 16, dtype=np.uint8)
            lib.bqc_synth_reference(seed, i, n, a.ctypes.data)
            packed.append(a)
        return Genome(list(names), list(lengths), packed, seed)

    def write_fasta(self, path):
        lib = _lib.load_synth()
        n = len(self.names)
        names = (ctypes.c_char_p * n)(*[s.encode() for s in self.names])
        lens = (ctypes.c_uint64 * n)(*self.lengths)
        ptrs = (ctypes.c_void_p * n)(*[p.ctypes.data for p in self.packed])
        if lib.bqc_synth_write_fasta(str(path).encode(), n, names, lens, ptrs):
            raise IOError(path)


@dataclass
class Library:
    """Library / alignment properties of a synthetic data set (defaults = SURVEY 8d standard)."""
    seed: int = 20260101
    n_pairs: int = 1000
    read_len: int = 150
    ins_mean: float = 400.0
    ins_sd: float = 60.0
    ins_min: int = 150
    ins_max: int = 1000
    sub_rate: float = 0.005
    n_rate: float = 0.001
    indel_read_frac: float = 0.03
    max_indels: int = 1
    softclip_frac: float = 0.03
    low_quality: int = 0
    mapq60_frac: float = 0.9
    dup_frac: float = 0.02
    qcfail_frac: float = 0.005
    one_unmapped_frac: float = 0.01
    both_unmapped_frac: float = 0.005
    secondary_frac: float = 0.005
    supplementary_frac: float = 0.005
    n_lanes: int = 1
    first_pair_id: int = 0
    emit_unmapped_tail: int = 1
    regions: dict = field(default_factory=dict)  # contig index -> (begin, end); empty = whole genome

    def stress(self):
        """cfg 4: high-error / low-quality library."""
        self.sub_rate, self.softclip_frac, self.indel_read_frac, self.max_indels = 0.05, 0.30, 0.15, 3
        self.low_quality, self.mapq60_frac = 1, -1.0
        return self


class _Params:
    def __init__(self, genome, lib_):
        self.c = _lib.bqc_synth_params()
        L = _lib.load_synth()
        L.bqc_synth_default_params(ctypes.byref(self.c))
        n = len(genome.names)
        self._names = (ctypes.c_char_p * n)(*[s.encode() for s in genome.names])
        self._lens = (ctypes.c_uint64 * n)(*genome.lengths)
        self._ptrs = (ctypes.c_void_p * n)(*[p.ctypes.data for p in genome.packed])
        c = self.c
        c.n_contigs, c.names, c.lengths, c.packed = n, self._names, self._lens, self._ptrs
        for k in ("seed", "n_pairs", "read_len", "ins_mean", "ins_sd", "ins_min", "ins_max", "sub_rate", "n_rate",
                  "indel_read_frac", "max_indels", "softclip_frac", "low_quality", "mapq60_frac", "dup_frac",
                  "qcfail_frac", "one_unmapped_frac", "both_unmapped_frac", "secondary_frac", "supplementary_frac",
                  "n_lanes", "first_pair_id", "emit_unmapped_tail"):
            setattr(c, k, getattr(lib_, k))
        if lib_.regions:
            b = [0] * n
            e = [0] * n
            for i, (lo, hi) in lib_.regions.items():
                b[i], e[i] = lo, hi
            self._rb = (ctypes.c_uint64 * n)(*b)
            self._re = (ctypes.c_uint64 * n)(*e)
            c.region_begin, c.region_end = self._rb, self._re


def generate(genome, lib_):
    """Return (records uint8[n_bytes + 64 pad], offsets uint64[n_records+1]) -- coordinate-sorted inflated BAM records."""
    L = _lib.load_synth()
    p = _Params(genome, lib_)
    est_rec = int(lib_.n_pairs * 2.05) + 1024
    per = 4 + 32 + 12 + 40 + (lib_.read_len + 1) // 2 + lib_.read_len + 24
    for _ in range(3):
        out = np.zeros(est_rec * per + 64, dtype=np.uint8)
        offs = np.zeros(est_rec + 2, dtype=np.uint64)
        nb, nr = ctypes.c_uint64(), ctypes.c_uint64()
        rc = L.bqc_synth_records(ctypes.byref(p.c), out.ctypes.data, out.size - 64, ctypes.byref(nb), offs.ctypes.data,
                                 offs.size, ctypes.byref(nr))
        if rc == 0:
            return out[: nb.value + 64], offs[: nr.value + 1].copy()
        est_rec = int(max(nr.value, est_rec) * 1.3) + 1024
    raise RuntimeError("synthetic generator capacity")


def header_text(genome, lib_, sample_id="S1"):
    L = _lib.load_synth()
    p = _Params(genome, lib_)
    n = L.bqc_synth_header_text(ctypes.byref(p.c), sample_id.encode(), None, 0)
    buf = ctypes.create_string_buffer(n + 1)
    L.bqc_synth_header_text(ctypes.byref(p.c), sample_id.encode(), buf, n)
    return buf.raw[:n].decode()


def write_sam(path, genome, lib_, records, n_bytes, sample_id="S1"):
    """SAM text of the records (header + one line per record), written by the C generator."""
    L = _lib.load_synth()
    p = _Params(genome, lib_)
    if L.bqc_synth_write_sam(str(path).encode(), ctypes.byref(p.c), sample_id.encode(), records.ctypes.data, n_bytes):
        raise IOError(path)


def write_bam(path, genome, lib_, records, n_bytes, sample_id="S1", level=-1):
    """level -1: raw uncompressed BAM stream; 0..9: BGZF."""
    L = _lib.load_synth()
    p = _Params(genome, lib_)
    if L.bqc_synth_write_bam(str(path).encode(), ctypes.byref(p.c), sample_id.encode(), records.ctypes.data, n_bytes, level):
        raise IOError(path)


def bgzf_compress(data, level=1):
    L = _lib.load_synth()
    a = np.ascontiguousarray(data, dtype=np.uint8)
    out = np.zeros(int(a.size * 1.01) + (a.size // 0xff00 + 2) * 64 + 1024, dtype=np.uint8)
    n = L.bqc_synth_bgzf_compress(a.ctypes.data, a.size, level, out.ctypes.data, out.size)
    if n == 0:
        raise RuntimeError("bgzf_compress capacity")
    return out[:n]


def lane_ids(lib_):
    return ["L%d" % (i + 1) for i in range(lib_.n_lanes)]
