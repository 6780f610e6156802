"""Python mirror of the C ABI (include/bamqc_b200.h).  Names follow the reference: lanes (read groups),
mates (QualityCheck r1/r2, src/bamqualcheck.cpp:17), q/k pairs (ReadQualityHasher grid, :28-36)."""
import ctypes

import numpy as np

from . import _lib

FIELDS = dict(
    SCALARS=0, POSCOV=1, INSERT=2, EIGHTMER=3, TRIPLET=4, READLEN=5, NCOUNT=6, GCCOUNT=7, AVGQUAL=8, MAPQ=9,
    MISMATCH=10, DEL=11, INS=12, DNA_A=13, DNA_C=14, DNA_G=15, DNA_T=16, DNA_N=17, QUALSUM=18, SC5=19, SC3=20,
    READNR=21, SUMCOUNT=22, F2TABLE=23)
SCALAR_NAMES = ["supplementary", "duplicates", "QCfailed", "not_primary_alignment", "readcount", "totalbps",
                "bothunmapped", "firstunmapped", "secondunmapped", "first_and_or_second_mapped",
                "FF_RR_orientation", "properpair_count", "auto_properpair_count"]
DEFAULT_CHROMS = ",".join("chr%d" % i for i in range(1, 23))  # src/CommandLineParser.hpp:34


BQC_ERR_ARG = 33


def parse_sam_header(text):
    """The '@' header lines at the front of SAM text -> (dict with text, ref_names, ref_lengths, lane_ids, sample_id,
    offset of the first alignment line), through the same parser as a BAM header."""
    b = text.encode() if isinstance(text, str) else bytes(text)
    lib = _lib.load_library()
    h = _lib.bqc_bam_header()
    used = ctypes.c_size_t()
    rc = lib.bqc_parse_sam_header(b, len(b), ctypes.byref(h), ctypes.byref(used))
    if rc:
        raise BamQCError(rc, "malformed SAM header")
    try:
        out = {"text": h.text.decode(), "ref_names": [h.ref_names[i].decode() for i in range(h.n_ref)],
               "ref_lengths": [int(h.ref_lengths[i]) for i in range(h.n_ref)],
               "lane_ids": [h.lane_ids[i].decode() for i in range(h.n_lanes)],
               "sample_id": h.sample_id.decode() if h.sample_id else ""}
    finally:
        lib.bqc_free_bam_header(ctypes.byref(h))
    return out, used.value


class BamQCError(RuntimeError):
    def __init__(self, code, message, record=None):
        super().__init__(f"[bqc error {code}] {message}")
        self.code, self.record = code, record


def _as_u8(data):
    if isinstance(data, (bytes, bytearray, memoryview)):
        data = np.frombuffer(data, dtype=np.uint8)
    a = np.ascontiguousarray(data)
    assert a.dtype == np.uint8
    return a


class Batch:
    """A record batch resident in HBM (bqc_batch)."""

    def __init__(self, engine, handle):
        self.engine, self.handle = engine, handle
        self.n_records = int(engine.lib.bqc_batch_records(handle))
        self.n_bytes = int(engine.lib.bqc_batch_bytes(handle))

    def free(self):
        if self.handle:
            self.engine.lib.bqc_batch_free(self.engine.handle, self.handle)
            self.handle = None


class Engine:
    """One statistics engine on one GPU (bqc_engine)."""

    def __init__(self, lane_ids=("L1",), ref_names=(), chroms=DEFAULT_CHROMS, isize=1000, klist=(32,), qlist=(17,),
                 e=0.01, seed=1, device=0, max_read_len=0, staging_bytes=0, cov_ring_log2=0, host_threads=0):
        self.lib = _lib.load_library()
        self.lane_ids = [l if isinstance(l, str) else l.decode() for l in lane_ids]
        self.ref_names = [r if isinstance(r, str) else r.decode() for r in ref_names]
        self.klist, self.qlist = list(klist), list(qlist)
        main = set(chroms.split(",")) if isinstance(chroms, str) else set(chroms)
        # initChroms (src/bamqualcheck.cpp:106-123): names that exist in the BAM header
        self.main_chrom = np.array([1 if r in main else 0 for r in self.ref_names] or [0], dtype=np.uint8)
        cfg = _lib.bqc_config()
        self._keep = []
        cfg.device, cfg.isize = device, isize
        cfg.n_lanes = len(self.lane_ids)
        arr = (ctypes.c_char_p * len(self.lane_ids))(*[l.encode() for l in self.lane_ids])
        cfg.lane_ids = arr
        cfg.n_ref = len(self.ref_names)
        cfg.main_chrom = self.main_chrom.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
        ka = (ctypes.c_int32 * max(1, len(self.klist)))(*self.klist)
        qa = (ctypes.c_uint64 * max(1, len(self.qlist)))(*self.qlist)
        cfg.n_k, cfg.klist, cfg.n_q, cfg.q_cutoff = len(self.klist), ka, len(self.qlist), qa
        cfg.q_base, cfg.e, cfg.seed = 33, e, seed
        cfg.max_read_len, cfg.staging_bytes, cfg.cov_ring_log2 = max_read_len, staging_bytes, cov_ring_log2
        cfg.host_threads = host_threads
        self._keep += [arr, ka, qa]
        h = ctypes.c_void_p()
        rc = self.lib.bqc_create(ctypes.byref(cfg), ctypes.byref(h))
        if rc:
            raise BamQCError(rc, self.lib.bqc_last_error(None).decode())
        self.handle = h
        self.device = device
        self._sam_refs_set = False

    # ---- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "handle", None):
            self.lib.bqc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            info = _lib.bqc_error_info()
            self.lib.bqc_get_error(self.handle, ctypes.byref(info))
            msg = self.lib.bqc_last_error(self.handle).decode()
            if info.code:
                raise BamQCError(info.code, info.message.decode(), int(info.record))
            raise BamQCError(rc, msg)

    # ---- inputs -----------------------------------------------------------------------------------
    def set_reference(self, rid, packed, n_bases):
        p = _as_u8(packed)
        assert p.size * 4 >= n_bases
        self._check(self.lib.bqc_set_reference(self.handle, rid, p.ctypes.data, n_bases))

    def reset(self):
        self._check(self.lib.bqc_reset(self.handle))

    def acquire_staging(self):
        p, cap = ctypes.c_void_p(), ctypes.c_size_t()
        self._check(self.lib.bqc_acquire_staging(self.handle, ctypes.byref(p), ctypes.byref(cap)))
        buf = (ctypes.c_uint8 * cap.value).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint8)

    def submit(self, data, offsets=None, n_bytes=None):
        a = _as_u8(data)
        n = a.size if n_bytes is None else n_bytes
        if offsets is None:
            self._check(self.lib.bqc_submit(self.handle, a.ctypes.data, n, None, 0))
        else:
            o = np.ascontiguousarray(offsets, dtype=np.uint64)
            self._check(self.lib.bqc_submit(self.handle, a.ctypes.data, n, o.ctypes.data, o.size - 1))

    def submit_stream(self, data, last=False, n_bytes=None):
        """Next chunk of the inflated record stream (need not end on a record boundary)."""
        a = _as_u8(data)
        n = a.size if n_bytes is None else n_bytes
        self._check(self.lib.bqc_submit_stream(self.handle, a.ctypes.data if n else None, n, 1 if last else 0))

    def submit_bgzf(self, data, skip=0, last=False):
        """Whole BGZF blocks (compressed .bam bytes); inflated and framed on the device."""
        a = _as_u8(data)
        self._check(self.lib.bqc_submit_bgzf(self.handle, a.ctypes.data if a.size else None, a.size, skip, 1 if last else 0))

    def _sam_refs(self):  # bqc_set_ref_names once, before the first SAM text
        if not self._sam_refs_set:
            names = (ctypes.c_char_p * max(1, len(self.ref_names)))(*[r.encode() for r in self.ref_names])
            self._check(self.lib.bqc_set_ref_names(self.handle, len(self.ref_names), names))
            self._sam_refs_set = True

    def submit_sam(self, data, last=False):
        """SAM alignment lines (no header lines), ending at a line end unless `last`; encoded to BAM records on the
        device.  RNAME/RNEXT are looked up in `ref_names`."""
        self._sam_refs()
        a = _as_u8(data.encode() if isinstance(data, str) else data)
        self._check(self.lib.bqc_submit_sam(self.handle, a.ctypes.data if a.size else None, a.size, 1 if last else 0))

    def sam_to_bam(self, text):
        """The BAM records (block_size included) that submit_sam counts for `text`, as bytes."""
        self._sam_refs()
        a = _as_u8(text.encode() if isinstance(text, str) else text)
        out = np.empty(2 * a.size + 64, dtype=np.uint8)
        nb, nr = ctypes.c_uint64(), ctypes.c_uint64()
        rc = self.lib.bqc_sam_to_bam(self.handle, a.ctypes.data if a.size else None, a.size, out.ctypes.data, out.size, ctypes.byref(nb), ctypes.byref(nr))
        if rc == BQC_ERR_ARG:   # a host-encoded submission (B arrays) may need more than twice the text
            out = np.empty(8 * a.size + 64, dtype=np.uint8)
            rc = self.lib.bqc_sam_to_bam(self.handle, a.ctypes.data if a.size else None, a.size, out.ctypes.data, out.size, ctypes.byref(nb), ctypes.byref(nr))
        self._check(rc)
        return out[:nb.value].tobytes()

    @property
    def sam_host_lines(self):
        """Non-empty SAM lines that went through the host encoder (submissions outside the device grammar)."""
        return int(self.lib.bqc_sam_host_lines(self.handle))

    @property
    def frames_repaired(self):
        return int(self.lib.bqc_frames_repaired(self.handle))

    @property
    def records_seen(self):
        return int(self.lib.bqc_records_seen(self.handle))

    def prepare(self, data, offsets=None):
        a = _as_u8(data)
        h = ctypes.c_void_p()
        if offsets is None:
            rc = self.lib.bqc_batch_prepare(self.handle, a.ctypes.data, a.size, None, 0, ctypes.byref(h))
        else:
            o = np.ascontiguousarray(offsets, dtype=np.uint64)
            rc = self.lib.bqc_batch_prepare(self.handle, a.ctypes.data, a.size, o.ctypes.data, o.size - 1, ctypes.byref(h))
        self._check(rc)
        return Batch(self, h)

    def run(self, batch):
        self._check(self.lib.bqc_batch_run(self.handle, batch.handle))

    def sync(self):
        self._check(self.lib.bqc_sync(self.handle))

    def finish(self):
        self._check(self.lib.bqc_finish(self.handle))

    @property
    def stream(self):
        return self.lib.bqc_stream(self.handle)

    @property
    def kernel_launches(self):
        return int(self.lib.bqc_kernel_launches(self.handle))

    def profile_enable(self, on=True):
        self.lib.bqc_profile_enable(self.handle, int(on))  # 2: serialised (coverage kernels on the compute stream)

    def profile_read(self):
        """{family: (milliseconds, launch groups)} since the previous read (CUDA events on the compute stream)."""
        ms = (ctypes.c_double * 12)()
        n = (ctypes.c_uint64 * 12)()
        self._check(self.lib.bqc_profile_read(self.handle, ms, n))
        names = ["k_stats", "k_eightmer", "k_sketch", "k_cov", "merge", "host_framing", "host_scan_pass1", "host_scan_pass2",
                 "k_inflate", "k_frame", "k_sam", "_11"]
        return {names[i]: (float(ms[i]), int(n[i])) for i in range(12)}

    # ---- multi-GPU merge ----------------------------------------------------------------------------
    def counters_len(self):
        return int(self.lib.bqc_counters_len(self.handle))

    def sketch_len(self):
        return int(self.lib.bqc_sketch_len(self.handle))

    def export_to(self, counters_ptr, sketch_ptr):
        self._check(self.lib.bqc_counters_export(self.handle, counters_ptr))
        if self.sketch_len():
            self._check(self.lib.bqc_sketch_export_u8(self.handle, sketch_ptr))

    def import_from(self, counters_ptr, sketch_ptr):
        self._check(self.lib.bqc_counters_import(self.handle, counters_ptr))
        if self.sketch_len():
            self._check(self.lib.bqc_sketch_import_u8(self.handle, sketch_ptr))

    def merge_from(self, other):
        self._check(self.lib.bqc_merge_from(self.handle, other.handle))

    # ---- one record stream cut across several engines: the coverage statistic (bamqc_b200.h) ------------
    def cov_defer(self, mode=1):
        """1: a piece of a stream whose entry state is unknown; 2: the first piece of the stream; 0: stand-alone."""
        self._check(self.lib.bqc_cov_defer(self.handle, int(mode)))

    def cov_shard_boundary(self, lane=0):
        sh = _lib.bqc_cov_shard()
        self._check(self.lib.bqc_cov_shard_boundary_lane(self.handle, int(lane), ctypes.byref(sh)))
        return sh

    def cov_shard_function(self, have_prev, prev_rid, prev_b, lane=0):
        out = np.zeros(1002, dtype=np.uint16)
        self._check(self.lib.bqc_cov_shard_function_lane(self.handle, int(lane), int(have_prev), int(prev_rid), int(prev_b), out.ctypes.data))
        return out

    def cov_shard_run(self, have_prev, prev_rid, prev_b, p_in, lane=0):
        sh = _lib.bqc_cov_shard()
        self._check(self.lib.bqc_cov_shard_run_lane(self.handle, int(lane), int(have_prev), int(prev_rid), int(prev_b), int(p_in), ctypes.byref(sh)))
        return sh

    def poscov_adjust(self, delta, lane=0):
        d = np.ascontiguousarray(delta, dtype=np.int64)
        assert d.size == 101
        self._check(self.lib.bqc_poscov_adjust(self.handle, lane, d.ctypes.data))

    # ---- results ------------------------------------------------------------------------------------
    def table(self, field, lane=0, sub=0):
        f = FIELDS[field] if isinstance(field, str) else field
        n = ctypes.c_uint64()
        self._check(self.lib.bqc_result_table(self.handle, lane, f, sub, None, 0, ctypes.byref(n)))
        out = np.zeros(max(1, n.value), dtype=np.uint64)
        self._check(self.lib.bqc_result_table(self.handle, lane, f, sub, out.ctypes.data, out.size, None))
        return out[: n.value]

    def scalars(self, lane=0):
        return dict(zip(SCALAR_NAMES, (int(x) for x in self.table("SCALARS", lane))))

    def sketch(self, lane=0, qk=0):
        n = ctypes.c_uint64()
        self._check(self.lib.bqc_result_sketch(self.handle, lane, qk, None, 0, ctypes.byref(n)))
        out = np.zeros(n.value, dtype=np.uint64)
        self._check(self.lib.bqc_result_sketch(self.handle, lane, qk, out.ctypes.data, out.size, None))
        return out

    def estimates(self, lane=0, qk=0):
        out = (ctypes.c_uint64 * 4)()
        self._check(self.lib.bqc_result_estimates(self.handle, lane, qk, out))
        return dict(sumCount=int(out[0]), F0=int(out[1]), f1=int(out[2]), F2=int(out[3]))

    def avgqual(self, lane=0, mate=0):
        n = ctypes.c_uint64()
        self._check(self.lib.bqc_result_avgqual(self.handle, lane, mate, None, 0, ctypes.byref(n)))
        out = np.zeros(max(1, n.value), dtype=np.float64)
        self._check(self.lib.bqc_result_avgqual(self.handle, lane, mate, out.ctypes.data, out.size, None))
        return out[: n.value]

    def write_bamqc(self, sample_id, path):
        rc = self.lib.bqc_write_bamqc(self.handle, sample_id.encode(), str(path).encode())
        if rc:
            raise BamQCError(rc, "could not write " + str(path))
