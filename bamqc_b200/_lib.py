"""ctypes loaders for libbamqc_b200.so (the product: CUDA engine + host front end) and libbamqc_synth.so (the seeded
synthetic data generator used by the tests and bench.py), both built in-tree by ``bamqc_b200/csrc/Makefile``.

There is no Python or CPU fallback: if the product library is missing, importing the engine fails loudly.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SYNTH = None


def library_path():
    return os.path.join(_HERE, "libbamqc_b200.so")


def build(verbose=False):
    """Compile the CUDA extension for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libbamqc_b200.so failed")
    return library_path()


class bqc_config(ctypes.Structure):
    _fields_ = [
        ("device", ctypes.c_int32), ("isize", ctypes.c_int32), ("n_lanes", ctypes.c_int32),
        ("lane_ids", ctypes.POINTER(ctypes.c_char_p)), ("n_ref", ctypes.c_int32),
        ("main_chrom", ctypes.POINTER(ctypes.c_uint8)), ("n_k", ctypes.c_int32),
        ("klist", ctypes.POINTER(ctypes.c_int32)), ("n_q", ctypes.c_int32),
        ("q_cutoff", ctypes.POINTER(ctypes.c_uint64)), ("q_base", ctypes.c_uint32), ("e", ctypes.c_double),
        ("seed", ctypes.c_int32), ("max_read_len", ctypes.c_int32), ("staging_bytes", ctypes.c_uint64),
        ("cov_ring_log2", ctypes.c_uint32), ("host_threads", ctypes.c_int32),
    ]


class bqc_error_info(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int32), ("record", ctypes.c_uint64), ("message", ctypes.c_char * 256)]


class bqc_cov_shard(ctypes.Structure):
    _fields_ = [("n", ctypes.c_uint64), ("first_rid", ctypes.c_int32), ("last_rid", ctypes.c_int32),
                ("first_b", ctypes.c_uint32), ("last_b", ctypes.c_uint32), ("span", ctypes.c_uint64),
                ("head", ctypes.c_int32 * 2001), ("tail", ctypes.c_int32 * 2001)]


class bqc_bam_header(ctypes.Structure):
    _fields_ = [
        ("text", ctypes.c_char_p), ("n_ref", ctypes.c_int32), ("ref_names", ctypes.POINTER(ctypes.c_char_p)),
        ("ref_lengths", ctypes.POINTER(ctypes.c_int64)), ("n_lanes", ctypes.c_int32),
        ("lane_ids", ctypes.POINTER(ctypes.c_char_p)), ("sample_id", ctypes.c_char_p),
    ]


class bqc_synth_params(ctypes.Structure):
    _fields_ = [
        ("seed", ctypes.c_uint64), ("n_contigs", ctypes.c_int32), ("names", ctypes.POINTER(ctypes.c_char_p)),
        ("lengths", ctypes.POINTER(ctypes.c_uint64)), ("packed", ctypes.POINTER(ctypes.c_void_p)),
        ("region_begin", ctypes.POINTER(ctypes.c_uint64)), ("region_end", ctypes.POINTER(ctypes.c_uint64)),
        ("n_pairs", ctypes.c_uint64), ("read_len", ctypes.c_int32), ("ins_mean", ctypes.c_double),
        ("ins_sd", ctypes.c_double), ("ins_min", ctypes.c_int32), ("ins_max", ctypes.c_int32),
        ("sub_rate", ctypes.c_double), ("n_rate", ctypes.c_double), ("indel_read_frac", ctypes.c_double),
        ("max_indels", ctypes.c_int32), ("softclip_frac", ctypes.c_double), ("low_quality", ctypes.c_int32),
        ("mapq60_frac", ctypes.c_double), ("dup_frac", ctypes.c_double), ("qcfail_frac", ctypes.c_double),
        ("one_unmapped_frac", ctypes.c_double), ("both_unmapped_frac", ctypes.c_double),
        ("secondary_frac", ctypes.c_double), ("supplementary_frac", ctypes.c_double), ("n_lanes", ctypes.c_int32),
        ("first_pair_id", ctypes.c_uint64), ("emit_unmapped_tail", ctypes.c_int32),
    ]


_vp, _u64, _i32, _u32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32, ctypes.c_uint32
_P = ctypes.POINTER

# every exported entry point of include/bamqc_b200.h and include/bamqc_synth.h: (restype, argtypes)
PROTOTYPES = {
    "bqc_create": (ctypes.c_int, [_P(bqc_config), _P(_vp)]),
    "bqc_destroy": (None, [_vp]),
    "bqc_last_error": (ctypes.c_char_p, [_vp]),
    "bqc_set_reference": (ctypes.c_int, [_vp, _i32, _vp, _u64]),
    "bqc_reset": (ctypes.c_int, [_vp]),
    "bqc_acquire_staging": (ctypes.c_int, [_vp, _P(_vp), _P(ctypes.c_size_t)]),
    "bqc_submit": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _vp, _u64]),
    "bqc_submit_stream": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_int]),
    "bqc_submit_bgzf": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int]),
    "bqc_stream_unknown_start": (ctypes.c_int, [_vp]),
    "bqc_stream_skipped": (ctypes.c_int, [_vp, _P(_u64)]),
    "bqc_frames_repaired": (_u64, [_vp]),
    "bqc_set_ref_names": (ctypes.c_int, [_vp, _i32, _P(ctypes.c_char_p)]),
    "bqc_submit_sam": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_int]),
    "bqc_sam_to_bam": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _vp, _u64, _P(_u64), _P(_u64)]),
    "bqc_sam_host_lines": (_u64, [_vp]),
    "bqc_records_seen": (_u64, [_vp]),
    "bqc_batch_prepare": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _vp, _u64, _P(_vp)]),
    "bqc_batch_run": (ctypes.c_int, [_vp, _vp]),
    "bqc_batch_free": (None, [_vp, _vp]),
    "bqc_batch_records": (_u64, [_vp]),
    "bqc_batch_bytes": (_u64, [_vp]),
    "bqc_sync": (ctypes.c_int, [_vp]),
    "bqc_stream": (_vp, [_vp]),
    "bqc_kernel_launches": (_u64, [_vp]),
    "bqc_get_error": (ctypes.c_int, [_vp, _P(bqc_error_info)]),
    "bqc_finish": (ctypes.c_int, [_vp]),
    "bqc_profile_enable": (None, [_vp, ctypes.c_int]),
    "bqc_profile_read": (ctypes.c_int, [_vp, _P(ctypes.c_double), _P(_u64)]),
    "bqc_read_len_capacity": (_u32, [_vp]),
    "bqc_reserve_read_len": (ctypes.c_int, [_vp, _u32]),
    "bqc_counters_len": (_u64, [_vp]),
    "bqc_counters_export": (ctypes.c_int, [_vp, _vp]),
    "bqc_counters_import": (ctypes.c_int, [_vp, _vp]),
    "bqc_sketch_len": (_u64, [_vp]),
    "bqc_sketch_export_u8": (ctypes.c_int, [_vp, _vp]),
    "bqc_sketch_import_u8": (ctypes.c_int, [_vp, _vp]),
    "bqc_merge_from": (ctypes.c_int, [_vp, _vp]),
    "bqc_cov_defer": (ctypes.c_int, [_vp, ctypes.c_int]),
    "bqc_cov_shard_boundary": (ctypes.c_int, [_vp, _P(bqc_cov_shard)]),
    "bqc_cov_shard_function": (ctypes.c_int, [_vp, _i32, _i32, _u32, _vp]),
    "bqc_cov_shard_run": (ctypes.c_int, [_vp, _i32, _i32, _u32, _u32, _P(bqc_cov_shard)]),
    "bqc_cov_shard_boundary_lane": (ctypes.c_int, [_vp, _i32, _P(bqc_cov_shard)]),
    "bqc_cov_shard_function_lane": (ctypes.c_int, [_vp, _i32, _i32, _i32, _u32, _vp]),
    "bqc_cov_shard_run_lane": (ctypes.c_int, [_vp, _i32, _i32, _i32, _u32, _u32, _P(bqc_cov_shard)]),
    "bqc_cov_shards_combine": (None, [_vp, _i32, _vp]),
    "bqc_cov_apply": (_u32, [_vp, _u32]),
    "bqc_poscov_adjust": (ctypes.c_int, [_vp, _i32, _vp]),
    "bqc_n_lanes": (_i32, [_vp]),
    "bqc_lane_id": (ctypes.c_char_p, [_vp, _i32]),
    "bqc_qk_lists": (None, [_vp, _P(_P(_i32)), _P(_u32), _P(_P(_u64)), _P(_u32)]),
    "bqc_result_table": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _u64, _P(_u64)]),
    "bqc_result_sketch": (ctypes.c_int, [_vp, _i32, _i32, _vp, _u64, _P(_u64)]),
    "bqc_result_estimates": (ctypes.c_int, [_vp, _i32, _i32, _P(_u64)]),
    "bqc_result_avgqual": (ctypes.c_int, [_vp, _i32, _i32, _vp, _u64, _P(_u64)]),
    "bqc_write_bamqc": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_char_p]),
    "bqc_parse_bam_header": (ctypes.c_size_t, [_vp, ctypes.c_size_t, _P(bqc_bam_header)]),
    "bqc_free_bam_header": (None, [_P(bqc_bam_header)]),
    "bqc_parse_sam_header": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_size_t, _P(bqc_bam_header), _P(ctypes.c_size_t)]),
    "bqc_frame_records": (_u64, [_vp, ctypes.c_size_t, _vp, _u64]),
    "bqc_frame_records_mt": (_u64, [_vp, ctypes.c_size_t, _vp, _u64, _i32, _i32]),
    "bqc_bgzf_inflate": (_u64, [_vp, _u64, _vp, _u64, _i32]),
    "bqc_fasta_open": (_vp, [ctypes.c_char_p]),
    "bqc_fasta_contig": (ctypes.c_int64, [_vp, ctypes.c_char_p, _P(_vp)]),
    "bqc_fasta_close": (None, [_vp]),
    "bqc_main": (ctypes.c_int, [ctypes.c_int, _P(ctypes.c_char_p)]),
}

# include/bamqc_synth.h (libbamqc_synth.so)
SYNTH_PROTOTYPES = {
    "bqc_synth_default_params": (None, [_P(bqc_synth_params)]),
    "bqc_synth_reference": (None, [_u64, _i32, _u64, _vp]),
    "bqc_synth_write_fasta": (ctypes.c_int, [ctypes.c_char_p, _i32, _P(ctypes.c_char_p), _P(_u64), _P(_vp)]),
    "bqc_synth_header_text": (ctypes.c_size_t, [_P(bqc_synth_params), ctypes.c_char_p, ctypes.c_char_p, ctypes.c_size_t]),
    "bqc_synth_records": (ctypes.c_int, [_P(bqc_synth_params), _vp, _u64, _P(_u64), _vp, _u64, _P(_u64)]),
    "bqc_synth_write_bam": (ctypes.c_int, [ctypes.c_char_p, _P(bqc_synth_params), ctypes.c_char_p, _vp, _u64, ctypes.c_int]),
    "bqc_synth_bgzf_compress": (_u64, [_vp, _u64, ctypes.c_int, _vp, _u64]),
    "bqc_synth_write_sam": (ctypes.c_int, [ctypes.c_char_p, _P(bqc_synth_params), ctypes.c_char_p, _vp, _u64]),
}


def load_synth():
    """Load libbamqc_synth.so (generator only: no CUDA, no product code)."""
    global _SYNTH
    if _SYNTH is not None:
        return _SYNTH
    path = os.path.join(_HERE, "libbamqc_synth.so")
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `make -C bamqc_b200/csrc`")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SYNTH_PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _SYNTH = lib
    return lib


def load_library():
    """Load libbamqc_b200.so and attach prototypes.  Raises if it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C bamqc_b200/csrc).  bamqc_b200 has no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
