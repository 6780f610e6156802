/* bamqc_b200.h -- C ABI of the B200-native per-record statistics engine for BamQC's `bamqualcheck`.
 *
 * The reference (DecodeGenetics/BamQC) has no plugin / FFI interface: the statistics pass is the body of
 * the `while (!atEnd(inStream))` loop in src/bamqualcheck.cpp:303-444, with state `struct Counts`
 * (src/bamqualcheck.cpp:14-38) and output writeOutput() (src/bamqualcheck.cpp:156-233).  This header is the
 * seam a maintainer would cut there (SURVEY.md section 8b): the host keeps BGZF inflate, header parsing and
 * FASTA loading; whole inflated BAM records go in; per-lane count tables come out.  Plain pointers and
 * sizes only; every function returns 0 on success unless stated otherwise.  INTEGRATION.md shows the
 * reference-side stub.
 *
 * Threading: calls on one engine are not re-entrant (one submit thread per engine); any number of host
 * threads may fill staging buffers.  One engine drives one GPU.
 */
#ifndef BAMQC_B200_H_
#define BAMQC_B200_H_
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct bqc_engine bqc_engine;
typedef struct bqc_batch bqc_batch; /* a record batch resident in HBM (kernel-only timing, replay) */

/* Error codes (bqc_error_info.code); 1-3 are the reference's own fatal conditions. */
enum {
    BQC_OK = 0,
    BQC_ERR_RG_NOT_Z = 1,       /* src/bamqualcheck.cpp:81-97,315  "Read does not have Z"            */
    BQC_ERR_NO_MATE_FLAG = 2,   /* src/bamqualcheck.cpp:385-389    "No first or second flag in read" */
    BQC_ERR_AS_TAG = 3,         /* src/TripletCounting.hpp:116-127,155  missing / unreadable / negative AS */
    BQC_ERR_BAD_RECORD = 4,     /* src/bamqualcheck.cpp:306-310    record does not parse               */
    BQC_ERR_NO_RG = 5,          /* record without RG tag (undefined behaviour in the reference)      */
    BQC_ERR_UNSUPPORTED = 16,   /* value outside the engine's fixed table capacities (see config)    */
    BQC_ERR_CUDA = 32,          /* CUDA runtime failure; bqc_last_error() has the text               */
    BQC_ERR_ARG = 33
};

/* Configuration == ProgramOptions (src/CommandLineParser.hpp:13-41) + header-derived tables
 * (lane map src/bamqualcheck.cpp:44-66,286; main-chromosome set :106-123,292). */
typedef struct bqc_config {
    int32_t device;               /* CUDA device ordinal */
    int32_t isize;                /* -i: insert-size histogram upper bound (default 1000) */
    int32_t n_lanes;              /* number of @RG lines, lane index = order of appearance */
    const char* const* lane_ids;  /* n_lanes RG ID strings */
    int32_t n_ref;                /* number of BAM reference sequences */
    const uint8_t* main_chrom;    /* n_ref bytes: 1 if the reference is in the -c set */
    int32_t n_k;                  /* -k list */
    const int32_t* klist;
    int32_t n_q;                  /* -q list */
    const uint64_t* q_cutoff;
    uint32_t q_base;              /* 33 */
    double e;                     /* -e (sketch geometry, src/kmerstream/StreamCounter.hpp:25-43) */
    int32_t seed;                 /* -s (RepHash table, src/kmerstream/RepHash.cpp:4-17); 0 is rejected */
    int32_t max_read_len;         /* initial per-cycle table capacity; 0 => 512.  The tables grow with the longest read seen, like
                                     the reference's String<>s (src/QualityCheck.hpp:85-109), up to 1800 (what k_stats can keep in shared memory); beyond => BQC_ERR_UNSUPPORTED */
    uint64_t staging_bytes;       /* capacity of each pinned staging buffer; 0 => 256 MiB */
    uint32_t cov_ring_log2;       /* unused (the coverage statistic no longer keeps a depth ring); kept for ABI stability */
    int32_t host_threads;         /* host threads of the framing pre-pass of host-framed submissions; 0 => min(16, cores) */
} bqc_config;

typedef struct bqc_error_info {
    int32_t code;       /* BQC_ERR_* */
    uint64_t record;    /* global index (submission order) of the first offending record */
    char message[256];  /* the reference's message for codes 1-3 */
} bqc_error_info;

/* ---- lifetime -------------------------------------------------------------------------------- */
int bqc_create(const bqc_config* cfg, bqc_engine** out);
void bqc_destroy(bqc_engine* e);
const char* bqc_last_error(bqc_engine* e); /* text of the last failure on this engine (or global if NULL) */

/* Reference genome, 2-bit packed (base i in byte i/4, bits 2*(i%4); A=0 C=1 G=2 T=3; N packed as A,
 * which is what Dna5->Dna conversion does at src/TripletCounting.hpp:228).  Replaces the streaming FASTA
 * cursor of src/TripletCounting.hpp:60-104,254-259.  Copies host -> HBM. */
int bqc_set_reference(bqc_engine* e, int32_t rid, const uint8_t* packed2bit, uint64_t n_bases);

/* Zero every statistic (start of a run).  The reference genome stays resident. */
int bqc_reset(bqc_engine* e);

/* ---- streaming path (host buffers; replaces the loop body src/bamqualcheck.cpp:313-443) ------- */
/* Borrow a pinned staging buffer (blocks until the GPU has finished with it). */
int bqc_acquire_staging(bqc_engine* e, void** pinned, size_t* capacity);
/* Submit n_bytes of whole inflated BAM records (block_size prefixes included) that start at `data`.
 * `data` may be a staging buffer from bqc_acquire_staging (zero extra copies) or any host memory.
 * record_offsets (n_records+1 entries) may be NULL: the engine then frames the records itself (on the device;
 * n_bytes must end on a record boundary).
 * Asynchronous: returns once the copies and kernels are enqueued. */
int bqc_submit(bqc_engine* e, const void* data, size_t n_bytes, const uint64_t* record_offsets, uint64_t n_records);
/* Submit the next n_bytes of the inflated record stream; chunks need not end on record boundaries (what
 * readRecord() hides at src/bamqualcheck.cpp:306).  The partial record at the end of a chunk is carried into the
 * next one on the device; the records are framed on the device (speculated window starts, verified against the
 * sequential chain; kernel_frame.cuh).  `last` != 0 marks the end of the stream: a trailing partial record is then
 * the reference's "Could not read record" error (BQC_ERR_BAD_RECORD).  With several read groups the lane of every
 * record is looked up from its RG tag on the device as well.  BQC_HOST_FRAMING=1 in the environment switches to the
 * host framer (same results). */
int bqc_submit_stream(bqc_engine* e, const void* data, size_t n_bytes, int last);
/* Submit whole BGZF blocks (the compressed bytes of a .bam file) -- SURVEY section 8f rank 1: the blocks are copied
 * to the device as they are, inflated there (one warp per block, kernel_inflate.cuh) and the inflated stream then
 * takes the bqc_submit_stream path on the device.  data must start at a block boundary and hold whole blocks; any
 * size (the call splits it to the staging capacity).  skip_bytes: inflated bytes at the front that are not records
 * (the BAM header, for the first call of a file).  With BQC_HOST_FRAMING=1 the blocks are
 * inflated with zlib on the host threads instead (same results). */
int bqc_submit_bgzf(bqc_engine* e, const void* data, size_t n_bytes, size_t skip_bytes, int last);
/* A later piece of a file that was cut at BGZF block boundaries begins somewhere inside a record.  Called before the
 * first submission, bqc_stream_unknown_start makes the engine look for the first record boundary itself (the first
 * position from which six records in a row are plausible); bqc_stream_skipped then tells how many inflated bytes lie in
 * front of it -- they are the end of the previous piece's last record and have to be submitted there
 * (bqc_submit_stream(..., last = 1)); that piece ending exactly on a record boundary is the proof that the guess was
 * right (otherwise it reports BQC_ERR_BAD_RECORD and the caller falls back to a single stream). */
int bqc_stream_unknown_start(bqc_engine* e);
int bqc_stream_skipped(bqc_engine* e, uint64_t* skipped);   /* 0: known; -1: the first submission has not been framed yet (poll; may be
                                                               called from another thread); > 0: the engine's error code */
/* ---- SAM text -------------------------------------------------------------------------------------
 * The @SQ names in header order (n == cfg.n_ref), for RNAME/RNEXT: the first of duplicate names wins, an unknown name
 * is -1.  Call it before the first SAM submission. */
int bqc_set_ref_names(bqc_engine* e, int32_t n, const char* const* names);
/* Submit SAM alignment lines (no '@' header lines), asynchronously like bqc_submit_stream; pinned or pageable memory,
 * at most the staging capacity.  The text must end at a line end unless `last` is set (then a final line without
 * '\n' counts); otherwise BQC_ERR_ARG.  Empty lines are skipped and a trailing '\r' is dropped.  The lines are encoded
 * to BAM records on the device; a submission holding a line outside the device's grammar (B arrays, for one; see
 * csrc/sam_parse.h) is encoded on the host instead, with the same records.  A line the encoder rejects is
 * BQC_ERR_BAD_RECORD at that line's record index; the records in front of it still run. */
int bqc_submit_sam(bqc_engine* e, const void* text, size_t n, int last);
/* The BAM records (block_size included, back to back) that bqc_submit_sam would count for text[0..n), copied into
 * out[0..cap).  Synchronous; counts nothing.  On BQC_ERR_BAD_RECORD *n_records is the index of the rejected line's
 * record and out holds the records in front of it. */
int bqc_sam_to_bam(bqc_engine* e, const void* text, size_t n, uint8_t* out, uint64_t cap, uint64_t* n_bytes, uint64_t* n_records);
/* Non-empty lines encoded on the host so far (submissions that fell back, by bqc_submit_sam or bqc_sam_to_bam). */
uint64_t bqc_sam_host_lines(bqc_engine* e);

/* Number of stream buffers whose speculative framing failed verification and were re-framed sequentially. */
uint64_t bqc_frames_repaired(bqc_engine* e);
/* Records submitted so far (waits for the submissions in flight to be framed). */
uint64_t bqc_records_seen(bqc_engine* e);

/* ---- resident path (records already in HBM; kernel-only timing and replay) --------------------- */
int bqc_batch_prepare(bqc_engine* e, const void* data, size_t n_bytes, const uint64_t* record_offsets,
                      uint64_t n_records, bqc_batch** out);
int bqc_batch_run(bqc_engine* e, bqc_batch* b); /* enqueue the statistics kernels for b; batches must be
                                                   run in the order they were prepared after a bqc_reset */
void bqc_batch_free(bqc_engine* e, bqc_batch* b);
uint64_t bqc_batch_records(const bqc_batch* b);
uint64_t bqc_batch_bytes(const bqc_batch* b);

/* ---- completion -------------------------------------------------------------------------------- */
int bqc_sync(bqc_engine* e);             /* wait for all enqueued work; returns sticky error code if any */
void* bqc_stream(bqc_engine* e);         /* cudaStream_t the kernels run on (for CUDA-event timing) */
uint64_t bqc_kernel_launches(bqc_engine* e); /* kernels launched by this engine so far */
int bqc_get_error(bqc_engine* e, bqc_error_info* out); /* sticky device/host error (code 0 if none) */

/* Optional device timing of each kernel family with CUDA events on the compute stream.
 * bqc_profile_read: milliseconds and launch-group counts accumulated since the previous read, per family:
 * 0 k_stats, 1 k_eightmer, 2 k_sketch, 3 coverage kernels, 4 merge/export, 5-6 host framing / header
 * pre-pass of host-framed submissions (wall clock), 7 unused, 8 k_inflate, 9 framing kernels, 10 SAM text kernels. */
void bqc_profile_enable(bqc_engine* e, int on);
int bqc_profile_read(bqc_engine* e, double ms_out[12], uint64_t n_out[12]);

/* End of input: flush the last two coverage windows (src/bamqualcheck.cpp:447-453).  After this the
 * device tables are final for this GPU.  Idempotent until the next bqc_reset. */
int bqc_finish(bqc_engine* e);

/* ---- multi-GPU merge (StreamCounter::join semantics, src/kmerstream/StreamCounter.hpp:95-112) --- */
/* The additive part of the result: one flat uint64 array (all lanes).  Sum across GPUs, import on the
 * root.  dev_* pointers are device pointers on this engine's GPU. */
uint64_t bqc_counters_len(bqc_engine* e);                 /* number of uint64 */
/* The layout of the block depends on the per-cycle capacity, which grows with the longest read an engine has seen:
 * before exporting, bring every engine to the largest capacity of the group (all-reduce max of the capacities).
 * bqc_reserve_read_len grows the capacity to exactly n rounded up to a multiple of 8 (never shrinks it), so an engine
 * reserved to another engine's capacity has the same layout and bqc_counters_len. */
uint32_t bqc_read_len_capacity(bqc_engine* e);
int bqc_reserve_read_len(bqc_engine* e, uint32_t n);
int bqc_counters_export(bqc_engine* e, void* dev_u64);    /* device -> device copy */
int bqc_counters_import(bqc_engine* e, const void* dev_u64);
/* The sketch: one uint8 per 4-bit counter (so that 8 GPUs x 15 fits); import clamps to 15. */
uint64_t bqc_sketch_len(bqc_engine* e);                   /* number of uint8 */
int bqc_sketch_export_u8(bqc_engine* e, void* dev_u8);
int bqc_sketch_import_u8(bqc_engine* e, const void* dev_u8);
/* Same merge inside one process (engines on different GPUs of one box; peer copy + merge kernels). */
int bqc_merge_from(bqc_engine* dst, bqc_engine* src);

/* ---- one record stream cut across several engines (SURVEY 8e "the exception") ---------------------- */
/* Every statistic but one is a sum over records, so engines can take any pieces of the input.  The coverage
 * windows (OverallNumbers::coverage, src/OverallNumbers.hpp:79-135) are anchored by the records before them: an
 * engine that gets a later piece of a coordinate-ordered stream collects the records that take part
 * (bqc_cov_defer) and resolves them once the pieces have told each other where they begin and end:
 *   1. bqc_cov_shard_boundary  -> n, first/last (rid, begin) of the piece;
 *   2. bqc_cov_shard_function  <- the last qualifying record before the piece (from 1.), -> the piece's anchor
 *                                 recurrence as a function of the state at its entry (1002 x uint16);
 *   3. bqc_cov_shard_run       <- the state at its entry (chain the functions of the pieces before it, starting
 *                                 from 0), -> its histogram goes into its own poscov; head/tail/span describe the
 *                                 windows that were open at its entry and at its end;
 *   4. bqc_cov_shards_combine  (host arithmetic, any rank) -> what to add to the SUM of the pieces' poscov tables,
 *                                 including the end-of-run flush (src/bamqualcheck.cpp:447-453); apply it to the
 *                                 merged result with bqc_poscov_adjust.
 * Pieces are numbered in stream order.  With several read groups every lane's records, in file order, are a stream of
 * their own: run steps 1-4 once per lane with the *_lane calls and apply each lane's delta with
 * bqc_poscov_adjust(e, lane, ...).  The calls without a lane are the lane 0 case. */
typedef struct bqc_cov_shard {
    uint64_t n;                  /* records of the piece that take part in the statistic */
    int32_t first_rid, last_rid;
    uint32_t first_b, last_b;
    uint64_t span;               /* virtual coordinate of the window start of the piece's last record */
    int32_t head[2001];          /* own depth (difference array) over the two windows open at its entry */
    int32_t tail[2001];          /* ... open at its end */
} bqc_cov_shard;
int bqc_cov_defer(bqc_engine* e, int on);   /* after bqc_reset, before the first submission.  1: a piece whose entry state is
                                               unknown (records are collected, resolved in step 3); 2: the FIRST piece of the
                                               stream (runs like a normal engine; only the end-of-run flush is left to step 4);
                                               0: back to a stand-alone engine */
int bqc_cov_shard_boundary(bqc_engine* e, bqc_cov_shard* out);
int bqc_cov_shard_function(bqc_engine* e, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint16_t* table1002);
int bqc_cov_shard_run(bqc_engine* e, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint32_t p_in, bqc_cov_shard* out);
int bqc_cov_shard_boundary_lane(bqc_engine* e, int32_t lane, bqc_cov_shard* out);
int bqc_cov_shard_function_lane(bqc_engine* e, int32_t lane, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint16_t* table1002);
int bqc_cov_shard_run_lane(bqc_engine* e, int32_t lane, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint32_t p_in, bqc_cov_shard* out);
void bqc_cov_shards_combine(const bqc_cov_shard* shards, int32_t n_shards, int64_t delta[101]);
int bqc_poscov_adjust(bqc_engine* e, int32_t lane, const int64_t delta[101]);
/* State after a piece whose function is `table1002`, entered in state p (0..1000 or 2000). */
uint32_t bqc_cov_apply(const uint16_t* table1002, uint32_t p);

/* ---- configuration read-back ------------------------------------------------------------------- */
int32_t bqc_n_lanes(bqc_engine* e);
const char* bqc_lane_id(bqc_engine* e, int32_t lane);
void bqc_qk_lists(bqc_engine* e, const int32_t** klist, uint32_t* n_k, const uint64_t** qlist, uint32_t* n_q);

/* ---- results (host side; valid after bqc_finish, until bqc_reset/destroy) ----------------------- */
/* Field ids of the per-lane tables; *_M fields exist per mate (0 = first, 1 = second). */
enum {
    BQC_F_SCALARS = 0,   /* 13: supplementary, duplicates, QCfailed, not_primary_alignment, readcount, totalbps,
                            bothunmapped, firstunmapped, secondunmapped, first_and_or_second_mapped,
                            FF_RR_orientation, properpair_count, auto_properpair_count (OverallNumbers.hpp:12-24) */
    BQC_F_POSCOV,        /* 101 */
    BQC_F_INSERT,        /* isize+1 (first mate only) */
    BQC_F_EIGHTMER,      /* 65536 */
    BQC_F_TRIPLET,       /* 1024: [ctx 64][fwdFirst,fwdSecond,revFirst,revSecond][base 4] */
    BQC_F_READLEN_M, BQC_F_NCOUNT_M, BQC_F_GCCOUNT_M, BQC_F_AVGQUAL_M, BQC_F_MAPQ_M, BQC_F_MISMATCH_M,
    BQC_F_DEL_M, BQC_F_INS_M,
    BQC_F_DNA_A_M, BQC_F_DNA_C_M, BQC_F_DNA_G_M, BQC_F_DNA_T_M, BQC_F_DNA_N_M,
    BQC_F_QUALSUM_M, BQC_F_SC5_M, BQC_F_SC3_M, BQC_F_READNR_M,
    BQC_F_SUMCOUNT_QK,   /* per (q,k): index = qi*n_k+ki passed as `sub` */
    BQC_F_F2TABLE_QK,
    BQC_F__COUNT
};
/* Copy a table to the caller.  `sub` = mate for *_M fields, q*n_k+k index for *_QK fields, else 0.
 * Lengths are trimmed exactly like the reference's growing String<>s (SURVEY Appendix B).
 * out may be NULL to query *n only.  64-bit values; the writer truncates to `unsigned` where the
 * reference declares one. */
int bqc_result_table(bqc_engine* e, int32_t lane, int32_t field, int32_t sub, uint64_t* out, uint64_t cap, uint64_t* n);
/* Sketch of (lane, q, k) as the reference's packed uint64 words (32 levels x size). */
int bqc_result_sketch(bqc_engine* e, int32_t lane, int32_t qk, uint64_t* out, uint64_t cap, uint64_t* n);
/* KmerStream estimators (src/kmerstream/StreamCounter.hpp:114-172,308-317): out4 = sumCount,F0,f1,F2 */
int bqc_result_estimates(bqc_engine* e, int32_t lane, int32_t qk, uint64_t out4[4]);
/* Per-cycle mean quality (src/QualityCheck.hpp:273-279). */
int bqc_result_avgqual(bqc_engine* e, int32_t lane, int32_t mate, double* out, uint64_t cap, uint64_t* n);
/* The `.bamqc` text, byte-compatible with writeOutput() (src/bamqualcheck.cpp:156-233). */
int bqc_write_bamqc(bqc_engine* e, const char* sample_id, const char* path);

/* ---- host front end shared by the CLI and the Python layer ------------------------------------- */
/* Parse an uncompressed BAM header.  Returns bytes consumed (offset of the first record), 0 on error.
 * Outputs are malloc'ed; free with bqc_free(). */
typedef struct bqc_bam_header {
    char* text;          /* SAM header text (NUL terminated) */
    int32_t n_ref;
    char** ref_names;
    int64_t* ref_lengths;
    int32_t n_lanes;     /* @RG ID values in order of appearance (src/bamqualcheck.cpp:44-66) */
    char** lane_ids;
    char* sample_id;     /* last @RG SM */
} bqc_bam_header;
size_t bqc_parse_bam_header(const uint8_t* data, size_t n, bqc_bam_header* out);
/* Parse the header lines ('@' lines) at the front of SAM text into the same structure; *consumed is the length of the
 * header lines (the offset of the first alignment line).  0 on success, BQC_ERR_ARG on a malformed header. */
int bqc_parse_sam_header(const char* text, size_t n, bqc_bam_header* out, size_t* consumed);
void bqc_free_bam_header(bqc_bam_header* h);
/* Find record boundaries in [data, data+n): fills offsets (cap entries) with the start of each whole
 * record plus the end of the last whole one; returns the number of whole records. */
uint64_t bqc_frame_records(const uint8_t* data, size_t n, uint64_t* offsets, uint64_t cap);
/* Same result with `threads` host threads (speculated slice starts, verified when stitching). n_ref bounds
 * the plausible refID range (0 = unknown). */
uint64_t bqc_frame_records_mt(const uint8_t* data, size_t n, uint64_t* offsets, uint64_t cap, int32_t threads, int32_t n_ref);
/* Inflate a BGZF byte range with `threads` host threads.  Returns inflated size, or 0 on error / cap. */
uint64_t bqc_bgzf_inflate(const uint8_t* in, uint64_t n, uint8_t* out, uint64_t cap, int32_t threads);
/* Load a FASTA file and pack contig `name` (id up to first space/tab, src/TripletCounting.hpp:99-102)
 * to 2 bits (N and other non-ACGT -> A).  Returns a handle that serves several contigs. */
typedef struct bqc_fasta bqc_fasta;
bqc_fasta* bqc_fasta_open(const char* path);
int64_t bqc_fasta_contig(bqc_fasta* f, const char* name, const uint8_t** packed); /* length or -1 */
void bqc_fasta_close(bqc_fasta* f);
/* The whole `bamqualcheck` command (same argv as the reference CLI). */
int bqc_main(int argc, const char* const* argv);

#ifdef __cplusplus
}
#endif
#endif /* BAMQC_B200_H_ */
