// engine.cu -- host side of the statistics engine behind include/bamqc_b200.h: device memory, the
// pinned double-buffered staging ring, record framing + the sequential coverage anchor scan
// (src/OverallNumbers.hpp:79-110), kernel launches, the end-of-run merge helpers and result access.
//
// There is deliberately no CPU implementation of the statistics here: if CUDA is unavailable
// bqc_create() fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <random>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/bamqc_b200.h"
#include "kernels.cuh"
#include "kernel_frame.cuh"
#include "kernel_inflate.cuh"
#include "kernel_sam.cuh"
#include "sam_text.h"

using namespace bqc;

static thread_local std::string g_last_error;

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t err__ = (call);                                                                \
        if (err__ != cudaSuccess) {                                                                \
            set_error(e, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__); \
            return BQC_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

// Persistent host worker pool (framing and the scan pre-pass run once per staging buffer; spawning threads
// every time costs more than the work for small buffers).
class HostPool {
   public:
    explicit HostPool(int workers) {
        for (int i = 0; i < workers; ++i) th_.emplace_back([this] { loop(); });
    }
    ~HostPool() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; ++gen_; }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    // run fn(0..n-1) on the workers and the calling thread; returns when all are done
    void run(int n, const std::function<void(int)>& fn) {
        if (n <= 1 || th_.empty()) { for (int i = 0; i < n; ++i) fn(i); return; }
        {
            std::lock_guard<std::mutex> g(m_);
            fn_ = &fn; n_ = n; next_ = 0; done_ = 0; ++gen_;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> g(m_);
        cv_done_.wait(g, [this] { return done_ == n_; });
        fn_ = nullptr;
    }
   private:
    void work() {
        for (;;) {
            int i;
            const std::function<void(int)>* f;
            { std::lock_guard<std::mutex> g(m_); if (!fn_ || next_ >= n_) return; i = next_++; f = fn_; }
            (*f)(i);
            { std::lock_guard<std::mutex> g(m_); if (++done_ == n_) cv_done_.notify_all(); }
        }
    }
    void loop() {
        uint64_t seen = 0;
        for (;;) {
            { std::unique_lock<std::mutex> g(m_); cv_.wait(g, [&] { return gen_ != seen; }); seen = gen_; if (stop_) return; }
            work();
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_, cv_done_;
    const std::function<void(int)>* fn_ = nullptr;
    int n_ = 0, next_ = 0, done_ = 0;
    uint64_t gen_ = 0;
    bool stop_ = false;
};
static void run_parallel(HostPool* pool, int n, const std::function<void(int)>& fn) {
    if (pool) { pool->run(n, fn); return; }
    std::vector<std::thread> th;
    for (int t = 1; t < n; ++t) th.emplace_back(fn, t);
    if (n > 0) fn(0);
    for (auto& t : th) t.join();
}

struct DeviceBatch {
    uint8_t* bytes = nullptr;        // allocation: kFrameHead bytes of head room, then the staged data
    const uint8_t* base = nullptr;   // what the record offsets are relative to (bytes + kFrameHead when the host framed, bytes when the device did)
    uint32_t* offsets = nullptr;
    uint8_t* rec_lane = nullptr;
    uint32_t* lane_index = nullptr;  // several read groups: record indices grouped by lane + where each lane's list starts
    uint32_t* lane_range = nullptr;
    unsigned long long* lane_lb = nullptr;   // look-back states + ticket of k_lane_partition
    uint64_t lane_lb_bytes = 0;
    uint64_t n_records = 0, n_bytes = 0;
    uint32_t max_lseq = 0;
    uint64_t first_record = 0;
    bool owns = false;
    uint64_t records_after = 0;      // records seen once this batch has run (resident path replays)
};
struct bqc_batch {
    DeviceBatch d;
};

struct Slot {  // one half of the staging double buffer
    uint8_t* pinned = nullptr;
    uint32_t* h_offsets = nullptr;
    uint8_t* h_lane = nullptr;
    DeviceBatch dev;
    cudaEvent_t done = nullptr;
    bool in_flight = false;
    bool queued = false;           // handed to the commit thread, not yet enqueued on the GPU
    // device framing (kernel_frame.cuh)
    FrameResult* h_frame = nullptr;  // pinned
    FrameResult* d_frame = nullptr;
    uint32_t *d_ws = nullptr, *d_we = nullptr, *d_wc = nullptr, *d_ws2 = nullptr, *d_we2 = nullptr, *d_wc2 = nullptr, *d_bsum = nullptr, *d_bbase = nullptr;
    cudaEvent_t framed = nullptr;
    cudaEvent_t inflated = nullptr;    // k_inflate of this slot finished (recorded on its inflate stream)
    // device inflate (kernel_inflate.cuh)
    uint8_t* d_cin = nullptr;          // compressed BGZF bytes of the submission
    InflateBlock* h_blocks = nullptr;  // pinned
    InflateBlock* d_blocks = nullptr;
    uint32_t* d_ictl = nullptr;        // ticket, error
    // SAM text (kernel_sam.cuh), allocated on the first SAM submission: the text, its line ends, the packed per-line
    // sizes and their tile sums, and a batch with room for the encoded records (up to twice the text)
    uint8_t* d_text = nullptr;
    uint32_t* d_lend = nullptr;
    unsigned long long *d_sz = nullptr, *d_sbsum = nullptr;
    SamCtl* d_sctl = nullptr;
    DeviceBatch sam;
};

struct bqc_engine {
    bqc_config cfg;
    std::vector<std::string> lane_ids;
    std::unordered_map<std::string, uint32_t> lane_map;
    std::vector<uint8_t> main_chrom;
    std::vector<int32_t> klist;
    std::vector<uint64_t> qlist;
    Layout L;
    int n_sm = 0;
    uint32_t n_lanes = 1, n_qk = 1;
    uint64_t sketch_words_per_qk = 0;  // uint32 words
    uint64_t staging_bytes = 0, max_records_per_slot = 0;

    // device state
    uint64_t* d_counters = nullptr;
    uint32_t* d_sketch = nullptr;
    // coverage (kernel_cov.cuh): carried anchor state + the two open windows per lane, scratch for the batch in flight
    CovCarry* d_cov_carry = nullptr;   // [n_lanes]
    int32_t* d_cov_d = nullptr;        // [n_lanes][2][kCovD]
    uint8_t* d_cov_scratch = nullptr;  // one allocation, carved by ensure_cov_scratch
    uint64_t cov_scratch_cap = 0;      // records
    uint8_t* d_cov_q = nullptr;        // the compact qualifying records (rid, begin, interval, record index)
    uint64_t cov_q_cap = 0;
    bool cov_deferred = false;         // shard mode: records are collected, the statistic is resolved by bqc_cov_shard_*
    bool cov_head_piece = false;       // shard mode of the FIRST piece of a stream: its entry state is known, so it runs like a
                                       // normal engine; only the end-of-run flush is left to bqc_cov_shards_combine
    uint64_t cov_acc_bound = 0;        // shard mode: upper bound of the records collected so far
    uint8_t* d_cov_lq = nullptr;       // shard mode, several lanes: the collected records grouped by lane (rid, begin, interval),
    std::vector<uint32_t> cov_lane_range;  // ... lane l owns [range[l], range[l + 1]); empty until cov_lane_split, freed by bqc_reset
    uint16_t* d_cov_fn = nullptr;      // shard mode: [1024] shard function; [2048 int32] head
    uint64_t cov_ctl_bytes = 0;        // tickets + look-back states at the front of the scratch (zeroed per launch group)
    CovScratch cov_scratch = {};
    unsigned long long* d_error = nullptr;
    const uint32_t** d_ref = nullptr;
    uint64_t* d_ref_len = nullptr;
    uint8_t* d_main_chrom = nullptr;
    HashTables* d_hash = nullptr;  // one per k
    char* d_lane_names = nullptr;      // @RG IDs back to back + their offsets (k_frame_lanes)
    uint32_t* d_lane_off = nullptr;
    std::vector<uint32_t*> ref_bufs;
    std::vector<uint64_t> ref_len;
    cudaStream_t compute = nullptr, copy = nullptr, covs = nullptr;  // covs: coverage scatter + flush (HBM bound) overlaps the table kernels
    cudaStream_t frames = nullptr; // framing kernels: the H2D copy of the next buffer (copy stream) overlaps them
    // k_inflate: consecutive submissions alternate between two streams.  One warp inflates one BGZF block from start to
    // end (~6 ms for 64 KiB), and a 256 MB submission holds about as many blocks as the GPU has warp slots, so a launch
    // alone ends in a long tail of half-empty SMs; the next submission's launch fills it.
    cudaStream_t inflates[2] = {nullptr, nullptr};
    cudaEvent_t cov_done = nullptr, cov_go = nullptr;
    static const int kSlots = 4;  // depth of the staging pipeline: framing / anchor pass / H2D / kernels each hold one
    Slot slots[kSlots];
    int next_slot = 0;
    cudaEvent_t copied = nullptr;

    // host state
    std::vector<uint64_t> frame_offsets;
    int host_threads = 1;
    std::unique_ptr<HostPool> pool;
    // streaming path: the caller thread frames and pre-scans buffer i+1 while the commit thread runs the
    // sequential anchor pass, the H2D copies and the kernel launches of buffer i
    struct Task {
        int slot; const uint8_t* h2d_src; size_t span; uint64_t n_records; uint32_t max_lseq;
        int mode;          // 0: framed by the host (offsets + meta in the slot), 1: raw stream bytes, framed on the device,
                           // 2: BGZF blocks, inflated and framed on the device, 3: SAM text, encoded on the device
        uint32_t n_blocks = 0, inflated = 0, skip = 0;  // mode 2: BGZF blocks, their total inflated size, leading non-record bytes;
                                                        // mode 3: skip = 1 when the last line has no newline
        bool seek = false;  // the stream starts inside a record: find the first record boundary (k_frame_seek)
        bool must_align;   // the bytes must end on a record boundary (whole-record submissions, last stream chunk)
    };
    std::deque<Task> ingest;       // stream tasks whose H2D copy + framing kernels are enqueued, not yet launched
    int last_stream_slot = -1;     // slot of the previous stream submission (source of the carried partial record)
    bool stream_seek = false;      // bqc_stream_unknown_start: the next stream submission starts inside a record
    std::atomic<int64_t> stream_skipped{-1};   // bytes in front of the first record boundary that was found (-1: not known yet)
    bool device_framing = true;    // BQC_HOST_FRAMING=1 turns it off (A/B tests)
    bool trace = false;            // BQC_TRACE=1: per-buffer timings of the commit thread on stderr
    bool force_bad_frames = false; // BQC_FRAME_FORCE_REPAIR=1: every speculation is treated as failed (tests the repair path)
    std::vector<uint8_t> host_carry;  // partial record carried between stream submissions when the host frames
    std::thread commit_thread;
    std::mutex cm;
    std::condition_variable ccv, ccv_idle;
    std::deque<Task> cq;
    bool cstop = false, cbusy = false;
    int async_rc = 0;
    int tune_stats_bps = 0, tune_sketch_threads = 1024, tune_stats_stage = 1;  // BQC_STATS_STAGE=0: k_stats reads records straight from global memory (A/B tests)
    int tune_sketch_v2 = 3;   // BQC_SKETCH_V2: 0 = k_sketch32 of round 1 (per-base ballot, pair table), 1/2/3/4 = k_sketch32v2 with
                              // 1024/512/640/768 threads per CTA (64/88/86/80 registers).  Measured per 10 M cfg2 records (serialised):
                              // 6.2 / 7.3 / 4.85 / 4.55 / 7.25 ms -- the restructured kernel needs ~86 registers to keep its loads in flight.
                              // With SEQ/QUAL streamed as aligned 8-byte words (each sector fetched 4x instead of 8-16x): 3.96 ms at 640
                              // threads (94 registers), 4.06 at 512, 7.6 at 768 (80 registers: spills the stream)
    int tune_lane_index = 1;  // BQC_LANE_INDEX=0: every lane's pass filters the whole batch (round 1 behaviour, A/B)
    int tune_inflate_streams = 2;                        // BQC_INFLATE_STREAMS=1: every k_inflate on the framing stream (one launch at a time), A/B
    int tune_cov_bps = 6;                                // BQC_COV_BPS: k_cov_tiles CTAs per SM
    int tune_cov_overlap = 2;                            // BQC_COV_OVERLAP: 1 = coverage kernels on their own stream next to the table kernels, 0 = on the
                                                         // compute stream, 2 = by batch size.  Measured on one box, kernel-only M records/s, one resident batch
                                                         // of 64 / 128 / 256 / 512 / 1024 / 2048 MB: own stream 469 / 587 / 678 / 732 / 785 / 806, compute stream
                                                         // 416 / 540 / 643 / 728 / 794 / 823; three 1 GB batches (cfg 2): 12.0 ms on one stream, 12.5 on two
    int tune_tickets = 1;                                // BQC_TICKETS: 1 = the persistent table kernels take warps of 32 records from ticket counters, 0 = static
                                                         // grid-stride split, 2 = tickets for k_eightmer / k_sketch32v2 only.  cfg 2, same box: 11.50 ms (1) vs 12.16
                                                         // (0) per 10 M records; cfg 3 at 30x on 2-8 GPUs: k_stats 9 % slower with tickets (DESIGN.md 3.1)
    uint32_t* d_tab_tickets = nullptr;                   // [256] work counters of the table kernels (kernels.cuh BatchView::tickets)
    bool cov_overlap_now = false;                        // decision for the batch in flight (run_device_batch)
    uint64_t records_seen = 0, frames_repaired = 0;
    std::atomic<uint64_t> launches{0};   // kernels launched (commit thread, anchor thread, caller)
    bool finished = false;
    std::string last_error;
    bqc_error_info host_error = {0, 0, {0}};
    int stats_blocks_per_sm = 0;

    // optional per-kernel-family timing (CUDA events on the compute stream)
    bool profiling = false;
    bool prof_serial = false;      // bqc_profile_enable(e, 2): the coverage kernels run on the compute stream so that the per-family
                                   // times do not overlap (exclusive shares for the roofline report); slower than the default
    struct ProfEv { int family; cudaEvent_t a, b; };
    std::mutex prof_m;             // ProfScope is used from the commit and the anchor thread
    std::vector<ProfEv> prof_pending;
    std::vector<cudaEvent_t> prof_pool;
    double prof_ms[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t prof_n[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t blocks_per_slot = 0;  // capacity of the BGZF block table of a slot
    // SAM text: the @SQ names (bqc_set_ref_names) as the host encoder's map and as the device's sorted table
    bool have_sam_refs = false;
    std::map<std::string, int32_t> sam_ref_id;
    char* d_sam_blob = nullptr;
    uint32_t* d_sam_off = nullptr;
    int32_t* d_sam_id = nullptr;
    SamRefs sam_refs = {nullptr, nullptr, nullptr, 0};
    uint64_t sam_line_cap = 0, sam_rec_cap = 0, sam_byte_cap = 0;   // per slot
    std::atomic<uint64_t> sam_host_lines{0};
    int inflate_bps = 0;

    // results (after finish)
    bool have_results = false;
    std::vector<uint64_t> h_counters;
    std::vector<uint32_t> h_sketch;
};

static void set_error(bqc_engine* e, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    if (e) e->last_error = buf;
}

// ------------------------------------------------------------------------------------------------
// RepHash tables (src/kmerstream/RepHash.cpp:4-17, RepHash.hpp:8-13,57-61)
// ------------------------------------------------------------------------------------------------
static const unsigned char kTwin[32] = {0,  20, 2,  7,  4,  5,  6,  3,  8,  9,  10, 11, 12, 13, 14, 15,
                                        16, 17, 18, 19, 1,  21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31};
static void build_hash_tables(int seed, int k, HashTables& T) {
    uint64_t hv[32][2];  // [i][0]=hi [1]=lo
    std::mt19937 mt((uint32_t)seed);  // == MTRand(seed).randInt() (mersennetwister.h); golden-tested
    for (int i = 0; i < 32; ++i) {
        uint64_t a = mt(), b = mt(), c = mt(), d = mt();
        hv[i][0] = (a << 32) | b;
        hv[i][1] = (c << 32) | d;
    }
    auto rotlk = [&](const uint64_t* x, uint64_t* o) {  // fastleftshiftk: 128-bit rotate left by k (1..63)
        o[0] = (x[0] << k) | (x[1] >> (64 - k));
        o[1] = (x[1] << k) | (x[0] >> (64 - k));
    };
    static const char nt16[] = "=ACMGRSVTWYHKDBN";
    auto bitrev4 = [](int n) { return ((n & 1) << 3) | ((n & 2) << 1) | ((n & 4) >> 1) | ((n & 8) >> 3); };
    memset(&T, 0, sizeof(T));
    for (int s = 0; s < 2; ++s)
        for (int n = 0; n < 16; ++n) {
            int ch = nt16[s ? bitrev4(n) : n] & 31;  // reverse reads: IUPAC complement = nibble bit reversal (R7)
            const uint64_t* fwd = hv[ch];
            const uint64_t* twn = hv[kTwin[ch]];
            const uint64_t* hsrc = s ? twn : fwd;  // table feeding the forward state h
            const uint64_t* tsrc = s ? fwd : twn;  // table feeding the twin state ht
            T.t[s][0][n][0] = hsrc[0];
            T.t[s][0][n][1] = hsrc[1];
            rotlk(hsrc, T.t[s][1][n]);
            rotlk(tsrc, T.t[s][2][n]);
            T.t[s][3][n][0] = tsrc[0];
            T.t[s][3][n][1] = tsrc[1];
        }
}

static size_t round_up_pow2(size_t size) {  // StreamCounter.hpp:11-21
    size--;
    size |= size >> 1; size |= size >> 2; size |= size >> 4; size |= size >> 8; size |= size >> 16; size |= size >> 32;
    size++;
    return size;
}

// ------------------------------------------------------------------------------------------------
// create / destroy
// ------------------------------------------------------------------------------------------------
static void free_device_batch(DeviceBatch& d) {
    if (!d.owns) return;
    cudaFree(d.bytes);
    cudaFree(d.offsets);
    cudaFree(d.rec_lane);
    cudaFree(d.lane_index);
    cudaFree(d.lane_range);
    cudaFree(d.lane_lb);
    d = DeviceBatch();
}

extern "C" void bqc_destroy(bqc_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    if (e->commit_thread.joinable()) {
        { std::lock_guard<std::mutex> g(e->cm); e->cstop = true; }
        e->ccv.notify_all();
        e->commit_thread.join();
    }
    if (e->compute) cudaStreamSynchronize(e->compute);
    if (e->copy) cudaStreamSynchronize(e->copy);
    if (e->covs) cudaStreamSynchronize(e->covs);
    if (e->frames) cudaStreamSynchronize(e->frames);
    for (auto& s : e->slots) {
        if (s.pinned) cudaFreeHost(s.pinned);
        if (s.h_offsets) cudaFreeHost(s.h_offsets);
        if (s.h_lane) cudaFreeHost(s.h_lane);
        if (s.h_frame) cudaFreeHost(s.h_frame);
        if (s.h_blocks) cudaFreeHost(s.h_blocks);
        cudaFree(s.d_cin); cudaFree(s.d_blocks); cudaFree(s.d_ictl);
        cudaFree(s.d_frame); cudaFree(s.d_ws); cudaFree(s.d_we); cudaFree(s.d_wc); cudaFree(s.d_ws2); cudaFree(s.d_we2); cudaFree(s.d_wc2); cudaFree(s.d_bsum); cudaFree(s.d_bbase);
        free_device_batch(s.dev);
        cudaFree(s.d_text); cudaFree(s.d_lend); cudaFree(s.d_sz); cudaFree(s.d_sbsum); cudaFree(s.d_sctl);
        free_device_batch(s.sam);
        if (s.done) cudaEventDestroy(s.done);
        if (s.framed) cudaEventDestroy(s.framed);
        if (s.inflated) cudaEventDestroy(s.inflated);
    }
    for (auto p : e->ref_bufs) cudaFree(p);
    cudaFree(e->d_counters);
    cudaFree(e->d_sketch);
    cudaFree(e->d_cov_carry);
    cudaFree(e->d_cov_d);
    cudaFree(e->d_cov_scratch);
    cudaFree(e->d_cov_q);
    cudaFree(e->d_cov_lq);
    cudaFree(e->d_cov_fn);
    cudaFree(e->d_tab_tickets);
    cudaFree(e->d_error);
    cudaFree((void*)e->d_ref);
    cudaFree(e->d_ref_len);
    cudaFree(e->d_main_chrom);
    cudaFree(e->d_hash);
    cudaFree(e->d_lane_names);
    cudaFree(e->d_lane_off);
    cudaFree(e->d_sam_blob); cudaFree(e->d_sam_off); cudaFree(e->d_sam_id);
    if (e->copied) cudaEventDestroy(e->copied);
    if (e->cov_done) cudaEventDestroy(e->cov_done);
    if (e->cov_go) cudaEventDestroy(e->cov_go);
    if (e->covs) cudaStreamDestroy(e->covs);
    if (e->frames) cudaStreamDestroy(e->frames);
    for (auto& st : e->inflates) if (st) cudaStreamDestroy(st);
    if (e->compute) cudaStreamDestroy(e->compute);
    if (e->copy) cudaStreamDestroy(e->copy);
    delete e;
}

extern "C" const char* bqc_last_error(bqc_engine* e) { return e ? e->last_error.c_str() : g_last_error.c_str(); }

static int alloc_device_batch(bqc_engine* e, DeviceBatch& d, uint64_t bytes_cap, uint64_t rec_cap) {
    d.owns = true;
    // head room in front (a carried partial record) and the same slack behind: the host-framed stream path puts the
    // carried bytes in front of a full chunk and copies both to bytes + kFrameHead
    CU(cudaMalloc(&d.bytes, kFrameHead + bytes_cap + kFrameHead + 256));
    CU(cudaMemset(d.bytes, 0, kFrameHead + bytes_cap + kFrameHead + 256));
    d.base = d.bytes + kFrameHead;
    CU(cudaMalloc(&d.offsets, (rec_cap + 1) * sizeof(uint32_t)));
    if (e->n_lanes > 1) {
        CU(cudaMalloc(&d.rec_lane, rec_cap + 1));
        CU(cudaMalloc(&d.lane_index, (rec_cap + 1) * 4));
        CU(cudaMalloc(&d.lane_range, (e->n_lanes + 1) * 4));
        d.lane_lb_bytes = (rec_cap / 1024 + 4) * 8;
        CU(cudaMalloc(&d.lane_lb, d.lane_lb_bytes));
    }
    return 0;
}

static int drain_commits(bqc_engine* e);
extern "C" int bqc_reset(bqc_engine* e) {
    CU(cudaSetDevice(e->cfg.device));
    drain_commits(e);
    e->async_rc = 0;
    CU(cudaStreamSynchronize(e->compute));
    CU(cudaStreamSynchronize(e->copy));
    CU(cudaStreamSynchronize(e->covs));
    CU(cudaStreamSynchronize(e->frames));
    for (auto& st : e->inflates) CU(cudaStreamSynchronize(st));
    e->last_stream_slot = -1;
    e->stream_seek = false;
    e->stream_skipped = -1;
    e->host_carry.clear();
    CU(cudaMemsetAsync(e->d_counters, 0, e->n_lanes * e->L.lane_stride * 8, e->compute));
    CU(cudaMemsetAsync(e->d_sketch, 0, e->n_lanes * e->n_qk * e->sketch_words_per_qk * 4, e->compute));
    // OverallNumbers(): first = true, v1 = v2 = 0 (src/OverallNumbers.hpp:50-57)
    CU(cudaMemsetAsync(e->d_cov_d, 0, (uint64_t)e->n_lanes * 2 * kCovD * 4, e->compute));
    k_cov_init<<<(e->n_lanes + 63) / 64, 64, 0, e->compute>>>(e->d_cov_carry, e->n_lanes);
    CU(cudaMemsetAsync(e->d_error, 0xFF, 8, e->compute));
    CU(cudaStreamSynchronize(e->compute));  // the coverage stream starts from a clean state
    e->records_seen = 0;
    e->cov_acc_bound = 0;
    cudaFree(e->d_cov_lq);
    e->d_cov_lq = nullptr;
    e->cov_lane_range.clear();
    e->finished = false;
    e->have_results = false;
    e->host_error.code = 0;
    for (auto& s : e->slots) s.in_flight = false;
    return 0;
}

extern "C" int bqc_create(const bqc_config* cfg, bqc_engine** out) {
    bqc_engine* e = nullptr;
    if (!cfg || !out) { set_error(nullptr, "bqc_create: null argument"); return BQC_ERR_ARG; }
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) {
        set_error(nullptr, "bqc_create: no CUDA device available (%s); this engine has no CPU fallback", cudaGetErrorString(ce));
        return BQC_ERR_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { set_error(nullptr, "bqc_create: bad device %d", cfg->device); return BQC_ERR_ARG; }
    if (cfg->n_lanes < 1 || cfg->n_k < 0 || cfg->n_q < 0 || cfg->isize < 0) { set_error(nullptr, "bqc_create: bad configuration"); return BQC_ERR_ARG; }
    if (cfg->n_lanes > 255) { set_error(nullptr, "bqc_create: more than 255 read groups (the per-record lane index is one byte)"); return BQC_ERR_ARG; }
    if (cfg->seed == 0) { set_error(nullptr, "bqc_create: seed 0 (time-based hash seed, src/kmerstream/RepHash.cpp:5-7) is not reproducible and is rejected"); return BQC_ERR_ARG; }
    for (int i = 0; i < cfg->n_k; ++i)
        if (cfg->klist[i] < 1 || cfg->klist[i] > 63) { set_error(nullptr, "bqc_create: k must be in 1..63 (src/kmerstream/RepHash.hpp:34-35)"); return BQC_ERR_ARG; }
    e = new bqc_engine();
    e->cfg = *cfg;
    e->n_lanes = (uint32_t)cfg->n_lanes;
    for (int i = 0; i < cfg->n_lanes; ++i) {
        e->lane_ids.push_back(cfg->lane_ids ? cfg->lane_ids[i] : "");
        e->lane_map[e->lane_ids.back()] = (uint32_t)i;  // later duplicates overwrite, like laneNames[id] = size
    }
    e->main_chrom.assign(cfg->main_chrom, cfg->main_chrom + cfg->n_ref);
    e->klist.assign(cfg->klist, cfg->klist + cfg->n_k);
    e->qlist.assign(cfg->q_cutoff, cfg->q_cutoff + cfg->n_q);
    e->n_qk = (uint32_t)(cfg->n_k * cfg->n_q);
    // StreamCounter geometry (src/kmerstream/StreamCounter.hpp:25-38)
    double er = cfg->e;
    size_t numcounts = (size_t)(48.0 / (er * er) + 1);
    size_t f2size = round_up_pow2((size_t)(2.0 / (er * er) + 1));
    if (numcounts < 8192) numcounts = 8192;
    size_t sksize = round_up_pow2((numcounts + 15) / 16);
    if (f2size > (1u << 26) || sksize > (1u << 24)) { set_error(e, "bqc_create: -e %g needs tables beyond the supported size", er); delete e; return BQC_ERR_ARG; }
    uint32_t cyc = cfg->max_read_len > 0 ? (uint32_t)cfg->max_read_len : 512u;
    cyc = pad8(cyc);
    e->L = make_layout(cyc, (uint32_t)cfg->isize, e->n_qk, (uint32_t)f2size, (uint32_t)sksize);
    e->sketch_words_per_qk = 32ull * sksize * 2ull;
    e->staging_bytes = cfg->staging_bytes ? cfg->staging_bytes : (256ull << 20);
    if (e->staging_bytes > 0xF0000000ull) e->staging_bytes = 0xF0000000ull;
    e->max_records_per_slot = e->staging_bytes / 36 + 16;  // a record is at least 37 bytes (block_size + 32 fixed + a NUL name)
    e->blocks_per_slot = e->staging_bytes / 4096 + 4096;   // BGZF blocks per submission (larger inputs are split)
    e->sam_line_cap = e->staging_bytes / kSamMinLine + 16;   // a fast SAM line is at least 22 bytes; more lines fall back
    e->sam_rec_cap = e->sam_line_cap;
    e->sam_byte_cap = std::min<uint64_t>(2 * e->staging_bytes, 0xF0000000ull);   // a fast line encodes to at most twice its text
    if (const char* v = getenv("BQC_STATS_BPS")) e->tune_stats_bps = atoi(v);
    if (const char* v = getenv("BQC_STATS_STAGE")) e->tune_stats_stage = atoi(v);
    if (const char* v = getenv("BQC_COV_BPS")) e->tune_cov_bps = std::max(1, std::min(6, atoi(v)));
    if (const char* v = getenv("BQC_HOST_FRAMING")) e->device_framing = atoi(v) == 0;
    if (const char* v = getenv("BQC_TRACE")) e->trace = atoi(v) != 0;
    if (const char* v = getenv("BQC_FRAME_FORCE_REPAIR")) e->force_bad_frames = atoi(v) != 0;
    if (const char* v = getenv("BQC_SKETCH_V2")) e->tune_sketch_v2 = atoi(v);
    if (const char* v = getenv("BQC_COV_OVERLAP")) e->tune_cov_overlap = atoi(v);
    if (const char* v = getenv("BQC_TICKETS")) e->tune_tickets = atoi(v);
    if (const char* v = getenv("BQC_INFLATE_STREAMS")) e->tune_inflate_streams = atoi(v);
    if (const char* v = getenv("BQC_LANE_INDEX")) e->tune_lane_index = atoi(v);
    if (const char* v = getenv("BQC_SKETCH_THREADS")) e->tune_sketch_threads = std::max(32, std::min(1024, atoi(v) & ~31));
    e->host_threads = cfg->host_threads > 0 ? cfg->host_threads : (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    if (e->host_threads > 1) e->pool.reset(new HostPool(e->host_threads - 1));

    int rc = [&]() -> int {
        CU(cudaSetDevice(cfg->device));
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, cfg->device));
        e->n_sm = prop.multiProcessorCount;
        CU(cudaStreamCreateWithFlags(&e->compute, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&e->copy, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&e->covs, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&e->frames, cudaStreamNonBlocking));
        for (auto& st : e->inflates) CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&e->cov_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&e->cov_go, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&e->copied, cudaEventDisableTiming));
        CU(cudaMalloc(&e->d_counters, e->n_lanes * e->L.lane_stride * 8));
        CU(cudaMalloc(&e->d_sketch, std::max<uint64_t>(4, e->n_lanes * e->n_qk * e->sketch_words_per_qk * 4)));
        CU(cudaMalloc(&e->d_cov_carry, e->n_lanes * sizeof(CovCarry)));
        CU(cudaMalloc(&e->d_cov_d, (uint64_t)e->n_lanes * 2 * kCovD * 4));
        CU(cudaMalloc(&e->d_error, 8));
        int nref = std::max(1, cfg->n_ref);
        CU(cudaMalloc((void**)&e->d_ref, nref * sizeof(uint32_t*)));
        CU(cudaMemset((void*)e->d_ref, 0, nref * sizeof(uint32_t*)));
        CU(cudaMalloc(&e->d_ref_len, nref * 8));
        CU(cudaMemset(e->d_ref_len, 0, nref * 8));
        CU(cudaMalloc(&e->d_main_chrom, nref));
        CU(cudaMemset(e->d_main_chrom, 0, nref));
        if (cfg->n_ref) CU(cudaMemcpy(e->d_main_chrom, e->main_chrom.data(), cfg->n_ref, cudaMemcpyHostToDevice));
        e->ref_bufs.assign(nref, nullptr);
        e->ref_len.assign(nref, 0);
        if (e->n_lanes > 1) {
            std::string cat;
            std::vector<uint32_t> off(1, 0);
            for (const std::string& id : e->lane_ids) { cat += id; off.push_back((uint32_t)cat.size()); }
            CU(cudaMalloc(&e->d_lane_names, std::max<size_t>(1, cat.size())));
            CU(cudaMemcpy(e->d_lane_names, cat.data(), cat.size(), cudaMemcpyHostToDevice));
            CU(cudaMalloc(&e->d_lane_off, off.size() * 4));
            CU(cudaMemcpy(e->d_lane_off, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
        }
        if (cfg->n_k) {
            std::vector<HashTables> ht(cfg->n_k);
            for (int i = 0; i < cfg->n_k; ++i) build_hash_tables(cfg->seed, cfg->klist[i], ht[i]);
            CU(cudaMalloc(&e->d_hash, sizeof(HashTables) * cfg->n_k));
            CU(cudaMemcpy(e->d_hash, ht.data(), sizeof(HashTables) * cfg->n_k, cudaMemcpyHostToDevice));
        }
        for (auto& s : e->slots) {
            CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s.framed, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s.inflated, cudaEventDisableTiming));
        }
        // opt in to large dynamic shared memory
        CU(cudaFuncSetAttribute(k_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kInflateStreams * sizeof(InflateTabs))));
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&e->inflate_bps, k_inflate, (int)kInflateWarps * 32, kInflateStreams * sizeof(InflateTabs)));
        if (e->inflate_bps < 1) e->inflate_bps = 1;
        CU(cudaFuncSetAttribute(k_stats<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CU(cudaFuncSetAttribute(k_stats<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CU(cudaFuncSetAttribute(k_stats<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CU(cudaFuncSetAttribute(k_eightmer, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
        CU(cudaFuncSetAttribute(k_sketch<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
        CU(cudaFuncSetAttribute(k_cov_tables, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCovBlockSmem));
        CU(cudaFuncSetAttribute(k_cov_codes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCovCodesSmem));
        CU(cudaFuncSetAttribute(k_sketch32, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024 + (int)sizeof(HashPairTable) + (int)(kSketchThreads / 32 * kSketchQueue * 8)));
        CU(cudaFuncSetAttribute(k_sketch32v2<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sketch32v2_smem(32768u, 1024)));
        CU(cudaFuncSetAttribute(k_sketch32v2<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sketch32v2_smem(32768u, 512)));
        CU(cudaFuncSetAttribute(k_sketch32v2<640>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sketch32v2_smem(32768u, 640)));
        CU(cudaFuncSetAttribute(k_sketch32v2<768>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sketch32v2_smem(32768u, 768)));
        return 0;
    }();
    if (rc) { g_last_error = e->last_error; bqc_destroy(e); return rc; }
    rc = bqc_reset(e);
    if (rc) { g_last_error = e->last_error; bqc_destroy(e); return rc; }
    *out = e;
    return 0;
}

extern "C" int bqc_set_reference(bqc_engine* e, int32_t rid, const uint8_t* packed, uint64_t n_bases) {
    if (rid < 0 || rid >= e->cfg.n_ref) { set_error(e, "bqc_set_reference: rid %d out of range", rid); return BQC_ERR_ARG; }
    CU(cudaSetDevice(e->cfg.device));
    uint64_t words = (n_bases + 15) / 16 + 4;  // +4: the triplet walk may touch one word past the end
    uint32_t* buf = nullptr;
    CU(cudaMalloc(&buf, words * 4));
    CU(cudaMemset(buf, 0, words * 4));
    CU(cudaMemcpy(buf, packed, (n_bases + 3) / 4, cudaMemcpyHostToDevice));
    if (e->ref_bufs[rid]) cudaFree(e->ref_bufs[rid]);
    e->ref_bufs[rid] = buf;
    e->ref_len[rid] = n_bases;
    CU(cudaMemcpy((void*)(e->d_ref + rid), &buf, sizeof(buf), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_ref_len + rid, &n_bases, 8, cudaMemcpyHostToDevice));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// host framing + coverage anchor scan
// ------------------------------------------------------------------------------------------------
static inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }

extern "C" uint64_t bqc_frame_records(const uint8_t* data, size_t n, uint64_t* offsets, uint64_t cap) {
    uint64_t nrec = 0;
    size_t p = 0;
    while (p + 4 <= n) {
        uint32_t bs = rd32(data + p);
        if (bs < 32 || p + 4 + (size_t)bs > n) break;
        if (nrec + 1 >= cap) break;
        offsets[nrec++] = p;
        p += 4 + (size_t)bs;
        // the chain p -> block_size -> next p is a dependent load per record; records of one library have
        // nearly the same size, so the header 24 records ahead is prefetched at the predicted address
        const size_t pf = p + 24 * (4 + (size_t)bs);
        if (pf + 64 < n) {
            __builtin_prefetch(data + pf);
            __builtin_prefetch(data + pf + 64);
        }
    }
    if (cap) offsets[nrec] = p;
    return nrec;
}

// Plausibility of "a record starts at p" (SAM/BAM spec field ranges).  Only used to SPECULATE where a
// thread may start framing; the stitched result is accepted only where the true chain reaches it.
static inline bool plausible_record(const uint8_t* d, size_t n, size_t p, int64_t n_ref) {
    if (p + 36 > n) return false;
    uint32_t bs = rd32(d + p);
    if (bs < 34 || bs > (1u << 28) || p + 4 + (size_t)bs > n) return false;
    int32_t rid = (int32_t)rd32(d + p + 4), pos = (int32_t)rd32(d + p + 8), nrid = (int32_t)rd32(d + p + 24), npos = (int32_t)rd32(d + p + 28);
    if (rid < -1 || rid >= n_ref || nrid < -1 || nrid >= n_ref || pos < -1 || npos < -1) return false;
    uint32_t lname = d[p + 12], ncig = d[p + 16] | (d[p + 17] << 8);
    int32_t lseq = (int32_t)rd32(d + p + 20);
    if (lname < 1 || lseq < 0) return false;
    uint64_t need = 32ull + lname + 4ull * ncig + ((uint64_t)lseq + 1) / 2 + (uint64_t)lseq;
    if (need > bs) return false;
    return d[p + 36 + lname - 1] == 0;
}

// Multi-threaded framing.  The record chain is a dependent load per record (~20 ns each on a host core),
// so T threads frame T slices concurrently from speculated starts (first position whose next 6 hops all look
// like records); the slices are then stitched in order and a slice is accepted only if the chain of the
// previous slice ends exactly on its start -- otherwise the rest is framed sequentially.  The result is
// identical to the sequential walk.
static uint64_t frame_records_mt(const uint8_t* data, size_t n, uint64_t* offsets, uint64_t cap, int threads, int64_t n_ref, HostPool* pool = nullptr) {
    const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, n >> 22));
    if (T <= 1) return bqc_frame_records(data, n, offsets, cap);
    const uint64_t NONE = ~0ull;
    struct Part { uint64_t start, end; std::vector<uint64_t> offs; };
    std::vector<Part> parts((size_t)T);
    auto find_start = [&](int t) {
        Part& P = parts[(size_t)t];
        P.start = NONE;
        if (t == 0) { P.start = 0; return; }
        size_t lo = n * (size_t)t / (size_t)T, hi = std::min(n, lo + (1u << 20));
        for (size_t p = lo; p < hi; ++p) {
            size_t q = p;
            int hops = 0;
            while (hops < 6 && plausible_record(data, n, q, n_ref)) { q += 4 + (size_t)rd32(data + q); ++hops; if (q == n) { hops = 6; break; } }
            if (hops == 6) { P.start = p; return; }
        }
    };
    auto frame_part = [&](int t) {
        Part& P = parts[(size_t)t];
        if (P.start == NONE) return;
        uint64_t stop = n;
        for (int u = t + 1; u < T; ++u)
            if (parts[(size_t)u].start != NONE) { stop = parts[(size_t)u].start; break; }
        P.offs.reserve((size_t)((stop - P.start) / 200 + 16));
        size_t p = (size_t)P.start;
        while (p < stop && p + 4 <= n) {
            uint32_t bs = rd32(data + p);
            if (bs < 32 || p + 4 + (size_t)bs > n) break;
            P.offs.push_back(p);
            p += 4 + (size_t)bs;
            const size_t pf = p + 24 * (4 + (size_t)bs);
            if (pf + 64 < n) { __builtin_prefetch(data + pf); __builtin_prefetch(data + pf + 64); }
        }
        P.end = p;
    };
    run_parallel(pool, T, find_start);
    run_parallel(pool, T, frame_part);
    // stitch
    uint64_t nrec = 0, pos = 0;
    bool ok = true;
    for (int t = 0; t < T && ok; ++t) {
        Part& P = parts[(size_t)t];
        if (P.start == NONE) continue;
        if (P.start != pos) { ok = false; break; }  // speculation missed: the true chain does not land here
        if (nrec + P.offs.size() + 1 >= cap) { ok = false; break; }
        memcpy(offsets + nrec, P.offs.data(), P.offs.size() * 8);
        nrec += P.offs.size();
        pos = P.end;
        if (pos < n) {  // the slice stopped early: either at the next start (fine) or on a bad record
            uint64_t stop = n;
            for (int u = t + 1; u < T; ++u)
                if (parts[(size_t)u].start != NONE) { stop = parts[(size_t)u].start; break; }
            if (pos < stop) { ok = false; break; }
        }
    }
    if (!ok || pos != n) {  // continue sequentially from the last accepted position (rare)
        uint64_t more = bqc_frame_records(data + pos, n - pos, offsets + nrec, cap - nrec);
        for (uint64_t i = 0; i <= more; ++i) offsets[nrec + i] += pos;
        return nrec + more;
    }
    offsets[nrec] = pos;
    return nrec;
}

extern "C" uint64_t bqc_frame_records_mt(const uint8_t* data, size_t n, uint64_t* offsets, uint64_t cap, int32_t threads, int32_t n_ref) {
    return frame_records_mt(data, n, offsets, cap, threads, n_ref > 0 ? n_ref : (1 << 24));
}

// lane of a record from its RG:Z tag (only needed when the header declares several read groups)
static uint32_t host_lane(const bqc_engine* e, const uint8_t* r, uint32_t avail) {
    uint32_t lname = r[12], ncig = r[16] | (r[17] << 8);
    int32_t lseq = (int32_t)rd32(r + 20);
    uint64_t pos = 36ull + lname + 4ull * ncig + ((uint64_t)(lseq > 0 ? lseq : 0) + 1) / 2 + (uint64_t)(lseq > 0 ? lseq : 0);
    while (pos + 3 <= avail) {
        uint8_t k0 = r[pos], k1 = r[pos + 1], ty = r[pos + 2];
        pos += 3;
        uint64_t sz;
        switch (ty) {
            case 'A': case 'c': case 'C': sz = 1; break;
            case 's': case 'S': sz = 2; break;
            case 'i': case 'I': case 'f': sz = 4; break;
            case 'Z': case 'H': { uint64_t q = pos; while (q < avail && r[q]) ++q; sz = q - pos + 1; break; }
            case 'B': { if (pos + 5 > avail) return 0; uint8_t sub = r[pos]; uint32_t cnt = rd32(r + pos + 1); sz = 5ull + (uint64_t)cnt * ((sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4); break; }
            default: return 0;
        }
        if (k0 == 'R' && k1 == 'G') {
            if (ty != 'Z') return 0;
            uint64_t end = std::min<uint64_t>(pos + sz, avail);
            std::string v((const char*)r + pos, (const char*)r + end);
            while (!v.empty() && v.back() == '\0') v.pop_back();
            auto it = e->lane_map.find(v);
            return it == e->lane_map.end() ? 0u : it->second;  // unknown RG aliases lane 0 (laneNames[...] inserts 0)
        }
        pos += sz;
    }
    return 0;
}

// Host pre-pass of a host-framed submission (host threads): touch every record header once; 32-bit offsets, lane
// and longest read.  (The coverage statistic needs nothing from the host any more: kernel_cov.cuh.)
static void host_scan_pass1(bqc_engine* e, const uint8_t* data, const uint64_t* offs, uint64_t n_records, uint32_t* o32, uint8_t* lane_out, uint32_t& max_lseq) {
    max_lseq = 0;
    const uint64_t base_off = offs[0];
    const int T = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)e->host_threads, n_records / 65536));
    std::vector<uint32_t> tmax((size_t)T, 0);
    auto pass1 = [&](int t) {
        uint64_t r0 = n_records * (uint64_t)t / (uint64_t)T, r1 = n_records * (uint64_t)(t + 1) / (uint64_t)T;
        uint32_t mx = 0;
        for (uint64_t r = r0; r < r1; ++r) {
            const uint8_t* p = data + offs[r];
            if (r + 16 < r1) __builtin_prefetch(data + offs[r + 16]);
            o32[r] = (uint32_t)(offs[r] - base_off);
            uint32_t avail = (uint32_t)(offs[r + 1] - offs[r]);
            uint32_t lane = 0;
            if (avail >= 36) {
                int32_t lseq = (int32_t)rd32(p + 20);
                if (lseq > 0 && (uint32_t)lseq > mx) mx = (uint32_t)lseq;
                if (e->n_lanes > 1) lane = host_lane(e, p, avail);
            }
            if (lane_out) lane_out[r] = (uint8_t)lane;
        }
        tmax[(size_t)t] = mx;
    };
    auto t_p1 = std::chrono::steady_clock::now();
    run_parallel(e->pool.get(), T, pass1);
    for (uint32_t v : tmax) max_lseq = std::max(max_lseq, v);
    o32[n_records] = (uint32_t)(offs[n_records] - base_off);
    if (e->profiling) { e->prof_ms[6] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_p1).count(); e->prof_n[6] += 1; }
}

// ------------------------------------------------------------------------------------------------
// per-family kernel timing
// ------------------------------------------------------------------------------------------------
struct ProfScope {  // records an event pair around the launches of one kernel family
    bqc_engine* e;
    bqc_engine::ProfEv ev;
    bool on;
    cudaStream_t st;
    ProfScope(bqc_engine* e_, int family, cudaStream_t stream = nullptr) : e(e_), on(e_->profiling), st(stream ? stream : e_->compute) {
        if (!on) return;
        auto get = [&]() { cudaEvent_t x; if (e->prof_pool.empty()) cudaEventCreate(&x); else { x = e->prof_pool.back(); e->prof_pool.pop_back(); } return x; };
        ev.family = family;
        {
            std::lock_guard<std::mutex> g(e->prof_m);
            ev.a = get();
            ev.b = get();
        }
        cudaEventRecord(ev.a, st);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(ev.b, st);
        std::lock_guard<std::mutex> g(e->prof_m);
        e->prof_pending.push_back(ev);
    }
};
extern "C" void bqc_profile_enable(bqc_engine* e, int on) { e->profiling = on != 0; e->prof_serial = on == 2; }
static inline cudaStream_t cov_stream(bqc_engine* e) {
    if (e->prof_serial || e->tune_cov_overlap == 0) return e->compute;
    return (e->tune_cov_overlap == 1 || e->cov_overlap_now) ? e->covs : e->compute;
}
// Accumulated device time per kernel family since the last call: 0 k_stats, 1 k_eightmer, 2 k_sketch,
// 3 coverage flush (3 kernels per launch group), 4 merge/export.  Synchronises the compute stream.
extern "C" int bqc_profile_read(bqc_engine* e, double ms_out[12], uint64_t n_out[12]) {
    CU(cudaSetDevice(e->cfg.device));
    drain_commits(e);
    CU(cudaStreamSynchronize(e->compute));
    CU(cudaStreamSynchronize(e->covs));
    CU(cudaStreamSynchronize(e->frames));
    for (auto& p : e->prof_pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) { e->prof_ms[p.family] += ms; e->prof_n[p.family] += 1; }
        e->prof_pool.push_back(p.a);
        e->prof_pool.push_back(p.b);
    }
    e->prof_pending.clear();
    for (int i = 0; i < 12; ++i) { ms_out[i] = e->prof_ms[i]; n_out[i] = e->prof_n[i]; e->prof_ms[i] = 0; e->prof_n[i] = 0; }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// kernel launches for one device-resident batch
// ------------------------------------------------------------------------------------------------
// Scratch of the coverage kernels for a batch of up to n records: one allocation, grown on demand (rare: the first
// batch, or a larger resident batch).  Layout: control words that are zeroed before every launch group (tickets,
// look-back states), then the per-record and per-block arrays.  The compact records themselves live in their own
// allocation because shard mode keeps collecting them over the whole run (`keep` entries survive a growth).  With
// several read groups a one-byte lane tag per record follows the four arrays.
static int ensure_cov_q(bqc_engine* e, uint64_t n_records, uint64_t keep) {
    if (n_records <= e->cov_q_cap && e->d_cov_q) return 0;
    const uint64_t N = std::max<uint64_t>(n_records + n_records / 4, 1u << 16);
    const uint64_t tag = e->n_lanes > 1 ? N : 0;
    uint8_t* m = nullptr;
    CU(cudaStreamSynchronize(e->covs));
    CU(cudaMalloc(&m, N * 16 + tag));
    if (e->d_cov_q && keep) {
        for (int a = 0; a < 4; ++a) CU(cudaMemcpy(m + (uint64_t)a * N * 4, e->d_cov_q + (uint64_t)a * e->cov_q_cap * 4, keep * 4, cudaMemcpyDeviceToDevice));
        if (tag) CU(cudaMemcpy(m + N * 16, e->d_cov_q + e->cov_q_cap * 16, keep, cudaMemcpyDeviceToDevice));
    }
    cudaFree(e->d_cov_q);
    e->d_cov_q = m;
    e->cov_q_cap = N;
    CovScratch& S = e->cov_scratch;
    S.q_rid = (int32_t*)m;
    S.q_b = (uint32_t*)(m + N * 4);
    S.q_iv = (uint32_t*)(m + N * 8);
    S.q_rec = (uint32_t*)(m + N * 12);
    S.q_lane = tag ? m + N * 16 : nullptr;
    return 0;
}
static int ensure_cov_scratch(bqc_engine* e, uint64_t n_records) {
    if (n_records <= e->cov_scratch_cap && e->d_cov_scratch) return 0;
    const uint64_t N = std::max<uint64_t>(n_records + n_records / 8, 1u << 16);
    const uint64_t nblk = N / kCovRB + 2, nprep = N / kCovPrepTile + 2, ntile = 2 * N + 16;  // <= 2000 virtual positions per record
    auto up = [](uint64_t x) { return (x + 255) & ~255ull; };
    uint64_t o = 0;
    const uint64_t o_tickets = o; o += up(16);
    const uint64_t o_lbp = o; o += up(nprep * 8);
    const uint64_t o_lbc = o; o += up(nblk * 8);
    const uint64_t ctl = o;
    const uint64_t o_base = o; o += up(N * 8);
    const uint64_t o_ab = o; o += up(N * 4);
    const uint64_t o_tab = o; o += up(nblk * 1024 * 2);
    const uint64_t o_desc = o; o += up(nblk * 16);
    const uint64_t o_state = o; o += up(nblk * 4);
    const uint64_t o_first = o; o += up(ntile * 4);
    CU(cudaStreamSynchronize(e->covs));
    if (e->d_cov_scratch) { cudaFree(e->d_cov_scratch); e->d_cov_scratch = nullptr; e->cov_scratch_cap = 0; }
    CU(cudaMalloc(&e->d_cov_scratch, o));
    uint8_t* m = e->d_cov_scratch;
    CovScratch& S = e->cov_scratch;
    S.tickets = (uint32_t*)(m + o_tickets);
    S.lb_prep = (unsigned long long*)(m + o_lbp);
    S.lb_codes = (unsigned long long*)(m + o_lbc);
    S.base = (unsigned long long*)(m + o_base);
    S.ab = (uint32_t*)(m + o_ab);
    S.tables = (uint16_t*)(m + o_tab);
    S.desc = (uint4*)(m + o_desc);
    S.state_in = (uint32_t*)(m + o_state);
    S.first_rec = (uint32_t*)(m + o_first);
    e->cov_scratch_cap = N;
    e->cov_ctl_bytes = ctl;
    return 0;
}

static EngineView make_view(bqc_engine* e) {
    EngineView E;
    E.L = e->L;
    E.counters = e->d_counters;
    E.sketch = e->d_sketch;
    E.ref = e->d_ref;
    E.ref_len = e->d_ref_len;
    E.main_chrom = e->d_main_chrom;
    E.n_ref = e->cfg.n_ref;
    E.error = e->d_error;
    E.insert_smem = std::min<uint32_t>(pad8(e->L.isize1), 4096u);
    return E;
}

struct BatchLaunch {  // launch geometry shared by the coverage and the table kernels of one batch
    EngineView E;
    uint32_t cycb;
    size_t stats_smem;
    int bps;
    bool staged;
    size_t stats_smem0;   // shared memory of the unstaged kernel (lane-indexed batches)
};

// The reference's per-cycle String<>s grow with the longest read seen (src/QualityCheck.hpp:85-109); here the result
// block has a per-cycle capacity, and a batch with a longer read moves every table to a larger layout before its
// kernels are launched.  The limit is what k_stats can keep in shared memory (per-cycle rows of both mates).
// A batch grows the capacity by at least half, so that a file of slowly increasing read lengths moves the block a few
// times only; `exact` grows to pad8(need) instead, which is how two engines that grew along different steps are brought
// to one layout before their blocks are added (bqc_merge_from, bqc_reserve_read_len).
static const uint32_t kMaxReadLen = 1800;   // 2 mates x 9 padded per-cycle rows + 6 per-read histograms of that length: 216 KB of the 227 KB
static int grow_read_len(bqc_engine* e, uint32_t need, bool exact = false) {
    if (need <= e->L.cyc || need > kMaxReadLen) return 0;   // longer: the kernel reports BQC_ERR_UNSUPPORTED
    CU(cudaSetDevice(e->cfg.device));
    const uint32_t cyc2 = exact ? pad8(need) : std::min<uint32_t>(pad8(kMaxReadLen), pad8(std::max<uint32_t>(need, e->L.cyc + e->L.cyc / 2)));
    const Layout A = e->L, Bn = make_layout(cyc2, A.isize1 - 1, A.n_qk, A.f2size, A.sk_size);
    std::vector<uint3> segs;
    auto seg = [&](uint32_t so, uint32_t d_o, uint32_t n) { segs.push_back(make_uint3(so, d_o, n)); };
    seg(A.o_scalars, Bn.o_scalars, S_COUNT);
    seg(A.o_poscov, Bn.o_poscov, kPoscov);
    seg(A.o_insert, Bn.o_insert, pad8(A.isize1));
    seg(A.o_eightmer, Bn.o_eightmer, kEightmer);
    seg(A.o_triplet, Bn.o_triplet, kTriplet);
    for (uint32_t m = 0; m < 2; ++m) {
        const uint32_t a = A.o_mate0 + m * A.mate_stride, b = Bn.o_mate0 + m * Bn.mate_stride;
        seg(a + A.m_readlen, b + Bn.m_readlen, pad8(A.cyc + 1));
        seg(a + A.m_ncount, b + Bn.m_ncount, pad8(A.cyc + 1));
        seg(a + A.m_gccount, b + Bn.m_gccount, pad8(A.cyc + 1));
        seg(a + A.m_avgq, b + Bn.m_avgq, kQCap);
        seg(a + A.m_ceilq, b + Bn.m_ceilq, kQCap);
        seg(a + A.m_mapq, b + Bn.m_mapq, kMapqCap);
        seg(a + A.m_mismatch, b + Bn.m_mismatch, A.mmcap);
        seg(a + A.m_del, b + Bn.m_del, A.delcap);
        seg(a + A.m_ins, b + Bn.m_ins, A.mmcap);
        for (uint32_t r = 0; r < PC_ROWS; ++r) seg(a + A.m_pc + r * pad8(A.cyc), b + Bn.m_pc + r * pad8(Bn.cyc), pad8(A.cyc));
        seg(a + A.m_readnr, b + Bn.m_readnr, 8);
    }
    seg(A.o_qk, Bn.o_qk, A.n_qk * A.qk_stride);
    uint64_t* d2 = nullptr;
    uint3* dseg = nullptr;
    CU(cudaStreamSynchronize(e->covs));      // the coverage kernels add to poscov in the old block
    CU(cudaStreamSynchronize(e->compute));
    CU(cudaMalloc(&d2, e->n_lanes * Bn.lane_stride * 8));
    CU(cudaMemset(d2, 0, e->n_lanes * Bn.lane_stride * 8));
    CU(cudaMalloc(&dseg, segs.size() * sizeof(uint3)));
    CU(cudaMemcpy(dseg, segs.data(), segs.size() * sizeof(uint3), cudaMemcpyHostToDevice));
    k_relayout<<<dim3(64, (unsigned)segs.size()), 256, 0, e->compute>>>((const unsigned long long*)e->d_counters, (unsigned long long*)d2, dseg, (uint32_t)segs.size(), A.lane_stride,
                                                                        Bn.lane_stride, e->n_lanes);
    e->launches += 1;
    CU(cudaStreamSynchronize(e->compute));
    cudaFree(dseg);
    cudaFree(e->d_counters);
    e->d_counters = d2;
    e->L = Bn;
    e->have_results = false;
    return 0;
}

static int batch_launch_setup(bqc_engine* e, const DeviceBatch& d, BatchLaunch& BL) {
    if (d.max_lseq > e->L.cyc) { int rc = grow_read_len(e, d.max_lseq); if (rc) return rc; }
    BL.E = make_view(e);
    uint32_t cycb = pad8(std::max<uint32_t>(d.max_lseq, 8u));
    if (cycb > e->L.cyc) cycb = e->L.cyc;  // longer reads are reported as unsupported by the kernel
    BL.cycb = cycb;
    StatsSmem S = stats_smem_layout(cycb, BL.E.insert_smem);
    int bps = 0;
    BL.stats_smem0 = (size_t)S.total * 4;
    BL.staged = e->tune_stats_stage != 0 && !(e->n_lanes > 1 && e->tune_lane_index);
    if (BL.staged) {  // the per-warp staging areas on top of the tables: only while both fit
        BL.stats_smem = (size_t)S.stage * 4 + (size_t)(kStatsThreads / 32) * kStatsStage + kStatsMbarBytes;
        if (BL.stats_smem > 227u * 1024u || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_stats<1>, (int)kStatsThreads, BL.stats_smem) != cudaSuccess || bps < 1) {
            cudaGetLastError();
            BL.staged = false;
            bps = 0;
        }
    }
    if (!BL.staged) {
        BL.stats_smem = (size_t)S.total * 4;
        if (BL.stats_smem <= 227u * 1024u) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_stats<0>, (int)kStatsThreads, BL.stats_smem));
    }
    if (bps < 1) { set_error(e, "k_stats does not fit: %zu bytes of shared memory", BL.stats_smem); return BQC_ERR_ARG; }
    if (e->tune_stats_bps > 0 && e->tune_stats_bps < bps) bps = e->tune_stats_bps;
    BL.bps = bps;
    e->stats_blocks_per_sm = bps;
    return 0;
}

// The anchor recurrence, the virtual coordinates and the depth histogram of the records collected in the compact
// arrays of S (a batch, or a whole shard), from the state in CovCarry; n_bound >= the number of compact records.
static int launch_cov_resolve(bqc_engine* e, uint32_t lane, const CovScratch& S, const BatchView& B, uint64_t n_bound, bool tables_done) {
    cudaStream_t cs = cov_stream(e);
    CovCarry* carry = e->d_cov_carry + lane;
    int32_t* cd = e->d_cov_d + (uint64_t)lane * 2 * kCovD;
    unsigned long long* poscov = (unsigned long long*)(e->d_counters + (uint64_t)lane * e->L.lane_stride + e->L.o_poscov);
    const uint32_t nblk = (uint32_t)((n_bound + kCovRB - 1) / kCovRB);
    if (!tables_done) k_cov_tables<<<nblk, kCovBlockThreads, kCovBlockSmem, cs>>>(S, carry);
    k_cov_link<<<1, 1024, 0, cs>>>(S, carry);
    k_cov_codes<<<(int)std::min<uint32_t>(nblk, (uint32_t)e->n_sm * 2u), kCovBlockThreads, kCovCodesSmem, cs>>>(S, carry);
    k_cov_tiles<<<e->n_sm * e->tune_cov_bps, kCovTileThreads, 0, cs>>>(B, S, carry, cd, poscov);
    e->launches += tables_done ? 3 : 4;
    return 0;
}

// OverallNumbers::coverage for one device-resident batch (kernel_cov.cuh), on its own stream so that it overlaps the
// table kernels.  The caller has made e->covs wait for the batch's data.  Nothing comes back to the host: the anchor
// state and the two open windows are carried on the device from batch to batch.  Shard mode only collects the
// records that take part (bqc_cov_shard_* resolve them at the end).
static int launch_cov(bqc_engine* e, const DeviceBatch& d, const BatchLaunch& BL) {
    const uint64_t n = d.n_records;
    cudaStream_t cs = cov_stream(e);
    if (n) {
        int rc = ensure_cov_scratch(e, n);
        if (rc) return rc;
        rc = ensure_cov_q(e, e->cov_acc_bound + n, e->cov_acc_bound);
        if (rc) return rc;
        const CovScratch& S = e->cov_scratch;
        BatchView B;
        B.bytes = d.base;
        B.offsets = d.offsets;
        B.rec_lane = d.rec_lane;
        B.index = (e->n_lanes > 1 && e->tune_lane_index) ? d.lane_index : nullptr;
        B.index_range = d.lane_range;
        B.n_records = (uint32_t)n;
        B.cycb = BL.cycb;
        B.first_record = d.first_record;
        const uint32_t nprep = (uint32_t)((n + kCovPrepTile - 1) / kCovPrepTile);
        const int gprep = (int)std::min<uint32_t>(nprep, (uint32_t)e->n_sm * 2u);
        ProfScope prof(e, 3, cs);
        // shard mode with several read groups: one pass over all lanes into one tagged queue (its running total in
        // carry[0].nq), grouped by lane when the run has ended (cov_lane_split)
        const bool tagged = e->cov_deferred && e->n_lanes > 1;
        if (tagged) {
            CU(cudaMemsetAsync(e->d_cov_scratch, 0, e->cov_ctl_bytes, cs));
            k_cov_prep<true><<<gprep, kCovPrepThreads, 0, cs>>>(BL.E, B, 0, S, e->d_cov_carry, 1u);
            e->launches += 1;
        }
        for (uint32_t lane = 0; lane < e->n_lanes && !tagged; ++lane) {
            CovCarry* carry = e->d_cov_carry + lane;
            CU(cudaMemsetAsync(e->d_cov_scratch, 0, e->cov_ctl_bytes, cs));
            k_cov_prep<false><<<gprep, kCovPrepThreads, 0, cs>>>(BL.E, B, lane, S, carry, e->cov_deferred ? 1u : 0u);
            e->launches += 1;
            if (e->cov_deferred) continue;
            rc = launch_cov_resolve(e, lane, S, B, n, false);
            if (rc) return rc;
            k_cov_carry<<<1, 1024, 0, cs>>>(B, S, carry, e->d_cov_d + (uint64_t)lane * 2 * kCovD);
            e->launches += 1;
        }
        if (e->cov_deferred) e->cov_acc_bound += n;
    }
    CU(cudaEventRecord(e->cov_done, cs));
    CU(cudaGetLastError());
    return 0;
}

static int launch_tables(bqc_engine* e, const DeviceBatch& d, const BatchLaunch& BL) {
    const uint64_t n = d.n_records;
    const EngineView& E = BL.E;
    for (uint32_t lane = 0; lane < e->n_lanes && n; ++lane) {
        // the table kernels see the whole batch once
        BatchView B;
        B.bytes = d.base;
        B.offsets = d.offsets;
        B.rec_lane = d.rec_lane;
        B.index = (e->n_lanes > 1 && e->tune_lane_index) ? d.lane_index : nullptr;
        B.index_range = d.lane_range;
        B.n_records = (uint32_t)n;
        B.cycb = BL.cycb;
        B.first_record = d.first_record;
        if (e->tune_tickets && 2u + e->qlist.size() * e->klist.size() <= 256u) {
            if (!e->d_tab_tickets) CU(cudaMalloc(&e->d_tab_tickets, 256 * 4));
            CU(cudaMemsetAsync(e->d_tab_tickets, 0, 256 * 4, e->compute));
            B.tickets = e->d_tab_tickets;
        }
        int grid = (int)std::min<uint64_t>((n + kStatsThreads - 1) / kStatsThreads, (uint64_t)e->n_sm * BL.bps);
        {
            ProfScope prof(e, 0);
            BatchView Bs = B;
            if (e->tune_tickets == 2) Bs.tickets = nullptr;   // (A/B: tickets for the 8-mer and sketch kernels only)
            if (B.index) k_stats<0><<<grid, kStatsThreads, BL.stats_smem0, e->compute>>>(E, Bs, lane);   // a lane's records are not contiguous: no span to stage
            else if (BL.staged && e->tune_stats_stage == 2) k_stats<2><<<grid, kStatsThreads, BL.stats_smem, e->compute>>>(E, Bs, lane);
            else if (BL.staged) k_stats<1><<<grid, kStatsThreads, BL.stats_smem, e->compute>>>(E, Bs, lane);
            else k_stats<0><<<grid, kStatsThreads, BL.stats_smem, e->compute>>>(E, Bs, lane);
        }
        int g8 = (int)std::min<uint64_t>((n + kEightThreads - 1) / kEightThreads, (uint64_t)e->n_sm);
        if (g8 < 1) g8 = 1;
        { ProfScope prof(e, 1); k_eightmer<<<g8, kEightThreads, 32768 * 4, e->compute>>>(E, B, lane); }
        e->launches += 2;
        for (uint32_t qi = 0; qi < e->qlist.size(); ++qi)
            for (uint32_t ki = 0; ki < e->klist.size(); ++ki) {
                SketchParams SP;
                SP.k = (uint32_t)e->klist[ki];
                SP.q_thresh = (int32_t)(int8_t)(char)(e->cfg.q_base + e->qlist[qi]);
                SP.qk = qi * (uint32_t)e->klist.size() + ki;
                int gs = (int)std::min<uint64_t>((n + kSketchThreads - 1) / kSketchThreads, (uint64_t)e->n_sm);
                ProfScope prof(e, 2);
                if (SP.k == 32u && e->L.f2size <= 32768u && e->tune_sketch_v2 && SP.q_thresh >= 33 && SP.q_thresh <= 127)
                {
                    if (e->tune_sketch_v2 == 2) k_sketch32v2<512><<<(int)std::min<uint64_t>((n + 511) / 512, (uint64_t)e->n_sm), 512, sketch32v2_smem(e->L.f2size, 512), e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                    else if (e->tune_sketch_v2 == 3) k_sketch32v2<640><<<(int)std::min<uint64_t>((n + 639) / 640, (uint64_t)e->n_sm), 640, sketch32v2_smem(e->L.f2size, 640), e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                    else if (e->tune_sketch_v2 == 4) k_sketch32v2<768><<<(int)std::min<uint64_t>((n + 767) / 768, (uint64_t)e->n_sm), 768, sketch32v2_smem(e->L.f2size, 768), e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                    else k_sketch32v2<1024><<<gs, 1024, sketch32v2_smem(e->L.f2size, 1024), e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                }
                else if (SP.k == 32u && e->L.f2size <= 32768u)
                    k_sketch32<<<gs, e->tune_sketch_threads, e->L.f2size * 4 + sizeof(HashPairTable) + kSketchThreads / 32 * kSketchQueue * 8, e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                else if (e->L.f2size <= 32768u)
                    k_sketch<true><<<gs, kSketchThreads, e->L.f2size * 4, e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                else
                    k_sketch<false><<<gs, kSketchThreads, 0, e->compute>>>(E, B, lane, SP, e->d_hash + ki);
                e->launches += 1;
            }
    }
    CU(cudaGetLastError());
    return 0;
}

// coverage first (its own stream, released once the compute stream has reached this batch), then the tables
static int run_device_batch(bqc_engine* e, const DeviceBatch& d) {
    BatchLaunch BL;
    int rc = batch_launch_setup(e, d, BL);
    if (rc) return rc;
    // small batches: the coverage kernels (many short launches) hide behind k_stats; large ones: they only delay the CTAs of
    // the persistent table kernels.  Either way the two streams hand over through cov_go / cov_done.
    e->cov_overlap_now = d.n_bytes < (384ull << 20);
    CU(cudaEventRecord(e->cov_go, e->compute));
    CU(cudaStreamWaitEvent(e->covs, e->cov_go, 0));
    rc = launch_cov(e, d, BL);
    if (rc) return rc;
    rc = launch_tables(e, d, BL);
    if (rc) return rc;
    CU(cudaStreamWaitEvent(e->compute, e->cov_done, 0));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// streaming path
// ------------------------------------------------------------------------------------------------
static int ensure_slot(bqc_engine* e, Slot& s) {
    if (s.pinned) return 0;
    CU(cudaSetDevice(e->cfg.device));
    const uint64_t rc_ = e->max_records_per_slot;
    // kFrameHead bytes of head room in front of the staging area: a carried partial record goes there
    CU(cudaHostAlloc((void**)&s.pinned, kFrameHead + e->staging_bytes + 256, cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&s.h_offsets, (rc_ + 1) * 4, cudaHostAllocDefault));
    if (e->n_lanes > 1) CU(cudaHostAlloc((void**)&s.h_lane, rc_ + 1, cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&s.h_frame, sizeof(FrameResult), cudaHostAllocDefault));
    const uint64_t nwin = (kFrameHead + e->staging_bytes + kFrameWindow - 1) / kFrameWindow + 1;
    const uint64_t nblk = (nwin + kFrameThreads - 1) / kFrameThreads;
    CU(cudaMalloc(&s.d_frame, sizeof(FrameResult)));
    CU(cudaMalloc(&s.d_ws, nwin * 4));
    CU(cudaMalloc(&s.d_we, nwin * 4));
    CU(cudaMalloc(&s.d_wc, nwin * 4));
    CU(cudaMalloc(&s.d_ws2, nwin * 4));
    CU(cudaMalloc(&s.d_we2, nwin * 4));
    CU(cudaMalloc(&s.d_wc2, nwin * 4));
    CU(cudaMalloc(&s.d_bsum, nblk * 4));
    CU(cudaMalloc(&s.d_bbase, nblk * 4));
    CU(cudaMalloc(&s.d_cin, e->staging_bytes + 256));
    CU(cudaMemset(s.d_cin, 0, e->staging_bytes + 256));
    CU(cudaHostAlloc((void**)&s.h_blocks, e->blocks_per_slot * sizeof(InflateBlock), cudaHostAllocDefault));
    CU(cudaMalloc(&s.d_blocks, e->blocks_per_slot * sizeof(InflateBlock)));
    CU(cudaMalloc(&s.d_ictl, 8));
    return alloc_device_batch(e, s.dev, e->staging_bytes, rc_);
}

// Several read groups: group the record indices by lane (k_lane_partition, one cheap pass over the lane bytes per
// lane) on `st`, after rec_lane is there.  n_ptr: device-side record count of a device-framed buffer, or NULL.
static int launch_lane_partition(bqc_engine* e, DeviceBatch& d, const uint32_t* n_ptr, uint64_t n, cudaStream_t st) {
    if (e->n_lanes <= 1 || !e->tune_lane_index) return 0;
    const uint64_t nb = n_ptr ? e->max_records_per_slot : n;
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((nb + 1023) / 1024, (uint64_t)e->n_sm * 2));
    for (uint32_t lane = 0; lane < e->n_lanes; ++lane) {
        CU(cudaMemsetAsync(d.lane_lb, 0, d.lane_lb_bytes, st));
        k_lane_partition<<<grid, 1024, 0, st>>>(d.rec_lane, n_ptr, (uint32_t)n, lane, d.lane_index, d.lane_range, d.lane_lb + 1, (uint32_t*)d.lane_lb);
        e->launches += 1;
    }
    CU(cudaGetLastError());
    return 0;
}

// host-framed task: copies and launches
static int commit_task(bqc_engine* e, const bqc_engine::Task& t) {
    Slot& s = e->slots[t.slot];
    DeviceBatch& d = s.dev;
    const uint64_t n_records = t.n_records;
    d.max_lseq = t.max_lseq;
    d.n_records = n_records;
    d.n_bytes = t.span;
    d.first_record = e->records_seen;
    d.base = d.bytes + kFrameHead;
    CU(cudaMemcpyAsync(d.bytes + kFrameHead, t.h2d_src, t.span, cudaMemcpyHostToDevice, e->copy));
    CU(cudaMemcpyAsync(d.offsets, s.h_offsets, (n_records + 1) * 4, cudaMemcpyHostToDevice, e->copy));
    if (e->n_lanes > 1) {
        CU(cudaMemcpyAsync(d.rec_lane, s.h_lane, n_records, cudaMemcpyHostToDevice, e->copy));
        int rcp = launch_lane_partition(e, d, nullptr, n_records, e->copy);
        if (rcp) return rcp;
    }
    CU(cudaEventRecord(e->copied, e->copy));
    CU(cudaStreamWaitEvent(e->compute, e->copied, 0));
    int rc = run_device_batch(e, d);
    if (rc) return rc;
    CU(cudaEventRecord(s.done, e->compute));
    e->records_seen += n_records;
    return 0;
}

// stream task, stage A: carry the partial record of the previous buffer, copy the new bytes, frame on the device
static int sam_stage_a(bqc_engine* e, const bqc_engine::Task& t);
static int sam_stage_b(bqc_engine* e, const bqc_engine::Task& t);
static int stream_stage_a(bqc_engine* e, const bqc_engine::Task& t) {
    if (t.mode == 3) return sam_stage_a(e, t);
    Slot& s = e->slots[t.slot];
    DeviceBatch& d = s.dev;
    const Slot* prev = e->last_stream_slot >= 0 ? &e->slots[e->last_stream_slot] : nullptr;
    const uint32_t n_new = t.mode == 2 ? t.inflated : (uint32_t)t.span;
    k_frame_tail<<<1, 256, 0, e->frames>>>(prev ? prev->dev.bytes : nullptr, prev ? prev->d_frame : nullptr, d.bytes, s.d_frame, n_new, t.skip);
    if (t.mode == 2) {
        // compressed bytes + block table over PCIe, inflate on the device into the stream region of the buffer
        CU(cudaMemcpyAsync(s.d_cin, t.h2d_src, t.span, cudaMemcpyHostToDevice, e->copy));
        CU(cudaMemcpyAsync(s.d_blocks, s.h_blocks, (size_t)t.n_blocks * sizeof(InflateBlock), cudaMemcpyHostToDevice, e->copy));
        CU(cudaEventRecord(e->copied, e->copy));
        cudaStream_t is = e->tune_inflate_streams > 1 ? e->inflates[t.slot & 1] : e->frames;
        CU(cudaStreamWaitEvent(is, e->copied, 0));
        CU(cudaMemsetAsync(s.d_ictl, 0, 8, is));
        if (t.n_blocks) {
            const int grid = (int)std::min<uint64_t>(((uint64_t)t.n_blocks + kInflateStreams - 1) / kInflateStreams, (uint64_t)e->n_sm * e->inflate_bps);
            ProfScope prof(e, 8, is);
            k_inflate<<<grid, kInflateWarps * 32, kInflateStreams * sizeof(InflateTabs), is>>>(s.d_cin, s.d_blocks, t.n_blocks, d.bytes + kFrameHead, s.d_ictl);
            e->launches += 1;
        }
        if (is != e->frames) {
            CU(cudaEventRecord(s.inflated, is));
            CU(cudaStreamWaitEvent(e->frames, s.inflated, 0));
        }
    } else {
        CU(cudaMemcpyAsync(d.bytes + kFrameHead, t.h2d_src, t.span, cudaMemcpyHostToDevice, e->copy));
        CU(cudaEventRecord(e->copied, e->copy));
        CU(cudaStreamWaitEvent(e->frames, e->copied, 0));
    }
    ProfScope prof_frame(e, 9, e->frames);
    if (t.seek) { k_frame_seek<<<1, 256, 0, e->frames>>>(d.bytes, s.d_frame, std::max(1, e->cfg.n_ref)); e->launches += 1; }
    const uint32_t nwin = (uint32_t)((kFrameHead + (uint64_t)n_new + kFrameWindow - 1) / kFrameWindow);
    const uint32_t nblk = (nwin + kFrameThreads - 1) / kFrameThreads;
    const uint32_t rec_cap = (uint32_t)e->max_records_per_slot;
    k_frame_speculate<<<nblk, kFrameThreads, 0, e->frames>>>(d.bytes, s.d_frame, std::max(1, e->cfg.n_ref), nwin, s.d_ws, s.d_we, s.d_wc);
    for (int round = 0; round < 2; ++round) {  // two Jacobi rounds each way: the final state is back in d_ws/d_we/d_wc
        k_frame_relax<<<nblk, kFrameThreads, 0, e->frames>>>(d.bytes, s.d_frame, nwin, s.d_ws, s.d_we, s.d_wc, s.d_ws2, s.d_we2, s.d_wc2);
        k_frame_relax<<<nblk, kFrameThreads, 0, e->frames>>>(d.bytes, s.d_frame, nwin, s.d_ws2, s.d_we2, s.d_wc2, s.d_ws, s.d_we, s.d_wc);
    }
    k_frame_blocksum<<<nblk, kFrameThreads, 0, e->frames>>>(nwin, s.d_wc, s.d_bsum);
    k_frame_verify<<<1, 1024, 0, e->frames>>>(s.d_frame, nwin, nblk, s.d_ws, s.d_we, s.d_bsum, s.d_bbase, d.offsets, rec_cap, e->force_bad_frames ? 1u : 0u, t.mode == 2 ? s.d_ictl : nullptr);
    k_frame_repair<<<1, 32, 0, e->frames>>>(d.bytes, s.d_frame, e->cfg.n_ref, e->d_main_chrom, d.offsets, nullptr, rec_cap);
    k_frame_emit<<<nblk, kFrameThreads, 0, e->frames>>>(d.bytes, s.d_frame, e->cfg.n_ref, e->d_main_chrom, nwin, s.d_ws, s.d_wc, s.d_bbase, d.offsets, nullptr);
    e->launches += 10;
    if (e->n_lanes > 1) {  // several read groups: the lane of every record, from its RG tag, then the records grouped by lane
        k_frame_lanes<<<e->n_sm * 4, 256, 0, e->frames>>>(d.bytes, s.d_frame, d.offsets, e->d_lane_names, e->d_lane_off, e->n_lanes, d.rec_lane);
        e->launches += 1;
        int rcp = launch_lane_partition(e, d, &s.d_frame->n_records, 0, e->frames);
        if (rcp) return rcp;
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(s.h_frame, s.d_frame, sizeof(FrameResult), cudaMemcpyDeviceToHost, e->frames));
    CU(cudaEventRecord(s.framed, e->frames));
    e->last_stream_slot = t.slot;
    return 0;
}

// stage B: read the frame header back (record count, longest read), launch the coverage and the table kernels
static int stream_stage_b(bqc_engine* e, const bqc_engine::Task& t) {
    if (t.mode == 3) return sam_stage_b(e, t);
    Slot& s = e->slots[t.slot];
    DeviceBatch& d = s.dev;
    auto t_b0 = std::chrono::steady_clock::now();
    CU(cudaEventSynchronize(s.framed));
    auto t_b1 = std::chrono::steady_clock::now();
    const FrameResult fr = *s.h_frame;
    if (fr.inflate_bad) {
        e->host_error.code = BQC_ERR_BAD_RECORD;
        e->host_error.record = e->records_seen;
        snprintf(e->host_error.message, sizeof(e->host_error.message), "ERROR: Could not read record from BAM File (BGZF block %u of the submission does not inflate)", fr.inflate_bad - 1);
        set_error(e, "%s", e->host_error.message);
        return BQC_ERR_BAD_RECORD;
    }
    if (fr.tail_overflow) {
        e->host_error.code = fr.tail_overflow == 2 ? BQC_ERR_ARG : BQC_ERR_BAD_RECORD;
        e->host_error.record = e->records_seen + fr.n_records;
        snprintf(e->host_error.message, sizeof(e->host_error.message), "%s", fr.tail_overflow == 2 ? "too many records for one staging buffer" : "ERROR: Could not read record from BAM File (record chain broken or record larger than 1 MiB)");
        set_error(e, "%s", e->host_error.message);
        return e->host_error.code;
    }
    if (t.must_align && fr.end != fr.total) {
        e->host_error.code = BQC_ERR_BAD_RECORD;
        e->host_error.record = e->records_seen + fr.n_records;
        snprintf(e->host_error.message, sizeof(e->host_error.message), "bqc_submit: bytes do not end on a record boundary");
        set_error(e, "%s", e->host_error.message);
        return BQC_ERR_BAD_RECORD;
    }
    if (fr.repaired) e->frames_repaired += 1;
    if (t.seek) e->stream_skipped = (int64_t)fr.start - (int64_t)kFrameHead - (int64_t)t.skip;
    const uint64_t n = fr.n_records;
    d.max_lseq = fr.max_lseq;
    d.n_records = n;
    d.n_bytes = fr.end - fr.start;
    d.first_record = e->records_seen;
    d.base = d.bytes;
    e->records_seen += n;
    if (n) {
        CU(cudaStreamWaitEvent(e->compute, s.framed, 0));
        int rc = run_device_batch(e, d);
        if (rc) return rc;
        if (e->trace) {
            auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            fprintf(stderr, "[bqc trace] slot %d: repaired %u, wait framed %.2f ms, launches %.2f ms, n=%llu\n", t.slot, fr.repaired, ms(t_b0, t_b1),
                    ms(t_b1, std::chrono::steady_clock::now()), (unsigned long long)n);
        }
    }
    CU(cudaEventRecord(s.done, e->compute));
    return 0;
}

static void commit_loop(bqc_engine* e) {
    cudaSetDevice(e->cfg.device);
    for (;;) {
        bqc_engine::Task t;
        bool have_new = false, have_old = false;
        {
            std::unique_lock<std::mutex> g(e->cm);
            e->ccv.wait(g, [&] { return e->cstop || !e->cq.empty() || !e->ingest.empty(); });
            if (e->cq.empty() && e->ingest.empty()) return;  // stop requested and nothing left
            // keep up to two stream buffers in the copy + framing stage so that the H2D copy of the next buffer
            // overlaps the launches of this one
            // (tasks complete in submission order: a host-framed task waits for the stream tasks before it)
            const bool take_new = !e->cq.empty() && (e->cq.front().mode != 0 ? e->ingest.size() < 2 : e->ingest.empty());
            if (take_new) {
                t = e->cq.front();
                e->cq.pop_front();
                have_new = true;
            } else {
                t = e->ingest.front();
                e->ingest.pop_front();
                have_old = true;
            }
            e->cbusy = true;
        }
        int rc = e->async_rc;
        bool finished_slot = false;
        if (have_new) {
            if (t.mode == 0) {
                if (!rc) rc = commit_task(e, t);
                finished_slot = true;
            }
            else if (!rc) { rc = stream_stage_a(e, t); if (rc) finished_slot = true; }
            else finished_slot = true;
        } else if (have_old) {
            if (!rc) rc = stream_stage_b(e, t);
            finished_slot = true;
        }
        {
            std::lock_guard<std::mutex> g(e->cm);
            if (have_new && t.mode != 0 && !finished_slot) e->ingest.push_back(t);
            if (finished_slot) {
                e->slots[t.slot].queued = false;
                e->slots[t.slot].in_flight = rc == 0;
            }
            e->cbusy = false;
            if (rc && !e->async_rc) e->async_rc = rc;
        }
        e->ccv_idle.notify_all();
    }
}

// wait until the commit thread has enqueued everything handed to it; returns its sticky error
static int drain_commits(bqc_engine* e) {
    std::unique_lock<std::mutex> g(e->cm);
    e->ccv_idle.wait(g, [&] { return e->cq.empty() && e->ingest.empty() && !e->cbusy; });
    return e->async_rc;
}

static int wait_slot(bqc_engine* e, Slot& s) {
    {
        std::unique_lock<std::mutex> g(e->cm);
        e->ccv_idle.wait(g, [&] { return !s.queued; });
    }
    if (s.in_flight) {
        CU(cudaEventSynchronize(s.done));
        s.in_flight = false;
    }
    return 0;
}

extern "C" int bqc_acquire_staging(bqc_engine* e, void** pinned, size_t* capacity) {
    Slot& s = e->slots[e->next_slot];
    int rc = ensure_slot(e, s);
    if (rc) return rc;
    rc = wait_slot(e, s);
    if (rc) return rc;
    *pinned = s.pinned + kFrameHead;
    *capacity = e->staging_bytes;
    return 0;
}

// where the H2D copy of a submission reads from: the caller's page-locked memory directly (it stays unchanged
// until bqc_sync), pageable memory is staged through the slot's pinned buffer before returning
static const uint8_t* h2d_source(bqc_engine* e, Slot& s, const uint8_t* first, size_t span) {
    if (first >= s.pinned && first + span <= s.pinned + kFrameHead + e->staging_bytes + 256) return first;
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, first) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (pinned) return first;
    memcpy(s.pinned + kFrameHead, first, span);
    return s.pinned + kFrameHead;
}

static void enqueue_task(bqc_engine* e, Slot& s, const bqc_engine::Task& t) {
    {
        std::lock_guard<std::mutex> g(e->cm);
        if (!e->commit_thread.joinable()) e->commit_thread = std::thread(commit_loop, e);
        s.queued = true;
        e->cq.push_back(t);
    }
    e->ccv.notify_all();
    e->next_slot = (e->next_slot + 1) % bqc_engine::kSlots;
}

static int submit_host_framed(bqc_engine* e, Slot& s, const uint8_t* src, size_t n_bytes, const uint64_t* record_offsets, uint64_t n_records) {
    std::vector<uint64_t>& own_offsets = e->frame_offsets;
    if (!record_offsets) {
        if (own_offsets.size() < n_bytes / 36 + 2) own_offsets.resize(n_bytes / 36 + 2);
        auto t_f0 = std::chrono::steady_clock::now();
        n_records = frame_records_mt(src, n_bytes, own_offsets.data(), own_offsets.size(), e->host_threads, std::max(1, e->cfg.n_ref), e->pool.get());
        if (e->profiling) { e->prof_ms[5] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_f0).count(); e->prof_n[5] += 1; }
        if (own_offsets[n_records] != n_bytes) {
            e->host_error.code = BQC_ERR_BAD_RECORD;
            e->host_error.record = e->records_seen + n_records;
            set_error(e, "bqc_submit: bytes do not end on a record boundary");
            return BQC_ERR_BAD_RECORD;
        }
        record_offsets = own_offsets.data();
    }
    if (n_records > e->max_records_per_slot) { set_error(e, "bqc_submit: too many records for one staging buffer"); return BQC_ERR_ARG; }
    if (n_records == 0) return 0;
    // the header pre-pass on the caller's thread (+ pool); copies and launches on the commit thread
    bqc_engine::Task t;
    t.slot = e->next_slot;
    t.n_records = n_records;
    t.mode = 0;
    t.must_align = true;
    host_scan_pass1(e, src, record_offsets, n_records, s.h_offsets, e->n_lanes > 1 ? s.h_lane : nullptr, t.max_lseq);
    const uint8_t* first = src + record_offsets[0];
    t.span = (size_t)(record_offsets[n_records] - record_offsets[0]);
    t.h2d_src = h2d_source(e, s, first, t.span);
    enqueue_task(e, s, t);
    return 0;
}

static int submit_common(bqc_engine* e, const void* data, size_t n_bytes, const uint64_t* record_offsets, uint64_t n_records, bool stream, bool last) {
    if (e->finished) { set_error(e, "bqc_submit after bqc_finish (call bqc_reset)"); return BQC_ERR_ARG; }
    if (n_bytes > e->staging_bytes) { set_error(e, "bqc_submit: %zu bytes exceed the staging capacity %llu", n_bytes, (unsigned long long)e->staging_bytes); return BQC_ERR_ARG; }
    if (e->async_rc) return e->async_rc;
    CU(cudaSetDevice(e->cfg.device));
    Slot& s = e->slots[e->next_slot];
    int rc = ensure_slot(e, s);
    if (rc) return rc;
    rc = wait_slot(e, s);
    if (rc) return rc;
    const uint8_t* src = (const uint8_t*)data;
    const bool on_device = !record_offsets && e->device_framing;
    if (on_device) {
        if (n_bytes == 0 && !(stream && last)) return 0;
        bqc_engine::Task t;
        t.slot = e->next_slot;
        t.n_records = 0;
        t.max_lseq = 0;
        t.mode = 1;
        t.seek = e->stream_seek;
        e->stream_seek = false;
        t.must_align = !stream || last;
        t.span = n_bytes;
        t.h2d_src = n_bytes ? h2d_source(e, s, src, n_bytes) : s.pinned + kFrameHead;
        enqueue_task(e, s, t);
        return 0;
    }
    if (!stream) return submit_host_framed(e, s, src, n_bytes, record_offsets, n_records);
    // stream bytes framed by the host (several read groups, or BQC_HOST_FRAMING=1): the partial record at the end
    // of a chunk is kept on the host and put in front of the next chunk inside the pinned buffer's head room
    const size_t carry = e->host_carry.size();
    uint8_t* buf = s.pinned + kFrameHead - carry;
    if (src != s.pinned + kFrameHead) memmove(s.pinned + kFrameHead, src, n_bytes);
    if (carry) memcpy(buf, e->host_carry.data(), carry);
    const size_t filled = carry + n_bytes;
    std::vector<uint64_t>& offs = e->frame_offsets;
    if (offs.size() < filled / 36 + 2) offs.resize(filled / 36 + 2);
    n_records = frame_records_mt(buf, filled, offs.data(), offs.size(), e->host_threads, std::max(1, e->cfg.n_ref), e->pool.get());
    const size_t whole = (size_t)offs[n_records];
    if (filled - whole > kFrameHead || (last && whole != filled)) {
        e->host_error.code = BQC_ERR_BAD_RECORD;
        e->host_error.record = e->records_seen + n_records;
        snprintf(e->host_error.message, sizeof(e->host_error.message), "ERROR: Could not read record from BAM File (record chain broken or record larger than 1 MiB)");
        set_error(e, "%s", e->host_error.message);
        return BQC_ERR_BAD_RECORD;
    }
    e->host_carry.assign(buf + whole, buf + filled);
    if (n_records == 0) return 0;
    return submit_host_framed(e, s, buf, whole, offs.data(), n_records);
}

extern "C" int bqc_submit(bqc_engine* e, const void* data, size_t n_bytes, const uint64_t* record_offsets, uint64_t n_records) {
    return submit_common(e, data, n_bytes, record_offsets, n_records, false, false);
}

extern "C" int bqc_submit_stream(bqc_engine* e, const void* data, size_t n_bytes, int last) {
    return submit_common(e, data, n_bytes, nullptr, 0, true, last != 0);
}

// Index the BGZF blocks at the front of in[0..n): block table entries relative to `in`, until a limit is reached or
// the next block is incomplete.  Returns the bytes consumed; bad = malformed block header.
static uint64_t index_bgzf(const uint8_t* in, uint64_t n, InflateBlock* blocks, uint64_t max_blocks, uint64_t max_out, uint64_t max_in, uint32_t& n_blocks, uint64_t& inflated, bool& bad) {
    uint64_t p = 0, o = 0;
    n_blocks = 0;
    bad = false;
    while (p + 18 <= n && n_blocks < max_blocks) {
        if (in[p] != 0x1f || in[p + 1] != 0x8b || in[p + 2] != 8 || !(in[p + 3] & 4)) { bad = true; break; }
        const uint32_t xlen = in[p + 10] | (in[p + 11] << 8);
        if (p + 12 + xlen > n) break;
        uint64_t x = p + 12, xend = x + xlen;
        int bsize = -1;
        while (x + 4 <= xend) {  // extra subfields; BC carries the block size (SAM/BAM specification 4.1)
            const uint32_t slen = in[x + 2] | (in[x + 3] << 8);
            if (in[x] == 'B' && in[x + 1] == 'C' && slen == 2 && x + 6 <= xend) bsize = in[x + 4] | (in[x + 5] << 8);
            x += 4 + slen;
        }
        if (bsize < 0) { bad = true; break; }
        const uint64_t blen = (uint64_t)bsize + 1;
        if (p + blen > n) break;
        if (blen < 12ull + xlen + 8) { bad = true; break; }
        if (p + blen > max_in) break;
        const uint32_t isize = rd32(in + p + blen - 4);
        if (isize > 65536u) { bad = true; break; }
        if (o + isize > max_out) break;
        InflateBlock b;
        b.cbeg = (uint32_t)(p + 12 + xlen);
        b.clen = (uint32_t)(blen - 12 - xlen - 8);
        b.obeg = (uint32_t)o;
        b.isize = isize;
        blocks[n_blocks++] = b;
        o += isize;
        p += blen;
    }
    inflated = o;
    return p;
}

extern "C" int bqc_submit_bgzf(bqc_engine* e, const void* data, size_t n_bytes, size_t skip_bytes, int last) {
    if (e->finished) { set_error(e, "bqc_submit_bgzf after bqc_finish (call bqc_reset)"); return BQC_ERR_ARG; }
    if (e->async_rc) return e->async_rc;
    CU(cudaSetDevice(e->cfg.device));
    const uint8_t* src = (const uint8_t*)data;
    const bool on_device = e->device_framing;
    size_t p = 0;
    bool any = false;
    while (p < n_bytes || (last && !any)) {
        Slot& s = e->slots[e->next_slot];
        int rc = ensure_slot(e, s);
        if (rc) return rc;
        rc = wait_slot(e, s);
        if (rc) return rc;
        uint32_t nb = 0;
        uint64_t inflated = 0;
        bool bad = false;
        const uint64_t used = index_bgzf(src + p, n_bytes - p, s.h_blocks, e->blocks_per_slot, e->staging_bytes, e->staging_bytes, nb, inflated, bad);
        if (bad || (used == 0 && p < n_bytes)) {
            e->host_error.code = BQC_ERR_BAD_RECORD;
            e->host_error.record = e->records_seen;
            snprintf(e->host_error.message, sizeof(e->host_error.message), "ERROR: Could not read record from BAM File (malformed or truncated BGZF block)");
            set_error(e, "%s", e->host_error.message);
            return BQC_ERR_BAD_RECORD;
        }
        const bool final_chunk = last && p + used >= n_bytes;
        if (skip_bytes > inflated) { set_error(e, "bqc_submit_bgzf: skip_bytes lies beyond the first %llu inflated bytes", (unsigned long long)inflated); return BQC_ERR_ARG; }
        if (on_device) {
            bqc_engine::Task t;
            t.slot = e->next_slot;
            t.n_records = 0;
            t.max_lseq = 0;
            t.mode = 2;
            t.seek = e->stream_seek;
            e->stream_seek = false;
            t.must_align = final_chunk;
            t.span = (size_t)used;
            t.n_blocks = nb;
            t.inflated = (uint32_t)inflated;
            t.skip = (uint32_t)skip_bytes;
            t.h2d_src = used ? h2d_source(e, s, src + p, (size_t)used) : s.pinned + kFrameHead;
            enqueue_task(e, s, t);
        } else {
            // several read groups / BQC_HOST_FRAMING=1: zlib on the host threads, then the host-framed stream path
            uint8_t* buf = s.pinned + kFrameHead;
            const uint8_t* cin = src + p;
            std::vector<uint8_t> moved;
            if (cin < s.pinned + kFrameHead + e->staging_bytes + 256 && cin + used > s.pinned) {  // the caller filled this very staging buffer
                moved.assign(cin, cin + used);
                cin = moved.data();
            }
            if (inflated && bqc_bgzf_inflate(cin, used, buf, e->staging_bytes, e->host_threads) != inflated) {
                e->host_error.code = BQC_ERR_BAD_RECORD;
                e->host_error.record = e->records_seen;
                snprintf(e->host_error.message, sizeof(e->host_error.message), "ERROR: Could not read record from BAM File (BGZF block does not inflate)");
                set_error(e, "%s", e->host_error.message);
                return BQC_ERR_BAD_RECORD;
            }
            rc = submit_common(e, buf + skip_bytes, (size_t)(inflated - skip_bytes), nullptr, 0, true, final_chunk);
            if (rc) return rc;
        }
        skip_bytes = 0;
        p += (size_t)used;
        any = true;
    }
    return 0;
}

extern "C" int bqc_stream_unknown_start(bqc_engine* e) {
    if (!e->device_framing) { set_error(e, "bqc_stream_unknown_start needs device framing"); return BQC_ERR_ARG; }
    if (e->records_seen || e->last_stream_slot >= 0) { set_error(e, "bqc_stream_unknown_start: call it before the first submission"); return BQC_ERR_ARG; }
    e->stream_seek = true;
    e->stream_skipped = -1;
    return 0;
}
extern "C" int bqc_stream_skipped(bqc_engine* e, uint64_t* skipped) {
    const int64_t v = e->stream_skipped.load();
    if (v < 0) return e->async_rc ? e->async_rc : -1;   // -1: the first submission has not been framed yet (poll again)
    *skipped = (uint64_t)v;
    return 0;
}
extern "C" uint64_t bqc_frames_repaired(bqc_engine* e) { drain_commits(e); return e->frames_repaired; }
extern "C" uint64_t bqc_records_seen(bqc_engine* e) { drain_commits(e); return e->records_seen; }

// ------------------------------------------------------------------------------------------------
// SAM text (kernel_sam.cuh): whole lines in, BAM records out on the device; a submission with a line outside the
// fast grammar (sam_parse.h) is encoded on the host with sam_line_to_bam and run as host-framed batches
// ------------------------------------------------------------------------------------------------
static int ensure_sam_slot(bqc_engine* e, Slot& s) {
    if (s.d_text) return 0;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaMalloc(&s.d_text, e->staging_bytes + 512));
    CU(cudaMemset(s.d_text, 0, e->staging_bytes + 512));
    CU(cudaMalloc(&s.d_lend, (e->sam_line_cap + 1) * 4));
    CU(cudaMalloc(&s.d_sz, (e->sam_line_cap + 1) * 8));
    const uint64_t tiles = e->sam_line_cap / (kSamScanThreads * kSamScanPer) + 2;
    const uint64_t nl_blocks = (e->staging_bytes + 1) / (kSamNlThreads * kSamNlPer) + 2;
    CU(cudaMalloc(&s.d_sbsum, std::max(tiles, nl_blocks) * 8));
    CU(cudaMalloc(&s.d_sctl, sizeof(SamCtl)));
    return alloc_device_batch(e, s.sam, e->sam_byte_cap, e->sam_rec_cap);
}

// stage A: text over PCIe, line ends, sizes, scan, records; the frame header goes back to the host
static int sam_stage_a(bqc_engine* e, const bqc_engine::Task& t) {
    Slot& s = e->slots[t.slot];
    DeviceBatch& d = s.sam;
    CU(cudaMemcpyAsync(s.d_text, t.h2d_src, t.span, cudaMemcpyHostToDevice, e->copy));
    CU(cudaEventRecord(e->copied, e->copy));
    CU(cudaStreamWaitEvent(e->frames, e->copied, 0));
    const uint32_t n = (uint32_t)t.span + t.skip;
    {
        ProfScope prof(e, 10, e->frames);
        if (t.skip) CU(cudaMemsetAsync(s.d_text + t.span, '\n', 1, e->frames));
        CU(cudaMemsetAsync(s.d_sctl, 0, sizeof(SamCtl), e->frames));
        const uint32_t nl_blocks = (uint32_t)((n + kSamNlThreads * kSamNlPer - 1) / (kSamNlThreads * kSamNlPer));
        k_sam_nl_count<<<nl_blocks, kSamNlThreads, 0, e->frames>>>(s.d_text, n, s.d_sbsum);
        k_sam_scan_top<<<1, 1024, 0, e->frames>>>(s.d_sbsum, nl_blocks, nullptr, 1, 0, &s.d_sctl->lines);
        k_sam_nl_emit<<<nl_blocks, kSamNlThreads, 0, e->frames>>>(s.d_text, n, s.d_sbsum, s.d_lend, e->sam_line_cap);
        // lines of 300-700 bytes: a few per thread already fill the GPU; the grid-stride loop takes the rest
        const uint64_t est = std::min<uint64_t>(e->sam_line_cap, n / 200 + 1);
        const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((est + kSamLineThreads - 1) / kSamLineThreads, (uint64_t)e->n_sm * 16));
        k_sam_size<<<grid, kSamLineThreads, 0, e->frames>>>(s.d_text, s.d_lend, s.d_sctl, e->sam_line_cap, e->sam_refs, s.d_sz);
        const uint32_t tiles = (uint32_t)(std::min<uint64_t>(e->sam_line_cap, n) / (kSamScanThreads * kSamScanPer) + 1);
        k_sam_scan_tiles<<<tiles, kSamScanThreads, 0, e->frames>>>(s.d_sz, &s.d_sctl->lines, e->sam_line_cap, s.d_sbsum);
        k_sam_scan_top<<<1, 1024, 0, e->frames>>>(s.d_sbsum, 0, &s.d_sctl->lines, kSamScanThreads * kSamScanPer, e->sam_line_cap, &s.d_sctl->packed);
        k_sam_scan_apply<<<tiles, kSamScanThreads, 0, e->frames>>>(s.d_sz, &s.d_sctl->lines, e->sam_line_cap, s.d_sbsum);
        k_sam_encode<<<grid, kSamLineThreads, 0, e->frames>>>(s.d_text, s.d_lend, s.d_sctl, e->sam_line_cap, e->sam_rec_cap, e->sam_byte_cap, e->sam_refs, s.d_sz,
                                                                d.bytes, d.offsets, s.d_frame);
        e->launches += 8;
    }
    if (e->n_lanes > 1) {  // several read groups: as for a device-framed stream
        k_frame_lanes<<<e->n_sm * 4, 256, 0, e->frames>>>(d.bytes, s.d_frame, d.offsets, e->d_lane_names, e->d_lane_off, e->n_lanes, d.rec_lane);
        e->launches += 1;
        int rcp = launch_lane_partition(e, d, &s.d_frame->n_records, 0, e->frames);
        if (rcp) return rcp;
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(s.h_frame, s.d_frame, sizeof(FrameResult), cudaMemcpyDeviceToHost, e->frames));
    CU(cudaEventRecord(s.framed, e->frames));
    return 0;
}

// The host encoder over every line of text[0..n): records into enc, their starts (and the end) into offs.  Returns
// false at the first line sam_line_to_bam rejects (enc/offs then hold the records in front of it).
static bool sam_host_encode(bqc_engine* e, const uint8_t* text, size_t n, std::vector<uint8_t>& enc, std::vector<uint64_t>& offs) {
    enc.clear();
    offs.assign(1, 0);
    std::string line;
    uint64_t lines = 0;
    bool ok = true;
    for (size_t p = 0; p < n;) {
        const uint8_t* q = (const uint8_t*)memchr(text + p, '\n', n - p);
        const size_t end = q ? (size_t)(q - text) : n;
        line.assign((const char*)text + p, end - p);
        p = end + 1;
        if (!line.empty() && line.back() == '\r') line.pop_back();
        if (line.empty()) continue;
        ++lines;
        if (!sam_line_to_bam(line, e->sam_ref_id, enc)) { ok = false; break; }
        offs.push_back(enc.size());
    }
    e->sam_host_lines += lines;
    return ok;
}

static int sam_bad_line(bqc_engine* e) {
    e->host_error.code = BQC_ERR_BAD_RECORD;
    e->host_error.record = e->records_seen;
    snprintf(e->host_error.message, sizeof(e->host_error.message), "ERROR: Could not read record from BAM File (malformed SAM line, record %llu)", (unsigned long long)e->records_seen);
    set_error(e, "%s", e->host_error.message);
    return BQC_ERR_BAD_RECORD;
}

// stage B: run the device's records, or encode the submission on the host and run it as host-framed batches
static int sam_stage_b(bqc_engine* e, const bqc_engine::Task& t) {
    Slot& s = e->slots[t.slot];
    CU(cudaEventSynchronize(s.framed));
    const FrameResult fr = *s.h_frame;
    if (!fr.bad) {
        DeviceBatch& d = s.sam;
        d.max_lseq = fr.max_lseq;
        d.n_records = fr.n_records;
        d.n_bytes = fr.end;
        d.first_record = e->records_seen;
        d.base = d.bytes;
        e->records_seen += fr.n_records;
        if (fr.n_records) {
            CU(cudaStreamWaitEvent(e->compute, s.framed, 0));
            int rc = run_device_batch(e, d);
            if (rc) return rc;
        }
        CU(cudaEventRecord(s.done, e->compute));
        return 0;
    }
    std::vector<uint8_t> enc;
    std::vector<uint64_t> offs;
    const bool ok = sam_host_encode(e, t.h2d_src, t.span, enc, offs);
    const uint64_t n = offs.size() - 1;
    for (uint64_t r0 = 0; r0 < n;) {   // batches that fit the slot's host-framed capacities, one after the other
        uint64_t r1 = r0 + 1;
        while (r1 < n && r1 - r0 < e->max_records_per_slot && offs[r1 + 1] - offs[r0] <= e->staging_bytes) ++r1;
        if (offs[r1] - offs[r0] > e->staging_bytes) { set_error(e, "bqc_submit_sam: a record is larger than the staging buffer"); return BQC_ERR_ARG; }
        bqc_engine::Task b = t;
        b.mode = 0;
        b.n_records = r1 - r0;
        b.span = (size_t)(offs[r1] - offs[r0]);
        b.h2d_src = enc.data() + offs[r0];
        host_scan_pass1(e, enc.data(), offs.data() + r0, b.n_records, s.h_offsets, e->n_lanes > 1 ? s.h_lane : nullptr, b.max_lseq);
        int rc = commit_task(e, b);
        if (rc) return rc;
        CU(cudaEventSynchronize(s.done));   // the slot's buffers are reused by the next batch
        r0 = r1;
    }
    if (!ok) return sam_bad_line(e);
    CU(cudaEventRecord(s.done, e->compute));
    return 0;
}

extern "C" int bqc_set_ref_names(bqc_engine* e, int32_t n, const char* const* names) {
    if (n != e->cfg.n_ref || (n > 0 && !names)) { set_error(e, "bqc_set_ref_names: %d names for an engine of %d references", n, e->cfg.n_ref); return BQC_ERR_ARG; }
    CU(cudaSetDevice(e->cfg.device));
    { int arc = drain_commits(e); if (arc) return arc; }
    for (auto& sl : e->slots) { int rc = wait_slot(e, sl); if (rc) return rc; }
    std::vector<std::string> v(names, names + n);
    std::string blob;
    std::vector<uint32_t> off;
    std::vector<int32_t> id;
    sam_refs_build(v, blob, off, id);
    e->sam_ref_id.clear();
    for (int32_t i = 0; i < n; ++i) e->sam_ref_id.insert({v[i], i});   // first of duplicate names wins
    cudaFree(e->d_sam_blob); cudaFree(e->d_sam_off); cudaFree(e->d_sam_id);
    e->d_sam_blob = nullptr; e->d_sam_off = nullptr; e->d_sam_id = nullptr;
    CU(cudaMalloc(&e->d_sam_blob, blob.size() + 1));
    CU(cudaMalloc(&e->d_sam_off, off.size() * 4));
    CU(cudaMalloc(&e->d_sam_id, id.size() * 4 + 4));
    CU(cudaMemcpy(e->d_sam_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_sam_off, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
    if (!id.empty()) CU(cudaMemcpy(e->d_sam_id, id.data(), id.size() * 4, cudaMemcpyHostToDevice));
    e->sam_refs = {e->d_sam_blob, e->d_sam_off, e->d_sam_id, (int32_t)id.size()};
    e->have_sam_refs = true;
    return 0;
}

static int sam_check(bqc_engine* e, const char* fn, const uint8_t* text, size_t n, bool last) {
    if (e->finished) { set_error(e, "%s after bqc_finish (call bqc_reset)", fn); return BQC_ERR_ARG; }
    if (!e->have_sam_refs) { set_error(e, "%s: call bqc_set_ref_names first", fn); return BQC_ERR_ARG; }
    if (n > e->staging_bytes) { set_error(e, "%s: %zu bytes exceed the staging capacity %llu", fn, n, (unsigned long long)e->staging_bytes); return BQC_ERR_ARG; }
    if (n && !last && text[n - 1] != '\n') { set_error(e, "%s: the text does not end at a line end", fn); return BQC_ERR_ARG; }
    return 0;
}

extern "C" int bqc_submit_sam(bqc_engine* e, const void* text, size_t n, int last) {
    const uint8_t* src = (const uint8_t*)text;
    int rc = sam_check(e, "bqc_submit_sam", src, n, last != 0);
    if (rc) return rc;
    if (e->async_rc) return e->async_rc;
    if (n == 0) return 0;
    CU(cudaSetDevice(e->cfg.device));
    Slot& s = e->slots[e->next_slot];
    if ((rc = ensure_slot(e, s)) || (rc = ensure_sam_slot(e, s)) || (rc = wait_slot(e, s))) return rc;
    bqc_engine::Task t;
    t.slot = e->next_slot;
    t.n_records = 0;
    t.max_lseq = 0;
    t.mode = 3;
    t.must_align = true;
    t.span = n;
    t.skip = src[n - 1] != '\n' ? 1u : 0u;
    t.h2d_src = h2d_source(e, s, src, n);
    enqueue_task(e, s, t);
    return 0;
}

extern "C" int bqc_sam_to_bam(bqc_engine* e, const void* text, size_t n, uint8_t* out, uint64_t cap, uint64_t* n_bytes, uint64_t* n_records) {
    const uint8_t* src = (const uint8_t*)text;
    *n_bytes = 0;
    *n_records = 0;
    int rc = sam_check(e, "bqc_sam_to_bam", src, n, true);
    if (rc) return rc;
    if (n == 0) return 0;
    CU(cudaSetDevice(e->cfg.device));
    { int arc = drain_commits(e); if (arc) return arc; }
    Slot& s = e->slots[e->next_slot];
    if ((rc = ensure_slot(e, s)) || (rc = ensure_sam_slot(e, s)) || (rc = wait_slot(e, s))) return rc;
    bqc_engine::Task t;
    t.slot = e->next_slot;
    t.mode = 3;
    t.span = n;
    t.skip = src[n - 1] != '\n' ? 1u : 0u;
    t.h2d_src = h2d_source(e, s, src, n);
    if ((rc = sam_stage_a(e, t))) return rc;
    CU(cudaEventSynchronize(s.framed));
    const FrameResult fr = *s.h_frame;
    if (!fr.bad) {
        if (fr.end > cap) { set_error(e, "bqc_sam_to_bam: %u record bytes exceed the output capacity", fr.end); return BQC_ERR_ARG; }
        CU(cudaMemcpy(out, s.sam.bytes, fr.end, cudaMemcpyDeviceToHost));
        *n_bytes = fr.end;
        *n_records = fr.n_records;
        return 0;
    }
    std::vector<uint8_t> enc;
    std::vector<uint64_t> offs;
    const bool ok = sam_host_encode(e, t.h2d_src, t.span, enc, offs);
    if (offs.back() > cap) { set_error(e, "bqc_sam_to_bam: %llu record bytes exceed the output capacity", (unsigned long long)offs.back()); return BQC_ERR_ARG; }
    memcpy(out, enc.data(), (size_t)offs.back());
    *n_bytes = offs.back();
    *n_records = offs.size() - 1;
    if (!ok) { set_error(e, "bqc_sam_to_bam: SAM line of record %llu is malformed", (unsigned long long)*n_records); return BQC_ERR_BAD_RECORD; }
    return 0;
}

extern "C" uint64_t bqc_sam_host_lines(bqc_engine* e) { drain_commits(e); return e->sam_host_lines; }

// ------------------------------------------------------------------------------------------------
// resident path
// ------------------------------------------------------------------------------------------------
extern "C" int bqc_batch_prepare(bqc_engine* e, const void* data, size_t n_bytes, const uint64_t* record_offsets, uint64_t n_records, bqc_batch** out) {
    *out = nullptr;
    if (n_bytes >= 0xFFFFFF00ull) { set_error(e, "bqc_batch_prepare: a batch must be smaller than 4 GiB"); return BQC_ERR_ARG; }
    CU(cudaSetDevice(e->cfg.device));
    drain_commits(e);
    const uint8_t* src = (const uint8_t*)data;
    std::vector<uint64_t> own_offsets;
    if (!record_offsets) {
        own_offsets.resize(n_bytes / 36 + 2);
        n_records = frame_records_mt(src, n_bytes, own_offsets.data(), own_offsets.size(), e->host_threads, std::max(1, e->cfg.n_ref), e->pool.get());
        record_offsets = own_offsets.data();
    }
    bqc_batch* b = new bqc_batch();
    DeviceBatch& d = b->d;
    int rc = alloc_device_batch(e, d, n_bytes, n_records);
    if (rc) { free_device_batch(d); delete b; return rc; }
    std::vector<uint32_t> o32(n_records + 1);
    std::vector<uint8_t> lanes(e->n_lanes > 1 ? n_records + 1 : 0);
    host_scan_pass1(e, src, record_offsets, n_records, o32.data(), lanes.empty() ? nullptr : lanes.data(), d.max_lseq);
    size_t span = n_records ? (size_t)(record_offsets[n_records] - record_offsets[0]) : 0;
    d.n_records = n_records;
    d.n_bytes = span;
    d.first_record = e->records_seen;
    e->records_seen += n_records;
    d.records_after = e->records_seen;
    if (n_records) {
        CU(cudaMemcpy(d.bytes + kFrameHead, src + record_offsets[0], span, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d.offsets, o32.data(), (n_records + 1) * 4, cudaMemcpyHostToDevice));
        if (e->n_lanes > 1) {
            CU(cudaMemcpy(d.rec_lane, lanes.data(), n_records, cudaMemcpyHostToDevice));
            rc = launch_lane_partition(e, d, nullptr, n_records, e->compute);
            if (rc) return rc;
            CU(cudaStreamSynchronize(e->compute));
        }
    }
    *out = b;
    return 0;
}
extern "C" int bqc_batch_run(bqc_engine* e, bqc_batch* b) {
    CU(cudaSetDevice(e->cfg.device));
    if (e->finished) { set_error(e, "bqc_batch_run after bqc_finish (call bqc_reset)"); return BQC_ERR_ARG; }
    drain_commits(e);
    e->records_seen = b->d.records_after;  // (the coverage anchor state is carried on the device)
    return run_device_batch(e, b->d);
}
extern "C" void bqc_batch_free(bqc_engine* e, bqc_batch* b) {
    if (!b) return;
    if (e) cudaSetDevice(e->cfg.device);
    free_device_batch(b->d);
    delete b;
}
extern "C" uint64_t bqc_batch_records(const bqc_batch* b) { return b->d.n_records; }
extern "C" uint64_t bqc_batch_bytes(const bqc_batch* b) { return b->d.n_bytes; }

// ------------------------------------------------------------------------------------------------
// completion
// ------------------------------------------------------------------------------------------------
static const char* reference_message(int code) {
    switch (code) {
        case BQC_ERR_RG_NOT_Z: return "Read does not have Z";
        case BQC_ERR_NO_MATE_FLAG: return "ERROR: No first or second flag in read";
        case BQC_ERR_AS_TAG: return "ERROR: Read has no AS tag / could not read AS tag";
        case BQC_ERR_BAD_RECORD: return "ERROR: Could not read record from BAM File";
        case BQC_ERR_NO_RG: return "ERROR: record without RG tag";
        case BQC_ERR_UNSUPPORTED: return "ERROR: value outside the engine's table capacities (read length / histogram index)";
        default: return "";
    }
}

extern "C" int bqc_get_error(bqc_engine* e, bqc_error_info* out) {
    memset(out, 0, sizeof(*out));
    unsigned long long key = ~0ull;
    if (cudaSetDevice(e->cfg.device) != cudaSuccess || cudaMemcpy(&key, e->d_error, 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        if (!e->host_error.code) { set_error(e, "bqc_get_error: reading the device error word failed"); return BQC_ERR_CUDA; }
        key = ~0ull;
    }
    // the first offending record in file order wins, whether the host or the device found it
    if (e->host_error.code && (key == ~0ull || ((unsigned long long)e->host_error.record << 8 | (uint32_t)e->host_error.code) <= key)) { *out = e->host_error; return 0; }
    if (key != ~0ull) {
        out->code = (int32_t)(key & 255);
        out->record = key >> 8;
        snprintf(out->message, sizeof(out->message), "%s (record %llu)", reference_message(out->code), (unsigned long long)out->record);
    }
    return 0;
}

extern "C" int bqc_sync(bqc_engine* e) {
    CU(cudaSetDevice(e->cfg.device));
    const int arc = drain_commits(e);
    if (arc) {   // the work enqueued in front of the failure still runs: its errors are final once it has
        cudaStreamSynchronize(e->copy);
        cudaStreamSynchronize(e->covs);
        cudaStreamSynchronize(e->compute);
        return arc;
    }
    CU(cudaStreamSynchronize(e->copy));
    CU(cudaStreamSynchronize(e->covs));
    CU(cudaStreamSynchronize(e->compute));
    bqc_error_info ei;
    int rc = bqc_get_error(e, &ei);
    if (rc) return rc;
    if (ei.code) set_error(e, "%s", ei.message);
    return ei.code;
}

extern "C" int32_t bqc_n_lanes(bqc_engine* e) { return (int32_t)e->n_lanes; }
extern "C" const char* bqc_lane_id(bqc_engine* e, int32_t lane) { return (lane >= 0 && (uint32_t)lane < e->n_lanes) ? e->lane_ids[lane].c_str() : ""; }
extern "C" void bqc_qk_lists(bqc_engine* e, const int32_t** klist, uint32_t* n_k, const uint64_t** qlist, uint32_t* n_q) {
    *klist = e->klist.data();
    *n_k = (uint32_t)e->klist.size();
    *qlist = e->qlist.data();
    *n_q = (uint32_t)e->qlist.size();
}
extern "C" void* bqc_stream(bqc_engine* e) { return (void*)e->compute; }
extern "C" uint64_t bqc_kernel_launches(bqc_engine* e) { return e->launches; }

extern "C" int bqc_finish(bqc_engine* e) {
    CU(cudaSetDevice(e->cfg.device));
    { int arc = drain_commits(e); if (arc) return arc; }
    if (!e->finished) {
        // src/bamqualcheck.cpp:447-453: update_coverage(); update_vectors(); update_coverage() for every lane
        for (uint32_t lane = 0; lane < e->n_lanes; ++lane) {
            unsigned long long* poscov = (unsigned long long*)(e->d_counters + (uint64_t)lane * e->L.lane_stride + e->L.o_poscov);
            ProfScope prof(e, 3, cov_stream(e));
            if (e->cov_deferred || e->cov_head_piece) continue;  // shard mode: bqc_cov_shards_combine flushes the last windows
            k_cov_final<<<1, 32, 0, cov_stream(e)>>>(e->d_cov_carry + lane, e->d_cov_d + (uint64_t)lane * 2 * kCovD, poscov);
            e->launches += 1;
        }
        CU(cudaEventRecord(e->cov_done, cov_stream(e)));
        CU(cudaStreamWaitEvent(e->compute, e->cov_done, 0));
        e->finished = true;
    }
    e->have_results = false;
    return bqc_sync(e);
}

// ------------------------------------------------------------------------------------------------
// one record stream cut across several engines: the coverage statistic (include/bamqc_b200.h, cov_math.h "Shards")
// ------------------------------------------------------------------------------------------------
extern "C" int bqc_cov_defer(bqc_engine* e, int on) {
    if (e->records_seen || e->cov_acc_bound) { set_error(e, "bqc_cov_defer: call it right after bqc_reset"); return BQC_ERR_ARG; }
    e->cov_deferred = on == 1;
    e->cov_head_piece = on == 2;
    return 0;
}

// Shard mode with several read groups collects every lane's records in one queue, in file order, each tagged with its
// lane (launch_cov), so that the queue needs no more room than with one lane.  The first shard call after the run
// groups it by lane: k_lane_partition over the tags (lane by lane, file order inside a lane), then one gather into a
// copy whose lane l owns [cov_lane_range[l], cov_lane_range[l + 1]).  Kept until bqc_reset.  n: the records collected.
static int cov_lane_split(bqc_engine* e, uint32_t n) {
    const uint64_t N = std::max<uint32_t>(n, 1u);
    const uint64_t o_range = N * 16, o_lb = (o_range + (e->n_lanes + 1) * 4 + 7) & ~7ull, lb_bytes = (N / 1024 + 4) * 8;
    cudaFree(e->d_cov_lq);
    CU(cudaMalloc(&e->d_cov_lq, o_lb + lb_bytes));
    uint8_t* m = e->d_cov_lq;
    uint32_t* index = (uint32_t*)(m + N * 12);
    uint32_t* range = (uint32_t*)(m + o_range);
    unsigned long long* lb = (unsigned long long*)(m + o_lb);
    cudaStream_t st = cov_stream(e);
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((n + 1023) / 1024, (uint64_t)e->n_sm * 2));
    ProfScope prof(e, 3, st);
    for (uint32_t lane = 0; lane < e->n_lanes; ++lane) {
        CU(cudaMemsetAsync(lb, 0, lb_bytes, st));
        k_lane_partition<<<grid, 1024, 0, st>>>(e->cov_scratch.q_lane, nullptr, n, lane, index, range, lb + 1, (uint32_t*)lb);
    }
    if (n) k_cov_lane_gather<<<grid, 1024, 0, st>>>(e->cov_scratch, index, n, (int32_t*)m, (uint32_t*)(m + N * 4), (uint32_t*)(m + N * 8));
    e->launches += e->n_lanes + (n ? 1u : 0u);
    CU(cudaGetLastError());
    std::vector<uint32_t> r(e->n_lanes + 1);
    CU(cudaMemcpyAsync(r.data(), range, (e->n_lanes + 1) * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    e->cov_lane_range.swap(r);
    return 0;
}

// Every shard call: checks its arguments, synchronises the engine and returns how many records of `lane` were
// collected (grouping them by lane first, see cov_lane_split).
static int cov_shard_sync(bqc_engine* e, const char* fn, int32_t lane, uint32_t& nq) {
    if (!e->cov_deferred && !e->cov_head_piece) { set_error(e, "%s: engine is not in shard mode (bqc_cov_defer)", fn); return BQC_ERR_ARG; }
    if (lane < 0 || (uint32_t)lane >= e->n_lanes) { set_error(e, "%s: bad lane", fn); return BQC_ERR_ARG; }
    CU(cudaSetDevice(e->cfg.device));
    { int arc = drain_commits(e); if (arc) return arc; }
    CU(cudaStreamSynchronize(e->compute));
    CU(cudaStreamSynchronize(e->covs));
    CovCarry c;
    CU(cudaMemcpy(&c, e->d_cov_carry, sizeof(c), cudaMemcpyDeviceToHost));
    nq = c.nq;
    if (e->cov_deferred && e->n_lanes > 1) {
        if (e->cov_lane_range.empty()) { int rc = cov_lane_split(e, c.nq); if (rc) return rc; }
        nq = e->cov_lane_range[lane + 1] - e->cov_lane_range[lane];
    }
    return 0;
}

// The compact records of `lane` as the resolving kernels see them: the whole queue with one lane, the lane's segment
// of the grouped copy with several (no record index: a record that needs its bytes again is refused in shard mode).
static CovScratch cov_lane_scratch(bqc_engine* e, int32_t lane) {
    CovScratch S = e->cov_scratch;
    if (e->cov_deferred && e->n_lanes > 1) {
        const uint64_t N = std::max<uint32_t>(e->cov_lane_range.back(), 1u), a = e->cov_lane_range[lane];
        S.q_rid = (int32_t*)e->d_cov_lq + a;
        S.q_b = (uint32_t*)(e->d_cov_lq + N * 4) + a;
        S.q_iv = (uint32_t*)(e->d_cov_lq + N * 8) + a;
        S.q_rec = nullptr;
        S.q_lane = nullptr;
    }
    return S;
}

// With several lanes the carry of a lane does not hold the lane's record count: set it before its records are resolved.
static int cov_lane_set_nq(bqc_engine* e, int32_t lane, uint32_t nq) {
    if (e->cov_deferred && e->n_lanes > 1)
        CU(cudaMemcpyAsync(&e->d_cov_carry[lane].nq, &nq, 4, cudaMemcpyHostToDevice, cov_stream(e)));
    return 0;
}

extern "C" int bqc_cov_shard_boundary_lane(bqc_engine* e, int32_t lane, bqc_cov_shard* out) {
    memset(out, 0, sizeof(*out));
    uint32_t nq = 0;
    int rc = cov_shard_sync(e, "bqc_cov_shard_boundary", lane, nq);
    if (rc) return rc;
    if (e->cov_head_piece) {  // already resolved batch by batch: what matters to the pieces behind is the last record
        CovCarry c;
        CU(cudaMemcpy(&c, e->d_cov_carry + lane, sizeof(c), cudaMemcpyDeviceToHost));
        out->n = c.first ? 0 : 1;   // (a count is not kept; non-zero = some record took part)
        out->last_rid = c.rid_prev;
        out->last_b = c.b_prev;
        return 0;
    }
    out->n = nq;
    if (nq) {
        const CovScratch S = cov_lane_scratch(e, lane);
        CU(cudaMemcpy(&out->first_rid, S.q_rid, 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(&out->first_b, S.q_b, 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(&out->last_rid, S.q_rid + (nq - 1), 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(&out->last_b, S.q_b + (nq - 1), 4, cudaMemcpyDeviceToHost));
    }
    return 0;
}

extern "C" int bqc_cov_shard_function_lane(bqc_engine* e, int32_t lane, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint16_t* table1002) {
    uint32_t nq = 0;
    int rc = cov_shard_sync(e, "bqc_cov_shard_function", lane, nq);
    if (rc) return rc;
    for (uint32_t s = 0; s < kCovStates; ++s) table1002[s] = (uint16_t)s;   // no record: the state passes through
    if (e->cov_head_piece) {  // the first piece ends in the state it carries
        CovCarry c;
        CU(cudaMemcpy(&c, e->d_cov_carry + lane, sizeof(c), cudaMemcpyDeviceToHost));
        if (!c.first) for (uint32_t s = 0; s < kCovStates; ++s) table1002[s] = (uint16_t)cov_state_index(c.p_prev);
        return 0;
    }
    if (!nq) return 0;
    rc = ensure_cov_scratch(e, nq);
    if (rc) return rc;
    if (!e->d_cov_fn) CU(cudaMalloc(&e->d_cov_fn, 1024 * 2 + kCovD * 4));
    const CovScratch S = cov_lane_scratch(e, lane);
    CovCarry* carry = e->d_cov_carry + lane;
    const uint32_t nblk = (nq + kCovRB - 1) / kCovRB;
    rc = cov_lane_set_nq(e, lane, nq);
    if (rc) return rc;
    k_cov_set_state<<<1, 1, 0, cov_stream(e)>>>(carry, have_prev ? 0u : 1u, prev_rid, prev_b, 0u);
    k_cov_tables<<<nblk, kCovBlockThreads, kCovBlockSmem, cov_stream(e)>>>(S, carry);
    k_cov_shard_function<<<1, 1024, 0, cov_stream(e)>>>(S, carry, e->d_cov_fn);
    e->launches += 3;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(cov_stream(e)));
    CU(cudaMemcpy(table1002, e->d_cov_fn, kCovStates * 2, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int bqc_cov_shard_run_lane(bqc_engine* e, int32_t lane, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint32_t p_in, bqc_cov_shard* out) {
    uint32_t nq = 0;
    int rc = cov_shard_sync(e, "bqc_cov_shard_run", lane, nq);
    if (rc) return rc;
    memset(out->head, 0, sizeof(out->head));
    memset(out->tail, 0, sizeof(out->tail));
    out->span = 0;
    out->n = nq;
    CovCarry* carry = e->d_cov_carry + lane;
    int32_t* cd = e->d_cov_d + (uint64_t)lane * 2 * kCovD;
    if (e->cov_head_piece) {  // nothing left to resolve: report the two windows that are still open
        CovCarry c;
        CU(cudaMemcpy(&c, carry, sizeof(c), cudaMemcpyDeviceToHost));
        out->n = c.first ? 0 : 1;
        out->span = c.xc;
        CU(cudaMemcpy(out->tail, cd + (uint64_t)c.parity * kCovD, sizeof(out->tail), cudaMemcpyDeviceToHost));
        return 0;
    }
    if (!nq) return 0;
    rc = ensure_cov_scratch(e, nq);
    if (rc) return rc;
    if (!e->d_cov_fn) CU(cudaMalloc(&e->d_cov_fn, 1024 * 2 + kCovD * 4));
    int32_t* d_head = (int32_t*)(e->d_cov_fn + 1024);
    const CovScratch S = cov_lane_scratch(e, lane);
    BatchView B;
    memset(&B, 0, sizeof(B));
    CU(cudaMemsetAsync(e->d_cov_scratch, 0, e->cov_ctl_bytes, cov_stream(e)));
    CU(cudaMemsetAsync(cd, 0, 2 * kCovD * 4, cov_stream(e)));
    rc = cov_lane_set_nq(e, lane, nq);
    if (rc) return rc;
    k_cov_set_state<<<1, 1, 0, cov_stream(e)>>>(carry, have_prev ? 0u : 1u, prev_rid, prev_b, p_in);
    {
        ProfScope prof(e, 3, cov_stream(e));
        rc = launch_cov_resolve(e, (uint32_t)lane, S, B, nq, false);
        if (rc) return rc;
        k_cov_head<<<1, 1024, 0, cov_stream(e)>>>(B, S, carry, d_head);
        k_cov_carry<<<1, 1024, 0, cov_stream(e)>>>(B, S, carry, cd);
        e->launches += 3;
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(cov_stream(e)));
    CovCarry c;
    CU(cudaMemcpy(&c, carry, sizeof(c), cudaMemcpyDeviceToHost));
    out->span = c.xc;
    CU(cudaMemcpy(out->head, d_head, sizeof(out->head), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out->tail, cd + (uint64_t)c.parity * kCovD, sizeof(out->tail), cudaMemcpyDeviceToHost));
    e->have_results = false;
    return 0;
}

extern "C" int bqc_cov_shard_boundary(bqc_engine* e, bqc_cov_shard* out) { return bqc_cov_shard_boundary_lane(e, 0, out); }
extern "C" int bqc_cov_shard_function(bqc_engine* e, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint16_t* table1002) {
    return bqc_cov_shard_function_lane(e, 0, have_prev, prev_rid, prev_b, table1002);
}
extern "C" int bqc_cov_shard_run(bqc_engine* e, int32_t have_prev, int32_t prev_rid, uint32_t prev_b, uint32_t p_in, bqc_cov_shard* out) {
    return bqc_cov_shard_run_lane(e, 0, have_prev, prev_rid, prev_b, p_in, out);
}

extern "C" void bqc_cov_shards_combine(const bqc_cov_shard* shards, int32_t n_shards, int64_t delta[101]) {
    std::vector<CovShardPiece> pc((size_t)std::max(0, n_shards));
    for (int32_t k = 0; k < n_shards; ++k) { pc[k].n = shards[k].n; pc[k].span = shards[k].span; pc[k].head = shards[k].head; pc[k].tail = shards[k].tail; }
    long long d[101];
    cov_shards_combine(pc.data(), n_shards, d);
    for (int i = 0; i <= 100; ++i) delta[i] = d[i];
}

extern "C" uint32_t bqc_cov_apply(const uint16_t* table1002, uint32_t p) { return cov_state_value(table1002[cov_state_index(p)]); }

extern "C" int bqc_poscov_adjust(bqc_engine* e, int32_t lane, const int64_t delta[101]) {
    if (lane < 0 || (uint32_t)lane >= e->n_lanes) { set_error(e, "bqc_poscov_adjust: bad lane"); return BQC_ERR_ARG; }
    CU(cudaSetDevice(e->cfg.device));
    long long* d = nullptr;
    CU(cudaMalloc(&d, 101 * 8));
    CU(cudaMemcpy(d, delta, 101 * 8, cudaMemcpyHostToDevice));
    k_poscov_adjust<<<1, 128, 0, e->compute>>>((unsigned long long*)(e->d_counters + (uint64_t)lane * e->L.lane_stride + e->L.o_poscov), d);
    e->launches += 1;
    CU(cudaStreamSynchronize(e->compute));
    cudaFree(d);
    e->have_results = false;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// multi-GPU merge helpers
// ------------------------------------------------------------------------------------------------
extern "C" uint32_t bqc_read_len_capacity(bqc_engine* e) { return e->L.cyc; }
extern "C" int bqc_reserve_read_len(bqc_engine* e, uint32_t n) {
    CU(cudaSetDevice(e->cfg.device));
    { int arc = drain_commits(e); if (arc) return arc; }
    if (n > kMaxReadLen) { set_error(e, "bqc_reserve_read_len: reads longer than %u are not supported", kMaxReadLen); return BQC_ERR_ARG; }
    return grow_read_len(e, n, true);
}
extern "C" uint64_t bqc_counters_len(bqc_engine* e) { return (uint64_t)e->n_lanes * e->L.lane_stride; }
extern "C" int bqc_counters_export(bqc_engine* e, void* dev) {
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaMemcpyAsync(dev, e->d_counters, bqc_counters_len(e) * 8, cudaMemcpyDeviceToDevice, e->compute));
    CU(cudaStreamSynchronize(e->compute));
    return 0;
}
extern "C" int bqc_counters_import(bqc_engine* e, const void* dev) {
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaMemcpyAsync(e->d_counters, dev, bqc_counters_len(e) * 8, cudaMemcpyDeviceToDevice, e->compute));
    CU(cudaStreamSynchronize(e->compute));
    e->have_results = false;
    return 0;
}
extern "C" uint64_t bqc_sketch_len(bqc_engine* e) { return (uint64_t)e->n_lanes * e->n_qk * e->sketch_words_per_qk * 8; }
extern "C" int bqc_sketch_export_u8(bqc_engine* e, void* dev) {
    CU(cudaSetDevice(e->cfg.device));
    uint64_t nwords = bqc_sketch_len(e) / 8;
    if (nwords) {
        k_sketch_export_u8<<<e->n_sm * 8, 256, 0, e->compute>>>(e->d_sketch, nwords, (uint8_t*)dev);
        e->launches += 1;
    }
    CU(cudaStreamSynchronize(e->compute));
    return 0;
}
extern "C" int bqc_sketch_import_u8(bqc_engine* e, const void* dev) {
    CU(cudaSetDevice(e->cfg.device));
    uint64_t nwords = bqc_sketch_len(e) / 8;
    if (nwords) {
        k_sketch_import_u8<<<e->n_sm * 8, 256, 0, e->compute>>>(e->d_sketch, nwords, (const uint8_t*)dev);
        e->launches += 1;
    }
    CU(cudaStreamSynchronize(e->compute));
    e->have_results = false;
    return 0;
}
extern "C" int bqc_merge_from(bqc_engine* dst, bqc_engine* src) {
    bqc_engine* e = dst;
    { int arc = drain_commits(dst); if (arc) return arc; }   // a batch still with the commit thread may grow either layout
    { int arc = drain_commits(src); if (arc) { set_error(e, "bqc_merge_from: the source engine failed: %s", src->last_error.c_str()); return arc; } }
    if (dst->L.cyc != src->L.cyc) {  // one of them met a longer read: same layout first
        int rc = dst->L.cyc < src->L.cyc ? grow_read_len(dst, src->L.cyc, true) : grow_read_len(src, dst->L.cyc, true);
        if (rc) return rc;
    }
    if (bqc_counters_len(dst) != bqc_counters_len(src) || bqc_sketch_len(dst) != bqc_sketch_len(src)) { set_error(e, "bqc_merge_from: engines differ in configuration"); return BQC_ERR_ARG; }
    CU(cudaSetDevice(src->cfg.device));
    CU(cudaStreamSynchronize(src->compute));
    CU(cudaSetDevice(dst->cfg.device));
    uint64_t nc = bqc_counters_len(dst), nw = bqc_sketch_len(dst) / 8;
    uint64_t* tc = nullptr;
    uint32_t* ts = nullptr;
    CU(cudaMalloc(&tc, nc * 8));
    CU(cudaMalloc(&ts, std::max<uint64_t>(4, nw * 4)));
    CU(cudaMemcpyPeerAsync(tc, dst->cfg.device, src->d_counters, src->cfg.device, nc * 8, dst->compute));
    if (nw) CU(cudaMemcpyPeerAsync(ts, dst->cfg.device, src->d_sketch, src->cfg.device, nw * 4, dst->compute));
    k_counters_add<<<dst->n_sm * 4, 256, 0, dst->compute>>>((unsigned long long*)dst->d_counters, (const unsigned long long*)tc, nc);
    if (nw) k_sketch_merge<<<dst->n_sm * 8, 256, 0, dst->compute>>>(dst->d_sketch, ts, nw);
    dst->launches += 2;
    CU(cudaStreamSynchronize(dst->compute));
    cudaFree(tc);
    cudaFree(ts);
    dst->have_results = false;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
static int fetch_results(bqc_engine* e) {
    if (e->have_results) return 0;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaStreamSynchronize(e->compute));
    e->h_counters.resize(bqc_counters_len(e));
    e->h_sketch.resize(bqc_sketch_len(e) / 8);
    CU(cudaMemcpy(e->h_counters.data(), e->d_counters, e->h_counters.size() * 8, cudaMemcpyDeviceToHost));
    if (!e->h_sketch.empty()) CU(cudaMemcpy(e->h_sketch.data(), e->d_sketch, e->h_sketch.size() * 4, cudaMemcpyDeviceToHost));
    e->have_results = true;
    return 0;
}

static uint64_t top_nonzero(const uint64_t* p, uint64_t n) {  // highest non-zero index + 1
    while (n && p[n - 1] == 0) --n;
    return n;
}

extern "C" int bqc_result_table(bqc_engine* e, int32_t lane, int32_t field, int32_t sub, uint64_t* out, uint64_t cap, uint64_t* n_out) {
    int rc = fetch_results(e);
    if (rc) return rc;
    if (lane < 0 || (uint32_t)lane >= e->n_lanes) { set_error(e, "bqc_result_table: bad lane"); return BQC_ERR_ARG; }
    const Layout& L = e->L;
    const uint64_t* G = e->h_counters.data() + (uint64_t)lane * L.lane_stride;
    const uint64_t* src = nullptr;
    uint64_t n = 0;
    auto mateblk = [&](int m) { return G + L.o_mate0 + (uint64_t)m * L.mate_stride; };
    auto maxlen = [&](int m) { uint64_t t = top_nonzero(mateblk(m) + L.m_readlen, L.cyc + 1); return t ? t - 1 : 0; };  // max read length seen
    auto seen = [&](int m) { return top_nonzero(mateblk(m) + L.m_readlen, L.cyc + 1) != 0; };
    bool per_mate = field >= BQC_F_READLEN_M && field <= BQC_F_READNR_M;
    if (per_mate && (sub < 0 || sub > 1)) { set_error(e, "bqc_result_table: mate must be 0 or 1"); return BQC_ERR_ARG; }
    switch (field) {
        case BQC_F_SCALARS: src = G + L.o_scalars; n = 13; break;
        case BQC_F_POSCOV: src = G + L.o_poscov; n = 101; break;
        case BQC_F_INSERT: src = G + L.o_insert; n = L.isize1; break;
        case BQC_F_EIGHTMER: src = G + L.o_eightmer; n = kEightmer; break;
        case BQC_F_TRIPLET: src = G + L.o_triplet; n = kTriplet; break;
        case BQC_F_READLEN_M: src = mateblk(sub) + L.m_readlen; n = top_nonzero(src, L.cyc + 1); break;
        case BQC_F_NCOUNT_M: src = mateblk(sub) + L.m_ncount; n = seen(sub) ? maxlen(sub) + 1 : 0; break;
        case BQC_F_GCCOUNT_M: src = mateblk(sub) + L.m_gccount; n = seen(sub) ? maxlen(sub) + 1 : 0; break;
        case BQC_F_AVGQUAL_M: src = mateblk(sub) + L.m_avgq; n = top_nonzero(mateblk(sub) + L.m_ceilq, kQCap); break;
        case BQC_F_MAPQ_M: src = mateblk(sub) + L.m_mapq; n = top_nonzero(src, kMapqCap); break;
        case BQC_F_MISMATCH_M: src = mateblk(sub) + L.m_mismatch; n = top_nonzero(src, L.mmcap); break;
        case BQC_F_DEL_M: src = mateblk(sub) + L.m_del; n = top_nonzero(src, L.delcap); break;
        case BQC_F_INS_M: src = mateblk(sub) + L.m_ins; n = top_nonzero(src, L.mmcap); break;
        case BQC_F_DNA_A_M: case BQC_F_DNA_C_M: case BQC_F_DNA_G_M: case BQC_F_DNA_T_M: case BQC_F_DNA_N_M:
            src = mateblk(sub) + L.m_pc + (uint64_t)(field - BQC_F_DNA_A_M) * pad8(L.cyc); n = maxlen(sub); break;
        case BQC_F_QUALSUM_M: src = mateblk(sub) + L.m_pc + (uint64_t)PC_QUAL * pad8(L.cyc); n = maxlen(sub); break;
        case BQC_F_SC5_M: src = mateblk(sub) + L.m_pc + (uint64_t)PC_SC5 * pad8(L.cyc); n = maxlen(sub); break;
        case BQC_F_SC3_M: src = mateblk(sub) + L.m_pc + (uint64_t)PC_SC3 * pad8(L.cyc); n = maxlen(sub); break;
        case BQC_F_READNR_M: src = mateblk(sub) + L.m_readnr; n = 1; break;
        case BQC_F_SUMCOUNT_QK:
            if (sub < 0 || (uint32_t)sub >= e->n_qk) { set_error(e, "bqc_result_table: bad (q,k) index"); return BQC_ERR_ARG; }
            src = G + L.o_qk + (uint64_t)sub * L.qk_stride; n = 1; break;
        case BQC_F_F2TABLE_QK:
            if (sub < 0 || (uint32_t)sub >= e->n_qk) { set_error(e, "bqc_result_table: bad (q,k) index"); return BQC_ERR_ARG; }
            src = G + L.o_qk + (uint64_t)sub * L.qk_stride + 8; n = L.f2size; break;
        default: set_error(e, "bqc_result_table: unknown field %d", field); return BQC_ERR_ARG;
    }
    if (n_out) *n_out = n;
    if (out) {
        if (cap < n) { set_error(e, "bqc_result_table: buffer too small"); return BQC_ERR_ARG; }
        memcpy(out, src, n * 8);
    }
    return 0;
}

extern "C" int bqc_result_sketch(bqc_engine* e, int32_t lane, int32_t qk, uint64_t* out, uint64_t cap, uint64_t* n_out) {
    int rc = fetch_results(e);
    if (rc) return rc;
    if (lane < 0 || (uint32_t)lane >= e->n_lanes || qk < 0 || (uint32_t)qk >= e->n_qk) { set_error(e, "bqc_result_sketch: bad index"); return BQC_ERR_ARG; }
    uint64_t n = e->sketch_words_per_qk / 2;
    if (n_out) *n_out = n;
    if (out) {
        if (cap < n) { set_error(e, "bqc_result_sketch: buffer too small"); return BQC_ERR_ARG; }
        memcpy(out, e->h_sketch.data() + ((uint64_t)lane * e->n_qk + qk) * e->sketch_words_per_qk, n * 8);
    }
    return 0;
}

// (size_t)(double) as g++ compiles it on x86-64, including NaN -> 2^63 (empty sketch, SURVEY D.3)
static uint64_t double_to_size(double v) {
    if (std::isnan(v)) return 9223372036854775808ULL;
    if (v >= 9223372036854775808.0) return (uint64_t)(int64_t)(v - 9223372036854775808.0) ^ 0x8000000000000000ULL;
    return (uint64_t)(int64_t)v;
}

// KmerStream estimators from per-level nibble statistics (src/kmerstream/StreamCounter.hpp:114-172,308-317)
extern "C" int bqc_result_estimates(bqc_engine* e, int32_t lane, int32_t qk, uint64_t out4[4]) {
    int rc = fetch_results(e);
    if (rc) return rc;
    if (lane < 0 || (uint32_t)lane >= e->n_lanes || qk < 0 || (uint32_t)qk >= e->n_qk) { set_error(e, "bqc_result_estimates: bad index"); return BQC_ERR_ARG; }
    const Layout& L = e->L;
    const uint64_t* G = e->h_counters.data() + (uint64_t)lane * L.lane_stride + L.o_qk + (uint64_t)qk * L.qk_stride;
    const uint32_t* sk = e->h_sketch.data() + ((uint64_t)lane * e->n_qk + qk) * e->sketch_words_per_qk;
    const size_t R = (size_t)L.sk_size * 16;
    size_t nz[32], r0[32], r1[32];
    for (int lv = 0; lv < 32; ++lv) {
        size_t z = 0, o = 0;
        const uint32_t* w = sk + (uint64_t)lv * L.sk_size * 2;
        for (uint32_t i = 0; i < L.sk_size * 2; ++i) {
            uint32_t x = w[i];
            for (int j = 0; j < 8; ++j) {
                uint32_t v = (x >> (4 * j)) & 15u;
                z += (v == 0);
                o += (v == 1);
            }
        }
        r0[lv] = z;
        r1[lv] = o;
        nz[lv] = R - z;
    }
    out4[0] = G[0];
    {   // F0
        double sum = 0;
        int n = 0;
        double limit = 0.2;
        while (n == 0 && limit > 1e-8) {
            for (size_t i = 0; i < 32; i++) {
                size_t ts = nz[i];
                if (ts <= (1 - limit) * R && ts >= limit * R) {
                    double est = (log(1.0 - ts / ((double)R)) / log(1.0 - 1.0 / R)) * pow(2.0, i + 1);
                    sum += est;
                    n++;
                    break;
                }
            }
            limit = limit / 1.5;
        }
        out4[1] = double_to_size(sum / n);
    }
    {   // f1
        double sum = 0;
        int n = 0;
        double limit = 0.2;
        while (n == 0 && limit > 1e-8) {
            for (size_t i = 0; i < 32; i++) {
                if ((r0[i] <= (1 - limit) * R) && (r0[i] >= limit * R)) {
                    sum += (R - 1) * (r1[i] / ((double)r0[i])) * pow(2.0, i + 1);
                    n++;
                    break;
                }
            }
            limit = limit / 1.5;
        }
        out4[2] = double_to_size(sum / n);
    }
    {   // F2, sequential summation order as in the reference
        double sum = 0, sqsum = 0;
        for (size_t i = 0; i < L.f2size; i++) {
            double c = (double)G[8 + i];
            sum += c;
            sqsum += c * c;
        }
        out4[3] = double_to_size(sqsum + (sqsum - sum * sum) / L.f2size);
    }
    return 0;
}

extern "C" int bqc_result_avgqual(bqc_engine* e, int32_t lane, int32_t mate, double* out, uint64_t cap, uint64_t* n_out) {
    uint64_t n = 0;
    int rc = bqc_result_table(e, lane, BQC_F_QUALSUM_M, mate, nullptr, 0, &n);
    if (rc) return rc;
    if (n_out) *n_out = n;
    if (!out) return 0;
    if (cap < n) { set_error(e, "bqc_result_avgqual: buffer too small"); return BQC_ERR_ARG; }
    std::vector<uint64_t> q(n);
    uint64_t nr = 0;
    bqc_result_table(e, lane, BQC_F_QUALSUM_M, mate, q.data(), n, nullptr);
    bqc_result_table(e, lane, BQC_F_READNR_M, mate, &nr, 1, nullptr);
    unsigned readnr = (unsigned)nr;  // `unsigned qualcount_readnr` (src/QualityCheck.hpp:46)
    for (uint64_t i = 0; i < n; ++i) out[i] = (q[i] / (double)readnr);  // src/QualityCheck.hpp:277
    return 0;
}
