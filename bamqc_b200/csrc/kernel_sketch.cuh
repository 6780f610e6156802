// kernel_sketch.cuh -- k_sketch32: the default-configuration (k = 32) fast path of the KmerStream sketch
// update: ReadQualityHasher::operator() (src/ReadQualityHasher.hpp:30-68) -> RepHash::update
// (src/kmerstream/RepHash.hpp:101-114) -> StreamCounter::operator() (src/kmerstream/StreamCounter.hpp:67-93).
// Same arithmetic as the generic k_sketch in kernels.cuh; the differences are mechanical:
//   * 16 bases (one 8-byte SEQ chunk) per outer iteration, fully unrolled, next chunks prefetched one
//     iteration ahead so the loads overlap the hash updates of the current chunk;
//   * with k = 32 the base leaving the window sits at the same nibble of the chunk two iterations back,
//     so the lagging SEQ stream needs no loads at all;
//   * the four 128-bit table lookups per base collapse into one 32-byte row indexed by (in, out):
//     row = { H[in] ^ rotl_k(H[out]),  rotl_k(Ht[in]) ^ Ht[out] }.
#pragma once
#include "sketch_sched.h"

namespace bqc {

// Only the low 64 bits of both 128-bit states are ever used (hash = h.lo ^ ht.lo) and a base stays in the window
// for k = 32 steps, so each state can be carried in 96 bits without changing a single hash:
//   h  = XOR_j rotl^j(H[s_j]), j = 0..31: its low word takes at most the top 31 bits of H.hi, bits of H.lo that rotate
//        up into hi would need 64 more steps to come back -> keep (lo, top 32 bits of hi); the 32-bit hi part simply
//        shifts left and a base's contribution leaves it by itself after 32 steps;
//   ht = XOR_m rotl^m(Ht[s]), m = 31..0, rotated RIGHT each step: bits come back into lo from the LOW end of hi ->
//        keep (lo, low 32 bits of hi) with bits 0..32 of Ht.hi cleared in the table (they never reach lo in 32 steps).
// One 32-byte row per (strand, in, out): {a_lo, b_lo, a_hi32, b_hi32} with a = H[in] ^ rotl_k(H[out]) and
// b = rotl_k(Ht''[in]) ^ Ht''[out]; the generic k_sketch keeps the full 128-bit arithmetic of the reference.
struct HashPairRow {
    uint64_t a_lo, b_lo;
    uint32_t a_hi, b_hi;
    uint32_t pad[2];
};
struct HashPairTable {  // [strand][in 0..15][out 0..16]
    HashPairRow row[2][16][17];
};

// Valid k-mer hashes are rare on low-quality stretches (one base under the cutoff silences the next k windows), so
// probing the sketch straight from the per-base loop would run the ~70 instructions of a probe for a handful of
// active lanes.  Instead each lane appends its hash to a per-warp queue in shared memory (ballot + rank) and the
// warp probes 32 queued hashes at a time with every lane busy.  The order of the updates does not matter: F2 and
// sumCount are sums, the sketch counters saturate at 15.
static const uint32_t kSketchQueue = 64;  // entries per warp (at most 31 waiting + 32 new)

struct SketchProbe {  // one in-flight probe per lane: the word was loaded, the 4-bit increment is still to be done
    uint32_t word;       // index of the sketch word (kNone: nothing pending)
    uint32_t sh, old;
    __device__ __forceinline__ void finish(uint32_t* sk) {
        if (word != kNone) {
            while (((old >> sh) & 15u) != 15u) {  // 4-bit saturating increment
                const uint32_t assumed = old;
                old = atomicCAS(sk + word, assumed, assumed + (1u << sh));
                if (old == assumed) break;
            }
            word = kNone;
        }
    }
};

// k_sketch32v2: the increment is pipelined one stage further.  A probe goes through three drains of the warp's queue:
// the sketch word is loaded (issue), the CAS of the incremented word is sent (cas), and only then is its outcome looked
// at (check) -- the L2 round trips of the load and of the CAS both overlap the hashing of the next 8 bases of every
// lane instead of stalling the warp (the blocking CAS loop of SketchProbe held 38 % of the stall samples of the
// kernel, profiles/r2).  A CAS that lost a race (rare: another warp hit the same 32-bit word in between) is
// repeated in place.
struct SketchProbe2 {
    uint32_t word, sh, old;              // stage 1: word index (kNone: empty), nibble shift, loaded value
    uint32_t cword, csh, cexp, cold;     // stage 2: CAS sent with expected value cexp, cold = what it returned
    __device__ __forceinline__ void check(uint32_t* sk) {    // stage 2 -> done
        if (cword != kNone) {
            while (cold != cexp && ((cold >> csh) & 15u) != 15u) {
                cexp = cold;
                cold = atomicCAS(sk + cword, cexp, cexp + (1u << csh));
            }
            cword = kNone;
        }
    }
    __device__ __forceinline__ void advance(uint32_t* sk) {  // check the CAS in flight, send the CAS of the loaded word
        check(sk);
        if (word != kNone) {
            if (((old >> sh) & 15u) != 15u) {  // 4-bit saturating increment
                cword = word;
                csh = sh;
                cexp = old;
                cold = atomicCAS(sk + word, old, old + (1u << sh));
            }
            word = kNone;
        }
    }
    __device__ __forceinline__ void finish(uint32_t* sk) {
        advance(sk);
        check(sk);
    }
};

__global__ void __launch_bounds__(kSketchThreads, 1) k_sketch32(EngineView E, BatchView B, uint32_t lane, SketchParams SP, const HashTables* __restrict__ HT) {
    extern __shared__ uint32_t sm[];                 // F2 table (f2size u32), the pair table, the per-warp hash queues
    const Layout& L = E.L;
    HashPairTable* PT = reinterpret_cast<HashPairTable*>(sm + L.f2size);
    uint64_t* queue = reinterpret_cast<uint64_t*>(PT + 1) + (threadIdx.x >> 5) * kSketchQueue;
    for (uint32_t i = threadIdx.x; i < L.f2size; i += blockDim.x) sm[i] = 0;
    for (uint32_t i = threadIdx.x; i < 2 * 16 * 17; i += blockDim.x) {
        const uint32_t s = i / (16 * 17), in = (i / 17) % 16, out = i % 17;
        // HT->t[s][which][n][0] = hi, [1] = lo; which: 0 H[in], 1 rotl_k(H[out]), 2 rotl_k(Ht[in]), 3 Ht[out]
        // (rotl_32 swaps and mixes the halves: rotl_32(X).lo = X.lo << 32 | X.hi >> 32, .hi = X.hi << 32 | X.lo >> 32)
        HashPairRow r;
        r.a_lo = HT->t[s][0][in][1] ^ HT->t[s][1][out][1];
        r.a_hi = (uint32_t)(HT->t[s][0][in][0] >> 32);                 // top 32 bits of H[in].hi; the out term has none
        // Ht'' = Ht with hi bits 0..32 cleared: rotl_32(Ht'')[in].lo differs from the stored rotl_32(Ht)[in].lo in bit 0
        r.b_lo = (HT->t[s][2][in][1] & ~1ULL) ^ HT->t[s][3][out][1];
        r.b_hi = (uint32_t)HT->t[s][2][in][0];                         // low 32 bits of rotl_32(Ht[in]).hi = Ht[in].lo >> 32
        r.pad[0] = r.pad[1] = 0;
        PT->row[s][in][out] = r;
    }
    __syncthreads();
    uint64_t* G = E.counters + (uint64_t)lane * L.lane_stride + L.o_qk + (uint64_t)SP.qk * L.qk_stride;
    uint32_t* sk = E.sketch + ((uint64_t)lane * L.n_qk + SP.qk) * 32ull * (L.sk_size * 2ull);
    const uint32_t words_per_level = L.sk_size * 2u;
    const uint64_t idx_mask = (uint64_t)L.sk_size * 16ull - 1ull;
    const uint32_t f2mask = L.f2size - 1u;
    const int32_t q_thresh = SP.q_thresh;
    uint32_t warp_count = 0;                         // k-mers hashed by this warp (same value in every lane; < 2^32 per launch)
    const uint32_t lane_id = threadIdx.x & 31u;
    const uint32_t lt_mask = (1u << lane_id) - 1u;
    uint32_t qn = 0;                                 // queued hashes of this warp (uniform)
    SketchProbe probe = {kNone, 0u, 0u};

    // StreamCounter::operator() (src/kmerstream/StreamCounter.hpp:67-93) for one hash per participating lane
    auto probe_issue = [&](uint64_t hv) {
        probe.finish(sk);
        atomicAdd(sm + ((uint32_t)hv & f2mask), 1u);
        uint32_t w = hv ? (uint32_t)(__ffsll((long long)hv) - 1) : 63u;  // bitScanForward, 63 for 0
        if (w > 31u) w = 31u;
        const uint64_t index = (hv >> (w + 1u)) & idx_mask;
        probe.word = w * words_per_level + (uint32_t)(index >> 3);
        probe.sh = ((uint32_t)index & 7u) * 4u;
        probe.old = __ldcg(sk + probe.word);   // tested one drain later: the L2 latency overlaps the hashing in between
    };

    const LaneRecords LR = lane_records(B, lane);
    for (uint32_t r0 = blockIdx.x * blockDim.x + threadIdx.x - lane_id; r0 < LR.n; r0 += gridDim.x * blockDim.x) {
        const uint32_t ri = r0 + lane_id;
        const uint32_t rec = ri < LR.n ? LR[ri] : 0u;
        RecHdr h;
        bool act = ri < LR.n && lane_match(B, rec, lane);
        if (act) {
            const uint32_t off = B.offsets[rec];
            act = decode_hdr(B.bytes + off, B.offsets[rec + 1] - off, h);
        }
        act = act && !(h.flag & 0xF00u) && (h.flag & 0xC0u) && (uint32_t)h.lseq >= 32u;
        const uint32_t Ls = act ? (uint32_t)h.lseq : 0u;
        const uint32_t maxL = __reduce_max_sync(0xFFFFFFFFu, Ls);
        const uint32_t s = act ? ((h.flag >> 4) & 1u) : 0u;
        const uint8_t* seqp = act ? h.p + h.o_seq : B.bytes;
        const uint8_t* qualp = act ? h.p + h.o_qual : B.bytes;
        const HashPairRow* rows = &PT->row[s][0][0];
        uint64_t hlo = 0, tlo = 0;
        uint32_t hhi = 0, thi = 0;   // top 32 bits of h.hi, low 32 bits of ht.hi
        uint64_t seq_cur = ldu64(seqp), q_lo = ldu64(qualp), q_hi = ldu64(qualp + 8);
        uint64_t hist1 = 0, hist2 = 0;
        uint32_t run = 0;
        const uint32_t nchunks = (maxL + 15u) >> 4;
        for (uint32_t c = 0; c < nchunks; ++c) {
            // prefetch the next chunk of both streams (reads past a short record stay inside the padded batch)
            const uint64_t seq_next = ldu64(seqp + 8 * (c + 1));
            const uint64_t q_lo_next = ldu64(qualp + 16 * (c + 1)), q_hi_next = ldu64(qualp + 16 * (c + 1) + 8);
            const bool has_out = c >= 2;
#pragma unroll
            for (uint32_t j = 0; j < 16; ++j) {
                const uint32_t i = c * 16 + j;
                bool emit = false;
                if (i < Ls) {
                    const uint32_t nin = (uint32_t)(seq_cur >> (4 * (j ^ 1))) & 15u;
                    const uint32_t nout = has_out ? ((uint32_t)(hist2 >> (4 * (j ^ 1))) & 15u) : 16u;
                    const uint32_t q = (uint32_t)((j < 8 ? q_lo : q_hi) >> (8 * (j & 7))) & 255u;
                    const uint32_t ridx = nin * 17u + nout;
                    const ulonglong2 ab = *reinterpret_cast<const ulonglong2*>(rows + ridx);        // a_lo, b_lo
                    const uint2 abh = *reinterpret_cast<const uint2*>(&rows[ridx].a_hi);            // a_hi32, b_hi32
                    // h = rotl1(h) ^ H[in] ^ rotl_k(H[out])
                    hlo = ((hlo << 1) | (uint64_t)(hhi >> 31)) ^ ab.x;
                    hhi = (hhi << 1) ^ abh.x;
                    // ht = rotr1(ht ^ rotl_k(Ht[in]) ^ Ht[out])
                    const uint64_t xl = tlo ^ ab.y;
                    const uint32_t xh = thi ^ abh.y;
                    tlo = (xl >> 1) | ((uint64_t)xh << 63);
                    thi = xh >> 1;
                    const bool valid = (nin != 15u) && ((int8_t)(q + 33u) >= (int8_t)q_thresh);
                    run = valid ? run + 1u : 0u;
                    emit = run >= 32u;
                }
                const uint32_t em = __ballot_sync(0xFFFFFFFFu, emit);
                if (em) {  // warp-uniform
                    if (emit) queue[qn + __popc(em & lt_mask)] = hlo ^ tlo;
                    const uint32_t n = __popc(em);
                    qn += n;
                    warp_count += n;
                    if (qn >= 32u) {
                        __syncwarp();
                        qn -= 32u;
                        probe_issue(queue[qn + lane_id]);
                        __syncwarp();
                    }
                }
            }
            hist2 = hist1;
            hist1 = seq_cur;
            seq_cur = seq_next;
            q_lo = q_lo_next;
            q_hi = q_hi_next;
        }
    }
    __syncwarp();
    if (lane_id < qn) probe_issue(queue[lane_id]);  // what is left in the queue
    probe.finish(sk);
    if (lane_id == 0 && warp_count) atomicAdd((unsigned long long*)G, (unsigned long long)warp_count);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < L.f2size; i += blockDim.x) {
        uint32_t v = sm[i];
        if (v) atomicAdd((unsigned long long*)(G + 8 + i), (unsigned long long)v);
    }
}

// ------------------------------------------------------------------------------------------------
// k_sketch32v2 -- same arithmetic, restructured around what ncu showed in k_sketch32 (profiles/r1, profiles/r2):
//   * one __ballot_sync per base for the queue append, an `i < Ls` guard around every base and a signed-char quality
//     test + run counter in front of it (56 of ~80 warp instructions per base);
//   * the (in, out) pair table: a warp's lanes read different 32-byte rows that fall on the same banks -- 14 shared
//     memory wavefronts per 16-byte load where 4 are the minimum, i.e. the LSU pipe busy half of the kernel's time
//     and every hash step waiting ~3x longer for its row.
// Here a read is processed in sub-chunks of 8 bases, and a warp's 32 reads in two passes:
//   pass 1  each lane walks its whole read, word-parallel (sketch_sched.h): the 8-base validity mask (quality in
//           [q, 94] as one unsigned per-byte range test, base != N, inside the read) and a 32-bit validity history
//           give the sub-chunks in which a window of 32 valid bases ends.  Only those are hashed: each run of them is
//           cut into pieces of at most kPieceEmit sub-chunks, appended to a per-warp list in shared memory;
//   pass 2  the lanes take the pieces 32 at a time.  A piece is hashed from zero state kPieceWarm sub-chunks before its
//           first emitting one (exact: a window's hash depends on its 32 bases only), and per sub-chunk: the emit bits
//           again, ONE warp prefix sum of the emit counts for every lane's place in the warp's hash queue, and the 8
//           hash updates, unconditional; an emitted hash is one predicated 8-byte store at the lane's next slot.
// With binned NovaSeq-like qualities and -q 17, about 9 % of the windows are valid and 5 of the 19 sub-chunks of a
// 150 bp read emit; the pieces spread that work evenly over the lanes.  When the rounds of pieces would take the warp
// no fewer steps than walking its reads from start to end (clean data: splitting only adds warm-up), or the list
// overflows, the warp walks every lane's own read as one piece from sub-chunk 0 instead.
// The hash tables are split by linearity -- row(in, out) = row_in(in) ^ row_out(out) -- into two 16-row tables that
// are REPLICATED across the banks: a row holds 8 copies of its 16-byte part and 16 copies of its 8-byte part, lane l
// reads copy l mod 8 (l mod 16), so the lanes of a quarter (half) warp never share a bank whatever they look up:
// 4 + 4 + 2 wavefronts per base instead of ~28.  The first 32 bases of a read look up an all-zero `out` table.
// Then the warp probes the sketch for 32 queued hashes at a time with every lane busy, as before.  Taken when the
// quality threshold is an ordinary one ((char)(33 + q) in 33..127); k_sketch32 stays for the others.
// ------------------------------------------------------------------------------------------------
static const uint32_t kSketchSub = 8;                                  // bases per sub-chunk
static const uint32_t kSketchQueue2 = 31 + 32 * kSketchSub + 1;        // queue entries per warp: leftover + one sub-chunk of every lane
static const uint32_t kPlanSkip = 15;                                  // batches of 32 reads walked whole, unplanned, after a plan chose that
static const uint32_t kPieceCap = 96;                                  // piece descriptors per warp (3 rounds; fits 1024 threads in 227 KB)
// shared memory: [F2 table][in tables: 2 strands x 16 rows x 256 B][out tables: 2 strands x 16 rows x 128 B][zero: 16 x 128 B][queues][piece lists]
static const uint32_t kSkIn = 2 * 16 * 256, kSkOut = 2 * 16 * 128, kSkZero = 16 * 128;
__host__ __device__ inline uint32_t sketch32v2_smem(uint32_t f2size, uint32_t threads) {
    return f2size * 4u + kSkIn + kSkOut + kSkZero + (threads / 32u) * (kSketchQueue2 * 8u + kPieceCap * 4u);
}

// exclusive prefix sum over the warp of a count in 0..8 without a dependent shuffle chain: one ballot per bit
__device__ __forceinline__ uint32_t warp_prefix_small(uint32_t cnt, uint32_t lt_mask, uint32_t& total) {
    const uint32_t b0 = __ballot_sync(0xFFFFFFFFu, cnt & 1u), b1 = __ballot_sync(0xFFFFFFFFu, cnt & 2u);
    const uint32_t b2 = __ballot_sync(0xFFFFFFFFu, cnt & 4u), b3 = __ballot_sync(0xFFFFFFFFu, cnt & 8u);
    total = __popc(b0) + 2u * __popc(b1) + 4u * __popc(b2) + 8u * __popc(b3);
    return __popc(b0 & lt_mask) + 2u * __popc(b1 & lt_mask) + 4u * __popc(b2 & lt_mask) + 8u * __popc(b3 & lt_mask);
}

template <uint32_t THREADS>
__global__ void __launch_bounds__(THREADS, 1) k_sketch32v2(EngineView E, BatchView B, uint32_t lane, SketchParams SP, const HashTables* __restrict__ HT) {
    extern __shared__ __align__(16) uint32_t sm[];
    const Layout& L = E.L;
    uint8_t* tin = reinterpret_cast<uint8_t*>(sm + L.f2size);
    uint8_t* tout = tin + kSkIn;
    uint8_t* tzero = tout + kSkOut;
    uint64_t* queue = reinterpret_cast<uint64_t*>(tzero + kSkZero) + (threadIdx.x >> 5) * kSketchQueue2;
    uint32_t* pieces = reinterpret_cast<uint32_t*>(reinterpret_cast<uint64_t*>(tzero + kSkZero) + (THREADS / 32u) * kSketchQueue2) + (threadIdx.x >> 5) * kPieceCap;
    for (uint32_t i = threadIdx.x; i < L.f2size; i += blockDim.x) sm[i] = 0;
    // in row (strand s, nibble n): copies of {a_lo = H[in].lo, b_lo = rotl_k(Ht''[in]).lo} then of {a_hi, b_hi} (see k_sketch32);
    // out row: copies of {rotl_k(H[out]).lo, Ht[out].lo}
    for (uint32_t i = threadIdx.x; i < 2 * 16 * 8; i += blockDim.x) {
        const uint32_t s = i / 128, n = (i / 8) % 16, c = i % 8;
        uint64_t* pi = reinterpret_cast<uint64_t*>(tin + (s * 16 + n) * 256 + c * 16);
        pi[0] = HT->t[s][0][n][1];
        pi[1] = HT->t[s][2][n][1] & ~1ULL;
        uint64_t* po = reinterpret_cast<uint64_t*>(tout + (s * 16 + n) * 128 + c * 16);
        po[0] = HT->t[s][1][n][1];
        po[1] = HT->t[s][3][n][1];
    }
    for (uint32_t i = threadIdx.x; i < 2 * 16 * 16; i += blockDim.x) {
        const uint32_t s = i / 256, n = (i / 16) % 16, c = i % 16;
        uint32_t* ph = reinterpret_cast<uint32_t*>(tin + (s * 16 + n) * 256 + 128 + c * 8);
        ph[0] = (uint32_t)(HT->t[s][0][n][0] >> 32);
        ph[1] = (uint32_t)HT->t[s][2][n][0];
    }
    for (uint32_t i = threadIdx.x; i < kSkZero / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(tzero)[i] = 0;
    __syncthreads();
    uint64_t* G = E.counters + (uint64_t)lane * L.lane_stride + L.o_qk + (uint64_t)SP.qk * L.qk_stride;
    uint32_t* sk = E.sketch + ((uint64_t)lane * L.n_qk + SP.qk) * 32ull * (L.sk_size * 2ull);
    const uint32_t words_per_level = L.sk_size * 2u;
    const uint64_t idx_mask = (uint64_t)L.sk_size * 16ull - 1ull;
    const uint32_t f2mask = L.f2size - 1u;
    // valid(q) <=> (signed char)(q + 33) >= (signed char)thr with thr in 33..127  <=>  thr - 33 <= q <= 94
    const uint32_t q_lo_ok = (uint32_t)SP.q_thresh - 33u, q_span = 94u - q_lo_ok;
    unsigned long long warp_count = 0;               // k-mers hashed by this warp (same value in every lane)
    const uint32_t lane_id = threadIdx.x & 31u;
    const uint32_t sm_in = (uint32_t)__cvta_generic_to_shared(tin), sm_out = (uint32_t)__cvta_generic_to_shared(tout);
    const uint32_t zero_lo = (uint32_t)__cvta_generic_to_shared(tzero) + (lane_id & 7u) * 16u;
    const uint32_t lt_mask = (1u << lane_id) - 1u;
    const uint32_t queue_s = (uint32_t)__cvta_generic_to_shared(queue);
    uint32_t qn = 0;                                 // queued hashes of this warp (uniform, < 32 between sub-chunks)
    SketchProbe2 probe = {kNone, 0u, 0u, kNone, 0u, 0u, 0u};
    uint32_t plan_skip = 0;                          // batches of 32 reads still to walk whole without planning (uniform)

    auto probe_issue = [&](uint64_t hv) {            // StreamCounter::operator() (src/kmerstream/StreamCounter.hpp:67-93)
        probe.advance(sk);
        atomicAdd(sm + ((uint32_t)hv & f2mask), 1u);
        uint32_t w = hv ? (uint32_t)(__ffsll((long long)hv) - 1) : 63u;  // bitScanForward, 63 for 0
        if (w > 31u) w = 31u;
        const uint64_t index = (hv >> (w + 1u)) & idx_mask;
        probe.word = w * words_per_level + (uint32_t)(index >> 3);
        probe.sh = ((uint32_t)index & 7u) * 4u;
        probe.old = __ldcg(sk + probe.word);
    };

    const LaneRecords LR = lane_records(B, lane);
    uint32_t* const ticket = B.tickets ? B.tickets + 2u + SP.qk : nullptr;
    uint32_t r0 = blockIdx.x * blockDim.x + threadIdx.x - lane_id;
    for (;;) {
        if (ticket) r0 = warp_take32(ticket, lane_id);
        if (r0 >= LR.n) break;
        const uint32_t ri = r0 + lane_id;
        if (!ticket) r0 += gridDim.x * blockDim.x;
        const uint32_t rec = ri < LR.n ? LR[ri] : 0u;
        RecHdr h;
        bool act = ri < LR.n && lane_match(B, rec, lane);
        if (act) {
            const uint32_t off = B.offsets[rec];
            act = decode_hdr(B.bytes + off, B.offsets[rec + 1] - off, h);
        }
        act = act && !(h.flag & 0xF00u) && (h.flag & 0xC0u) && (uint32_t)h.lseq >= 32u;
        const uint32_t Ls = act ? (uint32_t)h.lseq : 0u;
        const uint32_t maxL = __reduce_max_sync(0xFFFFFFFFu, Ls);
        const uint32_t s = act ? ((h.flag >> 4) & 1u) : 0u;
        const uint8_t* seqp = act ? h.p + h.o_seq : B.bytes;
        const uint8_t* qualp = act ? h.p + h.o_qual : B.bytes;
        const uint32_t nsub = (maxL + kSketchSub - 1u) / kSketchSub;
        auto align64 = [](uint64_t a, uint64_t b, uint32_t sh) { return (a >> sh) | ((b << 1) << (63u - sh)); };

        // ---- pass 1: the emitting sub-chunks of this lane's read -> pieces in the warp's list
        // SEQ and QUAL are read as streams of ALIGNED 8-byte words, each loaded once and realigned in registers (one
        // SEQ word = 16 bases = two sub-chunks, one QUAL word per sub-chunk), two sub-chunks ahead of their use.  A lane
        // reads its own record, so every load touches 32 sectors per warp whatever its width: with the unaligned 4- and
        // 8-byte loads of the first version (two aligned loads each) a sector was fetched 16 times for SEQ and 8 times for
        // QUAL and the L1 data pipe was the busiest unit of the kernel (78 %, profiles/r2); now it is 4 times each.
        // A warp whose last plan was the whole-read walk skips the next kPlanSkip plans and walks whole reads straight
        // away: on clean data (every window valid) or where the list overflows (long reads), pass 1 would cost its
        // walk over the reads and save nothing; the quality profile of neighbouring reads changes slowly.
        uint32_t npieces = 0;                         // pieces of the warp (uniform; > kPieceCap: the list overflowed)
        const bool plan = plan_skip == 0u && nsub <= kPieceMaxSub;
        if (plan) {
            __syncwarp();                             // the list of the previous 32 reads has been read
            const uint64_t* sA = reinterpret_cast<const uint64_t*>((uintptr_t)seqp & ~(uintptr_t)7);
            const uint64_t* qA = reinterpret_cast<const uint64_t*>((uintptr_t)qualp & ~(uintptr_t)7);
            const uint32_t ssh = ((uint32_t)(uintptr_t)seqp & 7u) * 8u, qsh = ((uint32_t)(uintptr_t)qualp & 7u) * 8u;
            uint64_t A0 = __ldg(sA), A1 = __ldg(sA + 1);
            uint64_t Q0 = __ldg(qA), Q1 = __ldg(qA + 1), Q2 = __ldg(qA + 2);
            uint32_t hv = 0;
            PieceSplitter split = {0u, 0u};
            auto append = [&](bool close, uint32_t p_es, uint32_t p_end) {
                const uint32_t b = __ballot_sync(0xFFFFFFFFu, close);
                if (b) {  // warp-uniform
                    const uint32_t i = npieces + __popc(b & lt_mask);
                    if (close && i < kPieceCap) pieces[i] = piece_desc(lane_id, p_es, p_end);
                    npieces += __popc(b);
                }
            };
            // 16 bases (sub-chunks c, c + 1) per step; sub-chunk nsub, when c + 1 == nsub, is past every read: it emits
            // nothing and closes what is open, as the flush would
            for (uint32_t c = 0; c < nsub; c += 2u) {
                const uint64_t A2 = __ldg(sA + (c >> 1) + 2u);              // reads past a short record stay inside the padded batch
                const uint64_t Q3 = __ldg(qA + c + 3u), Q4 = __ldg(qA + c + 4u);
                const uint32_t e = sketch_emit16(hv, sketch_valid16(align64(Q0, Q1, qsh), align64(Q1, Q2, qsh), align64(A0, A1, ssh), c, Ls, q_lo_ok, q_span));
                uint32_t p_es = 0, p_end = 0;
                bool close = split.step(c, (e & 0xFFu) != 0u, p_es, p_end);
                close |= split.step(c + 1u, (e >> 8) != 0u, p_es, p_end);
                append(close, p_es, p_end);
                A0 = A1; A1 = A2;
                Q0 = Q2; Q1 = Q3; Q2 = Q4;
            }
            uint32_t p_es = 0, p_end = 0;
            const bool close = split.flush(nsub, p_es, p_end);
            append(close, p_es, p_end);
            __syncwarp();
        }
        // rounds of 32 pieces take the longest piece of each round (pieces in the order they were found: longest-first
        // would save about 6 % of the steps at -q 17 in a model of the synthetic library); walking the reads from
        // sub-chunk 0 takes nsub steps
        uint32_t split_steps = 0;
        const uint32_t split_rounds = (npieces + 31u) / 32u;
        if (plan && npieces <= kPieceCap) {
            for (uint32_t r = 0; r < split_rounds; ++r) {
                const uint32_t i = r * 32u + lane_id;
                const uint32_t d = i < npieces ? pieces[i] : 0u;
                split_steps += __reduce_max_sync(0xFFFFFFFFu, (d >> 16) - piece_warm_start((d >> 8) & 255u));
            }
        }
        const bool use_pieces = plan && npieces <= kPieceCap && split_steps < nsub;
        if (plan) plan_skip = use_pieces ? 0u : kPlanSkip;
        else if (plan_skip) --plan_skip;
        const uint32_t nrounds = use_pieces ? split_rounds : 1u;

        // ---- pass 2: the hash updates, one piece per lane and round
        for (uint32_t r = 0; r < nrounds; ++r) {
            uint32_t own = lane_id, es = 0, end = use_pieces ? 0u : nsub;   // unsplit: the lane's own read, sub-chunks 0..nsub-1
            if (use_pieces && r * 32u + lane_id < npieces) {
                const uint32_t d = pieces[r * 32u + lane_id];
                own = d & 31u;
                es = (d >> 8) & 255u;
                end = d >> 16;
            }
            const uint32_t ws = piece_warm_start(es);
            const uint32_t steps = __reduce_max_sync(0xFFFFFFFFu, end - ws);
            // the owning lane's read
            const uint8_t* pseq = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)(uintptr_t)seqp, own));
            const uint8_t* pqual = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)(uintptr_t)qualp, own));
            const uint32_t pLs = __shfl_sync(0xFFFFFFFFu, Ls, own), ps = __shfl_sync(0xFFFFFFFFu, s, own);
            // this lane's copies: the row offset (nibble << 8, nibble << 7) is added to these shared-memory addresses
            const uint32_t in_lo = sm_in + ps * 4096u + (lane_id & 7u) * 16u, in_hi = sm_in + ps * 4096u + 128u + (lane_id & 15u) * 8u;
            const uint32_t out_lo = sm_out + ps * 2048u + (lane_id & 7u) * 16u;
            // a piece starts at any sub-chunk: SEQ as aligned 4-byte words (one per sub-chunk), QUAL as aligned 8-byte words,
            // realigned in registers and loaded one sub-chunk ahead; never past word end + 1 of the piece's read.  One
            // 4-byte SEQ load per sub-chunk instead of an 8-byte one per two keeps a piece free to start at an odd
            // sub-chunk; with pass 1 that is more global loads per read than one walk, but each hashed sub-chunk saved
            // drops 24 table LDS (80 shared wavefronts) from the same L1 pipe
            const uint32_t* sW = reinterpret_cast<const uint32_t*>((uintptr_t)pseq & ~(uintptr_t)3);
            const uint64_t* qA = reinterpret_cast<const uint64_t*>((uintptr_t)pqual & ~(uintptr_t)7);
            const uint32_t ssh = ((uint32_t)(uintptr_t)pseq & 3u) * 8u, qsh = ((uint32_t)(uintptr_t)pqual & 7u) * 8u;
            uint32_t S0 = __ldg(sW + ws), S1 = __ldg(sW + ws + 1u);
            uint64_t Q0 = __ldg(qA + ws), Q1 = __ldg(qA + ws + 1u);
            uint64_t hlo = 0, tlo = 0;
            uint32_t hhi = 0, thi = 0;                // top 32 bits of h.hi, low 32 bits of ht.hi
            uint32_t lag0 = 0, lag1 = 0, lag2 = 0, lag3 = 0;  // SEQ words of the last 4 sub-chunks, oldest first (the base leaving a 32-window sits 4 words back)
            uint32_t hv = 0;                          // validity of the last 32 bases, oldest in bit 0
            for (uint32_t t = 0; t < steps; ++t) {
                const uint32_t c = ws + t;
                const uint32_t nx = min(c + 2u, end + 1u);
                const uint32_t S2 = __ldg(sW + nx);
                const uint64_t Q2 = __ldg(qA + nx);
                const uint32_t seq_cur = __funnelshift_r(S0, S1, ssh);
                uint32_t emit = sketch_emit8(hv, sketch_valid8(align64(Q0, Q1, qsh), seq_cur, c, pLs, q_lo_ok, q_span));
                if (c < es || c >= end) emit = 0u;    // warm-up (hashed by the previous piece) or past the piece
                uint32_t total;
                const uint32_t excl = warp_prefix_small(__popc(emit), lt_mask, total);
                uint32_t qp = queue_s + 8u * (qn + excl);                   // this lane's next queue slot
                // h = rotl1(h) ^ H[in] ^ rotl_k(H[out]), ht = rotr1(ht ^ rotl_k(Ht[in]) ^ Ht[out]); the first 32 bases
                // after the (re)start look up the all-zero `out` table
                const uint32_t outw = lag0;
                const uint32_t o_base = c >= ws + 4u ? out_lo : zero_lo;
#pragma unroll
                for (uint32_t j = 0; j < 8; ++j) {
                    const uint32_t sh = 4u * (j ^ 1u);
                    const uint32_t ni = sh >= 8u ? (seq_cur >> (sh - 8u)) & 0xF00u : (seq_cur << (8u - sh)) & 0xF00u;   // nibble << 8
                    const uint32_t no = sh >= 7u ? (outw >> (sh - 7u)) & 0x780u : (outw << (7u - sh)) & 0x780u;         // nibble << 7
                    uint64_t a_lo, b_lo, oa_lo, ob_lo;
                    uint32_t a_hi, b_hi;
                    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(a_lo), "=l"(b_lo) : "r"(in_lo + ni));
                    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(a_hi), "=r"(b_hi) : "r"(in_hi + ni));
                    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(oa_lo), "=l"(ob_lo) : "r"(o_base + no));
                    hlo = ((hlo << 1) | (uint64_t)(hhi >> 31)) ^ a_lo ^ oa_lo;
                    hhi = (hhi << 1) ^ a_hi;
                    const uint64_t xl = tlo ^ b_lo ^ ob_lo;
                    const uint32_t xh = thi ^ b_hi;
                    tlo = (xl >> 1) | ((uint64_t)xh << 63);
                    thi = xh >> 1;
                    if ((emit >> j) & 1u) {
                        const uint64_t hval = hlo ^ tlo;
                        asm volatile("st.shared.u64 [%0], %1;" ::"r"(qp), "l"(hval) : "memory");
                        qp += 8u;
                    }
                }
                lag0 = lag1; lag1 = lag2; lag2 = lag3; lag3 = seq_cur;
                S0 = S1; S1 = S2;
                Q0 = Q1; Q1 = Q2;
                if (total) {  // warp-uniform
                    __syncwarp();
                    warp_count += total;
                    const uint32_t have = qn + total;
                    uint32_t done = 0;
                    for (; done + 32u <= have; done += 32u) probe_issue(queue[done + lane_id]);
                    const uint32_t rest = have - done;
                    if (done && rest) {                                     // what is left moves to the front of the queue
                        const uint64_t v = lane_id < rest ? queue[done + lane_id] : 0ull;
                        __syncwarp();
                        if (lane_id < rest) queue[lane_id] = v;
                    }
                    qn = rest;
                    __syncwarp();
                }
            }
        }
    }
    __syncwarp();
    if (lane_id < qn) probe_issue(queue[lane_id]);  // what is left in the queue
    probe.finish(sk);
    if (lane_id == 0 && warp_count) atomicAdd((unsigned long long*)G, warp_count);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < L.f2size; i += blockDim.x) {
        uint32_t v = sm[i];
        if (v) atomicAdd((unsigned long long*)(G + 8 + i), (unsigned long long)v);
    }
}

}  // namespace bqc
