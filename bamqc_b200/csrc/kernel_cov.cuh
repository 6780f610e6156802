// kernel_cov.cuh -- OverallNumbers::coverage + update_coverage / update_vectors (src/OverallNumbers.hpp:59-135,
// src/bamqualcheck.cpp:430-433, 447-453) entirely on the device.  Included by kernels.cuh (namespace bqc).
//
// The reference keeps two 1000-position depth windows anchored at data-dependent positions and histograms a window
// when the read stream moves past it -- the only order-dependent statistic of the program.  Here (cov_math.h):
//   k_cov_prep    ordered compaction of the records that take part (primary, mapped, not duplicate, on a main
//                 contig): (rid, begin, covered interval relative to begin) -- single pass, decoupled look-back;
//   k_cov_tables  the anchor recurrence as a function of the unknown state at the start of each block of 2048
//                 compact records: blocks without a "candidate" (contig change or gap >= 1000) have a closed form,
//                 blocks with a contig change end in a known state, the rest are simulated for all 1002 states;
//   k_cov_link    chains the block functions from the carried state (one thread, one step per block);
//   k_cov_codes   with the state at block entry known: state of every record in closed form, its virtual
//                 coordinate X = 1000 * window + pos as a prefix sum (look-back across blocks), covered interval
//                 [X + a, X + b) clipped where the reference's writes leave its two windows;
//   k_cov_tiles   depth histogram: the virtual axis is cut into tiles of 1024 positions, one warp per tile; the warp
//                 builds the tile's difference array in shared memory from the records that overlap it (a record only
//                 writes into its two windows and window starts never decrease, even for unsorted input, so those
//                 are the records whose window start lies in the tile or in the two before), marks the positions that
//                 hold an event in a bitmap, prefix-sums the events and adds run lengths of equal depth to
//                 poscov[min(depth, 100)] -- it touches the events, not the positions;
//   k_cov_carry   the two windows that are still open after the batch's last record (the reference's v1 | v2)
//                 become a 2001-entry difference array that the next batch (or k_cov_final) starts from.
// There is no depth array in global memory and no host work: cost is proportional to the records plus 1/32 of the
// occupied virtual span.  All state lives in CovCarry on the device, so batches replay without the host.
#pragma once
#include "cov_math.h"

namespace bqc {

static const uint32_t kCovRB = 2048;        // compact records per anchor block
static const uint32_t kCovBlockThreads = 1024;
static const uint32_t kCovTile = 1024;      // virtual positions per tile: one warp, 32 positions per lane
static const uint32_t kCovTileThreads = 256;
static const uint32_t kCovD = 2048;         // entries of a carry difference array (2001 used)
static const uint32_t kCovPrepTile = 1024;  // records per compaction tile
static const uint32_t kCovPrepPer = 1;      // records per thread (one: every header is its own dependent load chain)
static const uint32_t kCovPrepThreads = kCovPrepTile / kCovPrepPer;
enum { COV_CLOSED = 0, COV_CONST = 1, COV_TABLE = 2 };

struct CovCarry {  // per lane
    uint32_t first;              // no qualifying record yet (OverallNumbers::first)
    int32_t rid_prev;            // last qualifying record: contig, begin, state p = begin - shift
    uint32_t b_prev;
    uint32_t p_prev;
    unsigned long long xc;       // virtual coordinate of the start of its window v1 (a multiple of 1000): poscov is final
                                 // below xc, the carry difference array covers [xc, xc + 2000] = the reference's v1 | v2
    uint32_t parity;             // which of the two carry difference arrays is current
    // batch in flight
    uint32_t nq;                 // qualifying records
    uint32_t ntiles;             // tiles of [xc, xl)
    uint32_t vt_last;            // tile that holds the window start of the batch's last record (ntiles - 1 or ntiles)
    unsigned long long xl;       // window start of the batch's last qualifying record = the next xc
    int32_t n_rid;               // state after it (becomes *_prev in k_cov_carry)
    uint32_t n_b, n_p, pad1;
};

struct CovScratch {  // sized for the largest batch; reused by every batch and lane (one stream)
    int32_t* q_rid;
    uint32_t* q_b;
    uint32_t* q_iv;
    uint32_t* q_rec;                 // batch index of the record (complex CIGARs are re-walked)
    uint8_t* q_lane;                 // several read groups: lane of the record (shard mode collects all lanes in one queue)
    unsigned long long* base;       // virtual coordinate of the record's begin
    uint32_t* ab;                    // covered interval [a, b) relative to base: a | b << 11; complex: p | bit 31
    uint16_t* tables;                // [block][1024] state -> state (COV_TABLE blocks)
    uint4* desc;                     // [block] {type, a, b, -}
    uint32_t* state_in;              // [block] state at block entry
    uint32_t* first_rec;             // [tile] first compact record whose window start lies in the tile or beyond
    unsigned long long* lb_prep;     // look-back states
    unsigned long long* lb_codes;
    uint32_t* tickets;               // [0] prep, [1] codes
};

__global__ void k_cov_init(CovCarry* carry, uint32_t n_lanes) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lanes) return;
    CovCarry c = {};
    c.first = 1u;
    carry[i] = c;
}

// ------------------------------------------------------------------------------------------------
// Decoupled look-back (tiles handed out in ticket order, so a tile only ever waits for tiles that are running or
// done).  state[t]: bits 63..62 = 0 empty / 1 aggregate / 2 inclusive prefix, low 62 bits = value.  Called by the 32
// lanes of one warp; returns the exclusive prefix of `tile` (first_prefix for tile 0) in every lane.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long cov_lookback(unsigned long long* state, uint32_t tile, unsigned long long aggregate, unsigned long long first_prefix) {
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned long long kVal = (1ull << 62) - 1ull;
    unsigned long long prefix = first_prefix;
    if (tile != 0) {
        if (lane == 0) atomicExch(state + tile, (1ull << 62) | (aggregate & kVal));
        prefix = 0;
        long long look = (long long)tile - 1;
        for (;;) {
            const long long t = look - (long long)lane;
            unsigned long long st = 2ull << 62;  // before tile 0: inclusive, contributes nothing
            if (t >= 0) {
                do { st = *((volatile unsigned long long*)(state + t)); } while ((st >> 62) == 0);
            }
            const uint32_t incl_mask = __ballot_sync(0xFFFFFFFFu, (st >> 62) == 2ull);
            const uint32_t firsti = incl_mask ? (uint32_t)(__ffs((int)incl_mask) - 1) : 32u;
            unsigned long long contrib = lane <= firsti ? (st & kVal) : 0ull;
            for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xFFFFFFFFu, contrib, o);
            prefix += contrib;
            if (incl_mask) break;
            look -= 32;
        }
        prefix &= kVal;  // aggregates may be negative (62-bit two's complement); prefixes are not
    }
    if (lane == 0) atomicExch(state + tile, (2ull << 62) | ((prefix + aggregate) & kVal));
    return prefix;
}

// inclusive scan of one value per thread over the CTA (blockDim.x <= 1024, multiple of 32); ws: 33 words of smem
__device__ __forceinline__ uint32_t cov_block_scan(uint32_t v, uint32_t* ws, uint32_t& total) {
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    uint32_t incl = v;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    __syncthreads();  // ws may still be read from a previous call
    if (lane == 31u) ws[w] = incl;
    __syncthreads();
    if (w == 0) {
        const uint32_t nw = blockDim.x >> 5;
        const uint32_t x = lane < nw ? ws[lane] : 0u;
        uint32_t xi = x;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, xi, o);
            if (lane >= (uint32_t)o) xi += t;
        }
        ws[lane] = xi - x;
        if (lane == 31u) ws[32] = xi;
    }
    __syncthreads();
    total = ws[32];
    return incl + ws[w];
}

// The covered intervals of a record relative to its begin (src/OverallNumbers.hpp:112-134): read-oriented CIGAR, S
// adds to the offset, M and D cover [c, c + n) and advance it, everything else is ignored.  emit(s, e) per maximal
// run of contiguous covered positions.
template <typename F>
__device__ __forceinline__ void cov_walk_cigar(const uint8_t* p, F emit) {
    const uint32_t x = ldu32(p + 12), y = ldu32(p + 16);
    const uint32_t lname = x & 255u, ncig = y & 0xFFFFu;
    const bool rc = ((y >> 16) & 0x10u) != 0;
    const uint8_t* cig = p + 36u + lname;
    uint32_t c = 0, s = 0, e = 0;
    bool have = false;
    for (uint32_t i = 0; i < ncig; ++i) {
        const uint32_t ce = ldu32(cig + 4u * (rc ? (ncig - 1u - i) : i));
        const uint32_t op = ce & 15u, n = ce >> 4;
        if (op == 4u) c += n;
        if (op == 0u || op == 2u) {
            if (n) {
                if (have && c != e) { emit(s, e); have = false; }
                if (!have) { s = c; have = true; }
                e = c + n;
            }
            c += n;
        }
    }
    if (have) emit(s, e);
}

// ------------------------------------------------------------------------------------------------
// k_cov_prep: which records take part (src/bamqualcheck.cpp:318-327,385-389,392,430: primary, first or last, mapped,
// not duplicate, rID in the -c set) and their (rid, begin, interval), compacted in file order.
// ------------------------------------------------------------------------------------------------
// append != 0 (shard mode): the records are added behind the carry->nq already collected instead of replacing them.
// kTagged (shard mode, several read groups): every record of the batch whatever its lane, each tagged with its lane
// in S.q_lane; the queue is grouped by lane once the run has ended (engine.cu cov_lane_split).
template <bool kTagged>
__global__ void __launch_bounds__(kCovPrepThreads, 2) k_cov_prep(EngineView E, BatchView B, uint32_t lane, CovScratch S, CovCarry* carry, uint32_t append) {
    __shared__ uint32_t ws[33];
    __shared__ uint32_t s_tile;
    __shared__ unsigned long long s_base;
    const LaneRecords LR = kTagged ? LaneRecords{B.n_records, nullptr} : lane_records(B, lane);
    const uint32_t ntile = (LR.n + kCovPrepTile - 1u) / kCovPrepTile;
    const uint32_t have = append ? carry->nq : 0u;   // only tile 0 uses it, and the last tile overwrites it after tile 0 has published
    for (;;) {
        if (threadIdx.x == 0) s_tile = atomicAdd(S.tickets + 0, 1u);
        __syncthreads();
        const uint32_t tile = s_tile;
        if (tile >= ntile) break;
        int32_t rid[kCovPrepPer];
        uint32_t b[kCovPrepPer], iv[kCovPrepPer], recno[kCovPrepPer], flags = 0;
        const uint32_t r0 = tile * kCovPrepTile + kCovPrepPer * threadIdx.x;
#pragma unroll
        for (uint32_t k = 0; k < kCovPrepPer; ++k) {
            rid[k] = -1; b[k] = 0; iv[k] = 0; recno[k] = 0;
            if (r0 + k >= LR.n) continue;
            const uint32_t r = LR[r0 + k];
            recno[k] = r;
            if (!kTagged && !lane_match(B, r, lane)) continue;
            const uint32_t off = B.offsets[r], avail = B.offsets[r + 1] - off;
            if (avail < 36u) continue;
            const uint8_t* p = B.bytes + off;
            const uint32_t x = ldu32(p + 12), y = ldu32(p + 16);
            const uint32_t flag = y >> 16, ncig = y & 0xFFFFu, lname = x & 255u;
            const int32_t id = (int32_t)ldu32(p + 4);
            if ((flag & 0x900u) || !(flag & 0xC0u) || (flag & 0x4u) || (flag & 0x400u)) continue;
            if (id < 0 || id >= E.n_ref || !E.main_chrom[id]) continue;
            if (36u + lname + 4u * ncig > avail) continue;  // malformed: k_stats reports the record
            uint32_t s0 = 0, e0 = 0, nint = 0;
            cov_walk_cigar(p, [&](uint32_t s, uint32_t e) { if (nint == 0) { s0 = s; e0 = e; } ++nint; });
            rid[k] = id;
            b[k] = ldu32(p + 8);
            iv[k] = cov_pack_iv(s0, e0 - s0, nint > 1u);
            if (append && nint > 1u) report_error(E, B.first_record + r, 16);  // the record bytes are gone when a shard is resolved
            flags |= 1u << k;
        }
        uint32_t total;
        const uint32_t cnt = __popc(flags);
        const uint32_t excl = cov_block_scan(cnt, ws, total) - cnt;
        if (threadIdx.x < 32) {
            const unsigned long long pre = cov_lookback(S.lb_prep, tile, total, (unsigned long long)have);
            if (threadIdx.x == 0) {
                s_base = pre;
                if (tile == ntile - 1u) carry->nq = (uint32_t)(pre + total);
            }
        }
        __syncthreads();
        uint32_t o = (uint32_t)s_base + excl;
#pragma unroll
        for (uint32_t k = 0; k < kCovPrepPer; ++k)
            if (flags & (1u << k)) {
                S.q_rid[o] = rid[k]; S.q_b[o] = b[k]; S.q_iv[o] = iv[k]; S.q_rec[o] = recno[k];
                if (kTagged) S.q_lane[o] = B.rec_lane[recno[k]];
                ++o;
            }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// Block analysis shared by k_cov_tables and k_cov_codes: positions 1..n are the block's compact records, position 0
// is the record before the block.  Candidate ordinal 0 is that record (its "stretch" is the head of the block).
// ------------------------------------------------------------------------------------------------
struct CovBlock {
    uint32_t* sb;     // [RB+1] begins
    int32_t* srid;    // [RB+1] contigs
    uint32_t* cg;     // [RB+2] per candidate: gap                         (k_cov_codes: advance of X at the candidate)
    uint32_t* cGs;    // [RB+2] begin of the stretch's last record - begin of the candidate   (k_cov_codes: state after it)
    uint32_t* cGj;    // [RB+2] begin of the stretch's last record - begin of j*
    uint16_t* cord;   // [RB+2] per position: ordinal of the governing candidate
    uint16_t* cpos;   // [RB+2] per candidate: position; cpos[nc + 1] = n + 1
    uint16_t* cjs;    // [RB+2] per candidate: j* (first position of the stretch whose begin differs), 0 = none
    uint8_t* cdef;    // [RB+2] per candidate: resets from every state (contig change, first record ever, gap in [2001, 2^32 - 2001])
    uint32_t* ws;     // [36]
    uint32_t n, nc;
    bool isfirst;
};
static const uint32_t kCovBlockSmem = ((kCovRB + 1) * 8 + (kCovRB + 2) * (12 + 6 + 1) + 36 * 4 + 64 + 15) & ~15u;
static const uint32_t kCovCodesSmem = kCovBlockSmem + (kCovRB + 1) * 4;  // + window starts (k_cov_codes)

__device__ __forceinline__ void cov_block_carve(CovBlock& K, uint8_t* smem) {
    K.sb = (uint32_t*)smem;
    K.srid = (int32_t*)(K.sb + kCovRB + 1);
    K.cg = (uint32_t*)(K.srid + kCovRB + 1);
    K.cGs = K.cg + kCovRB + 2;
    K.cGj = K.cGs + kCovRB + 2;
    K.ws = K.cGj + kCovRB + 2;
    K.cord = (uint16_t*)(K.ws + 36);
    K.cpos = K.cord + kCovRB + 2;
    K.cjs = K.cpos + kCovRB + 2;
    K.cdef = (uint8_t*)(K.cjs + kCovRB + 2);
}

// blockDim.x == kCovBlockThreads; every thread owns positions 2t+1, 2t+2
__device__ __forceinline__ void cov_block_analyse(CovBlock& K, const CovScratch& S, const CovCarry* carry, uint32_t blk, uint32_t nq) {
    const uint32_t r0 = blk * kCovRB;
    const uint32_t n = min(kCovRB, nq - r0);
    K.n = n;
    K.isfirst = blk == 0 && carry->first != 0;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) { K.sb[i + 1] = S.q_b[r0 + i]; K.srid[i + 1] = S.q_rid[r0 + i]; }
    if (threadIdx.x == 0) {
        if (blk) { K.sb[0] = S.q_b[r0 - 1]; K.srid[0] = S.q_rid[r0 - 1]; }
        else if (K.isfirst) { K.sb[0] = S.q_b[0]; K.srid[0] = S.q_rid[0]; }
        else { K.sb[0] = carry->b_prev; K.srid[0] = carry->rid_prev; }
    }
    __syncthreads();
    uint32_t f = 0;
#pragma unroll
    for (uint32_t k = 0; k < 2; ++k) {
        const uint32_t i = 2u * threadIdx.x + 1u + k;
        if (i <= n) {
            const bool other = K.srid[i] != K.srid[i - 1] || (K.isfirst && i == 1u);
            const uint32_t g = K.sb[i] - K.sb[i - 1];
            if (other || g >= kCovV) f |= ((other || cov_gap_definite(g)) ? 3u : 1u) << (2u * k);
        }
    }
    uint32_t total;
    const uint32_t cnt = (f & 1u) + ((f >> 2) & 1u);
    uint32_t ord = cov_block_scan(cnt, K.ws, total) - cnt;  // candidates before position 2t+1
    K.nc = total;
    if (threadIdx.x == 0) { K.cord[0] = 0; K.cpos[0] = 0; K.cg[0] = 0; K.cdef[0] = 0; K.cjs[0] = 0; K.cpos[total + 1] = (uint16_t)(n + 1u); }
#pragma unroll
    for (uint32_t k = 0; k < 2; ++k) {
        const uint32_t i = 2u * threadIdx.x + 1u + k;
        if (i <= n) {
            if ((f >> (2u * k)) & 1u) {
                ++ord;
                K.cpos[ord] = (uint16_t)i;
                K.cg[ord] = K.sb[i] - K.sb[i - 1];
                K.cdef[ord] = (uint8_t)((f >> (2u * k + 1u)) & 1u);
                K.cjs[ord] = 0;
            }
            K.cord[i] = (uint16_t)ord;
        }
    }
    __syncthreads();
#pragma unroll
    for (uint32_t k = 0; k < 2; ++k) {  // j*: the first record of a stretch that leaves the candidate's position
        const uint32_t i = 2u * threadIdx.x + 1u + k;
        if (i <= n) {
            const uint32_t c = K.cord[i];
            if (K.cpos[c] != i && K.sb[i] != K.sb[i - 1] && K.sb[i - 1] == K.sb[K.cpos[c]]) K.cjs[c] = (uint16_t)i;
        }
    }
    __syncthreads();
    for (uint32_t c = threadIdx.x; c <= K.nc; c += blockDim.x) {
        const uint32_t last = (uint32_t)K.cpos[c + 1] - 1u;
        K.cGs[c] = K.sb[last] - K.sb[K.cpos[c]];
        K.cGj[c] = K.cjs[c] ? K.sb[last] - K.sb[K.cjs[c]] : 0u;
    }
    __syncthreads();
}

// candidate c applied to state p: the record itself, then its stretch up to the next candidate
__device__ __forceinline__ uint32_t cov_block_apply(const CovBlock& K, uint32_t c, uint32_t p) {
    uint32_t q = p;
    if (c) { bool reset; q = cov_step(p, K.cg[c], K.cdef[c] != 0, reset); }
    return cov_stretch(q, K.cGs[c], K.cGj[c]);
}

__global__ void __launch_bounds__(kCovBlockThreads) k_cov_tables(CovScratch S, const CovCarry* carry) {
    extern __shared__ __align__(16) uint8_t cov_smem[];
    __shared__ uint32_t s_lastdef;
    const uint32_t nq = carry->nq;
    const uint32_t blk = blockIdx.x;
    if (blk * kCovRB >= nq) return;
    CovBlock K;
    cov_block_carve(K, cov_smem);
    cov_block_analyse(K, S, carry, blk, nq);
    if (threadIdx.x == 0) s_lastdef = 0;
    __syncthreads();
    for (uint32_t c = 1u + threadIdx.x; c <= K.nc; c += blockDim.x)
        if (K.cdef[c]) atomicMax(&s_lastdef, c);
    __syncthreads();
    const uint32_t lastdef = s_lastdef;
    if (K.nc == 0) {  // closed form: the whole block is the stretch of the record before it
        if (threadIdx.x == 0) S.desc[blk] = make_uint4(COV_CLOSED, K.cGs[0], K.cGj[0], 0u);
    } else if (lastdef) {  // whatever comes in, the state after the last contig change is known
        if (threadIdx.x == 0) {
            uint32_t p = 0;
            for (uint32_t c = lastdef; c <= K.nc; ++c) p = cov_block_apply(K, c, p);
            S.desc[blk] = make_uint4(COV_CONST, p, 0u, 0u);
        }
    } else {  // every possible state at block entry, one per thread
        if (threadIdx.x < kCovStates) {
            uint32_t p = cov_state_value(threadIdx.x);
            for (uint32_t c = 0; c <= K.nc; ++c) p = cov_block_apply(K, c, p);
            S.tables[(size_t)blk * 1024u + threadIdx.x] = (uint16_t)cov_state_index(p);
        }
        if (threadIdx.x == 0) S.desc[blk] = make_uint4(COV_TABLE, 0u, 0u, 0u);
    }
}

// State at the entry of every block.  A COV_CONST block ends in a known state, so the chain falls into independent
// segments (one thread each); inside a segment the blocks are applied one after the other.
static const uint32_t kCovLinkChunk = 2048;
__global__ void __launch_bounds__(1024) k_cov_link(CovScratch S, const CovCarry* carry) {
    __shared__ uint4 sd[kCovLinkChunk];
    __shared__ uint32_t s_p;
    const uint32_t nq = carry->nq;
    const uint32_t nblk = (nq + kCovRB - 1u) / kCovRB;
    if (threadIdx.x == 0) s_p = carry->p_prev;
    for (uint32_t b0 = 0; b0 < nblk; b0 += kCovLinkChunk) {
        const uint32_t m = min(kCovLinkChunk, nblk - b0);
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) sd[i] = S.desc[b0 + i];
        __syncthreads();
        const uint32_t p_chunk = s_p;
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) {
            if (i != 0u && sd[i - 1].x != COV_CONST) continue;   // not the start of a segment
            uint32_t p = i ? sd[i - 1].y : p_chunk;
            for (uint32_t k = i;; ++k) {
                S.state_in[b0 + k] = p;
                const uint4 d = sd[k];
                if (d.x == COV_CLOSED) p = cov_stretch(p, d.y, d.z);
                else if (d.x == COV_CONST) p = d.y;
                else p = cov_state_value(S.tables[(size_t)(b0 + k) * 1024u + cov_state_index(p)]);
                if (k + 1u == m) { s_p = p; break; }
                if (d.x == COV_CONST) break;
            }
        }
    }
}

__global__ void __launch_bounds__(kCovBlockThreads) k_cov_codes(CovScratch S, CovCarry* carry) {
    extern __shared__ __align__(16) uint8_t cov_smem[];
    __shared__ uint32_t s_blk;
    __shared__ unsigned long long s_x0;
    const uint32_t nq = carry->nq;
    const uint32_t nblk = (nq + kCovRB - 1u) / kCovRB;
    const unsigned long long xc = carry->xc;
    const unsigned long long x_prev = xc + carry->p_prev;  // virtual coordinate of the last record before the batch
    CovBlock K;
    cov_block_carve(K, cov_smem);
    int32_t* vrel = (int32_t*)(cov_smem + kCovBlockSmem);  // [RB+1] window start of every position relative to the block's X0
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_blk = atomicAdd(S.tickets + 1, 1u);
        __syncthreads();
        const uint32_t blk = s_blk;
        if (blk >= nblk) break;
        cov_block_analyse(K, S, carry, blk, nq);
        const uint32_t p_in = S.state_in[blk];
        // the candidates with the true state: cGs[c] <- state right after candidate c, cg[c] <- advance of X at c.  A
        // definite candidate starts from a reset whatever came before, so every run [definite candidate .. next one)
        // is walked by its own thread; the walker also leaves the advance of X for the definite candidate that ends
        // its run (2000 - p of the record before it).
        for (uint32_t c0 = threadIdx.x; c0 <= K.nc; c0 += blockDim.x) {
            if (c0 != 0u && !K.cdef[c0]) continue;
            uint32_t p = p_in;
            for (uint32_t c = c0;; ++c) {
                uint32_t q = p;
                if (c == c0) { if (c) q = 0u; }
                else {
                    bool reset;
                    const uint32_t g = K.cg[c];
                    q = cov_step(p, g, false, reset);
                    K.cg[c] = cov_dx(p, g, reset);
                }
                p = cov_stretch(q, K.cGs[c], K.cGj[c]);
                K.cGs[c] = q;
                if (c == K.nc) break;
                if (K.cdef[c + 1u]) { K.cg[c + 1u] = (K.isfirst && c == 0u) ? 0u : 2u * kCovV - p; break; }
            }
        }
        __syncthreads();
        uint32_t pst[2], dx[2];
#pragma unroll
        for (uint32_t k = 0; k < 2; ++k) {
            const uint32_t i = 2u * threadIdx.x + 1u + k;
            pst[k] = 0; dx[k] = 0;
            if (i <= K.n) {
                const uint32_t c = K.cord[i], cp = K.cpos[c], q = K.cGs[c];
                if (c && cp == i) { pst[k] = q; dx[k] = K.cg[c]; }
                else {
                    const uint32_t js = K.cjs[c], g = K.sb[i] - K.sb[i - 1];
                    if (q == kCovEdge && i == js) { pst[k] = 0; dx[k] = 0; }  // the reset after an edge record: X stays (2000 - p = 0)
                    else { pst[k] = cov_stretch(q, K.sb[i] - K.sb[cp], js ? K.sb[i] - K.sb[js] : 0u); dx[k] = g; }
                }
            }
        }
        // X: prefix sum of the advances (two's complement: a backward step inside the windows moves X back)
        uint32_t total;
        const uint32_t incl = cov_block_scan(dx[0] + dx[1], K.ws, total);
        if (threadIdx.x < 32) {
            const unsigned long long pre = cov_lookback(S.lb_codes, blk, (unsigned long long)(long long)(int32_t)total, x_prev);
            if (threadIdx.x == 0) s_x0 = pre;
        }
        {
            int32_t xr = (int32_t)(incl - dx[0] - dx[1]);
            if (threadIdx.x == 0) vrel[0] = -(int32_t)p_in;
#pragma unroll
            for (uint32_t k = 0; k < 2; ++k) {
                const uint32_t i = 2u * threadIdx.x + 1u + k;
                xr += (int32_t)dx[k];
                if (i <= K.n) vrel[i] = xr - (int32_t)pst[k];
            }
        }
        __syncthreads();
        const unsigned long long X0 = s_x0;
        int32_t xr = (int32_t)(incl - dx[0] - dx[1]);
#pragma unroll
        for (uint32_t k = 0; k < 2; ++k) {
            const uint32_t i = 2u * threadIdx.x + 1u + k;
            xr += (int32_t)dx[k];
            if (i <= K.n) {
                const unsigned long long X = X0 + (long long)xr;
                const uint32_t r = blk * kCovRB + i - 1u;
                const uint32_t iv = S.q_iv[r], p = pst[k];
                const uint32_t lim = 2u * kCovV - p;  // positions from here on leave the two windows (lost, R9)
                uint32_t code;
                if (iv & kCovComplex) code = p | kCovComplex;
                else {
                    const uint32_t c0 = iv & 2047u, len = (iv >> 11) & 2047u;
                    code = min(c0, lim) | (min(c0 + len, lim) << 11);
                }
                S.base[r] = X;
                S.ab[r] = code;
                // window starts never decrease (and advance by at most 2000 per record): the record is the first one at or
                // beyond every tile boundary it crosses
                const unsigned long long V = X0 + (long long)vrel[i], Vp = X0 + (long long)vrel[i - 1];
                const uint32_t t1 = (uint32_t)((V - xc) / kCovTile);
                for (uint32_t tt = r ? (uint32_t)((Vp - xc) / kCovTile) + 1u : 0u; tt <= t1; ++tt) S.first_rec[tt] = r;
                if (r == nq - 1u) {
                    carry->xl = V;
                    carry->ntiles = (uint32_t)((V - xc + kCovTile - 1u) / kCovTile);
                    carry->vt_last = t1;
                    carry->n_rid = K.srid[i];
                    carry->n_b = K.sb[i];
                    carry->n_p = p;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// depth histogram of one tile of <= 1024 positions by one warp (update_coverage, src/OverallNumbers.hpp:66-77:
// poscov[min(depth, 100)]++ per position).  The events of the tile sit in a difference array in shared memory and a
// bitmap (one word per lane) marks the positions that hold one, so the pass touches the bitmap and the events, not
// the positions: lane l owns positions [32 l, 32 l + 32); depth at its first position = d0 + warp prefix sum of the
// events before it; between events the depth is constant and a whole run goes into the histogram with one add
// (lanes without events are aggregated per depth).  The events are cleared on the way, so the difference array is
// all zero again afterwards.  No block-wide barrier: the 8 warps of a CTA work on different tiles.  Returns the depth
// after the last position.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int32_t cov_warp_tile(int32_t* diff, const uint32_t* bm, uint32_t len, int32_t d0, uint32_t* hist) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t m0 = bm[lane];
    int32_t* my = diff + 32u * lane;
    int32_t sum = 0;
    for (uint32_t m = m0; m; m &= m - 1u) sum += my[__ffs((int)m) - 1];
    int32_t incl = sum;
    for (int o = 1; o < 32; o <<= 1) {
        const int32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    int32_t d = d0 + incl - sum;   // depth before this lane's first position
    const uint32_t first = 32u * lane;
    const uint32_t nvalid = first >= len ? 0u : min(32u, len - first);
    // lanes whose 32 positions hold no event and lie inside the range: one add per depth
    const bool plain = m0 == 0u && nvalid == 32u;
    const uint32_t key = plain ? min((uint32_t)d, 100u) : (0x100u | lane);
    const uint32_t grp = __match_any_sync(0xFFFFFFFFu, key);
    if (plain) {
        if ((uint32_t)(__ffs((int)grp) - 1) == lane) atomicAdd(hist + key, 32u * (uint32_t)__popc(grp));
    } else if (nvalid) {
        uint32_t pos = 0;
        for (uint32_t m = m0; m; m &= m - 1u) {
            const uint32_t b = (uint32_t)__ffs((int)m) - 1u;
            if (b > pos) atomicAdd(hist + min((uint32_t)d, 100u), b - pos);
            d += my[b];
            my[b] = 0;
            pos = b;
        }
        if (nvalid > pos) atomicAdd(hist + min((uint32_t)d, 100u), nvalid - pos);
    }
    __syncwarp();
    return d0 + __shfl_sync(0xFFFFFFFFu, incl, 31);
}

// adds the covered interval(s) of compact record j, clipped to [T0, T1), to a difference array over [T0, T1] and marks
// the positions in the bitmap (bm may be NULL)
__device__ __forceinline__ void cov_tile_add(const CovScratch& S, const BatchView& B, uint32_t j, unsigned long long T0, unsigned long long T1, int32_t* diff, uint32_t* bm) {
    const long long rel = (long long)(S.base[j] - T0);        // begin of the record relative to the range (may be negative)
    const int32_t len = (int32_t)(T1 - T0);
    if (rel >= (long long)len || rel < -4096) return;           // an interval reaches at most 2000 positions
    const int32_t r = (int32_t)rel;
    const uint32_t code = S.ab[j];
    auto add = [&](int32_t a, int32_t b) {                     // [a, b) relative to the range
        if (b <= 0 || a >= len || a >= b) return;
        const uint32_t s = (uint32_t)max(a, 0);
        atomicAdd(diff + s, 1);
        if (bm) atomicOr(bm + (s >> 5), 1u << (s & 31u));
        if (b < len) {
            atomicAdd(diff + b, -1);
            if (bm) atomicOr(bm + ((uint32_t)b >> 5), 1u << ((uint32_t)b & 31u));
        }
    };
    if (!(code & kCovComplex)) {
        add(r + (int32_t)(code & 2047u), r + (int32_t)((code >> 11) & 2047u));
    } else {
        const uint32_t lim = 2u * kCovV - (code & 2047u);
        cov_walk_cigar(B.bytes + B.offsets[S.q_rec[j]], [&](uint32_t s, uint32_t e) { add(r + (int32_t)min(s, lim), r + (int32_t)min(e, lim)); });
    }
}

// One warp per tile of 1024 positions.  A record writes into [V, V + 2000) (V = start of its window v1): the records
// of a tile are those whose V lies in the tile or in the two before it.
__global__ void __launch_bounds__(kCovTileThreads) k_cov_tiles(BatchView B, CovScratch S, const CovCarry* carry, const int32_t* carry_d, unsigned long long* poscov) {
    __shared__ __align__(16) int32_t diff_all[(kCovTileThreads / 32) * kCovTile];
    __shared__ uint32_t bm_all[kCovTileThreads];
    __shared__ uint32_t hist[104];
    const uint32_t ntiles = carry->ntiles, nq = carry->nq;
    if (nq == 0 || blockIdx.x * (kCovTileThreads / 32u) >= ntiles) return;
    const unsigned long long xc = carry->xc, xl = carry->xl;
    const uint32_t vt_last = carry->vt_last;
    const int32_t* D = carry_d + (size_t)carry->parity * kCovD;
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    int32_t* diff = diff_all + w * kCovTile;
    uint32_t* bm = bm_all + w * 32u;
    for (uint32_t i = threadIdx.x; i < 104u; i += blockDim.x) hist[i] = 0;
    for (uint32_t i = lane; i < kCovTile; i += 32u) diff[i] = 0;
    __syncthreads();
    const uint32_t tstep = gridDim.x * (kCovTileThreads / 32u);
    uint32_t t = blockIdx.x * (kCovTileThreads / 32u) + w;
    uint32_t jlo = 0, jhi = 0;
    if (t < ntiles) { jlo = t >= 2u ? S.first_rec[t - 2u] : 0u; jhi = t + 1u <= vt_last ? S.first_rec[t + 1u] : nq; }
    for (; t < ntiles; t += tstep) {
        const unsigned long long T0 = xc + (unsigned long long)t * kCovTile;
        const unsigned long long T1 = min(T0 + kCovTile, xl);
        const uint32_t len = (uint32_t)(T1 - T0);
        bm[lane] = 0;
        // the record range of this warp's next tile is fetched while this one is worked on
        const uint32_t tn = t + tstep;
        uint32_t njlo = 0, njhi = 0;
        if (tn < ntiles) { njlo = S.first_rec[tn - 2u]; njhi = tn + 1u <= vt_last ? S.first_rec[tn + 1u] : nq; }
        __syncwarp();
        for (uint32_t j = jlo + lane; j < jhi; j += 32u) cov_tile_add(S, B, j, T0, T1, diff, bm);
        int32_t d0 = 0;
        if (t < 2u) {  // the two windows that were open when the batch started: positions xc .. xc + 2000
            const uint32_t o = t * kCovTile;
            for (uint32_t i = lane; i < len && o + i <= 2u * kCovV; i += 32u) {
                const int32_t v = D[o + i];
                if (v) { atomicAdd(diff + i, v); atomicOr(bm + (i >> 5), 1u << (i & 31u)); }
            }
            if (t == 1u) {  // depth they carry into tile 1
                for (uint32_t i = lane; i < kCovTile; i += 32u) d0 += D[i];
                for (int o2 = 16; o2 > 0; o2 >>= 1) d0 += __shfl_xor_sync(0xFFFFFFFFu, d0, o2);
            }
        }
        __syncwarp();
        cov_warp_tile(diff, bm, len, d0, hist);
        jlo = njlo; jhi = njhi;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < 101u; i += blockDim.x)
        if (hist[i]) atomicAdd(poscov + i, (unsigned long long)hist[i]);
}

// The two windows still open after the batch's last record become the next carry: a difference array over
// [xl, xl + 2000], entry 0 holding the depth at xl.  Then the batch's end state becomes the carried state.
__global__ void __launch_bounds__(1024) k_cov_carry(BatchView B, CovScratch S, CovCarry* carry, int32_t* carry_d) {
    __shared__ int32_t dn[kCovD];
    const uint32_t nq = carry->nq;
    if (nq == 0) return;  // nothing took part: state and carry stay
    const unsigned long long xc = carry->xc, xl = carry->xl;
    const int32_t* D = carry_d + (size_t)carry->parity * kCovD;
    int32_t* Dn = carry_d + (size_t)(carry->parity ^ 1u) * kCovD;
    for (uint32_t i = threadIdx.x; i < kCovD; i += blockDim.x) dn[i] = 0;
    __syncthreads();
    const uint32_t vt_last = carry->vt_last;
    const uint32_t jlo = vt_last >= 2u ? S.first_rec[vt_last - 2u] : 0u;   // window start > xl - 2000
    for (uint32_t j = jlo + threadIdx.x; j < nq; j += blockDim.x) cov_tile_add(S, B, j, xl, xl + kCovD, dn, nullptr);
    for (uint32_t d = threadIdx.x; d <= 2u * kCovV; d += blockDim.x) {
        const int32_t v = D[d];
        if (v) {
            const unsigned long long x = xc + d;
            if (x <= xl) atomicAdd(dn, v);
            else atomicAdd(dn + (uint32_t)(x - xl), v);   // x - xl <= 2000
        }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kCovD; i += blockDim.x) Dn[i] = dn[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        carry->first = 0;
        carry->rid_prev = carry->n_rid;
        carry->b_prev = carry->n_b;
        carry->p_prev = carry->n_p;
        carry->xc = xl;
        carry->parity ^= 1u;
        carry->nq = 0;
        carry->ntiles = 0;
    }
}

// End of the run (src/bamqualcheck.cpp:447-453): update_coverage(); update_vectors(); update_coverage() -- the two
// open windows, 2000 positions (all of depth 0 if no record ever took part).
__global__ void __launch_bounds__(32) k_cov_final(const CovCarry* carry, const int32_t* carry_d, unsigned long long* poscov) {
    __shared__ __align__(16) int32_t diff[kCovTile];
    __shared__ uint32_t bm[32];
    __shared__ uint32_t hist[104];
    const int32_t* D = carry_d + (size_t)carry->parity * kCovD;
    const uint32_t lane = threadIdx.x;
    for (uint32_t i = lane; i < 104u; i += 32u) hist[i] = 0;
    for (uint32_t i = lane; i < kCovTile; i += 32u) diff[i] = 0;
    int32_t depth = 0;
    for (uint32_t o = 0; o < 2u * kCovV; o += kCovTile) {
        const uint32_t len = min(kCovTile, 2u * kCovV - o);
        bm[lane] = 0;
        __syncwarp();
        for (uint32_t i = lane; i < len; i += 32u) {
            const int32_t v = D[o + i];
            if (v) { diff[i] = v; atomicOr(bm + (i >> 5), 1u << (i & 31u)); }
        }
        __syncwarp();
        depth = cov_warp_tile(diff, bm, len, depth, hist);
    }
    __syncwarp();
    for (uint32_t i = lane; i < 101u; i += 32u)
        if (hist[i]) atomicAdd(poscov + i, (unsigned long long)hist[i]);
}

// ------------------------------------------------------------------------------------------------
// Shards (cov_math.h): the whole shard's anchor recurrence as a function of the state at its entry -- the block
// descriptors of k_cov_tables applied one after the other for all 1002 states at once -- and the shard's own depth
// over the two windows that were open at its entry.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_cov_shard_function(CovScratch S, const CovCarry* carry, uint16_t* out) {
    __shared__ uint4 sd[1024];
    const uint32_t nq = carry->nq;
    const uint32_t nblk = (nq + kCovRB - 1u) / kCovRB;
    uint32_t p = cov_state_value(min(threadIdx.x, kCovStates - 1u));
    for (uint32_t b0 = 0; b0 < nblk; b0 += 1024u) {
        const uint32_t m = min(1024u, nblk - b0);
        __syncthreads();
        if (threadIdx.x < m) sd[threadIdx.x] = S.desc[b0 + threadIdx.x];
        __syncthreads();
        for (uint32_t k = 0; k < m; ++k) {
            const uint4 d = sd[k];
            if (d.x == COV_CLOSED) p = cov_stretch(p, d.y, d.z);
            else if (d.x == COV_CONST) p = d.y;
            else p = cov_state_value(S.tables[(size_t)(b0 + k) * 1024u + cov_state_index(p)]);
        }
    }
    if (threadIdx.x < kCovStates) out[threadIdx.x] = (uint16_t)cov_state_index(p);
}

// own depth (difference array) over [xc, xc + 2000]: the records whose window start lies in tiles 0 and 1
__global__ void __launch_bounds__(1024) k_cov_head(BatchView B, CovScratch S, const CovCarry* carry, int32_t* head) {
    __shared__ int32_t dn[kCovD];
    const uint32_t nq = carry->nq;
    for (uint32_t i = threadIdx.x; i < kCovD; i += blockDim.x) dn[i] = 0;
    __syncthreads();
    if (nq) {
        const unsigned long long xc = carry->xc;
        const uint32_t jhi = 2u <= carry->vt_last ? S.first_rec[2] : nq;
        for (uint32_t j = threadIdx.x; j < jhi; j += blockDim.x) cov_tile_add(S, B, j, xc, xc + 2u * kCovV + 1u, dn, nullptr);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kCovD; i += blockDim.x) head[i] = dn[i];
}

// Several read groups: the collected records in the order of `index` (k_lane_partition over S.q_lane: lane by lane,
// file order inside a lane), so that every lane's records are one contiguous segment of (rid, b, iv).
__global__ void k_cov_lane_gather(CovScratch S, const uint32_t* __restrict__ index, uint32_t n, int32_t* rid, uint32_t* b, uint32_t* iv) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t j = index[i];
        rid[i] = S.q_rid[j];
        b[i] = S.q_b[j];
        iv[i] = S.q_iv[j];
    }
}

__global__ void k_cov_set_state(CovCarry* carry, uint32_t first, int32_t rid_prev, uint32_t b_prev, uint32_t p_prev) {
    carry->first = first;
    carry->rid_prev = rid_prev;
    carry->b_prev = b_prev;
    carry->p_prev = p_prev;
    carry->xc = 0;
}

__global__ void k_poscov_adjust(unsigned long long* poscov, const long long* delta) {
    if (threadIdx.x <= 100u) poscov[threadIdx.x] += (unsigned long long)delta[threadIdx.x];
}

}  // namespace bqc
