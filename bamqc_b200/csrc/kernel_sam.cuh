// kernel_sam.cuh -- SAM text -> BAM records on the device (bqc_submit_sam, bqc_sam_to_bam).
//
// One submission holds whole lines.  The kernels, in order, on the framing stream:
//   k_sam_nl_count / k_sam_scan_top / k_sam_nl_emit   the line ends (newline positions, in order) by a block-sum scan
//   k_sam_size                                        one thread per line: the fast grammar (sam_parse.h) without
//                                                     writing; record size, or the line is counted as not fast
//   k_sam_scan_tiles / k_sam_scan_top / k_sam_scan_apply  exclusive scan of (record count << 36 | bytes) per line
//   k_sam_encode                                      one thread per line writes its record and offset, and fills the
//                                                     FrameResult stage B reads back
// A submission with any line that is not fast, more lines than the slot holds or more record bytes than it holds
// encodes nothing here: FrameResult::bad is set and the host encodes the whole submission (engine.cu).
#pragma once
#include <stdint.h>

#include "kernel_frame.cuh"
#include "sam_parse.h"

namespace bqc {

static const uint32_t kSamNlThreads = 256, kSamNlPer = 64;        // newline scan: 64 bytes per thread, 16 KB per CTA
static const uint32_t kSamScanThreads = 1024, kSamScanPer = 4;    // size scan: 4096 lines per CTA
static const uint32_t kSamLineThreads = 256;
static const int kSamBytesShift = 36;                             // packed per-line value: records << 36 | bytes

struct SamCtl {
    unsigned long long lines;    // newlines in the submission
    unsigned long long packed;   // sum of the packed per-line values
    uint32_t slow;               // lines outside the fast grammar
    uint32_t max_lseq;
};

// inclusive block scan of one 64-bit value per thread (blockDim.x a multiple of 32, at most 1024)
__device__ __forceinline__ unsigned long long sam_block_scan(unsigned long long v, unsigned long long* ws, unsigned long long& total) {
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    unsigned long long incl = v;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    __syncthreads();
    if (lane == 31u) ws[w] = incl;
    __syncthreads();
    if (w == 0) {
        const uint32_t nw = blockDim.x >> 5;
        const unsigned long long x = lane < nw ? ws[lane] : 0ull;
        unsigned long long xi = x;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, xi, o);
            if (lane >= (uint32_t)o) xi += t;
        }
        ws[lane] = xi - x;
        if (lane == 31u) ws[32] = xi;
    }
    __syncthreads();
    total = ws[32];
    return incl + ws[w];
}

// newlines in this thread's 64 bytes (16-byte loads; the text buffer has >= 256 bytes of slack behind n)
__device__ __forceinline__ uint32_t sam_nl_mask_count(const uint8_t* __restrict__ text, uint64_t at, uint32_t n, uint64_t* bits) {
    uint32_t c = 0;
    bits[0] = 0;
    if (at >= n) return 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint4 v = *reinterpret_cast<const uint4*>(text + at + 16 * k);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t m = __vcmpeq4(w[j], 0x0A0A0A0Au);   // 0xFF in every byte that is '\n'
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const uint32_t pos = 16 * k + 4 * j + b;
                if (((m >> (8 * b)) & 1u) && at + pos < n) { bits[0] |= 1ull << pos; ++c; }
            }
        }
    }
    return c;
}

__global__ void __launch_bounds__(kSamNlThreads) k_sam_nl_count(const uint8_t* __restrict__ text, uint32_t n, unsigned long long* __restrict__ bsum) {
    __shared__ unsigned long long ws[33];
    uint64_t bits;
    const uint32_t c = sam_nl_mask_count(text, ((uint64_t)blockIdx.x * kSamNlThreads + threadIdx.x) * kSamNlPer, n, &bits);
    unsigned long long total;
    sam_block_scan(c, ws, total);
    if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// one CTA: exclusive scan of v[0..nb) in place, the sum into *total.  n_items (device) overrides nb as
// ceil(min(*n_items, cap) / per) when given.
__global__ void __launch_bounds__(1024) k_sam_scan_top(unsigned long long* v, uint32_t nb, const unsigned long long* __restrict__ n_items, uint32_t per,
                                                       uint64_t cap, unsigned long long* total) {
    __shared__ unsigned long long ws[33];
    if (n_items) nb = (uint32_t)((min(*n_items, (unsigned long long)cap) + per - 1) / per);
    unsigned long long carry = 0;
    for (uint32_t base = 0; base < nb; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long x = i < nb ? v[i] : 0ull;
        unsigned long long t;
        const unsigned long long incl = sam_block_scan(x, ws, t);
        if (i < nb) v[i] = carry + incl - x;
        carry += t;
    }
    if (threadIdx.x == 0) *total = carry;
}

// the line ends: position of every newline, in order (at most cap of them are written)
__global__ void __launch_bounds__(kSamNlThreads) k_sam_nl_emit(const uint8_t* __restrict__ text, uint32_t n, const unsigned long long* __restrict__ bsum,
                                                               uint32_t* __restrict__ lend, uint64_t cap) {
    __shared__ unsigned long long ws[33];
    uint64_t bits;
    const uint64_t at = ((uint64_t)blockIdx.x * kSamNlThreads + threadIdx.x) * kSamNlPer;
    const uint32_t c = sam_nl_mask_count(text, at, n, &bits);
    unsigned long long total;
    uint64_t idx = bsum[blockIdx.x] + sam_block_scan(c, ws, total) - c;
    while (bits) {
        const int b = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        if (idx < cap) lend[idx] = (uint32_t)(at + b);
        ++idx;
    }
}

__device__ __forceinline__ void sam_line(const uint8_t* text, const uint32_t* lend, uint64_t i, uint32_t& b, uint32_t& e) {
    b = i ? lend[i - 1] + 1u : 0u;
    e = lend[i];
}

__global__ void __launch_bounds__(kSamLineThreads) k_sam_size(const uint8_t* __restrict__ text, const uint32_t* __restrict__ lend, SamCtl* ctl, uint64_t cap,
                                                              SamRefs R, unsigned long long* __restrict__ sz) {
    const unsigned long long lines = ctl->lines;
    if (lines > cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctl->slow, 1u);
        return;
    }
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < lines; i0 += stride) {
        const uint64_t i = i0 + threadIdx.x;
        uint32_t ls = 0, slow = 0;
        if (i < lines) {
            uint32_t b, e;
            sam_line(text, lend, i, b, e);
            const int64_t r = sam_fast_line(text + b, e - b, R, nullptr, ls);
            if (r < 0) { slow = 1; ls = 0; }
            sz[i] = r > 0 ? (1ull << kSamBytesShift) | (unsigned long long)r : 0ull;
        }
        const uint32_t mx = __reduce_max_sync(0xFFFFFFFFu, ls), ns = __reduce_add_sync(0xFFFFFFFFu, slow);
        if ((threadIdx.x & 31u) == 0) {
            if (mx) atomicMax(&ctl->max_lseq, mx);
            if (ns) atomicAdd(&ctl->slow, ns);
        }
    }
}

// per tile of kSamScanThreads * kSamScanPer values: their sum
__global__ void __launch_bounds__(kSamScanThreads) k_sam_scan_tiles(const unsigned long long* __restrict__ v, const unsigned long long* __restrict__ n_items,
                                                                    uint64_t cap, unsigned long long* __restrict__ tsum) {
    __shared__ unsigned long long ws[33];
    const unsigned long long n = min(*n_items, (unsigned long long)cap);
    const uint64_t base = (uint64_t)blockIdx.x * kSamScanThreads * kSamScanPer;
    if (base >= n) return;
    unsigned long long s = 0;
#pragma unroll
    for (uint32_t k = 0; k < kSamScanPer; ++k) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kSamScanPer + k;
        if (i < n) s += v[i];
    }
    unsigned long long total;
    sam_block_scan(s, ws, total);
    if (threadIdx.x == 0) tsum[blockIdx.x] = total;
}

// exclusive scan in place, tile offsets from k_sam_scan_top
__global__ void __launch_bounds__(kSamScanThreads) k_sam_scan_apply(unsigned long long* __restrict__ v, const unsigned long long* __restrict__ n_items,
                                                                    uint64_t cap, const unsigned long long* __restrict__ tsum) {
    __shared__ unsigned long long ws[33];
    const unsigned long long n = min(*n_items, (unsigned long long)cap);
    const uint64_t base = (uint64_t)blockIdx.x * kSamScanThreads * kSamScanPer;
    if (base >= n) return;
    unsigned long long x[kSamScanPer], s = 0;
#pragma unroll
    for (uint32_t k = 0; k < kSamScanPer; ++k) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kSamScanPer + k;
        x[k] = i < n ? v[i] : 0ull;
        s += x[k];
    }
    unsigned long long total;
    unsigned long long run = tsum[blockIdx.x] + sam_block_scan(s, ws, total) - s;
#pragma unroll
    for (uint32_t k = 0; k < kSamScanPer; ++k) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kSamScanPer + k;
        if (i < n) v[i] = run;
        run += x[k];
    }
}

// write the records (sz holds the exclusive prefix of the packed values) and the frame header
__global__ void __launch_bounds__(kSamLineThreads) k_sam_encode(const uint8_t* __restrict__ text, const uint32_t* __restrict__ lend, const SamCtl* __restrict__ ctl,
                                                                uint64_t line_cap, uint64_t rec_cap, uint64_t byte_cap, SamRefs R,
                                                                const unsigned long long* __restrict__ sz, uint8_t* __restrict__ out, uint32_t* __restrict__ offsets,
                                                                FrameResult* fr) {
    const unsigned long long lines = ctl->lines, packed = ctl->packed;
    const unsigned long long mask = (1ull << kSamBytesShift) - 1ull;
    const uint64_t n_rec = packed >> kSamBytesShift, n_bytes = packed & mask;
    const bool ok = lines <= line_cap && ctl->slow == 0 && n_rec <= rec_cap && n_bytes <= byte_cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        fr->n_records = ok ? (uint32_t)n_rec : 0u;
        fr->max_lseq = ctl->max_lseq;
        fr->bad = ok ? 0u : 1u;
        fr->start = 0;
        fr->end = ok ? (uint32_t)n_bytes : 0u;
        fr->total = fr->end;
        fr->tail_overflow = 0;
        fr->repaired = 0;
        fr->inflate_bad = 0;
        if (ok) offsets[n_rec] = (uint32_t)n_bytes;
    }
    if (!ok) return;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < lines; i += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned long long cur = sz[i], next = i + 1 < lines ? sz[i + 1] : packed;
        if (((next - cur) & mask) == 0) continue;   // empty line
        const uint32_t off = (uint32_t)(cur & mask);
        offsets[cur >> kSamBytesShift] = off;
        uint32_t b, e, ls;
        sam_line(text, lend, i, b, e);
        sam_fast_line(text + b, e - b, R, out + off, ls);
    }
}

}  // namespace bqc
