// sketch_sched.h -- where k_sketch32v2 has to hash: word-parallel validity and emit masks of one 8-base sub-chunk,
// and the split of a read's emitting sub-chunks into pieces that a warp spreads over its lanes.
// Host/device: the same functions are exercised on the CPU by tests/test_sketch_sched_cpu.py (via
// sketch_sched_selftest.cpp) against a per-base restatement of the rolling hash.
//
// A window of k = 32 bases is emitted iff all 32 bases are valid (quality q with (q - q_lo) <= q_span unsigned, base
// != N, inside the read).  Its hash depends on those 32 bases only, so hashing may restart from zero state anywhere:
// restarted at sub-chunk a with the all-zero `out` table for the first 32 updates, the hash is exact for every window
// ending at or after base 8a + 31, and the 32-bit validity history is rebuilt over the same 32 bases.  A piece
// therefore hashes from kPieceWarm sub-chunks before its first emitting sub-chunk (clipped at 0, where the walk
// starts exactly as at the start of a read) and emits only from its own emitting sub-chunks on.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define BQC_SK __host__ __device__ __forceinline__
#else
#define BQC_SK inline
#endif

namespace bqc {

static const uint32_t kPieceEmit = 4;    // emitting sub-chunks per piece at most
static const uint32_t kPieceWarm = 4;    // warm-up sub-chunks in front of a piece: 32 bases = one window
static_assert(kPieceEmit >= 2, "pass 1 appends at most one piece per two sub-chunks");

// bit j set iff quality byte j of q8 satisfies (q - q_lo) <= q_span as unsigned 8-bit values; q_lo, q_span in 0..127
BQC_SK uint32_t sketch_qual_ok8(uint64_t q8, uint32_t q_lo, uint32_t q_span) {
    const uint64_t H = 0x8080808080808080ULL, ones = 0x0101010101010101ULL;
    const uint64_t y = ones * q_lo;
    const uint64_t d = ((q8 | H) - y) ^ (~q8 & H);                                  // per-byte q - q_lo mod 256 (y < 128)
    const uint64_t ok = ~(d | ((d & ~H) + ones * (127u - q_span))) & H;            // d < 128 and d + 127 - span < 128
    uint64_t x = ok >> 7;                                                           // bit 8j
    x = (x | (x >> 7)) & 0x0003000300030003ULL;
    x = (x | (x >> 14)) & 0x0000000F0000000FULL;
    return (uint32_t)((x | (x >> 28)) & 0xFFu);
}

// bit j set iff base j of the 8 SEQ nibbles (BAM order: base 2i in the high nibble of byte i) is not N (15)
BQC_SK uint32_t sketch_not_n8(uint32_t s) {
    const uint32_t w = ((s & 0x0F0F0F0Fu) << 4) | ((s >> 4) & 0x0F0F0F0Fu);       // base j in nibble j
    uint32_t x = ~(w & (w >> 1) & (w >> 2) & (w >> 3)) & 0x11111111u;             // bit 4j
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    return (x | (x >> 12)) & 0xFFu;
}

// validity of the 8 bases of sub-chunk c of a read of Ls bases
BQC_SK uint32_t sketch_valid8(uint64_t q8, uint32_t s, uint32_t c, uint32_t Ls, uint32_t q_lo, uint32_t q_span) {
    const uint32_t left = Ls > 8u * c ? Ls - 8u * c : 0u;
    const uint32_t in_read = left >= 8u ? 0xFFu : (1u << left) - 1u;
    return sketch_qual_ok8(q8, q_lo, q_span) & sketch_not_n8(s) & in_read;
}

// hv: validity of the 32 bases before the sub-chunk, oldest in bit 0.  Returns the 8 emit bits (bit j: the window
// ending at base j of the sub-chunk has 32 valid bases) and advances hv by the sub-chunk.
BQC_SK uint32_t sketch_emit8(uint32_t& hv, uint32_t valid8) {
    const uint64_t x = (uint64_t)hv | ((uint64_t)valid8 << 32);
    uint64_t y = x & (x >> 1);
    y &= y >> 2;
    y &= y >> 4;
    y &= y >> 8;
    y &= y >> 16;                                                                   // bit i: bits i..i+31 of x all set
    hv = (uint32_t)(x >> 8);
    return (uint32_t)(y >> 1) & 0xFFu;
}

// the same for 16 bases (two sub-chunks c, c + 1; SEQ word s16 = 16 nibbles, QUAL words q0, q1): pass 1 walks whole
// reads, and one emit chain per 16 bases halves its cost over the 8-base forms that pass 2 uses per sub-chunk
BQC_SK uint32_t sketch_not_n16(uint64_t s) {
    const uint64_t w = ((s & 0x0F0F0F0F0F0F0F0FULL) << 4) | ((s >> 4) & 0x0F0F0F0F0F0F0F0FULL);
    uint64_t x = ~(w & (w >> 1) & (w >> 2) & (w >> 3)) & 0x1111111111111111ULL;
    x = (x | (x >> 3)) & 0x0303030303030303ULL;
    x = (x | (x >> 6)) & 0x000F000F000F000FULL;
    x = (x | (x >> 12)) & 0x000000FF000000FFULL;
    return (uint32_t)((x | (x >> 24)) & 0xFFFFu);
}
BQC_SK uint32_t sketch_valid16(uint64_t q0, uint64_t q1, uint64_t s, uint32_t c, uint32_t Ls, uint32_t q_lo, uint32_t q_span) {
    const uint32_t left = Ls > 8u * c ? Ls - 8u * c : 0u;
    const uint32_t in_read = left >= 16u ? 0xFFFFu : (1u << left) - 1u;
    return (sketch_qual_ok8(q0, q_lo, q_span) | (sketch_qual_ok8(q1, q_lo, q_span) << 8)) & sketch_not_n16(s) & in_read;
}
BQC_SK uint32_t sketch_emit16(uint32_t& hv, uint32_t valid16) {
    const uint64_t x = (uint64_t)hv | ((uint64_t)valid16 << 32);
    uint64_t y = x & (x >> 1);
    y &= y >> 2;
    y &= y >> 4;
    y &= y >> 8;
    y &= y >> 16;
    hv = (uint32_t)(x >> 16);
    return (uint32_t)(y >> 1) & 0xFFFFu;
}

// piece descriptor: owning lane (bits 0..4), first emitting sub-chunk (8..15), end sub-chunk, exclusive (16..23).
// The 8-bit fields hold reads of up to kPieceMaxSub sub-chunks (2040 bases, the engine takes 1800); a warp with a
// longer read does not split.
static const uint32_t kPieceMaxSub = 255;
BQC_SK uint32_t piece_desc(uint32_t lane, uint32_t es, uint32_t end) { return lane | (es << 8) | (end << 16); }
BQC_SK uint32_t piece_warm_start(uint32_t es) { return es > kPieceWarm ? es - kPieceWarm : 0u; }

// Splits the emitting sub-chunks of one read, fed in order, into pieces of at most kPieceEmit emitting sub-chunks.
// With kPieceEmit >= 2 at most one piece closes in two consecutive sub-chunks (pass 1 appends once per 16 bases).
struct PieceSplitter {
    uint32_t es, n;   // open piece: first emitting sub-chunk, emitting sub-chunks so far (n == 0: none open)
    // feed sub-chunk c; returns true when a piece [es, end) closes
    BQC_SK bool step(uint32_t c, bool emitting, uint32_t& p_es, uint32_t& p_end) {
        if (!emitting) {
            if (!n) return false;
            p_es = es; p_end = c; n = 0;
            return true;
        }
        if (!n) es = c;
        if (++n < kPieceEmit) return false;
        p_es = es; p_end = c + 1u; n = 0;
        return true;
    }
    // after the last sub-chunk nsub - 1
    BQC_SK bool flush(uint32_t nsub, uint32_t& p_es, uint32_t& p_end) {
        if (!n) return false;
        p_es = es; p_end = nsub; n = 0;
        return true;
    }
};

}  // namespace bqc
