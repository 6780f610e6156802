// sketch_sched_selftest.cpp -- CPU check of bamqc_b200/csrc/sketch_sched.h (test infrastructure; built and run by
// tests/test_sketch_sched_cpu.py).
//   (1) sketch_qual_ok8 / sketch_not_n8 against the per-base tests for every quality byte, threshold and nibble;
//   (2) random reads (lengths 31..1800, both strands, qualities 0..255, N anywhere, valid runs of exactly 31/32/33
//       bases at every alignment to the sub-chunks) hashed two ways with a k = 32 rolling hash of the same form as
//       RepHash (h = rotl1(h) ^ H[in] ^ rotl32(H[out])):
//         a. per base from the start of the read, a window emitted when its 32 bases are valid;
//         b. as k_sketch32v2 does it: pass 1 word-parallel over the read, 16 bases per step -> emitting sub-chunks -> pieces, then every
//            piece restarted from zero state at piece_warm_start with the zero `out` table for 4 sub-chunks and the
//            emits masked to the piece's emitting sub-chunks; and the unsplit walk (one piece per read, no warm-up).
//       The multisets of emitted hashes must be equal, and equal to the hash of each window computed directly.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>

#include "../bamqc_b200/csrc/sketch_sched.h"

using namespace bqc;

static uint64_t rng_state = 0x2545F4914F6CDD1DULL;
static uint64_t rnd() {
    uint64_t z = (rng_state += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
static uint64_t rotl(uint64_t x, uint32_t r) { r &= 63u; return r ? (x << r) | (x >> (64u - r)) : x; }

static uint64_t H[2][16];
static uint64_t mismatches = 0;

struct Read {
    std::vector<uint8_t> seq, qual;   // packed SEQ (high nibble first) and QUAL, padded
    uint32_t L, strand;
};
static uint32_t nib(const Read& r, uint32_t i) { return (r.seq[i >> 1] >> ((i & 1) ? 0 : 4)) & 15u; }
static bool valid_base(const Read& r, uint32_t i, uint32_t q_lo, uint32_t q_span) {
    return i < r.L && (uint32_t)(r.qual[i] - q_lo) <= q_span && nib(r, i) != 15u;
}
static uint64_t ld64(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }
static uint32_t ld32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }

// a: per base from the start of the read
static void per_base(const Read& r, uint32_t q_lo, uint32_t q_span, std::vector<uint64_t>& out) {
    uint64_t h = 0;
    uint32_t run = 0;
    for (uint32_t i = 0; i < r.L; ++i) {
        h = rotl(h, 1) ^ H[r.strand][nib(r, i)] ^ (i >= 32 ? rotl(H[r.strand][nib(r, i - 32)], 32) : 0);
        run = valid_base(r, i, q_lo, q_span) ? run + 1 : 0;
        if (run >= 32) {
            out.push_back(h);
            uint64_t d = 0;   // the window's hash computed directly
            for (uint32_t j = 0; j < 32; ++j) d ^= rotl(H[r.strand][nib(r, i - j)], j);
            if (d != h) ++mismatches;
        }
    }
}

// b: one piece: hash sub-chunks ws..end-1 from zero state, emit only in es..end-1
static void hash_piece(const Read& r, uint32_t ws, uint32_t es, uint32_t end, uint32_t q_lo, uint32_t q_span, std::vector<uint64_t>& out) {
    uint64_t h = 0;
    uint32_t hv = 0;
    for (uint32_t c = ws; c < end; ++c) {
        const uint32_t s = ld32(&r.seq[4 * c]);
        const uint32_t emit = sketch_emit8(hv, sketch_valid8(ld64(&r.qual[8 * c]), s, c, r.L, q_lo, q_span));
        const uint32_t so = c >= ws + kPieceWarm ? ld32(&r.seq[4 * (c - 4)]) : 0u;
        for (uint32_t j = 0; j < 8; ++j) {
            const uint32_t ni = (s >> (4 * (j ^ 1))) & 15u, no = (so >> (4 * (j ^ 1))) & 15u;
            h = rotl(h, 1) ^ H[r.strand][ni] ^ (c >= ws + kPieceWarm ? rotl(H[r.strand][no], 32) : 0);
            if (c >= es && ((emit >> j) & 1u)) out.push_back(h);
        }
    }
}

static void scheduled(const Read& r, uint32_t q_lo, uint32_t q_span, bool split, std::vector<uint64_t>& out) {
    const uint32_t nsub = (r.L + 7) / 8;
    if (!split) { hash_piece(r, 0, 0, nsub, q_lo, q_span, out); return; }
    uint32_t hv = 0;
    PieceSplitter ps = {0, 0};
    uint32_t es, end, covered = 0;
    std::vector<uint32_t> emitting(nsub, 0);
    auto piece = [&](uint32_t a, uint32_t b) {
        for (uint32_t c = a; c < b; ++c) {
            if (!emitting[c]) ++mismatches;        // a piece holds emitting sub-chunks only ...
        }
        if (b - a > kPieceEmit || a < covered) ++mismatches;
        covered = b;
        hash_piece(r, piece_warm_start(a), a, b, q_lo, q_span, out);
    };
    emitting.push_back(0);
    for (uint32_t c = 0; c < nsub; c += 2) {   // 16 bases per step, one piece closes at most, as in the kernel
        const uint32_t e = sketch_emit16(hv, sketch_valid16(ld64(&r.qual[8 * c]), ld64(&r.qual[8 * c + 8]), ld64(&r.seq[4 * c]), c, r.L, q_lo, q_span));
        emitting[c] = (e & 0xFF) != 0;
        emitting[c + 1] = (e >> 8) != 0;
        if (c + 1 >= nsub && emitting[c + 1]) ++mismatches;   // past the read
        uint32_t e0 = 0, e1 = 0;
        bool close = ps.step(c, emitting[c] != 0, e0, e1);
        uint32_t f0 = 0, f1 = 0;
        const bool close2 = ps.step(c + 1, emitting[c + 1] != 0, f0, f1);
        if (close && close2) ++mismatches;
        if (close) piece(e0, e1);
        if (close2) piece(f0, f1);
    }
    if (ps.flush(nsub, es, end)) piece(es, end);
}

static void check_masks() {
    for (uint32_t q_lo = 0; q_lo <= 94; ++q_lo) {
        const uint32_t q_span = 94 - q_lo;
        for (uint32_t q = 0; q < 256; ++q) {
            for (uint32_t pos = 0; pos < 8; ++pos) {
                const uint64_t w = (rnd() & ~(0xFFULL << (8 * pos))) | ((uint64_t)q << (8 * pos));
                const uint32_t m = sketch_qual_ok8(w, q_lo, q_span);
                for (uint32_t j = 0; j < 8; ++j) {
                    const uint32_t b = (uint32_t)(w >> (8 * j)) & 255u;
                    if ((((m >> j) & 1u) != 0) != ((uint32_t)(b - q_lo) <= q_span)) ++mismatches;
                }
            }
        }
    }
    for (uint32_t t = 0; t < 100000; ++t) {
        uint32_t s = (uint32_t)rnd();
        if (t & 1) s |= (uint32_t)rnd() & (uint32_t)rnd() & 0xF0F0F0F0u, s |= 0x0F0F0F0Fu & (uint32_t)rnd() & (uint32_t)rnd();
        const uint32_t m = sketch_not_n8(s);
        for (uint32_t j = 0; j < 8; ++j) {
            const uint32_t n = (s >> (4 * (j ^ 1))) & 15u;
            if ((((m >> j) & 1u) != 0) != (n != 15u)) ++mismatches;
        }
    }
}

int main(int argc, char** argv) {
    const uint32_t nreads = argc > 1 ? (uint32_t)atoi(argv[1]) : 20000;
    for (auto& t : H) for (auto& v : t) v = rnd();
    check_masks();
    const uint32_t lens[] = {31, 32, 33, 39, 40, 41, 63, 64, 65, 150, 151, 250, 700, 1500, 1800};
    uint64_t windows = 0;
    for (uint32_t n = 0; n < nreads; ++n) {
        Read r;
        r.L = n % 3 ? lens[rnd() % 15] : 31 + (uint32_t)(rnd() % 1770);
        r.strand = (uint32_t)(rnd() & 1);
        const uint32_t pad = 8 * ((r.L + 7) / 8) + 72;
        r.seq.assign(pad, 0);
        r.qual.assign(pad, 0);
        for (uint32_t i = 0; i < pad; ++i) r.qual[i] = (uint8_t)rnd();   // bytes past the read: anything
        for (uint32_t i = 0; i < pad; ++i) r.seq[i] = (uint8_t)rnd();
        const uint32_t q_lo = (uint32_t)(rnd() % 95), q_span = 94 - q_lo;
        const uint32_t mode = (uint32_t)(rnd() % 4);
        for (uint32_t i = 0; i < r.L; ++i) {
            uint32_t q;
            if (mode == 0) q = (uint32_t)(rnd() & 255);                                 // any byte
            else if (mode == 1) q = rnd() % 20 ? q_lo + (uint32_t)(rnd() % (q_span + 1)) : (uint32_t)(rnd() & 255);
            else q = q_lo + (uint32_t)(rnd() % (q_span + 1));                           // valid; runs cut below
            r.qual[i] = (uint8_t)q;
            uint32_t nb = rnd() % 64 ? 1u << (rnd() & 3) : (rnd() % 2 ? 15u : (uint32_t)(rnd() & 15));
            if (mode == 1 && rnd() % 50 == 0) nb = 15u;
            r.seq[i >> 1] = (uint8_t)((i & 1) ? (r.seq[i >> 1] & 0xF0) | nb : (r.seq[i >> 1] & 0x0F) | (nb << 4));
        }
        if (mode >= 2) {   // valid runs of exactly 31, 32 or 33 bases separated by one invalid base (or N), any alignment
            uint32_t i = (uint32_t)(rnd() % 9);
            while (i < r.L) {
                const uint32_t run = 31 + (uint32_t)(rnd() % 3);
                i += run;
                if (i >= r.L) break;
                if (rnd() & 1) r.qual[i] = (uint8_t)(q_lo == 0 ? 95 + rnd() % 161 : (rnd() & 1 ? q_lo - 1 : 95 + rnd() % 161));
                else r.seq[i >> 1] = (uint8_t)((i & 1) ? r.seq[i >> 1] | 0x0F : r.seq[i >> 1] | 0xF0);
                i += 1 + (mode == 3 ? (uint32_t)(rnd() % 8) : 0u);
            }
        }
        std::vector<uint64_t> a, b, c;
        per_base(r, q_lo, q_span, a);
        scheduled(r, q_lo, q_span, true, b);
        scheduled(r, q_lo, q_span, false, c);
        std::sort(a.begin(), a.end());
        std::sort(b.begin(), b.end());
        std::sort(c.begin(), c.end());
        if (a != b || a != c) {
            if (mismatches < 10) fprintf(stderr, "read %u L=%u q_lo=%u mode=%u: %zu per-base, %zu pieces, %zu unsplit\n", n, r.L, q_lo, mode, a.size(), b.size(), c.size());
            ++mismatches;
        }
        windows += a.size();
    }
    printf("%u reads, %llu windows, %llu mismatching\n", nreads, (unsigned long long)windows, (unsigned long long)mismatches);
    return mismatches ? 1 : 0;
}
