// sam_parse.h -- the SAM grammar the device encodes ("fast lines"), host/device.  kernel_sam.cuh runs it one thread per
// line; tests/sam_selftest.cpp runs the same code on the CPU against sam_line_to_bam (sam_text.h).
//
// A line is fast only where the host encoder's atoi/atoll/atof/cast behaviour is reproduced bit for bit:
//   - every byte is printable ASCII (0x20..0x7E) or TAB, at least 11 fields, no mandatory field empty;
//   - QNAME 1..254 bytes (the host's (uint8_t)(length + 1) wraps at 255);
//   - FLAG, MAPQ: 1..9 digits;  POS, PNEXT, TLEN: -?[0-9]{1,18}, then the host's int32/uint16/uint8 casts;
//   - RNAME, RNEXT: '*', '=' or a name looked up in the @SQ names (first of duplicate names wins, unknown -> -1);
//   - CIGAR: '*' or ([0-9]{1,9}[MIDNSHP=X])+ with at most 65535 operations;
//   - SEQ, QUAL: any of those bytes; QUAL '*' or of another length than SEQ gives the 0xFF fill;
//   - tags TAG:T:VALUE of type A, Z, H, i (-?[0-9]{1,18}) and f on the exact decimal fast path: at most 15
//     significant digits and a decimal exponent of at most 22 in magnitude, where one correctly rounded double
//     multiply or divide by an exact power of ten is the correctly rounded value strtod returns.
// Everything else (B arrays, other types, inf/nan/hex floats, '+', spaces, longer numbers) is not fast: the whole
// submission then goes through the host encoder, so the records counted never depend on which path ran.
//
// Size bound: a fast line of L bytes (newline included) encodes to at most 2 L bytes, block_size included.
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define BQC_SP __host__ __device__ __forceinline__
#else
#define BQC_SP inline
#endif

namespace bqc {

static const uint32_t kSamMinLine = 22;   // 10 tabs, a newline and one byte per mandatory field

// @SQ names in bytewise order, the first of duplicate names kept: name k is blob[off[k] .. off[k + 1]), its id id[k]
struct SamRefs {
    const char* blob;
    const uint32_t* off;
    const int32_t* id;
    int32_t n;
};

BQC_SP int32_t sam_ref_lookup(const SamRefs& R, const uint8_t* s, uint32_t len) {
    int32_t lo = 0, hi = R.n;   // std::string ordering: unsigned bytes, a proper prefix first
    while (lo < hi) {
        const int32_t mid = (lo + hi) >> 1;
        const uint32_t a = R.off[mid], m = R.off[mid + 1] - a;
        const uint32_t k = m < len ? m : len;
        int c = 0;
        for (uint32_t i = 0; i < k && !c; ++i) c = (int)(uint8_t)R.blob[a + i] - (int)s[i];
        if (!c) c = m < len ? -1 : (m > len ? 1 : 0);
        if (!c) return R.id[mid];
        if (c < 0) lo = mid + 1; else hi = mid;
    }
    return -1;
}

BQC_SP bool sam_digit(uint8_t c) { return c >= '0' && c <= '9'; }

// [0-9]{1,maxd}
BQC_SP bool sam_uint(const uint8_t* p, uint32_t n, uint32_t maxd, uint64_t& v) {
    if (n == 0 || n > maxd) return false;
    v = 0;
    for (uint32_t i = 0; i < n; ++i) {
        if (!sam_digit(p[i])) return false;
        v = v * 10 + (p[i] - '0');
    }
    return true;
}

// -?[0-9]{1,18}: exactly atoll's value
BQC_SP bool sam_int(const uint8_t* p, uint32_t n, int64_t& v) {
    const bool neg = n && p[0] == '-';
    uint64_t u;
    if (!sam_uint(p + neg, n - neg, 18, u)) return false;
    v = neg ? -(int64_t)u : (int64_t)u;
    return true;
}

// atof's value cast to float, on the exact fast path only
BQC_SP bool sam_float(const uint8_t* p, uint32_t n, float& out) {
    uint32_t i = 0;
    const bool neg = n && p[0] == '-';
    i += neg;
    uint64_t m = 0;
    int32_t sig = 0, nd = 0, frac = 0;
    bool dot = false;
    for (; i < n; ++i) {
        const uint8_t c = p[i];
        if (sam_digit(c)) {
            ++nd;
            if (dot) ++frac;
            if (m == 0 && c == '0') continue;
            if (++sig > 15) return false;
            m = m * 10 + (c - '0');
        } else if (c == '.' && !dot) {
            dot = true;
        } else {
            break;
        }
    }
    if (nd == 0) return false;
    int32_t ex = 0;
    if (i < n) {
        if (p[i] != 'e' && p[i] != 'E') return false;
        ++i;
        const bool eneg = i < n && p[i] == '-';
        if (i < n && (p[i] == '-' || p[i] == '+')) ++i;
        uint64_t u;
        if (!sam_uint(p + i, n - i, 3, u)) return false;
        ex = eneg ? -(int32_t)u : (int32_t)u;
    }
    double d = 0.0;
    if (m) {
        const int32_t e10 = ex - frac;
        if (e10 < -22 || e10 > 22) return false;
        double p10 = 1.0;   // 10^k is exact in double up to k = 22
        for (int32_t k = 0; k < (e10 < 0 ? -e10 : e10); ++k) p10 *= 10.0;
#ifdef __CUDA_ARCH__
        d = e10 >= 0 ? __dmul_rn((double)m, p10) : __ddiv_rn((double)m, p10);
#else
        d = e10 >= 0 ? (double)m * p10 : (double)m / p10;
#endif
    }
    if (neg) d = -d;
#ifdef __CUDA_ARCH__
    out = __double2float_rn(d);
#else
    out = (float)d;
#endif
    return true;
}

// nt16 code of a SEQ byte: strchr("=ACMGRSVTWYHKDBN", toupper(c)), 15 when absent
BQC_SP uint8_t sam_nt16(uint8_t c) {
    switch (c >= 'a' && c <= 'z' ? c - 32 : c) {
        case '=': return 0;  case 'A': return 1;  case 'C': return 2;  case 'M': return 3;
        case 'G': return 4;  case 'R': return 5;  case 'S': return 6;  case 'V': return 7;
        case 'T': return 8;  case 'W': return 9;  case 'Y': return 10; case 'H': return 11;
        case 'K': return 12; case 'D': return 13; case 'B': return 14; default: return 15;
    }
}

BQC_SP int sam_cigar_op(uint8_t c) {
    switch (c) {
        case 'M': return 0; case 'I': return 1; case 'D': return 2; case 'N': return 3; case 'S': return 4;
        case 'H': return 5; case 'P': return 6; case '=': return 7; case 'X': return 8; default: return -1;
    }
}

BQC_SP void sam_put(uint8_t* out, uint64_t at, uint64_t v, int nbytes) {
    for (int k = 0; k < nbytes; ++k) out[at + k] = (uint8_t)(v >> (8 * k));
}

// One alignment line p[0..n) without its '\n' (a trailing '\r' is dropped here).  Returns the record's size in
// bytes with its block_size, 0 for an empty line (not a record), -1 when the line is not fast.  out (may be null)
// receives the record; lseq the length of SEQ.
BQC_SP int64_t sam_fast_line(const uint8_t* p, uint32_t n, const SamRefs& R, uint8_t* out, uint32_t& lseq) {
    if (n && p[n - 1] == '\r') --n;
    if (n == 0) return 0;
    uint32_t fb[11], fe[11];
    uint32_t nf = 0, st = 0;   // fields so far; start of the current one
    for (uint32_t i = 0; i < n; ++i) {
        const uint8_t c = p[i];
        if (c == '\t') {
            if (nf < 11) { fb[nf] = st; fe[nf] = i; }
            ++nf;
            st = i + 1;
        } else if (c < 0x20 || c > 0x7E) {
            return -1;
        }
    }
    if (nf < 11) { fb[nf] = st; fe[nf] = n; }
    ++nf;
    if (nf < 11) return -1;
    for (uint32_t k = 0; k < 11; ++k)
        if (fe[k] == fb[k]) return -1;
    const uint32_t lq = fe[0] - fb[0];
    if (lq > 254) return -1;
    uint64_t flag, mapq;
    int64_t pos, pnext, tlen;
    if (!sam_uint(p + fb[1], fe[1] - fb[1], 9, flag) || !sam_uint(p + fb[4], fe[4] - fb[4], 9, mapq)) return -1;
    if (!sam_int(p + fb[3], fe[3] - fb[3], pos) || !sam_int(p + fb[7], fe[7] - fb[7], pnext) || !sam_int(p + fb[8], fe[8] - fb[8], tlen)) return -1;
    auto rid_of = [&](uint32_t k, int32_t same) -> int32_t {
        const uint32_t len = fe[k] - fb[k];
        if (len == 1 && p[fb[k]] == '*') return -1;
        if (len == 1 && p[fb[k]] == '=') return same;
        return sam_ref_lookup(R, p + fb[k], len);
    };
    const int32_t rid = rid_of(2, -1), nrid = rid_of(6, rid);
    // CIGAR
    uint32_t ncig = 0;
    const bool cig_star = fe[5] - fb[5] == 1 && p[fb[5]] == '*';
    if (!cig_star) {
        uint32_t nd = 0;
        for (uint32_t i = fb[5]; i < fe[5]; ++i) {
            if (sam_digit(p[i])) { if (++nd > 9) return -1; continue; }
            if (nd == 0 || sam_cigar_op(p[i]) < 0) return -1;
            nd = 0;
            if (++ncig > 65535) return -1;
        }
        if (nd) return -1;
    }
    const bool seq_star = fe[9] - fb[9] == 1 && p[fb[9]] == '*';
    const uint32_t ls = seq_star ? 0 : fe[9] - fb[9];
    const uint32_t lqual = fe[10] - fb[10];
    const bool qual_fill = (lqual == 1 && p[fb[10]] == '*') || lqual != ls;
    uint64_t o = 36 + lq + 1 + 4ull * ncig + (ls + 1) / 2 + ls;   // end of the fixed part, name, CIGAR, SEQ, QUAL
    // tags
    for (uint32_t t = 11, a = fe[10] + 1; t < nf; ++t) {
        uint32_t b = a;
        while (b < n && p[b] != '\t') ++b;
        const uint32_t len = b - a;
        if (len < 5 || p[a + 2] != ':' || p[a + 4] != ':') return -1;
        const uint8_t ty = p[a + 3];
        const uint8_t* v = p + a + 5;
        const uint32_t vn = len - 5;
        if (out) { out[o] = p[a]; out[o + 1] = p[a + 1]; }
        o += 2;
        if (ty == 'A') {
            if (out) { out[o] = 'A'; out[o + 1] = vn ? v[0] : 0; }
            o += 2;
        } else if (ty == 'i') {
            int64_t x;
            if (!sam_int(v, vn, x)) return -1;
            uint8_t t;
            int nb;
            if (x >= 0) { if (x <= 255) { t = 'C'; nb = 1; } else if (x <= 65535) { t = 'S'; nb = 2; } else { t = 'I'; nb = 4; } }
            else { if (x >= -128) { t = 'c'; nb = 1; } else if (x >= -32768) { t = 's'; nb = 2; } else { t = 'i'; nb = 4; } }
            if (out) { out[o] = t; sam_put(out, o + 1, (uint64_t)x, nb); }
            o += 1 + nb;
        } else if (ty == 'f') {
            float f;
            if (!sam_float(v, vn, f)) return -1;
            if (out) {
#ifdef __CUDA_ARCH__
                const uint32_t bits = __float_as_uint(f);
#else
                uint32_t bits;
                memcpy(&bits, &f, 4);
#endif
                out[o] = 'f';
                sam_put(out, o + 1, bits, 4);
            }
            o += 5;
        } else if (ty == 'Z' || ty == 'H') {
            if (out) {
                out[o] = ty;
                for (uint32_t i = 0; i < vn; ++i) out[o + 1 + i] = v[i];
                out[o + 1 + vn] = 0;
            }
            o += 2 + vn;
        } else {
            return -1;
        }
        a = b + 1;
    }
    lseq = ls;
    if (!out) return (int64_t)o;
    sam_put(out, 0, o - 4, 4);
    sam_put(out, 4, (uint32_t)rid, 4);
    sam_put(out, 8, (uint32_t)((uint32_t)pos - 1u), 4);
    out[12] = (uint8_t)(lq + 1);
    out[13] = (uint8_t)mapq;
    sam_put(out, 14, 4680, 2);
    sam_put(out, 16, ncig, 2);
    sam_put(out, 18, (uint16_t)flag, 2);
    sam_put(out, 20, ls, 4);
    sam_put(out, 24, (uint32_t)nrid, 4);
    sam_put(out, 28, (uint32_t)((uint32_t)pnext - 1u), 4);
    sam_put(out, 32, (uint32_t)tlen, 4);
    uint64_t w = 36;
    for (uint32_t i = 0; i < lq; ++i) out[w++] = p[fb[0] + i];
    out[w++] = 0;
    if (!cig_star) {
        uint64_t x = 0;
        for (uint32_t i = fb[5]; i < fe[5]; ++i) {
            if (sam_digit(p[i])) { x = x * 10 + (p[i] - '0'); continue; }
            sam_put(out, w, (uint32_t)(x << 4) | (uint32_t)sam_cigar_op(p[i]), 4);
            w += 4;
            x = 0;
        }
    }
    const uint8_t* sq = p + fb[9];
    for (uint32_t i = 0; i < ls; i += 2) out[w++] = (uint8_t)((sam_nt16(sq[i]) << 4) | (i + 1 < ls ? sam_nt16(sq[i + 1]) : 0));
    const uint8_t* qu = p + fb[10];
    for (uint32_t i = 0; i < ls; ++i) out[w++] = qual_fill ? 0xFF : (uint8_t)(qu[i] - 33);
    return (int64_t)o;
}

}  // namespace bqc
