// synth.cpp -- seeded synthetic BAM / FASTA generator (see include/bamqc_synth.h).
//
// The reference repository ships no test data (SURVEY.md section 4).  This generator produces the
// SURVEY section 8(d) data sets: coordinate-sorted FR proper pairs over an iid-uniform ACGT genome with
// substitutions, indels, soft clips, N bases, duplicates, QC-fails, unmapped mates, secondary and
// supplementary records, and the aux tags the statistics pass consumes (RG:Z, NM, AS).  It keeps clear
// of the inputs on which the reference itself has undefined behaviour (SURVEY Appendix C "hazards"):
// every record has SEQ/QUAL/RG, mapped reads have a CIGAR that starts and ends with M or S, NM >= I+D,
// reads stay away from contig ends, read length >= 32.
#include "../../include/bamqc_synth.h"

#include <zlib.h>

#include <algorithm>
#include <thread>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <queue>
#include <string>
#include <vector>

namespace {

struct Rng {  // xoshiro256** seeded through splitmix64
    uint64_t s[4];
    static uint64_t splitmix(uint64_t& x) {
        uint64_t z = (x += 0x9E3779B97F4A7C15ULL);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        return z ^ (z >> 31);
    }
    explicit Rng(uint64_t seed) {
        for (int i = 0; i < 4; ++i) s[i] = splitmix(seed);
    }
    static inline uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    inline uint64_t next() {
        const uint64_t result = rotl(s[1] * 5, 7) * 9;
        const uint64_t t = s[1] << 17;
        s[2] ^= s[0];
        s[3] ^= s[1];
        s[1] ^= s[2];
        s[0] ^= s[3];
        s[2] ^= t;
        s[3] = rotl(s[3], 45);
        return result;
    }
    inline double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
    inline uint32_t below(uint32_t n) { return (uint32_t)(((next() >> 32) * (uint64_t)n) >> 32); }
    inline bool chance(double p) { return uniform() < p; }
    double normal() {
        double u1 = uniform(), u2 = uniform();
        if (u1 < 1e-300) u1 = 1e-300;
        return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2);
    }
};

inline int refBase(const uint8_t* packed, uint64_t i) { return (packed[i >> 2] >> ((i & 3) * 2)) & 3; }

const uint8_t kNibbleOfBase[4] = {1, 2, 4, 8};  // A C G T in BAM 4-bit codes

struct Mate {
    bool mapped = false, reverse = false;
    int32_t rid = -1;
    int64_t pos = -1;
    std::vector<uint32_t> cigar;
    std::vector<uint8_t> seq;   // BAM nibble codes, one per base, stored (reference) orientation
    std::vector<uint8_t> qual;  // raw phred, stored orientation
    int nm = 0, as = 0, mapq = 0;
    int64_t refSpan = 0;
};

void drawQuals(Rng& g, const bqc_synth_params& P, int L, bool reverse, std::vector<uint8_t>& q) {
    q.resize(L);
    for (int j = 0; j < L; ++j) {  // j = cycle in read orientation
        uint32_t x = g.below(100);
        uint8_t v;
        if (!P.low_quality) {
            v = x < 2 ? 2 : x < 7 ? 12 : x < 20 ? 23 : 37;
            if (j >= L - 10 && g.below(100) < 30) v = 2;
        } else {
            v = x < 15 ? 2 : x < 40 ? 8 : x < 70 ? 15 : x < 90 ? 23 : 37;
        }
        q[reverse ? L - 1 - j : j] = v;
    }
}

// Build one mapped mate.  If anchorEnd, `anchor` is the exclusive reference end of the alignment,
// otherwise its reference start.
void buildMapped(Rng& g, const bqc_synth_params& P, int rid, const uint8_t* ref, int64_t anchor, bool anchorEnd, bool reverse, Mate& m) {
    const int L = P.read_len;
    m.mapped = true;
    m.reverse = reverse;
    m.rid = rid;
    m.cigar.clear();
    m.seq.assign(L, 0);
    int sl = 0, sr = 0;
    if (g.chance(P.softclip_frac)) {
        uint32_t mode = g.below(100);
        int a = 5 + (int)g.below(36), b = 5 + (int)g.below(36);
        if (mode < 45) sl = a;
        else if (mode < 90) sr = b;
        else { sl = a; sr = b; }
    }
    const int A = L - sl - sr;  // read bases inside the alignment
    // indels: (offset in aligned read bases, type, len), offsets >= 10 from both ends and >= 10 apart
    struct Indel { int off, type, len; };
    std::vector<Indel> indels;
    if (A >= 60 && g.chance(P.indel_read_frac)) {
        int n = 1 + (P.max_indels > 1 ? (int)g.below((uint32_t)P.max_indels) : 0);
        int lo = 10;
        for (int i = 0; i < n; ++i) {
            int hi = A - 10 - (n - 1 - i) * 16 - 3;
            if (hi <= lo) break;
            int off = lo + (int)g.below((uint32_t)(hi - lo));
            Indel d = {off, (int)g.below(2), 1 + (int)g.below(3)};
            indels.push_back(d);
            lo = off + d.len + 10;
        }
    }
    int64_t span = A;
    int sumI = 0, sumD = 0;
    for (auto& d : indels) {
        if (d.type == 0) { span -= d.len; sumI += d.len; }
        else { span += d.len; sumD += d.len; }
    }
    m.refSpan = span;
    m.pos = anchorEnd ? anchor - span : anchor;
    // CIGAR and bases
    int rp = 0;             // read cursor
    int64_t cp = m.pos;     // reference cursor
    int mism = 0, mbases = 0;
    auto putRandom = [&](int n) { for (int i = 0; i < n; ++i) m.seq[rp++] = kNibbleOfBase[g.below(4)]; };
    auto putMatch = [&](int n) {
        for (int i = 0; i < n; ++i, ++cp) {
            int b = refBase(ref, (uint64_t)cp);
            if (g.chance(P.sub_rate)) { b = (b + 1 + (int)g.below(3)) & 3; ++mism; }
            m.seq[rp++] = kNibbleOfBase[b];
        }
        mbases += n;
    };
    if (sl) { m.cigar.push_back(((uint32_t)sl << 4) | 4); putRandom(sl); }
    int done = 0;  // aligned read bases consumed
    for (auto& d : indels) {
        int mlen = d.off - done;
        m.cigar.push_back(((uint32_t)mlen << 4) | 0);
        putMatch(mlen);
        done = d.off;
        if (d.type == 0) { m.cigar.push_back(((uint32_t)d.len << 4) | 1); putRandom(d.len); done += d.len; }
        else { m.cigar.push_back(((uint32_t)d.len << 4) | 2); cp += d.len; }
    }
    m.cigar.push_back(((uint32_t)(A - done) << 4) | 0);
    putMatch(A - done);
    if (sr) { m.cigar.push_back(((uint32_t)sr << 4) | 4); putRandom(sr); }
    drawQuals(g, P, L, reverse, m.qual);
    for (int j = 0; j < L; ++j)
        if (g.chance(P.n_rate)) {
            if (m.seq[j] != 15) { m.seq[j] = 15; m.qual[j] = 2; }
        }
    // N inside the alignment counts as a mismatch for NM (cheap recount)
    m.nm = mism + sumI + sumD;
    int as = mbases - 5 * mism - 7 * (int)indels.size();
    m.as = as < 0 ? 0 : as;
    if (P.mapq60_frac < 0) m.mapq = (int)g.below(61);
    else m.mapq = g.chance(P.mapq60_frac) ? 60 : (int)g.below(60);
}

void buildUnmapped(Rng& g, const bqc_synth_params& P, Mate& m) {
    const int L = P.read_len;
    m.mapped = false;
    m.reverse = false;
    m.cigar.clear();
    m.seq.resize(L);
    for (int j = 0; j < L; ++j) m.seq[j] = kNibbleOfBase[g.below(4)];
    drawQuals(g, P, L, false, m.qual);
    for (int j = 0; j < L; ++j)
        if (g.chance(P.n_rate * 5)) { m.seq[j] = 15; m.qual[j] = 2; }
    m.nm = m.as = m.mapq = 0;
    m.refSpan = 0;
}

int reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

template <typename T>
void put(std::vector<uint8_t>& b, T v) {
    size_t o = b.size();
    b.resize(o + sizeof(T));
    memcpy(&b[o], &v, sizeof(T));
}

void serialize(const Mate& m, const Mate& mate, uint16_t flag, int32_t tlen, uint64_t pairId, int lane, std::vector<uint8_t>& b, bool withAlnTags) {
    b.clear();
    put<int32_t>(b, 0);  // block_size patched below
    // an unmapped mate is placed at its mapped mate's position (SAM convention)
    int32_t rid = m.mapped ? m.rid : (mate.mapped ? mate.rid : -1);
    int32_t pos = m.mapped ? (int32_t)m.pos : (mate.mapped ? (int32_t)mate.pos : -1);
    int32_t nrid = mate.mapped ? mate.rid : rid;
    int32_t npos = mate.mapped ? (int32_t)mate.pos : pos;
    put<int32_t>(b, rid);
    put<int32_t>(b, pos);
    char name[24];
    int ln = snprintf(name, sizeof(name), "p%09llu", (unsigned long long)pairId) + 1;
    put<uint8_t>(b, (uint8_t)ln);
    put<uint8_t>(b, (uint8_t)m.mapq);
    put<uint16_t>(b, (uint16_t)(pos >= 0 ? reg2bin(pos, pos + (m.refSpan > 0 ? m.refSpan : 1)) : 4680));
    put<uint16_t>(b, (uint16_t)m.cigar.size());
    put<uint16_t>(b, flag);
    put<int32_t>(b, (int32_t)m.seq.size());
    put<int32_t>(b, nrid);
    put<int32_t>(b, npos);
    put<int32_t>(b, tlen);
    b.insert(b.end(), (const uint8_t*)name, (const uint8_t*)name + ln);
    for (uint32_t c : m.cigar) put<uint32_t>(b, c);
    size_t L = m.seq.size();
    for (size_t i = 0; i < L; i += 2) {
        uint8_t hi = m.seq[i], lo = (i + 1 < L) ? m.seq[i + 1] : 0;
        b.push_back((uint8_t)((hi << 4) | lo));
    }
    b.insert(b.end(), m.qual.begin(), m.qual.end());
    // aux: RG:Z:L<k>  NM  AS
    char rg[16];
    int lr = snprintf(rg, sizeof(rg), "L%d", lane + 1) + 1;
    b.push_back('R'); b.push_back('G'); b.push_back('Z');
    b.insert(b.end(), (const uint8_t*)rg, (const uint8_t*)rg + lr);
    if (withAlnTags) {
        b.push_back('N'); b.push_back('M');
        if (m.nm < 256) { b.push_back('C'); b.push_back((uint8_t)m.nm); }
        else { b.push_back('S'); put<uint16_t>(b, (uint16_t)m.nm); }
        b.push_back('A'); b.push_back('S');
        if (m.as < 256) { b.push_back('C'); b.push_back((uint8_t)m.as); }
        else { b.push_back('S'); put<uint16_t>(b, (uint16_t)m.as); }
    }
    int32_t bs = (int32_t)(b.size() - 4);
    memcpy(&b[0], &bs, 4);
}

struct Pending {
    int64_t pos;
    uint64_t order;
    std::vector<uint8_t> bytes;
    bool operator<(const Pending& o) const { return pos != o.pos ? pos > o.pos : order > o.order; }  // min-heap
};

struct Sink {
    uint8_t* out;
    uint64_t cap, n = 0;
    uint64_t* offs;
    uint64_t offCap, nrec = 0;
    bool overflow = false;
    void add(const std::vector<uint8_t>& b) {
        if (n + b.size() > cap || nrec + 1 >= offCap) overflow = true;
        if (!overflow) {
            offs[nrec] = n;
            memcpy(out + n, b.data(), b.size());
        }
        n += b.size();
        ++nrec;
    }
};

}  // namespace

extern "C" {

void bqc_synth_default_params(bqc_synth_params* p) {
    memset(p, 0, sizeof(*p));
    p->seed = 20260101;
    p->read_len = 150;
    p->ins_mean = 400;
    p->ins_sd = 60;
    p->ins_min = 150;
    p->ins_max = 1000;
    p->sub_rate = 0.005;
    p->n_rate = 0.001;
    p->indel_read_frac = 0.03;
    p->max_indels = 1;
    p->softclip_frac = 0.03;
    p->low_quality = 0;
    p->mapq60_frac = 0.9;
    p->dup_frac = 0.02;
    p->qcfail_frac = 0.005;
    p->one_unmapped_frac = 0.01;
    p->both_unmapped_frac = 0.005;
    p->secondary_frac = 0.005;
    p->supplementary_frac = 0.005;
    p->n_lanes = 1;
    p->first_pair_id = 0;
    p->emit_unmapped_tail = 1;
}

void bqc_synth_reference(uint64_t seed, int32_t contig_index, uint64_t n_bases, uint8_t* packed_out) {
    Rng g(seed * 0x9E3779B97F4A7C15ULL + 0x1234567ULL * (uint64_t)(contig_index + 1));
    uint64_t nwords = (n_bases + 31) / 32;
    for (uint64_t w = 0; w < nwords; ++w) {
        uint64_t v = g.next();
        memcpy(packed_out + 8 * w, &v, 8);
    }
}

int bqc_synth_write_fasta(const char* path, int32_t n_contigs, const char* const* names, const uint64_t* lengths, const uint8_t* const* packed) {
    FILE* f = fopen(path, "wb");
    if (!f) return 1;
    std::vector<char> line(61);
    for (int c = 0; c < n_contigs; ++c) {
        fprintf(f, ">%s\n", names[c]);
        for (uint64_t i = 0; i < lengths[c]; i += 60) {
            int n = (int)std::min<uint64_t>(60, lengths[c] - i);
            for (int j = 0; j < n; ++j) line[j] = "ACGT"[refBase(packed[c], i + j)];
            line[n] = '\n';
            fwrite(line.data(), 1, (size_t)n + 1, f);
        }
    }
    fclose(f);
    return 0;
}

size_t bqc_synth_header_text(const bqc_synth_params* p, const char* sample_id, char* out, size_t cap) {
    std::string h = "@HD\tVN:1.6\tSO:coordinate\n";
    for (int c = 0; c < p->n_contigs; ++c) h += "@SQ\tSN:" + std::string(p->names[c]) + "\tLN:" + std::to_string(p->lengths[c]) + "\n";
    for (int l = 0; l < p->n_lanes; ++l) h += "@RG\tID:L" + std::to_string(l + 1) + "\tSM:" + std::string(sample_id) + "\n";
    if (out && cap) {
        size_t n = std::min(cap, h.size());
        memcpy(out, h.data(), n);
    }
    return h.size();
}

int bqc_synth_records(const bqc_synth_params* pp, uint8_t* out, uint64_t out_cap, uint64_t* n_bytes, uint64_t* offsets_out, uint64_t offsets_cap, uint64_t* n_records) {
    const bqc_synth_params& P = *pp;
    Rng g(P.seed ^ 0xA5A5A5A5DEADBEEFULL);
    Sink sink = {out, out_cap, 0, offsets_out, offsets_cap, 0, false};
    const int64_t margin = 64;
    // total usable region length -> mean gap between fragment starts
    double total = 0;
    for (int c = 0; c < P.n_contigs; ++c) {
        int64_t b = P.region_begin ? (int64_t)P.region_begin[c] : 0, e = P.region_end ? (int64_t)P.region_end[c] : (int64_t)P.lengths[c];
        b = std::max<int64_t>(b, margin);
        e = std::min<int64_t>(e, (int64_t)P.lengths[c] - P.ins_max - margin);
        if (e > b) total += (double)(e - b);
    }
    const double meanGap = P.n_pairs ? total / (double)P.n_pairs : 1e18;
    std::priority_queue<Pending> heap;
    uint64_t order = 0, pairId = P.first_pair_id;
    std::vector<std::vector<uint8_t>> unmappedTail;
    std::vector<uint8_t> buf;
    Mate m1, m2;
    for (int c = 0; c < P.n_contigs; ++c) {
        int64_t b = P.region_begin ? (int64_t)P.region_begin[c] : 0, e = P.region_end ? (int64_t)P.region_end[c] : (int64_t)P.lengths[c];
        b = std::max<int64_t>(b, margin);
        e = std::min<int64_t>(e, (int64_t)P.lengths[c] - P.ins_max - margin);
        if (e <= b) continue;
        const uint8_t* ref = P.packed[c];
        double x = (double)b + (-std::log(1.0 - g.uniform())) * meanGap;
        while (x < (double)e) {
            int64_t s = (int64_t)x;
            x += (-std::log(1.0 - g.uniform())) * meanGap;
            while (!heap.empty() && heap.top().pos <= s) {
                sink.add(heap.top().bytes);
                heap.pop();
            }
            int lane = P.n_lanes > 1 ? (int)g.below((uint32_t)P.n_lanes) : 0;
            double kind = g.uniform();
            uint64_t id = pairId++;
            if (kind < P.both_unmapped_frac) {
                buildUnmapped(g, P, m1);
                buildUnmapped(g, P, m2);
                if (P.emit_unmapped_tail) {
                    serialize(m1, m2, (uint16_t)(0x1 | 0x4 | 0x8 | 0x40), 0, id, lane, buf, false);
                    unmappedTail.push_back(buf);
                    serialize(m2, m1, (uint16_t)(0x1 | 0x4 | 0x8 | 0x80), 0, id, lane, buf, false);
                    unmappedTail.push_back(buf);
                }
                continue;
            }
            int ins = (int)std::lround(P.ins_mean + P.ins_sd * g.normal());
            ins = std::max(P.ins_min, std::min(P.ins_max, ins));
            if (ins < P.read_len + 8) ins = P.read_len + 8;
            bool firstIsLeft = g.below(2) == 0;
            uint16_t pairFlags = 0;
            if (g.chance(P.dup_frac)) pairFlags |= 0x400;
            if (g.chance(P.qcfail_frac)) pairFlags |= 0x200;
            bool oneUnmapped = kind < P.both_unmapped_frac + P.one_unmapped_frac;
            Mate left, right;
            buildMapped(g, P, c, ref, s, false, false, left);
            if (oneUnmapped) {
                buildUnmapped(g, P, right);
                bool mappedIsFirst = firstIsLeft;
                uint16_t fm = (uint16_t)(0x1 | 0x8 | (mappedIsFirst ? 0x40 : 0x80) | pairFlags);
                uint16_t fu = (uint16_t)(0x1 | 0x4 | (mappedIsFirst ? 0x80 : 0x40) | pairFlags);
                serialize(left, right, fm, 0, id, lane, buf, true);
                sink.add(buf);
                serialize(right, left, fu, 0, id, lane, buf, false);
                sink.add(buf);
                continue;
            }
            buildMapped(g, P, c, ref, s + ins, true, true, right);
            if (right.pos < left.pos) right.pos = left.pos, right.refSpan = right.refSpan;  // cannot happen with ins >= read_len + 8
            int32_t tl = (int32_t)(right.pos + right.refSpan - left.pos);
            uint16_t fl = (uint16_t)(0x1 | 0x2 | 0x20 | (firstIsLeft ? 0x40 : 0x80) | pairFlags);
            uint16_t fr = (uint16_t)(0x1 | 0x2 | 0x10 | (firstIsLeft ? 0x80 : 0x40) | pairFlags);
            serialize(left, right, fl, tl, id, lane, buf, true);
            sink.add(buf);
            if (g.chance(P.secondary_frac)) {  // extra secondary copy of the left mate
                Mate sec = left;
                sec.mapq = 0;
                serialize(sec, right, (uint16_t)(fl | 0x100), tl, id, lane, buf, true);
                sink.add(buf);
            }
            if (g.chance(P.supplementary_frac)) {  // extra supplementary record: <h>H<L-h>M at the same position
                Mate sup;
                sup.mapped = true;
                sup.rid = c;
                sup.pos = left.pos;
                int h = 20 + (int)g.below(60), ml = P.read_len - h;
                sup.cigar.push_back(((uint32_t)h << 4) | 5);
                sup.cigar.push_back(((uint32_t)ml << 4) | 0);
                sup.seq.resize(ml);
                sup.qual.assign(ml, 30);
                for (int j = 0; j < ml; ++j) sup.seq[j] = kNibbleOfBase[refBase(ref, (uint64_t)(left.pos + j))];
                sup.refSpan = ml;
                sup.nm = 0;
                sup.as = ml;
                sup.mapq = left.mapq;
                serialize(sup, right, (uint16_t)(fl | 0x800), tl, id, lane, buf, true);
                sink.add(buf);
            }
            serialize(right, left, fr, -tl, id, lane, buf, true);
            Pending pd;
            pd.pos = right.pos;
            pd.order = order++;
            pd.bytes = buf;
            heap.push(std::move(pd));
        }
        while (!heap.empty()) {  // contig change: flush
            sink.add(heap.top().bytes);
            heap.pop();
        }
    }
    for (auto& u : unmappedTail) sink.add(u);
    if (!sink.overflow) offsets_out[sink.nrec] = sink.n;
    *n_bytes = sink.n;
    *n_records = sink.nrec;
    return sink.overflow ? 1 : 0;
}

static void bamHeaderBytes(const bqc_synth_params* p, const char* sample_id, std::vector<uint8_t>& h) {
    size_t lt = bqc_synth_header_text(p, sample_id, nullptr, 0);
    std::string text(lt, '\0');
    bqc_synth_header_text(p, sample_id, &text[0], lt);
    h.clear();
    h.insert(h.end(), {'B', 'A', 'M', 1});
    put<int32_t>(h, (int32_t)lt);
    h.insert(h.end(), text.begin(), text.end());
    put<int32_t>(h, p->n_contigs);
    for (int c = 0; c < p->n_contigs; ++c) {
        size_t ln = strlen(p->names[c]) + 1;
        put<int32_t>(h, (int32_t)ln);
        h.insert(h.end(), (const uint8_t*)p->names[c], (const uint8_t*)p->names[c] + ln);
        put<int32_t>(h, (int32_t)p->lengths[c]);
    }
}

static size_t bgzfBlock(const uint8_t* in, size_t n, int level, uint8_t* out) {
    // out needs >= n + 64 bytes
    static const uint8_t hdr[12] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0};
    memcpy(out, hdr, 12);
    out[12] = 'B'; out[13] = 'C'; out[14] = 2; out[15] = 0;
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
    zs.next_in = (Bytef*)in;
    zs.avail_in = (uInt)n;
    zs.next_out = out + 18;
    zs.avail_out = (uInt)(n + 64 - 18 - 8);
    deflate(&zs, Z_FINISH);
    size_t clen = zs.total_out;
    deflateEnd(&zs);
    uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), in, (uInt)n);
    uint32_t isize = (uint32_t)n;
    memcpy(out + 18 + clen, &crc, 4);
    memcpy(out + 22 + clen, &isize, 4);
    uint16_t bsize = (uint16_t)(18 + clen + 8 - 1);
    memcpy(out + 16, &bsize, 2);
    return 18 + clen + 8;
}

uint64_t bqc_synth_bgzf_compress(const uint8_t* in, uint64_t n, int level, uint8_t* out, uint64_t cap) {
    // blocks are independent: compressed by all host threads in groups, concatenated in order
    const size_t chunk = 0xff00;
    const uint64_t nblk = (n + chunk - 1) / chunk;
    const unsigned T = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(std::thread::hardware_concurrency(), nblk / 8));
    const uint64_t group = 256;  // blocks per work item
    const uint64_t ngroups = (nblk + group - 1) / group;
    std::vector<std::vector<uint8_t>> parts((size_t)ngroups);
    std::atomic<uint64_t> next(0);
    auto work = [&]() {
        std::vector<uint8_t> tmp(chunk + 1024);
        for (;;) {
            const uint64_t g = next.fetch_add(1);
            if (g >= ngroups) break;
            std::vector<uint8_t>& dst = parts[(size_t)g];
            for (uint64_t b = g * group; b < std::min(nblk, (g + 1) * group); ++b) {
                const uint64_t p = b * chunk;
                const size_t m = (size_t)std::min<uint64_t>(chunk, n - p);
                const size_t len = bgzfBlock(in + p, m, level, tmp.data());
                dst.insert(dst.end(), tmp.begin(), tmp.begin() + len);
            }
        }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < T; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    uint64_t o = 0;
    for (auto& part : parts) {
        if (o + part.size() > cap) return 0;
        memcpy(out + o, part.data(), part.size());
        o += part.size();
    }
    std::vector<uint8_t> tmp(1024);
    size_t b = bgzfBlock(in, 0, level, tmp.data());  // EOF block
    if (o + b > cap) return 0;
    memcpy(out + o, tmp.data(), b);
    return o + b;
}

int bqc_synth_write_bam(const char* path, const bqc_synth_params* p, const char* sample_id, const uint8_t* records, uint64_t n_bytes, int compress_level) {
    std::vector<uint8_t> h;
    bamHeaderBytes(p, sample_id, h);
    FILE* f = fopen(path, "wb");
    if (!f) return 1;
    if (compress_level < 0) {
        fwrite(h.data(), 1, h.size(), f);
        fwrite(records, 1, n_bytes, f);
        fclose(f);
        return 0;
    }
    const size_t chunk = 0xff00;
    std::vector<uint8_t> tmp(chunk + 1024), stage;
    stage.reserve(chunk);
    auto flush = [&](const uint8_t* d, size_t n) {
        size_t b = bgzfBlock(d, n, compress_level, tmp.data());
        fwrite(tmp.data(), 1, b, f);
    };
    // header in its own block(s), then the record stream
    for (size_t o = 0; o < h.size(); o += chunk) flush(h.data() + o, std::min(chunk, h.size() - o));
    for (uint64_t o = 0; o < n_bytes; o += chunk) flush(records + o, (size_t)std::min<uint64_t>(chunk, n_bytes - o));
    flush(records, 0);
    fclose(f);
    return 0;
}

// SAM text of the records (SAM/BAM specification 1.4 and 4.2): the header of bqc_synth_header_text, one line per
// record.  B arrays, every integer type and f are written; the text encodes back to the same field values.
int bqc_synth_write_sam(const char* path, const bqc_synth_params* p, const char* sample_id, const uint8_t* records, uint64_t n_bytes) {
    FILE* f = fopen(path, "wb");
    if (!f) return 1;
    std::string line, head(bqc_synth_header_text(p, sample_id, nullptr, 0), '\0');
    bqc_synth_header_text(p, sample_id, &head[0], head.size());
    fwrite(head.data(), 1, head.size(), f);
    static const char kOps[] = "MIDNSHP=X??????", kNt[] = "=ACMGRSVTWYHKDBN";
    auto rd = [](const uint8_t* q, int n) { uint64_t v = 0; memcpy(&v, q, n); return v; };
    auto ref = [&](int32_t id) { return id >= 0 && id < p->n_contigs ? std::string(p->names[id]) : std::string("*"); };
    char num[64];
    for (uint64_t o = 0; o + 4 <= n_bytes;) {
        const uint32_t bs = (uint32_t)rd(records + o, 4);
        const uint8_t* r = records + o + 4;
        const uint8_t* end = r + bs;
        o += 4 + (uint64_t)bs;
        const int32_t rid = (int32_t)rd(r, 4), pos = (int32_t)rd(r + 4, 4), nrid = (int32_t)rd(r + 20, 4), npos = (int32_t)rd(r + 24, 4), tlen = (int32_t)rd(r + 28, 4);
        const uint32_t lname = r[8], mapq = r[9], ncig = (uint32_t)rd(r + 12, 2), flag = (uint32_t)rd(r + 14, 2), lseq = (uint32_t)rd(r + 16, 4);
        const uint8_t* q = r + 32;
        line.assign((const char*)q, lname ? lname - 1 : 0);
        q += lname;
        snprintf(num, sizeof(num), "\t%u\t", flag);
        line += num + ref(rid);
        snprintf(num, sizeof(num), "\t%d\t%u\t", pos + 1, mapq);
        line += num;
        if (!ncig) line += '*';
        for (uint32_t k = 0; k < ncig; ++k, q += 4) {
            const uint32_t c = (uint32_t)rd(q, 4);
            snprintf(num, sizeof(num), "%u%c", c >> 4, kOps[c & 15]);
            line += num;
        }
        line += '\t';
        line += nrid < 0 ? "*" : (nrid == rid ? "=" : ref(nrid));
        snprintf(num, sizeof(num), "\t%d\t%d\t", npos + 1, tlen);
        line += num;
        if (!lseq) line += '*';
        for (uint32_t k = 0; k < lseq; ++k) line += kNt[(q[k / 2] >> (k % 2 ? 0 : 4)) & 15];
        q += (lseq + 1) / 2;
        line += '\t';
        if (!lseq || q[0] == 0xFF) line += '*';
        else for (uint32_t k = 0; k < lseq; ++k) line += (char)(q[k] + 33);
        q += lseq;
        while (q + 3 <= end) {   // tags
            const char t0 = (char)q[0], t1 = (char)q[1], ty = (char)q[2];
            q += 3;
            line += '\t'; line += t0; line += t1;
            auto ival = [&](char t, const uint8_t* v) -> long long {
                switch (t) {
                    case 'c': return (int8_t)v[0]; case 'C': return v[0]; case 's': return (int16_t)rd(v, 2); case 'S': return (uint16_t)rd(v, 2);
                    case 'i': return (int32_t)rd(v, 4); default: return (uint32_t)rd(v, 4);
                }
            };
            auto isz = [](char t) { return t == 'c' || t == 'C' || t == 'A' ? 1 : t == 's' || t == 'S' ? 2 : 4; };
            if (ty == 'A') { line += ":A:"; line += (char)q[0]; q += 1; }
            else if (ty == 'Z' || ty == 'H') {
                line += ty == 'Z' ? ":Z:" : ":H:";
                const uint8_t* z = q;
                while (z < end && *z) ++z;
                line.append((const char*)q, z - q);
                q = z + 1;
            } else if (ty == 'f') { float x; memcpy(&x, q, 4); snprintf(num, sizeof(num), ":f:%.9g", x); line += num; q += 4; }
            else if (ty == 'B') {
                const char sub = (char)q[0];
                const uint32_t cnt = (uint32_t)rd(q + 1, 4);
                q += 5;
                line += ":B:"; line += sub;
                for (uint32_t k = 0; k < cnt; ++k, q += isz(sub)) {
                    if (sub == 'f') { float x; memcpy(&x, q, 4); snprintf(num, sizeof(num), ",%.9g", x); }
                    else snprintf(num, sizeof(num), ",%lld", ival(sub, q));
                    line += num;
                }
            } else { snprintf(num, sizeof(num), ":i:%lld", ival(ty, q)); line += num; q += isz(ty); }
        }
        line += '\n';
        if (fwrite(line.data(), 1, line.size(), f) != line.size()) { fclose(f); return 1; }
    }
    return fclose(f) ? 1 : 0;
}

}  // extern "C"
