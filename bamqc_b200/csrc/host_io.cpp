// host_io.cpp -- the host front end that stays on CPU threads (BASELINE.json north_star): BGZF inflate,
// BAM header parsing (the SeqAn BamStream stand-in, src/bamqualcheck.cpp:262,286,292), FASTA -> 2-bit
// loading (replaces the streaming cursor of src/TripletCounting.hpp:60-104), the `.bamqc` writer
// (src/bamqualcheck.cpp:156-233) and the `bamqualcheck` command line (src/CommandLineParser.hpp:43-149).
// Everything here talks to the GPU engine only through include/bamqc_b200.h.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <cerrno>
#include <atomic>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <iostream>
#include <map>
#include <set>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../include/bamqc_b200.h"
#include "sam_text.h"

// ------------------------------------------------------------------------------------------------
// BAM header
// ------------------------------------------------------------------------------------------------
static char* dup_cstr(const std::string& s) {
    char* p = (char*)malloc(s.size() + 1);
    memcpy(p, s.data(), s.size());
    p[s.size()] = 0;
    return p;
}

extern "C" size_t bqc_parse_bam_header(const uint8_t* d, size_t n, bqc_bam_header* out) {
    memset(out, 0, sizeof(*out));
    if (n < 12 || memcmp(d, "BAM\1", 4) != 0) return 0;
    int32_t l_text;
    memcpy(&l_text, d + 4, 4);
    if (l_text < 0 || 8 + (size_t)l_text + 4 > n) return 0;
    std::string text((const char*)d + 8, (size_t)l_text);
    size_t p = 8 + (size_t)l_text;
    int32_t n_ref;
    memcpy(&n_ref, d + p, 4);
    p += 4;
    if (n_ref < 0) return 0;
    std::vector<std::string> names;
    std::vector<int64_t> lens;
    for (int i = 0; i < n_ref; ++i) {
        if (p + 4 > n) return 0;
        int32_t l_name;
        memcpy(&l_name, d + p, 4);
        p += 4;
        if (l_name < 0 || p + (size_t)l_name + 4 > n) return 0;
        names.push_back(std::string((const char*)d + p, l_name > 0 ? (size_t)l_name - 1 : 0));
        p += (size_t)l_name;
        int32_t l_ref;
        memcpy(&l_ref, d + p, 4);
        p += 4;
        lens.push_back(l_ref);
    }
    // @RG lines: ID -> lane (order of appearance), last SM -> sample id (src/bamqualcheck.cpp:44-66)
    std::vector<std::string> lanes;
    std::map<std::string, unsigned> laneNames;
    std::string sample;
    std::istringstream hs(text);
    std::string line;
    while (std::getline(hs, line)) {
        if (line.compare(0, 3, "@RG") != 0) continue;
        std::istringstream ls(line);
        std::string field;
        bool firstField = true;
        while (std::getline(ls, field, '\t')) {
            if (firstField) { firstField = false; continue; }
            if (field.size() < 3 || field[2] != ':') continue;
            std::string key = field.substr(0, 2), value = field.substr(3);
            if (key == "ID" && !laneNames.count(value)) {
                laneNames[value] = (unsigned)lanes.size();
                lanes.push_back(value);
            }
            if (key == "SM") sample = value;
        }
    }
    out->text = dup_cstr(text);
    out->n_ref = n_ref;
    out->ref_names = (char**)calloc((size_t)std::max(1, n_ref), sizeof(char*));
    out->ref_lengths = (int64_t*)calloc((size_t)std::max(1, n_ref), sizeof(int64_t));
    for (int i = 0; i < n_ref; ++i) {
        out->ref_names[i] = dup_cstr(names[i]);
        out->ref_lengths[i] = lens[i];
    }
    out->n_lanes = (int32_t)lanes.size();
    out->lane_ids = (char**)calloc(std::max<size_t>(1, lanes.size()), sizeof(char*));
    for (size_t i = 0; i < lanes.size(); ++i) out->lane_ids[i] = dup_cstr(lanes[i]);
    out->sample_id = dup_cstr(sample);
    return p;
}

extern "C" void bqc_free_bam_header(bqc_bam_header* h) {
    if (!h) return;
    free(h->text);
    for (int i = 0; i < h->n_ref; ++i) free(h->ref_names[i]);
    free(h->ref_names);
    free(h->ref_lengths);
    for (int i = 0; i < h->n_lanes; ++i) free(h->lane_ids[i]);
    free(h->lane_ids);
    free(h->sample_id);
    memset(h, 0, sizeof(*h));
}

// SAM header lines ('@' at the start; a trailing '\r' dropped) -> the binary BAM header -> the same parser
extern "C" int bqc_parse_sam_header(const char* text, size_t n, bqc_bam_header* out, size_t* consumed) {
    std::string head;
    size_t p = 0;
    while (p < n && text[p] == '@') {
        const char* q = (const char*)memchr(text + p, '\n', n - p);
        const size_t end = q ? (size_t)(q - text) : n;
        size_t len = end - p;
        if (len && text[p + len - 1] == '\r') --len;
        head.append(text + p, len);
        head += '\n';
        p = q ? end + 1 : n;
    }
    *consumed = p;
    const std::vector<uint8_t> bam = sam_header_to_bam(head);
    return bqc_parse_bam_header(bam.data(), bam.size(), out) ? 0 : BQC_ERR_ARG;
}

// ------------------------------------------------------------------------------------------------
// BGZF
// ------------------------------------------------------------------------------------------------
struct BgzfBlock {
    uint64_t bbeg;   // start of the block (gzip member header)
    uint64_t cbeg;   // start of the raw deflate payload
    uint32_t clen;   // payload length
    uint32_t isize;  // inflated size
    uint64_t obeg;   // offset in the output
};

// Index the blocks of in[0..n).  Stops at the first incomplete block; returns bytes consumed.
static uint64_t bgzf_index(const uint8_t* in, uint64_t n, std::vector<BgzfBlock>& blocks, uint64_t max_out, bool& bad) {
    uint64_t p = 0, o = 0;
    bad = false;
    while (p + 18 <= n) {
        if (in[p] != 0x1f || in[p + 1] != 0x8b || in[p + 2] != 8 || !(in[p + 3] & 4)) { bad = true; break; }
        uint16_t xlen;
        memcpy(&xlen, in + p + 10, 2);
        if (p + 12 + xlen > n) break;
        uint64_t x = p + 12, xend = x + xlen;
        int bsize = -1;
        while (x + 4 <= xend) {
            uint16_t slen;
            memcpy(&slen, in + x + 2, 2);
            if (in[x] == 'B' && in[x + 1] == 'C' && slen == 2) {
                uint16_t b;
                memcpy(&b, in + x + 4, 2);
                bsize = b;
            }
            x += 4 + slen;
        }
        if (bsize < 0) { bad = true; break; }
        uint64_t blen = (uint64_t)bsize + 1;
        if (p + blen > n) break;
        if (blen < 12ull + xlen + 8) { bad = true; break; }
        BgzfBlock b;
        memcpy(&b.isize, in + p + blen - 4, 4);
        if (o + b.isize > max_out) break;
        b.bbeg = p;
        b.cbeg = p + 12 + xlen;
        b.clen = (uint32_t)(blen - 12 - xlen - 8);
        b.obeg = o;
        o += b.isize;
        blocks.push_back(b);
        p += blen;
    }
    return p;
}

static bool inflate_blocks(const uint8_t* in, const std::vector<BgzfBlock>& blocks, uint8_t* out, int threads) {
    std::atomic<size_t> next(0);
    std::atomic<bool> ok(true);
    auto work = [&]() {
        z_stream zs;
        memset(&zs, 0, sizeof(zs));
        if (inflateInit2(&zs, -15) != Z_OK) { ok = false; return; }
        for (;;) {
            size_t i0 = next.fetch_add(16);
            if (i0 >= blocks.size()) break;
            for (size_t i = i0; i < std::min(blocks.size(), i0 + 16); ++i) {
                const BgzfBlock& b = blocks[i];
                if (!b.isize) continue;
                inflateReset(&zs);
                zs.next_in = (Bytef*)(in + b.cbeg);
                zs.avail_in = b.clen;
                zs.next_out = out + b.obeg;
                zs.avail_out = b.isize;
                if (inflate(&zs, Z_FINISH) != Z_STREAM_END) ok = false;
            }
        }
        inflateEnd(&zs);
    };
    threads = std::max(1, threads);
    if (threads == 1 || blocks.size() < 32) {
        work();
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < threads; ++t) pool.emplace_back(work);
        for (auto& t : pool) t.join();
    }
    return ok;
}

extern "C" uint64_t bqc_bgzf_inflate(const uint8_t* in, uint64_t n, uint8_t* out, uint64_t cap, int32_t threads) {
    std::vector<BgzfBlock> blocks;
    bool bad = false;
    uint64_t used = bgzf_index(in, n, blocks, cap, bad);
    if (bad || used != n) return 0;
    if (!inflate_blocks(in, blocks, out, threads)) return 0;
    return blocks.empty() ? 0 : blocks.back().obeg + blocks.back().isize;
}

// ------------------------------------------------------------------------------------------------
// FASTA -> 2 bit
// ------------------------------------------------------------------------------------------------
struct bqc_fasta {
    std::vector<std::string> names;
    std::vector<std::vector<uint8_t>> packed;
    std::vector<int64_t> lengths;
};

// FASTA -> 2 bits per base on all host threads (a human reference is 3 GB of text; one byte at a time on one thread it
// took longer than the whole statistics pass of a 30x genome on the GPU).  The file is read once, records are found
// with memchr, and every record's sequence bytes are cut into chunks: pass 1 counts the bases of each chunk (white
// space skipped), a prefix sum gives the chunk's first base index, pass 2 packs.  Two chunks can share an output
// byte at their boundary, so the first and last byte of a chunk are merged with atomic ORs.
struct FastaLut {  // per byte: 0..3 = 2-bit code, 4 = white space (not a base)
    uint8_t v[256];
    FastaLut() {
        for (int i = 0; i < 256; ++i) v[i] = 0;  // Dna5 -> Dna keeps the low two bits: N (4) -> A (0), SURVEY R6
        v['C'] = v['c'] = 1;
        v['G'] = v['g'] = 2;
        v['T'] = v['t'] = 3;
        v['\n'] = v['\r'] = v[' '] = v['\t'] = 4;
    }
};
static const FastaLut kFastaLut;

extern "C" bqc_fasta* bqc_fasta_open(const char* path) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return nullptr;
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return nullptr; }
    const size_t n = (size_t)st.st_size;
    const char* d = nullptr;
    void* map = nullptr;
    std::vector<char> fallback;
    if (n) {
        map = mmap(nullptr, n, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
        if (map == MAP_FAILED) {  // e.g. a pipe or an odd file system: read it
            map = nullptr;
            fallback.resize(n);
            size_t got = 0;
            while (got < n) {
                const ssize_t r = read(fd, fallback.data() + got, n - got);
                if (r <= 0) break;
                got += (size_t)r;
            }
            if (got != n) { close(fd); return nullptr; }
            d = fallback.data();
        } else {
            d = (const char*)map;
        }
    }
    close(fd);
    bqc_fasta* fa = new bqc_fasta();
    // records: '>' at the start of a line opens a header line; the sequence runs to the next such '>'.  '>' is rare
    // inside sequence text, so the scan is a memchr for '>' plus a look at the byte before it.
    struct Rec { size_t seq_beg, seq_end; };
    std::vector<Rec> recs;
    size_t p = 0;
    while (p < n) {
        const char* q = (const char*)memchr(d + p, '>', n - p);
        if (!q) break;
        const size_t at = (size_t)(q - d);
        if (at > 0 && d[at - 1] != '\n') { p = at + 1; continue; }  // not at a line start: an ordinary character
        const char* eol = (const char*)memchr(d + at, '\n', n - at);
        const size_t hend = eol ? (size_t)(eol - d) : n;
        std::string hdr(d + at + 1, d + hend);
        std::string name = hdr.substr(0, hdr.find(' '));
        name = name.substr(0, name.find('\t'));  // src/TripletCounting.hpp:99-102
        while (!name.empty() && (name.back() == '\r' || name.back() == '\n')) name.pop_back();
        if (!recs.empty()) recs.back().seq_end = at;
        fa->names.push_back(name);
        recs.push_back({std::min(n, hend + 1), n});
        p = std::min(n, hend + 1);
    }
    const unsigned T = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    const uint8_t* lut = kFastaLut.v;
    fa->packed.resize(recs.size());
    fa->lengths.assign(recs.size(), 0);
    for (size_t r = 0; r < recs.size(); ++r) {
        const size_t beg = recs[r].seq_beg, end = recs[r].seq_end;
        const size_t span = end > beg ? end - beg : 0;
        const unsigned parts = (unsigned)std::max<size_t>(1, std::min<size_t>(T, span >> 20));
        std::vector<size_t> count(parts + 1, 0);
        auto bounds = [&](unsigned t) { return beg + span * t / parts; };
        auto pass1 = [&](unsigned t) {
            size_t c = 0;
            for (size_t i = bounds(t), e = bounds(t + 1); i < e; ++i) c += lut[(unsigned char)d[i]] != 4;
            count[t + 1] = c;
        };
        {
            std::vector<std::thread> th;
            for (unsigned t = 1; t < parts; ++t) th.emplace_back(pass1, t);
            pass1(0);
            for (auto& x : th) x.join();
        }
        for (unsigned t = 0; t < parts; ++t) count[t + 1] += count[t];
        const size_t len = count[parts];
        std::vector<uint8_t>& out = fa->packed[r];
        out.assign((len + 3) / 4 + 16, 0);
        fa->lengths[r] = (int64_t)len;
        auto pass2 = [&](unsigned t) {
            size_t k = count[t];
            const size_t k_end = count[t + 1];
            if (k == k_end) return;
            const size_t first_byte = k >> 2, last_byte = (k_end - 1) >> 2;
            uint8_t acc = 0;
            size_t cur_byte = first_byte;
            auto store = [&](size_t byte, uint8_t v) {
                if (byte == first_byte || byte == last_byte) __atomic_fetch_or(&out[byte], v, __ATOMIC_RELAXED);  // may be shared with a neighbour chunk
                else out[byte] = v;
            };
            for (size_t i = bounds(t), e = bounds(t + 1); i < e; ++i) {
                const uint8_t code = lut[(unsigned char)d[i]];
                if (code == 4) continue;
                const size_t byte = k >> 2;
                if (byte != cur_byte) { store(cur_byte, acc); acc = 0; cur_byte = byte; }
                acc |= (uint8_t)(code << ((k & 3) * 2));
                ++k;
            }
            store(cur_byte, acc);
        };
        {
            std::vector<std::thread> th;
            for (unsigned t = 1; t < parts; ++t) th.emplace_back(pass2, t);
            pass2(0);
            for (auto& x : th) x.join();
        }
    }
    if (map) munmap(map, n);
    return fa;
}
extern "C" int64_t bqc_fasta_contig(bqc_fasta* f, const char* name, const uint8_t** packed) {
    for (size_t i = 0; i < f->names.size(); ++i)
        if (f->names[i] == name) {
            *packed = f->packed[i].data();
            return f->lengths[i];
        }
    return -1;
}
extern "C" void bqc_fasta_close(bqc_fasta* f) { delete f; }

// ------------------------------------------------------------------------------------------------
// `.bamqc` writer  (src/bamqualcheck.cpp:130-233, src/OverallNumbers.hpp:170-216, src/TripletCounting.hpp:271-301)
// ------------------------------------------------------------------------------------------------
namespace {
struct Table {
    std::vector<uint64_t> v;
};
bool get_table(bqc_engine* e, int lane, int field, int sub, std::vector<uint64_t>& v) {
    uint64_t n = 0;
    if (bqc_result_table(e, lane, field, sub, nullptr, 0, &n)) return false;
    v.assign(n, 0);
    return bqc_result_table(e, lane, field, sub, v.data(), n, nullptr) == 0;
}
void print_u32(std::ostream& o, const std::vector<uint64_t>& v) {  // String<unsigned>
    for (uint64_t x : v) o << " " << (unsigned)x;
    o << std::endl;
}
void print_u64(std::ostream& o, const std::vector<uint64_t>& v) {  // String<uint64_t>
    for (uint64_t x : v) o << " " << x;
    o << std::endl;
}
}  // namespace

extern "C" int bqc_write_bamqc(bqc_engine* e, const char* sample_id, const char* path) {
    std::ofstream out(path, std::ios::out | std::ios::binary);
    if (!out.good()) return BQC_ERR_ARG;
    // lanes in std::map<CharString> key order (src/bamqualcheck.cpp:163)
    int n_lanes = bqc_n_lanes(e);
    std::map<std::string, int> order;
    for (int l = 0; l < n_lanes; ++l) order[bqc_lane_id(e, l)] = l;  // duplicates collapse like the reference map
    uint32_t n_q = 0, n_k = 0;
    const int32_t* klist = nullptr;
    const uint64_t* qlist = nullptr;
    bqc_qk_lists(e, &klist, &n_k, &qlist, &n_q);

    for (auto& kv : order) {
        int lane = kv.second;
        std::vector<uint64_t> sc, t;
        if (!get_table(e, lane, BQC_F_SCALARS, 0, sc)) return BQC_ERR_ARG;
        out << "sample_id " << sample_id << std::endl;
        out << "lane " << kv.first << std::endl;
        out << "total_read_pairs " << (unsigned)sc[4] / 2 << std::endl;
        out << "total_bps " << sc[5] << std::endl;
        out << "supplementary_alignments " << (unsigned)sc[0] << std::endl;
        out << "marked_duplicate " << (unsigned)sc[1] << std::endl;
        out << "QC_failed " << (unsigned)sc[2] << std::endl;
        out << "not_primary_alignment " << (unsigned)sc[3] << std::endl;
        out << "both_reads_unmapped " << (unsigned)sc[6] << std::endl;
        out << "first_read_unmapped " << (unsigned)sc[7] << std::endl;
        out << "second_read_unmapped " << (unsigned)sc[8] << std::endl;
        out << "first_and_or_second_read_mapped " << (unsigned)sc[9] << std::endl;
        out << "FF_RR_oriented_pairs " << (unsigned)sc[10] << std::endl;
        out << "total_proper_pairs " << (unsigned)sc[11] << std::endl;
        out << "total_proper_pairs_autosome " << (unsigned)sc[12] << std::endl;
        get_table(e, lane, BQC_F_POSCOV, 0, t);
        out << "genome_coverage_histogram"; print_u32(out, t);
        get_table(e, lane, BQC_F_INSERT, 0, t);
        out << "insert_size_histogram"; print_u32(out, t);
        struct { const char* name; int field; bool wide; } hists[] = {
            {"read_length_histogram", BQC_F_READLEN_M, false}, {"N_count_histogram", BQC_F_NCOUNT_M, false},
            {"GC_content_histogram", BQC_F_GCCOUNT_M, true},   {"average_base_qual_histogram", BQC_F_AVGQUAL_M, false},
            {"mapping_qual_histogram", BQC_F_MAPQ_M, false},   {"mismatch_count_histogram", BQC_F_MISMATCH_M, false},
            {"deletion_count_histogram", BQC_F_DEL_M, false},  {"insertion_count_histogram", BQC_F_INS_M, false},
            {"Ns_by_position", BQC_F_DNA_N_M, true},           {"As_by_position", BQC_F_DNA_A_M, true},
            {"Cs_by_position", BQC_F_DNA_C_M, true},           {"Gs_by_position", BQC_F_DNA_G_M, true},
            {"Ts_by_position", BQC_F_DNA_T_M, true}};
        for (auto& h : hists)
            for (int m = 0; m < 2; ++m) {
                get_table(e, lane, h.field, m, t);
                out << h.name << (m ? "_second" : "_first");
                if (h.wide) print_u64(out, t);
                else print_u32(out, t);
            }
        for (int m = 0; m < 2; ++m) {
            uint64_t n = 0;
            bqc_result_avgqual(e, lane, m, nullptr, 0, &n);
            std::vector<double> aq(n);
            bqc_result_avgqual(e, lane, m, aq.data(), n, nullptr);
            out << "average_base_qual_by_position" << (m ? "_second" : "_first");
            for (double x : aq) out << " " << x;
            out << std::endl;
        }
        for (int m = 0; m < 2; ++m) {
            get_table(e, lane, BQC_F_SC5_M, m, t);
            out << "soft_clipping_5_prime_by_position" << (m ? "_second" : "_first"); print_u32(out, t);
            get_table(e, lane, BQC_F_SC3_M, m, t);
            out << "soft_clipping_3_prime_by_position" << (m ? "_second" : "_first"); print_u32(out, t);
        }
        // ten_most_abundant_kmers: top 10 counts descending, equal counts by ascending table index
        std::vector<uint64_t> em;
        get_table(e, lane, BQC_F_EIGHTMER, 0, em);
        {
            std::vector<uint64_t> v(em);
            std::partial_sort(v.begin(), v.begin() + 10, v.end(), std::greater<uint64_t>());
            std::set<int> used;
            for (int i = 0; i < 10; ++i) {
                int pos = (int)(std::find(em.begin(), em.end(), v[i]) - em.begin());
                while (used.count(pos)) pos = (int)(std::find(em.begin() + pos + 1, em.end(), v[i]) - em.begin());
                used.insert(pos);
                char kmer[9];
                for (int b = 0; b < 8; ++b) kmer[b] = "ACGT"[(pos >> (2 * (7 - b))) & 3];
                kmer[8] = 0;
                out << "nr_" << i + 1 << "_most_abundant_8mer " << kmer << " " << v[i] << std::endl;
            }
        }
        out << "8mer_count"; print_u64(out, em);
        for (uint32_t i = 0; i < n_q; ++i)
            for (uint32_t j = 0; j < n_k; ++j) {
                uint64_t est[4];
                if (bqc_result_estimates(e, lane, (int)(i * n_k + j), est)) return BQC_ERR_ARG;
                out << klist[j] << "mer_count_after_qual_clipping_" << qlist[i] << " " << est[0] << std::endl;
                out << "distinct_" << klist[j] << "mer_count_after_qual_clipping_" << qlist[i] << " " << est[1] << std::endl;
                out << "unique_" << klist[j] << "mer_count_after_qual_clipping_" << qlist[i] << " " << est[2] << std::endl;
                out << klist[j] << "mer_F2_after_qual_clipping_" << qlist[i] << " " << est[3] << std::endl;
            }
        std::vector<uint64_t> tr;
        get_table(e, lane, BQC_F_TRIPLET, 0, tr);
        const char bases[] = {'A', 'C', 'G', 'T'};
        const struct { const char* suffix; int grp; } groups[] = {{"_1st_FW", 0}, {"_1st_RC", 2}, {"_2nd_FW", 1}, {"_2nd_RC", 3}};
        for (int b = 0; b < 4; ++b)
            for (auto& g : groups) {
                out << "triplet_counts_" << bases[b] << g.suffix;
                for (int ctx = 0; ctx < 64; ++ctx) out << " " << tr[(size_t)ctx * 16 + g.grp * 4 + b];
                out << std::endl;
            }
    }
    return out.good() ? 0 : BQC_ERR_ARG;
}

// ------------------------------------------------------------------------------------------------
// bamqualcheck command line
// ------------------------------------------------------------------------------------------------
namespace {
struct Cli {
    std::string bam, ref = "genome.fa", out;
    std::string chroms =
        "chr1,chr2,chr3,chr4,chr5,chr6,chr7,chr8,chr9,chr10,chr11,chr12,chr13,chr14,chr15,chr16,"
        "chr17,chr18,chr19,chr20,chr21,chr22";
    std::vector<int32_t> klist;
    std::vector<uint64_t> qlist;
    double e = 0.01;
    int seed = 1, isize = 1000, threads = 0, max_read_len = 0;
    std::vector<int> devices = {0};
    uint64_t staging_mb = 0;
    bool timing = false;
};
}  // namespace

// ------------------------------------------------------------------------------------------------
// the command: helpers shared by the SAM and the file path
// ------------------------------------------------------------------------------------------------
namespace {
typedef std::chrono::steady_clock::time_point TimePoint;

bool probe_output(const Cli& c) {
    std::ofstream probe(c.out.c_str(), std::ios::out | std::ios::binary);
    if (!probe.good()) {
        std::cerr << "ERROR: Could not open output file " << c.out << '\n';
        return false;
    }
    return true;
}

int report_submit_error(bqc_engine* eng, const Cli& c) {
    bqc_error_info ei;
    bqc_get_error(eng, &ei);
    if (ei.code == BQC_ERR_BAD_RECORD) std::cerr << "ERROR: Could not read record from BAM File " << c.bam << "\n";
    else std::cerr << "ERROR: " << bqc_last_error(eng) << std::endl;
    return 1;
}

// the reference's messages for the fatal records (src/bamqualcheck.cpp:91,308,387; src/TripletCounting.hpp:116-127)
int report_finish_error(bqc_engine* eng, const Cli& c) {
    bqc_error_info ei;
    bqc_get_error(eng, &ei);
    if (ei.code == BQC_ERR_RG_NOT_Z) std::cout << "Read does not have Z" << "\n";
    else if (ei.code == BQC_ERR_BAD_RECORD) std::cerr << "ERROR: Could not read record from BAM File " << c.bam << "\n";
    else if (ei.code == BQC_ERR_NO_MATE_FLAG) std::cerr << "ERROR: No first or second flag in read in:  " << c.bam << "\n";
    else std::cerr << (ei.code ? ei.message : bqc_last_error(eng)) << std::endl;
    return ei.code ? ei.code : 1;
}

bqc_engine* make_engine(const Cli& c, const bqc_bam_header& hdr, int device, std::vector<uint8_t>& main_chrom) {
    main_chrom.assign((size_t)std::max(1, hdr.n_ref), 0);
    {   // initChroms (src/bamqualcheck.cpp:106-123): the -c names that exist in the BAM header
        std::istringstream cs(c.chroms);
        std::string name;
        while (std::getline(cs, name, ','))
            for (int i = 0; i < hdr.n_ref; ++i)
                if (name == hdr.ref_names[i]) { main_chrom[i] = 1; break; }
    }
    if (hdr.n_lanes == 0) {
        std::cerr << "ERROR: BAM header declares no read group (@RG); bamqualcheck needs at least one.\n";
        return nullptr;
    }
    bqc_config cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.device = device;
    cfg.isize = c.isize;
    cfg.n_lanes = hdr.n_lanes;
    cfg.lane_ids = hdr.lane_ids;
    cfg.n_ref = hdr.n_ref;
    cfg.main_chrom = main_chrom.data();
    cfg.n_k = (int32_t)c.klist.size();
    cfg.klist = c.klist.data();
    cfg.n_q = (int32_t)c.qlist.size();
    cfg.q_cutoff = c.qlist.data();
    cfg.q_base = 33;
    cfg.e = c.e;
    cfg.seed = c.seed;
    cfg.max_read_len = c.max_read_len;
    cfg.staging_bytes = c.staging_mb << 20;
    cfg.host_threads = c.threads;
    bqc_engine* eng = nullptr;
    if (bqc_create(&cfg, &eng)) {
        std::cerr << "ERROR: " << bqc_last_error(nullptr) << std::endl;
        return nullptr;
    }
    return eng;
}

// reference genome: every BAM reference that the FASTA holds goes to HBM
bool load_reference(bqc_engine* eng, bqc_fasta* fa, const bqc_bam_header& hdr) {
    for (int i = 0; i < hdr.n_ref; ++i) {
        const uint8_t* packed = nullptr;
        int64_t len = bqc_fasta_contig(fa, hdr.ref_names[i], &packed);
        if (len >= 0 && bqc_set_reference(eng, i, packed, (uint64_t)len)) {
            std::cerr << "ERROR: " << bqc_last_error(eng) << std::endl;
            return false;
        }
    }
    return true;
}

// ---- streaming file input ----------------------------------------------------------------------------------
struct RangeReader {  // sequential pread over [pos, end) of a file (end == ~0: to the end of the file / pipe)
    int fd = -1;
    bool seekable = true;
    uint64_t pos = 0, end = ~0ull;
    size_t read(uint8_t* buf, size_t n) {
        size_t got = 0;
        while (got < n && pos < end) {
            const size_t want = (size_t)std::min<uint64_t>(n - got, end - pos);
            const ssize_t r = seekable ? pread(fd, buf + got, want, (off_t)pos) : ::read(fd, buf + got, want);
            if (r <= 0) break;
            got += (size_t)r;
            pos += (uint64_t)r;
        }
        return got;
    }
};

// whole BGZF blocks at the front of buf[0..n): bytes and inflated size, stopping before `max_out` inflated bytes are
// exceeded; bad = not a BGZF block header (SAM/BAM specification 4.1)
size_t bgzf_whole_prefix(const uint8_t* buf, size_t n, uint64_t max_out, uint64_t& inflated, bool& bad) {
    size_t p = 0;
    inflated = 0;
    bad = false;
    while (p + 18 <= n) {
        if (buf[p] != 0x1f || buf[p + 1] != 0x8b || buf[p + 2] != 8 || !(buf[p + 3] & 4)) { bad = true; break; }
        const uint32_t xlen = buf[p + 10] | (buf[p + 11] << 8);
        if (p + 12 + xlen > n) break;
        size_t x = p + 12, xend = x + xlen;
        int bsize = -1;
        while (x + 4 <= xend) {
            const uint32_t slen = buf[x + 2] | (buf[x + 3] << 8);
            if (buf[x] == 'B' && buf[x + 1] == 'C' && slen == 2 && x + 6 <= xend) bsize = buf[x + 4] | (buf[x + 5] << 8);
            x += 4 + slen;
        }
        if (bsize < 0) { bad = true; break; }
        const size_t blen = (size_t)bsize + 1;
        if (p + blen > n) break;
        uint32_t isize;
        memcpy(&isize, buf + p + blen - 4, 4);
        if (isize > 65536u) { bad = true; break; }
        if (inflated + isize > max_out) break;
        inflated += isize;
        p += blen;
    }
    return p;
}

// A BGZF block boundary at or after `from`: the 16-byte member header with the BC subfield, confirmed by three hops.
// Returns ~0 if none is found within 1 MiB (then the file is not cut there).
uint64_t find_bgzf_block(int fd, uint64_t from, uint64_t file_size) {
    std::vector<uint8_t> buf((size_t)std::min<uint64_t>(file_size - from, (1u << 20) + (4u << 16)));
    RangeReader rr;
    rr.fd = fd; rr.pos = from; rr.end = file_size;
    const size_t n = rr.read(buf.data(), buf.size());
    for (size_t p = 0; p + 18 <= n && p < (1u << 20); ++p) {
        size_t q = p;
        int hops = 0;
        while (hops < 4 && q + 18 <= n) {
            if (!(buf[q] == 0x1f && buf[q + 1] == 0x8b && buf[q + 2] == 8 && buf[q + 3] == 4 && buf[q + 10] == 6 && buf[q + 11] == 0 && buf[q + 12] == 'B' &&
                  buf[q + 13] == 'C' && buf[q + 14] == 2 && buf[q + 15] == 0))
                break;
            q += (size_t)(buf[q + 16] | (buf[q + 17] << 8)) + 1;
            ++hops;
        }
        if (hops == 4 || (hops >= 1 && from + q == file_size)) return from + p;
    }
    return ~0ull;
}

struct Piece {  // one engine and the byte range of the file it reads
    bqc_engine* eng = nullptr;
    std::vector<uint8_t> main_chrom;
    uint64_t beg = 0, end = 0;
    size_t skip = 0;           // piece 0: inflated bytes of the BAM header in its first block
    std::atomic<int> rc{0};
    Piece() {}
    Piece(const Piece&) {}
};

// Piece k of a BGZF file: whole blocks go to the device as they are.  Pieces after the first begin inside a record:
// the engine finds the first record boundary, the bytes in front of it are inflated here and handed to the piece
// before (get_head), whose last record they complete.
int stream_bgzf_piece(const Cli& c, int fd, Piece& P, bool unknown_start, bool is_last, const std::function<bool(std::vector<uint8_t>&)>& get_next_head) {
    bqc_engine* eng = P.eng;
    if (unknown_start && bqc_stream_unknown_start(eng)) return report_submit_error(eng, c);
    RangeReader rr;
    rr.fd = fd; rr.pos = P.beg; rr.end = P.end;
    std::vector<uint8_t> carry;
    size_t skip = P.skip;
    bool eof = false, any = false;
    while (!eof || !carry.empty() || !any) {
        void* pin;
        size_t cap;
        if (bqc_acquire_staging(eng, &pin, &cap)) return report_submit_error(eng, c);
        uint8_t* buf = (uint8_t*)pin;
        size_t filled = carry.size();
        memcpy(buf, carry.data(), filled);
        carry.clear();
        const size_t target = std::max<size_t>(1u << 20, cap / 4);   // ~4x compression: the inflated bytes have to fit the same buffer
        if (!eof && filled < target) {
            const size_t got = rr.read(buf + filled, target - filled);
            if (got < target - filled) eof = true;
            filled += got;
        }
        uint64_t inflated = 0;
        bool bad = false;
        const size_t used = bgzf_whole_prefix(buf, filled, cap, inflated, bad);
        if (bad || (used == 0 && filled > 0 && (eof || filled >= target))) {
            std::cerr << "ERROR: Could not read record from BAM File " << c.bam << "\n";
            return 1;
        }
        carry.assign(buf + used, buf + filled);
        const bool final_chunk = eof && carry.empty();
        if (used || final_chunk) {
            if (bqc_submit_bgzf(eng, buf, used, skip, (final_chunk && is_last) ? 1 : 0)) return report_submit_error(eng, c);
            skip = 0;
            any = true;
        }
        if (final_chunk) break;
    }
    if (!is_last) {  // the end of this piece's last record lies in the next piece
        std::vector<uint8_t> head;
        if (!get_next_head(head)) return 1;
        if (bqc_submit_stream(eng, head.empty() ? nullptr : head.data(), head.size(), 1)) return report_submit_error(eng, c);
    }
    return 0;
}

// the first `want` inflated bytes of the BGZF stream that starts at file offset `from`
bool inflate_head(int fd, uint64_t from, uint64_t file_size, uint64_t want, std::vector<uint8_t>& out) {
    out.clear();
    if (!want) return true;
    std::vector<uint8_t> buf((size_t)std::min<uint64_t>(file_size - from, want + (4u << 20)));
    RangeReader rr;
    rr.fd = fd; rr.pos = from; rr.end = file_size;
    const size_t n = rr.read(buf.data(), buf.size());
    std::vector<BgzfBlock> blocks;
    bool bad = false;
    bgzf_index(buf.data(), n, blocks, ~0ull, bad);
    if (bad || blocks.empty()) return false;
    size_t nb = 0;
    while (nb < blocks.size() && blocks[nb].obeg < want) ++nb;
    blocks.resize(nb);
    if (blocks.empty() || blocks.back().obeg + blocks.back().isize < want) return false;
    out.resize((size_t)(blocks.back().obeg + blocks.back().isize));
    if (!inflate_blocks(buf.data(), blocks, out.data(), 1)) return false;
    out.resize((size_t)want);
    return true;
}

int finish_and_write(const Cli& c, std::vector<Piece>& pieces, const bqc_bam_header& hdr, TimePoint t_start, TimePoint t_setup) {
    const int N = (int)pieces.size();
    for (Piece& P : pieces)
        if (bqc_finish(P.eng)) {
            bqc_error_info ei;
            bqc_get_error(P.eng, &ei);
            // a piece that does not end on a record boundary: the guessed start of the next piece was wrong (or the file is
            // damaged, which the single-stream pass then reports)
            if (N > 1 && ei.code == BQC_ERR_BAD_RECORD) return 2;
            report_finish_error(P.eng, c);
            return 1;
        }
    if (N > 1) {
        // the coverage windows across the cuts (include/bamqc_b200.h: bqc_cov_shard_*), one lane (read group) after the
        // other: each lane's records are a stream of their own; then everything is summed
        const int n_lanes = bqc_n_lanes(pieces[0].eng);
        std::vector<std::vector<int64_t>> delta((size_t)n_lanes, std::vector<int64_t>(101));
        for (int lane = 0; lane < n_lanes; ++lane) {
            std::vector<bqc_cov_shard> sh((size_t)N);
            for (int k = 0; k < N; ++k)
                if (bqc_cov_shard_boundary_lane(pieces[k].eng, lane, &sh[k])) return report_submit_error(pieces[k].eng, c);
            std::vector<int> have_prev(N, 0);
            std::vector<int32_t> prid(N, 0);
            std::vector<uint32_t> pb(N, 0);
            for (int k = 1; k < N; ++k) {
                have_prev[k] = have_prev[k - 1]; prid[k] = prid[k - 1]; pb[k] = pb[k - 1];
                if (sh[k - 1].n) { have_prev[k] = 1; prid[k] = sh[k - 1].last_rid; pb[k] = sh[k - 1].last_b; }
            }
            std::vector<std::vector<uint16_t>> fn((size_t)N, std::vector<uint16_t>(1002));
            for (int k = 0; k < N; ++k)
                if (bqc_cov_shard_function_lane(pieces[k].eng, lane, have_prev[k], prid[k], pb[k], fn[k].data())) return report_submit_error(pieces[k].eng, c);
            uint32_t p = 0;
            for (int k = 0; k < N; ++k) {
                if (bqc_cov_shard_run_lane(pieces[k].eng, lane, have_prev[k], prid[k], pb[k], p, &sh[k])) return report_submit_error(pieces[k].eng, c);
                if (sh[k].n) p = bqc_cov_apply(fn[k].data(), p);
            }
            bqc_cov_shards_combine(sh.data(), N, delta[lane].data());
        }
        for (int k = 1; k < N; ++k)
            if (bqc_merge_from(pieces[0].eng, pieces[k].eng)) return report_submit_error(pieces[0].eng, c);
        for (int lane = 0; lane < n_lanes; ++lane)
            if (bqc_poscov_adjust(pieces[0].eng, lane, delta[lane].data())) return report_submit_error(pieces[0].eng, c);
    }
    auto t_stats = std::chrono::steady_clock::now();
    if (bqc_write_bamqc(pieces[0].eng, hdr.sample_id, c.out.c_str())) {
        std::cerr << "ERROR: Could not open output file " << c.out << '\n';
        return 1;
    }
    auto t_end = std::chrono::steady_clock::now();
    if (c.timing) {
        auto sec = [](TimePoint a, TimePoint b) { return std::chrono::duration<double>(b - a).count(); };
        unsigned long long recs = 0;
        for (Piece& P : pieces) recs += bqc_records_seen(P.eng);
        fprintf(stderr, "BAMQC_TIMING records=%llu setup_s=%.4f stats_s=%.4f write_s=%.4f total_s=%.4f threads=%d devices=%d\n", recs, sec(t_start, t_setup), sec(t_setup, t_stats),
                sec(t_stats, t_end), sec(t_start, t_end), c.threads, N);
    }
    return 0;
}

// A .bam file (BGZF, or the raw uncompressed BAM stream the tests use): read in staging-sized pieces, never as a
// whole (src/bamqualcheck.cpp:303-306 streams too).  With several devices the file is cut into contiguous byte
// ranges at BGZF block boundaries, one engine per range, all reading concurrently.
int run_file(Cli& c, TimePoint t_start) {
    const int fd = open(c.bam.c_str(), O_RDONLY);
    if (fd < 0) {
        std::cerr << "ERROR: Could not open " << c.bam << " for reading.\n";
        return 1;
    }
    struct stat st;
    const bool seekable = fstat(fd, &st) == 0 && S_ISREG(st.st_mode);
    const uint64_t file_size = seekable ? (uint64_t)st.st_size : ~0ull;
    if (!probe_output(c)) { close(fd); return 1; }
    // ---- header: read (and inflate) a prefix large enough to hold it ------------------------------------
    std::vector<uint8_t> front;          // the first bytes of the file as read
    RangeReader rr;
    rr.fd = fd; rr.seekable = seekable; rr.end = file_size;
    auto grow_front = [&](size_t more) { const size_t o = front.size(); front.resize(o + more); front.resize(o + rr.read(front.data() + o, more)); return front.size() > o; };
    grow_front(1u << 20);
    const bool raw = front.size() >= 4 && memcmp(front.data(), "BAM\1", 4) == 0;
    bqc_bam_header hdr;
    size_t hdr_bytes = 0;
    std::vector<BgzfBlock> blocks;       // BGZF blocks of `front`
    std::vector<uint8_t> head;
    for (;;) {
        if (raw) hdr_bytes = bqc_parse_bam_header(front.data(), front.size(), &hdr);
        else {
            blocks.clear();
            bool bad = false;
            bgzf_index(front.data(), front.size(), blocks, ~0ull, bad);
            if (bad || (blocks.empty() && front.size() >= (1u << 17))) break;
            if (!blocks.empty()) {
                head.resize((size_t)(blocks.back().obeg + blocks.back().isize));
                if (!inflate_blocks(front.data(), blocks, head.data(), c.threads)) break;
                hdr_bytes = bqc_parse_bam_header(head.data(), head.size(), &hdr);
            }
        }
        if (hdr_bytes) break;
        if (!grow_front(std::max<size_t>(front.size(), 1u << 20))) break;   // the header did not fit: read on
    }
    if (!hdr_bytes) {
        std::cerr << "ERROR: Could not open " << c.bam << " for reading.\n";
        close(fd);
        return 1;
    }
    // ---- engines: one per device; with several, the record stream is cut into contiguous pieces -----------
    uint64_t rec_beg = 0;   // file offset of the first BGZF block that holds records
    size_t skip = 0;
    if (!raw) {
        size_t k = 0;
        while (k < blocks.size() && blocks[k].obeg + blocks[k].isize <= hdr_bytes) ++k;
        if (k < blocks.size()) { rec_beg = blocks[k].bbeg; skip = hdr_bytes - (size_t)blocks[k].obeg; }
        else { rec_beg = blocks.empty() ? 0 : blocks.back().bbeg + (blocks.back().cbeg - blocks.back().bbeg) + blocks.back().clen + 8; skip = 0; }
    }
    std::vector<int> devices = c.devices;
    if (raw || !seekable) devices.resize(1);   // pieces need BGZF block boundaries and device-side framing
    std::vector<uint64_t> cut(1, rec_beg);
    if (devices.size() > 1) {
        const uint64_t span = file_size - rec_beg;
        const size_t n = (size_t)std::min<uint64_t>(devices.size(), std::max<uint64_t>(1, span >> 22));   // at least 4 MB of file per piece
        for (size_t k = 1; k < n; ++k) {
            const uint64_t at = find_bgzf_block(fd, rec_beg + span * k / n, file_size);
            if (at != ~0ull && at > cut.back() && at < file_size) cut.push_back(at);
        }
        devices.resize(cut.size());
    }
    const int N = (int)devices.size();
    int rc = 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
        std::vector<Piece> pieces((size_t)(attempt ? 1 : N));
        const int M = (int)pieces.size();
        for (int k = 0; k < M && !rc; ++k) {
            pieces[k].eng = make_engine(c, hdr, devices[k], pieces[k].main_chrom);
            if (!pieces[k].eng) rc = 1;
            pieces[k].beg = k ? cut[k] : rec_beg;
            pieces[k].end = k + 1 < M ? cut[k + 1] : file_size;
        }
        bqc_fasta* fa = rc ? nullptr : bqc_fasta_open(c.ref.c_str());
        if (!rc && !fa) std::cerr << "ERROR: Could not open fasta file " << c.ref << std::endl;  // the reference continues too (:291)
        if (fa) {
            std::vector<std::thread> th;
            std::atomic<int> bad(0);
            for (int k = 0; k < M; ++k) th.emplace_back([&, k] { if (!load_reference(pieces[k].eng, fa, hdr)) bad = 1; });
            for (auto& t : th) t.join();
            bqc_fasta_close(fa);
            if (bad) rc = 1;
        }
        auto t_setup = std::chrono::steady_clock::now();
        if (!rc && raw) {
            // the uncompressed stream: the engine frames it on the device
            bqc_engine* eng = pieces[0].eng;
            std::vector<uint8_t> pending(front.begin() + (ptrdiff_t)hdr_bytes, front.end());
            bool eof = false, first = true;
            while ((!eof || !pending.empty() || first) && !rc) {
                first = false;
                void* pin;
                size_t cap;
                if (bqc_acquire_staging(eng, &pin, &cap)) { rc = report_submit_error(eng, c); break; }
                uint8_t* buf = (uint8_t*)pin;
                size_t filled = std::min(cap, pending.size());
                memcpy(buf, pending.data(), filled);
                pending.erase(pending.begin(), pending.begin() + (ptrdiff_t)filled);
                if (pending.empty() && !eof && filled < cap) {
                    const size_t got = rr.read(buf + filled, cap - filled);
                    if (got < cap - filled) eof = true;
                    filled += got;
                }
                if (bqc_submit_stream(eng, buf, filled, (eof && pending.empty()) ? 1 : 0)) rc = report_submit_error(eng, c);
            }
        } else if (!rc) {
            if (M > 1)
                for (int k = 0; k < M; ++k) bqc_cov_defer(pieces[k].eng, k == 0 ? 2 : 1);
            pieces[0].skip = skip;
            if (!seekable) {  // a pipe: what was read for the header is replayed from memory first
                // (single piece) the front bytes from rec_beg on are fed through a temporary reader below
            }
            std::vector<std::thread> th;
            std::vector<int> prc((size_t)M, 0);
            for (int k = 0; k < M; ++k)
                th.emplace_back([&, k] {
                    auto next_head = [&](std::vector<uint8_t>& out) -> bool {
                        uint64_t skipped = 0;
                        for (;;) {   // until piece k+1 has framed its first buffer
                            const int r = bqc_stream_skipped(pieces[k + 1].eng, &skipped);
                            if (r == 0) break;
                            if (r > 0 || pieces[k + 1].rc.load()) return false;
                            std::this_thread::sleep_for(std::chrono::milliseconds(1));
                        }
                        return inflate_head(fd, pieces[k + 1].beg, file_size, skipped, out);
                    };
                    prc[k] = seekable ? stream_bgzf_piece(c, fd, pieces[k], k > 0, k + 1 == M, next_head) : 0;
                    if (prc[k]) pieces[k].rc = 1;
                });
            for (auto& t : th) t.join();
            if (!seekable) {
                // BGZF from a pipe: the bytes already read (from the first record block on), then the rest of the pipe
                bqc_engine* eng = pieces[0].eng;
                std::vector<uint8_t> carry(front.begin() + (ptrdiff_t)rec_beg, front.end());
                size_t sk = skip;
                bool eof = false, any = false;
                while ((!eof || !carry.empty() || !any) && !rc) {
                    void* pin;
                    size_t cap;
                    if (bqc_acquire_staging(eng, &pin, &cap)) { rc = report_submit_error(eng, c); break; }
                    uint8_t* buf = (uint8_t*)pin;
                    const size_t target = std::max<size_t>(1u << 20, cap / 4);
                    size_t filled = std::min(carry.size(), target);
                    memcpy(buf, carry.data(), filled);
                    carry.erase(carry.begin(), carry.begin() + (ptrdiff_t)filled);
                    if (carry.empty() && !eof && filled < target) {
                        const size_t got = rr.read(buf + filled, target - filled);
                        if (got < target - filled) eof = true;
                        filled += got;
                    }
                    uint64_t inflated = 0;
                    bool bad = false;
                    const size_t used = bgzf_whole_prefix(buf, filled, cap, inflated, bad);
                    if (bad || (used == 0 && filled > 0 && eof && carry.empty())) { std::cerr << "ERROR: Could not read record from BAM File " << c.bam << "\n"; rc = 1; break; }
                    carry.insert(carry.begin(), buf + used, buf + filled);
                    const bool final_chunk = eof && carry.empty();
                    if (used || final_chunk) {
                        if (bqc_submit_bgzf(eng, buf, used, sk, final_chunk ? 1 : 0)) { rc = report_submit_error(eng, c); break; }
                        sk = 0;
                        any = true;
                    }
                    if (final_chunk) break;
                }
            }
            for (int k = 0; k < M; ++k)
                if (prc[k]) rc = 1;
        }
        if (!rc) rc = finish_and_write(c, pieces, hdr, t_start, t_setup);
        if (rc == 2 && attempt == 0) {  // a piece did not begin where its predecessor ended: one stream on one device
            std::cerr << "note: the file could not be cut at the guessed record boundaries; reading it as one stream\n";
            for (Piece& P : pieces) bqc_destroy(P.eng);
            rc = 0;
            continue;
        }
        if (rc == 2) rc = 1;
        for (Piece& P : pieces)
            if (P.eng) bqc_destroy(P.eng);
        break;
    }
    bqc_free_bam_header(&hdr);
    close(fd);
    return rc;
}
}  // namespace

extern "C" int bqc_main(int argc, const char* const* argv) {
    Cli c;
    std::string kmer = "32", qcut = "17";
    bool haveR = false, haveO = false;
    std::vector<std::string> positional;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto need = [&](const char* name) -> std::string {
            if (i + 1 >= argc) {
                std::cerr << "bamqualcheck: option requires an argument -- " << name << std::endl;
                exit(1);
            }
            return argv[++i];
        };
        if (a == "-h" || a == "--help") {
            std::cout << "bamqualcheck [OPTIONS] BAMFILE   (BAMFILE '-' reads SAM text from stdin)\n  -r, --reference FILENAME   Reference genome filename.\n"
                         "  -i, --insert-size INT      Upper bound for the insert size in insert size histogram. Default: 1000.\n"
                         "  -c, --chromosomes STRING   Comma separated list of the main chromosome names.\n"
                         "  -o, --output-file OUT      Output filename.\n  -k, --kmer-size STRING     Comma-separated list of k-mer sizes. Default: 32.\n"
                         "  -q, --quality-cutoff STRING Comma-separated list of PHRED quality thresholds. Default: 17.\n"
                         "  -e, --error-rate DOUBLE    Error rate guaranteed. Default: 0.01.\n  -s, --seed INT             Seed value for the randomness. Default: 1.\n"
                         "  --device INT | --devices LIST (e.g. 0-7: the BAM file is cut into one piece per GPU), --threads INT,\n"
                         "  --max-read-len INT, --staging-mb INT, --timing   (engine options)\n";
            return 0;
        }
        if (a == "--version") { std::cout << "bamqualcheck version: dev (bamqc-b200)\n"; return 0; }
        if (a == "-r" || a == "--reference") { c.ref = need("r"); haveR = true; }
        else if (a == "-i" || a == "--insert-size") c.isize = atoi(need("i").c_str());
        else if (a == "-c" || a == "--chromosomes") c.chroms = need("c");
        else if (a == "-o" || a == "--output-file") { c.out = need("o"); haveO = true; }
        else if (a == "-k" || a == "--kmer-size") kmer = need("k");
        else if (a == "-q" || a == "--quality-cutoff") qcut = need("q");
        else if (a == "-e" || a == "--error-rate") c.e = atof(need("e").c_str());
        else if (a == "-s" || a == "--seed") c.seed = atoi(need("s").c_str());
        else if (a == "--device") c.devices = {atoi(need("device").c_str())};
        else if (a == "--devices") {   // 0,1,2 or 0-7: the file is cut into one contiguous piece per device
            c.devices.clear();
            std::stringstream ds(need("devices"));
            std::string item;
            while (std::getline(ds, item, ',')) {
                const size_t dash = item.find('-');
                if (dash != std::string::npos && dash > 0) for (int d = atoi(item.substr(0, dash).c_str()); d <= atoi(item.substr(dash + 1).c_str()); ++d) c.devices.push_back(d);
                else if (!item.empty()) c.devices.push_back(atoi(item.c_str()));
            }
            if (c.devices.empty()) c.devices = {0};
        }
        else if (a == "--max-read-len") c.max_read_len = atoi(need("max-read-len").c_str());
        else if (a == "--staging-mb") c.staging_mb = (uint64_t)atoll(need("staging-mb").c_str());
        else if (a == "--threads") c.threads = atoi(need("threads").c_str());
        else if (a == "--timing") c.timing = true;
        else positional.push_back(a);
    }
    if (!haveR || !haveO || positional.size() != 1) {
        std::cerr << "bamqualcheck: options -r and -o and exactly one BAMFILE argument are required" << std::endl;
        return 1;
    }
    c.bam = positional[0];
    {   // src/CommandLineParser.hpp:121-141
        std::stringstream sq(qcut);
        size_t j;
        while (sq >> j) { c.qlist.push_back(j); if (sq.peek() == ',') sq.ignore(); }
        std::stringstream sk(kmer);
        int i;
        while (sk >> i) { c.klist.push_back(i); if (sk.peek() == ',') sk.ignore(); }
    }
    const bool sam = c.bam == "-";
    if (c.threads <= 0) c.threads = (int)std::max(1u, std::thread::hardware_concurrency());
    auto t_start = std::chrono::steady_clock::now();
    if (!sam) return run_file(c, t_start);
    // ---- SAM text on stdin (src/bamqualcheck.cpp:252-260): one device ------------------------------------
    // The header lines are read first; the alignment lines then go straight from read() into the staging buffers,
    // each cut at its last line end (the partial line is carried into the next buffer), and are encoded on the GPU.
    std::cerr << "Reading from stdin" << std::endl;  // src/CommandLineParser.hpp:96
    auto read_some = [](char* dst, size_t cap, bool& eof) -> size_t {
        for (;;) {
            const ssize_t r = read(0, dst, cap);
            if (r < 0 && errno == EINTR) continue;
            if (r <= 0) { eof = true; return 0; }
            return (size_t)r;
        }
    };
    std::vector<char> head;
    bool eof = false;
    for (size_t line = 0;;) {   // until the first line that does not start with '@' (or the end of the input)
        while (line < head.size() && head[line] == '@') {
            const char* q = (const char*)memchr(head.data() + line, '\n', head.size() - line);
            if (!q) break;
            line = (size_t)(q - head.data()) + 1;
        }
        if ((line < head.size() && head[line] != '@') || eof) break;
        const size_t at = head.size();
        head.resize(at + (1u << 20));
        head.resize(at + read_some(head.data() + at, 1u << 20, eof));
    }
    if (!probe_output(c)) return 1;
    bqc_bam_header hdr;
    size_t consumed = 0;
    if (bqc_parse_sam_header(head.data(), head.size(), &hdr, &consumed)) {
        std::cerr << "ERROR: Could not open " << c.bam << " for reading.\n";
        return 1;
    }
    std::vector<uint8_t> main_chrom;
    bqc_engine* eng = make_engine(c, hdr, c.devices[0], main_chrom);
    if (!eng) return 1;
    if (bqc_set_ref_names(eng, hdr.n_ref, hdr.ref_names)) { std::cerr << "ERROR: " << bqc_last_error(eng) << std::endl; return 1; }
    bqc_fasta* fa = bqc_fasta_open(c.ref.c_str());
    if (!fa) std::cerr << "ERROR: Could not open fasta file " << c.ref << std::endl;  // the reference continues too (:291)
    if (fa && !load_reference(eng, fa, hdr)) return 1;
    auto t_setup = std::chrono::steady_clock::now();
    int rc = 0;
    {
        std::vector<char> carry(head.begin() + (ptrdiff_t)consumed, head.end());
        head = std::vector<char>();
        while (!rc) {
            void* pin;
            size_t cap;
            if (bqc_acquire_staging(eng, &pin, &cap)) { rc = 1; break; }
            char* buf = (char*)pin;
            if (carry.size() > cap) { std::cerr << "ERROR: SAM record larger than the staging buffer\n"; rc = 1; break; }
            memcpy(buf, carry.data(), carry.size());
            size_t filled = carry.size();
            while (filled < cap && !eof) filled += read_some(buf + filled, cap - filled, eof);
            size_t cut = filled;
            if (!eof) {
                while (cut > 0 && buf[cut - 1] != '\n') --cut;
                if (cut == 0) { std::cerr << "ERROR: SAM record larger than the staging buffer\n"; rc = 1; break; }
            }
            carry.assign(buf + cut, buf + filled);
            if (bqc_submit_sam(eng, buf, cut, eof ? 1 : 0)) {
                bqc_sync(eng);   // the device's error word is final once the work in flight has run
                report_finish_error(eng, c);
                rc = 1;
            }
            if (eof) break;
        }
    }
    if (!rc && bqc_finish(eng)) { bqc_sync(eng); report_finish_error(eng, c); rc = 1; }
    auto t_stats = std::chrono::steady_clock::now();
    if (!rc && bqc_write_bamqc(eng, hdr.sample_id, c.out.c_str())) {
        std::cerr << "ERROR: Could not open output file " << c.out << '\n';
        rc = 1;
    }
    auto t_end = std::chrono::steady_clock::now();
    if (c.timing) {
        auto sec = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
        fprintf(stderr, "BAMQC_TIMING records=%llu setup_s=%.4f stats_s=%.4f write_s=%.4f total_s=%.4f threads=%d devices=1 sam_host_lines=%llu\n", (unsigned long long)bqc_records_seen(eng), sec(t_start, t_setup), sec(t_setup, t_stats), sec(t_stats, t_end), sec(t_start, t_end), c.threads, (unsigned long long)bqc_sam_host_lines(eng));
    }
    if (fa) bqc_fasta_close(fa);
    bqc_destroy(eng);
    bqc_free_bam_header(&hdr);
    return rc;
}
