// CPU check of the device SAM grammar (bamqc_b200/csrc/sam_parse.h) against the host encoder (sam_text.h) on random,
// deliberately odd alignment lines: every line the fast path accepts must encode byte for byte like sam_line_to_bam,
// so every line the host would encode differently, or reject, must be refused by the fast path.
//
//   sam_selftest N            N random lines (plus the fixed boundary cases); prints "<k> mismatching"
//   sam_selftest --time FILE  the host encoder's rate on the alignment lines of a SAM file, one thread
//   sam_selftest --emit FILE N  the lines of the N-line run that the fast path accepts, one per line (for the device
//                             encoder's check against the host encoder; @SQ names: kNames)
#include <chrono>
#include <cstdio>
#include <fstream>
#include <random>

#include "../bamqc_b200/csrc/sam_text.h"
#include "../bamqc_b200/csrc/sam_parse.h"

using bqc::SamRefs;

static std::mt19937_64 rng(12345);
static uint64_t rnd(uint64_t n) { return rng() % n; }
static bool coin(int pct) { return (int)rnd(100) < pct; }

static const char* kInts[] = {"-2147483649", "-2147483648", "-32769", "-32768", "-129", "-128", "-1", "-0", "0", "1", "127", "128", "255", "256",
                              "65535", "65536", "2147483647", "2147483648", "4294967295", "4294967296", "999999999", "1000000000",
                              "123456789012345678", "1234567890123456789", "12345678901234567890", "-123456789012345678", "+5", "007",
                              " 5", "5 ", "", "-", "5x", "0x10", "42"};
static const char* kFloats[] = {"1e22", "1e23", "-0", "0", "0.1", "0.3333333333333333", "0.333333333333333", "nan", "NaN", "inf", "-inf",
                                "0x1p3", "1.5x", "1.5", "-2.25e-5", "123456789012345", "1234567890123456", "1e-22", "1e-23", "5.", ".5",
                                ".", "1E5", "1e+05", "1e", "1e-", "", "-", "+1", " 1", "3.4028235e38", "1e-45", "0.000000000000000000001",
                                "100000000000000000000", "0e999", "12.5e-3", "1.000000000000001"};
static const char* kNames[] = {"chr1", "chr2", "chr10", "chrX", "chr1", "c", "chr1_alt", "chr", "HLA-A*01:01", "chrM"};
static const char* kRnames[] = {"*", "=", "chr1", "chr2", "chr10", "chrX", "c", "chr1_alt", "chr", "chrY", "chr1 ", "HLA-A*01:01", "", "chrM", "=="};

static std::string printable(size_t n, bool tabs_ok = false) {
    std::string s;
    for (size_t i = 0; i < n; ++i) {
        char c = (char)(0x20 + rnd(95));
        if (tabs_ok && coin(1)) c = '\t';
        s += c;
    }
    return s;
}
static std::string pick_int() {
    if (coin(70)) return kInts[rnd(sizeof(kInts) / sizeof(kInts[0]))];
    std::string s = coin(30) ? "-" : "";
    const size_t nd = 1 + rnd(20);
    for (size_t i = 0; i < nd; ++i) s += (char)('0' + rnd(10));
    return s;
}
static std::string pick_float() {
    if (coin(50)) return kFloats[rnd(sizeof(kFloats) / sizeof(kFloats[0]))];
    std::string s = coin(30) ? "-" : "";
    const size_t nd = 1 + rnd(18), dot = rnd(nd + 2);
    for (size_t i = 0; i < nd; ++i) {
        if (i == dot) s += '.';
        s += (char)('0' + rnd(10));
    }
    if (coin(50)) s += (coin(50) ? "e" : "E") + std::string(coin(30) ? "-" : coin(20) ? "+" : "") + std::to_string(rnd(40));
    return s;
}
static std::string pick_cigar(size_t lseq) {
    const int r = (int)rnd(100);
    if (r < 10) return "*";
    if (r < 15) { const char* bad[] = {"5", "M", "5Q", "5m", "0M", "1234567890M", "12345678901M", "5M5", "", "5M*"}; return bad[rnd(10)]; }
    std::string s;
    const char* ops = "MIDNSHP=X";
    size_t n = 1 + rnd(6);
    for (size_t i = 0; i < n; ++i) s += std::to_string(coin(90) ? 1 + rnd(lseq + 1) : rnd(4000000000ull)) + ops[rnd(9)];
    return s;
}
static std::string pick_seq(size_t& lseq) {
    if (coin(5)) { lseq = 0; return "*"; }
    lseq = coin(5) ? 1 + rnd(3) : 20 + rnd(300);
    const char* al = coin(80) ? "ACGT" : "ACGTNacgtn.=*XRYKMbdhv";
    const size_t na = strlen(al);
    std::string s;
    for (size_t i = 0; i < lseq; ++i) s += al[rnd(na)];
    return s;
}
static std::string pick_tag() {
    const char* tg[] = {"RG", "AS", "NM", "XS", "MD", "zz", "a1", "X"};
    std::string t = coin(95) ? tg[rnd(7)] : tg[7];
    const int r = (int)rnd(100);
    if (r < 10) return t + ":A:" + (coin(80) ? std::string(1, (char)('!' + rnd(90))) : coin(50) ? "" : "ab");
    if (r < 40) return t + ":i:" + pick_int();
    if (r < 55) return t + ":f:" + pick_float();
    if (r < 75) return t + ":Z:" + printable(rnd(40));
    if (r < 80) return t + ":H:" + printable(rnd(10));
    if (r < 90) {
        const char* sub = "cCsSiIfx";
        std::string s = t + ":B:" + sub[rnd(8)];
        const size_t n = rnd(6);
        for (size_t i = 0; i < n; ++i) s += "," + (coin(10) ? std::string() : coin(50) ? pick_int() : pick_float());
        if (coin(10)) s += ",,";
        return s;
    }
    const char* bad[] = {"XX:Q:5", "XX:i", "X:i:5", "XXi:5", "XX:i:", "XX:f:", "XX", "XX:Z", "", "XX::5"};
    return bad[rnd(10)];
}

static std::string make_line() {
    std::vector<std::string> f;
    const int qn = (int)rnd(100);
    f.push_back(qn < 2 ? printable(254) : qn < 4 ? printable(255) : qn < 5 ? "" : "read" + std::to_string(rnd(1000000)) + printable(rnd(20)));
    for (char& c : f.back()) if (c == '\t') c = '_';
    f.push_back(coin(85) ? std::to_string(rnd(4096)) : pick_int());
    f.push_back(kRnames[rnd(sizeof(kRnames) / sizeof(kRnames[0]))]);
    f.push_back(coin(80) ? std::to_string(rnd(250000000)) : pick_int());
    f.push_back(coin(85) ? std::to_string(rnd(61)) : pick_int());
    size_t lseq = 0;
    std::string seq = pick_seq(lseq);
    f.push_back(pick_cigar(lseq));
    f.push_back(kRnames[rnd(sizeof(kRnames) / sizeof(kRnames[0]))]);
    f.push_back(coin(80) ? std::to_string(rnd(250000000)) : pick_int());
    f.push_back(coin(80) ? std::to_string((int64_t)rnd(2000) - 1000) : pick_int());
    f.push_back(seq);
    const int qr = (int)rnd(100);
    std::string qual;
    if (qr < 10) qual = "*";
    else if (qr < 15) qual = printable(lseq + 1 + rnd(3));
    else if (qr < 17 && lseq) qual = printable(lseq - 1);
    else { for (size_t i = 0; i < lseq; ++i) qual += (char)('!' + rnd(94)); }
    if (qual.empty() && coin(50)) qual = "*";
    f.push_back(qual);
    const size_t nt = coin(70) ? 1 + rnd(6) : 0;
    for (size_t i = 0; i < nt; ++i) f.push_back(pick_tag());
    if (coin(2) && f.size() > 1) f.resize(1 + rnd(f.size() - 1));   // fewer fields
    std::string line;
    for (size_t i = 0; i < f.size(); ++i) line += (i ? "\t" : "") + f[i];
    const int m = (int)rnd(1000);
    if (m < 10) line += '\t';                                   // trailing TAB
    else if (m < 20) line += '\r';                              // CRLF
    else if (m < 25) line[rnd(line.size())] = (char)(0x80 + rnd(128));
    else if (m < 30) line[rnd(line.size())] = '\0';
    else if (m < 35) line[rnd(line.size())] = '\r';
    else if (m < 37) line.insert(rnd(line.size()), 1, ' ');
    else if (m < 39) line = coin(50) ? "" : "\r";
    return line;
}

static std::string cigar_line(size_t nops) {
    std::string cig;
    for (size_t i = 0; i < nops; ++i) cig += "1M";
    return "big\t0\tchr1\t100\t60\t" + cig + "\t=\t100\t0\tACGT\tIIII\tAS:i:5";
}

int main(int argc, char** argv) {
    std::vector<std::string> names(kNames, kNames + sizeof(kNames) / sizeof(kNames[0]));
    std::map<std::string, int32_t> ref_id;
    for (size_t i = 0; i < names.size(); ++i) ref_id.insert({names[i], (int32_t)i});
    std::string blob;
    std::vector<uint32_t> off;
    std::vector<int32_t> id;
    sam_refs_build(names, blob, off, id);
    const SamRefs R = {blob.data(), off.data(), id.data(), (int32_t)id.size()};

    if (argc == 3 && std::string(argv[1]) == "--time") {
        std::ifstream in(argv[2], std::ios::binary);
        std::vector<std::string> lines;
        std::string line;
        uint64_t bytes = 0;
        std::vector<std::string> sq;   // the file's @SQ names
        while (std::getline(in, line)) {
            if (line.empty() || line[0] != '@') { bytes += line.size() + 1; lines.push_back(line); }
            else if (line.compare(0, 3, "@SQ") == 0)
                for (const std::string& f : split_tabs(line))
                    if (f.compare(0, 3, "SN:") == 0) sq.push_back(f.substr(3));
        }
        ref_id.clear();
        for (size_t i = 0; i < sq.size(); ++i) ref_id.insert({sq[i], (int32_t)i});
        std::vector<uint8_t> enc;
        enc.reserve(bytes * 2);
        const auto t0 = std::chrono::steady_clock::now();
        for (std::string& l : lines) {
            if (!l.empty() && l.back() == '\r') l.pop_back();
            if (!l.empty() && !sam_line_to_bam(l, ref_id, enc)) { printf("rejected line\n"); return 1; }
        }
        const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        printf("{\"lines\": %zu, \"text_bytes\": %llu, \"seconds\": %.4f, \"mlines_per_s\": %.4f, \"mb_per_s\": %.2f}\n", lines.size(),
               (unsigned long long)bytes, s, lines.size() / s / 1e6, bytes / s / 1e6);
        return 0;
    }

    const bool emit = argc == 4 && std::string(argv[1]) == "--emit";
    FILE* ef = emit ? fopen(argv[2], "wb") : nullptr;
    if (emit && !ef) return 1;
    const uint64_t n = strtoull(argc > 1 ? argv[emit ? 3 : 1] : "200000", nullptr, 10);
    std::vector<std::string> lines;
    for (size_t k : {65534, 65535, 65536}) lines.push_back(cigar_line(k));
    for (const char* fx : kFloats) lines.push_back(std::string("r\t99\tchr1\t1\t60\t4M\t=\t1\t0\tACGT\tIIII\tXF:f:") + fx);
    for (const char* ix : kInts) {
        lines.push_back(std::string("r\t99\tchr1\t1\t60\t4M\t=\t1\t0\tACGT\tIIII\tXI:i:") + ix);
        lines.push_back(std::string("r\t") + ix + "\tchr1\t" + ix + "\t" + ix + "\t4M\t=\t" + ix + "\t" + ix + "\tACGT\tIIII");
    }
    uint64_t bad = 0, fast = 0, slow = 0, empty = 0;
    std::vector<uint8_t> host, dev;
    for (uint64_t i = 0; i < n + lines.size(); ++i) {
        const std::string line = i < lines.size() ? lines[i] : make_line();
        std::string stripped = line;
        if (!stripped.empty() && stripped.back() == '\r') stripped.pop_back();
        uint32_t lseq = 0;
        const int64_t sz = bqc::sam_fast_line((const uint8_t*)line.data(), (uint32_t)line.size(), R, nullptr, lseq);
        if (stripped.empty()) {
            if (sz != 0) { ++bad; printf("empty line not skipped\n"); }
            ++empty;
            continue;
        }
        if (sz < 0) { ++slow; continue; }
        ++fast;
        if (ef) { fwrite(line.data(), 1, line.size(), ef); fputc('\n', ef); }
        host.clear();
        const bool ok = sam_line_to_bam(stripped, ref_id, host);
        dev.assign((size_t)sz, 0xAB);
        const int64_t sz2 = bqc::sam_fast_line((const uint8_t*)line.data(), (uint32_t)line.size(), R, dev.data(), lseq);
        const bool bound = (uint64_t)sz <= 2 * (line.size() + 1);
        if (!ok || sz2 != sz || host != dev || !bound || lseq != (uint32_t)(int32_t)(host.size() >= 24 ? host[20] | host[21] << 8 | host[22] << 16 | host[23] << 24 : 0)) {
            if (bad < 10) printf("MISMATCH (host ok %d, sizes %zu / %lld, bound %d): %.200s\n", ok, host.size(), (long long)sz, bound, stripped.c_str());
            ++bad;
        }
    }
    if (ef) fclose(ef);
    printf("%llu lines: %llu fast, %llu not fast, %llu empty; %llu mismatching\n", (unsigned long long)(n + lines.size()), (unsigned long long)fast,
           (unsigned long long)slow, (unsigned long long)empty, (unsigned long long)bad);
    return bad ? 1 : 0;
}
