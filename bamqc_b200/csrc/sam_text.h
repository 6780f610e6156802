// sam_text.h -- SAM text -> BAM records on the host (SAM/BAM specification sections 1.4 and 4.2): the header lines
// become a binary BAM header so that one header parser serves both formats, and every alignment line becomes one BAM
// record.  This encoder defines what the engine counts for SAM input: the device parser (sam_parse.h, kernel_sam.cuh)
// accepts only lines it reproduces byte for byte, and every other submission is encoded here
// (tests/sam_selftest.cpp checks the two against each other).
#pragma once
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <map>
#include <sstream>
#include <string>
#include <vector>

namespace {
template <typename T> void put_le(std::vector<uint8_t>& v, T x) { uint8_t b[sizeof(T)]; memcpy(b, &x, sizeof(T)); v.insert(v.end(), b, b + sizeof(T)); }

std::vector<std::string> split_tabs(const std::string& line) {
    std::vector<std::string> out;
    size_t p = 0;
    for (;;) {
        size_t q = line.find('\t', p);
        out.push_back(line.substr(p, q == std::string::npos ? std::string::npos : q - p));
        if (q == std::string::npos) break;
        p = q + 1;
    }
    return out;
}

// binary BAM header (magic, text, reference list) from SAM header lines
std::vector<uint8_t> sam_header_to_bam(const std::string& text) {
    std::vector<uint8_t> h = {'B', 'A', 'M', 1};
    put_le<int32_t>(h, (int32_t)text.size());
    h.insert(h.end(), text.begin(), text.end());
    std::vector<std::pair<std::string, int32_t>> refs;
    std::istringstream is(text);
    std::string line;
    while (std::getline(is, line)) {
        if (line.compare(0, 3, "@SQ") != 0) continue;
        std::string name;
        int64_t len = 0;
        for (const std::string& f : split_tabs(line)) {
            if (f.compare(0, 3, "SN:") == 0) name = f.substr(3);
            else if (f.compare(0, 3, "LN:") == 0) len = atoll(f.c_str() + 3);
        }
        refs.push_back({name, (int32_t)len});
    }
    put_le<int32_t>(h, (int32_t)refs.size());
    for (auto& r : refs) {
        put_le<int32_t>(h, (int32_t)r.first.size() + 1);
        h.insert(h.end(), r.first.begin(), r.first.end());
        h.push_back(0);
        put_le<int32_t>(h, r.second);
    }
    return h;
}

// one SAM alignment line -> one BAM record appended to out (block_size prefix included); false if malformed
bool sam_line_to_bam(const std::string& line, const std::map<std::string, int32_t>& ref_id, std::vector<uint8_t>& out) {
    const std::vector<std::string> f = split_tabs(line);
    if (f.size() < 11) return false;
    auto rid_of = [&](const std::string& name, int32_t same) -> int32_t {
        if (name == "*") return -1;
        if (name == "=") return same;
        auto it = ref_id.find(name);
        return it == ref_id.end() ? -1 : it->second;
    };
    const int32_t rid = rid_of(f[2], -1), pos = (int32_t)atoll(f[3].c_str()) - 1;
    const int32_t nrid = rid_of(f[6], rid), npos = (int32_t)atoll(f[7].c_str()) - 1, tlen = (int32_t)atoll(f[8].c_str());
    const uint32_t flag = (uint32_t)atoi(f[1].c_str()), mapq = (uint32_t)atoi(f[4].c_str());
    std::vector<uint32_t> cigar;
    if (f[5] != "*") {
        static const char ops[] = "MIDNSHP=X";
        uint64_t n = 0;
        bool have = false;
        for (char ch : f[5]) {
            if (ch >= '0' && ch <= '9') { n = n * 10 + (uint64_t)(ch - '0'); have = true; continue; }
            const char* o = strchr(ops, ch);
            if (!o || !have) return false;
            cigar.push_back((uint32_t)(n << 4) | (uint32_t)(o - ops));
            n = 0;
            have = false;
        }
        if (have) return false;
    }
    const std::string seq = f[9] == "*" ? std::string() : f[9];
    const size_t start = out.size();
    put_le<int32_t>(out, 0);  // block_size, patched below
    put_le<int32_t>(out, rid);
    put_le<int32_t>(out, pos);
    out.push_back((uint8_t)(f[0].size() + 1));
    out.push_back((uint8_t)mapq);
    put_le<uint16_t>(out, 4680);  // bin: not used by the statistics
    put_le<uint16_t>(out, (uint16_t)cigar.size());
    put_le<uint16_t>(out, (uint16_t)flag);
    put_le<int32_t>(out, (int32_t)seq.size());
    put_le<int32_t>(out, nrid);
    put_le<int32_t>(out, npos);
    put_le<int32_t>(out, tlen);
    out.insert(out.end(), f[0].begin(), f[0].end());
    out.push_back(0);
    for (uint32_t c : cigar) put_le<uint32_t>(out, c);
    static const char nt16[] = "=ACMGRSVTWYHKDBN";
    for (size_t i = 0; i < seq.size(); i += 2) {
        auto code = [&](char ch) -> uint8_t {
            const char* q = strchr(nt16, toupper((unsigned char)ch));
            return q && ch ? (uint8_t)(q - nt16) : 15;
        };
        out.push_back((uint8_t)((code(seq[i]) << 4) | (i + 1 < seq.size() ? code(seq[i + 1]) : 0)));
    }
    if (f[10] == "*" || f[10].size() != seq.size()) out.insert(out.end(), seq.size(), 0xFF);
    else for (char ch : f[10]) out.push_back((uint8_t)(ch - 33));
    for (size_t t = 11; t < f.size(); ++t) {  // TAG:TYPE:VALUE
        const std::string& a = f[t];
        if (a.size() < 5 || a[2] != ':' || a[4] != ':') return false;
        const char ty = a[3];
        const std::string val = a.substr(5);
        out.push_back((uint8_t)a[0]);
        out.push_back((uint8_t)a[1]);
        if (ty == 'A') { out.push_back('A'); out.push_back(val.empty() ? 0 : (uint8_t)val[0]); }
        else if (ty == 'i') {  // the smallest BAM integer type that holds the value
            const long long v = atoll(val.c_str());
            if (v >= 0) {
                if (v <= 255) { out.push_back('C'); out.push_back((uint8_t)v); }
                else if (v <= 65535) { out.push_back('S'); put_le<uint16_t>(out, (uint16_t)v); }
                else { out.push_back('I'); put_le<uint32_t>(out, (uint32_t)v); }
            } else {
                if (v >= -128) { out.push_back('c'); out.push_back((uint8_t)(int8_t)v); }
                else if (v >= -32768) { out.push_back('s'); put_le<int16_t>(out, (int16_t)v); }
                else { out.push_back('i'); put_le<int32_t>(out, (int32_t)v); }
            }
        } else if (ty == 'f') { out.push_back('f'); put_le<float>(out, (float)atof(val.c_str())); }
        else if (ty == 'Z' || ty == 'H') { out.push_back((uint8_t)ty); out.insert(out.end(), val.begin(), val.end()); out.push_back(0); }
        else if (ty == 'B') {
            if (val.empty()) return false;
            const char sub = val[0];
            std::vector<std::string> items;
            std::stringstream ss(val.size() > 2 ? val.substr(2) : std::string());
            std::string item;
            while (std::getline(ss, item, ',')) items.push_back(item);
            out.push_back('B');
            out.push_back((uint8_t)sub);
            put_le<int32_t>(out, (int32_t)items.size());
            for (const std::string& it : items) {
                switch (sub) {
                    case 'c': out.push_back((uint8_t)(int8_t)atoi(it.c_str())); break;
                    case 'C': out.push_back((uint8_t)atoi(it.c_str())); break;
                    case 's': put_le<int16_t>(out, (int16_t)atoi(it.c_str())); break;
                    case 'S': put_le<uint16_t>(out, (uint16_t)atoi(it.c_str())); break;
                    case 'i': put_le<int32_t>(out, (int32_t)atoll(it.c_str())); break;
                    case 'I': put_le<uint32_t>(out, (uint32_t)atoll(it.c_str())); break;
                    case 'f': put_le<float>(out, (float)atof(it.c_str())); break;
                    default: return false;
                }
            }
        } else return false;
    }
    const int32_t bs = (int32_t)(out.size() - start - 4);
    memcpy(out.data() + start, &bs, 4);
    return true;
}
}  // namespace

// The @SQ names as the device's lookup table (sam_parse.h SamRefs): sorted like std::map<std::string, int32_t>, the
// first of duplicate names kept, as sam_line_to_bam's map does.
inline void sam_refs_build(const std::vector<std::string>& names, std::string& blob, std::vector<uint32_t>& off, std::vector<int32_t>& id) {
    std::map<std::string, int32_t> m;
    for (size_t i = 0; i < names.size(); ++i) m.insert({names[i], (int32_t)i});
    blob.clear();
    off.assign(1, 0);
    id.clear();
    for (auto& kv : m) {
        blob += kv.first;
        off.push_back((uint32_t)blob.size());
        id.push_back(kv.second);
    }
}
