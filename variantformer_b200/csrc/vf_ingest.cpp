// vf_ingest.cpp — libvf_ingest.so: FASTA / VCF ingest for stage 1 (include/vf_ingest.h).
// Plain text, gzip or BGZF in; byte-per-base sequences and per-chromosome sorted variant arrays out.
// BGZF members are inflated in parallel, VCF lines are parsed in parallel chunks and merged in file order.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <memory>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/vf_ingest.h"

namespace {

thread_local char g_err[512] = "";
void set_err(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int resolve_threads(int n) {
    if (n > 0) return n;
    unsigned h = std::thread::hardware_concurrency();
    return h ? (int)h : 4;
}

template <class F>
void parallel_for(int64_t n, int n_threads, F&& body) {             // body(index), dynamic scheduling
    if (n <= 0) return;
    const int nt = (int)std::min<int64_t>(n, n_threads);
    if (nt <= 1) { for (int64_t i = 0; i < n; ++i) body(i); return; }
    std::atomic<int64_t> next(0);
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t)
        th.emplace_back([&]() { for (int64_t i; (i = next.fetch_add(1)) < n;) body(i); });
    for (auto& x : th) x.join();
}

bool read_file(const char* path, std::vector<uint8_t>& out) {
    FILE* f = fopen(path, "rb");
    if (!f) { set_err("cannot open %s", path); return false; }
    fseek(f, 0, SEEK_END);
    const long long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    out.resize((size_t)n);
    const size_t got = n ? fread(out.data(), 1, (size_t)n, f) : 0;
    fclose(f);
    if ((long long)got != n) { set_err("short read on %s", path); return false; }
    return true;
}

// ---- gzip / BGZF ------------------------------------------------------------------------------------------------
struct Member { size_t off, csize, usize, uoff; };

// BGZF: every gzip member carries an extra subfield 'B','C' with BSIZE (member size - 1); ISIZE is its last 4 bytes.
bool scan_bgzf(const std::vector<uint8_t>& z, std::vector<Member>& ms) {
    size_t p = 0, u = 0;
    while (p < z.size()) {
        if (p + 18 > z.size() || z[p] != 0x1f || z[p + 1] != 0x8b || z[p + 2] != 8 || !(z[p + 3] & 4)) return false;
        const size_t xlen = z[p + 10] | (z[p + 11] << 8);
        size_t q = p + 12, bsize = 0;
        const size_t xend = q + xlen;
        if (xend > z.size()) return false;
        while (q + 4 <= xend) {
            const size_t slen = z[q + 2] | (z[q + 3] << 8);
            if (z[q] == 'B' && z[q + 1] == 'C' && slen == 2) bsize = (z[q + 4] | (z[q + 5] << 8)) + 1;
            q += 4 + slen;
        }
        if (!bsize || p + bsize > z.size()) return false;
        const uint8_t* t = &z[p + bsize - 4];
        const size_t isize = t[0] | (t[1] << 8) | (t[2] << 16) | ((size_t)t[3] << 24);
        ms.push_back({p, bsize, isize, u});
        u += isize;
        p += bsize;
    }
    return !ms.empty();
}

bool inflate_member(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, size_t* produced) {
    z_stream s;
    memset(&s, 0, sizeof(s));
    if (inflateInit2(&s, 15 + 16) != Z_OK) return false;
    s.next_in = const_cast<Bytef*>(src); s.avail_in = (uInt)n;
    s.next_out = dst; s.avail_out = (uInt)cap;
    const int rc = inflate(&s, Z_FINISH);
    *produced = s.total_out;
    inflateEnd(&s);
    return rc == Z_STREAM_END;
}

// whole file -> text (decompressed if needed)
bool load_text(const char* path, int n_threads, std::vector<uint8_t>& text) {
    std::vector<uint8_t> raw;
    if (!read_file(path, raw)) return false;
    if (raw.size() < 2 || raw[0] != 0x1f || raw[1] != 0x8b) { text.swap(raw); return true; }
    std::vector<Member> ms;
    if (scan_bgzf(raw, ms)) {                                        // BGZF: independent members, inflate in parallel
        text.resize(ms.back().uoff + ms.back().usize);
        std::atomic<bool> ok(true);
        parallel_for((int64_t)ms.size(), n_threads, [&](int64_t i) {
            const Member& m = ms[(size_t)i];
            size_t got = 0;
            if (m.usize == 0) return;                                // (the empty EOF block)
            if (!inflate_member(&raw[m.off], m.csize, &text[m.uoff], m.usize, &got) || got != m.usize) ok = false;
        });
        if (!ok) { set_err("corrupt BGZF block in %s", path); return false; }
        return true;
    }
    // generic gzip (possibly several members): one stream
    z_stream s;
    memset(&s, 0, sizeof(s));
    if (inflateInit2(&s, 15 + 32) != Z_OK) { set_err("zlib init failed"); return false; }
    text.resize(std::max<size_t>(raw.size() * 4, 1 << 20));
    size_t in_pos = 0;
    s.next_out = text.data(); s.avail_out = (uInt)std::min<size_t>(text.size(), 1u << 30);
    size_t out_pos = 0;
    for (;;) {
        s.next_in = raw.data() + in_pos;
        s.avail_in = (uInt)std::min<size_t>(raw.size() - in_pos, 1u << 30);
        const uInt in_before = s.avail_in, out_before = s.avail_out;
        const int rc = inflate(&s, Z_NO_FLUSH);
        in_pos += in_before - s.avail_in;
        out_pos += out_before - s.avail_out;
        if (rc == Z_STREAM_END) {
            if (in_pos >= raw.size()) break;
            inflateReset(&s);                                        // next member
        } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
            inflateEnd(&s);
            set_err("corrupt gzip stream in %s (zlib %d)", path, rc);
            return false;
        } else if (rc == Z_BUF_ERROR && s.avail_in == 0 && in_pos >= raw.size()) {
            inflateEnd(&s);
            set_err("truncated gzip stream in %s", path);
            return false;
        }
        if (s.avail_out == 0) {
            if (out_pos == text.size()) text.resize(text.size() * 2);
            s.next_out = text.data() + out_pos;
            s.avail_out = (uInt)std::min<size_t>(text.size() - out_pos, 1u << 30);
        }
    }
    inflateEnd(&s);
    text.resize(out_pos);
    return true;
}

}  // namespace

// ---- FASTA ------------------------------------------------------------------------------------------------------
struct vf_fasta {
    std::vector<std::string> names;
    std::vector<std::vector<uint8_t>> seqs;
};

struct vf_vcf {
    struct Chrom {
        std::string name;
        std::vector<int64_t> pos;
        std::vector<int32_t> ref_len, alt_off, alt_len;
        std::vector<uint8_t> gt, pool;
    };
    std::vector<Chrom> chroms;
};

namespace {

struct Rec { int64_t pos; int32_t ref_len; uint8_t gt; std::string alt; };
struct ChunkOut { std::vector<std::string> order; std::map<std::string, std::vector<Rec>> per; };

inline const uint8_t* find_tab(const uint8_t* p, const uint8_t* e) {
    const void* t = memchr(p, '\t', (size_t)(e - p));
    return t ? (const uint8_t*)t : e;
}

char iupac2(char a, char b) {
    auto up = [](char c) { return (char)((c >= 'a' && c <= 'z') ? c - 32 : c); };
    a = up(a); b = up(b);
    if (a > b) std::swap(a, b);
    if (a == 'A' && b == 'C') return 'M';
    if (a == 'A' && b == 'G') return 'R';
    if (a == 'A' && b == 'T') return 'W';
    if (a == 'C' && b == 'G') return 'S';
    if (a == 'C' && b == 'T') return 'Y';
    if (a == 'G' && b == 'T') return 'K';
    return 'N';
}

// The columns every sample of a data line shares: POS, REF length and the ALT list.
struct LineFixed {
    bool pos_ok;
    int64_t pos;                                                     // 1-based, as in the file
    int32_t ref_len;
    std::vector<std::pair<const uint8_t*, const uint8_t*>> alts;
};

void parse_fixed(const uint8_t* const* f, const uint8_t* const* fe, LineFixed& L) {
    L.alts.clear();
    for (const uint8_t* a = f[4]; a <= fe[4];) {
        const uint8_t* c = (const uint8_t*)memchr(a, ',', (size_t)(fe[4] - a));
        if (!c) c = fe[4];
        L.alts.emplace_back(a, c);
        if (c >= fe[4]) break;
        a = c + 1;
    }
    L.pos_ok = true;
    L.pos = 0;
    for (const uint8_t* d = f[1]; d < fe[1]; ++d) {
        if (*d < '0' || *d > '9') { L.pos_ok = false; break; }
        L.pos = L.pos * 10 + (*d - '0');
    }
    L.ref_len = (int32_t)(fe[3] - f[3]);
}

// One sample column [samp, samp_e) of a line -> record (false: dropped).  The genotype is the first ':'-separated
// subfield, alleles separated by '/' or '|'.
bool decode_sample(const LineFixed& L, const uint8_t* samp, const uint8_t* samp_e, Rec& r) {
    int als[8]; int na = 0;
    {
        const uint8_t* g = samp;
        const uint8_t* ge = (const uint8_t*)memchr(g, ':', (size_t)(samp_e - g));
        if (!ge) ge = samp_e;
        while (g <= ge) {
            const uint8_t* s2 = g;
            while (s2 < ge && *s2 != '/' && *s2 != '|') ++s2;
            if (s2 == g || *g == '.') return false;                  // missing allele
            int v = 0;
            for (const uint8_t* d = g; d < s2; ++d) { if (*d < '0' || *d > '9') return false; v = v * 10 + (*d - '0'); }
            if (na < 8) als[na] = v;
            ++na;
            if (s2 >= ge) break;
            g = s2 + 1;
        }
    }
    if (na == 0) return false;
    if (na == 1) { als[1] = als[0]; na = 2; }
    if (na > 8) na = 8;
    int nz[8]; int nnz = 0;
    bool all_same = true;
    for (int i = 0; i < na; ++i) { if (als[i] > 0) nz[nnz++] = als[i]; if (als[i] != als[0]) all_same = false; }
    if (nnz == 0) return false;                                      // hom-ref
    const auto& alts = L.alts;
    for (int i = 0; i < nnz; ++i) if (nz[i] > (int)alts.size()) return false;
    const auto a0 = alts[(size_t)nz[0] - 1];
    if (a0.first == a0.second || *a0.first == '<' || (a0.second - a0.first == 1 && *a0.first == '*')) return false;
    if (!L.pos_ok) return false;
    r.pos = L.pos - 1;
    r.ref_len = L.ref_len;
    if (all_same) {
        r.gt = 2; r.alt.assign((const char*)a0.first, (size_t)(a0.second - a0.first));
    } else if (nnz == 2 && r.ref_len == 1 && a0.second - a0.first == 1 &&
               alts[(size_t)nz[1] - 1].second - alts[(size_t)nz[1] - 1].first == 1) {
        r.gt = 2; r.alt.assign(1, iupac2((char)*a0.first, (char)*alts[(size_t)nz[1] - 1].first));
    } else {
        r.gt = 1; r.alt.assign((const char*)a0.first, (size_t)(a0.second - a0.first));
    }
    return true;
}

// one data line [p, e) -> the record of sample column `col` (false: dropped)
bool parse_line(const uint8_t* p, const uint8_t* e, int col, std::string& chrom, Rec& r) {
    const uint8_t* f[10];                                            // field starts of the first 10 columns
    int nf = 0;
    const uint8_t* q = p;
    const uint8_t* fe[10];
    const uint8_t* samp = nullptr; const uint8_t* samp_e = nullptr;
    for (int c = 0; q <= e; ++c) {
        const uint8_t* t = find_tab(q, e);
        if (c < 10) { f[nf] = q; fe[nf] = t; ++nf; }
        if (c == col) { samp = q; samp_e = t; }
        if (t >= e) break;
        q = t + 1;
        if (c >= col && c >= 9) break;
    }
    if (nf < 5) return false;
    chrom.assign((const char*)f[0], (size_t)(fe[0] - f[0]));
    if (!samp) return false;                                         // "./."
    LineFixed L;
    parse_fixed(f, fe, L);
    return decode_sample(L, samp, samp_e, r);
}

// Data text after the header, cut into chunks of ~4 MB at line ends (parsed in parallel, merged in file order).
std::vector<std::pair<size_t, size_t>> line_chunks(const uint8_t* b, size_t p, size_t n) {
    std::vector<std::pair<size_t, size_t>> chunks;
    const size_t target = 4u << 20;
    for (size_t s = std::min(p, n); s < n;) {
        size_t e = std::min(n, s + target);
        if (e < n) {
            const void* nl = memchr(b + e, '\n', n - e);
            e = nl ? (size_t)((const uint8_t*)nl - b) + 1 : n;
        }
        chunks.emplace_back(s, e);
        s = e;
    }
    return chunks;
}

// records of one (sample, chromosome), in file order -> the sorted arrays vf_vcf_copy hands out (stable by position)
void pack_chrom(std::vector<const Rec*>& rs, vf_vcf::Chrom& ch) {
    std::stable_sort(rs.begin(), rs.end(), [](const Rec* a, const Rec* b2) { return a->pos < b2->pos; });
    const size_t m = rs.size();
    ch.pos.resize(m); ch.ref_len.resize(m); ch.alt_off.resize(m); ch.alt_len.resize(m); ch.gt.resize(m);
    size_t pool = 0;
    for (const Rec* r : rs) pool += r->alt.size();
    ch.pool.resize(pool);
    size_t w = 0;
    for (size_t i = 0; i < m; ++i) {
        const Rec* r = rs[i];
        ch.pos[i] = r->pos; ch.ref_len[i] = r->ref_len; ch.gt[i] = r->gt;
        ch.alt_off[i] = (int32_t)w; ch.alt_len[i] = (int32_t)r->alt.size();
        memcpy(ch.pool.data() + w, r->alt.data(), r->alt.size());
        w += r->alt.size();
    }
}

// BED intervals per chromosome, sorted and merged: does [p0, p1) intersect one of them?
struct Regions {
    std::map<std::string, std::vector<std::pair<int64_t, int64_t>>> iv;
    bool parse(const char* bed) {
        for (const char* p = bed; *p;) {
            const char* e = strchr(p, '\n');
            if (!e) e = p + strlen(p);
            std::string line(p, (size_t)(e - p));
            p = *e ? e + 1 : e;
            while (!line.empty() && (line.back() == '\r' || line.back() == ' ' || line.back() == '\t')) line.pop_back();
            if (line.empty() || line[0] == '#' || !line.compare(0, 5, "track") || !line.compare(0, 7, "browser")) continue;
            char chrom[256];
            long long a = 0, b = 0;
            if (sscanf(line.c_str(), "%255s %lld %lld", chrom, &a, &b) != 3 || a < 0 || b < a) {
                set_err("regions: malformed BED line '%.200s'", line.c_str());
                return false;
            }
            if (b > a) iv[chrom].emplace_back(a, b);
        }
        for (auto& kv : iv) {
            auto& v = kv.second;
            std::sort(v.begin(), v.end());
            size_t k = 0;
            for (size_t i = 1; i < v.size(); ++i) {
                if (v[i].first <= v[k].second) v[k].second = std::max(v[k].second, v[i].second);
                else v[++k] = v[i];
            }
            v.resize(v.empty() ? 0 : k + 1);
        }
        return true;
    }
    bool hit(const std::string& chrom, int64_t p0, int64_t p1) const {
        auto it = iv.find(chrom);
        if (it == iv.end()) return false;
        const auto& v = it->second;
        auto u = std::lower_bound(v.begin(), v.end(), std::make_pair(p1, (int64_t)INT64_MIN));   // first start >= p1
        return u != v.begin() && std::prev(u)->second > p0;
    }
};

}  // namespace

// ---- multi-sample VCF ---------------------------------------------------------------------------------------------
struct vf_vcf_cohort {
    std::vector<std::string> samples;
    std::vector<std::string> chroms;
    std::vector<vf_vcf::Chrom> data;                                 // [sample * chroms.size() + chrom]
    const vf_vcf::Chrom* at(int s, int c) const {
        if (s < 0 || s >= (int)samples.size() || c < 0 || c >= (int)chroms.size()) return nullptr;
        return &data[(size_t)s * chroms.size() + (size_t)c];
    }
};

extern "C" {

const char* vf_ingest_last_error(void) { return g_err; }

vf_fasta* vf_fasta_open(const char* path, int n_threads) {
    const int nt = resolve_threads(n_threads);
    std::vector<uint8_t> text;
    if (!load_text(path, nt, text)) return nullptr;
    struct Span { size_t name_b, name_e, body_b, body_e; };
    std::vector<Span> spans;
    const uint8_t* b = text.data();
    const size_t n = text.size();
    size_t p = 0;
    while (p < n) {
        if (b[p] != '>') {                                           // stray text before the first header: skip the line
            const void* nl = memchr(b + p, '\n', n - p);
            p = nl ? (size_t)((const uint8_t*)nl - b) + 1 : n;
            continue;
        }
        const void* nl = memchr(b + p, '\n', n - p);
        const size_t he = nl ? (size_t)((const uint8_t*)nl - b) : n;
        size_t ne = p + 1;
        while (ne < he && b[ne] != ' ' && b[ne] != '\t' && b[ne] != '\r') ++ne;
        size_t q = std::min(he + 1, n), body_b = q;
        for (;;) {                                                   // body ends at the next line that starts with '>'
            if (q >= n) break;
            if (b[q] == '>') break;
            const void* nl2 = memchr(b + q, '\n', n - q);
            q = nl2 ? (size_t)((const uint8_t*)nl2 - b) + 1 : n;
        }
        spans.push_back({p + 1, ne, body_b, q});
        p = q;
    }
    vf_fasta* f = new vf_fasta;
    f->names.resize(spans.size());
    f->seqs.resize(spans.size());
    parallel_for((int64_t)spans.size(), nt, [&](int64_t i) {
        const Span& s = spans[(size_t)i];
        f->names[(size_t)i].assign((const char*)b + s.name_b, s.name_e - s.name_b);
        std::vector<uint8_t>& out = f->seqs[(size_t)i];
        out.resize(s.body_e - s.body_b);
        size_t w = 0, q = s.body_b;
        while (q < s.body_e) {
            const void* nl = memchr(b + q, '\n', s.body_e - q);
            size_t le = nl ? (size_t)((const uint8_t*)nl - b) : s.body_e;
            size_t ce = le;
            while (ce > q && (b[ce - 1] == '\r')) --ce;
            memcpy(out.data() + w, b + q, ce - q);
            w += ce - q;
            q = le + 1;
        }
        out.resize(w);
    });
    return f;
}
int vf_fasta_num_seqs(const vf_fasta* f) { return f ? (int)f->names.size() : -1; }
const char* vf_fasta_name(const vf_fasta* f, int i) {
    return (f && i >= 0 && i < (int)f->names.size()) ? f->names[(size_t)i].c_str() : nullptr;
}
int64_t vf_fasta_length(const vf_fasta* f, int i) {
    return (f && i >= 0 && i < (int)f->seqs.size()) ? (int64_t)f->seqs[(size_t)i].size() : -1;
}
int64_t vf_fasta_copy(const vf_fasta* f, int i, uint8_t* dst, int64_t cap) {
    if (!f || i < 0 || i >= (int)f->seqs.size()) { set_err("vf_fasta_copy: bad sequence index %d", i); return -1; }
    const auto& s = f->seqs[(size_t)i];
    if ((int64_t)s.size() > cap) { set_err("vf_fasta_copy: buffer too small"); return -1; }
    memcpy(dst, s.data(), s.size());
    return (int64_t)s.size();
}
void vf_fasta_close(vf_fasta* f) { delete f; }

vf_vcf* vf_vcf_open(const char* path, const char* sample, int n_threads) {
    const int nt = resolve_threads(n_threads);
    std::vector<uint8_t> text;
    if (!load_text(path, nt, text)) return nullptr;
    const uint8_t* b = text.data();
    const size_t n = text.size();
    // header: skip '##', take the sample column from '#CHROM'
    size_t p = 0;
    int col = 9;
    while (p < n && b[p] == '#') {
        const void* nl = memchr(b + p, '\n', n - p);
        const size_t le = nl ? (size_t)((const uint8_t*)nl - b) : n;
        if (le - p > 6 && !memcmp(b + p, "#CHROM", 6) && sample) {
            size_t ce = le;
            while (ce > p && b[ce - 1] == '\r') --ce;
            int c = 0; bool found = false;
            for (size_t q = p; q <= ce; ++c) {
                const uint8_t* t = find_tab(b + q, b + ce);
                if (c >= 9 && strlen(sample) == (size_t)(t - (b + q)) && !memcmp(b + q, sample, strlen(sample))) {
                    col = c; found = true; break;
                }
                if (t >= b + ce) break;
                q = (size_t)(t - b) + 1;
            }
            if (!found) { set_err("sample %s not found in %s", sample, path); return nullptr; }
        }
        p = le + 1;
    }
    // data: chunks of ~4 MB cut at line ends, parsed in parallel, merged in file order (keeps the sort stable)
    const auto chunks = line_chunks(b, p, n);
    std::vector<ChunkOut> outs(chunks.size());
    parallel_for((int64_t)chunks.size(), nt, [&](int64_t ci) {
        ChunkOut& o = outs[(size_t)ci];
        size_t q = chunks[(size_t)ci].first;
        const size_t ce = chunks[(size_t)ci].second;
        std::string chrom, last;
        std::vector<Rec>* cur = nullptr;
        Rec r;
        while (q < ce) {
            const void* nl = memchr(b + q, '\n', ce - q);
            const size_t le = nl ? (size_t)((const uint8_t*)nl - b) : ce;
            size_t te = le;
            while (te > q && b[te - 1] == '\r') --te;
            if (te > q && b[q] != '#' && parse_line(b + q, b + te, col, chrom, r)) {
                if (!cur || chrom != last) {
                    auto it = o.per.find(chrom);
                    if (it == o.per.end()) { o.order.push_back(chrom); it = o.per.emplace(chrom, std::vector<Rec>()).first; }
                    cur = &it->second; last = chrom;
                }
                cur->push_back(std::move(r));
            }
            q = le + 1;
        }
    });
    vf_vcf* v = new vf_vcf;
    std::map<std::string, size_t> index;
    std::vector<std::vector<const Rec*>> recs;
    for (const ChunkOut& o : outs)
        for (const std::string& name : o.order) {
            auto it = index.find(name);
            if (it == index.end()) {
                it = index.emplace(name, v->chroms.size()).first;
                v->chroms.emplace_back(); v->chroms.back().name = name; recs.emplace_back();
            }
            for (const Rec& r : o.per.at(name)) recs[it->second].push_back(&r);
        }
    parallel_for((int64_t)v->chroms.size(), nt, [&](int64_t c) { pack_chrom(recs[(size_t)c], v->chroms[(size_t)c]); });
    return v;
}
int vf_vcf_num_chroms(const vf_vcf* v) { return v ? (int)v->chroms.size() : -1; }
const char* vf_vcf_chrom(const vf_vcf* v, int c) {
    return (v && c >= 0 && c < (int)v->chroms.size()) ? v->chroms[(size_t)c].name.c_str() : nullptr;
}
int64_t vf_vcf_num_records(const vf_vcf* v, int c) {
    return (v && c >= 0 && c < (int)v->chroms.size()) ? (int64_t)v->chroms[(size_t)c].pos.size() : -1;
}
int64_t vf_vcf_alt_bytes(const vf_vcf* v, int c) {
    return (v && c >= 0 && c < (int)v->chroms.size()) ? (int64_t)v->chroms[(size_t)c].pool.size() : -1;
}
int vf_vcf_copy(const vf_vcf* v, int c, int64_t* pos, int32_t* ref_len, int32_t* alt_off, int32_t* alt_len,
                uint8_t* gt, uint8_t* alt_pool) {
    if (!v || c < 0 || c >= (int)v->chroms.size()) { set_err("vf_vcf_copy: bad chromosome index %d", c); return -1; }
    const vf_vcf::Chrom& ch = v->chroms[(size_t)c];
    const size_t m = ch.pos.size();
    memcpy(pos, ch.pos.data(), m * sizeof(int64_t));
    memcpy(ref_len, ch.ref_len.data(), m * sizeof(int32_t));
    memcpy(alt_off, ch.alt_off.data(), m * sizeof(int32_t));
    memcpy(alt_len, ch.alt_len.data(), m * sizeof(int32_t));
    memcpy(gt, ch.gt.data(), m);
    memcpy(alt_pool, ch.pool.data(), ch.pool.size());
    return 0;
}
void vf_vcf_close(vf_vcf* v) { delete v; }

vf_vcf_cohort* vf_vcf_open_cohort(const char* path, const char* const* samples, int n_samples, const char* regions_bed,
                                  int n_threads) {
    if (samples && n_samples < 1) { set_err("vf_vcf_open_cohort: %d samples requested", n_samples); return nullptr; }
    Regions regions;
    if (regions_bed && !regions.parse(regions_bed)) return nullptr;
    const int nt = resolve_threads(n_threads);
    std::vector<uint8_t> text;
    if (!load_text(path, nt, text)) return nullptr;
    const uint8_t* b = text.data();
    const size_t n = text.size();
    // header: skip '##', the sample names are the '#CHROM' line's columns from the tenth on
    size_t p = 0;
    std::vector<std::string> header;
    bool have_header = false;
    while (p < n && b[p] == '#') {
        const void* nl = memchr(b + p, '\n', n - p);
        const size_t le = nl ? (size_t)((const uint8_t*)nl - b) : n;
        if (le - p > 6 && !memcmp(b + p, "#CHROM", 6) && !have_header) {
            size_t ce = le;
            while (ce > p && b[ce - 1] == '\r') --ce;
            int c = 0;
            for (size_t q = p; q <= ce; ++c) {
                const uint8_t* t = find_tab(b + q, b + ce);
                if (c >= 9) header.emplace_back((const char*)b + q, (size_t)(t - (b + q)));
                if (t >= b + ce) break;
                q = (size_t)(t - b) + 1;
            }
            have_header = true;
        }
        p = le + 1;
    }
    if (!have_header) { set_err("no #CHROM header line in %s", path); return nullptr; }
    std::unique_ptr<vf_vcf_cohort> v(new vf_vcf_cohort);
    std::vector<int> cols;                                           // column of every requested sample
    std::map<std::string, int> first_col;                            // name -> its first column (as vf_vcf_open picks)
    for (size_t i = 0; i < header.size(); ++i) first_col.emplace(header[i], (int)i + 9);
    if (!samples) {
        if (first_col.size() != header.size()) { set_err("duplicate sample names in the header of %s", path); return nullptr; }
        v->samples = header;
    } else {
        for (int i = 0; i < n_samples; ++i) v->samples.emplace_back(samples[i] ? samples[i] : "");
    }
    std::map<std::string, int> seen;
    for (const std::string& s : v->samples) {
        auto it = first_col.find(s);
        if (it == first_col.end()) { set_err("sample %s not found in %s", s.c_str(), path); return nullptr; }
        if (!seen.emplace(s, 0).second) { set_err("sample %s requested twice", s.c_str()); return nullptr; }
        cols.push_back(it->second);
    }
    const int S = (int)cols.size();
    if (S == 0) { set_err("no sample columns in %s", path); return nullptr; }   // a sites-only VCF
    const int max_col = *std::max_element(cols.begin(), cols.end());
    // data: every line is split once and each requested column decoded from it
    const auto chunks = line_chunks(b, p, n);
    struct CohortChunk {
        std::vector<std::string> order;                              // chromosomes in order of their first kept record
        std::vector<std::vector<Rec>> recs;                          // [local chrom * S + sample]
    };
    std::vector<CohortChunk> outs(chunks.size());
    parallel_for((int64_t)chunks.size(), nt, [&](int64_t ci) {
        CohortChunk& o = outs[(size_t)ci];
        size_t q0 = chunks[(size_t)ci].first;
        const size_t ce = chunks[(size_t)ci].second;
        std::vector<const uint8_t*> cb((size_t)max_col + 1), cend((size_t)max_col + 1);
        std::string chrom, last;
        int cur = -1;
        LineFixed L;
        Rec r;
        while (q0 < ce) {
            const void* nl = memchr(b + q0, '\n', ce - q0);
            const size_t le = nl ? (size_t)((const uint8_t*)nl - b) : ce;
            size_t te = le;
            while (te > q0 && b[te - 1] == '\r') --te;
            const uint8_t* e = b + te;
            if (te > q0 && b[q0] != '#') {
                int nc = 0;
                for (const uint8_t* q = b + q0; q <= e && nc <= max_col;) {
                    const uint8_t* t = find_tab(q, e);
                    cb[(size_t)nc] = q; cend[(size_t)nc] = t; ++nc;
                    if (t >= e) break;
                    q = t + 1;
                }
                if (nc >= 5) {
                    parse_fixed(cb.data(), cend.data(), L);
                    chrom.assign((const char*)cb[0], (size_t)(cend[0] - cb[0]));
                    if (regions_bed && (!L.pos_ok || !regions.hit(chrom, L.pos - 1, L.pos - 1 + std::max<int32_t>(L.ref_len, 1)))) {
                        q0 = le + 1;
                        continue;
                    }
                    for (int s = 0; s < S; ++s) {
                        if (cols[(size_t)s] >= nc || !decode_sample(L, cb[(size_t)cols[(size_t)s]], cend[(size_t)cols[(size_t)s]], r))
                            continue;
                        if (cur < 0 || chrom != last) {
                            auto it = std::find(o.order.begin(), o.order.end(), chrom);
                            cur = (int)(it - o.order.begin());
                            if (it == o.order.end()) { o.order.push_back(chrom); o.recs.resize(o.recs.size() + (size_t)S); }
                            last = chrom;
                        }
                        o.recs[(size_t)cur * S + s].push_back(std::move(r));
                    }
                }
            }
            q0 = le + 1;
        }
    });
    std::map<std::string, size_t> index;
    for (const CohortChunk& o : outs)
        for (const std::string& name : o.order)
            if (index.emplace(name, v->chroms.size()).second) v->chroms.push_back(name);
    const size_t C = v->chroms.size();
    std::vector<std::vector<const Rec*>> recs((size_t)S * C);
    for (const CohortChunk& o : outs)
        for (size_t lc = 0; lc < o.order.size(); ++lc) {
            const size_t c = index.at(o.order[lc]);
            for (int s = 0; s < S; ++s)
                for (const Rec& r : o.recs[lc * S + (size_t)s]) recs[(size_t)s * C + c].push_back(&r);
        }
    v->data.resize((size_t)S * C);
    parallel_for((int64_t)(S * C), nt, [&](int64_t i) { pack_chrom(recs[(size_t)i], v->data[(size_t)i]); });
    return v.release();
}
int vf_vcf_cohort_num_samples(const vf_vcf_cohort* v) { return v ? (int)v->samples.size() : -1; }
const char* vf_vcf_cohort_sample_name(const vf_vcf_cohort* v, int s) {
    return (v && s >= 0 && s < (int)v->samples.size()) ? v->samples[(size_t)s].c_str() : nullptr;
}
int vf_vcf_cohort_num_chroms(const vf_vcf_cohort* v) { return v ? (int)v->chroms.size() : -1; }
const char* vf_vcf_cohort_chrom(const vf_vcf_cohort* v, int c) {
    return (v && c >= 0 && c < (int)v->chroms.size()) ? v->chroms[(size_t)c].c_str() : nullptr;
}
int64_t vf_vcf_cohort_num_records(const vf_vcf_cohort* v, int s, int c) {
    const vf_vcf::Chrom* ch = v ? v->at(s, c) : nullptr;
    return ch ? (int64_t)ch->pos.size() : -1;
}
int64_t vf_vcf_cohort_alt_bytes(const vf_vcf_cohort* v, int s, int c) {
    const vf_vcf::Chrom* ch = v ? v->at(s, c) : nullptr;
    return ch ? (int64_t)ch->pool.size() : -1;
}
int vf_vcf_cohort_copy(const vf_vcf_cohort* v, int s, int c, int64_t* pos, int32_t* ref_len, int32_t* alt_off,
                       int32_t* alt_len, uint8_t* gt, uint8_t* alt_pool) {
    const vf_vcf::Chrom* ch = v ? v->at(s, c) : nullptr;
    if (!ch) { set_err("vf_vcf_cohort_copy: bad sample %d / chromosome %d", s, c); return -1; }
    const size_t m = ch->pos.size();
    memcpy(pos, ch->pos.data(), m * sizeof(int64_t));
    memcpy(ref_len, ch->ref_len.data(), m * sizeof(int32_t));
    memcpy(alt_off, ch->alt_off.data(), m * sizeof(int32_t));
    memcpy(alt_len, ch->alt_len.data(), m * sizeof(int32_t));
    memcpy(gt, ch->gt.data(), m);
    memcpy(alt_pool, ch->pool.data(), ch->pool.size());
    return 0;
}
void vf_vcf_cohort_close(vf_vcf_cohort* v) { delete v; }

}  // extern "C"
