// rt_prepare.cpp -- native host I/O of prepare-orfs (DESIGN.md section 9):
//   * GTF loader: exon and CDS lines parsed in chunks on all cores, attribute strings interned, merged in file order;
//   * FASTA loader: the file read and indexed by all cores, bases translated to 1-byte codes (A C G T -> 0-3, anything
//     else -> 4) straight into the caller's buffer; nothing is written next to the input;
//   * candidate-ORF index writer: rows formatted on all cores, written in order by a write-behind thread.
// No GPU is involved; these entry points also work on a CPU-only box.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

#include "ribotricer_b200.h"
#include "rt_host.h"

// ------------------------------------------------------------------------------------------------------------ GTF
enum { kGeneId, kTxId, kGeneName, kGeneType, kTxType, kAttrs };

struct rt_gtf {
    std::vector<int64_t> line_no;
    std::vector<uint8_t> feature;                // 0 exon, 1 CDS
    std::vector<int32_t> chrom, start, end;      // chrom: string id
    std::vector<uint8_t> strand;                 // 0 '+', 1 '-', 2 anything else
    std::vector<int32_t> attr;                   // kAttrs per line, string ids, -1 = absent
    std::string strings;                         // every distinct string, NUL terminated, in order of first appearance
    int64_t n_strings = 0;
};

namespace {

struct GtfChunk {
    const char *lo, *hi;
    int64_t n_lines = 0;                         // physical lines of the chunk
    std::vector<int64_t> line_no;                // chunk-local 0-based
    std::vector<uint8_t> feature, strand;
    std::vector<int32_t> chrom, start, end, attr;
    std::vector<std::string_view> names;         // local string table
    std::unordered_map<std::string_view, int32_t> ids;
    std::string err;                             // first error, at chunk-local line err_line
    int64_t err_line = -1;

    int32_t intern(std::string_view s) {
        auto it = ids.find(s);
        if (it != ids.end()) return it->second;
        const int32_t id = (int32_t)names.size();
        ids.emplace(s, id);
        names.push_back(s);
        return id;
    }
};

bool gtf_coord(std::string_view f, int32_t& v) {   // ASCII digits, 1 .. 2^31 - 1
    if (f.empty() || f.size() > 10) return false;
    long long x = 0;
    for (char c : f) {
        if (c < '0' || c > '9') return false;
        x = x * 10 + (c - '0');
    }
    if (x < 1 || x > 2147483647LL) return false;
    v = (int32_t)x;
    return true;
}

std::string_view strip_blanks(std::string_view s) {
    while (!s.empty() && s.front() == ' ') s.remove_prefix(1);
    while (!s.empty() && s.back() == ' ') s.remove_suffix(1);
    return s;
}

void parse_gtf_chunk(GtfChunk& ck) {
    int64_t line = 0;
    for (const char* p = ck.lo; p < ck.hi; ++line) {
        const char* eol = (const char*)memchr(p, '\n', (size_t)(ck.hi - p));
        const char* next = eol ? eol + 1 : ck.hi;
        const char* e = eol ? eol : ck.hi;
        if (e > p && e[-1] == '\r') --e;
        const char* q = p;
        p = next;
        if (e == q || *q == '#') continue;
        std::string_view f[9];
        int nf = 0;
        const char* a = q;
        for (;;) {
            const char* t = (const char*)memchr(a, '\t', (size_t)(e - a));
            if (nf < 9) f[nf] = std::string_view(a, (size_t)((t ? t : e) - a));
            ++nf;
            if (!t) break;
            a = t + 1;
        }
        auto fail = [&](std::string msg) { ck.err = std::move(msg); ck.err_line = line; };
        if (nf != 9) { fail("expected 9 tab-separated columns, found " + std::to_string(nf)); return; }
        int32_t s, en;
        if (!gtf_coord(f[3], s)) { fail("start is not a positive integer"); return; }
        if (!gtf_coord(f[4], en)) { fail("end is not a positive integer"); return; }
        if (s > en) { fail("start > end"); return; }
        const bool exon = f[2] == "exon", cds = f[2] == "CDS";
        if (!exon && !cds) continue;
        int32_t at[kAttrs + 2] = {-1, -1, -1, -1, -1, -1, -1};   // + gene_biotype, transcript_biotype
        std::string_view rest = f[8];
        while (!rest.empty()) {
            const size_t semi = rest.find(';');
            std::string_view piece = strip_blanks(rest.substr(0, semi));
            rest = semi == std::string_view::npos ? std::string_view() : rest.substr(semi + 1);
            if (piece.empty()) continue;
            const size_t sp = piece.find(' ');
            std::string_view key = piece.substr(0, sp);
            std::string_view val = sp == std::string_view::npos ? std::string_view() : strip_blanks(piece.substr(sp + 1));
            if (val.size() >= 2 && val.front() == '"' && val.back() == '"') val = val.substr(1, val.size() - 2);
            int slot = key == "gene_id" ? kGeneId : key == "transcript_id" ? kTxId : key == "gene_name" ? kGeneName
                     : key == "gene_type" ? kGeneType : key == "transcript_type" ? kTxType
                     : key == "gene_biotype" ? kAttrs : key == "transcript_biotype" ? kAttrs + 1 : -1;
            if (slot >= 0 && at[slot] < 0) at[slot] = ck.intern(val);
        }
        if (at[kGeneName] < 0) at[kGeneName] = at[kGeneId];
        if (at[kGeneType] < 0) at[kGeneType] = at[kAttrs];
        if (at[kTxType] < 0) at[kTxType] = at[kAttrs + 1];
        ck.line_no.push_back(line);
        ck.feature.push_back(exon ? 0 : 1);
        ck.chrom.push_back(ck.intern(f[0]));
        ck.start.push_back(s);
        ck.end.push_back(en);
        ck.strand.push_back(f[6] == "+" ? 0 : f[6] == "-" ? 1 : 2);
        ck.attr.insert(ck.attr.end(), at, at + kAttrs);
    }
    ck.n_lines = line;
}

}  // namespace

extern "C" {

// rt_gtf_load and rt_gtf_load_text once `text` holds the file
static int gtf_parse(const HostArr<char>& text, rt_gtf** out) {
    const int n_thr = host_threads(text.size() >> 20, 32, "RT_GTF_THREADS");
    const char* base = text.data();
    std::vector<const char*> cut = cut_lines(base, base + text.size(), n_thr);
    std::vector<GtfChunk> chunks((size_t)n_thr);
    for (int k = 0; k < n_thr; ++k) { chunks[(size_t)k].lo = cut[(size_t)k]; chunks[(size_t)k].hi = cut[(size_t)k + 1]; }
    run_parallel(n_thr, [&](int k) { parse_gtf_chunk(chunks[(size_t)k]); });
    // the first error in file order, with its 1-based line number
    int64_t lines_before = 0;
    for (const GtfChunk& ck : chunks) {
        if (!ck.err.empty()) {
            rt_io_set_error("GTF line " + std::to_string(lines_before + ck.err_line + 1) + ": " + ck.err);
            return RT_EINVAL;
        }
        lines_before += ck.n_lines;
    }
    // merge: global string ids in order of first appearance, columns concatenated in file order
    std::unique_ptr<rt_gtf> g(new rt_gtf());
    std::unordered_map<std::string_view, int32_t> ids;
    std::vector<std::vector<int32_t>> remap(chunks.size());
    size_t n = 0;
    for (size_t k = 0; k < chunks.size(); ++k) {
        for (std::string_view s : chunks[k].names) {
            auto it = ids.find(s);
            if (it == ids.end()) {
                it = ids.emplace(s, (int32_t)g->n_strings++).first;
                g->strings.append(s.data(), s.size());
                g->strings.push_back('\0');
            }
            remap[k].push_back(it->second);
        }
        n += chunks[k].line_no.size();
    }
    g->line_no.resize(n); g->feature.resize(n); g->strand.resize(n);
    g->chrom.resize(n); g->start.resize(n); g->end.resize(n); g->attr.resize(n * kAttrs);
    std::vector<size_t> row0(chunks.size() + 1, 0);
    std::vector<int64_t> line0(chunks.size() + 1, 1);
    for (size_t k = 0; k < chunks.size(); ++k) {
        row0[k + 1] = row0[k] + chunks[k].line_no.size();
        line0[k + 1] = line0[k] + chunks[k].n_lines;
    }
    run_parallel((int)chunks.size(), [&](int kk) {
        const size_t k = (size_t)kk;
        GtfChunk& ck = chunks[k];
        const size_t r0 = row0[k], m = ck.line_no.size();
        const std::vector<int32_t>& map = remap[k];
        for (size_t i = 0; i < m; ++i) {
            g->line_no[r0 + i] = line0[k] + ck.line_no[i];
            g->chrom[r0 + i] = map[(size_t)ck.chrom[i]];
            for (int a = 0; a < kAttrs; ++a) {
                const int32_t v = ck.attr[i * kAttrs + a];
                g->attr[(r0 + i) * kAttrs + a] = v < 0 ? -1 : map[(size_t)v];
            }
        }
        if (m) {
            memcpy(g->feature.data() + r0, ck.feature.data(), m);
            memcpy(g->strand.data() + r0, ck.strand.data(), m);
            memcpy(g->start.data() + r0, ck.start.data(), 4 * m);
            memcpy(g->end.data() + r0, ck.end.data(), 4 * m);
        }
    });
    *out = g.release();
    return RT_OK;
}

int rt_gtf_load(const char* path, rt_gtf** out) {
    if (!path || !out) return RT_EINVAL;
    *out = nullptr;
    HostArr<char> text;
    if (const int rc = read_file(path, text)) return rc;
    return gtf_parse(text, out);
}

int rt_gtf_load_text(rt_text* text, const char* path, rt_gtf** out) {
    if (!text || !path || !out) { rt_text_free(text); return RT_EINVAL; }
    *out = nullptr;
    HostArr<char> buf;
    adopt_text(text, buf);
    return gtf_parse(buf, out);
}

void rt_gtf_free(rt_gtf* g) { delete g; }
int64_t rt_gtf_n_lines(const rt_gtf* g) { return g ? (int64_t)g->line_no.size() : 0; }
int64_t rt_gtf_n_strings(const rt_gtf* g) { return g ? g->n_strings : 0; }
int64_t rt_gtf_string_bytes(const rt_gtf* g) { return g ? (int64_t)g->strings.size() : 0; }

int rt_gtf_copy(const rt_gtf* g, int64_t* line_no, uint8_t* feature, int32_t* chrom, int32_t* start, int32_t* end,
                uint8_t* strand, int32_t* attr, char* strings) {
    if (!g) return RT_EINVAL;
    const size_t n = g->line_no.size();
    if (line_no && n) memcpy(line_no, g->line_no.data(), 8 * n);
    if (feature && n) memcpy(feature, g->feature.data(), n);
    if (chrom && n) memcpy(chrom, g->chrom.data(), 4 * n);
    if (start && n) memcpy(start, g->start.data(), 4 * n);
    if (end && n) memcpy(end, g->end.data(), 4 * n);
    if (strand && n) memcpy(strand, g->strand.data(), n);
    if (attr && n) memcpy(attr, g->attr.data(), 4 * n * kAttrs);
    if (strings && !g->strings.empty()) memcpy(strings, g->strings.data(), g->strings.size());
    return RT_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------- FASTA
struct rt_fasta {
    HostArr<char> text;
    std::vector<std::string> names;
    std::vector<int64_t> length;
    struct Piece { int contig; size_t lo, hi; int64_t out; };   // a slice of one contig's text, its first base's rank
    std::vector<Piece> pieces;
    std::vector<size_t> piece0;                  // per contig: first piece (+ 1 sentinel)
    int n_thr = 1;
};

extern "C" {

// rt_fasta_load and rt_fasta_load_text once fa->text holds the file
static int fasta_parse(std::unique_ptr<rt_fasta> fa, rt_fasta** out) {
    const char* base = fa->text.data();
    const size_t size = fa->text.size();
    fa->n_thr = host_threads(size >> 20, 32, "RT_FASTA_THREADS");
    // 1. header lines: a '>' at the start of a line, found by all threads in slices of the file
    std::vector<std::vector<size_t>> found((size_t)fa->n_thr);
    run_parallel(fa->n_thr, [&](int k) {
        size_t at = size * (size_t)k / fa->n_thr;
        const size_t hi = size * (size_t)(k + 1) / fa->n_thr;
        for (; at < hi; ++at) {
            const char* q = (const char*)memchr(base + at, '>', hi - at);
            if (!q) break;
            at = (size_t)(q - base);
            if (at == 0 || base[at - 1] == '\n') found[(size_t)k].push_back(at);
        }
    });
    std::vector<size_t> heads;
    for (auto& v : found) heads.insert(heads.end(), v.begin(), v.end());
    const size_t first = heads.empty() ? size : heads[0];
    for (size_t i = 0; i < first; ++i)
        if (base[i] != '\n' && base[i] != '\r' && base[i] != ' ' && base[i] != '\t') {
            rt_io_set_error("FASTA: sequence before the first header");
            return RT_EINVAL;
        }
    // 2. names and the byte range of every contig's sequence, cut into pieces of at most 8 MB
    std::unordered_map<std::string, int> seen;
    constexpr size_t kPiece = 8u << 20;
    for (size_t c = 0; c < heads.size(); ++c) {
        const size_t h = heads[c], stop = c + 1 < heads.size() ? heads[c + 1] : size;
        const char* nl = (const char*)memchr(base + h, '\n', stop - h);
        const size_t body = nl ? (size_t)(nl - base) + 1 : stop;
        size_t ne = h + 1;
        while (ne < body && base[ne] != ' ' && base[ne] != '\t' && base[ne] != '\r' && base[ne] != '\n') ++ne;
        std::string name(base + h + 1, ne - h - 1);
        if (!seen.emplace(name, (int)c).second) { rt_io_set_error("duplicate FASTA contig " + name); return RT_EINVAL; }
        fa->names.push_back(name);
        fa->piece0.push_back(fa->pieces.size());
        for (size_t lo = body; lo < stop; lo += kPiece) fa->pieces.push_back({(int)c, lo, std::min(stop, lo + kPiece), 0});
    }
    fa->piece0.push_back(fa->pieces.size());
    // 3. bases per piece (everything but '\n' and '\r'), then each piece's rank within its contig
    std::vector<int64_t> count(fa->pieces.size());
    claim_parallel(fa->n_thr, fa->pieces.size(), [&](size_t i) {
        const auto& pc = fa->pieces[i];
        int64_t skip = 0;
        for (size_t j = pc.lo; j < pc.hi; ++j) skip += base[j] == '\n' || base[j] == '\r';
        count[i] = (int64_t)(pc.hi - pc.lo) - skip;
    });
    fa->length.assign(fa->names.size(), 0);
    for (size_t i = 0; i < fa->pieces.size(); ++i) {
        auto& pc = fa->pieces[i];
        pc.out = fa->length[(size_t)pc.contig];
        fa->length[(size_t)pc.contig] += count[i];
    }
    *out = fa.release();
    return RT_OK;
}

int rt_fasta_load(const char* path, rt_fasta** out) {
    if (!path || !out) return RT_EINVAL;
    *out = nullptr;
    std::unique_ptr<rt_fasta> fa(new rt_fasta());
    if (const int rc = read_file(path, fa->text)) return rc;
    return fasta_parse(std::move(fa), out);
}

int rt_fasta_load_text(rt_text* text, const char* path, rt_fasta** out) {
    if (!text || !path || !out) { rt_text_free(text); return RT_EINVAL; }
    *out = nullptr;
    std::unique_ptr<rt_fasta> fa(new rt_fasta());
    adopt_text(text, fa->text);
    return fasta_parse(std::move(fa), out);
}

void rt_fasta_free(rt_fasta* fa) { delete fa; }
int rt_fasta_n_contig(const rt_fasta* fa) { return fa ? (int)fa->names.size() : 0; }
const char* rt_fasta_contig_name(const rt_fasta* fa, int i) {
    return fa && i >= 0 && i < (int)fa->names.size() ? fa->names[(size_t)i].c_str() : nullptr;
}
int64_t rt_fasta_contig_len(const rt_fasta* fa, int i) {
    return fa && i >= 0 && i < (int)fa->length.size() ? fa->length[(size_t)i] : -1;
}

int rt_fasta_codes(const rt_fasta* fa, int n_sel, const int32_t* contigs, uint8_t* out) {
    if (!fa || n_sel < 0 || (n_sel && (!contigs || !out))) { rt_io_set_error("rt_fasta_codes: NULL argument"); return RT_EINVAL; }
    uint8_t lut[256];
    memset(lut, 4, sizeof lut);
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
    struct Job { size_t piece; int64_t at; };
    std::vector<Job> jobs;
    int64_t at = 0;
    for (int s = 0; s < n_sel; ++s) {
        const int c = contigs[s];
        if (c < 0 || c >= (int)fa->names.size()) { rt_io_set_error("rt_fasta_codes: contig id out of range"); return RT_EINVAL; }
        for (size_t i = fa->piece0[(size_t)c]; i < fa->piece0[(size_t)c + 1]; ++i) jobs.push_back({i, at + fa->pieces[i].out});
        at += fa->length[(size_t)c];
    }
    const char* base = fa->text.data();
    claim_parallel(fa->n_thr, jobs.size(), [&](size_t j) {
        const auto& pc = fa->pieces[jobs[j].piece];
        uint8_t* o = out + jobs[j].at;
        for (size_t i = pc.lo; i < pc.hi; ++i) {
            const unsigned char ch = (unsigned char)base[i];
            if (ch == '\n' || ch == '\r') continue;
            *o++ = lut[ch];
        }
    });
    return RT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------- index writer
namespace {

const char* const kTypeName[] = {"annotated", "uORF", "overlap_uORF", "super_uORF", "overlap_dORF", "dORF", "novel", "internal"};

}  // namespace

extern "C" {

int rt_orf_write(const char* path, int64_t n_tx, const char* tx_text, const int64_t* tx_text_off, const int32_t* tx_id_len,
                 int64_t n_rows, const int32_t* row_tx, const uint8_t* row_type, const uint8_t* row_codon,
                 const int64_t* iv_ptr, const int32_t* iv_start, const int32_t* iv_end) {
    if (!path || n_tx < 0 || n_rows < 0 || (n_rows && (!tx_text || !tx_text_off || !tx_id_len || !row_tx || !row_type ||
                                                       !row_codon || !iv_ptr || !iv_start || !iv_end))) {
        rt_io_set_error("rt_orf_write: NULL argument");
        return RT_EINVAL;
    }
    for (int64_t r = 0; r < n_rows; ++r)
        if (row_tx[r] < 0 || row_tx[r] >= n_tx || row_type[r] > 7 || iv_ptr[r + 1] <= iv_ptr[r]) {
            rt_io_set_error("rt_orf_write: row " + std::to_string(r) + " has no transcript, type or interval");
            return RT_EINVAL;
        }
    FILE* fh = fopen(path, "wb");
    if (!fh) { rt_io_set_error(std::string("cannot open ") + path); return RT_EINVAL; }
    static const char kHeader[] = "ORF_ID\tORF_type\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\t"
                                  "chrom\tstrand\tstart_codon\tcoordinate\n";
    const int n_thr = host_threads((size_t)n_rows * 64 >> 20, 32, "RT_WRITE_THREADS");
    constexpr int64_t kBatchRows = 1 << 16;
    auto format = [&](int64_t r0, int64_t r1, TextBuf& s) {
        for (int64_t r = r0; r < r1; ++r) {
            const int64_t t = row_tx[r], a = iv_ptr[r], b = iv_ptr[r + 1];
            const char* tt = tx_text + tx_text_off[t];
            const size_t tlen = (size_t)(tx_text_off[t + 1] - tx_text_off[t]);
            const char* type = kTypeName[row_type[r]];
            char* p = s.need(tlen + (size_t)tx_id_len[t] + 96 + 24 * (size_t)(b - a));
            if (!p) return false;
            int64_t length = 0;
            for (int64_t i = a; i < b; ++i) length += (int64_t)iv_end[i] - iv_start[i] + 1;
            memcpy(p, tt, (size_t)tx_id_len[t]); p += tx_id_len[t];
            *p++ = '_'; p = put_int(p, iv_start[a]);
            *p++ = '_'; p = put_int(p, iv_end[b - 1]);
            *p++ = '_'; p = put_int(p, length);
            *p++ = '\t';
            const size_t tl = strlen(type);
            memcpy(p, type, tl); p += tl;
            *p++ = '\t';
            memcpy(p, tt, tlen); p += tlen;
            *p++ = '\t';
            const unsigned cc = row_codon[r];
            *p++ = "ACGT"[(cc >> 4) & 3]; *p++ = "ACGT"[(cc >> 2) & 3]; *p++ = "ACGT"[cc & 3];
            *p++ = '\t';
            for (int64_t i = a; i < b; ++i) {
                if (i > a) *p++ = ',';
                p = put_int(p, iv_start[i]);
                *p++ = '-';
                p = put_int(p, iv_end[i]);
            }
            *p++ = '\n';
            s.advance_to(p);
        }
        return true;
    };
    // rounds of n_thr batches: formatted by all threads while the earlier rounds are written behind
    bool ok, formatted = true;
    {
        WriteBehind out(fh);
        ok = out.put_view(kHeader, sizeof kHeader - 1);
        std::vector<TextBuf> part((size_t)n_thr);
        std::vector<char> part_ok((size_t)n_thr);
        for (int64_t r0 = 0; r0 < n_rows && ok && formatted; r0 += kBatchRows * n_thr) {
            run_parallel(n_thr, [&](int k) {
                const int64_t lo = std::min(n_rows, r0 + k * kBatchRows), hi = std::min(n_rows, lo + kBatchRows);
                part_ok[(size_t)k] = format(lo, hi, part[(size_t)k]);
            });
            for (int k = 0; k < n_thr && ok && formatted; ++k) {
                formatted = part_ok[(size_t)k];
                if (formatted) ok = out.put(std::move(part[(size_t)k]));
            }
        }
        ok = out.finish() && ok;
    }
    if (fclose(fh) != 0) ok = false;
    if (!formatted) { rt_io_set_error("rt_orf_write: out of memory"); return RT_ENOMEM; }
    if (!ok) { rt_io_set_error(std::string("write failed: ") + path); return RT_EINVAL; }
    return RT_OK;
}

}  // extern "C"
