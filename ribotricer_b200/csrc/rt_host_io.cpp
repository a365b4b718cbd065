// rt_host_io.cpp -- native host I/O around the GPU path (SURVEY.md 8(f) "next #3"):
//   * candidate-ORF index loader: ORF.from_string rules (orf.py:121-182), interval sort (orf.py:100),
//     annotated prefix (detect_orfs.py:104-118) -> CSR arrays, without one Python object per row;
//   * {prefix}_translating_ORFs.tsv writer: rows formatted exactly as detect_orfs.py:304-323 prints
//     them (np.float64 / Python float shortest repr, str(list) profile).
// No GPU is involved; these entry points also work on a CPU-only box.
#include <algorithm>
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "ribotricer_b200.h"
#include "rt_host.h"

struct rt_index {
    HostArr<char> text;                  // the whole file; fields point into it
    HostArr<int64_t> exon_ptr;           // n_orf + 1
    HostArr<int32_t> exon_start, exon_end;
    HostArr<int32_t> orf_chrom;          // index into chrom_names
    HostArr<uint8_t> orf_strand;         // 0 '+', 1 '-', 2 anything else
    HostArr<uint32_t> field_len;         // 9 per ORF: lengths of fields 1..9
    HostArr<uint64_t> line_field;        // per ORF: offset of field 1 (64-bit, files > 4 GB)
    std::vector<std::string> chrom_names;
    int64_t n_annotated_prefix = 0;
    std::string error;
};

// An output file (TSV or WIG) with its write-behind thread.
struct rt_tsv {
    FILE* fh;
    WriteBehind out;
    explicit rt_tsv(FILE* f) : fh(f), out(f) {}
};

namespace {

thread_local std::string g_io_error;

// Shortest round-trip repr of a double in Python's float.__repr__ / numpy float64.__str__ style.
void append_repr(std::string& out, double x) {
    if (x != x) { out += "nan"; return; }
    if (x == 1.0 / 0.0) { out += "inf"; return; }
    if (x == -1.0 / 0.0) { out += "-inf"; return; }
    char tmp[64];
    auto res = std::to_chars(tmp, tmp + sizeof tmp, x, std::chars_format::scientific);   // d[.ddd]e[+-]XX, shortest
    const char* p = tmp;
    if (*p == '-') { out += '-'; ++p; }
    const char* e = std::find(p, (const char*)res.ptr, 'e');
    std::string digits;
    for (const char* q = p; q < e; ++q)
        if (*q != '.') digits += *q;
    int exp10 = 0;
    std::from_chars(e + 1 + (e[1] == '+' ? 1 : 0), res.ptr, exp10);
    const int nd = (int)digits.size();
    if (exp10 < -4 || exp10 >= 16) {            // repr switches to exponent notation here
        out += digits[0];
        if (nd > 1) { out += '.'; out.append(digits, 1, std::string::npos); }
        out += 'e';
        out += exp10 < 0 ? '-' : '+';
        const int a = exp10 < 0 ? -exp10 : exp10;
        if (a < 10) out += '0';
        out += std::to_string(a);
    } else if (exp10 < 0) {
        out += "0.";
        out.append((size_t)(-exp10 - 1), '0');
        out += digits;
    } else if (nd <= exp10 + 1) {
        out += digits;
        out.append((size_t)(exp10 + 1 - nd), '0');
        out += ".0";
    } else {
        out.append(digits, 0, (size_t)exp10 + 1);
        out += '.';
        out.append(digits, (size_t)exp10 + 1, std::string::npos);
    }
}

bool parse_int(const char*& p, const char* end, long long& v) {   // Python int(): optional blanks and sign
    while (p < end && (*p == ' ')) ++p;
    bool neg = false;
    if (p < end && (*p == '-' || *p == '+')) { neg = *p == '-'; ++p; }
    if (p >= end || *p < '0' || *p > '9') return false;
    long long x = 0;
    while (p < end && *p >= '0' && *p <= '9') { x = x * 10 + (*p - '0'); ++p; }
    while (p < end && (*p == ' ' || *p == '\r' || *p == '\n')) ++p;
    v = neg ? -x : x;
    return true;
}

}  // namespace

extern "C" {

const char* rt_io_last_error(void) { return g_io_error.c_str(); }

int rt_text_alloc(int64_t n, rt_text** out) {
    if (!out || n < 0) return RT_EINVAL;
    *out = nullptr;
    std::unique_ptr<rt_text> t(new (std::nothrow) rt_text());
    if (!t || !(t->p = static_cast<char*>(malloc((size_t)n + 1)))) { g_io_error = "out of memory"; return RT_ENOMEM; }
    t->n = (size_t)n;
    t->p[n] = '\0';
    *out = t.release();
    return RT_OK;
}

char* rt_text_data(rt_text* t) { return t ? t->p : nullptr; }
int64_t rt_text_len(const rt_text* t) { return t ? (int64_t)t->n : 0; }

void rt_text_free(rt_text* t) {
    if (!t) return;
    free(t->p);
    delete t;
}

}  // extern "C"

void rt_io_set_error(const std::string& msg) { g_io_error = msg; }   // rt_prepare.cpp reports through the same slot

extern "C" {

// rt_index_load and rt_index_load_text once ix->text holds the file
static int index_parse(std::unique_ptr<rt_index> ix, rt_index** out) {
    const size_t size = ix->text.size();
    const char* base = ix->text.data();
    const char* end = base + size;
    const char* body = (const char*)memchr(base, '\n', size);   // skip the header (detect_orfs.py:273)
    body = body ? body + 1 : end;
    const int n_thr = host_threads(size >> 22, 16, "RT_INDEX_THREADS");   // tests: chunked parse of a small file

    // 2. the rows, parsed in chunks cut at line ends
    struct Chunk {
        const char *lo, *hi;
        std::vector<int32_t> exon_start, exon_end, n_exon, chrom_local;
        std::vector<uint8_t> strand;
        std::vector<uint32_t> field_len;
        std::vector<uint64_t> line_field;
        std::vector<std::string> chrom_names;          // in order of first appearance within the chunk
        int64_t annotated_prefix = 0;                  // leading rows that hold the substring "annotated"
        bool all_annotated = true;
        int err = RT_OK;                               // first error of the chunk, at local row err_row
        int64_t err_row = 0;
    };
    std::vector<Chunk> chunks((size_t)n_thr);
    const std::vector<const char*> cut = cut_lines(body, end, n_thr);
    for (int k = 0; k < n_thr; ++k) { chunks[(size_t)k].lo = cut[(size_t)k]; chunks[(size_t)k].hi = cut[(size_t)k + 1]; }
    auto parse_chunk = [&](Chunk& ck) {
        std::unordered_map<std::string, int> chrom_id;
        std::vector<std::pair<long long, long long>> ivs;
        const size_t rows_guess = (size_t)(ck.hi - ck.lo) / 96 + 16;
        ck.n_exon.reserve(rows_guess); ck.chrom_local.reserve(rows_guess); ck.strand.reserve(rows_guess);
        ck.line_field.reserve(rows_guess); ck.field_len.reserve(9 * rows_guess);
        ck.exon_start.reserve(4 * rows_guess); ck.exon_end.reserve(4 * rows_guess);
        int64_t row = 0;
        for (const char* p = ck.lo; p < ck.hi; ++row) {
            const char* eol = (const char*)memchr(p, '\n', (size_t)(ck.hi - p));
            const char* line_end = eol ? eol : ck.hi;
            // split on tabs: exactly 11 fields (orf.py:144-151)
            const char* f[12];
            int tabs = 0;
            f[0] = p;
            for (const char* q = p; (q = (const char*)memchr(q, '\t', (size_t)(line_end - q))) != nullptr; ++q) {
                if (tabs < 10) f[tabs + 1] = q + 1;
                ++tabs;
            }
            if (tabs != 10) { ck.err = RT_ESTATE; ck.err_row = row; return; }
            f[11] = line_end + 1;
            if (ck.all_annotated) {   // detect_orfs.py:104-105 tests the whole line for the substring
                static const char kAnn[] = "annotated";
                if (std::search(p, line_end, kAnn, kAnn + 9) != line_end) ck.annotated_prefix++;
                else ck.all_annotated = false;
            }
            // coordinate = start-end[,start-end...] (orf.py:166-170)
            ivs.clear();
            const char* c = f[10];
            while (c < line_end) {
                const char* grp_end = (const char*)memchr(c, ',', (size_t)(line_end - c));
                if (!grp_end) grp_end = line_end;
                const char* dash = (const char*)memchr(c + 1, '-', (size_t)(grp_end - c - 1));   // a leading '-' is a sign
                long long s = 0, e = 0;
                const char* q = c;
                bool ok = dash != nullptr && parse_int(q, dash, s) && q == dash;
                q = dash ? dash + 1 : c;
                ok = ok && parse_int(q, grp_end, e) && q == grp_end;
                if (!ok || s < INT32_MIN || s > INT32_MAX || e < INT32_MIN || e > INT32_MAX) { ck.err = RT_EINVAL; ck.err_row = row; return; }
                ivs.emplace_back(s, e);
                c = grp_end + 1;
            }
            if (ivs.size() > 1)
                std::stable_sort(ivs.begin(), ivs.end(), [](const auto& a, const auto& b) { return a.first < b.first; });   // orf.py:100
            for (auto& iv : ivs) {
                ck.exon_start.push_back((int32_t)iv.first);
                ck.exon_end.push_back((int32_t)iv.second);
            }
            ck.n_exon.push_back((int32_t)ivs.size());
            ck.line_field.push_back((uint64_t)(f[1] - base));
            for (int k = 1; k <= 9; ++k) ck.field_len.push_back((uint32_t)(f[k + 1] - 1 - f[k]));
            std::string chrom(f[7], f[8] - 1);
            auto it = chrom_id.find(chrom);
            if (it == chrom_id.end()) {
                it = chrom_id.emplace(chrom, (int)ck.chrom_names.size()).first;
                ck.chrom_names.push_back(chrom);
            }
            ck.chrom_local.push_back(it->second);
            const size_t slen = (size_t)(f[9] - 1 - f[8]);
            ck.strand.push_back(slen == 1 && *f[8] == '+' ? 0 : slen == 1 && *f[8] == '-' ? 1 : 2);
            p = line_end + 1;
        }
    };
    run_parallel(n_thr, [&](int k) { parse_chunk(chunks[(size_t)k]); });
    // 3. the first error in file order, as the row-by-row loop of the reference would meet it
    {
        int64_t rows_before = 0;
        for (const Chunk& ck : chunks) {
            if (ck.err == RT_ESTATE) {
                g_io_error = "Error: unexpected number of columns found for index file\nplease run ribotricer prepare-orfs to regenerate";
                return RT_ESTATE;
            }
            if (ck.err != RT_OK) {
                g_io_error = "bad coordinate in index row " + std::to_string(rows_before + ck.err_row + 1);
                return ck.err;
            }
            rows_before += (int64_t)ck.n_exon.size();
        }
    }
    // 4. merge: chromosome ids in order of first appearance in the file, columns concatenated by all threads
    std::vector<std::vector<int>> chrom_map(chunks.size());
    {
        std::unordered_map<std::string, int> chrom_id;
        for (size_t k = 0; k < chunks.size(); ++k)
            for (const std::string& name : chunks[k].chrom_names) {
                auto it = chrom_id.find(name);
                if (it == chrom_id.end()) {
                    it = chrom_id.emplace(name, (int)ix->chrom_names.size()).first;
                    ix->chrom_names.push_back(name);
                }
                chrom_map[k].push_back(it->second);
            }
    }
    std::vector<size_t> row0(chunks.size() + 1, 0), exon0(chunks.size() + 1, 0);
    bool in_prefix = true;
    for (size_t k = 0; k < chunks.size(); ++k) {
        row0[k + 1] = row0[k] + chunks[k].n_exon.size();
        exon0[k + 1] = exon0[k] + chunks[k].exon_start.size();
        if (in_prefix) {
            ix->n_annotated_prefix += chunks[k].annotated_prefix;
            in_prefix = chunks[k].all_annotated;
        }
    }
    const size_t n_rows = row0.back(), n_exons = exon0.back();
    if (!(ix->exon_ptr.alloc(n_rows + 1) && ix->exon_start.alloc(n_exons) && ix->exon_end.alloc(n_exons) && ix->orf_chrom.alloc(n_rows) &&
          ix->orf_strand.alloc(n_rows) && ix->field_len.alloc(9 * n_rows) && ix->line_field.alloc(n_rows))) {
        g_io_error = "out of memory";
        return RT_ENOMEM;
    }
    ix->exon_ptr[0] = 0;
    run_parallel(n_thr, [&](int kk) {
        const size_t k = (size_t)kk;
        Chunk& ck = chunks[k];
        const size_t r0 = row0[k], e0 = exon0[k], m = ck.n_exon.size();
        if (!ck.exon_start.empty()) {
            memcpy(ix->exon_start.p + e0, ck.exon_start.data(), 4 * ck.exon_start.size());
            memcpy(ix->exon_end.p + e0, ck.exon_end.data(), 4 * ck.exon_end.size());
        }
        int64_t at = (int64_t)e0;
        for (size_t i = 0; i < m; ++i) {
            at += ck.n_exon[i];
            ix->exon_ptr[r0 + i + 1] = at;
            ix->orf_chrom[r0 + i] = chrom_map[k][(size_t)ck.chrom_local[i]];
        }
        if (m) {
            memcpy(ix->orf_strand.p + r0, ck.strand.data(), m);
            memcpy(ix->field_len.p + 9 * r0, ck.field_len.data(), 4 * 9 * m);
            memcpy(ix->line_field.p + r0, ck.line_field.data(), 8 * m);
        }
        Chunk().exon_start.swap(ck.exon_start);        // give the chunk's memory back early
        Chunk().exon_end.swap(ck.exon_end);
        Chunk().field_len.swap(ck.field_len);
    });
    *out = ix.release();
    return RT_OK;
}

int rt_index_load(const char* path, rt_index** out) {
    if (!path || !out) return RT_EINVAL;
    *out = nullptr;
    std::unique_ptr<rt_index> ix(new rt_index());
    // the file, read in slices by all threads
    if (const int rc = read_file(path, ix->text)) return rc;
    return index_parse(std::move(ix), out);
}

int rt_index_load_text(rt_text* text, const char* path, rt_index** out) {
    if (!text || !path || !out) { rt_text_free(text); return RT_EINVAL; }
    *out = nullptr;
    std::unique_ptr<rt_index> ix(new rt_index());
    adopt_text(text, ix->text);
    return index_parse(std::move(ix), out);
}

void rt_index_free(rt_index* ix) { delete ix; }
int64_t rt_index_n_orf(const rt_index* ix) { return ix ? (int64_t)ix->orf_chrom.size() : 0; }
int64_t rt_index_n_exon(const rt_index* ix) { return ix ? (int64_t)ix->exon_start.size() : 0; }
int64_t rt_index_n_annotated_prefix(const rt_index* ix) { return ix ? ix->n_annotated_prefix : 0; }
int rt_index_n_chrom(const rt_index* ix) { return ix ? (int)ix->chrom_names.size() : 0; }
const char* rt_index_chrom_name(const rt_index* ix, int i) {
    return ix && i >= 0 && i < (int)ix->chrom_names.size() ? ix->chrom_names[i].c_str() : nullptr;
}

int rt_index_copy(const rt_index* ix, int64_t* exon_ptr, int32_t* exon_start, int32_t* exon_end, int32_t* orf_chrom,
                  uint8_t* orf_strand) {
    if (!ix) return RT_EINVAL;
    // one thread per column when the index is large (the destination is usually fresh memory)
    struct Copy { void* dst; const void* src; size_t bytes; };
    std::vector<Copy> big;
    auto copy = [&](void* dst, const void* src, size_t bytes) {
        if (!dst || !bytes) return;
        if (bytes < (1u << 22)) memcpy(dst, src, bytes);
        else big.push_back({dst, src, bytes});
    };
    copy(exon_ptr, ix->exon_ptr.p, 8 * ix->exon_ptr.n);
    copy(exon_start, ix->exon_start.p, 4 * ix->exon_start.n);
    copy(exon_end, ix->exon_end.p, 4 * ix->exon_end.n);
    copy(orf_chrom, ix->orf_chrom.p, 4 * ix->orf_chrom.n);
    copy(orf_strand, ix->orf_strand.p, ix->orf_strand.n);
    run_parallel((int)big.size(), [&](int k) { memcpy(big[(size_t)k].dst, big[(size_t)k].src, big[(size_t)k].bytes); });
    return RT_OK;
}

// Field k (1..9: ORF_type .. start_codon) of row `orf`; not NUL terminated.
const char* rt_index_field(const rt_index* ix, int64_t orf, int k, int* len) {
    if (!ix || orf < 0 || orf >= (int64_t)ix->orf_chrom.size() || k < 1 || k > 9) return nullptr;
    uint64_t off = ix->line_field[orf];
    for (int j = 1; j < k; ++j) off += ix->field_len[9 * orf + (j - 1)] + 1;
    if (len) *len = (int)ix->field_len[9 * orf + (k - 1)];
    return ix->text.data() + off;
}

// Field 0 (ORF_ID) of every row.  A row's first field runs from the end of the previous line (the header's for row 0)
// to the tab before field 1.
int rt_index_ids(const rt_index* ix, int64_t* off, char* blob) {
    if (!ix || !off) return RT_EINVAL;
    const int64_t n = (int64_t)ix->orf_chrom.size();
    off[0] = 0;
    for (int64_t o = 0; o < n; ++o) {
        const char* end = ix->text.data() + ix->line_field[o] - 1;
        const char* p = end;
        while (p > ix->text.data() && p[-1] != '\n') --p;
        if (blob) memcpy(blob + off[o], p, (size_t)(end - p));
        off[o + 1] = off[o] + (end - p);
    }
    return RT_OK;
}

int rt_tsv_open(const char* path, int write_header, rt_tsv** out) {
    if (!path || !out) return RT_EINVAL;
    FILE* fh = fopen(path, "wb");
    if (!fh) { g_io_error = std::string("cannot open ") + path; return RT_EINVAL; }
    rt_tsv* t = new rt_tsv(fh);
    if (write_header)   // detect_orfs.py:241-260
        fputs("ORF_ID\tORF_type\tstatus\tphase_score\tread_count\tlength\tvalid_codons\tvalid_codons_ratio\t"
              "read_density\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\t"
              "start_codon\tprofile\n", fh);
    *out = t;
    return RT_OK;
}

// Rows of the selected ORFs (absolute ids, ascending = index order).  Result columns are indexed by
// (orf - orf_lo); prof_ptr[i]..prof_ptr[i+1] delimit the profile of orf_ids[i] in `prof`.
}  // extern "C"

namespace {

// The re-derived ORF id tid_start_end_len of row o (orf.py:101-103) at p; returns the end.  At most the transcript id
// plus 3 * 21 bytes.
char* put_oid(char* p, const rt_index* ix, int64_t o) {
    int tlen = 0;
    const char* tid = rt_index_field(ix, o, 2, &tlen);
    const int64_t e0 = ix->exon_ptr[o], e1 = ix->exon_ptr[o + 1];
    long long L = 0;
    for (int64_t e = e0; e < e1; ++e) L += (long long)ix->exon_end[e] - ix->exon_start[e] + 1;
    memcpy(p, tid, (size_t)tlen);
    p += tlen;
    *p++ = '_';
    p = put_int(p, e1 > e0 ? ix->exon_start[e0] : 0); *p++ = '_';
    p = put_int(p, e1 > e0 ? ix->exon_end[e1 - 1] : 0); *p++ = '_';
    return put_int(p, L);
}

// Rows [i0, i1) of the selection, formatted as detect_orfs.py:304-323 prints them.
bool format_rows(TextBuf& b, const rt_index* ix, int64_t i0, int64_t i1, const int64_t* orf_ids, int64_t orf_lo,
                 const double* score, const int32_t* valid, const int64_t* count, const int32_t* length,
                 const uint8_t* status, const int64_t* prof_ptr, const int32_t* prof) {
    std::string num;                                     // the three doubles of a row
    for (int64_t i = i0; i < i1; ++i) {
        const int64_t o = orf_ids[i], k = o - orf_lo;
        if (o < 0 || o >= (int64_t)ix->orf_chrom.size() || k < 0 || prof_ptr[i + 1] < prof_ptr[i]) return false;
        int flen[10];
        const char* f[10];
        size_t text = 0;
        for (int j = 1; j <= 9; ++j) {
            f[j] = rt_index_field(ix, o, j, &flen[j]);
            text += (size_t)flen[j];
        }
        const size_t n_prof = (size_t)(prof_ptr[i + 1] - prof_ptr[i]);
        // everything but the profile: the fields (transcript_id twice), 7 integers of <= 20 characters, 3 doubles of <= 25,
        // the status word, tabs and brackets; a profile value takes <= 11 characters and ", "
        char* p = b.need(2 * text + 7 * 21 + 3 * 26 + 64 + 13 * n_prof);
        if (!p) return false;
        auto put = [&](const char* d, int n) { memcpy(p, d, (size_t)n); p += n; };
        auto put_double = [&](double x) {
            num.clear();
            append_repr(num, x);
            put(num.data(), (int)num.size());
        };
        p = put_oid(p, ix, o);
        *p++ = '\t';
        put(f[1], flen[1]); *p++ = '\t';
        if (status[k]) put("translating", 11); else put("nontranslating", 14);
        *p++ = '\t';
        put_double(score[k]); *p++ = '\t';
        p = put_int(p, count[k]); *p++ = '\t';
        p = put_int(p, length[k]); *p++ = '\t';
        p = put_int(p, valid[k]); *p++ = '\t';
        const long long n_codons = length[k] / 3 > 1 ? length[k] / 3 : 1;        // detect_orfs.py:281
        put_double((double)valid[k] / (double)n_codons); *p++ = '\t';             // :285
        put_double((double)count[k] / (double)n_codons); *p++ = '\t';             // :287
        put(f[2], flen[2]); *p++ = '\t';
        put(f[3], flen[3]); *p++ = '\t';
        put(f[4], flen[4]); *p++ = '\t';
        put(f[5], flen[5]); *p++ = '\t';
        put(f[6], flen[6]); *p++ = '\t';
        put(f[7], flen[7]); *p++ = '\t';
        put(f[8], flen[8]); *p++ = '\t';
        if (flen[9] >= 3) put(f[9], 3);                                          // ORF.start_codon (orf.py:108-119): seq[:3],
        else put("None", 4);                                                     //   None when the field holds fewer than 3 characters
        *p++ = '\t';
        *p++ = '[';
        const int32_t* q = prof + prof_ptr[i];
        for (size_t j = 0; j < n_prof; ++j) {
            const int32_t v = q[j];
            if ((uint32_t)v < 10u) *p++ = (char)('0' + v);
            else p = put_int(p, v);
            *p++ = ',';
            *p++ = ' ';
        }
        if (n_prof) p -= 2;
        *p++ = ']';
        *p++ = '\n';
        b.advance_to(p);
    }
    return true;
}

}  // namespace

extern "C" {

int rt_tsv_write(rt_tsv* t, const rt_index* ix, int64_t n_sel, const int64_t* orf_ids, int64_t orf_lo,
                 const double* score, const int32_t* valid, const int64_t* count, const int32_t* length,
                 const uint8_t* status, const int64_t* prof_ptr, const int32_t* prof) {
    if (!t || !ix || n_sel < 0 || (n_sel && (!orf_ids || !score || !valid || !count || !length || !status || !prof_ptr || !prof)))
        return RT_EINVAL;
    // the profile column is most of the text: rows are formatted by several threads in slices balanced by
    // profile length, and handed in order to the file's write-behind thread
    const int64_t total = n_sel ? prof_ptr[n_sel] - prof_ptr[0] : 0;
    const int n_thr = host_threads((size_t)((total + n_sel * 40) / (1 << 21)), 16);
    std::vector<int64_t> cut(n_thr + 1, n_sel);
    cut[0] = 0;
    for (int k = 1; k < n_thr; ++k) {
        const int64_t target = prof_ptr[0] + total * k / n_thr;
        cut[k] = std::lower_bound(prof_ptr, prof_ptr + n_sel, target) - prof_ptr;
        if (cut[k] < cut[k - 1]) cut[k] = cut[k - 1];
    }
    std::vector<TextBuf> parts(n_thr);
    std::vector<char> ok(n_thr, 1);
    run_parallel(n_thr, [&](int k) {
        ok[k] = format_rows(parts[k], ix, cut[k], cut[k + 1], orf_ids, orf_lo, score, valid, count, length, status, prof_ptr, prof);
    });
    for (int k = 0; k < n_thr; ++k)
        if (!ok[k]) { g_io_error = "rt_tsv_write: ORF id outside the index or the result range, or out of memory"; return RT_EINVAL; }
    for (int k = 0; k < n_thr; ++k)
        if (!t->out.put(std::move(parts[k]))) { g_io_error = "rt_tsv_write: write failed"; return RT_EINVAL; }
    return RT_OK;
}

int rt_tsv_close(rt_tsv* t) {
    if (!t) return RT_EINVAL;
    const bool wrote = t->out.finish();
    const int rc = fclose(t->fh);
    delete t;
    if (!wrote || rc != 0) g_io_error = "write failed (disk full?)";
    return wrote && rc == 0 ? RT_OK : RT_EINVAL;
}

// For tests: Python-style repr of a double into buf (NUL terminated).
int rt_repr_double(double x, char* buf, int cap) {
    std::string s;
    append_repr(s, x);
    if ((int)s.size() + 1 > cap) return RT_EINVAL;
    memcpy(buf, s.c_str(), s.size() + 1);
    return (int)s.size();
}

}  // extern "C"

// ---- metagene sums (metagene.py:204-252) ---------------------------------------------------------------
// Row i of the ragged matrix flat[ptr[i] .. ptr[i+1]) is the coverage of one annotated ORF over its first <= width
// positions (leader included).  A row with reads is divided by its mean (metagene.py:214-219) and added, position by
// position, to the start-aligned sums and -- re-indexed to END at the last column (metagene.py:140-155) -- to the
// stop-aligned sums; the counts say how many rows reach a column.  Rows are summed in blocks of 2,048 by all cores and the
// block sums are added in block order, so the result does not depend on the number of threads.
extern "C" int rt_metagene_sums(const int32_t* flat, const int64_t* ptr, int64_t n_rows, int64_t width, double* start_sum,
                                int64_t* start_cnt, double* stop_sum, int64_t* stop_cnt) {
    if (n_rows < 0 || width < 0 || !ptr || !start_sum || !start_cnt || !stop_sum || !stop_cnt || (n_rows && ptr[n_rows] > ptr[0] && !flat))
        return RT_EINVAL;
    for (int64_t i = 0; i < n_rows; ++i)
        if (ptr[i + 1] < ptr[i] || ptr[i + 1] - ptr[i] > width) { g_io_error = "rt_metagene_sums: a row is longer than the matrix is wide"; return RT_EINVAL; }
    const int64_t kBlock = 2048, n_blocks = (n_rows + kBlock - 1) / kBlock, w = width;
    std::vector<double> sums((size_t)(n_blocks * 2 * w), 0.0);
    std::vector<int64_t> cnts((size_t)(n_blocks * 2 * w), 0);
    claim_parallel(host_threads((size_t)n_blocks, 16), (size_t)n_blocks, [&](size_t bb) {
        const int64_t b = (int64_t)bb;
        double* s5 = sums.data() + (size_t)(b * 2 * w);
        double* s3 = s5 + w;
        int64_t* c5 = cnts.data() + (size_t)(b * 2 * w);
        int64_t* c3 = c5 + w;
        for (int64_t i = b * kBlock; i < std::min(n_rows, (b + 1) * kBlock); ++i) {
            const int32_t* row = flat + ptr[i];
            const int64_t len = ptr[i + 1] - ptr[i];
            long long total = 0;
            for (int64_t k = 0; k < len; ++k) total += row[k];
            if (len == 0) continue;
            const double mean = (double)total / (double)len;
            if (!(mean > 0)) continue;                       // metagene.py:216: ORFs without reads are skipped
            const int64_t shift = w - len;
            for (int64_t k = 0; k < len; ++k) {
                const double v = (double)row[k] / mean;
                s5[k] += v;
                s3[shift + k] += v;
                c5[k]++;
                c3[shift + k]++;
            }
        }
    });
    for (int64_t k = 0; k < w; ++k) { start_sum[k] = stop_sum[k] = 0.0; start_cnt[k] = stop_cnt[k] = 0; }
    for (int64_t b = 0; b < n_blocks; ++b) {
        const double* s5 = sums.data() + (size_t)(b * 2 * w);
        const int64_t* c5 = cnts.data() + (size_t)(b * 2 * w);
        for (int64_t k = 0; k < w; ++k) {
            start_sum[k] += s5[k];
            stop_sum[k] += s5[w + k];
            start_cnt[k] += c5[k];
            stop_cnt[k] += c5[w + k];
        }
    }
    return RT_OK;
}

// ---- WIG writer (detect_orfs.py:327-351): one "variableStep chrom=" block per call ------------------
extern "C" {

int rt_wig_open(const char* path, rt_tsv** out) { return rt_tsv_open(path, 0, out); }

int rt_wig_block(rt_tsv* t, const char* chrom, int64_t n, const int64_t* pos, const int32_t* count) {
    if (!t || !chrom || n < 0 || (n && (!pos || !count))) return RT_EINVAL;
    // "pos<TAB>count<NL>" lines of [lo, hi): at most 20 + 11 + 2 characters each
    auto lines = [&](TextBuf& o, int64_t lo, int64_t hi) {
        char* p = o.need((size_t)(hi - lo) * 33);
        if (!p) return false;
        for (int64_t i = lo; i < hi; ++i) {
            p = put_int(p, pos[i]);
            *p++ = '\t';
            p = put_int(p, count[i]);
            *p++ = '\n';
        }
        o.advance_to(p);
        return true;
    };
    TextBuf head;
    const std::string title = std::string("variableStep chrom=") + chrom + "\n";
    head.append(title.data(), title.size());
    // a long block (a human chromosome holds millions of covered positions) is formatted by several threads, a slice of
    // the block each; the pieces go to the write-behind thread in order
    const int n_thr = host_threads((size_t)(n >> 16), 16);
    if (n_thr == 1) {
        if (!lines(head, 0, n) || !t->out.put(std::move(head))) return RT_EINVAL;
        return RT_OK;
    }
    std::vector<TextBuf> part((size_t)n_thr);
    std::vector<char> ok((size_t)n_thr, 1);
    run_parallel(n_thr, [&](int k) { ok[(size_t)k] = lines(part[(size_t)k], n * k / n_thr, n * (k + 1) / n_thr); });
    for (char c : ok)
        if (!c) return RT_EINVAL;
    if (!t->out.put(std::move(head))) return RT_EINVAL;
    for (TextBuf& o : part)
        if (!t->out.put(std::move(o))) return RT_EINVAL;
    return RT_OK;
}

int rt_wig_close(rt_tsv* t) { return rt_tsv_close(t); }

}  // extern "C"

// ---- record stream (4 B/read, format in ribotricer_b200.h): delta code of a coordinate-sorted library ----
namespace {

struct StreamWriter {
    uint32_t* rec;          // NULL: count only
    int32_t* hdr;
    int64_t cap;
    int64_t nb = 0;         // blocks opened so far
    int fill = RT_STREAM_BLOCK;   // records in the open block (RT_STREAM_BLOCK: none open)
    bool open(int32_t rid, int32_t at) {
        if (rec && nb > 0)
            for (int k = fill; k < RT_STREAM_BLOCK; ++k) rec[(nb - 1) * RT_STREAM_BLOCK + k] = RT_STREAM_NULL;
        if (rec && nb >= cap) return false;
        if (rec) {
            hdr[4 * nb] = rid;
            hdr[4 * nb + 1] = at;
            hdr[4 * nb + 2] = hdr[4 * nb + 3] = 0;
        }
        ++nb;
        fill = 0;
        return true;
    }
    void put(uint32_t w) {
        if (rec) rec[(nb - 1) * RT_STREAM_BLOCK + fill] = w;
        ++fill;
    }
    void close() {
        if (rec && nb > 0)
            for (int k = fill; k < RT_STREAM_BLOCK; ++k) rec[(nb - 1) * RT_STREAM_BLOCK + k] = RT_STREAM_NULL;
        fill = RT_STREAM_BLOCK;
    }
};

}  // namespace

// The usual group of a sorted library: kStreamGroup reads of one reference, each 0..32767 nt after the one before, none
// spliced or longer than 255.  Two branch-free loops the compiler vectorises (AVX2 clone picked at load time): the
// test, then one record per read.
constexpr int kStreamGroup = 64;

#if defined(__x86_64__) && defined(__GNUC__) && !defined(__clang__)
__attribute__((target_clones("avx2", "default")))
#endif
bool rt_stream_group_plain(const int32_t* __restrict__ ref_id, const int32_t* __restrict__ first, const int32_t* __restrict__ last,
                           const uint16_t* __restrict__ mlen, int32_t cur_ref, int64_t cur_pos) {
    const int64_t d0 = (int64_t)first[0] - cur_pos;
    uint32_t bad = (d0 < 0) | (d0 > 32767);
    for (int k = 1; k < kStreamGroup; ++k) bad |= (uint32_t)((uint32_t)first[k] - (uint32_t)first[k - 1]) > 32767u;
    for (int k = 0; k < kStreamGroup; ++k)
        bad |= (uint32_t)(ref_id[k] ^ cur_ref) | (uint32_t)(mlen[k] > 255) | (uint32_t)(last[k] - first[k] + 1 - (int32_t)mlen[k]);
    return bad == 0;
}

// The same test fused with the coding: `out` receives the group's records whether or not the group turns out plain
// (the caller only keeps them when it does), so every column is read once.
#if defined(__x86_64__) && defined(__GNUC__) && !defined(__clang__)
__attribute__((target_clones("avx2", "default")))
#endif
bool rt_stream_group_code(const int32_t* __restrict__ ref_id, const int32_t* __restrict__ first, const int32_t* __restrict__ last,
                          const uint16_t* __restrict__ mlen, const uint16_t* __restrict__ flag, const uint8_t* __restrict__ mapq,
                          const uint8_t* __restrict__ nh, int32_t cur_ref, int64_t cur_pos, uint32_t* __restrict__ out) {
    const int64_t d0 = (int64_t)first[0] - cur_pos;
    uint32_t delta[kStreamGroup];
    alignas(16) uint32_t rec[kStreamGroup];
    delta[0] = (uint32_t)d0;
    for (int k = 1; k < kStreamGroup; ++k) delta[k] = (uint32_t)first[k] - (uint32_t)first[k - 1];
    uint32_t bad = (d0 < 0) | (d0 > 32767);
    for (int k = 0; k < kStreamGroup; ++k) {
        const uint32_t f = flag[k], nn = nh[k], qq = mapq[k], l = mlen[k];
        const uint32_t state = nn == 0u ? (uint32_t)(qq == 255u) : 3u - (uint32_t)(nn == 1u);
        const uint32_t meta = ((f >> 2) & 1u) | ((f >> 7) & 0xeu) | (f & 0x10u) | (state << 5);
        bad |= (uint32_t)(delta[k] > 32767u) | (uint32_t)(ref_id[k] ^ cur_ref) | (uint32_t)(l > 255u) | (uint32_t)(last[k] - first[k] + 1 - (int32_t)l);
        rec[k] = delta[k] | (l << 16) | (meta << 24);
    }
#if defined(__x86_64__)
    if ((reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        // the staging buffer is written once and read by the copy engine: streaming stores keep it out of the caches
        // and spare the read-for-ownership of every line (rt_stream_pack_range fences before it returns)
        for (int k = 0; k < kStreamGroup; k += 4)
            _mm_stream_si128(reinterpret_cast<__m128i*>(out + k), _mm_load_si128(reinterpret_cast<const __m128i*>(rec + k)));
        return bad == 0;
    }
#endif
    memcpy(out, rec, sizeof rec);
    return bad == 0;
}

// Reads [0, m) of the decoder's columns as one run of stream blocks.  Returns the number of blocks, -1 when the
// reads cannot be coded (a span beyond the extension's 22 bits), -2 when `cap` blocks are not enough.  rec == NULL
// counts only.  Positions that descend inside a reference cost a block each.
int64_t rt_stream_pack_range(const int32_t* __restrict__ ref_id, const int32_t* __restrict__ first, const int32_t* __restrict__ last,
                             const uint16_t* __restrict__ mlen, const uint16_t* __restrict__ flag, const uint8_t* __restrict__ mapq,
                             const uint8_t* __restrict__ nh, int64_t m, uint32_t* rec, int32_t* hdr, int64_t cap) {
    StreamWriter w{rec, hdr, cap};
    int32_t cur_ref = m > 0 ? ref_id[0] : 0;
    int64_t cur_pos = m > 0 ? first[0] : 0;
    int64_t i = 0;
    // A core streams only ~12 GB/s through its L1 miss buffers; prefetches into L2 run ahead of them (measured on the
    // GPU box: 10 % off the coding time at 512 reads, nothing more further out).
    constexpr int64_t ahead_reads = 512;
    while (i < m) {
        if (i + ahead_reads + kStreamGroup <= m) {   // one 64-read group of every column, `ahead_reads` further on
            const int64_t a = i + ahead_reads;
            for (int k = 0; k < 4; ++k) {
                __builtin_prefetch(ref_id + a + 16 * k, 0, 2);
                __builtin_prefetch(first + a + 16 * k, 0, 2);
                __builtin_prefetch(last + a + 16 * k, 0, 2);
            }
            __builtin_prefetch(mlen + a, 0, 2); __builtin_prefetch(mlen + a + 32, 0, 2);
            __builtin_prefetch(flag + a, 0, 2); __builtin_prefetch(flag + a + 32, 0, 2);
            __builtin_prefetch(mapq + a, 0, 2);
            __builtin_prefetch(nh + a, 0, 2);
        }
        if (i + kStreamGroup <= m && w.fill == RT_STREAM_BLOCK) {     // start the next block here: the group may well be plain
            if (!(flag[i] & 0x704u)) {      // (a read the flags decide may carry any position: it must not become the block's)
                cur_ref = ref_id[i];
                cur_pos = first[i];
            }
            if (!w.open(cur_ref, (int32_t)cur_pos)) return -2;
        }
        if (i + kStreamGroup <= m && w.fill + kStreamGroup <= RT_STREAM_BLOCK &&
            (rec ? rt_stream_group_code(ref_id + i, first + i, last + i, mlen + i, flag + i, mapq + i, nh + i, cur_ref, cur_pos,
                                        rec + (w.nb - 1) * RT_STREAM_BLOCK + w.fill)
                 : rt_stream_group_plain(ref_id + i, first + i, last + i, mlen + i, cur_ref, cur_pos))) {
            w.fill += kStreamGroup;
            i += kStreamGroup;
            cur_pos = first[i - 1];
            continue;
        }
        const int64_t stop = std::min<int64_t>(m, i + kStreamGroup);
        for (; i < stop; ++i) {
            const unsigned f = flag[i];
            const unsigned nn = nh[i], qq = mapq[i];
            const unsigned state = nn == 0u ? (qq == 255u ? RT_STREAM_NH_ABSENT_MAPQ255 : RT_STREAM_NH_ABSENT)
                                            : (nn == 1u ? RT_STREAM_NH_ONE : RT_STREAM_NH_OTHER);
            // SAM 0x4 -> bit 0, 0x100 / 0x200 / 0x400 -> bits 1-3, 0x10 stays bit 4
            const unsigned meta = ((f >> 2) & 1u) | ((f >> 7) & 0xeu) | (f & 0x10u) | (state << 5);
            if (f & 0x704u) {      // the flags decide (bam.py:77-88): the reference never looks at position or length
                if (w.fill == RT_STREAM_BLOCK && !w.open(cur_ref, (int32_t)cur_pos)) return -2;
                w.put(meta << 24);
                continue;
            }
            const int32_t rid = ref_id[i];
            const int64_t at = first[i];
            const unsigned l = mlen[i];
            const int64_t extra = (int64_t)last[i] - at + 1 - (int64_t)l;
            int64_t d = at - cur_pos;
            const unsigned ext = (l > 255u) | (extra != 0);
            if (extra < 0 || extra >= (1 << 22)) return -1;
            // a read that starts before its predecessor (a CIGAR that opens with D or N, or a library that is not sorted
            // after all) starts a block of its own; the callers give up when that happens too often
            bool fresh = w.fill == RT_STREAM_BLOCK || rid != cur_ref || d >= (1ll << 30) || d < 0;
            if (!fresh) fresh = w.fill + 1 + (int)(d > 32767) + (int)ext > RT_STREAM_BLOCK;
            if (fresh) {
                if (!w.open(rid, (int32_t)at)) return -2;
                cur_ref = rid;
                d = 0;
            }
            if (d > 32767) {
                w.put(RT_STREAM_SPECIAL | ((uint32_t)(d & 0xffff) << 16) | (uint32_t)(d >> 16));
                d = 0;
            }
            w.put((uint32_t)d | ((l & 255u) << 16) | ((meta | (ext ? RT_STREAM_EXT : 0u)) << 24));
            if (ext) w.put(RT_STREAM_SPECIAL | RT_STREAM_KIND_EXT | (l >> 8) | ((uint32_t)(extra >> 16) << 8) | ((uint32_t)(extra & 0xffff) << 16));
            cur_pos = at;
        }
    }
    w.close();
#if defined(__x86_64__)
    _mm_sfence();       // the streaming stores of rt_stream_group_code, before anyone is told the records are there
#endif
    return w.nb;
}

extern "C" {

int rt_stream_pack(int64_t n, const int32_t* ref_id, const int32_t* first, const int32_t* last, const uint16_t* mlen,
                   const uint16_t* flag, const uint8_t* mapq, const uint8_t* nh, int n_threads, int64_t cap_blocks,
                   uint32_t* records, int32_t* hdr, int64_t* n_blocks) {
    if (n < 0 || !n_blocks || (n > 0 && (!ref_id || !first || !last || !mlen || !flag || !mapq || !nh)) || (records && !hdr))
        return RT_EINVAL;
    const int64_t n_ranges = (n + RT_STREAM_RANGE - 1) / RT_STREAM_RANGE;
    n_threads = n_threads > 0 ? (int)std::max<int64_t>(1, std::min<int64_t>(n_threads, n_ranges)) : host_threads((size_t)n_ranges, SIZE_MAX);
    std::vector<int64_t> blocks(n_ranges + 1, 0);
    auto sweep = [&](bool write) {
        std::atomic<int64_t> worst{0};
        claim_parallel(n_threads, (size_t)n_ranges, [&](size_t rr) {
            const int64_t r = (int64_t)rr;
            const int64_t at = r * RT_STREAM_RANGE, m = std::min<int64_t>(RT_STREAM_RANGE, n - at);
            int64_t got;
            if (write)
                got = rt_stream_pack_range(ref_id + at, first + at, last + at, mlen + at, flag + at, mapq + at, nh + at, m,
                                           records + blocks[r] * RT_STREAM_BLOCK, hdr + 4 * blocks[r], blocks[r + 1] - blocks[r]);
            else
                got = blocks[r + 1] = rt_stream_pack_range(ref_id + at, first + at, last + at, mlen + at, flag + at, mapq + at,
                                                           nh + at, m, nullptr, nullptr, 0);
            if (got < 0) {
                int64_t seen = worst.load();
                while (got < seen && !worst.compare_exchange_weak(seen, got)) {}
            }
        });
        return worst.load();
    };
    if (sweep(false) < 0) {
        g_io_error = "rt_stream_pack: the library cannot be delta-coded (a read spans 2^22 nt more than it matches); use the column "
                     "entry points";
        return RT_ESTATE;
    }
    for (int64_t r = 0; r < n_ranges; ++r) blocks[r + 1] += blocks[r];     // counts -> exclusive offsets
    // every descent of the positions costs a block: a library that is not coordinate-sorted would be mostly padding
    if (blocks[n_ranges] * RT_STREAM_BLOCK > 2 * n + 1024 * RT_STREAM_BLOCK * n_ranges) {       // (small libraries may be mostly padding)
        g_io_error = "rt_stream_pack: the stream would be more than half padding (the library is not coordinate-sorted); use the "
                     "column entry points";
        return RT_ESTATE;
    }
    *n_blocks = blocks[n_ranges];
    if (!records) return RT_OK;
    if (cap_blocks < blocks[n_ranges]) {
        g_io_error = "rt_stream_pack: cap_blocks is smaller than the stream (call with h_records = NULL for the size)";
        return RT_EINVAL;
    }
    if (sweep(true) < 0) return RT_ESTATE;
    return RT_OK;
}

}  // extern "C"

// ---- count-orfs-codon, host side (DESIGN.md section 11) ------------------------------------------------------------
// rt_codon_load_tsv selects the rows of a detected-ORFs TSV and matches them to the index, rt_codon_load_seq checks the
// orfs-seq nucleotide file against the index, rt_codon_write formats the tables the device computed.

struct rt_codon {
    HostArr<char> tsv;                   // the detected-ORFs TSV; profiles and gene keys point into it
    HostArr<char> seq;                   // the orfs-seq file (rt_codon_load_seq)
    std::vector<int64_t> row, line, prof_off, prof_len;   // per selected TSV row
    std::vector<int32_t> gene, gseq;
    std::vector<int64_t> gene_key;       // per gene: offset of "gene_id\tgene_name" in tsv
    std::vector<int32_t> gene_id_len, gene_key_len;
    int64_t n_gseq = 0, n_lines = 0;
    std::vector<int64_t> seq_off;        // per index row: offset of its letters in seq
};

namespace {

inline bool ws(char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '\v' || c == '\f'; }

// ORF_ID -> index row for the rows whose ORF_type is wanted; a later duplicate replaces an earlier one.  Open addressing
// over the oid hashes; a probe compares the oid formed again from the index.
struct OidTable {
    const rt_index* ix = nullptr;
    std::vector<uint64_t> hash;          // per index row (0: not a candidate)
    std::vector<int64_t> slot;           // row + 1, 0 empty
    uint64_t mask = 0;
    static uint64_t hash_of(const char* p, size_t n) {
        uint64_t h = std::hash<std::string_view>()(std::string_view(p, n));
        return h | 1;                    // 0 marks a row that is not a candidate
    }
    bool same(int64_t o, const char* p, size_t n) const {
        char buf[1 << 12];
        int tlen = 0;
        rt_index_field(ix, o, 2, &tlen);
        if ((size_t)tlen + 70 > sizeof buf) {
            std::string big((size_t)tlen + 70, '\0');
            const size_t m = (size_t)(put_oid(&big[0], ix, o) - big.data());
            return m == n && memcmp(big.data(), p, n) == 0;
        }
        const size_t m = (size_t)(put_oid(buf, ix, o) - buf);
        return m == n && memcmp(buf, p, n) == 0;
    }
    void build(const rt_index* index, const std::vector<std::string>& features) {
        ix = index;
        const int64_t n = (int64_t)ix->orf_chrom.size();
        hash.assign((size_t)n, 0);
        std::atomic<int64_t> n_cand{0};
        const int64_t block = 1 << 14;
        claim_parallel(host_threads((size_t)(n / block + 1), 16), (size_t)((n + block - 1) / block), [&](size_t bk) {
            std::string buf;
            int64_t cand = 0;
            for (int64_t o = (int64_t)bk * block; o < std::min(n, (int64_t)(bk + 1) * block); ++o) {
                int len = 0;
                const char* type = rt_index_field(ix, o, 1, &len);
                bool want = false;
                for (const std::string& f : features) want = want || (f.size() == (size_t)len && memcmp(f.data(), type, (size_t)len) == 0);
                if (!want) continue;
                int tlen = 0;
                rt_index_field(ix, o, 2, &tlen);
                buf.resize((size_t)tlen + 70);
                const size_t m = (size_t)(put_oid(&buf[0], ix, o) - buf.data());
                hash[(size_t)o] = hash_of(buf.data(), m);
                ++cand;
            }
            n_cand += cand;
        });
        uint64_t cap = 16;
        while (cap < 2 * (uint64_t)n_cand.load()) cap <<= 1;
        slot.assign(cap, 0);
        mask = cap - 1;
        std::string buf;
        for (int64_t o = 0; o < n; ++o) {
            if (!hash[(size_t)o]) continue;
            int tlen = 0;
            rt_index_field(ix, o, 2, &tlen);
            buf.resize((size_t)tlen + 70);
            const size_t m = (size_t)(put_oid(&buf[0], ix, o) - buf.data());
            for (uint64_t s = hash[(size_t)o] & mask;; s = (s + 1) & mask) {
                const int64_t r = slot[s] - 1;
                if (r < 0 || (hash[(size_t)r] == hash[(size_t)o] && same(r, buf.data(), m))) { slot[s] = o + 1; break; }
            }
        }
    }
    int64_t find(const char* p, size_t n) const {
        const uint64_t h = hash_of(p, n);
        for (uint64_t s = h & mask;; s = (s + 1) & mask) {
            const int64_t r = slot[s] - 1;
            if (r < 0) return -1;
            if (hash[(size_t)r] == h && same(r, p, n)) return r;
        }
    }
};

// Python's repr of S1 / n, the correctly rounded quotient of two integers (n > 0).
double exact_ratio(uint64_t s1, uint64_t n) {
    if (s1 < (1ull << 53) && n < (1ull << 53)) return (double)s1 / (double)n;
    // a quotient of at least 55 bits, its last bit set when the division is inexact, then one rounding to 53 bits
    const int bits_s = 64 - __builtin_clzll(s1), bits_n = 64 - __builtin_clzll(n);
    const int shift = std::max(0, 55 + bits_n - bits_s);
    const unsigned __int128 num = (unsigned __int128)s1 << shift;
    const unsigned __int128 q = num / n;
    const uint64_t sticky = num % n != 0;
    return std::ldexp((double)(uint64_t)(q | sticky), -shift);
}

// One row of a table: occurrences, total, mean, median, var (rule 9).  cell = n, S1, S2 low, S2 high, middle sum.
void put_stats(TextBuf& b, const uint64_t* cell, std::string& num) {
    const uint64_t n = cell[0], s1 = cell[1];
    const unsigned __int128 s2 = (unsigned __int128)cell[3] << 64 | cell[2];
    const unsigned __int128 var_num = (unsigned __int128)n * s2 - (unsigned __int128)s1 * s1;
    const unsigned __int128 var_den = (unsigned __int128)n * n;
    num.clear();
    append_repr(num, exact_ratio(s1, n));
    num += '\t';
    append_repr(num, (double)cell[4] / 2.0);
    num += '\t';
    append_repr(num, (double)var_num / (double)var_den);
    char* p = b.need(2 * 21 + num.size() + 4);
    if (!p) return;
    p = put_int(p, (long long)n); *p++ = '\t';
    p = put_int(p, (long long)s1); *p++ = '\t';
    memcpy(p, num.data(), num.size());
    p += num.size();
    *p++ = '\n';
    b.advance_to(p);
}

void put_codon(TextBuf& b, int c) {
    if (char* p = b.need(4)) {
        p[0] = "ACGT"[c >> 4]; p[1] = "ACGT"[(c >> 2) & 3]; p[2] = "ACGT"[c & 3]; p[3] = '\t';
        b.advance_to(p + 4);
    }
}

}  // namespace

extern "C" {

// rt_codon_load_tsv and rt_codon_load_tsv_text once h->tsv holds the file; `path` names it in messages
static int codon_parse_tsv(std::unique_ptr<rt_codon> h, const rt_index* ix, const char* path, int n_features,
                           const char* const* features, int report_all, rt_codon** out) {
    std::vector<std::string> feats;
    for (int k = 0; k < n_features; ++k) feats.emplace_back(features[k] ? features[k] : "");
    OidTable oids;
    oids.build(ix, feats);
    auto wanted = [&](const char* p, size_t n) {
        for (const std::string& f : feats)
            if (f.size() == n && memcmp(f.data(), p, n) == 0) return true;
        return false;
    };
    const char* base = h->tsv.data();
    const size_t size = h->tsv.size();
    const char* end = base + size;
    const char* body = (const char*)memchr(base, '\n', size);   // the first line is skipped, as count_orfs does
    body = body ? body + 1 : end;
    const int n_thr = host_threads(size >> 22, 16, "RT_CODON_THREADS");

    // 1. line-aligned chunks: fields, selection, ORF_ID lookup, gene keys interned per chunk
    struct Chunk {
        const char *lo, *hi;
        std::vector<int64_t> row, line, prof_off, prof_len;
        std::vector<int32_t> gene, gseq;
        std::vector<std::string_view> genes;            // "gene_id\tgene_name", first appearance within the chunk
        std::vector<uint64_t> gseqs;                    // local gene << 32 | chrom << 2 | strand
        int64_t lines = 0;
        int err = 0;                                    // 1: field count, 2: unknown ORF_ID; at local line err_line
        int64_t err_line = 0, err_fields = 0;
        std::string_view err_id;
    };
    std::vector<Chunk> chunks((size_t)n_thr);
    const std::vector<const char*> cut = cut_lines(body, end, n_thr);
    run_parallel(n_thr, [&](int k) {
        Chunk& ck = chunks[(size_t)k];
        std::unordered_map<std::string_view, int32_t> gene_id;
        std::unordered_map<uint64_t, int32_t> gseq_id;
        for (const char* p = cut[(size_t)k]; p < cut[(size_t)k + 1]; ++ck.lines) {
            const char* eol = (const char*)memchr(p, '\n', (size_t)(cut[(size_t)k + 1] - p));
            const char* lo = p;
            const char* hi = eol ? eol : cut[(size_t)k + 1];
            p = hi + 1;
            while (lo < hi && ws(*lo)) ++lo;                 // line.strip()
            while (hi > lo && ws(hi[-1])) --hi;
            const char* f[19];
            int n_f = 1;
            f[0] = lo;
            for (const char* q = lo; (q = (const char*)memchr(q, '\t', (size_t)(hi - q))) != nullptr; ++q) {
                if (n_f < 18) f[n_f] = q + 1;
                ++n_f;
            }
            if (n_f != 18) { ck.err = 1; ck.err_line = ck.lines; ck.err_fields = n_f; return; }
            f[18] = hi + 1;
            auto len = [&](int j) { return (size_t)(f[j + 1] - 1 - f[j]); };
            if (!wanted(f[1], len(1))) continue;
            if (!report_all && len(2) == 14 && memcmp(f[2], "nontranslating", 14) == 0) continue;
            const int64_t o = oids.find(f[0], len(0));
            if (o < 0) { ck.err = 2; ck.err_line = ck.lines; ck.err_id = std::string_view(f[0], len(0)); return; }
            const std::string_view key(f[11], (size_t)(f[13] - 1 - f[11]));
            auto g = gene_id.emplace(key, (int32_t)ck.genes.size());
            if (g.second) ck.genes.push_back(key);
            const uint64_t sk = (uint64_t)g.first->second << 32 | (uint64_t)ix->orf_chrom[o] << 2 | ix->orf_strand[o];
            auto s = gseq_id.emplace(sk, (int32_t)ck.gseqs.size());
            if (s.second) ck.gseqs.push_back(sk);
            ck.row.push_back(o);
            ck.line.push_back(ck.lines);
            ck.prof_off.push_back(f[17] - base);
            ck.prof_len.push_back(len(17));
            ck.gene.push_back(g.first->second);
            ck.gseq.push_back(s.first->second);
        }
    });
    // 2. the first error in file order; line 1 is the header
    int64_t lines_before = 2;
    for (const Chunk& ck : chunks) {
        if (ck.err == 1) {
            g_io_error = std::string(path) + " line " + std::to_string(lines_before + ck.err_line) + ": " +
                         std::to_string(ck.err_fields) + " tab-separated fields, 18 expected";
            return RT_EINVAL;
        }
        if (ck.err == 2) {
            g_io_error = std::string(path) + " line " + std::to_string(lines_before + ck.err_line) + ": ORF_ID " +
                         std::string(ck.err_id.substr(0, 200)) + " is not in the index with an ORF_type of the features";
            return RT_EINVAL;
        }
        lines_before += ck.lines;
    }
    h->n_lines = lines_before - 2;
    // 3. merge in file order: gene and (gene, chrom, strand) ids follow first appearance
    std::unordered_map<std::string_view, int32_t> gene_id;
    std::unordered_map<uint64_t, int32_t> gseq_id;
    std::vector<std::vector<int32_t>> gene_map(chunks.size()), gseq_map(chunks.size());
    size_t n_sel = 0;
    for (size_t k = 0; k < chunks.size(); ++k) {
        for (const std::string_view& key : chunks[k].genes) {
            auto g = gene_id.emplace(key, (int32_t)h->gene_key.size());
            if (g.second) {
                h->gene_key.push_back(key.data() - base);
                h->gene_key_len.push_back((int32_t)key.size());
                h->gene_id_len.push_back((int32_t)(std::find(key.begin(), key.end(), '\t') - key.begin()));
            }
            gene_map[k].push_back(g.first->second);
        }
        for (uint64_t sk : chunks[k].gseqs) {
            const uint64_t gk = (uint64_t)gene_map[k][(size_t)(sk >> 32)] << 32 | (sk & 0xffffffffu);
            auto s = gseq_id.emplace(gk, (int32_t)gseq_id.size());
            gseq_map[k].push_back(s.first->second);
        }
        n_sel += chunks[k].row.size();
    }
    h->n_gseq = (int64_t)gseq_id.size();
    h->row.resize(n_sel); h->line.resize(n_sel); h->prof_off.resize(n_sel); h->prof_len.resize(n_sel);
    h->gene.resize(n_sel); h->gseq.resize(n_sel);
    std::vector<size_t> sel0(chunks.size() + 1, 0);
    std::vector<int64_t> line0(chunks.size() + 1, 2);
    for (size_t k = 0; k < chunks.size(); ++k) {
        sel0[k + 1] = sel0[k] + chunks[k].row.size();
        line0[k + 1] = line0[k] + chunks[k].lines;
    }
    run_parallel(n_thr, [&](int kk) {
        const size_t k = (size_t)kk, s0 = sel0[k];
        const Chunk& ck = chunks[k];
        for (size_t i = 0; i < ck.row.size(); ++i) {
            h->row[s0 + i] = ck.row[i];
            h->line[s0 + i] = line0[k] + ck.line[i];
            h->prof_off[s0 + i] = ck.prof_off[i];
            h->prof_len[s0 + i] = ck.prof_len[i];
            h->gene[s0 + i] = gene_map[k][(size_t)ck.gene[i]];
            h->gseq[s0 + i] = gseq_map[k][(size_t)ck.gseq[i]];
        }
    });
    *out = h.release();
    return RT_OK;
}

int rt_codon_load_tsv(const rt_index* ix, const char* path, int n_features, const char* const* features, int report_all,
                      rt_codon** out) {
    if (!ix || !path || !out || n_features < 0 || (n_features && !features)) return RT_EINVAL;
    *out = nullptr;
    std::unique_ptr<rt_codon> h(new rt_codon());
    if (const int rc = read_file(path, h->tsv)) return rc;
    return codon_parse_tsv(std::move(h), ix, path, n_features, features, report_all, out);
}

int rt_codon_load_tsv_text(const rt_index* ix, rt_text* text, const char* path, int n_features, const char* const* features,
                           int report_all, rt_codon** out) {
    if (!ix || !text || !path || !out || n_features < 0 || (n_features && !features)) { rt_text_free(text); return RT_EINVAL; }
    *out = nullptr;
    std::unique_ptr<rt_codon> h(new rt_codon());
    adopt_text(text, h->tsv);
    return codon_parse_tsv(std::move(h), ix, path, n_features, features, report_all, out);
}

// rt_codon_load_seq and rt_codon_load_seq_text once h->seq holds the file; `path` names it in messages
static int codon_parse_seq(rt_codon* h, const rt_index* ix, const char* path) {
    const char* text = h->seq.data();
    const int64_t size = (int64_t)h->seq.size();
    const int64_t n = (int64_t)ix->orf_chrom.size();
    const std::string where = std::string(path) + " line ";
    const char* hint = "; was it written by orfs-seq from this index, without --protein?";
    static const char kHeader[] = "ORF_ID\tsequence";
    const char* nl = (const char*)memchr(text, '\n', (size_t)size);
    const int64_t head_end = nl ? nl - text : size;
    if (head_end != (int64_t)sizeof kHeader - 1 || memcmp(text, kHeader, sizeof kHeader - 1) != 0) {
        g_io_error = where + "1: the header is not ORF_ID<tab>sequence" + hint;
        return RT_EINVAL;
    }
    // every line's place is known from the index: row k is id, tab, length letters, newline at line_off[k]
    std::vector<int64_t> id_off((size_t)n + 1), L((size_t)n), line_off((size_t)n + 1);
    rt_index_ids(ix, id_off.data(), nullptr);
    line_off[0] = head_end + 1;
    for (int64_t k = 0; k < n; ++k) {
        int64_t len = 0;
        for (int64_t e = ix->exon_ptr[k]; e < ix->exon_ptr[k + 1]; ++e) len += (int64_t)ix->exon_end[e] - ix->exon_start[e] + 1;
        L[(size_t)k] = len;
        line_off[(size_t)k + 1] = line_off[(size_t)k] + (id_off[(size_t)k + 1] - id_off[(size_t)k]) + 1 + len + 1;
    }
    std::vector<char> ids((size_t)std::max<int64_t>(1, id_off[(size_t)n]));
    rt_index_ids(ix, id_off.data(), ids.data());
    static const struct Letters {
        bool ok[256] = {};
        Letters() { for (char c : std::string("ACGTN")) ok[(unsigned char)c] = true; }
    } letters;
    auto row_ok = [&](int64_t k) {
        const int64_t off = line_off[(size_t)k], id_len = id_off[(size_t)k + 1] - id_off[(size_t)k];
        const int64_t stop = off + id_len + 1 + L[(size_t)k];
        if (stop > size || memcmp(text + off, ids.data() + id_off[(size_t)k], (size_t)id_len) != 0 || text[off + id_len] != '\t')
            return false;
        if (stop < size && text[stop] != '\n') return false;
        for (const unsigned char* q = (const unsigned char*)text + off + id_len + 1; q < (const unsigned char*)text + stop; ++q)
            if (!letters.ok[*q]) return false;
        return true;
    };
    const int64_t block = 1 << 12, n_blocks = (n + block - 1) / block;
    std::vector<int64_t> first_bad((size_t)std::max<int64_t>(1, n_blocks), INT64_MAX);
    claim_parallel(host_threads((size_t)(size >> 22) + 1, 16, "RT_CODON_THREADS"), (size_t)n_blocks, [&](size_t b) {
        for (int64_t k = (int64_t)b * block; k < std::min(n, (int64_t)(b + 1) * block); ++k)
            if (!row_ok(k)) { first_bad[b] = k; return; }
    });
    const int64_t bad = *std::min_element(first_bad.begin(), first_bad.end());
    if (bad != INT64_MAX) {
        // rows before `bad` matched exactly, so its line starts at line_off[bad]
        const int64_t k = bad, off = line_off[(size_t)k], line_no = k + 2;
        const std::string want(ids.data() + id_off[(size_t)k], (size_t)(id_off[(size_t)k + 1] - id_off[(size_t)k]));
        if (off >= size) {
            g_io_error = std::string(path) + ": the file ends after line " + std::to_string(k + 1) + ", the index has " +
                         std::to_string(n) + " rows" + hint;
            return RT_EINVAL;
        }
        const char* eol = (const char*)memchr(text + off, '\n', (size_t)(size - off));
        const int64_t stop = eol ? eol - text : size;
        const char* tab = (const char*)memchr(text + off, '\t', (size_t)(stop - off));
        if (!tab || std::string(text + off, tab) != want) {
            const int64_t got = (tab ? tab - text : stop) - off;
            g_io_error = where + std::to_string(line_no) + ": ORF_ID " + std::string(text + off, (size_t)std::min<int64_t>(got, 200)) +
                         " is not " + want + ", the ORF_ID of index row " + std::to_string(k + 1) + hint;
            return RT_EINVAL;
        }
        const int64_t got = stop - (tab + 1 - text);
        if (got != L[(size_t)k]) {
            g_io_error = where + std::to_string(line_no) + ": the sequence of " + want + " has " + std::to_string(got) +
                         " letters, the index row has " + std::to_string(L[(size_t)k]) + " nt" + hint;
            return RT_EINVAL;
        }
        int64_t at = 0;
        while (letters.ok[(unsigned char)tab[1 + at]]) ++at;
        g_io_error = where + std::to_string(line_no) + ": the sequence of " + want + " holds a letter other than A, C, G, T and N at " +
                     "position " + std::to_string(at + 1) + hint;
        return RT_EINVAL;
    }
    const int64_t done = std::min(line_off[(size_t)n], size);
    if (done < size) {
        g_io_error = where + std::to_string(n + 2) + ": the file has more lines than the index has rows (" + std::to_string(n) + ")" + hint;
        return RT_EINVAL;
    }
    h->seq_off.resize((size_t)n);
    for (int64_t k = 0; k < n; ++k) h->seq_off[(size_t)k] = line_off[(size_t)k] + (id_off[(size_t)k + 1] - id_off[(size_t)k]) + 1;
    return RT_OK;
}

int rt_codon_load_seq(rt_codon* h, const rt_index* ix, const char* path) {
    if (!h || !ix || !path) return RT_EINVAL;
    if (const int rc = read_file(path, h->seq)) return rc;
    return codon_parse_seq(h, ix, path);
}

int rt_codon_load_seq_text(rt_codon* h, const rt_index* ix, rt_text* text, const char* path) {
    if (!h || !ix || !text || !path) { rt_text_free(text); return RT_EINVAL; }
    adopt_text(text, h->seq);
    return codon_parse_seq(h, ix, path);
}

void rt_codon_free(rt_codon* h) { delete h; }

int rt_codon_sizes(const rt_codon* h, int64_t* sizes) {
    if (!h || !sizes) return RT_EINVAL;
    sizes[0] = (int64_t)h->row.size();
    sizes[1] = (int64_t)h->gene_key.size();
    sizes[2] = h->n_gseq;
    sizes[3] = h->n_lines;
    return RT_OK;
}

int rt_codon_copy(const rt_codon* h, int64_t* row, int32_t* gene, int32_t* gseq, int64_t* line, int64_t* prof_off,
                  int64_t* prof_len, int64_t* seq_off) {
    if (!h) return RT_EINVAL;
    auto copy = [](void* dst, const void* src, size_t bytes) { if (dst && bytes) memcpy(dst, src, bytes); };
    const size_t n = h->row.size();
    copy(row, h->row.data(), 8 * n);
    copy(gene, h->gene.data(), 4 * n);
    copy(gseq, h->gseq.data(), 4 * n);
    copy(line, h->line.data(), 8 * n);
    copy(prof_off, h->prof_off.data(), 8 * n);
    copy(prof_len, h->prof_len.data(), 8 * n);
    copy(seq_off, h->seq_off.data(), 8 * h->seq_off.size());
    return RT_OK;
}

const char* rt_codon_gene(const rt_codon* h, int64_t g, int* id_len, int* name_len) {
    if (!h || g < 0 || g >= (int64_t)h->gene_key.size()) return nullptr;
    const int il = h->gene_id_len[(size_t)g];
    if (id_len) *id_len = il;
    if (name_len) *name_len = h->gene_key_len[(size_t)g] - il - 1;
    return h->tsv.data() + h->gene_key[(size_t)g];
}

const char* rt_codon_text(const rt_codon* h, int which, int64_t* len) {
    if (!h || (which != 0 && which != 1)) return nullptr;
    const HostArr<char>& t = which == 0 ? h->tsv : h->seq;
    if (len) *len = (int64_t)t.size();
    return t.data();
}

int rt_codon_write(const rt_codon* h, const uint64_t* gene_tab, const uint64_t* pooled_tab, const char* gene_path,
                   const char* pooled_path) {
    if (!h || !gene_path || !pooled_path || !pooled_tab || (!h->gene_key.empty() && !gene_tab)) return RT_EINVAL;
    const int64_t n_gene = (int64_t)h->gene_key.size();
    // genes by (gene_id, gene_name): byte order equals Python's str order
    auto part = [&](int64_t g, int which) {
        int il = 0, nl = 0;
        const char* p = rt_codon_gene(h, g, &il, &nl);
        return which == 0 ? std::string_view(p, (size_t)il) : std::string_view(p + il + 1, (size_t)nl);
    };
    std::vector<int64_t> order((size_t)n_gene);
    for (int64_t g = 0; g < n_gene; ++g) order[(size_t)g] = g;
    std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
        const int c = part(a, 0).compare(part(b, 0));
        return c != 0 ? c < 0 : part(a, 1) < part(b, 1);
    });
    const int n_thr = host_threads((size_t)(n_gene >> 10), 16);
    std::vector<TextBuf> parts((size_t)n_thr + 1);
    parts[0].append("gene_id\tcodon\tcodon_occurrences\ttotal_codon_coverage\tmean_codon_coverage\tmedian_codon_coverage\t"
                    "var_codon_coverage\n", 114);
    std::vector<char> ok_part((size_t)n_thr, 1);
    run_parallel(n_thr, [&](int k) {
        TextBuf& b = parts[(size_t)k + 1];
        std::string num;
        for (int64_t i = n_gene * k / n_thr; i < n_gene * (k + 1) / n_thr; ++i) {
            const int64_t g = order[(size_t)i];
            const std::string_view id = part(g, 0);
            for (int c = 0; c < 64; ++c) {
                const uint64_t* cell = gene_tab + 5 * (64 * g + c);
                if (!cell[0]) continue;
                if (!b.need(id.size() + 256)) { ok_part[(size_t)k] = 0; return; }   // room for the whole row
                b.append(id.data(), id.size());
                b.append("\t", 1);
                put_codon(b, c);
                put_stats(b, cell, num);
            }
        }
    });
    TextBuf pooled;
    pooled.append("codon\tcodon_occurrences\ttotal_codon_coverage\tmean_codon_coverage\tmedian_codon_coverage\t"
                  "var_codon_coverage\n", 106);
    std::string num;
    for (int c = 0; c < 64; ++c)
        if (pooled_tab[5 * c]) { put_codon(pooled, c); put_stats(pooled, pooled_tab + 5 * c, num); }
    if (!parts[0].base || !pooled.base || std::find(ok_part.begin(), ok_part.end(), 0) != ok_part.end()) {
        g_io_error = "out of memory";
        return RT_ENOMEM;
    }
    bool ok = true;
    FILE* fg = fopen(gene_path, "wb");
    if (!fg) { g_io_error = std::string("cannot open ") + gene_path; return RT_EINVAL; }
    {
        WriteBehind w(fg);
        for (TextBuf& b : parts) ok = ok && w.put(std::move(b));
        ok = w.finish() && ok;
    }
    ok = fclose(fg) == 0 && ok;
    FILE* fp = ok ? fopen(pooled_path, "wb") : nullptr;
    if (fp) {
        ok = fwrite(pooled.base, 1, pooled.len, fp) == pooled.len;
        ok = fclose(fp) == 0 && ok;
    } else {
        ok = false;
    }
    if (!ok) {
        g_io_error = std::string("cannot write ") + gene_path + " or " + pooled_path;
        remove(gene_path);
        remove(pooled_path);
        return RT_EINVAL;
    }
    return RT_OK;
}

}  // extern "C"
