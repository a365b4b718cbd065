// rt_host_io.cpp -- native host I/O around the GPU path (SURVEY.md 8(f) "next #3"):
//   * candidate-ORF index loader: ORF.from_string rules (orf.py:121-182), interval sort (orf.py:100),
//     annotated prefix (detect_orfs.py:104-118) -> CSR arrays, without one Python object per row;
//   * {prefix}_translating_ORFs.tsv writer: rows formatted exactly as detect_orfs.py:304-323 prints
//     them (np.float64 / Python float shortest repr, str(list) profile).
// No GPU is involved; these entry points also work on a CPU-only box.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <charconv>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "ribotricer_b200.h"

// A column of the parsed index: plain uninitialised storage (the threads that fill a large array also touch its pages
// first; a std::vector would have one thread zero-fill it)
template <class T>
struct Arr {
    T* p = nullptr;
    size_t n = 0;
    Arr() = default;
    Arr(const Arr&) = delete;
    Arr& operator=(const Arr&) = delete;
    ~Arr() { free(p); }
    bool alloc(size_t m) {
        free(p);
        p = static_cast<T*>(malloc(std::max<size_t>(m, 1) * sizeof(T)));
        n = p ? m : 0;
        return p != nullptr;
    }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
    T* data() const { return p; }
    size_t size() const { return n; }
    T* begin() const { return p; }
    T* end() const { return p + n; }
};

struct rt_index {
    char* text = nullptr;                // the whole file (malloc); fields point into it
    size_t text_size = 0;
    ~rt_index() { free(text); }
    Arr<int64_t> exon_ptr;               // n_orf + 1
    Arr<int32_t> exon_start, exon_end;
    Arr<int32_t> orf_chrom;              // index into chrom_names
    Arr<uint8_t> orf_strand;             // 0 '+', 1 '-', 2 anything else
    Arr<uint32_t> field_len;             // 9 per ORF: lengths of fields 1..9
    Arr<uint64_t> line_field;            // per ORF: offset of field 1 (64-bit, files > 4 GB)
    std::vector<std::string> chrom_names;
    int64_t n_annotated_prefix = 0;
    std::string error;
};

// Text under construction: a growable char buffer written through a raw pointer (no per-character capacity checks).
struct TextBuf {
    char* base = nullptr;
    size_t len = 0, cap = 0;
    TextBuf() = default;
    TextBuf(TextBuf&& o) noexcept : base(o.base), len(o.len), cap(o.cap) { o.base = nullptr; o.len = o.cap = 0; }
    TextBuf& operator=(TextBuf&& o) noexcept {
        if (this != &o) { free(base); base = o.base; len = o.len; cap = o.cap; o.base = nullptr; o.len = o.cap = 0; }
        return *this;
    }
    TextBuf(const TextBuf&) = delete;
    TextBuf& operator=(const TextBuf&) = delete;
    ~TextBuf() { free(base); }
    // room for n more bytes; returns where to write them (nullptr: out of memory)
    char* need(size_t n) {
        if (cap - len < n) {
            const size_t want = std::max(len + n, cap + cap / 2 + (1u << 16));
            char* q = static_cast<char*>(realloc(base, want));
            if (!q) return nullptr;
            base = q;
            cap = want;
        }
        return base + len;
    }
    void advance_to(char* p) { len = (size_t)(p - base); }
    void append(const char* d, size_t n) {
        if (char* p = need(n)) { memcpy(p, d, n); len += n; }
    }
};

// An output file with a write-behind thread: formatted text is queued and written in order while the caller formats
// the next piece (or waits for the GPU).  At most kPendingMax bytes wait in the queue.
struct rt_tsv {
    FILE* fh = nullptr;
    std::thread writer;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<TextBuf> queue;
    size_t pending = 0;
    bool closing = false, failed = false;
    static constexpr size_t kPendingMax = 1ull << 30;

    void run() {
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv.wait(lk, [&] { return closing || !queue.empty(); });
            if (queue.empty()) return;
            TextBuf b = std::move(queue.front());
            queue.pop_front();
            lk.unlock();
            const bool ok = b.len == 0 || fwrite(b.base, 1, b.len, fh) == b.len;
            lk.lock();
            pending -= b.len;
            if (!ok) failed = true;
            cv.notify_all();
        }
    }
    // false when an earlier write has failed
    bool put(TextBuf&& b) {
        std::unique_lock<std::mutex> lk(mu);
        if (failed) return false;
        if (b.len == 0) return true;
        if (!writer.joinable()) writer = std::thread([this] { run(); });
        cv.wait(lk, [&] { return pending < kPendingMax || failed; });
        pending += b.len;
        queue.push_back(std::move(b));
        cv.notify_all();
        return !failed;
    }
    bool put(const std::string& s) {
        TextBuf b;
        b.append(s.data(), s.size());
        return b.len == s.size() && put(std::move(b));
    }
    // drains the queue and stops the thread; false when any write failed
    bool finish() {
        {
            std::lock_guard<std::mutex> lk(mu);
            closing = true;
        }
        cv.notify_all();
        if (writer.joinable()) writer.join();
        return !failed;
    }
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

// Decimal digits of v at p; returns the end.  Coverage profiles are mostly one-digit numbers.
inline char* put_int(char* p, long long v) {
    static const char pairs[] =
        "00010203040506070809101112131415161718192021222324252627282930313233343536373839404142434445464748495051525354555657585960616263"
        "646566676869707172737475767778798081828384858687888990919293949596979899";
    unsigned long long u = (unsigned long long)v;
    if (v < 0) { *p++ = '-'; u = 0ull - u; }
    if (u < 10) { *p++ = (char)('0' + u); return p; }
    if (u < 100) { memcpy(p, pairs + 2 * u, 2); return p + 2; }
    char tmp[24];
    int k = 24;
    while (u >= 100) {
        const unsigned r = (unsigned)(u % 100);
        u /= 100;
        k -= 2;
        memcpy(tmp + k, pairs + 2 * r, 2);
    }
    if (u >= 10) { k -= 2; memcpy(tmp + k, pairs + 2 * u, 2); }
    else tmp[--k] = (char)('0' + u);
    memcpy(p, tmp + k, (size_t)(24 - k));
    return p + (24 - k);
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

}  // extern "C"

void rt_io_set_error(const std::string& msg) { g_io_error = msg; }   // rt_prepare.cpp reports through the same slot

extern "C" {

int rt_index_load(const char* path, rt_index** out) {
    if (!path || !out) return RT_EINVAL;
    *out = nullptr;
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { g_io_error = std::string("cannot open ") + path; return RT_EINVAL; }
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); g_io_error = std::string("cannot stat ") + path; return RT_EINVAL; }
    const size_t size = (size_t)st.st_size;
    std::unique_ptr<rt_index> ix(new rt_index());
    ix->text = static_cast<char*>(malloc(size + 1));
    if (!ix->text) { close(fd); g_io_error = "out of memory"; return RT_ENOMEM; }
    ix->text_size = size;
    int n_thr = (int)std::max<size_t>(1, std::min<size_t>({(size_t)std::thread::hardware_concurrency(), (size_t)16, size >> 22}));
    if (const char* e = getenv("RT_INDEX_THREADS")) n_thr = std::max(1, std::min(64, atoi(e)));   // tests: chunked parse of a small file
    // 1. the file, read in slices by all threads (the buffer's pages are first touched by the thread that fills them)
    {
        std::atomic<bool> ok{true};
        auto read_slice = [&](int k) {
            size_t at = size * (size_t)k / n_thr;
            const size_t hi = size * (size_t)(k + 1) / n_thr;
            while (at < hi) {
                const ssize_t got = pread(fd, ix->text + at, hi - at, (off_t)at);
                if (got <= 0) { ok = false; return; }
                at += (size_t)got;
            }
        };
        std::vector<std::thread> pool;
        for (int k = 1; k < n_thr; ++k) pool.emplace_back(read_slice, k);
        read_slice(0);
        for (auto& th : pool) th.join();
        close(fd);
        if (!ok) { g_io_error = "short read"; return RT_EINVAL; }
    }
    ix->text[size] = '\0';
    const char* base = ix->text;
    const char* end = base + size;
    const char* body = (const char*)memchr(base, '\n', size);   // skip the header (detect_orfs.py:273)
    body = body ? body + 1 : end;

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
    {
        const size_t span = (size_t)(end - body);
        const char* lo = body;
        for (int k = 0; k < n_thr; ++k) {
            const char* hi = end;
            if (k + 1 < n_thr) {
                const char* guess = body + span * (size_t)(k + 1) / n_thr;
                if (guess < lo) guess = lo;
                const char* nl = guess < end ? (const char*)memchr(guess, '\n', (size_t)(end - guess)) : nullptr;
                hi = nl ? nl + 1 : end;
            }
            chunks[(size_t)k].lo = lo;
            chunks[(size_t)k].hi = hi;
            lo = hi;
        }
    }
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
    {
        std::vector<std::thread> pool;
        for (int k = 1; k < n_thr; ++k) pool.emplace_back([&, k]() { parse_chunk(chunks[(size_t)k]); });
        parse_chunk(chunks[0]);
        for (auto& th : pool) th.join();
    }
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
    auto merge_chunk = [&](size_t k) {
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
    };
    {
        std::vector<std::thread> pool;
        for (size_t k = 1; k < chunks.size(); ++k) pool.emplace_back(merge_chunk, k);
        merge_chunk(0);
        for (auto& th : pool) th.join();
    }
    *out = ix.release();
    return RT_OK;
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
    std::vector<std::thread> pool;
    auto copy = [&](void* dst, const void* src, size_t bytes) {
        if (!dst || !bytes) return;
        if (bytes < (1u << 22)) memcpy(dst, src, bytes);
        else pool.emplace_back([=]() { memcpy(dst, src, bytes); });
    };
    copy(exon_ptr, ix->exon_ptr.p, 8 * ix->exon_ptr.n);
    copy(exon_start, ix->exon_start.p, 4 * ix->exon_start.n);
    copy(exon_end, ix->exon_end.p, 4 * ix->exon_end.n);
    copy(orf_chrom, ix->orf_chrom.p, 4 * ix->orf_chrom.n);
    copy(orf_strand, ix->orf_strand.p, ix->orf_strand.n);
    for (auto& th : pool) th.join();
    return RT_OK;
}

// Field k (1..9: ORF_type .. start_codon) of row `orf`; not NUL terminated.
const char* rt_index_field(const rt_index* ix, int64_t orf, int k, int* len) {
    if (!ix || orf < 0 || orf >= (int64_t)ix->orf_chrom.size() || k < 1 || k > 9) return nullptr;
    uint64_t off = ix->line_field[orf];
    for (int j = 1; j < k; ++j) off += ix->field_len[9 * orf + (j - 1)] + 1;
    if (len) *len = (int)ix->field_len[9 * orf + (k - 1)];
    return ix->text + off;
}

int rt_tsv_open(const char* path, int write_header, rt_tsv** out) {
    if (!path || !out) return RT_EINVAL;
    FILE* fh = fopen(path, "wb");
    if (!fh) { g_io_error = std::string("cannot open ") + path; return RT_EINVAL; }
    rt_tsv* t = new rt_tsv();
    t->fh = fh;
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
        const int64_t e0 = ix->exon_ptr[o], e1 = ix->exon_ptr[o + 1];
        long long L = 0;
        for (int64_t e = e0; e < e1; ++e) L += (long long)ix->exon_end[e] - ix->exon_start[e] + 1;
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
        // oid = tid_start_end_len (orf.py:101-103)
        put(f[2], flen[2]); *p++ = '_';
        p = put_int(p, e1 > e0 ? ix->exon_start[e0] : 0); *p++ = '_';
        p = put_int(p, e1 > e0 ? ix->exon_end[e1 - 1] : 0); *p++ = '_';
        p = put_int(p, L); *p++ = '\t';
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
    const int n_thr = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)std::thread::hardware_concurrency(), (int64_t)16,
                                                                  (total + n_sel * 40) / (1 << 21)}));
    std::vector<int64_t> cut(n_thr + 1, n_sel);
    cut[0] = 0;
    for (int k = 1; k < n_thr; ++k) {
        const int64_t target = prof_ptr[0] + total * k / n_thr;
        cut[k] = std::lower_bound(prof_ptr, prof_ptr + n_sel, target) - prof_ptr;
        if (cut[k] < cut[k - 1]) cut[k] = cut[k - 1];
    }
    std::vector<TextBuf> parts(n_thr);
    std::vector<char> ok(n_thr, 1);
    std::vector<std::thread> pool;
    for (int k = 1; k < n_thr; ++k)
        pool.emplace_back([&, k]() {
            ok[k] = format_rows(parts[k], ix, cut[k], cut[k + 1], orf_ids, orf_lo, score, valid, count, length, status, prof_ptr, prof);
        });
    ok[0] = format_rows(parts[0], ix, cut[0], cut[1], orf_ids, orf_lo, score, valid, count, length, status, prof_ptr, prof);
    for (auto& th : pool) th.join();
    for (int k = 0; k < n_thr; ++k)
        if (!ok[k]) { g_io_error = "rt_tsv_write: ORF id outside the index or the result range, or out of memory"; return RT_EINVAL; }
    for (int k = 0; k < n_thr; ++k)
        if (!t->put(std::move(parts[k]))) { g_io_error = "rt_tsv_write: write failed"; return RT_EINVAL; }
    return RT_OK;
}

int rt_tsv_close(rt_tsv* t) {
    if (!t) return RT_EINVAL;
    const bool wrote = t->finish();
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
    std::atomic<int64_t> next{0};
    auto run = [&]() {
        for (int64_t b; (b = next.fetch_add(1)) < n_blocks;) {
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
        }
    };
    {
        const int n_thr = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)std::thread::hardware_concurrency(), (int64_t)16, n_blocks}));
        std::vector<std::thread> pool;
        for (int t = 1; t < n_thr; ++t) pool.emplace_back(run);
        run();
        for (auto& th : pool) th.join();
    }
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
    const int n_thr = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)std::thread::hardware_concurrency(), (int64_t)16, n >> 16}));
    if (n_thr == 1) {
        if (!lines(head, 0, n) || !t->put(std::move(head))) return RT_EINVAL;
        return RT_OK;
    }
    std::vector<TextBuf> part((size_t)n_thr);
    std::vector<char> ok((size_t)n_thr, 1);
    std::vector<std::thread> pool;
    for (int k = 0; k < n_thr; ++k)
        pool.emplace_back([&, k]() { ok[(size_t)k] = lines(part[(size_t)k], n * k / n_thr, n * (k + 1) / n_thr); });
    for (auto& th : pool) th.join();
    for (char c : ok)
        if (!c) return RT_EINVAL;
    if (!t->put(std::move(head))) return RT_EINVAL;
    for (TextBuf& o : part)
        if (!t->put(std::move(o))) return RT_EINVAL;
    return RT_OK;
}

int rt_wig_close(rt_tsv* t) { return rt_tsv_close(t); }

}  // extern "C"

// ---- packed read records (11 B/read instead of 18): the filter cascade is decided here, on the host ----
#include <thread>

// bam.py:77-91 + common.py:33-69 for reads [0, m) of a chunk (same order as classify_read() in rt_kernels.cuh: the
// EARLIER test wins, so the selects run from the last test to the first) and the run-length code of ref_id.  One
// thread; branch-free and in blocks so that the compiler vectorises both loops (an AVX2 clone is picked at load time).
// Returns the number of runs, or -1 when there are more than `cap` (the chunk is not grouped by reference).
#if defined(__x86_64__) && defined(__GNUC__) && !defined(__clang__)
__attribute__((target_clones("avx2", "default")))
#endif
int64_t rt_pack_chunk(const int32_t* __restrict__ ref_id, const uint16_t* __restrict__ flag, const uint8_t* __restrict__ mapq,
                      const uint8_t* __restrict__ nh, int64_t m, uint8_t* __restrict__ meta, int64_t* run_start, int32_t* run_ref,
                      int64_t cap) {
    for (int64_t i = 0; i < m; ++i) {
        const unsigned f = flag[i];
        const unsigned nn = nh[i], qq = mapq[i];             // both loaded unconditionally: no control flow, the loop vectorises
        const unsigned uniq = (nn == 1u) | ((nn == 0u) & (qq == 255u));
        unsigned code = uniq ? 0u : (unsigned)RT_ST_MULTI;
        code = (f & 0x4) ? (unsigned)RT_ST_UNMAPPED : code;
        code = (f & 0x100) ? (unsigned)RT_ST_SECONDARY : code;
        code = (f & 0x400) ? (unsigned)RT_ST_DUPLICATE : code;
        code = (f & 0x200) ? (unsigned)RT_ST_QCFAIL : code;
        meta[i] = (uint8_t)(code | ((f >> 1) & 8u));
    }
    int64_t r = 0;
    if (m > 0) {
        run_start[0] = 0;
        run_ref[0] = ref_id[0];
        r = 1;
    }
    constexpr int64_t kBlock = 256;
    for (int64_t b = 1; b < m; b += kBlock) {
        const int64_t e = b + kBlock < m ? b + kBlock : m;
        int32_t diff = 0;
        for (int64_t i = b; i < e; ++i) diff |= ref_id[i] ^ ref_id[i - 1];
        if (diff == 0) continue;                    // the usual case: no reference changes inside the block
        for (int64_t i = b; i < e; ++i)
            if (ref_id[i] != ref_id[i - 1]) {
                if (r >= cap) return -1;
                run_start[r] = i;
                run_ref[r] = ref_id[i];
                ++r;
            }
    }
    run_start[r] = m;
    return r;
}

extern "C" {

int rt_pack_read_meta(int64_t n, const int32_t* ref_id, const uint16_t* flag, const uint8_t* mapq, const uint8_t* nh,
                      uint8_t* meta, int64_t run_cap, int64_t* run_start, int32_t* run_ref, int64_t* n_runs) {
    if (n < 0 || !n_runs || (n > 0 && (!ref_id || !flag || !mapq || !nh || !meta || !run_start || !run_ref)))
        return RT_EINVAL;
    // bam.py:77-91 + common.py:33-69, same order as classify_read() in rt_kernels.cuh
    auto work = [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; ++i) {
            const unsigned f = flag[i];
            unsigned code;
            if (f & 0x200) code = RT_ST_QCFAIL;
            else if (f & 0x400) code = RT_ST_DUPLICATE;
            else if (f & 0x100) code = RT_ST_SECONDARY;
            else if (f & 0x4) code = RT_ST_UNMAPPED;
            else code = (nh[i] != 0 ? nh[i] == 1 : mapq[i] == 255) ? 0u : (unsigned)RT_ST_MULTI;
            meta[i] = (uint8_t)(code | ((f & 0x10) ? 8u : 0u));
        }
    };
    const int n_thr = (int)std::max<int64_t>(1, std::min<int64_t>(std::thread::hardware_concurrency(), n / (1 << 20)));
    std::vector<std::thread> pool;
    for (int t = 0; t < n_thr; ++t) pool.emplace_back(work, n * t / n_thr, n * (t + 1) / n_thr);
    for (auto& th : pool) th.join();
    int64_t r = 0;
    for (int64_t i = 0; i < n; ++i)
        if (i == 0 || ref_id[i] != ref_id[i - 1]) {
            if (r >= run_cap) {
                g_io_error = "rt_pack_read_meta: more reference runs than run_cap (input not grouped by reference?)";
                return RT_ESTATE;
            }
            run_start[r] = i;
            run_ref[r] = ref_id[i];
            ++r;
        }
    if (n > 0) run_start[r] = n;
    *n_runs = r;
    return RT_OK;
}

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
    // GPU box: 10 % off the coding time at 512 reads, nothing more further out).  RT_PACK_PREFETCH overrides, 0 = off.
    static const int64_t ahead_reads = [] {
        const char* e = getenv("RT_PACK_PREFETCH");
        return e ? (int64_t)atoll(e) : (int64_t)512;
    }();
    while (i < m) {
        if (ahead_reads > 0 && i + ahead_reads + kStreamGroup <= m) {   // one 64-read group of every column, `ahead_reads` further on
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
    if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
    n_threads = (int)std::max<int64_t>(1, std::min<int64_t>(n_threads, n_ranges));
    std::vector<int64_t> blocks(n_ranges + 1, 0);
    auto sweep = [&](bool write) {
        std::atomic<int64_t> next{0};
        std::atomic<int64_t> worst{0};
        auto work = [&]() {
            for (;;) {
                const int64_t r = next.fetch_add(1);
                if (r >= n_ranges) break;
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
            }
        };
        std::vector<std::thread> pool;
        for (int t = 1; t < n_threads; ++t) pool.emplace_back(work);
        work();
        for (auto& th : pool) th.join();
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
