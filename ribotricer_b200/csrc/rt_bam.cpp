// rt_bam.cpp -- native BAM/BGZF decode straight to the read columns of the C ABI
// (SURVEY.md 8(f) "next #2"; replaces the two pysam passes of bam.py:65-71 on the host).
//
// Per alignment record it produces what split_bam reads through pysam:
//   ref_id  = reference_id                       flag = flag        mapq = mapping_quality
//   first / last / mlen = get_reference_positions()[0] / [-1] / len()   (bam.py:95-99): reference
//             positions of M, = and X operations only (D and N advance the reference, S I H P do not)
//   nh      = the NH aux tag as is_read_uniq_mapping sees it (common.py:53-56: `dict(get_tags())["NH"] == 1`):
//             0 = absent, 1 = present and equal to 1, anything else = present and different from 1
//             (2..254 the value itself; 255 for values <= 0, > 254 or of a non-numeric type).  When the tag
//             occurs twice the LAST one counts, as in dict().
//   pos / ref_end = reference_start / reference_end of infer_protocol.py:84-85 (ref_end = -1 for None:
//             unmapped flag or no CIGAR; else pos + reference length of the CIGAR, at least 1 as in htslib)
// The file is decoded as a pipeline of batches of BGZF blocks (see rt_bam_load): every worker inflates a batch
// (rt_inflate.cpp, CRC-32 checked, zlib as fallback), takes its turn in the one sequential step -- finding the record
// boundaries of the batch, which needs the offset the previous batch ended on -- and decodes its records into
// columns; the columns are concatenated by all threads at the end.  No GPU is involved.
#include <sys/mman.h>
#include <sys/stat.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstring>
#include <exception>
#include <condition_variable>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "ribotricer_b200.h"
#include "rt_bgzf.h"
#include "rt_host.h"

struct rt_bam {
    std::vector<std::string> ref_names;
    std::vector<int64_t> ref_lens;
    HostArr<int32_t> ref_id, first, last, pos, ref_end;   // uninitialised: first touched by the threads that fill them
    HostArr<uint16_t> mlen, flag;
    HostArr<uint8_t> mapq, nh;
    bool sorted = false;
};

namespace {

thread_local std::string g_bam_error;

inline uint16_t rd16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }
inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline int32_t rdi32(const uint8_t* p) { int32_t v; memcpy(&v, p, 4); return v; }

// Decode one alignment record (after its block_size field) into slot i of the columns.
// Returns false when the fixed fields, the CIGAR or an aux field run past the record (untrusted input).
struct ColView {
    int32_t *ref_id, *first, *last, *pos, *ref_end;
    uint16_t *mlen, *flag;
    uint8_t *mapq, *nh;
};

bool decode_record(const uint8_t* r, uint32_t len, const ColView& out, size_t i) {
    const int32_t ref = rdi32(r), pos = rdi32(r + 4);
    const uint32_t l_name = r[8];
    const uint32_t n_cigar = rd16(r + 12);
    const int32_t l_seq = rdi32(r + 16);
    if (l_seq < 0) return false;
    const uint64_t fixed = 32ull + l_name + 4ull * n_cigar + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq;
    if (fixed > len) return false;
    out.ref_id[i] = ref;
    out.mapq[i] = r[9];
    const uint16_t flag = rd16(r + 14);
    out.flag[i] = flag;
    const uint8_t* cig = r + 32 + l_name;
    int64_t cur = pos, first = 0, last = 0, n = 0;
    for (uint32_t k = 0; k < n_cigar; ++k) {
        const uint32_t v = rd32(cig + 4 * k), op = v & 15u, l = v >> 4;
        if (op == 0 || op == 7 || op == 8) {          // M = X
            if (n == 0) first = cur;
            last = cur + l - 1;
            n += l;
            cur += l;
        } else if (op == 2 || op == 3) {              // D N
            cur += l;
        }
    }
    out.first[i] = (int32_t)first;
    out.last[i] = (int32_t)last;
    out.mlen[i] = (uint16_t)std::min<int64_t>(n, 65535);
    out.pos[i] = pos;
    const int64_t rlen = cur - pos;
    out.ref_end[i] = ((flag & 4) || n_cigar == 0) ? -1 : (int32_t)(pos + (rlen ? rlen : 1));
    // aux fields: the NH tag as `dict(read.get_tags())["NH"] == 1` sees it
    const uint8_t* end = r + len;
    const uint8_t* a = r + fixed;
    int nh = 0;                                           // 0 absent, 1 equal to 1, else present and not 1
    while (a + 3 <= end) {
        const uint8_t t0 = a[0], t1 = a[1], ty = a[2];
        a += 3;
        size_t adv = 0;
        switch (ty) {
            case 'A': case 'c': case 'C': adv = 1; break;
            case 's': case 'S': adv = 2; break;
            case 'i': case 'I': case 'f': adv = 4; break;
            case 'Z': case 'H': {
                const uint8_t* z = (const uint8_t*)memchr(a, 0, (size_t)(end - a));
                if (!z) return false;
                adv = (size_t)(z - a) + 1;
                break;
            }
            case 'B': {
                if (a + 5 > end) return false;
                const uint8_t sub = a[0];
                const uint32_t cnt = rd32(a + 1);
                const size_t w = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
                adv = 5 + (size_t)cnt * w;
                break;
            }
            default: return false;                    // unknown aux type
        }
        if (adv > (size_t)(end - a)) return false;
        if (t0 == 'N' && t1 == 'H') {
            long long val = 0;
            bool numeric = true;
            switch (ty) {
                case 'c': val = (int8_t)a[0]; break;
                case 'C': val = a[0]; break;
                case 's': val = (int16_t)rd16(a); break;
                case 'S': val = rd16(a); break;
                case 'i': val = rdi32(a); break;
                case 'I': val = rd32(a); break;
                case 'f': { float f; memcpy(&f, a, 4); val = f == 1.0f ? 1 : 0; break; }   // 1.0 == 1 in Python
                default: numeric = false;
            }
            nh = !numeric ? 255 : val == 1 ? 1 : (val >= 2 && val <= 254) ? (int)val : 255;
        }
        a += adv;
    }
    out.nh[i] = (uint8_t)nh;
    return true;
}

// What the walk of one batch hands to the next: the bytes of the record (or header) that is not complete yet,
// the number of records before the next batch, and whether the header has been read.
struct Handoff {
    std::vector<uint8_t> carry;
    size_t n_before = 0;
    bool header_done = false;
};

constexpr size_t kRowBytes = 5 * 4 + 2 * 2 + 2;          // one record in the columns of a batch

struct BatchOut {
    size_t base = 0, n = 0;
    std::unique_ptr<uint8_t[]> mem;                       // [5][n] int32, [2][n] uint16, [2][n] uint8
    ColView view() const {
        int32_t* w = reinterpret_cast<int32_t*>(mem.get());
        uint16_t* h = reinterpret_cast<uint16_t*>(w + 5 * n);
        uint8_t* b = reinterpret_cast<uint8_t*>(h + 2 * n);
        return ColView{w, w + n, w + 2 * n, w + 3 * n, w + 4 * n, h, h + n, b, b + n};
    }
};

// BAM header at the start of the uncompressed stream.  1 = parsed (`used` bytes), 0 = more data needed, -1 = not a BAM.
int parse_header(const uint8_t* d, size_t n, rt_bam& bam, size_t& used) {
    if (n >= 4 && memcmp(d, "BAM\1", 4) != 0) return -1;
    if (n < 12) return 0;
    const uint32_t l_text = rd32(d + 4);
    if (n < 12 + (size_t)l_text) return 0;
    size_t q = 8 + (size_t)l_text;
    const uint32_t n_ref = rd32(d + q);
    q += 4;
    std::vector<std::string> names;
    std::vector<int64_t> lens;
    for (uint32_t r = 0; r < n_ref; ++r) {
        if (q + 4 > n) return 0;
        const uint32_t l_name = rd32(d + q);
        if (q + 8 + (size_t)l_name > n) return 0;
        names.emplace_back((const char*)d + q + 4, l_name ? l_name - 1 : 0);
        lens.push_back(rd32(d + q + 4 + l_name));
        q += 8 + (size_t)l_name;
    }
    const std::string text((const char*)d + 8, l_text);
    const size_t hd = text.find("@HD");
    if (hd != std::string::npos) {
        const size_t eol = text.find('\n', hd);
        bam.sorted = text.substr(hd, eol - hd).find("SO:coordinate") != std::string::npos;
    }
    bam.ref_names.swap(names);
    bam.ref_lens.swap(lens);
    used = q;
    return 1;
}

// fn(lo, hi) over [0, n) in slices of 1 Mi elements, on up to 16 threads (one when n is small)
template <class F>
void parallel_slices(size_t n, const F& fn) {
    const size_t slice = 1u << 20, n_slices = (n + slice - 1) / slice;
    claim_parallel(host_threads(n_slices, 16), n_slices, [&](size_t k) { fn(k * slice, std::min(n, (k + 1) * slice)); });
}

}  // namespace

extern "C" {

const char* rt_bam_last_error(void) { return g_bam_error.c_str(); }

int rt_bam_load(const char* path, int n_threads, rt_bam** out) {
    if (!path || !out) return RT_EINVAL;
    *out = nullptr;
    if (n_threads <= 0) n_threads = host_threads(SIZE_MAX, SIZE_MAX);    // every hardware thread
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { g_bam_error = std::string("cannot open ") + path; return RT_EINVAL; }
    struct stat st;
    fstat(fd, &st);
    const size_t size = (size_t)st.st_size;
    const uint8_t* base = size ? (const uint8_t*)mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0) : nullptr;
    close(fd);
    if (size && base == MAP_FAILED) { g_bam_error = "mmap failed"; return RT_EINVAL; }
    if (size) madvise((void*)base, size, MADV_SEQUENTIAL);
    size_t batch_bytes = 1u << 20;                     // uncompressed bytes per batch: stays in the worker's cache
    if (const char* e = getenv("RT_BAM_BATCH_BYTES")) batch_bytes = std::max<size_t>(1, strtoull(e, nullptr, 10));
    const bool zlib_only = getenv("RT_BAM_ZLIB") != nullptr;     // A/B switch: zlib's inflate instead of rt_inflate.cpp

    // The file is cut into batches of consecutive BGZF blocks.  A worker claims the next batch (block headers are parsed
    // under the claim lock, so batches are handed out in file order), inflates it into its own reusable buffer, then
    // waits for its turn in the WALK: the only sequential step, which needs to know where the first record of the batch
    // starts.  The walk finds the record boundaries, hands the unfinished tail (`carry`) and the running record count
    // to the next batch, and the worker decodes its records into columns of its own while the next batch is walked.
    std::unique_ptr<rt_bam> bam(new rt_bam());
    std::mutex claim_mu, walk_mu, out_mu;
    std::condition_variable walk_cv;
    size_t file_off = 0, next_batch = 0, walk_turn = 0;
    Handoff cur;
    std::vector<BatchOut> done;
    std::atomic<bool> failed{false};
    std::string fail_msg;
    auto set_fail = [&](const char* msg) {
        {
            std::lock_guard<std::mutex> lk(walk_mu);
            if (!failed.exchange(true)) fail_msg = msg;
        }
        walk_cv.notify_all();
    };

    auto worker = [&]() {
        std::vector<uint8_t> buf, strad;
        std::vector<Block> blocks;
        std::vector<uint32_t> rec_off;
        for (;;) {
            size_t k, n = 0;
            {
                std::lock_guard<std::mutex> lk(claim_mu);
                if (failed || file_off >= size) return;
                blocks.clear();
                while (file_off < size && n < batch_bytes) {
                    Block b;
                    size_t next;
                    if (!parse_block(base, size, file_off, b, next)) { set_fail("not a BGZF/BAM file (bad block header)"); return; }
                    b.out_off = n;
                    n += b.out_len;
                    blocks.push_back(b);
                    file_off = next;
                }
                k = next_batch++;
            }
            if (buf.size() < n) buf.resize(n);
            uint8_t* data = buf.data();
            bool ok = true;
            for (const Block& b : blocks) ok = ok && inflate_block(base + b.in_off, b.in_len, data + b.out_off, b.out_len, b.crc, zlib_only);
            if (!ok) { set_fail("BGZF block does not inflate to its announced size and CRC-32"); return; }

            // ---- the walk (one batch at a time, in file order)
            {
                std::unique_lock<std::mutex> lk(walk_mu);
                walk_cv.wait(lk, [&] { return walk_turn == k || failed; });
                if (failed) return;
            }
            Handoff h = std::move(cur), nxt;           // only the holder of the turn touches `cur`
            auto pass_on = [&](Handoff& v) {
                {
                    std::lock_guard<std::mutex> lk(walk_mu);
                    cur = std::move(v);
                    walk_turn = k + 1;
                }
                walk_cv.notify_all();
            };
            size_t p = 0;                               // where the first record that STARTS in this batch begins
            bool have_strad = false;
            if (!h.header_done) {                       // header: magic, text, references (may span batches)
                const uint8_t* hd = data;
                size_t hn = n;
                const size_t before = h.carry.size();
                if (before) {
                    h.carry.insert(h.carry.end(), data, data + n);
                    hd = h.carry.data();
                    hn = h.carry.size();
                }
                size_t used = 0;
                const int rc = parse_header(hd, hn, *bam, used);
                if (rc < 0) { set_fail("not a BAM file (bad magic)"); return; }
                if (rc == 0) {                          // incomplete: everything so far travels on
                    if (!before) h.carry.assign(data, data + n);
                    nxt.carry = std::move(h.carry);
                    pass_on(nxt);
                    continue;
                }
                p = used - before;                      // used > before, or the previous batch would have finished the header
                h.carry.clear();
            } else if (!h.carry.empty()) {              // the record that began in an earlier batch
                strad = std::move(h.carry);
                size_t take = 0;
                if (strad.size() < 4) {
                    take = std::min<size_t>(4 - strad.size(), n);
                    strad.insert(strad.end(), data, data + take);
                }
                bool complete = false;
                if (strad.size() >= 4) {
                    const uint32_t bs = rd32(strad.data());
                    if (bs < 32) { set_fail("corrupt BAM record"); return; }
                    const size_t need = 4 + (size_t)bs - strad.size();
                    if (need <= n - take) {
                        strad.insert(strad.end(), data + take, data + take + need);
                        p = take + need;
                        complete = true;
                    }
                }
                if (!complete) {                        // longer than this whole batch: keep collecting
                    strad.insert(strad.end(), data + take, data + n);
                    nxt.carry = std::move(strad);
                    nxt.n_before = h.n_before;
                    nxt.header_done = true;
                    pass_on(nxt);
                    strad.clear();
                    continue;
                }
                have_strad = true;
            }
            rec_off.clear();
            while (p + 4 <= n) {
                const uint32_t bs = rd32(data + p);
                if (bs < 32) { set_fail("corrupt BAM record"); return; }
                if (4 + (size_t)bs > n - p) break;
                rec_off.push_back((uint32_t)p);
                p += 4 + (size_t)bs;
            }
            const size_t m = rec_off.size() + (have_strad ? 1 : 0);
            nxt.carry.assign(data + p, data + n);
            nxt.n_before = h.n_before + m;
            nxt.header_done = true;
            pass_on(nxt);

            // ---- decode into columns of this batch
            if (m == 0) continue;
            BatchOut bo;
            bo.base = h.n_before;
            bo.n = m;
            bo.mem.reset(new uint8_t[m * kRowBytes]);
            const ColView v = bo.view();
            bool rec_ok = true;
            size_t i = 0;
            if (have_strad) rec_ok = decode_record(strad.data() + 4, rd32(strad.data()), v, i++);
            for (size_t j = 0; j < rec_off.size(); ++j, ++i)
                rec_ok = decode_record(data + rec_off[j] + 4, rd32(data + rec_off[j]), v, i) && rec_ok;
            if (!rec_ok) { set_fail("corrupt BAM record"); return; }
            std::lock_guard<std::mutex> lk(out_mu);
            done.push_back(std::move(bo));
        }
    };
    auto guarded = [&]() {
        try {
            worker();
        } catch (const std::exception& e) {              // bad_alloc on a huge record: refuse the file, do not terminate
            set_fail("out of memory while decoding");
        }
    };
    run_parallel(n_threads, [&](int) { guarded(); });
    if (size) munmap((void*)base, size);
    if (failed) { g_bam_error = fail_msg; return RT_EINVAL; }
    if (!cur.header_done) { g_bam_error = "truncated BAM header"; return RT_EINVAL; }
    if (!cur.carry.empty()) { g_bam_error = "truncated BAM record at end of file"; return RT_EINVAL; }

    // ---- the batches' columns, concatenated in file order by all threads (first touch of the final arrays included)
    const size_t total = cur.n_before;
    if (total > (size_t)INT64_MAX / kRowBytes) { g_bam_error = "too many records"; return RT_EINVAL; }
    rt_bam& B = *bam;
    if (!(B.ref_id.alloc(total) && B.first.alloc(total) && B.last.alloc(total) && B.pos.alloc(total) && B.ref_end.alloc(total) &&
          B.mlen.alloc(total) && B.flag.alloc(total) && B.mapq.alloc(total) && B.nh.alloc(total))) {
        g_bam_error = "out of memory";
        return RT_ENOMEM;
    }
    claim_parallel((int)std::min<size_t>((size_t)n_threads, done.size()), done.size(), [&](size_t j) {
        BatchOut& bo = done[j];
        const ColView v = bo.view();
        const size_t o = bo.base, m = bo.n;
        memcpy(B.ref_id.p + o, v.ref_id, 4 * m); memcpy(B.first.p + o, v.first, 4 * m); memcpy(B.last.p + o, v.last, 4 * m);
        memcpy(B.pos.p + o, v.pos, 4 * m); memcpy(B.ref_end.p + o, v.ref_end, 4 * m);
        memcpy(B.mlen.p + o, v.mlen, 2 * m); memcpy(B.flag.p + o, v.flag, 2 * m);
        memcpy(B.mapq.p + o, v.mapq, m); memcpy(B.nh.p + o, v.nh, m);
        bo.mem.reset();
    });
    *out = bam.release();
    return RT_OK;
}

void rt_bam_free(rt_bam* b) { delete b; }
int64_t rt_bam_n_reads(const rt_bam* b) { return b ? (int64_t)b->ref_id.size() : 0; }
int rt_bam_n_ref(const rt_bam* b) { return b ? (int)b->ref_names.size() : 0; }
const char* rt_bam_ref_name(const rt_bam* b, int i) {
    return b && i >= 0 && i < (int)b->ref_names.size() ? b->ref_names[i].c_str() : nullptr;
}
int64_t rt_bam_ref_len(const rt_bam* b, int i) { return b && i >= 0 && i < (int)b->ref_lens.size() ? b->ref_lens[i] : -1; }
int rt_bam_sorted(const rt_bam* b) { return b && b->sorted ? 1 : 0; }

int rt_bam_copy(const rt_bam* b, int32_t* ref_id, int32_t* first, int32_t* last, uint16_t* mlen, uint16_t* flag,
                uint8_t* mapq, uint8_t* nh) {
    if (!b) return RT_EINVAL;
    // the destination is usually fresh (untouched) memory: slices are copied by several threads so that its pages are
    // faulted in by all of them
    parallel_slices(b->ref_id.size(), [&](size_t lo, size_t hi) {
        const size_t m = hi - lo;
        if (ref_id) memcpy(ref_id + lo, b->ref_id.p + lo, 4 * m);
        if (first) memcpy(first + lo, b->first.p + lo, 4 * m);
        if (last) memcpy(last + lo, b->last.p + lo, 4 * m);
        if (mlen) memcpy(mlen + lo, b->mlen.p + lo, 2 * m);
        if (flag) memcpy(flag + lo, b->flag.p + lo, 2 * m);
        if (mapq) memcpy(mapq + lo, b->mapq.p + lo, m);
        if (nh) memcpy(nh + lo, b->nh.p + lo, m);
    });
    return RT_OK;
}

int rt_bam_copy_span(const rt_bam* b, int32_t* pos, int32_t* ref_end) {
    if (!b) return RT_EINVAL;
    parallel_slices(b->pos.size(), [&](size_t lo, size_t hi) {
        if (pos) memcpy(pos + lo, b->pos.p + lo, 4 * (hi - lo));
        if (ref_end) memcpy(ref_end + lo, b->ref_end.p + lo, 4 * (hi - lo));
    });
    return RT_OK;
}

int rt_bam_stream(const rt_bam* b, int n_threads, int64_t cap_blocks, uint32_t* records, int32_t* hdr, int64_t* n_blocks) {
    if (!b) return RT_EINVAL;
    return rt_stream_pack((int64_t)b->ref_id.size(), b->ref_id.data(), b->first.data(), b->last.data(), b->mlen.data(), b->flag.data(),
                          b->mapq.data(), b->nh.data(), n_threads, cap_blocks, records, hdr, n_blocks);
}

}  // extern "C"
