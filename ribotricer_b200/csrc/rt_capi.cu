// rt_capi.cu -- C ABI (include/ribotricer_b200.h) over the sm_100a kernels.
// Host-side state: genome layout, device-resident CSR index, scratch for the host-buffer calls.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "rt_bgzf.h"
#include "rt_host.h"
#include "rt_kernels.cuh"

// rt_host_io.cpp: one chunk of host columns as a run of record-stream blocks (-1: cannot be coded, -2: cap too small)
int64_t rt_stream_pack_range(const int32_t* ref_id, const int32_t* first, const int32_t* last, const uint16_t* mlen, const uint16_t* flag,
                             const uint8_t* mapq, const uint8_t* nh, int64_t m, uint32_t* rec, int32_t* hdr, int64_t cap);

namespace {

thread_local std::string g_last_error;

// Device memory for at least n elements of T, freed with its owner.  reserve() only grows and keeps nothing; it
// allocates one element and 16 bytes at the least, so an empty table is still a valid kernel argument.
template <class T>
struct DevArr {
    T* p = nullptr;
    size_t n = 0;
    DevArr() = default;
    DevArr(DevArr&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevArr& operator=(DevArr&& o) noexcept { std::swap(p, o.p); std::swap(n, o.n); return *this; }
    ~DevArr() { if (p) cudaFree(p); }
    cudaError_t reserve(size_t m) {
        if (m <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        const size_t bytes = std::max<size_t>(sizeof(T) * std::max<size_t>(m, 1), 16);
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) n = bytes / sizeof(T);
        return e;
    }
    // reserve(m), then the first m elements from the host (S: a host type of the same size, e.g. int64_t for long long)
    template <class S>
    cudaError_t upload(const S* src, size_t m) {
        static_assert(sizeof(S) == sizeof(T), "host and device elements differ in size");
        cudaError_t e = reserve(m);
        return e != cudaSuccess || m == 0 ? e : cudaMemcpy(p, src, sizeof(T) * m, cudaMemcpyHostToDevice);
    }
    template <class S>
    cudaError_t upload(const S* src, size_t m, cudaStream_t st) {
        static_assert(sizeof(S) == sizeof(T), "host and device elements differ in size");
        cudaError_t e = reserve(m);
        return e != cudaSuccess || m == 0 ? e : cudaMemcpyAsync(p, src, sizeof(T) * m, cudaMemcpyHostToDevice, st);
    }
};

// Page-locked host memory for n elements of T, freed with its owner.
template <class T>
struct PinnedArr {
    T* p = nullptr;
    size_t n = 0;
    PinnedArr() = default;
    PinnedArr(const PinnedArr&) = delete;
    PinnedArr& operator=(const PinnedArr&) = delete;
    ~PinnedArr() { if (p) cudaFreeHost(p); }
    cudaError_t alloc(size_t m) {
        if (p) cudaFreeHost(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaHostAlloc(&p, sizeof(T) * m, cudaHostAllocDefault);
        if (e == cudaSuccess) n = m;
        return e;
    }
};

// A non-blocking stream, destroyed with its owner; create() does nothing once the stream exists.
struct Stream {
    cudaStream_t s = nullptr;
    Stream() = default;
    Stream(const Stream&) = delete;
    Stream& operator=(const Stream&) = delete;
    ~Stream() { if (s) cudaStreamDestroy(s); }
    cudaError_t create() { return s ? cudaSuccess : cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking); }
    operator cudaStream_t() const { return s; }
};

// An event, destroyed with its owner; create() does nothing once the event exists.
struct Event {
    cudaEvent_t e = nullptr;
    Event() = default;
    Event(const Event&) = delete;
    Event& operator=(const Event&) = delete;
    ~Event() { if (e) cudaEventDestroy(e); }
    cudaError_t create(unsigned flags = cudaEventDefault) { return e ? cudaSuccess : cudaEventCreateWithFlags(&e, flags); }
    operator cudaEvent_t() const { return e; }
};

// stage_ms[k] = the time from ev[k] to ev[k + 1] for k < n: consecutive events bound consecutive stages.
cudaError_t stage_times(const Event* ev, int n, float* stage_ms) {
    for (int k = 0; k < n; ++k)
        if (cudaError_t e = cudaEventElapsedTime(&stage_ms[k], ev[k], ev[k + 1])) return e;
    return cudaSuccess;
}

}  // namespace

struct rt_ctx {
    int device = 0;
    int n_sm = 0;
    std::string err;
    int64_t launches = 0;
    std::atomic<int64_t> h2d_bytes{0};               // copied to the device by the host-buffer entry points so far

    // genome
    int n_contig = 0;
    int pad = 0;
    int64_t plane = 0;
    std::vector<int64_t> contig_len, contig_base;
    DevArr<int2> contig_tab;                         // per contig: (length, first slot >> 5)
    DevArr<double2> uv_table;                        // unit vectors of small codons (rt::fill_uv_table), for phase B's seam windows

    // read-length table
    DevArr<int32_t> len_table;
    bool have_len_table = false;
    int len_base = 20;   // first of the 16 read lengths K1 counts in registers
    int zone_delta_plus = 0, zone_delta_minus = 0;   // smallest P-site displacement from `first` on either strand

    Event ev_scored;                                 // rt_score_host: a part's columns are ready for their copy
    DevArr<unsigned long long> work_counter;         // 4 x u64: work counters of phase A (0) and the fallback (2), fallback count (3)

    // score plan: the work lists of the three scoring launches for one ORF range
    struct ScorePlan {
        int64_t lo = -1, hi = -1;
        DevArr<int32_t> fallback;       // ORFs redone by score_orfs_kernel; capacity hi - lo
        DevArr<int32_t> atom_list;      // atoms the range touches, similar lengths adjacent
        int64_t n_atom_list = 0;
        DevArr<rt::PassDesc> passes;    // compact layout: runs of adjacent atoms for atom_pass_kernel
        int64_t n_passes = 0;
        DevArr<rt::RefRec> refs;        // compose_refs_kernel: one slot per atom reference, groups of 32
        DevArr<rt::RefWarp> ref_warps;
        DevArr<rt::LongAcc> long_acc;   // one per ORF with more than 32 references
        int64_t n_ref_warps = 0;
    };

    // Everything rt_set_index derives from the index; rt_set_index and rt_set_genome replace it as a whole.
    struct Index {
        int64_t n_orf = 0;
        DevArr<uint64_t> orf_desc;
        DevArr<int32_t> orf_len;
        DevArr<uint64_t> exon_entries;
        std::vector<int64_t> bytes_prefix{0};            // n_orf + 1: prefix of 4L + 8E + 42
        std::vector<int64_t> nt_prefix{0};               // n_orf + 1: prefix of L

        // two-phase scoring: atoms (coverage intervals no ORF exon boundary splits) and per-ORF atom refs
        int64_t n_atoms = 0;
        DevArr<uint64_t> atoms;                          // (slot offset << 24) | len
        DevArr<rt::AtomSummary> summaries;               // per-library scratch, written by phase A
        DevArr<uint8_t> atom_nonzero;                    // per-library scratch: atom holds at least one read
        // compact layout: the coverage buffer holds the exon union only (atoms back to back, genome order)
        int layout = RT_LAYOUT_DENSE;
        int64_t compact_elems = 0;                       // int32 elements of a compact coverage buffer (with guard)
        DevArr<unsigned> cbits;                          // one bit per cmap word: the word has members
        unsigned compact_plus_end = 0, compact_end = 0;  // compact index after the last '+' slot / after the last slot
        DevArr<uint2> cmap;                              // per 32 dense slots: member mask | compact index after the last member
        DevArr<uint64_t> atoms_c;                        // the same tables with compact slot offsets
        DevArr<uint64_t> exon_entries_c;
        std::vector<uint64_t> h_atoms;                   // host copies used to build per-range atom lists
        std::vector<uint64_t> h_atoms_c;                 // ... with compact slot offsets
        std::vector<uint64_t> h_orf_refs_desc;           // per ORF: ref begin | n_refs << 40 | reverse << 63
        std::vector<uint32_t> h_ref_atom;                // atom id of every ref (0xffffffff: reads as zeros)
        std::vector<uint64_t> h_ref_ent;                 // refs in profile order

        std::vector<ScorePlan> plans;
    } ix;
    DevArr<unsigned> zone_buf, spill_buf;            // rt_bin_stream_fresh: zone boundaries; spill counter (16 B), spill list

    // scratch for the host-buffer entry points
    struct HostStage {                               // page-locked staging of one chunk's record stream
        PinnedArr<uint32_t> rec;
        PinnedArr<int32_t> hdr;
        Event copied;
        bool busy = false;
    } host_stage[16];
    std::mutex launch_mutex;                         // the packing threads of rt_bin_reads_host launch K1 one at a time
    DevArr<char> read_slot[16];
    Stream slot_stream[16];
    DevArr<int64_t> stats_buf;                       // stats, then length counts
    DevArr<char> score_buf;

    // sparse clear: slots touched by K1 since the last rt_clear_touched
    bool track_touched = false;
    DevArr<unsigned long long> touched_buf;
    DevArr<unsigned long long> n_touched;
    int64_t touched_reserved = 0;    // reads binned (weight +1) since the last clear

    // prepare-orfs (rt_orf_search / rt_orf_fetch): the last search's tables and rows stay on the device until fetched
    struct OrfBufs {
        DevArr<uint8_t> codes, ex_rev, tx_rev, seq, row_type, row_codon;
        DevArr<long long> ex_src, ex_dst, tx_seq, tx_exon, tx_rows, row_off, iv_count, iv_off;
        DevArr<int> ex_len, ex_start, ex_end, ex_before, row_tx, row_start, row_stop, iv_start, iv_end;
        DevArr<int2> tx_cds;
        DevArr<unsigned> claim;
    } orf;
    std::vector<int64_t> orf_iv_ptr;                 // n_rows + 1: interval offsets of the last search
    int64_t orf_rows = 0;

    // orfs-seq (rt_orf_seq_write): the uploaded tables and the two chunk buffers, kept for the next call
    struct SeqBufs {
        DevArr<uint8_t> codes, strand;
        DevArr<long long> exon_ptr, base, id_off, line_off;
        DevArr<int> ex_start, ex_end, contig;
        DevArr<char> ids, out[2];
        DevArr<unsigned> claim;
    } seq;
};

namespace {

int fail(rt_ctx* ctx, int code, const char* fmt, ...) {
    char msg[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(msg, sizeof msg, fmt, ap);
    va_end(ap);
    g_last_error = msg;
    if (ctx) ctx->err = msg;
    return code;
}

#define RT_CUDA(ctx, call)                                                                        \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? RT_ENOMEM : RT_ECUDA,             \
                        "%s failed: %s", #call, cudaGetErrorString(e__));                         \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// The touched-slot list holds one entry per read binned since the last clear; grow it keeping its content.
int ensure_touched_capacity(rt_ctx* ctx, int64_t reads) {
    if ((size_t)reads <= ctx->touched_buf.n) return RT_OK;
    DevArr<unsigned long long> bigger;
    RT_CUDA(ctx, bigger.reserve(std::max((size_t)reads, ctx->touched_buf.n * 2)));
    if (ctx->touched_buf.p) {
        RT_CUDA(ctx, cudaDeviceSynchronize());
        RT_CUDA(ctx, cudaMemcpy(bigger.p, ctx->touched_buf.p, sizeof(unsigned long long) * (size_t)ctx->touched_reserved,
                                cudaMemcpyDeviceToDevice));
    }
    ctx->touched_buf = std::move(bigger);
    return RT_OK;
}

// Two-phase scoring, host side: cut the exon entries of all ORFs at every entry boundary into atoms
// (no ORF exon boundary falls inside an atom; atoms longer than kAtomMaxNt are chopped) and express
// every ORF as its sequence of atoms in profile order.
int build_atoms(rt_ctx* ctx, const std::vector<uint64_t>& desc, const std::vector<uint64_t>& entries) {
    rt_ctx::Index& ix = ctx->ix;
    const uint64_t kZero = rt::kZeroOff;
    std::vector<uint64_t> pts;
    pts.reserve(entries.size() * 2);
    for (uint64_t ent : entries) {
        const uint64_t off = ent >> rt::kLenBits, len = ent & rt::kLenMask;
        if (off == kZero) continue;
        pts.push_back(off);
        pts.push_back(off + len);
    }
    // a human index has 10^7 boundaries: the sort (chunks, then a tree of merges) and the look-ups below run on all cores
    const int n_thr = host_threads(pts.size() >> 16, 16);
    auto parallel_for = [&](size_t n_items, auto&& body) {          // body(lo, hi) on slices of [0, n_items)
        run_parallel(n_thr, [&](int k) { body(n_items * k / n_thr, n_items * (k + 1) / n_thr); });
    };
    parallel_for(pts.size(), [&](size_t lo, size_t hi) { std::sort(pts.begin() + lo, pts.begin() + hi); });
    for (int width = 1; width < n_thr; width *= 2)   // merge k = 0, 2w, 4w, ...: the runs [k, k + w) and [k + w, k + 2w)
        run_parallel((n_thr + width - 1) / (2 * width), [&](int j) {
            const int k = 2 * width * j;
            const size_t a = pts.size() * k / n_thr, m = pts.size() * (k + width) / n_thr;
            const size_t b = pts.size() * std::min(k + 2 * width, n_thr) / n_thr;
            std::inplace_merge(pts.begin() + a, pts.begin() + m, pts.begin() + b);
        });
    pts.erase(std::unique(pts.begin(), pts.end()), pts.end());
    // which elementary intervals [pts[i], pts[i+1]) are covered by an entry
    std::vector<int32_t> diff(pts.size() + 1, 0);
    auto idx_of = [&](uint64_t v) { return (size_t)(std::lower_bound(pts.begin(), pts.end(), v) - pts.begin()); };
    // interval numbers of every entry's two ends, looked up once
    std::vector<uint32_t> ilo(entries.size(), 0), ihi(entries.size(), 0);
    parallel_for(entries.size(), [&](size_t lo, size_t hi) {
        for (size_t e = lo; e < hi; ++e) {
            const uint64_t off = entries[e] >> rt::kLenBits, len = entries[e] & rt::kLenMask;
            if (off == kZero) continue;
            ilo[e] = (uint32_t)idx_of(off);
            ihi[e] = (uint32_t)idx_of(off + len);
        }
    });
    for (size_t e = 0; e < entries.size(); ++e) {
        if ((entries[e] >> rt::kLenBits) == kZero) continue;
        diff[ilo[e]]++;
        diff[ihi[e]]--;
    }
    // atoms of interval i are [atom_begin[i], atom_begin[i+1])
    std::vector<uint32_t> atom_begin(pts.size() + 1, 0);
    ix.h_atoms.clear();
    int64_t cover = 0;
    for (size_t i = 0; i + 1 < pts.size(); ++i) {
        cover += diff[i];
        atom_begin[i] = (uint32_t)ix.h_atoms.size();
        if (cover > 0) {
            uint64_t at = pts[i];
            while (at < pts[i + 1]) {
                const uint64_t piece = std::min<uint64_t>(pts[i + 1] - at, (uint64_t)rt::kAtomMaxNt);
                ix.h_atoms.push_back((at << rt::kLenBits) | piece);
                at += piece;
            }
        }
    }
    if (!pts.empty()) atom_begin[pts.size() - 1] = atom_begin[pts.size()] = (uint32_t)ix.h_atoms.size();
    if (ix.h_atoms.size() >= 0xffffffffull) return fail(ctx, RT_EINVAL, "rt_set_index: too many atoms");
    // per-ORF refs in profile order
    const size_t n_orf = desc.size();
    ix.h_orf_refs_desc.assign(n_orf, 0);
    ix.h_ref_ent.clear();
    ix.h_ref_atom.clear();
    ix.h_ref_ent.reserve(entries.size() * 3 / 2);
    ix.h_ref_atom.reserve(entries.size() * 3 / 2);
    for (size_t o = 0; o < n_orf; ++o) {
        const uint64_t begin = desc[o] & rt::kBeginMask;
        const int n_ent = (int)((desc[o] >> 40) & rt::kMaxEntriesPerOrf);
        const bool rev = (desc[o] >> 63) != 0;
        const size_t ref_begin = ix.h_ref_ent.size();
        for (int k = 0; k < n_ent; ++k) {
            const size_t e = begin + (size_t)(rev ? n_ent - 1 - k : k);
            const uint64_t ent = entries[e];
            const uint64_t off = ent >> rt::kLenBits;
            if (off == kZero) {
                ix.h_ref_ent.push_back(ent);
                ix.h_ref_atom.push_back(0xffffffffu);   // reads-as-zero stretch: no atom
                continue;
            }
            const uint32_t a0 = atom_begin[ilo[e]], a1 = atom_begin[ihi[e]];
            for (uint32_t a = 0; a < a1 - a0; ++a) {
                const uint32_t atom = rev ? a1 - 1 - a : a0 + a;
                ix.h_ref_ent.push_back(ix.h_atoms[atom]);
                ix.h_ref_atom.push_back(atom);
            }
        }
        const size_t cnt = ix.h_ref_ent.size() - ref_begin;
        if (cnt > (size_t)rt::kMaxEntriesPerOrf) return fail(ctx, RT_EINVAL, "rt_set_index: ORF %zu has too many atoms", o);
        ix.h_orf_refs_desc[o] = (uint64_t)ref_begin | ((uint64_t)cnt << 40) | ((uint64_t)rev << 63);
    }
    ix.n_atoms = (int64_t)ix.h_atoms.size();
    // compact layout: atom i starts at the sum of the lengths of the atoms before it
    std::vector<uint64_t>& atoms_c = ix.h_atoms_c;
    atoms_c.assign(ix.h_atoms.size(), 0);
    std::vector<uint64_t> entries_c(entries.size());
    uint64_t cat = 0;
    for (size_t i = 0; i < atoms_c.size(); ++i) {
        const uint64_t len = ix.h_atoms[i] & rt::kLenMask;
        atoms_c[i] = (cat << rt::kLenBits) | len;
        cat += len;
    }
    ix.compact_elems = (int64_t)((cat + 31) / 32 * 32 + 32);
    ix.compact_end = (unsigned)std::min<uint64_t>(cat, 0xffffffffull);
    ix.compact_plus_end = ix.compact_end;        // atoms are in slot order: the first one of the '-' plane ends the '+' part
    for (size_t i = 0; i < atoms_c.size(); ++i)
        if ((ix.h_atoms[i] >> rt::kLenBits) >= (uint64_t)ctx->plane) {
            ix.compact_plus_end = (unsigned)(atoms_c[i] >> rt::kLenBits);
            break;
        }
    for (size_t k = 0; k < entries.size(); ++k) {
        const uint64_t off = entries[k] >> rt::kLenBits, len = entries[k] & rt::kLenMask;
        entries_c[k] = off == kZero ? entries[k] : ((atoms_c[atom_begin[ilo[k]]] >> rt::kLenBits) << rt::kLenBits) | len;
    }
    auto upload = [&](DevArr<uint64_t>& d, const std::vector<uint64_t>& vec) {
        cudaError_t e = d.reserve(vec.size() + 4);   // slack: atom_pass_kernel copies descriptor pairs
        return e == cudaSuccess ? d.upload(vec.data(), vec.size()) : e;
    };
    RT_CUDA(ctx, upload(ix.atoms, ix.h_atoms));
    RT_CUDA(ctx, upload(ix.atoms_c, atoms_c));
    RT_CUDA(ctx, upload(ix.exon_entries_c, entries_c));
    RT_CUDA(ctx, ix.summaries.reserve(ix.h_atoms.size()));
    RT_CUDA(ctx, ix.atom_nonzero.reserve(ix.h_atoms.size()));
    return RT_OK;   // the host copies stay: build_plan_host makes the atom lists and the families from them
}

constexpr size_t kReadBytes = 4 + 4 + 4 + 2 + 2 + 1 + 1;
constexpr int64_t kHostChunkReads = 4 << 20;
constexpr int64_t kPackChunkReads = 1 << 20;      // reads per chunk of the packing pipelines
// stream blocks a chunk may fill: 1.5 records per read (every second read spliced or far from its neighbour) + slack;
// a chunk that needs more goes as plain columns
constexpr int64_t kChunkBlockCap = kPackChunkReads * 3 / 2 / RT_STREAM_BLOCK + 64;
static_assert(kChunkBlockCap * (RT_STREAM_BLOCK * 4 + 16) + 64 <= kPackChunkReads * kReadBytes, "a chunk's stream fits its device slot");
constexpr int64_t kMaxPipes = 16;


}  // namespace

extern "C" {

int rt_abi_version(void) { return RT_ABI_VERSION; }

const char* rt_last_error(const rt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int rt_create(int device, rt_ctx** out) {
    if (!out) return fail(nullptr, RT_EINVAL, "rt_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, RT_ECUDA, "rt_create: no CUDA device (%s); there is no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, RT_EINVAL, "rt_create: device %d out of range [0,%d)", device, n);
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    RT_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, RT_ECUDA, "rt_create: device %d is sm_%d%d; this library is built for sm_100a only",
                    device, prop.major, prop.minor);
    std::unique_ptr<rt_ctx> ctx(new rt_ctx());
    ctx->device = device;
    ctx->n_sm = prop.multiProcessorCount;
    if (ctx->work_counter.reserve(4) != cudaSuccess || ctx->len_table.reserve(RT_LEN_TABLE) != cudaSuccess ||
        ctx->uv_table.reserve(rt::kUvEntries) != cudaSuccess)
        return fail(nullptr, RT_ENOMEM, "rt_create: cudaMalloc failed");
    rt::fill_uv_table_kernel<<<1, 256>>>(ctx->uv_table.p);
    if (cudaDeviceSynchronize() != cudaSuccess)
        return fail(nullptr, RT_ECUDA, "rt_create: %s", cudaGetErrorString(cudaGetLastError()));
    *out = ctx.release();
    return RT_OK;
}

void rt_destroy(rt_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    cudaDeviceSynchronize();   // no stream or page-locked buffer of the ctx goes while work of the ctx may still use it
    delete ctx;
}

int64_t rt_launch_count(const rt_ctx* ctx) { return ctx ? ctx->launches : 0; }
int64_t rt_h2d_bytes(const rt_ctx* ctx) { return ctx ? ctx->h2d_bytes.load() : 0; }

// ------------------------------------------------------------------------------------ genome
int rt_set_genome(rt_ctx* ctx, int n_contig, const int64_t* h_contig_len, int pad) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_set_genome: ctx is NULL");
    if (n_contig < 0 || (n_contig > 0 && !h_contig_len) || pad < 0 || pad > (1 << 20))
        return fail(ctx, RT_EINVAL, "rt_set_genome: bad arguments (n_contig=%d pad=%d)", n_contig, pad);
    DeviceGuard guard(ctx->device);
    ctx->n_contig = n_contig;
    ctx->pad = pad;
    ctx->contig_len.assign(h_contig_len, h_contig_len + n_contig);
    ctx->contig_base.assign(n_contig, 0);
    int64_t at = 0;
    for (int c = 0; c < n_contig; ++c) {
        if (h_contig_len[c] < 0 || h_contig_len[c] > 0x7fffffff - 2ll * pad - 64 - 2ll * RT_MAX_OFFSET)   // K1 adds an offset in 32 bits
            return fail(ctx, RT_EINVAL, "rt_set_genome: contig %d length %lld unsupported", c, (long long)h_contig_len[c]);
        ctx->contig_base[c] = at;
        at += (h_contig_len[c] + 2ll * pad + 1 + 31) / 32 * 32;
    }
    ctx->plane = n_contig ? at : 32;
    if (2 * ctx->plane >= (int64_t)rt::kZeroOff || 2 * ctx->plane / 32 >= 0xffffffffll)
        return fail(ctx, RT_EINVAL, "rt_set_genome: genome too large (2 x plane must stay below 2^37 slots)");
    std::vector<int2> tab((size_t)std::max(1, n_contig));
    for (int c = 0; c < n_contig; ++c) tab[c] = make_int2((int)h_contig_len[c], (int)(ctx->contig_base[c] >> 5));
    RT_CUDA(ctx, ctx->contig_tab.upload(tab.data(), tab.size()));
    // a new genome invalidates the index encoding
    ctx->ix = rt_ctx::Index();
    return RT_OK;
}

int64_t rt_plane_elems(const rt_ctx* ctx) { return ctx ? ctx->plane : 0; }

int rt_get_contig_base(const rt_ctx* ctx, int64_t* h_out) {
    if (!ctx || !h_out) return RT_EINVAL;
    std::copy(ctx->contig_base.begin(), ctx->contig_base.end(), h_out);
    return RT_OK;
}

int rt_set_length_table(rt_ctx* ctx, const int32_t* h_len_table) {
    if (!ctx || !h_len_table) return fail(ctx, RT_EINVAL, "rt_set_length_table: NULL argument");
    DeviceGuard guard(ctx->device);
    for (int i = 0; i < RT_LEN_TABLE; ++i)
        if (h_len_table[i] > RT_LEN_FILTERED && (h_len_table[i] < -RT_MAX_OFFSET || h_len_table[i] > RT_MAX_OFFSET))
            return fail(ctx, RT_EINVAL, "rt_set_length_table: entry %d = %d is neither a sentinel nor an offset in [-%d, %d]", i,
                        h_len_table[i], RT_MAX_OFFSET, RT_MAX_OFFSET);
    RT_CUDA(ctx, cudaMemcpy(ctx->len_table.p, h_len_table, sizeof(int32_t) * RT_LEN_TABLE, cudaMemcpyHostToDevice));
    ctx->have_len_table = true;
    ctx->len_base = 20;
    for (int i = 0; i < RT_LEN_TABLE; ++i)
        if (h_len_table[i] > RT_LEN_FILTERED) {
            ctx->len_base = i;
            break;
        }
    // zone boundaries of rt_bin_stream_fresh: how far before / behind `first` a P-site can lie at the least
    bool any = false;
    for (int i = 0; i < RT_LEN_TABLE; ++i)
        if (h_len_table[i] > RT_LEN_FILTERED) {
            const int plus = h_len_table[i], minus = i - 1 - h_len_table[i];
            ctx->zone_delta_plus = any ? std::min(ctx->zone_delta_plus, plus) : plus;
            ctx->zone_delta_minus = any ? std::min(ctx->zone_delta_minus, minus) : minus;
            any = true;
        }
    if (!any) ctx->zone_delta_plus = ctx->zone_delta_minus = 0;
    return RT_OK;
}

int rt_clear_coverage(rt_ctx* ctx, int32_t* d_cov, void* stream) {
    if (!ctx || !d_cov) return fail(ctx, RT_EINVAL, "rt_clear_coverage: NULL argument");
    if (ctx->plane == 0) return fail(ctx, RT_ESTATE, "rt_clear_coverage: call rt_set_genome first");
    DeviceGuard guard(ctx->device);
    const size_t elems = ctx->ix.layout == RT_LAYOUT_COMPACT ? (size_t)ctx->ix.compact_elems : 2 * (size_t)ctx->plane;
    RT_CUDA(ctx, cudaMemsetAsync(d_cov, 0, sizeof(int32_t) * elems, (cudaStream_t)stream));
    return RT_OK;
}

int rt_set_layout(rt_ctx* ctx, int layout) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_set_layout: ctx is NULL");
    if (layout != RT_LAYOUT_DENSE && layout != RT_LAYOUT_COMPACT) return fail(ctx, RT_EINVAL, "rt_set_layout: unknown layout %d", layout);
    if (layout == RT_LAYOUT_COMPACT) {
        if (ctx->ix.n_orf == 0) return fail(ctx, RT_ESTATE, "rt_set_layout: the compact layout is derived from the index; call rt_set_index first");
        if (ctx->ix.compact_elems >= 0xffffffffll) return fail(ctx, RT_EINVAL, "rt_set_layout: exon union too large for 32-bit compact slots");
        DeviceGuard guard(ctx->device);
        if (!ctx->ix.cmap.p) {
            const size_t words = (size_t)(2 * ctx->plane / 32);
            RT_CUDA(ctx, ctx->ix.cmap.reserve(words));
            RT_CUDA(ctx, cudaMemset(ctx->ix.cmap.p, 0, sizeof(uint2) * words));
            if (ctx->ix.n_atoms > 0) {
                const unsigned grid = (unsigned)std::min<int64_t>((ctx->ix.n_atoms + 7) / 8, (int64_t)ctx->n_sm * 16);
                rt::build_cmap_kernel<<<grid, 256>>>(ctx->ix.atoms.p, ctx->ix.atoms_c.p, ctx->ix.n_atoms, ctx->ix.cmap.p);
                ctx->launches++;
                RT_CUDA(ctx, cudaGetLastError());
            }
            {   // empty words carry the compact index of the next member (cmap_rank: zone boundaries of rt_bin_stream_fresh)
                const size_t tiles = (words + rt::kGapTile - 1) / rt::kGapTile;
                DevArr<unsigned> tile_buf;
                RT_CUDA(ctx, tile_buf.reserve(tiles));
                unsigned* d_tile = tile_buf.p;
                rt::cmap_tile_last_kernel<<<(unsigned)tiles, 256>>>(ctx->ix.cmap.p, (long long)words, d_tile);
                std::vector<unsigned> h_tile(tiles);
                RT_CUDA(ctx, cudaMemcpy(h_tile.data(), d_tile, sizeof(unsigned) * tiles, cudaMemcpyDeviceToHost));
                unsigned carry = 0;
                for (size_t t = 0; t < tiles; ++t) {      // exclusive prefix maximum
                    const unsigned last = h_tile[t];
                    h_tile[t] = carry;
                    carry = std::max(carry, last);
                }
                RT_CUDA(ctx, cudaMemcpy(d_tile, h_tile.data(), sizeof(unsigned) * tiles, cudaMemcpyHostToDevice));
                rt::cmap_fill_gaps_kernel<<<(unsigned)tiles, 256>>>(ctx->ix.cmap.p, (long long)words, d_tile);
                ctx->launches += 2;
                RT_CUDA(ctx, cudaGetLastError());
                RT_CUDA(ctx, cudaDeviceSynchronize());
            }
            RT_CUDA(ctx, ctx->ix.cbits.reserve((words + 31) / 32));
            rt::build_cbits_kernel<<<(unsigned)((words + 255) / 256), 256>>>(ctx->ix.cmap.p, (long long)words, ctx->ix.cbits.p);
            ctx->launches++;
            RT_CUDA(ctx, cudaGetLastError());
            RT_CUDA(ctx, cudaDeviceSynchronize());
        }
    }
    ctx->ix.layout = layout;
    return RT_OK;
}

int64_t rt_coverage_elems(const rt_ctx* ctx) {
    if (!ctx) return 0;
    return ctx->ix.layout == RT_LAYOUT_COMPACT ? ctx->ix.compact_elems : 2 * ctx->plane;
}

int rt_track_touched(rt_ctx* ctx, int enable) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_track_touched: ctx is NULL");
    DeviceGuard guard(ctx->device);
    if (enable && !ctx->n_touched.p) {
        RT_CUDA(ctx, ctx->n_touched.reserve(1));
        RT_CUDA(ctx, cudaMemset(ctx->n_touched.p, 0, sizeof(unsigned long long)));
    }
    ctx->track_touched = enable != 0;
    return RT_OK;
}

int rt_clear_touched(rt_ctx* ctx, int32_t* d_cov, void* stream) {
    if (!ctx || !d_cov) return fail(ctx, RT_EINVAL, "rt_clear_touched: NULL argument");
    if (!ctx->n_touched.p && ctx->ix.layout != RT_LAYOUT_COMPACT)
        return fail(ctx, RT_ESTATE, "rt_clear_touched: call rt_track_touched(ctx, 1) first");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (ctx->ix.layout == RT_LAYOUT_COMPACT) {   // the whole buffer is the exon union: a plain memset is the sparse clear
        RT_CUDA(ctx, cudaMemsetAsync(d_cov, 0, sizeof(int32_t) * (size_t)ctx->ix.compact_elems, st));
        return RT_OK;
    }
    if (ctx->touched_buf.p) {
        rt::clear_touched_kernel<<<(unsigned)ctx->n_sm * 8, 256, 0, st>>>(
            d_cov, ctx->touched_buf.p, ctx->n_touched.p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaMemsetAsync(ctx->n_touched.p, 0, sizeof(unsigned long long), st));
    ctx->touched_reserved = 0;
    return RT_OK;
}

// ------------------------------------------------------------------------------------ K1
}  // extern "C"

namespace {

// Checks and launch of rt_bin_reads: `a` arrives with its read columns filled in.
int launch_bin(rt_ctx* ctx, const char* who, rt::BinArgs& a, int32_t* d_cov, int64_t n, int protocol,
               int weight, int64_t* d_stats, int64_t* d_len_counts, void* stream) {
    if (weight != 1 && weight != -1) return fail(ctx, RT_EINVAL, "%s: weight must be +1 or -1", who);
    if (ctx->plane == 0) return fail(ctx, RT_ESTATE, "%s: call rt_set_genome first", who);
    if (!ctx->have_len_table) return fail(ctx, RT_ESTATE, "%s: call rt_set_length_table first", who);
    if (n < 0 || !d_cov || !d_stats || !d_len_counts) return fail(ctx, RT_EINVAL, "%s: NULL argument or negative n", who);
    if (n == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    a.cov = d_cov;
    a.n = n;
    a.protocol = protocol;
    a.weight = weight;
    a.len_base = ctx->len_base;
    a.len_table = ctx->len_table.p;
    a.contig_tab = ctx->contig_tab.p;
    a.n_contig = ctx->n_contig;
    a.pad = ctx->pad;
    a.plane_words = (unsigned)(ctx->plane >> 5);
    a.stats = reinterpret_cast<unsigned long long*>(d_stats);
    a.len_counts = reinterpret_cast<unsigned long long*>(d_len_counts);
    a.touched = nullptr;
    a.n_touched = nullptr;
    a.cmap = ctx->ix.layout == RT_LAYOUT_COMPACT ? ctx->ix.cmap.p : nullptr;
    a.cbits = ctx->ix.cbits.p;
    if (ctx->track_touched && weight == 1 && !a.cmap) {
        int rc = ensure_touched_capacity(ctx, ctx->touched_reserved + n);
        if (rc != RT_OK) return rc;
        ctx->touched_reserved += n;
        a.touched = ctx->touched_buf.p;
        a.n_touched = ctx->n_touched.p;
    }
    const int64_t per_block = (int64_t)rt::kBinThreads * rt::kBinReadsPerThread;
    const int64_t blocks = (n + per_block - 1) / per_block;
    if (blocks > 0x7fffffff) return fail(ctx, RT_EINVAL, "%s: n too large for one launch", who);
    cudaStream_t st = (cudaStream_t)stream;
    if (a.cmap) rt::bin_psites_kernel<true><<<(unsigned)blocks, rt::kBinThreads, 0, st>>>(a);
    else rt::bin_psites_kernel<false><<<(unsigned)blocks, rt::kBinThreads, 0, st>>>(a);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

}  // namespace

extern "C" {

int rt_bin_reads(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* d_ref_id, const int32_t* d_first,
                 const int32_t* d_last, const uint16_t* d_mlen, const uint16_t* d_flag, const uint8_t* d_mapq,
                 const uint8_t* d_nh, int protocol, int sorted_hint, int weight, int64_t* d_stats,
                 int64_t* d_len_counts, void* stream) {
    (void)sorted_hint;
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bin_reads: ctx is NULL");
    if (n > 0 && (!d_ref_id || !d_first || !d_last || !d_mlen || !d_flag || !d_mapq || !d_nh))
        return fail(ctx, RT_EINVAL, "rt_bin_reads: NULL column");
    rt::BinArgs a{};
    a.ref_id = d_ref_id; a.first = d_first; a.last = d_last; a.mlen = d_mlen; a.flag = d_flag;
    a.mapq = d_mapq; a.nh = d_nh;
    return launch_bin(ctx, "rt_bin_reads", a, d_cov, n, protocol, weight, d_stats, d_len_counts, stream);
}

static int launch_stream(rt_ctx* ctx, const char* who, bool fresh, int32_t* d_cov, int64_t n_blocks, const uint32_t* d_records,
                         const int32_t* d_hdr, int protocol, int weight, int64_t* d_stats, int64_t* d_len_counts, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "%s: ctx is NULL", who);
    if (weight != 1 && weight != -1) return fail(ctx, RT_EINVAL, "%s: weight must be +1 or -1", who);
    if (ctx->plane == 0) return fail(ctx, RT_ESTATE, "%s: call rt_set_genome first", who);
    if (!ctx->have_len_table) return fail(ctx, RT_ESTATE, "%s: call rt_set_length_table first", who);
    if (n_blocks < 0 || !d_cov || !d_stats || !d_len_counts || (n_blocks > 0 && (!d_records || !d_hdr)))
        return fail(ctx, RT_EINVAL, "%s: NULL argument or bad n_blocks", who);
    if ((reinterpret_cast<uintptr_t>(d_records) | reinterpret_cast<uintptr_t>(d_hdr)) & 15)
        return fail(ctx, RT_EINVAL, "%s: d_records and d_hdr must be 16-byte aligned", who);
    if (ctx->track_touched && ctx->ix.layout != RT_LAYOUT_COMPACT)
        return fail(ctx, RT_ESTATE, "%s: the touched-slot list of the dense layout is kept by rt_bin_reads only", who);
    if (fresh && ctx->ix.layout != RT_LAYOUT_COMPACT) return fail(ctx, RT_ESTATE, "%s: needs the compact layout (rt_set_layout)", who);
    if (fresh && (reinterpret_cast<uintptr_t>(d_cov) & 15)) return fail(ctx, RT_EINVAL, "%s: d_cov must be 16-byte aligned", who);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_blocks == 0) {
        if (fresh) RT_CUDA(ctx, cudaMemsetAsync(d_cov, 0, sizeof(int32_t) * (size_t)ctx->ix.compact_elems, st));
        return RT_OK;
    }
    rt::StreamArgs a{};
    a.cov = d_cov;
    a.rec = reinterpret_cast<const uint4*>(d_records);
    a.hdr = reinterpret_cast<const int4*>(d_hdr);
    a.n_blocks = n_blocks;
    a.protocol = protocol;
    a.weight = weight;
    a.len_base = ctx->len_base;
    a.cmap = ctx->ix.layout == RT_LAYOUT_COMPACT ? ctx->ix.cmap.p : nullptr;
    a.cbits = ctx->ix.cbits.p;
    a.len_table = ctx->len_table.p;
    a.contig_tab = ctx->contig_tab.p;
    a.n_contig = ctx->n_contig;
    a.pad = ctx->pad;
    a.plane_words = (unsigned)(ctx->plane >> 5);
    a.stats = reinterpret_cast<unsigned long long*>(d_stats);
    a.len_counts = reinterpret_cast<unsigned long long*>(d_len_counts);
    // persistent: a few CTAs per SM; every warp walks blocks with the next one in flight (cp.async.bulk)
    const unsigned grid = (unsigned)std::min<int64_t>((n_blocks + rt::kStreamWarps - 1) / rt::kStreamWarps, (int64_t)ctx->n_sm * rt::kStreamCtasPerSm);
    if (fresh) {
        // zone boundaries of the blocks (rank of the first position a read of the block can reach), made monotone
        const int64_t tiles = (n_blocks + 1 + rt::kZoneTile - 1) / rt::kZoneTile;
        RT_CUDA(ctx, ctx->zone_buf.reserve(2 * (size_t)(n_blocks + 1) + 4 * (size_t)tiles));
        RT_CUDA(ctx, ctx->spill_buf.reserve((size_t)n_blocks * RT_STREAM_BLOCK + 4));
        rt::ZoneArgs z{};
        z.hdr = a.hdr;
        z.n_blocks = n_blocks;
        z.bounds = ctx->zone_buf.p;
        z.cmap = ctx->ix.cmap.p;
        z.contig_tab = ctx->contig_tab.p;
        z.n_contig = ctx->n_contig;
        z.pad = ctx->pad;
        z.plane_words = a.plane_words;
        z.delta_plus = ctx->zone_delta_plus;
        z.delta_minus = ctx->zone_delta_minus;
        z.plus_end = ctx->ix.compact_plus_end;
        z.minus_end = ctx->ix.compact_end;
        unsigned long long* d_n_spill = reinterpret_cast<unsigned long long*>(ctx->spill_buf.p);
        unsigned* d_tile_max = z.bounds + 2 * (size_t)(n_blocks + 1);
        unsigned* d_tile_carry = d_tile_max + 2 * (size_t)tiles;
        a.zone_bounds = z.bounds;
        a.zone_carry = d_tile_carry;
        a.zone_tiles = tiles;
        a.spill = reinterpret_cast<unsigned*>(d_n_spill + 2);
        a.n_spill = d_n_spill;
        RT_CUDA(ctx, cudaMemsetAsync(d_n_spill, 0, sizeof(unsigned long long), st));
        // the few guard slots behind the last zone belong to no block
        RT_CUDA(ctx, cudaMemsetAsync(d_cov + ctx->ix.compact_end, 0, sizeof(int32_t) * (size_t)(ctx->ix.compact_elems - ctx->ix.compact_end), st));
        rt::zone_bounds_kernel<<<dim3((unsigned)tiles, 2), rt::kZoneTile, 0, st>>>(z, d_tile_max);
        rt::zone_carry_kernel<<<2, 1024, 0, st>>>(d_tile_max, d_tile_carry, tiles, z.plus_end);
        rt::bin_stream_kernel<true, true><<<grid, rt::kStreamThreads, 0, st>>>(a);
        rt::zone_spill_kernel<<<(unsigned)ctx->n_sm * 4, 256, 0, st>>>(d_cov, a.spill, d_n_spill);
        ctx->launches += 4;
    } else {
        if (a.cmap) rt::bin_stream_kernel<true, false><<<grid, rt::kStreamThreads, 0, st>>>(a);
        else rt::bin_stream_kernel<false, false><<<grid, rt::kStreamThreads, 0, st>>>(a);
        ctx->launches++;
    }
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

int rt_bin_stream(rt_ctx* ctx, int32_t* d_cov, int64_t n_blocks, const uint32_t* d_records, const int32_t* d_hdr, int protocol,
                  int weight, int64_t* d_stats, int64_t* d_len_counts, void* stream) {
    return launch_stream(ctx, "rt_bin_stream", false, d_cov, n_blocks, d_records, d_hdr, protocol, weight, d_stats, d_len_counts, stream);
}

int rt_bin_stream_fresh(rt_ctx* ctx, int32_t* d_cov, int64_t n_blocks, const uint32_t* d_records, const int32_t* d_hdr, int protocol,
                        int64_t* d_stats, int64_t* d_len_counts, void* stream) {
    return launch_stream(ctx, "rt_bin_stream_fresh", true, d_cov, n_blocks, d_records, d_hdr, protocol, 1, d_stats, d_len_counts, stream);
}

int rt_bin_stream_host(rt_ctx* ctx, int32_t* d_cov, int64_t n_blocks, const uint32_t* h_records, const int32_t* h_hdr, int protocol,
                       int64_t* h_stats, int64_t* h_len_counts) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bin_stream_host: ctx is NULL");
    if (!h_stats || !h_len_counts) return fail(ctx, RT_EINVAL, "rt_bin_stream_host: NULL output");
    if (n_blocks < 0 || (n_blocks > 0 && (!h_records || !h_hdr))) return fail(ctx, RT_EINVAL, "rt_bin_stream_host: NULL stream");
    DeviceGuard guard(ctx->device);
    const size_t acc_bytes = sizeof(int64_t) * (RT_N_STATS + RT_LEN_TABLE);
    RT_CUDA(ctx, ctx->stats_buf.reserve(RT_N_STATS + RT_LEN_TABLE));
    int64_t* d_stats = ctx->stats_buf.p;
    int64_t* d_len_counts = d_stats + RT_N_STATS;
    for (int s = 0; s < 2; ++s)
        RT_CUDA(ctx, ctx->slot_stream[s].create());
    RT_CUDA(ctx, cudaMemsetAsync(d_stats, 0, acc_bytes, ctx->slot_stream[0]));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    // chunks of 16 MB of records alternate between two device slots: copy of one || K1 of the other
    const int64_t chunk = (16 << 20) / (RT_STREAM_BLOCK * 4);
    const size_t rec_bytes = sizeof(uint32_t) * RT_STREAM_BLOCK * (size_t)chunk;
    int slot = 0;
    for (int64_t at = 0; at < n_blocks; at += chunk, slot ^= 1) {
        const int64_t m = std::min(chunk, n_blocks - at);
        RT_CUDA(ctx, ctx->read_slot[slot].reserve(rec_bytes + sizeof(int32_t) * 4 * (size_t)chunk));
        uint32_t* d_rec = reinterpret_cast<uint32_t*>(ctx->read_slot[slot].p);
        int32_t* d_hdr = reinterpret_cast<int32_t*>(ctx->read_slot[slot].p + rec_bytes);
        cudaStream_t st = ctx->slot_stream[slot];   // stream order protects the slot's previous use
        RT_CUDA(ctx, cudaMemcpyAsync(d_rec, h_records + at * RT_STREAM_BLOCK, sizeof(uint32_t) * RT_STREAM_BLOCK * (size_t)m, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(d_hdr, h_hdr + 4 * at, sizeof(int32_t) * 4 * (size_t)m, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += (int64_t)m * (RT_STREAM_BLOCK * 4 + 16);
        int rc = rt_bin_stream(ctx, d_cov, m, d_rec, d_hdr, protocol, 1, d_stats, d_len_counts, st);
        if (rc != RT_OK) return rc;
    }
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[1]));
    RT_CUDA(ctx, cudaMemcpy(h_stats, d_stats, sizeof(int64_t) * RT_N_STATS, cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(h_len_counts, d_len_counts, sizeof(int64_t) * RT_LEN_TABLE, cudaMemcpyDeviceToHost));
    return RT_OK;
}

int rt_bin_reads_host(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* h_ref_id, const int32_t* h_first,
                      const int32_t* h_last, const uint16_t* h_mlen, const uint16_t* h_flag,
                      const uint8_t* h_mapq, const uint8_t* h_nh, int protocol, int sorted_hint,
                      int64_t* h_stats, int64_t* h_len_counts) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bin_reads_host: ctx is NULL");
    if (!h_stats || !h_len_counts) return fail(ctx, RT_EINVAL, "rt_bin_reads_host: NULL output");
    if (n > 0 && (!h_ref_id || !h_first || !h_last || !h_mlen || !h_flag || !h_mapq || !h_nh))
        return fail(ctx, RT_EINVAL, "rt_bin_reads_host: NULL column");
    DeviceGuard guard(ctx->device);
    // the sparse-clear list of the dense layout is kept by the column kernel only
    const bool use_stream = sorted_hint && !(ctx->track_touched && ctx->ix.layout != RT_LAYOUT_COMPACT);
    const size_t acc_bytes = sizeof(int64_t) * (RT_N_STATS + RT_LEN_TABLE);
    RT_CUDA(ctx, ctx->stats_buf.reserve(RT_N_STATS + RT_LEN_TABLE));
    int64_t* d_stats = ctx->stats_buf.p;
    int64_t* d_len_counts = d_stats + RT_N_STATS;
    for (int s = 0; s < 2; ++s)
        RT_CUDA(ctx, ctx->slot_stream[s].create());
    RT_CUDA(ctx, cudaMemsetAsync(d_stats, 0, acc_bytes, ctx->slot_stream[0]));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    if (ctx->track_touched && ctx->ix.layout != RT_LAYOUT_COMPACT) {   // one growth up front instead of one per chunk
        int rc = ensure_touched_capacity(ctx, ctx->touched_reserved + n);
        if (rc != RT_OK) return rc;
    }
    // Host columns are the 18 B/read a BAM decoder produces.  With `use_stream` (a coordinate-sorted library) they cross
    // PCIe as a 4 B/read record stream: a few pipeline threads each take the next chunk of the library, delta-code it
    // into their own page-locked staging slot, start the copy on their own stream and launch K1 behind it -- so the
    // coding of some chunks, the copies of others and the kernels of yet others overlap.  A chunk that cannot be coded
    // (positions descend: not sorted after all) is sent as plain columns.
    const int64_t chunk = use_stream ? std::min<int64_t>(kPackChunkReads, std::max<int64_t>(n, 1))
                                      : std::min<int64_t>(kHostChunkReads, std::max<int64_t>(n, 1));
    const int64_t n_chunks = (n + chunk - 1) / chunk;
    // the delta coding is the bottleneck of this call (about 1.5 ns per read and thread): one pipeline per hardware thread
    const int n_pipes = use_stream ? (int)std::max<int64_t>(1, std::min<int64_t>({host_threads((size_t)n_chunks, kMaxPipes, "RT_PACK_PIPES"),
                                                                                 kMaxPipes, n_chunks}))
                                   : 2;
    const bool timing = getenv("RT_HOST_TIMING") != nullptr;
    std::atomic<long long> pack_ns{0}, wait_ns{0}, issue_ns{0};
    const auto t_begin = std::chrono::steady_clock::now();
    // per-slot layout: a chunk's record stream (records, then block headers) or its plain columns, widest column first
    const size_t slot_bytes = std::max((size_t)chunk, (size_t)(use_stream ? kPackChunkReads : 0)) * kReadBytes + 64;
    for (int s = 0; s < n_pipes; ++s) {
        RT_CUDA(ctx, ctx->slot_stream[s].create());
        RT_CUDA(ctx, ctx->read_slot[s].reserve(slot_bytes));
        rt_ctx::HostStage& hs = ctx->host_stage[s];
        if (use_stream && !hs.rec.p) {
            RT_CUDA(ctx, hs.rec.alloc(RT_STREAM_BLOCK * (size_t)kChunkBlockCap));
            RT_CUDA(ctx, hs.hdr.alloc(4 * (size_t)kChunkBlockCap));
            RT_CUDA(ctx, hs.copied.create(cudaEventDisableTiming));
        }
        hs.busy = false;
    }
    std::atomic<int64_t> next_chunk{0};
    std::atomic<int> status{RT_OK};
    std::string first_error;
    auto pipeline = [&](int s) {
        cudaSetDevice(ctx->device);
        char* base = ctx->read_slot[s].p;
        // a chunk is either a record stream (records, then block headers) or plain columns
        uint32_t* d_rec = reinterpret_cast<uint32_t*>(base);
        int32_t* d_hdr = reinterpret_cast<int32_t*>(d_rec + RT_STREAM_BLOCK * (size_t)kChunkBlockCap);
        int32_t* d_ref = reinterpret_cast<int32_t*>(base);
        int32_t* d_first = d_ref + chunk;
        int32_t* d_last = d_first + chunk;
        uint16_t* d_mlen = reinterpret_cast<uint16_t*>(d_last + chunk);
        uint16_t* d_flag = d_mlen + chunk;
        uint8_t* d_mapq = reinterpret_cast<uint8_t*>(d_flag + chunk);
        uint8_t* d_nh = d_mapq + chunk;
        cudaStream_t st = ctx->slot_stream[s];      // stream order protects the device slot's previous use
        rt_ctx::HostStage& hs = ctx->host_stage[s];
        auto check = [&](cudaError_t e, const char* what) {
            if (e == cudaSuccess) return true;
            std::lock_guard<std::mutex> lock(ctx->launch_mutex);
            if (status.exchange(RT_ECUDA) == RT_OK) first_error = std::string(what) + ": " + cudaGetErrorString(e);
            return false;
        };
        for (;;) {
            const int64_t c = next_chunk.fetch_add(1);
            if (c >= n_chunks || status.load() != RT_OK) break;
            const int64_t at = c * chunk, m = std::min(chunk, n - at);
            int64_t blocks = -1;
            const auto t0 = std::chrono::steady_clock::now();
            if (use_stream) {
                if (hs.busy && !check(cudaEventSynchronize(hs.copied), "cudaEventSynchronize")) break;   // staging slot free again
                hs.busy = false;
                const auto t1 = std::chrono::steady_clock::now();
                blocks = rt_stream_pack_range(h_ref_id + at, h_first + at, h_last + at, h_mlen + at, h_flag + at, h_mapq + at, h_nh + at, m,
                                              hs.rec.p, hs.hdr.p, kChunkBlockCap);
                if (timing) {
                    wait_ns += std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
                    pack_ns += std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t1).count();
                }
            }
            const auto t2 = std::chrono::steady_clock::now();
            int rc;
            if (blocks >= 0) {
                if (!check(cudaMemcpyAsync(d_rec, hs.rec.p, sizeof(uint32_t) * RT_STREAM_BLOCK * (size_t)blocks, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_hdr, hs.hdr.p, sizeof(int32_t) * 4 * (size_t)blocks, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaEventRecord(hs.copied, st), "cudaEventRecord"))
                    break;
                hs.busy = true;
                ctx->h2d_bytes += (int64_t)blocks * (RT_STREAM_BLOCK * 4 + 16);
                std::lock_guard<std::mutex> lock(ctx->launch_mutex);
                rc = rt_bin_stream(ctx, d_cov, blocks, d_rec, d_hdr, protocol, 1, d_stats, d_len_counts, st);
            } else {
                if (!check(cudaMemcpyAsync(d_first, h_first + at, 4 * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_last, h_last + at, 4 * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_mlen, h_mlen + at, 2 * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_ref, h_ref_id + at, 4 * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_flag, h_flag + at, 2 * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_mapq, h_mapq + at, m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_nh, h_nh + at, m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync"))
                    break;
                ctx->h2d_bytes += (int64_t)m * (int64_t)kReadBytes;
                std::lock_guard<std::mutex> lock(ctx->launch_mutex);
                rc = rt_bin_reads(ctx, d_cov, m, d_ref, d_first, d_last, d_mlen, d_flag, d_mapq, d_nh, protocol, 0, 1,
                                  d_stats, d_len_counts, st);
            }
            if (timing) issue_ns += std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t2).count();
            if (rc != RT_OK) {
                int expected = RT_OK;
                status.compare_exchange_strong(expected, rc);
                break;
            }
        }
    };
    run_parallel(n_pipes, pipeline);
    if (status.load() != RT_OK) return first_error.empty() ? status.load() : fail(ctx, status.load(), "rt_bin_reads_host: %s", first_error.c_str());
    const auto t_issued = std::chrono::steady_clock::now();
    for (int s = 0; s < n_pipes; ++s) {
        RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[s]));
        ctx->host_stage[s].busy = false;
    }
    if (timing) {
        const auto ms = [](auto d) { return std::chrono::duration<double, std::milli>(d).count(); };
        fprintf(stderr, "rt_bin_reads_host: %lld reads, %d pipes, chunk %lld: issue phase %.2f ms, drain %.2f ms; thread-ms packing %.2f, waiting for staging %.2f, "
                        "enqueueing %.2f\n", (long long)n, n_pipes, (long long)chunk, ms(t_issued - t_begin), ms(std::chrono::steady_clock::now() - t_issued),
                pack_ns.load() / 1e6, wait_ns.load() / 1e6, issue_ns.load() / 1e6);
    }
    RT_CUDA(ctx, cudaMemcpy(h_stats, d_stats, sizeof(int64_t) * RT_N_STATS, cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(h_len_counts, d_len_counts, sizeof(int64_t) * RT_LEN_TABLE, cudaMemcpyDeviceToHost));
    return RT_OK;
}

// ------------------------------------------------------------------------------------ index
int rt_set_index(rt_ctx* ctx, int64_t n_orf, const int64_t* h_exon_ptr, const int32_t* h_exon_start,
                 const int32_t* h_exon_end, const int32_t* h_orf_contig, const uint8_t* h_orf_strand) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_set_index: ctx is NULL");
    if (ctx->plane == 0) return fail(ctx, RT_ESTATE, "rt_set_index: call rt_set_genome first");
    if (n_orf < 0 || !h_exon_ptr || (n_orf > 0 && (!h_orf_contig || !h_orf_strand)))
        return fail(ctx, RT_EINVAL, "rt_set_index: NULL argument");
    DeviceGuard guard(ctx->device);
    const int64_t max_piece = (int64_t)rt::kLenMask;
    std::vector<uint64_t> desc((size_t)n_orf);
    std::vector<uint64_t> entries;
    entries.reserve((size_t)(h_exon_ptr[n_orf] - h_exon_ptr[0]) + 16);
    std::vector<int64_t> bytes_prefix((size_t)n_orf + 1, 0), nt_prefix((size_t)n_orf + 1, 0);
    auto push = [&](int64_t off, int64_t len) {   // off < 0: zeros
        while (len > 0) {
            const int64_t piece = std::min(len, max_piece);
            entries.push_back(((off < 0 ? rt::kZeroOff : (uint64_t)off) << rt::kLenBits) | (uint64_t)piece);
            if (off >= 0) off += piece;
            len -= piece;
        }
    };
    for (int64_t o = 0; o < n_orf; ++o) {
        const int64_t e0 = h_exon_ptr[o], e1 = h_exon_ptr[o + 1];
        if (e1 < e0) return fail(ctx, RT_EINVAL, "rt_set_index: exon_ptr not monotone at ORF %lld", (long long)o);
        const int c = h_orf_contig[o];
        const int s = h_orf_strand[o];
        const bool covered = c >= 0 && c < ctx->n_contig && (s == 0 || s == 1);
        const size_t begin = entries.size();
        int64_t L = 0;
        for (int64_t e = e0; e < e1; ++e) {
            const int64_t st = h_exon_start[e], en = h_exon_end[e];
            if (en < st) return fail(ctx, RT_EINVAL, "rt_set_index: ORF %lld has an empty interval %lld-%lld",
                                     (long long)o, (long long)st, (long long)en);
            L += en - st + 1;
            if (!covered) {
                push(-1, en - st + 1);
                continue;
            }
            // positions outside the padded contig have no slot: they read as 0 (missing dict key)
            const int64_t lo = 1 - ctx->pad, hi = ctx->contig_len[c] + ctx->pad;
            const int64_t a = std::max(st, lo), b = std::min(en, hi);
            if (a > b) {
                push(-1, en - st + 1);
                continue;
            }
            if (st < a) push(-1, a - st);
            push((int64_t)s * ctx->plane + ctx->contig_base[c] + ctx->pad + a, b - a + 1);
            if (b < en) push(-1, en - b);
        }
        if (L > 0x7fffffff) return fail(ctx, RT_EINVAL, "rt_set_index: ORF %lld longer than 2^31-1 nt", (long long)o);
        const size_t cnt = entries.size() - begin;
        if (cnt > (size_t)rt::kMaxEntriesPerOrf)
            return fail(ctx, RT_EINVAL, "rt_set_index: ORF %lld has too many intervals", (long long)o);
        if (begin >= rt::kBeginMask) return fail(ctx, RT_EINVAL, "rt_set_index: index too large");
        desc[o] = (uint64_t)begin | ((uint64_t)cnt << 40) | ((uint64_t)(s == 1) << 63);
        nt_prefix[o + 1] = nt_prefix[o] + L;
        bytes_prefix[o + 1] = bytes_prefix[o] + 4 * L + 8 * (e1 - e0) + 42;
    }
    // the old index goes only now, so that an index refused above leaves it intact; a failure from here on (a CUDA
    // error, too many atoms) leaves an empty index
    rt_ctx::Index& ix = ctx->ix;
    ix = rt_ctx::Index();
    ix.bytes_prefix = std::move(bytes_prefix);
    ix.nt_prefix = std::move(nt_prefix);
    {
        std::vector<int32_t> lens((size_t)n_orf);
        for (int64_t o = 0; o < n_orf; ++o) lens[o] = (int32_t)(ix.nt_prefix[o + 1] - ix.nt_prefix[o]);
        RT_CUDA(ctx, ix.orf_len.upload(lens.data(), lens.size()));
    }
    RT_CUDA(ctx, ix.orf_desc.upload(desc.data(), desc.size()));
    RT_CUDA(ctx, ix.exon_entries.upload(entries.data(), entries.size()));
    {
        const auto t_atoms = std::chrono::steady_clock::now();
        int rc = build_atoms(ctx, desc, entries);
        if (getenv("RT_HOST_TIMING"))
            fprintf(stderr, "rt_set_index: build_atoms %.1f ms (%zu ORFs, %zu exon entries, %zu atoms)\n",
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_atoms).count(), desc.size(), entries.size(),
                    ix.h_atoms.size());
        if (rc != RT_OK) return rc;
    }
    ix.n_orf = n_orf;
    return RT_OK;
}

int64_t rt_index_orfs(const rt_ctx* ctx) { return ctx ? ctx->ix.n_orf : 0; }

int64_t rt_index_score_bytes(const rt_ctx* ctx, int64_t lo, int64_t hi) {
    if (!ctx || lo < 0 || hi > ctx->ix.n_orf || lo > hi) return -1;
    return ctx->ix.bytes_prefix[hi] - ctx->ix.bytes_prefix[lo];
}

int64_t rt_index_total_nt(const rt_ctx* ctx, int64_t lo, int64_t hi) {
    if (!ctx || lo < 0 || hi > ctx->ix.n_orf || lo > hi) return -1;
    return ctx->ix.nt_prefix[hi] - ctx->ix.nt_prefix[lo];
}

int rt_shard_bounds(const rt_ctx* ctx, int n_shards, int64_t* h_bounds) {
    if (!ctx || n_shards < 1 || !h_bounds) return RT_EINVAL;
    const int64_t total = ctx->ix.bytes_prefix.back();
    h_bounds[0] = 0;
    for (int s = 1; s < n_shards; ++s) {
        const int64_t target = (int64_t)((__int128)total * s / n_shards);
        auto it = std::lower_bound(ctx->ix.bytes_prefix.begin(), ctx->ix.bytes_prefix.end(), target);
        h_bounds[s] = std::max<int64_t>(h_bounds[s - 1], it - ctx->ix.bytes_prefix.begin());
        if (h_bounds[s] > ctx->ix.n_orf) h_bounds[s] = ctx->ix.n_orf;
    }
    h_bounds[n_shards] = ctx->ix.n_orf;
    return RT_OK;
}

// ------------------------------------------------------------------------------------ K2+K3
}  // extern "C"

namespace {

// What get_plan works out on the host for the ORFs [lo, hi) before anything touches the device: pure functions of the
// index arrays of the ctx, so the part plans of rt_score_host can be built side by side.
struct PlanHost {
    int64_t lo = 0, hi = 0;
    std::vector<rt::PassDesc> passes;         // phase A
    std::vector<int32_t> alist;               // atoms of the range, similar lengths adjacent
    std::vector<rt::RefRec> refs;             // phase B slots
    std::vector<rt::RefWarp> warps;
    int n_long_b = 0;                         // ORFs with more than 32 references (phase B accumulators)
};

void build_plan_host(const rt_ctx* ctx, int64_t lo, int64_t hi, PlanHost& ph) {
    const int64_t n = hi - lo;
    const auto t_plan = std::chrono::steady_clock::now();
    ph.lo = lo;
    ph.hi = hi;
    const bool plan_timing = getenv("RT_HOST_TIMING") != nullptr;
    auto t_mark = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!plan_timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "  get_plan: %-28s %.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_mark).count());
        t_mark = now;
    };
    {   // atoms the ORFs of the range refer to; sorted by length inside windows so that the four atoms of
        // a warp are balanced while genomic neighbours stay close in time
        std::vector<uint8_t> used((size_t)ctx->ix.n_atoms, 0);
        for (int64_t o = lo; o < hi; ++o) {
            const uint64_t d = ctx->ix.h_orf_refs_desc[o];
            const uint64_t b = d & rt::kBeginMask, c = (d >> 40) & rt::kMaxEntriesPerOrf;
            for (uint64_t k = b; k < b + c; ++k)
                if (ctx->ix.h_ref_atom[k] != 0xffffffffu) used[ctx->ix.h_ref_atom[k]] = 1;
        }
        std::vector<int32_t>& alist = ph.alist;
        for (int64_t a = 0; a < ctx->ix.n_atoms; ++a)
            if (used[a]) alist.push_back((int32_t)a);
        {   // passes of the streamed phase A: consecutive atom ids are adjacent in the compact buffer
            std::vector<rt::PassDesc>& passes = ph.passes;
            const uint64_t* ac = ctx->ix.h_atoms_c.data();
            size_t i = 0;
            while (i < alist.size()) {
                const uint32_t a0 = (uint32_t)alist[i];
                uint32_t n = 0, pieces = 0, slots = 0;
                while (i < alist.size() && n < (uint32_t)rt::kPassPieces && (uint32_t)alist[i] == a0 + n) {
                    const uint32_t len = (uint32_t)(ac[a0 + n] & rt::kLenMask);
                    const uint32_t np = (len + rt::kPieceNt - 1) / rt::kPieceNt;
                    if (pieces + np > (uint32_t)rt::kPassPieces) break;
                    pieces += np;
                    slots += len;
                    ++n;
                    ++i;
                }
                const uint64_t s0 = ac[a0] >> rt::kLenBits, q0 = s0 & ~3ull, q1 = (s0 + slots + 3) & ~3ull;
                passes.push_back({a0, n | ((uint32_t)((q1 - q0) >> 2) << 8), (uint32_t)(q0 >> 2), (uint32_t)(s0 - q0)});
            }
        }
        constexpr size_t kAtomWindow = 4096;
        for (size_t w0 = 0; w0 < alist.size(); w0 += kAtomWindow) {
            auto b = alist.begin() + w0, e = alist.begin() + std::min(alist.size(), w0 + kAtomWindow);
            std::stable_sort(b, e, [&](int32_t x, int32_t y) {
                return (ctx->ix.h_atoms[x] & rt::kLenMask) > (ctx->ix.h_atoms[y] & rt::kLenMask);
            });
        }
    }
    lap("atom list + passes");
    {
        // Phase B work list.  FAMILIES: candidate ORFs of one transcript that share their stop are suffixes of the
        // longest one -- same atoms from some reference on (the index is cut into atoms at every ORF start).  The
        // longest ORF of a family (the parent) lays its references out, one per slot; an ORF whose reference list is a
        // proper suffix of it (a child) is just marked on the slot where it starts.  compose_refs_kernel forms
        // suffix sums over the parent's slots, so every reference is visited once per family instead of once per ORF.
        // Families never straddle a group of 32 slots; ORFs with more than 32 references stay alone and fill whole groups.
        std::vector<rt::RefRec>& refs = ph.refs;
        std::vector<rt::RefWarp>& warps = ph.warps;
        refs.reserve((size_t)(ctx->ix.h_ref_ent.size() / std::max<int64_t>(1, ctx->ix.n_orf) * n * 3 / 4 + 64));
        const rt::RefRec pad_rec{0xffffffffu, 0u, 0u, -1};
        int& n_long = ph.n_long_b;
        auto pad_group = [&]() {
            while (refs.size() % 32) refs.push_back(pad_rec);
            warps.resize(refs.size() / 32, rt::RefWarp{-1, 0, -1, 0});
        };
        auto desc_of = [&](int64_t o, uint64_t& rb, uint64_t& cnt, uint32_t& rev) {
            const uint64_t d = ctx->ix.h_orf_refs_desc[o];
            rb = d & rt::kBeginMask;
            cnt = (d >> 40) & (uint64_t)rt::kMaxEntriesPerOrf;
            rev = (uint32_t)(d >> 63);
        };
        // hash of a reference list, powers counted from its END, so that the hash of a suffix of a parent equals the
        // hash of the child that is that suffix
        const uint64_t kB = 0x9E3779B97F4A7C15ull;
        auto elem = [&](uint64_t k) {
            uint64_t x = ((uint64_t)ctx->ix.h_ref_atom[k] << 25) ^ (ctx->ix.h_ref_ent[k] & rt::kLenMask);
            x ^= x >> 31; x *= 0xD6E8FEB86659FD93ull; x ^= x >> 29;
            return x | 1ull;
        };
        std::vector<uint64_t> full_hash((size_t)n);
        std::unordered_multimap<uint64_t, int64_t> by_hash;
        by_hash.reserve((size_t)n * 2);
        for (int64_t o = lo; o < hi; ++o) {
            uint64_t rb, cnt; uint32_t rev;
            desc_of(o, rb, cnt, rev);
            uint64_t h = rev ? 0x5bd1e995ull : 0x1b873593ull, pw = 1;
            for (uint64_t k = cnt; k-- > 0;) { h += elem(rb + k) * pw; pw *= kB; }
            full_hash[o - lo] = h;
            if (cnt >= 1 && cnt <= 31) by_hash.emplace(h, o);          // a child has at most 31 references
        }
        lap("reference-list hashes");
        std::vector<int32_t> parent_of((size_t)n, -1);                   // -1: not a child
        std::vector<int64_t> order((size_t)n);
        for (int64_t i = 0; i < n; ++i) order[i] = lo + i;
        auto refs_of = [&](int64_t o) { return (ctx->ix.h_orf_refs_desc[o] >> 40) & (uint64_t)rt::kMaxEntriesPerOrf; };
        std::stable_sort(order.begin(), order.end(), [&](int64_t x, int64_t y) { return refs_of(x) > refs_of(y); });
        // children[o - lo]: (position in the parent's list, child ORF)
        std::vector<std::vector<std::pair<int, int64_t>>> children((size_t)n);
        for (int64_t o : order) {
            if (parent_of[o - lo] >= 0) continue;
            uint64_t rb, cnt; uint32_t rev;
            desc_of(o, rb, cnt, rev);
            if (cnt < 2 || cnt > 32) continue;
            uint64_t h = rev ? 0x5bd1e995ull : 0x1b873593ull, pw = 1;
            for (uint64_t k = cnt; k-- > 1;) {                           // proper suffixes starting at k = cnt-1 .. 1
                h += elem(rb + k) * pw;
                pw *= kB;
                auto range = by_hash.equal_range(h);
                for (auto it = range.first; it != range.second; ++it) {
                    const int64_t c = it->second;
                    if (c == o || parent_of[c - lo] >= 0 || !children[c - lo].empty()) continue;
                    uint64_t crb, ccnt; uint32_t crev;
                    desc_of(c, crb, ccnt, crev);
                    if (crev != rev || ccnt != cnt - k) continue;
                    // a child's first reference must hold two values: then every seam window of the references after it
                    // starts inside the child (with one value, the window two before the next reference would not)
                    if ((ctx->ix.h_ref_ent[crb] & rt::kLenMask) < 2) continue;
                    bool same = true;
                    for (uint64_t j = 0; j < ccnt && same; ++j)
                        same = ctx->ix.h_ref_atom[crb + j] == ctx->ix.h_ref_atom[rb + k + j] &&
                               (ctx->ix.h_ref_ent[crb + j] & rt::kLenMask) == (ctx->ix.h_ref_ent[rb + k + j] & rt::kLenMask);
                    if (!same) continue;
                    parent_of[c - lo] = (int32_t)(o - lo);
                    children[o - lo].push_back({(int)k, c});
                    break;                                               // one ORF per starting slot
                }
            }
        }
        lap("families (suffix matching)");
        for (int64_t o = lo; o < hi; ++o) {
            if (parent_of[o - lo] >= 0) continue;                        // laid out with its parent
            uint64_t rb, cnt; uint32_t rev;
            desc_of(o, rb, cnt, rev);
            if (cnt > 32 || refs.size() % 32 + std::max<uint64_t>(cnt, 1) > 32) pad_group();
            const size_t w0 = refs.size() / 32, first_slot = refs.size();
            uint64_t P = 0;
            const uint64_t L = (uint64_t)(ctx->ix.nt_prefix[o + 1] - ctx->ix.nt_prefix[o]);
            auto flags_of = [&](uint64_t len, uint64_t l_mod3) -> uint32_t {
                return ((uint32_t)(P % 3) << rt::kRefPmod3Shift) | (P >= 1 ? rt::kRefPge1 : 0u) | (P >= 2 ? rt::kRefPge2 : 0u) |
                       (P + len == L ? rt::kRefLast : 0u) | ((uint32_t)l_mod3 << rt::kRefLmod3Shift) | (rev ? rt::kRefRev : 0u);
            };
            for (uint64_t k = 0; k < cnt; ++k) {
                const uint32_t len = (uint32_t)(ctx->ix.h_ref_ent[rb + k] & rt::kLenMask);
                // L mod 3 of the ORF that starts on this slot; a long ORF carries its own on every slot (its last
                // group applies the trailing partial codon itself)
                const uint64_t lm3 = (k == 0 || cnt > 32) ? L % 3 : 0;
                refs.push_back({ctx->ix.h_ref_atom[rb + k], len | flags_of(len, lm3), (uint32_t)((len + P) % 3) | (k == 0 ? rt::kRefFamilyHead : 0u),
                                k == 0 ? (int32_t)o : -2});
                P += len;
            }
            if (cnt == 0) refs.push_back({0xffffffffu, flags_of(0, L % 3), rt::kRefFamilyHead, (int32_t)o});   // an ORF without intervals still gets its row
            for (const auto& ch : children[o - lo]) {
                rt::RefRec& r = refs[first_slot + (size_t)ch.first];
                const uint64_t Lc = (uint64_t)(ctx->ix.nt_prefix[ch.second + 1] - ctx->ix.nt_prefix[ch.second]);
                r.orf = (int32_t)ch.second;
                r.len_flags = (r.len_flags & ~(3u << rt::kRefLmod3Shift)) | ((uint32_t)(Lc % 3) << rt::kRefLmod3Shift);
            }
            if (cnt > 32) {
                pad_group();
                const int groups = (int)(refs.size() / 32 - w0);
                for (size_t g = w0; g < warps.size(); ++g) warps[g] = rt::RefWarp{n_long, groups, (int32_t)o, 0};
                ++n_long;
            }
        }
        pad_group();
        lap("slot layout");
    }
    if (plan_timing)
        fprintf(stderr, "get_plan [%lld, %lld): %.1f ms on the host\n", (long long)lo, (long long)hi,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_plan).count());
}

// The device side of a plan: the host arrays of `ph` uploaded, the plan entered into the (bounded) cache of the ctx.
int upload_plan(rt_ctx* ctx, PlanHost& ph, rt_ctx::ScorePlan** out) {
    const int64_t lo = ph.lo, hi = ph.hi, n = hi - lo;
    if (ctx->ix.plans.size() >= 24)   // bounded cache (rt_score_host keeps four part plans per range it is asked for)
        ctx->ix.plans.erase(ctx->ix.plans.begin());
    rt_ctx::ScorePlan p;
    p.lo = lo;
    p.hi = hi;
    RT_CUDA(ctx, p.fallback.reserve((size_t)n));
    p.n_passes = (int64_t)ph.passes.size();
    RT_CUDA(ctx, p.passes.upload(ph.passes.data(), ph.passes.size()));
    p.n_atom_list = (int64_t)ph.alist.size();
    RT_CUDA(ctx, p.atom_list.upload(ph.alist.data(), ph.alist.size()));
    p.n_ref_warps = (int64_t)ph.warps.size();
    RT_CUDA(ctx, p.refs.upload(ph.refs.data(), ph.refs.size()));
    RT_CUDA(ctx, p.ref_warps.upload(ph.warps.data(), ph.warps.size()));
    std::vector<rt::LongAcc> acc((size_t)std::max(1, ph.n_long_b));
    memset(acc.data(), 0, sizeof(rt::LongAcc) * acc.size());
    for (auto& a : acc) a.mn = 0xffffffffu;
    RT_CUDA(ctx, p.long_acc.upload(acc.data(), acc.size()));
    ctx->ix.plans.push_back(std::move(p));
    *out = &ctx->ix.plans.back();
    return RT_OK;
}

int get_plan(rt_ctx* ctx, int64_t lo, int64_t hi, rt_ctx::ScorePlan** out) {
    for (auto& p : ctx->ix.plans)
        if (p.lo == lo && p.hi == hi) {
            *out = &p;
            return RT_OK;
        }
    PlanHost ph;
    build_plan_host(ctx, lo, hi, ph);
    return upload_plan(ctx, ph, out);
}

// The plans of several ranges at once (the parts of rt_score_host): the host halves are built side by side, one thread per
// range that is not in the cache yet; the uploads follow one after the other in range order.
int prebuild_plans(rt_ctx* ctx, const std::vector<int64_t>& cut) {
    std::vector<PlanHost> todo;
    for (size_t i = 0; i + 1 < cut.size(); ++i) {
        const int64_t a = cut[i], b = cut[i + 1];
        bool cached = a == b;
        for (auto& p : ctx->ix.plans) cached = cached || (p.lo == a && p.hi == b);
        if (!cached) {
            todo.emplace_back();
            todo.back().lo = a;
            todo.back().hi = b;
        }
    }
    if (todo.size() < 2) return RT_OK;           // get_plan does a single one just as well
    run_parallel((int)todo.size(), [&](int k) { build_plan_host(ctx, todo[(size_t)k].lo, todo[(size_t)k].hi, todo[(size_t)k]); });
    for (PlanHost& ph : todo) {
        rt_ctx::ScorePlan* unused = nullptr;
        const int rc = upload_plan(ctx, ph, &unused);
        if (rc != RT_OK) return rc;
    }
    return RT_OK;
}

template <typename Kernel>
unsigned persistent_grid(rt_ctx* ctx, Kernel k, int64_t work_items) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, rt::kScoreWarps * 32, 0) != cudaSuccess) per_sm = 1;
    per_sm = std::max(per_sm, 1);
    const int64_t want = (work_items + rt::kScoreWarps - 1) / rt::kScoreWarps;
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)ctx->n_sm * per_sm));
}

}  // namespace

extern "C" {

int rt_score(rt_ctx* ctx, const int32_t* d_cov, int64_t orf_lo, int64_t orf_hi, const rt_score_params* params,
             const rt_score_out* d_out, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_score: ctx is NULL");
    if (!d_cov || !params || !d_out) return fail(ctx, RT_EINVAL, "rt_score: NULL argument");
    if (orf_lo < 0 || orf_hi > ctx->ix.n_orf || orf_lo > orf_hi)
        return fail(ctx, RT_EINVAL, "rt_score: ORF range [%lld,%lld) outside the index [0,%lld)", (long long)orf_lo,
                    (long long)orf_hi, (long long)ctx->ix.n_orf);
    if (orf_lo == orf_hi) return RT_OK;
    if (!d_out->score || !d_out->valid || !d_out->count || !d_out->length)
        return fail(ctx, RT_EINVAL, "rt_score: score/valid/count/length columns are required");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    rt_ctx::ScorePlan* plan = nullptr;
    int rc = get_plan(ctx, orf_lo, orf_hi, &plan);
    if (rc != RT_OK) return rc;
    RT_CUDA(ctx, cudaMemsetAsync(ctx->work_counter.p, 0, 4 * sizeof(unsigned long long), st));
    rt::ScoreArgs a;
    a.cov = d_cov;
    a.orf_desc = ctx->ix.orf_desc.p;
    const bool compact = ctx->ix.layout == RT_LAYOUT_COMPACT;
    a.exon_entries = compact ? ctx->ix.exon_entries_c.p : ctx->ix.exon_entries.p;
    a.orf_len = ctx->ix.orf_len.p;
    a.orf_lo = orf_lo;
    a.n_fallback = reinterpret_cast<unsigned*>(ctx->work_counter.p + 3);
    a.prm = *params;
    a.out = *d_out;
    const int threads = rt::kScoreWarps * 32;
    // the per-frame minima only matter for --min_reads_per_codon > 0 or when the caller asks for min_codon
    const bool want_min = d_out->min_codon != nullptr || params->min_reads_per_codon > 0.0;
    // phase A: every atom the range touches is scanned once
    if (plan->n_atom_list > 0) {
        if (compact) {
            // streamed phase A: the compact buffer is read once, front to back, through TMA into shared memory
            rt::PassArgs pa;
            pa.cov = d_cov;
            pa.atoms = ctx->ix.atoms_c.p;
            pa.passes = plan->passes.p;
            pa.n_passes = (unsigned)plan->n_passes;
            pa.out = ctx->ix.summaries.p;
            pa.nonzero = ctx->ix.atom_nonzero.p;
            const size_t smem = rt::kUvEntries * sizeof(double2) + (size_t)rt::kPassWarps * rt::kPassStages * rt::kPassStageBytes;
            const auto kern = want_min ? rt::atom_pass_kernel<true> : rt::atom_pass_kernel<false>;
            RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const int64_t want = (plan->n_passes + rt::kPassWarps - 1) / rt::kPassWarps;
            const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, ctx->n_sm));
            kern<<<grid, rt::kPassWarps * 32, smem, st>>>(pa);
        } else {
            rt::AtomArgs aa;
            aa.cov = d_cov;
            aa.atoms = ctx->ix.atoms.p;
            aa.list = plan->atom_list.p;
            aa.n_list = plan->n_atom_list;
            aa.work_counter = ctx->work_counter.p + 0;
            aa.out = ctx->ix.summaries.p;
            aa.nonzero = ctx->ix.atom_nonzero.p;
            const auto kern = want_min ? rt::atom_summary_kernel<true> : rt::atom_summary_kernel<false>;
            const int g = 32 / rt::kAtomLPO;
            kern<<<persistent_grid(ctx, kern, (plan->n_atom_list + g - 1) / g), threads, 0, st>>>(aa);
        }
        ctx->launches++;
    }
    // phase B: the ORFs of every family from the summaries of their atoms
    rt::RefComposeArgs ra;
    ra.refs = plan->refs.p;
    ra.warps = plan->ref_warps.p;
    ra.n_warps = plan->n_ref_warps;
    ra.summaries = ctx->ix.summaries.p;
    ra.atom_nonzero = ctx->ix.atom_nonzero.p;
    ra.uv_table = ctx->uv_table.p;
    ra.want_min = want_min ? 1 : 0;
    ra.orf_len = ctx->ix.orf_len.p;
    ra.orf_lo = orf_lo;
    ra.fallback = plan->fallback.p;
    ra.n_fallback = a.n_fallback;
    ra.long_acc = plan->long_acc.p;
    ra.prm = *params;
    ra.out = *d_out;
    if (ra.n_warps > 0) {
        if (want_min) rt::compose_refs_kernel<true><<<(unsigned)((ra.n_warps + 7) / 8), 256, 0, st>>>(ra);
        else rt::compose_refs_kernel<false><<<(unsigned)((ra.n_warps + 7) / 8), 256, 0, st>>>(ra);
    }
    ctx->launches++;
    // ORFs holding counts >= 2^20: redone by the generic kernel (normally none)
    a.list = plan->fallback.p;
    a.n_list = 0;
    a.n_list_dev = a.n_fallback;
    a.work_counter = ctx->work_counter.p + 2;
    rt::score_orfs_kernel<<<(unsigned)ctx->n_sm, threads, 0, st>>>(a);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

int rt_score_host(rt_ctx* ctx, const int32_t* d_cov, int64_t orf_lo, int64_t orf_hi, const rt_score_params* params,
                  const rt_score_out* h_out) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_score_host: ctx is NULL");
    if (!h_out || !params) return fail(ctx, RT_EINVAL, "rt_score_host: NULL argument");
    if (orf_lo < 0 || orf_hi > ctx->ix.n_orf || orf_lo > orf_hi) return fail(ctx, RT_EINVAL, "rt_score_host: bad ORF range");
    const int64_t n = orf_hi - orf_lo;
    if (n == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    // one scratch allocation, 8-byte columns first
    const size_t bytes = (size_t)n * (8 + 8 + 24 + 4 + 4 + 4 + 12 + 1) + 256;
    RT_CUDA(ctx, ctx->score_buf.reserve(bytes));
    char* p = ctx->score_buf.p;
    rt_score_out d{};
    d.score = reinterpret_cast<double*>(p); p += 8 * n;
    d.count = reinterpret_cast<int64_t*>(p); p += 8 * n;
    d.frame_s = h_out->frame_s ? reinterpret_cast<double*>(p) : nullptr; p += 24 * n;
    d.valid = reinterpret_cast<int32_t*>(p); p += 4 * n;
    d.length = reinterpret_cast<int32_t*>(p); p += 4 * n;
    d.min_codon = h_out->min_codon ? reinterpret_cast<int32_t*>(p) : nullptr; p += 4 * n;
    d.frame_K = h_out->frame_K ? reinterpret_cast<int32_t*>(p) : nullptr; p += 12 * n;
    d.status = reinterpret_cast<uint8_t*>(p);
    // A large range is scored in a few byte-balanced parts so that the result columns of part i cross PCIe (copy stream)
    // while part i + 1 is being scored; every part has its own cached plan, the columns are the same (sums are exact).
    int n_parts = n >= (1 << 20) ? 4 : 1;
    if (const char* e = getenv("RT_SCORE_HOST_PARTS")) n_parts = std::max(1, std::min(16, atoi(e)));
    n_parts = (int)std::min<int64_t>(n_parts, n);
    std::vector<int64_t> cut((size_t)n_parts + 1, orf_lo);
    cut[(size_t)n_parts] = orf_hi;
    const int64_t* bp = ctx->ix.bytes_prefix.data();
    for (int i = 1; i < n_parts; ++i) {
        const int64_t target = bp[orf_lo] + (bp[orf_hi] - bp[orf_lo]) * i / n_parts;
        cut[(size_t)i] = std::max<int64_t>(cut[(size_t)i - 1], std::lower_bound(bp + orf_lo, bp + orf_hi, target) - bp);
    }
    if (n_parts > 1) {                 // the parts' plans that are not cached yet: host halves built side by side
        const int rc = prebuild_plans(ctx, cut);
        if (rc != RT_OK) return rc;
    }
    RT_CUDA(ctx, ctx->slot_stream[0].create());
    cudaStream_t copy = n_parts > 1 ? ctx->slot_stream[0].s : nullptr;
    if (n_parts > 1) RT_CUDA(ctx, ctx->ev_scored.create(cudaEventDisableTiming));
    for (int i = 0; i < n_parts; ++i) {
        const int64_t a = cut[(size_t)i], b = cut[(size_t)i + 1], m = b - a, k = a - orf_lo;
        if (m == 0) continue;
        rt_score_out di{};
        di.score = d.score + k; di.count = d.count + k; di.valid = d.valid + k; di.length = d.length + k; di.status = d.status + k;
        di.min_codon = d.min_codon ? d.min_codon + k : nullptr;
        di.frame_K = d.frame_K ? d.frame_K + 3 * k : nullptr;
        di.frame_s = d.frame_s ? d.frame_s + 3 * k : nullptr;
        int rc = rt_score(ctx, d_cov, a, b, params, &di, nullptr);
        if (rc != RT_OK) return rc;
        if (copy) {
            RT_CUDA(ctx, cudaEventRecord(ctx->ev_scored, nullptr));
            RT_CUDA(ctx, cudaStreamWaitEvent(copy, ctx->ev_scored, 0));
        }
        auto back = [&](void* h, const void* dv, size_t elem) -> cudaError_t {
            return h ? cudaMemcpyAsync(static_cast<char*>(h) + elem * (size_t)k, dv, elem * (size_t)m, cudaMemcpyDeviceToHost, copy) : cudaSuccess;
        };
        RT_CUDA(ctx, back(h_out->score, di.score, 8));
        RT_CUDA(ctx, back(h_out->count, di.count, 8));
        RT_CUDA(ctx, back(h_out->valid, di.valid, 4));
        RT_CUDA(ctx, back(h_out->length, di.length, 4));
        RT_CUDA(ctx, back(h_out->min_codon, di.min_codon, 4));
        RT_CUDA(ctx, back(h_out->status, di.status, 1));
        if (di.frame_K) RT_CUDA(ctx, back(h_out->frame_K, di.frame_K, 12));
        if (di.frame_s) RT_CUDA(ctx, back(h_out->frame_s, di.frame_s, 24));
    }
    RT_CUDA(ctx, cudaStreamSynchronize(nullptr));
    if (copy) RT_CUDA(ctx, cudaStreamSynchronize(copy));
    return RT_OK;
}

// ------------------------------------------------------------------------------------ phasescore(values)
int rt_phasescore_values(rt_ctx* ctx, const double* h_values, int64_t n, double* h_score, int32_t* h_valid) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_phasescore_values: ctx is NULL");
    if (n < 0 || (n > 0 && !h_values) || !h_score || !h_valid)
        return fail(ctx, RT_EINVAL, "rt_phasescore_values: NULL argument");
    DeviceGuard guard(ctx->device);
    const size_t bytes = sizeof(double) * (size_t)std::max<int64_t>(n, 1) + 64;
    RT_CUDA(ctx, ctx->score_buf.reserve(bytes));
    double* d_vals = reinterpret_cast<double*>(ctx->score_buf.p);
    double* d_score = d_vals + std::max<int64_t>(n, 1);
    int* d_valid = reinterpret_cast<int*>(d_score + 1);
    if (n) RT_CUDA(ctx, cudaMemcpyAsync(d_vals, h_values, sizeof(double) * n, cudaMemcpyHostToDevice, nullptr));
    rt::phasescore_values_kernel<<<1, 32>>>(d_vals, n, d_score, d_valid);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpy(h_score, d_score, sizeof(double), cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(h_valid, d_valid, sizeof(int), cudaMemcpyDeviceToHost));
    return RT_OK;
}

// ------------------------------------------------------------------------------------ K4
int rt_gather_profiles(rt_ctx* ctx, const int32_t* d_cov, int64_t n_sel, const int64_t* d_orf_ids,
                       const int64_t* d_out_ptr, int32_t* d_out, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_gather_profiles: ctx is NULL");
    if (n_sel < 0 || !d_cov || (n_sel > 0 && (!d_orf_ids || !d_out_ptr || !d_out)))
        return fail(ctx, RT_EINVAL, "rt_gather_profiles: NULL argument");
    if (ctx->ix.n_orf == 0 && n_sel > 0) return fail(ctx, RT_ESTATE, "rt_gather_profiles: no index");
    if (n_sel == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    rt::GatherArgs a;
    a.cov = d_cov;
    a.orf_desc = ctx->ix.orf_desc.p;
    a.exon_entries = ctx->ix.layout == RT_LAYOUT_COMPACT ? ctx->ix.exon_entries_c.p : ctx->ix.exon_entries.p;
    a.orf_ids = d_orf_ids;
    a.out_ptr = d_out_ptr;
    a.out = d_out;
    a.n_sel = n_sel;
    const int64_t want = (n_sel + 7) / 8;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)ctx->n_sm * 8));
    rt::gather_profiles_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

// ------------------------------------------------------------------------------------ dense -> compact
int rt_compact_from_dense(rt_ctx* ctx, const int32_t* d_dense, int32_t* d_compact, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_compact_from_dense: ctx is NULL");
    if (!d_dense || !d_compact) return fail(ctx, RT_EINVAL, "rt_compact_from_dense: NULL argument");
    if (ctx->ix.n_orf == 0 || !ctx->ix.atoms_c.p) return fail(ctx, RT_ESTATE, "rt_compact_from_dense: call rt_set_index first");
    if (ctx->ix.n_atoms == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((ctx->ix.n_atoms + 7) / 8, (int64_t)ctx->n_sm * 16));
    rt::compact_from_dense_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ctx->ix.atoms.p, ctx->ix.atoms_c.p, ctx->ix.n_atoms, d_dense, d_compact);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

// ------------------------------------------------------------------------------------ covered positions (WIG)
int64_t rt_wig_tiles(int64_t n_slots) { return n_slots <= 0 ? 0 : (n_slots + rt::kWigTile - 1) / rt::kWigTile; }

int rt_wig_count(rt_ctx* ctx, const int32_t* d_cov, int64_t n_slots, uint32_t* d_tile_counts, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_wig_count: ctx is NULL");
    if (n_slots < 0 || (n_slots > 0 && (!d_cov || !d_tile_counts))) return fail(ctx, RT_EINVAL, "rt_wig_count: NULL argument");
    if (n_slots == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    rt::wig_count_kernel<<<(unsigned)rt_wig_tiles(n_slots), 256, 0, (cudaStream_t)stream>>>(d_cov, n_slots, d_tile_counts);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

int rt_wig_fill(rt_ctx* ctx, const int32_t* d_cov, int64_t n_slots, const int64_t* d_tile_offsets, int64_t* d_out_slot,
                int32_t* d_out_count, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_wig_fill: ctx is NULL");
    if (n_slots < 0 || (n_slots > 0 && (!d_cov || !d_tile_offsets || !d_out_slot || !d_out_count)))
        return fail(ctx, RT_EINVAL, "rt_wig_fill: NULL argument");
    if (n_slots == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    rt::wig_fill_kernel<<<(unsigned)rt_wig_tiles(n_slots), 256, 0, (cudaStream_t)stream>>>(
        d_cov, n_slots, reinterpret_cast<const long long*>(d_tile_offsets), reinterpret_cast<long long*>(d_out_slot), d_out_count);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

// ------------------------------------------------------------------------------------ interval sums
int rt_interval_sums(rt_ctx* ctx, const int32_t* d_cov, int64_t n_iv, const int64_t* d_iv_off, const int32_t* d_iv_len,
                     const int32_t* d_iv_group, int64_t* d_sums, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_interval_sums: ctx is NULL");
    if (n_iv < 0 || !d_cov || !d_sums || (n_iv > 0 && (!d_iv_off || !d_iv_len || !d_iv_group)))
        return fail(ctx, RT_EINVAL, "rt_interval_sums: NULL argument");
    if (ctx->ix.layout != RT_LAYOUT_DENSE)
        return fail(ctx, RT_ESTATE, "rt_interval_sums: interval offsets address the dense planes; switch the layout back first");
    if (n_iv == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n_iv + 7) / 8, (int64_t)ctx->n_sm * 8));
    rt::interval_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_cov, n_iv, reinterpret_cast<const long long*>(d_iv_off),
                                                                   d_iv_len, d_iv_group,
                                                                   reinterpret_cast<unsigned long long*>(d_sums));
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

// ------------------------------------------------------------------------------------ bootstrap medians
int rt_bootstrap_medians(rt_ctx* ctx, const double* h_values, int64_t n, const int64_t* h_idx, int64_t n_sel, int64_t reps,
                         double* h_out) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bootstrap_medians: ctx is NULL");
    if (n <= 0 || n_sel <= 0 || reps <= 0 || !h_values || !h_idx || !h_out)
        return fail(ctx, RT_EINVAL, "rt_bootstrap_medians: empty or NULL argument");
    if (reps > 0x7fffffff) return fail(ctx, RT_EINVAL, "rt_bootstrap_medians: too many replicates");
    for (int64_t i = 0; i < n_sel * reps; ++i)
        if (h_idx[i] < 0 || h_idx[i] >= n) return fail(ctx, RT_EINVAL, "rt_bootstrap_medians: index %lld outside [0,%lld)", (long long)h_idx[i], (long long)n);
    DeviceGuard guard(ctx->device);
    const size_t key_bytes = sizeof(unsigned long long) * (size_t)n_sel;
    const bool in_smem = key_bytes <= 160 * 1024;
    DevArr<double> vals, outb;
    DevArr<long long> idx;
    DevArr<unsigned long long> scratch;
    RT_CUDA(ctx, vals.upload(h_values, (size_t)n));
    RT_CUDA(ctx, idx.upload(h_idx, (size_t)(n_sel * reps)));
    RT_CUDA(ctx, outb.reserve((size_t)reps));
    if (!in_smem) RT_CUDA(ctx, scratch.reserve((size_t)n_sel * (size_t)reps));
    if (in_smem) RT_CUDA(ctx, cudaFuncSetAttribute(rt::bootstrap_median_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)key_bytes));
    rt::bootstrap_median_kernel<<<(unsigned)reps, 256, in_smem ? key_bytes : 0>>>(vals.p, idx.p, n_sel, reps, scratch.p,
                                                                                 in_smem ? 1 : 0, outb.p);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpy(h_out, outb.p, sizeof(double) * (size_t)reps, cudaMemcpyDeviceToHost));
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------ prepare-orfs
int rt_orf_search(rt_ctx* ctx, const rt_orf_query* q, int64_t* n_rows, int64_t* n_iv, float* stage_ms) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_orf_search: ctx is NULL");
    if (!q || !n_rows || !n_iv || q->n_tx < 0 || q->n_codes < 0 || q->min_orf_length < 0 ||
        (q->n_tx && (!q->exon_ptr || !q->exon_start || !q->exon_end || !q->tx_base || !q->tx_strand || !q->tx_cds)) ||
        (q->n_codes && !q->codes))
        return fail(ctx, RT_EINVAL, "rt_orf_search: NULL or negative argument");
    if (q->n_tx > 0x7fffffff) return fail(ctx, RT_EINVAL, "rt_orf_search: more than 2^31 - 1 transcripts");
    const int64_t n_tx = q->n_tx;
    const int64_t n_ex = n_tx ? q->exon_ptr[n_tx] : 0;
    // host side of the transcript table: per exon its source in codes, its place in the spliced buffer, its offset
    // within the transcript's ascending concatenation
    std::vector<int64_t> ex_src((size_t)n_ex), ex_dst((size_t)n_ex), tx_seq((size_t)n_tx + 1, 0);
    std::vector<int32_t> ex_len((size_t)n_ex), ex_before((size_t)n_ex);
    std::vector<uint8_t> ex_rev((size_t)n_ex);
    for (int64_t t = 0; t < n_tx; ++t) {
        const int64_t a = q->exon_ptr[t], b = q->exon_ptr[t + 1];
        if (a < 0 || b <= a || b > n_ex) return fail(ctx, RT_EINVAL, "rt_orf_search: transcript %lld has no exon", (long long)t);
        if (q->tx_strand[t] > 1) return fail(ctx, RT_EINVAL, "rt_orf_search: transcript %lld has no strand", (long long)t);
        int64_t n = 0;
        for (int64_t e = a; e < b; ++e) {
            if (q->exon_start[e] < 1 || q->exon_end[e] < q->exon_start[e] || (e > a && q->exon_start[e] <= q->exon_end[e - 1]) ||
                q->tx_base[t] < 0 || q->tx_base[t] + q->exon_end[e] > q->n_codes)
                return fail(ctx, RT_EINVAL, "rt_orf_search: exon %lld of transcript %lld is unsorted or outside the codes",
                            (long long)(e - a), (long long)t);
            ex_before[(size_t)e] = (int32_t)n;
            ex_len[(size_t)e] = q->exon_end[e] - q->exon_start[e] + 1;
            ex_src[(size_t)e] = q->tx_base[t] + q->exon_start[e] - 1;
            ex_rev[(size_t)e] = q->tx_strand[t];
            n += ex_len[(size_t)e];
            if (n > 0x7fffffff) return fail(ctx, RT_EINVAL, "rt_orf_search: transcript %lld is longer than 2^31 - 1", (long long)t);
        }
        for (int64_t e = a; e < b; ++e)
            ex_dst[(size_t)e] = tx_seq[(size_t)t] + (q->tx_strand[t] ? n - ex_before[(size_t)e] - ex_len[(size_t)e] : ex_before[(size_t)e]);
        tx_seq[(size_t)t + 1] = tx_seq[(size_t)t] + n;
    }
    const int64_t n_seq = tx_seq[(size_t)n_tx];
    DeviceGuard guard(ctx->device);
    rt_ctx::OrfBufs& B = ctx->orf;
    const size_t nt = (size_t)n_tx, ne = (size_t)n_ex;
    RT_CUDA(ctx, B.codes.reserve((size_t)q->n_codes));
    RT_CUDA(ctx, B.ex_src.reserve(ne));
    RT_CUDA(ctx, B.ex_dst.reserve(ne));
    RT_CUDA(ctx, B.ex_len.reserve(ne));
    RT_CUDA(ctx, B.ex_rev.reserve(ne));
    RT_CUDA(ctx, B.tx_seq.reserve(nt + 1));
    RT_CUDA(ctx, B.tx_cds.reserve(nt));
    RT_CUDA(ctx, B.tx_exon.reserve(nt + 1));
    RT_CUDA(ctx, B.tx_rev.reserve(nt));
    RT_CUDA(ctx, B.ex_start.reserve(ne));
    RT_CUDA(ctx, B.ex_end.reserve(ne));
    RT_CUDA(ctx, B.ex_before.reserve(ne));
    RT_CUDA(ctx, B.seq.reserve((size_t)n_seq + 4));
    RT_CUDA(ctx, B.tx_rows.reserve(nt));
    RT_CUDA(ctx, B.row_off.reserve(nt));
    RT_CUDA(ctx, B.claim.reserve(1));
    cudaStream_t st = 0;
    Event ev[RT_ORF_STAGES + 1];
    for (auto& e : ev) RT_CUDA(ctx, e.create());
    RT_CUDA(ctx, cudaEventRecord(ev[0], st));
    // 1. upload: contig codes, the transcript and exon tables
    RT_CUDA(ctx, B.codes.upload(q->codes, (size_t)q->n_codes, st));
    RT_CUDA(ctx, B.ex_src.upload(ex_src.data(), ne, st));
    RT_CUDA(ctx, B.ex_dst.upload(ex_dst.data(), ne, st));
    RT_CUDA(ctx, B.ex_len.upload(ex_len.data(), ne, st));
    RT_CUDA(ctx, B.ex_rev.upload(ex_rev.data(), ne, st));
    RT_CUDA(ctx, B.tx_seq.upload(tx_seq.data(), nt + 1, st));
    RT_CUDA(ctx, B.tx_cds.upload(reinterpret_cast<const int2*>(q->tx_cds), nt, st));
    RT_CUDA(ctx, B.tx_exon.upload(q->exon_ptr, nt + 1, st));
    RT_CUDA(ctx, B.tx_rev.upload(q->tx_strand, nt, st));
    RT_CUDA(ctx, B.ex_start.upload(q->exon_start, ne, st));
    RT_CUDA(ctx, B.ex_end.upload(q->exon_end, ne, st));
    RT_CUDA(ctx, B.ex_before.upload(ex_before.data(), ne, st));
    RT_CUDA(ctx, cudaEventRecord(ev[1], st));
    const unsigned big = (unsigned)std::max(1, ctx->n_sm * 8);
    // 2. spliced, oriented sequences
    if (n_ex) {
        rt::orf_splice_kernel<<<(unsigned)std::min<int64_t>((n_ex + 7) / 8, big), 256, 0, st>>>(
            B.codes.p, B.ex_src.p, B.ex_dst.p, B.ex_len.p, B.ex_rev.p, n_ex, B.seq.p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(ev[2], st));
    // 3. rows per transcript
    rt::OrfArgs A{B.tx_seq.p, B.tx_cds.p, B.seq.p, q->start_mask, q->stop_mask, (int)n_tx, q->min_orf_length, q->longest ? 1 : 0,
                  B.claim.p};
    const unsigned walk_grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n_tx + 7) / 8, big));
    if (n_tx) {
        RT_CUDA(ctx, cudaMemsetAsync(B.claim.p, 0, sizeof(unsigned), st));
        rt::orf_walk_kernel<false><<<walk_grid, 256, 0, st>>>(A, B.tx_rows.p, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(ev[3], st));
    // 4. exclusive scan of the row counts (host: one int64 per transcript)
    std::vector<int64_t> cnt((size_t)n_tx), off((size_t)n_tx + 1, 0);
    if (n_tx) RT_CUDA(ctx, cudaMemcpyAsync(cnt.data(), B.tx_rows.p, sizeof(long long) * nt, cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    for (int64_t t = 0; t < n_tx; ++t) off[(size_t)t + 1] = off[(size_t)t] + cnt[(size_t)t];
    const int64_t rows = off[(size_t)n_tx];
    const size_t nr = (size_t)rows;
    RT_CUDA(ctx, B.row_tx.reserve(nr));
    RT_CUDA(ctx, B.row_start.reserve(nr));
    RT_CUDA(ctx, B.row_stop.reserve(nr));
    RT_CUDA(ctx, B.row_type.reserve(nr));
    RT_CUDA(ctx, B.row_codon.reserve(nr));
    RT_CUDA(ctx, B.iv_count.reserve(nr));
    RT_CUDA(ctx, B.iv_off.reserve(nr));
    RT_CUDA(ctx, B.row_off.upload(off.data(), nt, st));
    RT_CUDA(ctx, cudaEventRecord(ev[4], st));
    // 5. the rows
    if (rows) {
        RT_CUDA(ctx, cudaMemsetAsync(B.claim.p, 0, sizeof(unsigned), st));
        rt::orf_walk_kernel<true><<<walk_grid, 256, 0, st>>>(A, B.tx_rows.p, B.row_off.p, B.row_tx.p, B.row_start.p, B.row_stop.p,
                                                               B.row_type.p, B.row_codon.p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(ev[5], st));
    // 6. intervals per row, their exclusive scan (host)
    const unsigned row_grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((rows + 255) / 256, (int64_t)big * 4));
    auto intervals = [&](bool count) {
        if (count)
            rt::orf_interval_kernel<true><<<row_grid, 256, 0, st>>>(rows, B.row_tx.p, B.row_start.p, B.row_stop.p, B.tx_exon.p,
                                                                      B.tx_seq.p, B.tx_rev.p, B.ex_start.p, B.ex_end.p, B.ex_before.p,
                                                                      B.iv_count.p, nullptr, nullptr, nullptr);
        else
            rt::orf_interval_kernel<false><<<row_grid, 256, 0, st>>>(rows, B.row_tx.p, B.row_start.p, B.row_stop.p, B.tx_exon.p,
                                                                       B.tx_seq.p, B.tx_rev.p, B.ex_start.p, B.ex_end.p, B.ex_before.p,
                                                                       nullptr, B.iv_off.p, B.iv_start.p, B.iv_end.p);
        ctx->launches++;
        return cudaGetLastError();
    };
    std::vector<int64_t>& ivp = ctx->orf_iv_ptr;
    ivp.assign((size_t)rows + 1, 0);
    if (rows) {
        RT_CUDA(ctx, intervals(true));
        std::vector<int64_t> ivc((size_t)rows);
        RT_CUDA(ctx, cudaMemcpyAsync(ivc.data(), B.iv_count.p, sizeof(long long) * nr, cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));
        for (int64_t r = 0; r < rows; ++r) ivp[(size_t)r + 1] = ivp[(size_t)r] + ivc[(size_t)r];
    }
    const int64_t ivs = ivp.back();
    RT_CUDA(ctx, B.iv_start.reserve((size_t)ivs));
    RT_CUDA(ctx, B.iv_end.reserve((size_t)ivs));
    RT_CUDA(ctx, B.iv_off.upload(ivp.data(), nr, st));
    RT_CUDA(ctx, cudaEventRecord(ev[6], st));
    // 7. the intervals
    if (rows) RT_CUDA(ctx, intervals(false));
    RT_CUDA(ctx, cudaEventRecord(ev[7], st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    if (stage_ms) RT_CUDA(ctx, stage_times(ev, RT_ORF_STAGES, stage_ms));
    ctx->orf_rows = rows;
    *n_rows = rows;
    *n_iv = ivs;
    return RT_OK;
}

int rt_orf_fetch(rt_ctx* ctx, int32_t* row_tx, int32_t* row_start, int32_t* row_stop, uint8_t* row_type, uint8_t* row_codon,
                 int64_t* iv_ptr, int32_t* iv_start, int32_t* iv_end) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_orf_fetch: ctx is NULL");
    const int64_t rows = ctx->orf_rows;
    if ((int64_t)ctx->orf_iv_ptr.size() != rows + 1) return fail(ctx, RT_ESTATE, "rt_orf_fetch: call rt_orf_search first");
    const int64_t ivs = ctx->orf_iv_ptr.back();
    DeviceGuard guard(ctx->device);
    const rt_ctx::OrfBufs& B = ctx->orf;
    cudaStream_t st = 0;
    auto down = [&](void* dst, const auto& src, int64_t m) {
        return dst && m ? cudaMemcpyAsync(dst, src.p, sizeof(*src.p) * (size_t)m, cudaMemcpyDeviceToHost, st) : cudaSuccess;
    };
    RT_CUDA(ctx, down(row_tx, B.row_tx, rows));
    RT_CUDA(ctx, down(row_start, B.row_start, rows));
    RT_CUDA(ctx, down(row_stop, B.row_stop, rows));
    RT_CUDA(ctx, down(row_type, B.row_type, rows));
    RT_CUDA(ctx, down(row_codon, B.row_codon, rows));
    RT_CUDA(ctx, down(iv_start, B.iv_start, ivs));
    RT_CUDA(ctx, down(iv_end, B.iv_end, ivs));
    if (iv_ptr) memcpy(iv_ptr, ctx->orf_iv_ptr.data(), 8 * (size_t)(rows + 1));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    return RT_OK;
}

// ---------------------------------------------------------------------------------------------------- orfs-seq
namespace {
constexpr int64_t kSeqChunkDefault = int64_t(64) << 20;

// Streams, events, page-locked buffers and the writer of one rt_orf_seq_write call; the destructor joins the writer and
// waits for both streams before the members are freed, so every early return leaves nothing behind.
struct SeqPipeline {
    Stream ks, cs;                             // kernels + uploads, copy-back
    Event ev[10];                              // upload begin / end, then per buffer b: kernel begin/end, copy begin/end
    PinnedArr<char> pinned[2];
    WriteBehind writer;
    explicit SeqPipeline(FILE* fh) : writer(fh) {}
    ~SeqPipeline() {
        writer.finish();                       // before the page-locked buffers it writes from are freed
        if (ks) cudaStreamSynchronize(ks);
        if (cs) cudaStreamSynchronize(cs);
    }
};

int seq_emit(rt_ctx* ctx, const rt_seq_query* q, const std::vector<int64_t>& line_off, const std::vector<int64_t>& cut,
             int64_t buf_bytes, FILE* fh, float* stage_ms) {
    const int64_t n = q->n_orf, n_ex = n ? q->exon_ptr[n] : 0, n_ids = n ? q->id_off[n] : 0;
    const int64_t n_chunks = (int64_t)cut.size() - 1;
    rt_ctx::SeqBufs& B = ctx->seq;
    const size_t nr = (size_t)n, ne = (size_t)n_ex;
    RT_CUDA(ctx, B.codes.reserve((size_t)q->n_codes));
    RT_CUDA(ctx, B.exon_ptr.reserve(nr + 1));
    RT_CUDA(ctx, B.ex_start.reserve(ne));
    RT_CUDA(ctx, B.ex_end.reserve(ne));
    RT_CUDA(ctx, B.contig.reserve(nr));
    RT_CUDA(ctx, B.strand.reserve(nr));
    RT_CUDA(ctx, B.base.reserve((size_t)q->n_contig));
    RT_CUDA(ctx, B.id_off.reserve(nr + 1));
    RT_CUDA(ctx, B.ids.reserve((size_t)n_ids));
    RT_CUDA(ctx, B.line_off.reserve(nr + 1));
    RT_CUDA(ctx, B.claim.reserve(1));
    SeqPipeline P(fh);
    RT_CUDA(ctx, P.ks.create());
    RT_CUDA(ctx, P.cs.create());
    for (auto& e : P.ev) RT_CUDA(ctx, e.create());
    const Event *k_begin = P.ev + 2, *k_end = P.ev + 4, *c_begin = P.ev + 6, *c_end = P.ev + 8;
    // 1. upload: the contig codes and the tables, once
    RT_CUDA(ctx, cudaEventRecord(P.ev[0], P.ks));
    RT_CUDA(ctx, B.codes.upload(q->codes, (size_t)q->n_codes, P.ks));
    RT_CUDA(ctx, B.exon_ptr.upload(q->exon_ptr, nr + 1, P.ks));
    RT_CUDA(ctx, B.ex_start.upload(q->exon_start, ne, P.ks));
    RT_CUDA(ctx, B.ex_end.upload(q->exon_end, ne, P.ks));
    RT_CUDA(ctx, B.contig.upload(q->orf_contig, nr, P.ks));
    RT_CUDA(ctx, B.strand.upload(q->orf_strand, nr, P.ks));
    RT_CUDA(ctx, B.base.upload(q->contig_base, (size_t)q->n_contig, P.ks));
    RT_CUDA(ctx, B.id_off.upload(q->id_off, nr + 1, P.ks));
    RT_CUDA(ctx, B.ids.upload(q->ids, (size_t)n_ids, P.ks));
    RT_CUDA(ctx, B.line_off.upload(line_off.data(), nr + 1, P.ks));
    RT_CUDA(ctx, cudaEventRecord(P.ev[1], P.ks));
    if (stage_ms) stage_ms[1] = stage_ms[2] = 0.f;
    if (n_chunks == 0) {
        RT_CUDA(ctx, cudaStreamSynchronize(P.ks));
        if (stage_ms) RT_CUDA(ctx, cudaEventElapsedTime(&stage_ms[0], P.ev[0], P.ev[1]));
        return RT_OK;
    }
    // 2. the chunks: kernel k+1 runs while chunk k is copied back and chunk k-1 is written
    for (int b = 0; b < 2 && b < n_chunks; ++b) {
        RT_CUDA(ctx, B.out[b].reserve((size_t)buf_bytes));
        RT_CUDA(ctx, P.pinned[b].alloc((size_t)buf_bytes));
    }
    const rt::SeqArgs A{B.codes.p, B.exon_ptr.p, B.ex_start.p, B.ex_end.p, B.contig.p, B.strand.p, B.base.p, B.id_off.p, B.ids.p,
                        B.line_off.p, B.claim.p};
    const int64_t big = std::max(1, ctx->n_sm * 8);
    auto bytes_of = [&](int64_t k) { return (size_t)(line_off[(size_t)cut[(size_t)k + 1]] - line_off[(size_t)cut[(size_t)k]]); };
    // chunk k is on the host: add its times, hand it to the writer
    auto collect = [&](int64_t k) -> int {
        const int b = (int)(k & 1);
        RT_CUDA(ctx, cudaEventSynchronize(c_end[b]));
        if (stage_ms) {
            float kms = 0.f, cms = 0.f;
            RT_CUDA(ctx, cudaEventElapsedTime(&kms, k_begin[b], k_end[b]));
            RT_CUDA(ctx, cudaEventElapsedTime(&cms, c_begin[b], c_end[b]));
            stage_ms[1] += kms;
            stage_ms[2] += cms;
        }
        if (!P.writer.put_view(P.pinned[b].p, bytes_of(k))) return fail(ctx, RT_EINVAL, "rt_orf_seq_write: write error");
        return RT_OK;
    };
    for (int64_t k = 0; k < n_chunks; ++k) {
        const int b = (int)(k & 1);
        const int64_t r0 = cut[(size_t)k], rows = cut[(size_t)k + 1] - r0;
        // device buffer b is free: chunk k-2's copy finished before collect(k-2) returned
        RT_CUDA(ctx, cudaMemsetAsync(B.claim.p, 0, sizeof(unsigned), P.ks));
        RT_CUDA(ctx, cudaEventRecord(k_begin[b], P.ks));
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((rows + rt::kSeqWarps - 1) / rt::kSeqWarps, big));
        if (q->protein)
            rt::orf_seq_kernel<true><<<grid, rt::kSeqWarps * 32, 0, P.ks>>>(A, r0, rows, B.out[b].p);
        else
            rt::orf_seq_kernel<false><<<grid, rt::kSeqWarps * 32, 0, P.ks>>>(A, r0, rows, B.out[b].p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
        RT_CUDA(ctx, cudaEventRecord(k_end[b], P.ks));
        if (k >= 1) {
            const int rc = collect(k - 1);
            if (rc != RT_OK) return rc;
        }
        // page-locked buffer b is free once chunk k-2 has been written
        if (k >= 2 && !P.writer.wait_written(k - 1)) return fail(ctx, RT_EINVAL, "rt_orf_seq_write: write error");
        RT_CUDA(ctx, cudaStreamWaitEvent(P.cs, k_end[b], 0));
        RT_CUDA(ctx, cudaEventRecord(c_begin[b], P.cs));
        RT_CUDA(ctx, cudaMemcpyAsync(P.pinned[b].p, B.out[b].p, bytes_of(k), cudaMemcpyDeviceToHost, P.cs));
        RT_CUDA(ctx, cudaEventRecord(c_end[b], P.cs));
    }
    const int rc = collect(n_chunks - 1);
    if (rc != RT_OK) return rc;
    if (!P.writer.wait_written(n_chunks)) return fail(ctx, RT_EINVAL, "rt_orf_seq_write: write error");
    if (stage_ms) RT_CUDA(ctx, cudaEventElapsedTime(&stage_ms[0], P.ev[0], P.ev[1]));
    return RT_OK;
}
}  // namespace

int rt_orf_seq_write(rt_ctx* ctx, const rt_seq_query* q, const char* path, float* stage_ms) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_orf_seq_write: ctx is NULL");
    if (!q || !path || q->n_orf < 0 || q->n_contig < 0 || q->n_codes < 0 || q->chunk_bytes < 0 ||
        (q->n_orf && (!q->exon_ptr || !q->orf_contig || !q->orf_strand || !q->id_off)) ||
        (q->n_contig && (!q->contig_base || !q->contig_len)) || (q->n_codes && !q->codes))
        return fail(ctx, RT_EINVAL, "rt_orf_seq_write: NULL or negative argument");
    const int64_t n = q->n_orf;
    const int64_t n_ex = n ? q->exon_ptr[n] : 0, n_ids = n ? q->id_off[n] : 0;
    if ((n_ex && (!q->exon_start || !q->exon_end)) || (n_ids && !q->ids) || (n && (q->exon_ptr[0] != 0 || q->id_off[0] != 0)))
        return fail(ctx, RT_EINVAL, "rt_orf_seq_write: NULL or negative argument");
    for (int c = 0; c < q->n_contig; ++c)
        if (q->contig_base[c] < 0 || q->contig_len[c] < 0 || q->contig_base[c] + q->contig_len[c] > q->n_codes)
            return fail(ctx, RT_EINVAL, "rt_orf_seq_write: contig %d lies outside the codes", c);
    // 1. host pass: every row checked, the length and offset of every line
    std::vector<int64_t> line_off((size_t)n + 1, 0);
    int64_t longest = 0;
    for (int64_t r = 0; r < n; ++r) {
        const int64_t a = q->exon_ptr[r], b = q->exon_ptr[r + 1], i0 = q->id_off[r], i1 = q->id_off[r + 1];
        if (b < a || b > n_ex || i1 < i0 || i1 > n_ids)
            return fail(ctx, RT_EINVAL, "rt_orf_seq_write: exon_ptr or id_off is not monotone at row %lld", (long long)r);
        const int id_len = (int)std::min<int64_t>(i1 - i0, 200);
        const int c = q->orf_contig[r];
        if (c < 0 || c >= q->n_contig)
            return fail(ctx, RT_EINVAL, "rt_orf_seq_write: ORF %.*s: contig %d is not in the contig table", id_len, q->ids + i0, c);
        int64_t L = 0;
        for (int64_t e = a; e < b; ++e) {
            const int32_t s = q->exon_start[e], t = q->exon_end[e];
            if (t < s)
                return fail(ctx, RT_EINVAL, "rt_orf_seq_write: ORF %.*s: interval %d-%d ends before it starts", id_len, q->ids + i0, s, t);
            if (s < 1 || t > q->contig_len[c])
                return fail(ctx, RT_EINVAL, "rt_orf_seq_write: ORF %.*s: interval %d-%d is outside its contig of %lld nt", id_len,
                            q->ids + i0, s, t, (long long)q->contig_len[c]);
            L += (int64_t)t - s + 1;
        }
        const int64_t line = (i1 - i0) + 1 + (q->protein ? L / 3 : L) + 1;
        line_off[(size_t)r + 1] = line_off[(size_t)r] + line;
        longest = std::max(longest, line);
    }
    // 2. chunks of whole lines, none smaller than the longest line
    const int64_t cap = std::max(q->chunk_bytes ? q->chunk_bytes : kSeqChunkDefault, longest);
    std::vector<int64_t> cut{0};
    int64_t buf_bytes = 0;
    for (int64_t r = 0; r < n;) {
        const int64_t limit = line_off[(size_t)r] + cap;
        int64_t r1 = std::upper_bound(line_off.begin() + r + 1, line_off.end(), limit) - line_off.begin() - 1;
        r1 = std::min<int64_t>(r1, r + 0x7fffffff);
        buf_bytes = std::max(buf_bytes, line_off[(size_t)r1] - line_off[(size_t)r]);
        cut.push_back(r1);
        r = r1;
    }
    // 3. the header, then the lines
    DeviceGuard guard(ctx->device);
    FILE* fh = fopen(path, "wb");
    if (!fh) return fail(ctx, RT_EINVAL, "rt_orf_seq_write: cannot open %s", path);
    static const char kHeader[] = "ORF_ID\tsequence\n";
    int rc = fwrite(kHeader, 1, sizeof kHeader - 1, fh) == sizeof kHeader - 1
                 ? RT_OK : fail(ctx, RT_EINVAL, "rt_orf_seq_write: cannot write %s", path);
    if (rc == RT_OK) rc = seq_emit(ctx, q, line_off, cut, buf_bytes, fh, stage_ms);
    if (fclose(fh) != 0 && rc == RT_OK) rc = fail(ctx, RT_EINVAL, "rt_orf_seq_write: cannot write %s", path);
    if (rc != RT_OK) remove(path);
    return rc;
}

// ---------------------------------------------------------------------- selected detected-ORF rows, count-orfs-codon
}  // extern "C"

namespace {
// The selected rows of a detected-ORFs TSV (rt_codon_load_tsv), the half rt_codon_counts and rt_count_orfs share.
// scan<slot_nt>() checks the query fields both take and scans per row its profile text, its length in nt and its slots
// of slot_nt nt; gather() copies the profile text together on all cores; reserve() and upload() put it on the device with
// the rows' index intervals for the emit kernels (rt::RowArgs); read_refusal() reads back the first refused row.
struct SelectedRows {
    rt_count_query q{};
    int64_t n = 0, n_ex = 0;
    HostArr<int64_t> prof_base, len_base, slot_base;         // n + 1 each
    HostArr<char> prof;
    DevArr<char> d_prof;
    DevArr<long long> d_prof_base, d_len_base, d_row, d_ex_ptr;
    DevArr<int> d_gene, d_ex_start, d_ex_end;
    DevArr<uint8_t> d_strand, d_flag;
    DevArr<unsigned> d_claim;

    template <int slot_nt>
    int scan(rt_ctx* ctx, const char* who, const rt_count_query& query) {
        q = query;
        if (q.n_sel < 0 || q.n_orf < 0 || q.n_gene < 0 ||
            (q.n_sel && (!q.row || !q.gene || !q.prof_off || !q.prof_len || !q.tsv || !q.exon_ptr || !q.orf_strand)))
            return fail(ctx, RT_EINVAL, "%s: NULL or negative argument", who);
        n = q.n_sel;
        n_ex = n ? q.exon_ptr[q.n_orf] : 0;
        if (!prof_base.alloc((size_t)n + 1) || !len_base.alloc((size_t)n + 1) || !slot_base.alloc((size_t)n + 1))
            return fail(ctx, RT_ENOMEM, "%s: out of host memory", who);
        prof_base[0] = len_base[0] = slot_base[0] = 0;
        for (int64_t i = 0; i < n; ++i) {
            const int64_t r = q.row[i];
            if (r < 0 || r >= q.n_orf || q.gene[i] < 0 || q.gene[i] >= q.n_gene)
                return fail(ctx, RT_EINVAL, "%s: selected row %lld lies outside the index or the gene table", who, (long long)i);
            int64_t L = 0;
            for (int64_t e = q.exon_ptr[r]; e < q.exon_ptr[r + 1]; ++e) L += (int64_t)q.exon_end[e] - q.exon_start[e] + 1;
            prof_base[(size_t)i + 1] = prof_base[(size_t)i] + q.prof_len[i];
            len_base[(size_t)i + 1] = len_base[(size_t)i] + L;
            slot_base[(size_t)i + 1] = slot_base[(size_t)i] + L / slot_nt;
        }
        return RT_OK;
    }
    int64_t slots() const { return slot_base[(size_t)n]; }

    // also(i) runs for every row i in the same pass; also_bytes is what it copies in all.
    template <class F>
    int gather(rt_ctx* ctx, const char* who, int64_t also_bytes, F&& also) {
        if (!prof.alloc((size_t)prof_base[(size_t)n])) return fail(ctx, RT_ENOMEM, "%s: out of host memory", who);
        const int64_t block = 1 << 10;
        claim_parallel(host_threads((size_t)((prof_base[(size_t)n] + also_bytes) >> 22) + 1, 32),
                       (size_t)((n + block - 1) / block), [&](size_t bk) {
            for (int64_t i = (int64_t)bk * block; i < std::min(n, (int64_t)(bk + 1) * block); ++i) {
                memcpy(prof.p + prof_base[(size_t)i], q.tsv + q.prof_off[i], (size_t)q.prof_len[i]);
                also(i);
            }
        });
        return RT_OK;
    }

    int reserve(rt_ctx* ctx) {
        const size_t nn = (size_t)n, no = (size_t)q.n_orf, ne = (size_t)n_ex;
        RT_CUDA(ctx, d_prof.reserve(prof.size()));
        RT_CUDA(ctx, d_prof_base.reserve(nn + 1));
        RT_CUDA(ctx, d_len_base.reserve(nn + 1));
        RT_CUDA(ctx, d_row.reserve(nn));
        RT_CUDA(ctx, d_gene.reserve(nn));
        RT_CUDA(ctx, d_ex_ptr.reserve(no + 1));
        RT_CUDA(ctx, d_ex_start.reserve(ne));
        RT_CUDA(ctx, d_ex_end.reserve(ne));
        RT_CUDA(ctx, d_strand.reserve(no));
        RT_CUDA(ctx, d_flag.reserve(nn));
        RT_CUDA(ctx, d_claim.reserve(1));
        return RT_OK;
    }

    int upload(rt_ctx* ctx, cudaStream_t st) {
        const size_t nn = (size_t)n, no = (size_t)q.n_orf, ne = (size_t)n_ex;
        RT_CUDA(ctx, d_prof.upload(prof.p, prof.size(), st));
        RT_CUDA(ctx, d_prof_base.upload(prof_base.data(), nn + 1, st));
        RT_CUDA(ctx, d_len_base.upload(len_base.data(), nn + 1, st));
        RT_CUDA(ctx, d_row.upload(q.row, nn, st));
        RT_CUDA(ctx, d_gene.upload(q.gene, nn, st));
        if (n) {
            RT_CUDA(ctx, d_ex_ptr.upload(q.exon_ptr, no + 1, st));
            RT_CUDA(ctx, d_ex_start.upload(q.exon_start, ne, st));
            RT_CUDA(ctx, d_ex_end.upload(q.exon_end, ne, st));
            RT_CUDA(ctx, d_strand.upload(q.orf_strand, no, st));
        }
        RT_CUDA(ctx, cudaMemsetAsync(d_claim.p, 0, sizeof(unsigned), st));
        return RT_OK;
    }

    rt::RowArgs args() const {
        return {d_prof.p, d_prof_base.p, d_len_base.p, d_row.p, d_ex_ptr.p, d_ex_start.p, d_ex_end.p, d_strand.p, d_gene.p,
                d_flag.p, (long long)n, d_claim.p};
    }
    // blocks of kCodonWarps warps, one warp a row, at most `cap` blocks
    unsigned emit_grid(int64_t cap) const {
        return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + rt::kCodonWarps - 1) / rt::kCodonWarps, cap));
    }

    // out[0] = first, the first refused row, and out[1] = its refusal bits
    int read_refusal(rt_ctx* ctx, cudaStream_t st, unsigned long long first, int64_t* out) {
        uint8_t f = 0;
        RT_CUDA(ctx, cudaMemcpyAsync(&f, d_flag.p + first, 1, cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));
        out[0] = (int64_t)first;
        out[1] = f;
        return RT_OK;
    }
};

// The stream, events and buffers of one rt_codon_counts call; everything is freed on every return.
struct CodonScratch {
    Stream st;
    Event ev[7];
    SelectedRows rows;                 // len_base: where the rows' letters start in `letters`
    HostArr<char> letters;
    DevArr<char> seq, temp;
    DevArr<long long> slot_base;
    DevArr<int> gseq;
    DevArr<unsigned long long> cnt, key, val, key2, val2, counters, gene_tab, pooled_tab;
    ~CodonScratch() { if (st) cudaStreamSynchronize(st); }
};

int bit_length(unsigned long long x) { return x ? 64 - __builtin_clzll(x) : 0; }
}  // namespace

extern "C" {

int rt_codon_counts(rt_ctx* ctx, const rt_codon_query* q, uint64_t* gene_tab, uint64_t* pooled_tab, int64_t* summary,
                    float* stage_ms) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_codon_counts: ctx is NULL");
    if (!q || !pooled_tab || !summary || q->n_gseq < 0 || (q->n_sel && (!q->gseq || !q->seq_off || !q->seq)) ||
        (q->n_gene && !gene_tab))
        return fail(ctx, RT_EINVAL, "rt_codon_counts: NULL or negative argument");
    if (q->n_gene > (1 << 26))
        return fail(ctx, RT_EINVAL, "count-orfs-codon handles at most 2^26 genes; the selection has %d", q->n_gene);
    DeviceGuard guard(ctx->device);
    CodonScratch S;
    SelectedRows& R = S.rows;
    const auto t_host = std::chrono::steady_clock::now();
    // 1. host: per selected row its profile text, length and codons, and its letters
    if (int rc = R.scan<3>(ctx, "rt_codon_counts", {q->n_sel, q->row, q->gene, q->prof_off, q->prof_len, q->tsv, q->n_orf,
                                                    q->exon_ptr, q->exon_start, q->exon_end, q->orf_strand, q->n_gene}))
        return rc;
    const int64_t n = R.n, n_slot = R.slots();
    for (int64_t i = 0; i < n; ++i)
        if (q->gseq[i] < 0 || q->gseq[i] >= q->n_gseq)
            return fail(ctx, RT_EINVAL, "rt_codon_counts: selected row %lld lies outside the gene tables", (long long)i);
    if (n_slot > (int64_t)0xffffffffll)
        return fail(ctx, RT_EINVAL, "count-orfs-codon handles at most 2^32 - 1 codons; the selection has %lld", (long long)n_slot);
    const int64_t* seq_base = R.len_base.data();
    if (!S.letters.alloc((size_t)seq_base[(size_t)n])) return fail(ctx, RT_ENOMEM, "rt_codon_counts: out of host memory");
    if (int rc = R.gather(ctx, "rt_codon_counts", seq_base[(size_t)n], [&](int64_t i) {
            memcpy(S.letters.p + seq_base[(size_t)i], q->seq + q->seq_off[q->row[i]],
                   (size_t)(seq_base[(size_t)i + 1] - seq_base[(size_t)i]));
        }))
        return rc;
    if (stage_ms) {
        for (int k = 0; k < RT_CODON_STAGES; ++k) stage_ms[k] = 0.f;
        stage_ms[0] = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_host).count();
    }
    for (int k = 0; k < 6; ++k) summary[k] = 0;
    summary[4] = -1;
    // 2. uploads
    RT_CUDA(ctx, S.st.create());
    for (auto& e : S.ev) RT_CUDA(ctx, e.create());
    const size_t ns = (size_t)n_slot, nn = (size_t)n;
    if (int rc = R.reserve(ctx)) return rc;
    RT_CUDA(ctx, S.seq.reserve(S.letters.size()));
    RT_CUDA(ctx, S.slot_base.reserve(nn + 1));
    RT_CUDA(ctx, S.gseq.reserve(nn));
    RT_CUDA(ctx, S.cnt.reserve(ns));
    RT_CUDA(ctx, S.key.reserve(ns));
    RT_CUDA(ctx, S.val.reserve(ns));
    RT_CUDA(ctx, S.key2.reserve(ns));
    RT_CUDA(ctx, S.val2.reserve(ns));
    RT_CUDA(ctx, S.counters.reserve(4));
    RT_CUDA(ctx, S.gene_tab.reserve(RT_CODON_CELL * 64 * (size_t)q->n_gene));
    RT_CUDA(ctx, S.pooled_tab.reserve(RT_CODON_CELL * 64));
    RT_CUDA(ctx, cudaEventRecord(S.ev[0], S.st));
    if (int rc = R.upload(ctx, S.st)) return rc;
    RT_CUDA(ctx, S.seq.upload(S.letters.p, S.letters.size(), S.st));
    RT_CUDA(ctx, S.slot_base.upload(R.slot_base.data(), nn + 1, S.st));
    RT_CUDA(ctx, S.gseq.upload(q->gseq, nn, S.st));
    const unsigned long long counters0[4] = {0, 0, ~0ull, 0};
    RT_CUDA(ctx, S.counters.upload(counters0, 4, S.st));
    RT_CUDA(ctx, cudaMemsetAsync(S.cnt.p, 0, sizeof(unsigned long long) * ns, S.st));
    RT_CUDA(ctx, cudaEventRecord(S.ev[1], S.st));
    // 3. codon_emit_kernel
    unsigned long long *cnt = S.cnt.p, *key = S.key.p, *val = S.val.p, *key2 = S.key2.p, *val2 = S.val2.p, *counters = S.counters.p;
    const rt::CodonArgs A{R.args(), S.seq.p, S.slot_base.p, S.gseq.p, cnt, key, val, counters};
    const int64_t big = std::max(1, ctx->n_sm * 8);
    if (n) {
        rt::codon_emit_kernel<<<R.emit_grid(big), rt::kCodonWarps * 32, 0, S.st>>>(A);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(S.ev[2], S.st));
    unsigned long long h_counters[4];
    RT_CUDA(ctx, cudaMemcpyAsync(h_counters, counters, sizeof h_counters, cudaMemcpyDeviceToHost, S.st));
    RT_CUDA(ctx, cudaStreamSynchronize(S.st));
    summary[0] = (int64_t)h_counters[0];
    summary[1] = (int64_t)h_counters[1];
    if (h_counters[2] != ~0ull) {                      // a refused profile: no tables
        if (int rc = R.read_refusal(ctx, S.st, h_counters[2], summary + 4)) return rc;
        if (stage_ms) RT_CUDA(ctx, stage_times(S.ev, 1, stage_ms + 1));
        return RT_OK;
    }
    // 4. dedup: stable sort by place, keep the first slot of every place
    const unsigned items = (unsigned)ns;
    const int place_bits = std::min(64, 32 + bit_length((unsigned long long)q->n_gseq));
    const int gene_bits = 32 + bit_length(64ull * (unsigned long long)q->n_gene);
    size_t t1 = 0, t2 = 0, t3 = 0;
    RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, t1, key, key2, val, val2, items, 0, place_bits, S.st));
    RT_CUDA(ctx, cub::DeviceRadixSort::SortKeys(nullptr, t2, val, val2, items, 0, gene_bits, S.st));
    RT_CUDA(ctx, cub::DeviceRadixSort::SortKeys(nullptr, t3, val, val2, items, 0, 38, S.st));
    RT_CUDA(ctx, S.temp.reserve(std::max({t1, t2, t3})));
    void* temp = S.temp.p;
    if (items) RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(temp, t1, key, key2, val, val2, items, 0, place_bits, S.st));
    // kept values -> cnt (free now), pooled keys -> key (free now)
    const unsigned keep_grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((int64_t)(ns + 255) / 256, big));
    if (items) {
        rt::codon_keep_kernel<<<keep_grid, 256, 0, S.st>>>(key2, val2, (long long)ns, cnt, key, counters + 3);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(S.ev[3], S.st));
    RT_CUDA(ctx, cudaMemcpyAsync(h_counters + 3, counters + 3, 8, cudaMemcpyDeviceToHost, S.st));
    RT_CUDA(ctx, cudaStreamSynchronize(S.st));
    const unsigned kept = (unsigned)h_counters[3];
    summary[3] = (int64_t)kept;
    summary[2] = summary[0] - summary[1] - summary[3];
    // 5. counts in order within every (gene, codon) and every codon
    if (kept) {
        RT_CUDA(ctx, cub::DeviceRadixSort::SortKeys(temp, t2, cnt, val2, kept, 0, gene_bits, S.st));
        RT_CUDA(ctx, cub::DeviceRadixSort::SortKeys(temp, t3, key, key2, kept, 0, 38, S.st));
    }
    RT_CUDA(ctx, cudaEventRecord(S.ev[4], S.st));
    // 6. codon_stats_kernel over the per-gene cells and the pooled cells
    unsigned long long *gtab = S.gene_tab.p, *ptab = S.pooled_tab.p;
    const int64_t gene_cells = 64 * (int64_t)q->n_gene;
    if (gene_cells) {
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((gene_cells + 7) / 8, big * 4));
        rt::codon_stats_kernel<<<grid, 256, 0, S.st>>>(val2, (long long)kept, gene_cells, gtab);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    rt::codon_stats_kernel<<<8, 256, 0, S.st>>>(key2, (long long)kept, 64, ptab);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaEventRecord(S.ev[5], S.st));
    // 7. copy-back
    if (gene_cells) RT_CUDA(ctx, cudaMemcpyAsync(gene_tab, gtab, 8 * RT_CODON_CELL * (size_t)gene_cells, cudaMemcpyDeviceToHost, S.st));
    RT_CUDA(ctx, cudaMemcpyAsync(pooled_tab, ptab, 8 * RT_CODON_CELL * 64, cudaMemcpyDeviceToHost, S.st));
    RT_CUDA(ctx, cudaEventRecord(S.ev[6], S.st));
    RT_CUDA(ctx, cudaStreamSynchronize(S.st));
    if (stage_ms) RT_CUDA(ctx, stage_times(S.ev, RT_CODON_STAGES - 1, stage_ms + 1));
    return RT_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------- count-orfs
namespace {
// The stream, events and buffers of one rt_count_orfs call; everything is freed on every return.
struct CountScratch {
    Stream st;
    Event ev[6];
    SelectedRows rows;                 // len_base: the slots of every row, one a nt
    DevArr<char> temp;
    DevArr<unsigned long long> key, key2, counters, total, length;
    DevArr<unsigned> val, val2;
    ~CountScratch() { if (st) cudaStreamSynchronize(st); }
};
}  // namespace

extern "C" {

int rt_count_orfs(rt_ctx* ctx, const rt_count_query* q, uint64_t* total, uint64_t* length, int64_t* summary,
                  float* stage_ms) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_count_orfs: ctx is NULL");
    if (!q || !summary || (q->n_gene && (!total || !length)))
        return fail(ctx, RT_EINVAL, "rt_count_orfs: NULL or negative argument");
    DeviceGuard guard(ctx->device);
    CountScratch S;
    SelectedRows& R = S.rows;
    const auto t_host = std::chrono::steady_clock::now();
    // 1. host: per selected line its profile text and row length
    if (int rc = R.scan<1>(ctx, "rt_count_orfs", *q)) return rc;
    const int64_t n = R.n, n_slot = R.slots();
    if (n_slot > (int64_t)0xffffffffll)
        return fail(ctx, RT_EINVAL, "count-orfs handles at most 2^32 - 1 nt in the selected rows; the selection has %lld",
                    (long long)n_slot);
    if (int rc = R.gather(ctx, "rt_count_orfs", 0, [](int64_t) {})) return rc;
    if (stage_ms) {
        for (int k = 0; k < RT_COUNT_STAGES; ++k) stage_ms[k] = 0.f;
        stage_ms[0] = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_host).count();
    }
    for (int k = 0; k < 4; ++k) summary[k] = 0;
    summary[2] = -1;
    // 2. uploads
    RT_CUDA(ctx, S.st.create());
    for (auto& e : S.ev) RT_CUDA(ctx, e.create());
    const size_t ns = (size_t)n_slot, ng = (size_t)q->n_gene;
    if (int rc = R.reserve(ctx)) return rc;
    RT_CUDA(ctx, S.key.reserve(ns));
    RT_CUDA(ctx, S.key2.reserve(ns));
    RT_CUDA(ctx, S.val.reserve(ns));
    RT_CUDA(ctx, S.val2.reserve(ns));
    RT_CUDA(ctx, S.counters.reserve(2));
    RT_CUDA(ctx, S.total.reserve(ng));
    RT_CUDA(ctx, S.length.reserve(ng));
    // the sort looks at the key bits in use: 32 of coordinate and those of the largest gene id, n_gene - 1.  A dropped
    // slot's key ~0 has all of them set, and a real key's gene field is at most n_gene - 1 < 2^bit_length(n_gene) - 1,
    // so a dropped slot sorts after every real key and never equals one.
    const unsigned items = (unsigned)ns;
    const int key_bits = 32 + bit_length((unsigned long long)q->n_gene);
    size_t temp_bytes = 0;
    RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, S.key.p, S.key2.p, S.val.p, S.val2.p, items, 0,
                                                 key_bits, S.st.s));
    RT_CUDA(ctx, S.temp.reserve(temp_bytes));
    RT_CUDA(ctx, cudaEventRecord(S.ev[0], S.st));
    if (int rc = R.upload(ctx, S.st)) return rc;
    const unsigned long long counters0[2] = {0, ~0ull};
    RT_CUDA(ctx, S.counters.upload(counters0, 2, S.st));
    RT_CUDA(ctx, cudaMemsetAsync(S.total.p, 0, sizeof(unsigned long long) * ng, S.st));
    RT_CUDA(ctx, cudaMemsetAsync(S.length.p, 0, sizeof(unsigned long long) * ng, S.st));
    RT_CUDA(ctx, cudaEventRecord(S.ev[1], S.st));
    // 3. count_emit_kernel
    const rt::CountArgs A{R.args(), S.key.p, S.val.p, S.counters.p};
    const int64_t big = std::max(1, ctx->n_sm * 8);
    if (n) {
        rt::count_emit_kernel<<<R.emit_grid(big), rt::kCodonWarps * 32, 0, S.st>>>(A);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(S.ev[2], S.st));
    unsigned long long h_counters[2];
    RT_CUDA(ctx, cudaMemcpyAsync(h_counters, S.counters.p, sizeof h_counters, cudaMemcpyDeviceToHost, S.st));
    RT_CUDA(ctx, cudaStreamSynchronize(S.st));
    summary[0] = (int64_t)h_counters[0];
    if (h_counters[1] != ~0ull) {                      // a refused profile: no counts
        if (int rc = R.read_refusal(ctx, S.st, h_counters[1], summary + 2)) return rc;
        if (stage_ms) RT_CUDA(ctx, stage_times(S.ev, 1, stage_ms + 1));
        return RT_OK;
    }
    // 4. stable sort by key: slots are in (line, oriented nt) order, so the first slot of every key is the first pair
    if (items)
        RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(S.temp.p, temp_bytes, S.key.p, S.key2.p, S.val.p, S.val2.p, items, 0,
                                                     key_bits, S.st.s));
    RT_CUDA(ctx, cudaEventRecord(S.ev[3], S.st));
    // 5. count_keep_kernel
    if (items) {
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((int64_t)(ns + 255) / 256, big));
        rt::count_keep_kernel<<<grid, 256, 0, S.st>>>(S.key2.p, S.val2.p, (long long)ns, S.total.p, S.length.p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(S.ev[4], S.st));
    // 6. copy-back
    if (ng) {
        RT_CUDA(ctx, cudaMemcpyAsync(total, S.total.p, 8 * ng, cudaMemcpyDeviceToHost, S.st));
        RT_CUDA(ctx, cudaMemcpyAsync(length, S.length.p, 8 * ng, cudaMemcpyDeviceToHost, S.st));
    }
    RT_CUDA(ctx, cudaEventRecord(S.ev[5], S.st));
    RT_CUDA(ctx, cudaStreamSynchronize(S.st));
    uint64_t kept = 0;
    for (size_t g = 0; g < ng; ++g) kept += length[g];
    summary[1] = (int64_t)kept;
    if (stage_ms) RT_CUDA(ctx, stage_times(S.ev, RT_COUNT_STAGES - 1, stage_ms + 1));
    return RT_OK;
}

}  // extern "C"

// -------------------------------------------------------------------------------------------------- BGZF text inputs
namespace {
constexpr size_t kInflatePiece = size_t(64) << 20;   // text bytes per page-locked copy-back buffer

// Streams, events and buffers of one rt_bgzf_inflate call; the destructor waits for the streams before the members are
// freed, so every early return leaves nothing behind.
struct InflatePipeline {
    Stream ks, us, cs;                                     // kernels, uploads, copy-back
    std::unique_ptr<Event[]> up_begin, up_end, k_begin, k_end;   // per kernel launch
    Event c_begin[2], c_end[2];                            // per page-locked buffer
    PinnedArr<char> pinned[2];
    DevArr<uint8_t> comp, text, status;
    DevArr<rt::BgzfBlock> tab;
    DevArr<unsigned> claim;                                // one work counter per launch
    explicit InflatePipeline(size_t n)
        : up_begin(new Event[n]), up_end(new Event[n]), k_begin(new Event[n]), k_end(new Event[n]) {}
    ~InflatePipeline() {
        for (cudaStream_t s : {ks.s, us.s, cs.s})
            if (s) cudaStreamSynchronize(s);
    }
};

float ms_since(std::chrono::steady_clock::time_point t) {
    return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t).count();
}

// The members inflated on the device and the text copied into `out`.  Launches of one member per resident warp (so each
// fills the GPU) run in order on one stream, each after the upload of its members' payload on another.  The text comes
// back in pieces of kInflatePiece bytes through two page-locked buffers, each piece as soon as the launches that write
// it have finished, and host threads drain a piece into `out` while the next piece is copied and later launches run: a
// single copy into pageable memory runs at the rate one thread faults in the destination's pages.
// ms[2..5]: upload (summed), kernels (first start to last end), copy-back into the page-locked buffers (summed), drain.
int inflate_on_device(rt_ctx* ctx, const uint8_t* base, size_t size, const std::vector<rt::BgzfBlock>& tab, size_t total,
                      char* out, std::vector<uint8_t>& status, float* ms) {
    const size_t nb = tab.size();
    DeviceGuard guard(ctx->device);
    int per_sm = 0;
    RT_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rt::bgzf_inflate_kernel, rt::kInflateWarps * 32, 0));
    const size_t ctas = (size_t)std::max(1, per_sm) * (size_t)std::max(1, ctx->n_sm);
    const size_t per_launch = ctas * rt::kInflateWarps;
    const size_t n_launch = (nb + per_launch - 1) / per_launch;
    InflatePipeline P(n_launch);
    RT_CUDA(ctx, P.ks.create());
    RT_CUDA(ctx, P.us.create());
    RT_CUDA(ctx, P.cs.create());
    for (size_t c = 0; c < n_launch; ++c)
        for (Event* e : {&P.up_begin[c], &P.up_end[c], &P.k_begin[c], &P.k_end[c]}) RT_CUDA(ctx, e->create());
    for (int b = 0; b < 2; ++b) {
        RT_CUDA(ctx, P.c_begin[b].create());
        RT_CUDA(ctx, P.c_end[b].create());
    }
    RT_CUDA(ctx, P.comp.reserve(size));
    RT_CUDA(ctx, P.text.reserve(total));
    RT_CUDA(ctx, P.status.reserve(nb));
    RT_CUDA(ctx, P.tab.reserve(nb));
    RT_CUDA(ctx, P.claim.reserve(n_launch));
    RT_CUDA(ctx, P.tab.upload(tab.data(), nb, P.ks));
    RT_CUDA(ctx, cudaMemsetAsync(P.claim.p, 0, sizeof(unsigned) * n_launch, P.ks));
    // 1. uploads and launches, in order
    std::vector<size_t> launch_out(n_launch);             // first text byte each launch writes
    for (size_t c = 0; c < n_launch; ++c) {
        const size_t m0 = c * per_launch, m1 = std::min(nb, m0 + per_launch);
        const size_t lo = tab[m0].in_off, hi = tab[m1 - 1].in_off + tab[m1 - 1].in_len;
        launch_out[c] = tab[m0].out_off;
        RT_CUDA(ctx, cudaEventRecord(P.up_begin[c], P.us));
        if (hi > lo) RT_CUDA(ctx, cudaMemcpyAsync(P.comp.p + lo, base + lo, hi - lo, cudaMemcpyHostToDevice, P.us));
        RT_CUDA(ctx, cudaEventRecord(P.up_end[c], P.us));
        RT_CUDA(ctx, cudaStreamWaitEvent(P.ks, P.up_end[c], 0));
        RT_CUDA(ctx, cudaEventRecord(P.k_begin[c], P.ks));
        const unsigned grid = (unsigned)std::min(ctas, (m1 - m0 + rt::kInflateWarps - 1) / rt::kInflateWarps);
        rt::bgzf_inflate_kernel<<<grid, rt::kInflateWarps * 32, 0, P.ks>>>(P.comp.p, P.tab.p + m0, (long long)(m1 - m0), P.text.p,
                                                                          P.status.p + m0, P.claim.p + c);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
        RT_CUDA(ctx, cudaEventRecord(P.k_end[c], P.ks));
    }
    RT_CUDA(ctx, cudaMemcpyAsync(status.data(), P.status.p, nb, cudaMemcpyDeviceToHost, P.ks));
    // 2. the text, piece by piece: copy-back of piece p overlaps the drain of piece p - 1
    const size_t n_pieces = (total + kInflatePiece - 1) / kInflatePiece;
    for (size_t b = 0; b < 2 && b < n_pieces; ++b) RT_CUDA(ctx, P.pinned[b].alloc(std::min(kInflatePiece, total)));
    auto piece_bytes = [&](size_t p) { return std::min(kInflatePiece, total - p * kInflatePiece); };
    auto drain = [&](size_t p) -> int {
        const int b = (int)(p & 1);
        RT_CUDA(ctx, cudaEventSynchronize(P.c_end[b]));
        float c_ms = 0.f;
        RT_CUDA(ctx, cudaEventElapsedTime(&c_ms, P.c_begin[b], P.c_end[b]));
        ms[4] += c_ms;
        const auto t = std::chrono::steady_clock::now();
        const size_t n = piece_bytes(p), slice = size_t(1) << 20, n_slices = (n + slice - 1) / slice;
        char* dst = out + p * kInflatePiece;
        const char* src = P.pinned[b].p;
        claim_parallel(host_threads(n_slices, 64), n_slices, [&](size_t k) {
            memcpy(dst + k * slice, src + k * slice, std::min(slice, n - k * slice));
        });
        ms[5] += ms_since(t);
        return RT_OK;
    };
    for (size_t p = 0; p < n_pieces; ++p) {
        const int b = (int)(p & 1);                        // buffer b was drained with piece p - 2
        const size_t hi = p * kInflatePiece + piece_bytes(p);
        const size_t last = (size_t)(std::upper_bound(launch_out.begin(), launch_out.end(), hi - 1) - launch_out.begin()) - 1;
        RT_CUDA(ctx, cudaStreamWaitEvent(P.cs, P.k_end[last], 0));
        RT_CUDA(ctx, cudaEventRecord(P.c_begin[b], P.cs));
        RT_CUDA(ctx, cudaMemcpyAsync(P.pinned[b].p, P.text.p + p * kInflatePiece, piece_bytes(p), cudaMemcpyDeviceToHost, P.cs));
        RT_CUDA(ctx, cudaEventRecord(P.c_end[b], P.cs));
        if (p >= 1)
            if (const int rc = drain(p - 1)) return rc;
    }
    if (n_pieces)
        if (const int rc = drain(n_pieces - 1)) return rc;
    RT_CUDA(ctx, cudaStreamSynchronize(P.ks));
    RT_CUDA(ctx, cudaStreamSynchronize(P.us));
    for (size_t c = 0; c < n_launch; ++c) {
        float u = 0.f;
        RT_CUDA(ctx, cudaEventElapsedTime(&u, P.up_begin[c], P.up_end[c]));
        ms[2] += u;
    }
    RT_CUDA(ctx, cudaEventElapsedTime(&ms[3], P.k_begin[0], P.k_end[n_launch - 1]));
    return RT_OK;
}
}  // namespace

extern "C" {

int rt_bgzf_inflate(rt_ctx* ctx, const char* path, rt_text** out, int64_t* summary, float* stage_ms) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bgzf_inflate: ctx is NULL");
    if (!path || !out) return fail(ctx, RT_EINVAL, "rt_bgzf_inflate: NULL argument");
    *out = nullptr;
    float ms[RT_BGZF_STAGES] = {};
    // 1. the file, read in slices by all threads
    auto t0 = std::chrono::steady_clock::now();
    HostArr<char> file;
    if (const int rc = read_file(path, file)) return fail(ctx, rc, "%s", rt_io_last_error());
    ms[0] = ms_since(t0);
    // 2. the member chain: block table and output offsets
    t0 = std::chrono::steady_clock::now();
    const uint8_t* base = reinterpret_cast<const uint8_t*>(file.data());
    const size_t size = file.size();
    std::vector<rt::BgzfBlock> tab;
    std::vector<size_t> at;                           // byte offset of every member, for messages
    unsigned long long total = 0;
    for (size_t off = 0; off < size;) {
        Block b;
        size_t next;
        const long long k = (long long)tab.size();
        if (!parse_block(base, size, off, b, next)) {
            const int why = block_refusal(base, size, off);
            if (why == 2 && k > 0)
                return fail(ctx, RT_EINVAL, "%s: BGZF block %lld at byte %zu: %zu bytes after the last member are not a BGZF member",
                            path, k, off, size - off);
            if (why == 1) return fail(ctx, RT_EINVAL, "%s: BGZF block %lld at byte %zu: truncated, the file ends inside it", path, k, off);
            return fail(ctx, RT_EINVAL, "%s: BGZF block %lld at byte %zu: not a BGZF member header", path, k, off);
        }
        tab.push_back({(unsigned long long)b.in_off, total, (unsigned)b.in_len, b.out_len, b.crc, 0u});
        at.push_back(off);
        total += b.out_len;
        off = next;
    }
    rt_text* raw = nullptr;
    if (rt_text_alloc((int64_t)total, &raw) != RT_OK)
        return fail(ctx, RT_ENOMEM, "rt_bgzf_inflate: no host memory for the %llu inflated bytes of %s", total, path);
    std::unique_ptr<rt_text, void (*)(rt_text*)> text(raw, rt_text_free);
    ms[1] = ms_since(t0);
    // 3. device: inflate, copy back
    const size_t nb = tab.size();
    std::vector<uint8_t> status(nb, 0);
    if (nb)
        if (const int rc = inflate_on_device(ctx, base, size, tab, (size_t)total, text->p, status, ms)) return rc;
    // 4. members the device refused, decoded again on the host (rt_inflate.cpp, then zlib)
    t0 = std::chrono::steady_clock::now();
    std::vector<size_t> redo;
    for (size_t k = 0; k < nb; ++k)
        if (status[k] != rt::kInfOk) redo.push_back(k);
    std::vector<char> ok(redo.size(), 0);
    claim_parallel(host_threads(redo.size(), SIZE_MAX), redo.size(), [&](size_t j) {
        const rt::BgzfBlock& b = tab[redo[j]];
        ok[j] = inflate_block(base + b.in_off, b.in_len, reinterpret_cast<uint8_t*>(text->p) + b.out_off, b.out_len, b.crc, false) &&
                (b.out_len != 0 || b.crc == 0);
    });
    if (summary) {
        summary[0] = (int64_t)nb;
        summary[1] = (int64_t)size;
        summary[2] = (int64_t)total;
        summary[3] = (int64_t)redo.size();
    }
    for (size_t j = 0; j < redo.size(); ++j)
        if (!ok[j]) {
            const rt::BgzfBlock& b = tab[redo[j]];
            return fail(ctx, RT_EINVAL, "%s: BGZF block %zu at byte %zu: does not inflate to its ISIZE of %u bytes and CRC-32 %08x", path,
                        redo[j], at[redo[j]], b.out_len, b.crc);
        }
    ms[6] = ms_since(t0);
    if (stage_ms)
        for (int k = 0; k < RT_BGZF_STAGES; ++k) stage_ms[k] = ms[k];
    *out = text.release();
    return RT_OK;
}

}  // extern "C"
