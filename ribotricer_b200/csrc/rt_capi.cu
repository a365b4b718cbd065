// rt_capi.cu -- C ABI (include/ribotricer_b200.h) over the sm_100a kernels.
// Host-side state: genome layout, device-resident CSR index, scratch for the host-buffer calls.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <mutex>
#include <string>
#include <unordered_map>
#include <thread>
#include <vector>

#include "rt_kernels.cuh"

// rt_host_io.cpp: filter cascade + run-length code of ref_id for one chunk of host columns
int64_t rt_pack_chunk(const int32_t* ref_id, const uint16_t* flag, const uint8_t* mapq, const uint8_t* nh, int64_t m, uint8_t* meta,
                      int64_t* run_start, int32_t* run_ref, int64_t cap);
// rt_host_io.cpp: one chunk of host columns as a run of record-stream blocks (-1: cannot be coded, -2: cap too small)
int64_t rt_stream_pack_range(const int32_t* ref_id, const int32_t* first, const int32_t* last, const uint16_t* mlen, const uint16_t* flag,
                             const uint8_t* mapq, const uint8_t* nh, int64_t m, uint32_t* rec, int32_t* hdr, int64_t cap);

namespace {

thread_local std::string g_last_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

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
    int2* d_contig_tab = nullptr;                    // per contig: (length, first slot >> 5)
    double2* d_uv_table = nullptr;                   // unit vectors of small codons (rt::fill_uv_table), for phase B's seam windows

    // read-length table
    int32_t* d_len_table = nullptr;
    bool have_len_table = false;
    int len_base = 20;   // first of the 16 read lengths K1 counts in registers
    int zone_delta_plus = 0, zone_delta_minus = 0;   // smallest P-site displacement from `first` on either strand

    // index
    int64_t n_orf = 0;
    uint64_t* d_orf_desc = nullptr;
    int32_t* d_orf_len = nullptr;
    cudaEvent_t ev_scored = nullptr;                 // rt_score_host: a part's columns are ready for their copy
    uint64_t* d_exon_entries = nullptr;
    std::vector<int64_t> bytes_prefix;  // n_orf + 1: prefix of 4L + 8E + 42
    std::vector<int64_t> nt_prefix;     // n_orf + 1: prefix of L
    unsigned long long* d_work_counter = nullptr;   // 4 x u64: work counters of phase A (0) and the fallback (2), fallback count (3)

    // two-phase scoring: atoms (coverage intervals no ORF exon boundary splits) and per-ORF atom refs
    int64_t n_atoms = 0;
    uint64_t* d_atoms = nullptr;                     // (slot offset << 24) | len
    rt::AtomSummary* d_summaries = nullptr;          // per-library scratch, written by phase A
    uint8_t* d_atom_nonzero = nullptr;               // per-library scratch: atom holds at least one read
    // compact layout: the coverage buffer holds the exon union only (atoms back to back, genome order)
    int layout = RT_LAYOUT_DENSE;
    int64_t compact_elems = 0;                       // int32 elements of a compact coverage buffer (with guard)
    unsigned* d_cbits = nullptr;                     // one bit per cmap word: the word has members
    unsigned compact_plus_end = 0, compact_end = 0;  // compact index after the last '+' slot / after the last slot
    DevBuf zone_buf, spill_buf;                      // rt_bin_stream_fresh: zone boundaries, spill list + its counter
    uint2* d_cmap = nullptr;                         // per 32 dense slots: member mask | compact index after the last member
    uint64_t* d_atoms_c = nullptr;                   // the same tables with compact slot offsets
    uint64_t* d_exon_entries_c = nullptr;
    std::vector<uint64_t> h_atoms;                   // host copies used to build per-range atom lists
    std::vector<uint64_t> h_atoms_c;                 // ... with compact slot offsets
    std::vector<uint64_t> h_orf_refs_desc;           // per ORF: ref begin | n_refs << 40 | reverse << 63
    std::vector<uint32_t> h_ref_atom;                // atom id of every ref (0xffffffff: reads as zeros)
    std::vector<uint64_t> h_ref_ent;                 // refs in profile order

    // score plan: the work lists of the three scoring launches for one ORF range
    struct ScorePlan {
        int64_t lo = -1, hi = -1;
        int32_t* d_fallback = nullptr;  // ORFs redone by score_orfs_kernel; capacity hi - lo
        int32_t* d_atom_list = nullptr; // atoms the range touches, similar lengths adjacent
        int64_t n_atom_list = 0;
        rt::PassDesc* d_passes = nullptr;      // compact layout: runs of adjacent atoms for atom_pass_kernel
        int64_t n_passes = 0;
        rt::RefRec* d_refs = nullptr;          // compose_refs_kernel: one slot per atom reference, groups of 32
        rt::RefWarp* d_ref_warps = nullptr;
        rt::LongAcc* d_long_acc = nullptr;     // one per ORF with more than 32 references
        int64_t n_ref_warps = 0;
    };
    std::vector<ScorePlan> plans;

    // scratch for the host-buffer entry points
    struct HostStage {                               // page-locked staging of one chunk's record stream
        uint32_t* rec = nullptr;
        int32_t* hdr = nullptr;
        cudaEvent_t copied = nullptr;
        bool busy = false;
    } host_stage[16];
    std::mutex launch_mutex;                         // the packing threads of rt_bin_reads_host launch K1 one at a time
    DevBuf read_slot[16];
    cudaStream_t slot_stream[16] = {};
    DevBuf stats_buf, score_buf;

    // sparse clear: slots touched by K1 since the last rt_clear_touched
    bool track_touched = false;
    DevBuf touched_buf;
    unsigned long long* d_n_touched = nullptr;
    int64_t touched_reserved = 0;    // reads binned (weight +1) since the last clear

    // prepare-orfs (rt_orf_search / rt_orf_fetch): the last search's tables and rows stay on the device until fetched
    DevBuf orf_buf[32];
    std::vector<int64_t> orf_iv_ptr;                 // n_rows + 1: interval offsets of the last search
    int64_t orf_rows = 0;
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
    const size_t need = sizeof(unsigned long long) * (size_t)reads;
    if (need <= ctx->touched_buf.cap) return RT_OK;
    DevBuf bigger;
    RT_CUDA(ctx, bigger.reserve(std::max(need, ctx->touched_buf.cap * 2)));
    if (ctx->touched_buf.p) {
        RT_CUDA(ctx, cudaDeviceSynchronize());
        RT_CUDA(ctx, cudaMemcpy(bigger.p, ctx->touched_buf.p, sizeof(unsigned long long) * (size_t)ctx->touched_reserved,
                                cudaMemcpyDeviceToDevice));
        ctx->touched_buf.release();
    }
    ctx->touched_buf = bigger;
    return RT_OK;
}

// Two-phase scoring, host side: cut the exon entries of all ORFs at every entry boundary into atoms
// (no ORF exon boundary falls inside an atom; atoms longer than kAtomMaxNt are chopped) and express
// every ORF as its sequence of atoms in profile order.
int build_atoms(rt_ctx* ctx, const std::vector<uint64_t>& desc, const std::vector<uint64_t>& entries) {
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
    const int n_thr = (int)std::max<size_t>(1, std::min<size_t>({(size_t)std::thread::hardware_concurrency(), (size_t)16, pts.size() >> 16}));
    auto parallel_for = [&](size_t n_items, auto&& body) {          // body(lo, hi) on slices of [0, n_items)
        std::vector<std::thread> pool;
        for (int k = 1; k < n_thr; ++k) pool.emplace_back([&, k]() { body(n_items * k / n_thr, n_items * (k + 1) / n_thr); });
        body(0, n_items / n_thr);
        for (auto& th : pool) th.join();
    };
    parallel_for(pts.size(), [&](size_t lo, size_t hi) { std::sort(pts.begin() + lo, pts.begin() + hi); });
    for (int width = 1; width < n_thr; width *= 2) {
        std::vector<std::thread> pool;
        for (int k = 0; k + width < n_thr; k += 2 * width)
            pool.emplace_back([&, k, width]() {
                const size_t a = pts.size() * k / n_thr, m = pts.size() * (k + width) / n_thr;
                const size_t b = pts.size() * std::min(k + 2 * width, n_thr) / n_thr;
                std::inplace_merge(pts.begin() + a, pts.begin() + m, pts.begin() + b);
            });
        for (auto& th : pool) th.join();
    }
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
    ctx->h_atoms.clear();
    int64_t cover = 0;
    for (size_t i = 0; i + 1 < pts.size(); ++i) {
        cover += diff[i];
        atom_begin[i] = (uint32_t)ctx->h_atoms.size();
        if (cover > 0) {
            uint64_t at = pts[i];
            while (at < pts[i + 1]) {
                const uint64_t piece = std::min<uint64_t>(pts[i + 1] - at, (uint64_t)rt::kAtomMaxNt);
                ctx->h_atoms.push_back((at << rt::kLenBits) | piece);
                at += piece;
            }
        }
    }
    if (!pts.empty()) atom_begin[pts.size() - 1] = atom_begin[pts.size()] = (uint32_t)ctx->h_atoms.size();
    if (ctx->h_atoms.size() >= 0xffffffffull) return fail(ctx, RT_EINVAL, "rt_set_index: too many atoms");
    // per-ORF refs in profile order
    const size_t n_orf = desc.size();
    ctx->h_orf_refs_desc.assign(n_orf, 0);
    ctx->h_ref_ent.clear();
    ctx->h_ref_atom.clear();
    ctx->h_ref_ent.reserve(entries.size() * 3 / 2);
    ctx->h_ref_atom.reserve(entries.size() * 3 / 2);
    for (size_t o = 0; o < n_orf; ++o) {
        const uint64_t begin = desc[o] & rt::kBeginMask;
        const int n_ent = (int)((desc[o] >> 40) & rt::kMaxEntriesPerOrf);
        const bool rev = (desc[o] >> 63) != 0;
        const size_t ref_begin = ctx->h_ref_ent.size();
        for (int k = 0; k < n_ent; ++k) {
            const size_t e = begin + (size_t)(rev ? n_ent - 1 - k : k);
            const uint64_t ent = entries[e];
            const uint64_t off = ent >> rt::kLenBits;
            if (off == kZero) {
                ctx->h_ref_ent.push_back(ent);
                ctx->h_ref_atom.push_back(0xffffffffu);   // reads-as-zero stretch: no atom
                continue;
            }
            const uint32_t a0 = atom_begin[ilo[e]], a1 = atom_begin[ihi[e]];
            for (uint32_t a = 0; a < a1 - a0; ++a) {
                const uint32_t atom = rev ? a1 - 1 - a : a0 + a;
                ctx->h_ref_ent.push_back(ctx->h_atoms[atom]);
                ctx->h_ref_atom.push_back(atom);
            }
        }
        const size_t cnt = ctx->h_ref_ent.size() - ref_begin;
        if (cnt > (size_t)rt::kMaxEntriesPerOrf) return fail(ctx, RT_EINVAL, "rt_set_index: ORF %zu has too many atoms", o);
        ctx->h_orf_refs_desc[o] = (uint64_t)ref_begin | ((uint64_t)cnt << 40) | ((uint64_t)rev << 63);
    }
    ctx->n_atoms = (int64_t)ctx->h_atoms.size();
    // compact layout: atom i starts at the sum of the lengths of the atoms before it
    std::vector<uint64_t>& atoms_c = ctx->h_atoms_c;
    atoms_c.assign(ctx->h_atoms.size(), 0);
    std::vector<uint64_t> entries_c(entries.size());
    uint64_t cat = 0;
    for (size_t i = 0; i < atoms_c.size(); ++i) {
        const uint64_t len = ctx->h_atoms[i] & rt::kLenMask;
        atoms_c[i] = (cat << rt::kLenBits) | len;
        cat += len;
    }
    ctx->compact_elems = (int64_t)((cat + 31) / 32 * 32 + 32);
    ctx->compact_end = (unsigned)std::min<uint64_t>(cat, 0xffffffffull);
    ctx->compact_plus_end = ctx->compact_end;        // atoms are in slot order: the first one of the '-' plane ends the '+' part
    for (size_t i = 0; i < atoms_c.size(); ++i)
        if ((ctx->h_atoms[i] >> rt::kLenBits) >= (uint64_t)ctx->plane) {
            ctx->compact_plus_end = (unsigned)(atoms_c[i] >> rt::kLenBits);
            break;
        }
    for (size_t k = 0; k < entries.size(); ++k) {
        const uint64_t off = entries[k] >> rt::kLenBits, len = entries[k] & rt::kLenMask;
        entries_c[k] = off == kZero ? entries[k] : ((atoms_c[atom_begin[ilo[k]]] >> rt::kLenBits) << rt::kLenBits) | len;
    }
    auto upload = [&](auto** dptr, const auto& vec) -> cudaError_t {
        using T = typename std::remove_reference<decltype(vec)>::type::value_type;
        cudaError_t e = cudaMalloc(dptr, sizeof(T) * (vec.size() + 4));   // slack: atom_pass_kernel copies descriptor pairs
        if (e == cudaSuccess && !vec.empty()) e = cudaMemcpy(*dptr, vec.data(), sizeof(T) * vec.size(), cudaMemcpyHostToDevice);
        return e;
    };
    RT_CUDA(ctx, upload(&ctx->d_atoms, ctx->h_atoms));
    RT_CUDA(ctx, upload(&ctx->d_atoms_c, atoms_c));
    RT_CUDA(ctx, upload(&ctx->d_exon_entries_c, entries_c));
    RT_CUDA(ctx, cudaMalloc(&ctx->d_summaries, sizeof(rt::AtomSummary) * std::max<size_t>(1, ctx->h_atoms.size())));
    RT_CUDA(ctx, cudaMalloc(&ctx->d_atom_nonzero, std::max<size_t>(1, ctx->h_atoms.size())));
    return RT_OK;   // the host copies stay: build_plan_host makes the atom lists and the families from them
}

void free_plan(rt_ctx::ScorePlan& p) {
    cudaFree(p.d_fallback);
    cudaFree(p.d_atom_list);
    cudaFree(p.d_passes);
    cudaFree(p.d_refs);
    cudaFree(p.d_ref_warps);
    cudaFree(p.d_long_acc);
}

constexpr size_t kReadBytes = 4 + 4 + 4 + 2 + 2 + 1 + 1;
constexpr size_t kPackedReadBytes = 4 + 4 + 2 + 1;
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
    rt_ctx* ctx = new rt_ctx();
    ctx->device = device;
    ctx->n_sm = prop.multiProcessorCount;
    if (cudaMalloc(&ctx->d_work_counter, 4 * sizeof(unsigned long long)) != cudaSuccess ||
        cudaMalloc(&ctx->d_len_table, sizeof(int32_t) * RT_LEN_TABLE) != cudaSuccess) {
        delete ctx;
        return fail(nullptr, RT_ENOMEM, "rt_create: cudaMalloc failed");
    }
    if (cudaMalloc(&ctx->d_uv_table, sizeof(double2) * rt::kUvEntries) != cudaSuccess) {
        delete ctx;
        return fail(nullptr, RT_ENOMEM, "rt_create: cudaMalloc failed");
    }
    rt::fill_uv_table_kernel<<<1, 256>>>(ctx->d_uv_table);
    if (cudaDeviceSynchronize() != cudaSuccess) {
        delete ctx;
        return fail(nullptr, RT_ECUDA, "rt_create: %s", cudaGetErrorString(cudaGetLastError()));
    }
    *out = ctx;
    return RT_OK;
}

void rt_destroy(rt_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    for (auto& b : ctx->orf_buf) b.release();
    cudaFree(ctx->d_contig_tab);
    cudaFree(ctx->d_uv_table);
    cudaFree(ctx->d_len_table);
    cudaFree(ctx->d_orf_desc);
    cudaFree(ctx->d_orf_len);
    cudaFree(ctx->d_exon_entries);
    cudaFree(ctx->d_atoms);
    cudaFree(ctx->d_summaries);
    cudaFree(ctx->d_atom_nonzero);
    cudaFree(ctx->d_cmap);
    cudaFree(ctx->d_cbits);
    cudaFree(ctx->d_atoms_c);
    cudaFree(ctx->d_exon_entries_c);
    cudaFree(ctx->d_work_counter);
    if (ctx->ev_scored) cudaEventDestroy(ctx->ev_scored);
    for (auto& p : ctx->plans) free_plan(p);
    for (int s = 0; s < 16; ++s) {
        if (ctx->host_stage[s].rec) cudaFreeHost(ctx->host_stage[s].rec);
        if (ctx->host_stage[s].hdr) cudaFreeHost(ctx->host_stage[s].hdr);
        if (ctx->host_stage[s].copied) cudaEventDestroy(ctx->host_stage[s].copied);
        ctx->read_slot[s].release();
        if (ctx->slot_stream[s]) cudaStreamDestroy(ctx->slot_stream[s]);
    }
    ctx->stats_buf.release();
    ctx->score_buf.release();
    ctx->touched_buf.release();
    cudaFree(ctx->d_n_touched);
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
    cudaFree(ctx->d_contig_tab);
    ctx->d_contig_tab = nullptr;
    std::vector<int2> tab((size_t)std::max(1, n_contig));
    for (int c = 0; c < n_contig; ++c) tab[c] = make_int2((int)h_contig_len[c], (int)(ctx->contig_base[c] >> 5));
    RT_CUDA(ctx, cudaMalloc(&ctx->d_contig_tab, sizeof(int2) * tab.size()));
    RT_CUDA(ctx, cudaMemcpy(ctx->d_contig_tab, tab.data(), sizeof(int2) * tab.size(), cudaMemcpyHostToDevice));
    // a new genome invalidates the index encoding
    ctx->n_orf = 0;
    ctx->layout = RT_LAYOUT_DENSE;
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
    RT_CUDA(ctx, cudaMemcpy(ctx->d_len_table, h_len_table, sizeof(int32_t) * RT_LEN_TABLE, cudaMemcpyHostToDevice));
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
    const size_t elems = ctx->layout == RT_LAYOUT_COMPACT ? (size_t)ctx->compact_elems : 2 * (size_t)ctx->plane;
    RT_CUDA(ctx, cudaMemsetAsync(d_cov, 0, sizeof(int32_t) * elems, (cudaStream_t)stream));
    return RT_OK;
}

int rt_set_layout(rt_ctx* ctx, int layout) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_set_layout: ctx is NULL");
    if (layout != RT_LAYOUT_DENSE && layout != RT_LAYOUT_COMPACT) return fail(ctx, RT_EINVAL, "rt_set_layout: unknown layout %d", layout);
    if (layout == RT_LAYOUT_COMPACT) {
        if (ctx->n_orf == 0) return fail(ctx, RT_ESTATE, "rt_set_layout: the compact layout is derived from the index; call rt_set_index first");
        if (ctx->compact_elems >= 0xffffffffll) return fail(ctx, RT_EINVAL, "rt_set_layout: exon union too large for 32-bit compact slots");
        DeviceGuard guard(ctx->device);
        if (!ctx->d_cmap) {
            const size_t words = (size_t)(2 * ctx->plane / 32);
            RT_CUDA(ctx, cudaMalloc(&ctx->d_cmap, sizeof(uint2) * words));
            RT_CUDA(ctx, cudaMemset(ctx->d_cmap, 0, sizeof(uint2) * words));
            if (ctx->n_atoms > 0) {
                const unsigned grid = (unsigned)std::min<int64_t>((ctx->n_atoms + 7) / 8, (int64_t)ctx->n_sm * 16);
                rt::build_cmap_kernel<<<grid, 256>>>(ctx->d_atoms, ctx->d_atoms_c, ctx->n_atoms, ctx->d_cmap);
                ctx->launches++;
                RT_CUDA(ctx, cudaGetLastError());
            }
            {   // empty words carry the compact index of the next member (cmap_rank: zone boundaries of rt_bin_stream_fresh)
                const size_t tiles = (words + rt::kGapTile - 1) / rt::kGapTile;
                DevBuf tile_buf;
                RT_CUDA(ctx, tile_buf.reserve(sizeof(unsigned) * tiles));
                unsigned* d_tile = static_cast<unsigned*>(tile_buf.p);
                rt::cmap_tile_last_kernel<<<(unsigned)tiles, 256>>>(ctx->d_cmap, (long long)words, d_tile);
                std::vector<unsigned> h_tile(tiles);
                RT_CUDA(ctx, cudaMemcpy(h_tile.data(), d_tile, sizeof(unsigned) * tiles, cudaMemcpyDeviceToHost));
                unsigned carry = 0;
                for (size_t t = 0; t < tiles; ++t) {      // exclusive prefix maximum
                    const unsigned last = h_tile[t];
                    h_tile[t] = carry;
                    carry = std::max(carry, last);
                }
                RT_CUDA(ctx, cudaMemcpy(d_tile, h_tile.data(), sizeof(unsigned) * tiles, cudaMemcpyHostToDevice));
                rt::cmap_fill_gaps_kernel<<<(unsigned)tiles, 256>>>(ctx->d_cmap, (long long)words, d_tile);
                ctx->launches += 2;
                RT_CUDA(ctx, cudaGetLastError());
                RT_CUDA(ctx, cudaDeviceSynchronize());
                tile_buf.release();
            }
            RT_CUDA(ctx, cudaMalloc(&ctx->d_cbits, sizeof(unsigned) * ((words + 31) / 32)));
            rt::build_cbits_kernel<<<(unsigned)((words + 255) / 256), 256>>>(ctx->d_cmap, (long long)words, ctx->d_cbits);
            ctx->launches++;
            RT_CUDA(ctx, cudaGetLastError());
            RT_CUDA(ctx, cudaDeviceSynchronize());
        }
    }
    ctx->layout = layout;
    return RT_OK;
}

int64_t rt_coverage_elems(const rt_ctx* ctx) {
    if (!ctx) return 0;
    return ctx->layout == RT_LAYOUT_COMPACT ? ctx->compact_elems : 2 * ctx->plane;
}

int rt_track_touched(rt_ctx* ctx, int enable) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_track_touched: ctx is NULL");
    DeviceGuard guard(ctx->device);
    if (enable && !ctx->d_n_touched) {
        RT_CUDA(ctx, cudaMalloc(&ctx->d_n_touched, sizeof(unsigned long long)));
        RT_CUDA(ctx, cudaMemset(ctx->d_n_touched, 0, sizeof(unsigned long long)));
    }
    ctx->track_touched = enable != 0;
    return RT_OK;
}

int rt_clear_touched(rt_ctx* ctx, int32_t* d_cov, void* stream) {
    if (!ctx || !d_cov) return fail(ctx, RT_EINVAL, "rt_clear_touched: NULL argument");
    if (!ctx->d_n_touched && ctx->layout != RT_LAYOUT_COMPACT)
        return fail(ctx, RT_ESTATE, "rt_clear_touched: call rt_track_touched(ctx, 1) first");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (ctx->layout == RT_LAYOUT_COMPACT) {   // the whole buffer is the exon union: a plain memset is the sparse clear
        RT_CUDA(ctx, cudaMemsetAsync(d_cov, 0, sizeof(int32_t) * (size_t)ctx->compact_elems, st));
        return RT_OK;
    }
    if (ctx->touched_buf.p) {
        rt::clear_touched_kernel<<<(unsigned)ctx->n_sm * 8, 256, 0, st>>>(
            d_cov, static_cast<const unsigned long long*>(ctx->touched_buf.p), ctx->d_n_touched);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_n_touched, 0, sizeof(unsigned long long), st));
    ctx->touched_reserved = 0;
    return RT_OK;
}

// ------------------------------------------------------------------------------------ K1
}  // extern "C"

namespace {

// Common part of rt_bin_reads / rt_bin_reads_packed: `a` arrives with its read columns filled in.
int launch_bin(rt_ctx* ctx, const char* who, rt::BinArgs& a, bool packed, int32_t* d_cov, int64_t n, int protocol,
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
    a.len_table = ctx->d_len_table;
    a.contig_tab = ctx->d_contig_tab;
    a.n_contig = ctx->n_contig;
    a.pad = ctx->pad;
    a.plane_words = (unsigned)(ctx->plane >> 5);
    a.stats = reinterpret_cast<unsigned long long*>(d_stats);
    a.len_counts = reinterpret_cast<unsigned long long*>(d_len_counts);
    a.touched = nullptr;
    a.n_touched = nullptr;
    a.cmap = ctx->layout == RT_LAYOUT_COMPACT ? ctx->d_cmap : nullptr;
    a.cbits = ctx->d_cbits;
    if (ctx->track_touched && weight == 1 && !a.cmap) {
        int rc = ensure_touched_capacity(ctx, ctx->touched_reserved + n);
        if (rc != RT_OK) return rc;
        ctx->touched_reserved += n;
        a.touched = static_cast<unsigned long long*>(ctx->touched_buf.p);
        a.n_touched = ctx->d_n_touched;
    }
    const int64_t per_block = (int64_t)rt::kBinThreads * rt::kBinReadsPerThread;
    const int64_t blocks = (n + per_block - 1) / per_block;
    if (blocks > 0x7fffffff) return fail(ctx, RT_EINVAL, "%s: n too large for one launch", who);
    cudaStream_t st = (cudaStream_t)stream;
    if (packed) {
        if (a.cmap) rt::bin_psites_kernel<true, true><<<(unsigned)blocks, rt::kBinThreads, 0, st>>>(a);
        else rt::bin_psites_kernel<false, true><<<(unsigned)blocks, rt::kBinThreads, 0, st>>>(a);
    } else {
        if (a.cmap) rt::bin_psites_kernel<true, false><<<(unsigned)blocks, rt::kBinThreads, 0, st>>>(a);
        else rt::bin_psites_kernel<false, false><<<(unsigned)blocks, rt::kBinThreads, 0, st>>>(a);
    }
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
    return launch_bin(ctx, "rt_bin_reads", a, false, d_cov, n, protocol, weight, d_stats, d_len_counts, stream);
}

int rt_bin_reads_packed(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* d_first, const int32_t* d_last,
                        const uint16_t* d_mlen, const uint8_t* d_meta, int64_t read_base, int64_t n_runs,
                        const int64_t* d_run_start, const int32_t* d_run_ref, int protocol, int weight,
                        int64_t* d_stats, int64_t* d_len_counts, void* stream) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bin_reads_packed: ctx is NULL");
    if (n > 0 && (!d_first || !d_last || !d_mlen || !d_meta || !d_run_start || !d_run_ref || n_runs < 1 ||
                  n_runs > 0x7fffffff || read_base < 0))
        return fail(ctx, RT_EINVAL, "rt_bin_reads_packed: NULL column or empty run table");
    rt::BinArgs a{};
    a.first = d_first; a.last = d_last; a.mlen = d_mlen; a.meta = d_meta;
    a.run_start = reinterpret_cast<const long long*>(d_run_start);
    a.run_ref = d_run_ref;
    a.n_runs = (int)n_runs;
    a.read_base = read_base;
    return launch_bin(ctx, "rt_bin_reads_packed", a, true, d_cov, n, protocol, weight, d_stats, d_len_counts, stream);
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
    if (ctx->track_touched && ctx->layout != RT_LAYOUT_COMPACT)
        return fail(ctx, RT_ESTATE, "%s: the touched-slot list of the dense layout is kept by rt_bin_reads only", who);
    if (fresh && ctx->layout != RT_LAYOUT_COMPACT) return fail(ctx, RT_ESTATE, "%s: needs the compact layout (rt_set_layout)", who);
    if (fresh && (reinterpret_cast<uintptr_t>(d_cov) & 15)) return fail(ctx, RT_EINVAL, "%s: d_cov must be 16-byte aligned", who);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_blocks == 0) {
        if (fresh) RT_CUDA(ctx, cudaMemsetAsync(d_cov, 0, sizeof(int32_t) * (size_t)ctx->compact_elems, st));
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
    a.cmap = ctx->layout == RT_LAYOUT_COMPACT ? ctx->d_cmap : nullptr;
    a.cbits = ctx->d_cbits;
    a.len_table = ctx->d_len_table;
    a.contig_tab = ctx->d_contig_tab;
    a.n_contig = ctx->n_contig;
    a.pad = ctx->pad;
    a.plane_words = (unsigned)(ctx->plane >> 5);
    a.stats = reinterpret_cast<unsigned long long*>(d_stats);
    a.len_counts = reinterpret_cast<unsigned long long*>(d_len_counts);
    // persistent: a few CTAs per SM; every warp walks blocks with the next one in flight (cp.async.bulk)
    const unsigned grid = (unsigned)std::min<int64_t>((n_blocks + rt::kStreamWarps - 1) / rt::kStreamWarps, (int64_t)ctx->n_sm * RT_STREAM_CTAS_PER_SM);
    if (fresh) {
        // zone boundaries of the blocks (rank of the first position a read of the block can reach), made monotone
        const int64_t tiles = (n_blocks + 1 + rt::kZoneTile - 1) / rt::kZoneTile;
        RT_CUDA(ctx, ctx->zone_buf.reserve(sizeof(unsigned) * (2 * (size_t)(n_blocks + 1) + 4 * (size_t)tiles)));
        RT_CUDA(ctx, ctx->spill_buf.reserve(sizeof(unsigned) * (size_t)n_blocks * RT_STREAM_BLOCK + 16));
        rt::ZoneArgs z{};
        z.hdr = a.hdr;
        z.n_blocks = n_blocks;
        z.bounds = static_cast<unsigned*>(ctx->zone_buf.p);
        z.cmap = ctx->d_cmap;
        z.contig_tab = ctx->d_contig_tab;
        z.n_contig = ctx->n_contig;
        z.pad = ctx->pad;
        z.plane_words = a.plane_words;
        z.delta_plus = ctx->zone_delta_plus;
        z.delta_minus = ctx->zone_delta_minus;
        z.plus_end = ctx->compact_plus_end;
        z.minus_end = ctx->compact_end;
        unsigned long long* d_n_spill = reinterpret_cast<unsigned long long*>(static_cast<char*>(ctx->spill_buf.p));
        unsigned* d_tile_max = z.bounds + 2 * (size_t)(n_blocks + 1);
        unsigned* d_tile_carry = d_tile_max + 2 * (size_t)tiles;
        a.zone_bounds = z.bounds;
        a.zone_carry = d_tile_carry;
        a.zone_tiles = tiles;
        a.spill = reinterpret_cast<unsigned*>(d_n_spill + 2);
        a.n_spill = d_n_spill;
        RT_CUDA(ctx, cudaMemsetAsync(d_n_spill, 0, sizeof(unsigned long long), st));
        // the few guard slots behind the last zone belong to no block
        RT_CUDA(ctx, cudaMemsetAsync(d_cov + ctx->compact_end, 0, sizeof(int32_t) * (size_t)(ctx->compact_elems - ctx->compact_end), st));
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
    RT_CUDA(ctx, ctx->stats_buf.reserve(acc_bytes));
    int64_t* d_stats = static_cast<int64_t*>(ctx->stats_buf.p);
    int64_t* d_len_counts = d_stats + RT_N_STATS;
    for (int s = 0; s < 2; ++s)
        if (!ctx->slot_stream[s]) RT_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking));
    RT_CUDA(ctx, cudaMemsetAsync(d_stats, 0, acc_bytes, ctx->slot_stream[0]));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    // chunks of 16 MB of records alternate between two device slots: copy of one || K1 of the other
    const int64_t chunk = (16 << 20) / (RT_STREAM_BLOCK * 4);
    const size_t rec_bytes = sizeof(uint32_t) * RT_STREAM_BLOCK * (size_t)chunk;
    int slot = 0;
    for (int64_t at = 0; at < n_blocks; at += chunk, slot ^= 1) {
        const int64_t m = std::min(chunk, n_blocks - at);
        RT_CUDA(ctx, ctx->read_slot[slot].reserve(rec_bytes + sizeof(int32_t) * 4 * (size_t)chunk));
        uint32_t* d_rec = static_cast<uint32_t*>(ctx->read_slot[slot].p);
        int32_t* d_hdr = reinterpret_cast<int32_t*>(static_cast<char*>(ctx->read_slot[slot].p) + rec_bytes);
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
    const bool use_stream = sorted_hint && !(ctx->track_touched && ctx->layout != RT_LAYOUT_COMPACT);
    const size_t acc_bytes = sizeof(int64_t) * (RT_N_STATS + RT_LEN_TABLE);
    RT_CUDA(ctx, ctx->stats_buf.reserve(acc_bytes));
    int64_t* d_stats = static_cast<int64_t*>(ctx->stats_buf.p);
    int64_t* d_len_counts = d_stats + RT_N_STATS;
    for (int s = 0; s < 2; ++s)
        if (!ctx->slot_stream[s]) RT_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking));
    RT_CUDA(ctx, cudaMemsetAsync(d_stats, 0, acc_bytes, ctx->slot_stream[0]));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    if (ctx->track_touched && ctx->layout != RT_LAYOUT_COMPACT) {   // one growth up front instead of one per chunk
        int rc = ensure_touched_capacity(ctx, ctx->touched_reserved + n);
        if (rc != RT_OK) return rc;
    }
    // Host columns are the 18 B/read a BAM decoder produces.  With `use_stream` (a coordinate-sorted library) they cross
    // PCIe as a 4 B/read record stream: a few pipeline threads each take the next chunk of the library, delta-code it
    // into their own page-locked staging slot, start the copy on their own stream and launch K1 behind it -- so the
    // coding of some chunks, the copies of others and the kernels of yet others overlap.  A chunk that cannot be coded
    // (positions descend: not sorted after all) is sent as plain columns.
    int64_t pack_chunk_reads = kPackChunkReads;
    if (const char* e = getenv("RT_PACK_CHUNK")) pack_chunk_reads = std::min<int64_t>(kPackChunkReads, std::max(1 << 16, atoi(e)));
    const int64_t chunk = use_stream ? std::min<int64_t>(pack_chunk_reads, std::max<int64_t>(n, 1))
                                      : std::min<int64_t>(kHostChunkReads, std::max<int64_t>(n, 1));
    const int64_t n_chunks = (n + chunk - 1) / chunk;
    // the delta coding is the bottleneck of this call (about 1.5 ns per read and thread): one pipeline per hardware thread
    int64_t want_pipes = std::min<int64_t>(kMaxPipes, (int64_t)std::thread::hardware_concurrency());
    if (const char* e = getenv("RT_PACK_PIPES")) want_pipes = std::min<int64_t>(kMaxPipes, std::max(1, atoi(e)));
    const int n_pipes = use_stream ? (int)std::max<int64_t>(1, std::min<int64_t>(want_pipes, n_chunks)) : 2;
    const bool timing = getenv("RT_HOST_TIMING") != nullptr;
    std::atomic<long long> pack_ns{0}, wait_ns{0}, issue_ns{0};
    const auto t_begin = std::chrono::steady_clock::now();
    // per-slot layout: a chunk's record stream (records, then block headers) or its plain columns, widest column first
    const size_t slot_bytes = std::max((size_t)chunk, (size_t)(use_stream ? kPackChunkReads : 0)) * kReadBytes + 64;
    for (int s = 0; s < n_pipes; ++s) {
        if (!ctx->slot_stream[s]) RT_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking));
        RT_CUDA(ctx, ctx->read_slot[s].reserve(slot_bytes));
        rt_ctx::HostStage& hs = ctx->host_stage[s];
        if (use_stream && !hs.rec) {
            RT_CUDA(ctx, cudaHostAlloc(&hs.rec, sizeof(uint32_t) * RT_STREAM_BLOCK * (size_t)kChunkBlockCap, cudaHostAllocDefault));
            RT_CUDA(ctx, cudaHostAlloc(&hs.hdr, sizeof(int32_t) * 4 * (size_t)kChunkBlockCap, cudaHostAllocDefault));
            RT_CUDA(ctx, cudaEventCreateWithFlags(&hs.copied, cudaEventDisableTiming));
        }
        hs.busy = false;
    }
    std::atomic<int64_t> next_chunk{0};
    std::atomic<int> status{RT_OK};
    std::string first_error;
    auto pipeline = [&](int s) {
        cudaSetDevice(ctx->device);
        char* base = static_cast<char*>(ctx->read_slot[s].p);
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
                                              hs.rec, hs.hdr, kChunkBlockCap);
                if (timing) {
                    wait_ns += std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
                    pack_ns += std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t1).count();
                }
            }
            const auto t2 = std::chrono::steady_clock::now();
            int rc;
            if (blocks >= 0) {
                if (!check(cudaMemcpyAsync(d_rec, hs.rec, sizeof(uint32_t) * RT_STREAM_BLOCK * (size_t)blocks, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
                    !check(cudaMemcpyAsync(d_hdr, hs.hdr, sizeof(int32_t) * 4 * (size_t)blocks, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") ||
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
    {
        std::vector<std::thread> pipes;
        for (int s = 1; s < n_pipes; ++s) pipes.emplace_back(pipeline, s);
        pipeline(0);
        for (auto& th : pipes) th.join();
    }
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

int rt_bin_reads_packed_host(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* h_first, const int32_t* h_last,
                             const uint16_t* h_mlen, const uint8_t* h_meta, int64_t n_runs, const int64_t* h_run_start,
                             const int32_t* h_run_ref, int protocol, int64_t* h_stats, int64_t* h_len_counts) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_bin_reads_packed_host: ctx is NULL");
    if (!h_stats || !h_len_counts) return fail(ctx, RT_EINVAL, "rt_bin_reads_packed_host: NULL output");
    if (n > 0 && (n_runs < 1 || !h_run_start || !h_run_ref || h_run_start[0] != 0 || h_run_start[n_runs] != n))
        return fail(ctx, RT_EINVAL, "rt_bin_reads_packed_host: the run table must cover reads [0, n)");
    DeviceGuard guard(ctx->device);
    const size_t acc_bytes = sizeof(int64_t) * (RT_N_STATS + RT_LEN_TABLE);
    const size_t run_bytes = n > 0 ? sizeof(int64_t) * (size_t)(n_runs + 1) + sizeof(int32_t) * (size_t)n_runs : 0;
    RT_CUDA(ctx, ctx->stats_buf.reserve(acc_bytes + run_bytes + 16));
    int64_t* d_stats = static_cast<int64_t*>(ctx->stats_buf.p);
    int64_t* d_len_counts = d_stats + RT_N_STATS;
    int64_t* d_run_start = d_len_counts + RT_LEN_TABLE;
    int32_t* d_run_ref = reinterpret_cast<int32_t*>(d_run_start + (n > 0 ? n_runs + 1 : 0));
    for (int s = 0; s < 2; ++s)
        if (!ctx->slot_stream[s]) RT_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking));
    RT_CUDA(ctx, cudaMemsetAsync(d_stats, 0, acc_bytes, ctx->slot_stream[0]));
    if (n > 0) {
        RT_CUDA(ctx, cudaMemcpyAsync(d_run_start, h_run_start, sizeof(int64_t) * (size_t)(n_runs + 1), cudaMemcpyHostToDevice, ctx->slot_stream[0]));
        RT_CUDA(ctx, cudaMemcpyAsync(d_run_ref, h_run_ref, sizeof(int32_t) * (size_t)n_runs, cudaMemcpyHostToDevice, ctx->slot_stream[0]));
    }
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    if (ctx->track_touched && ctx->layout != RT_LAYOUT_COMPACT) {
        int rc = ensure_touched_capacity(ctx, ctx->touched_reserved + n);
        if (rc != RT_OK) return rc;
    }
    const int64_t chunk = std::min<int64_t>(kHostChunkReads, std::max<int64_t>(n, 1));
    const size_t slot_bytes = (size_t)chunk * kPackedReadBytes + 64;
    int slot = 0;
    for (int64_t at = 0; at < n; at += chunk, slot ^= 1) {
        const int64_t m = std::min(chunk, n - at);
        RT_CUDA(ctx, ctx->read_slot[slot].reserve(slot_bytes));
        char* base = static_cast<char*>(ctx->read_slot[slot].p);
        int32_t* d_first = reinterpret_cast<int32_t*>(base);
        int32_t* d_last = d_first + chunk;
        uint16_t* d_mlen = reinterpret_cast<uint16_t*>(d_last + chunk);
        uint8_t* d_meta = reinterpret_cast<uint8_t*>(d_mlen + chunk);
        cudaStream_t st = ctx->slot_stream[slot];   // stream order protects the slot's previous use
        RT_CUDA(ctx, cudaMemcpyAsync(d_first, h_first + at, 4 * m, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(d_last, h_last + at, 4 * m, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(d_mlen, h_mlen + at, 2 * m, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(d_meta, h_meta + at, m, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += (int64_t)m * (int64_t)kPackedReadBytes;
        int rc = rt_bin_reads_packed(ctx, d_cov, m, d_first, d_last, d_mlen, d_meta, at, n_runs, d_run_start, d_run_ref,
                                     protocol, 1, d_stats, d_len_counts, st);
        if (rc != RT_OK) return rc;
    }
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[1]));
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
    ctx->bytes_prefix.assign((size_t)n_orf + 1, 0);
    ctx->nt_prefix.assign((size_t)n_orf + 1, 0);
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
        ctx->nt_prefix[o + 1] = ctx->nt_prefix[o] + L;
        ctx->bytes_prefix[o + 1] = ctx->bytes_prefix[o] + 4 * L + 8 * (e1 - e0) + 42;
    }
    cudaFree(ctx->d_orf_desc);
    cudaFree(ctx->d_orf_len);
    cudaFree(ctx->d_exon_entries);
    ctx->d_orf_desc = ctx->d_exon_entries = nullptr;
    ctx->d_orf_len = nullptr;
    ctx->n_orf = 0;
    for (auto& p : ctx->plans) free_plan(p);
    ctx->plans.clear();
    cudaFree(ctx->d_atoms);
    cudaFree(ctx->d_summaries);
    cudaFree(ctx->d_atom_nonzero);
    ctx->d_atom_nonzero = nullptr;
    cudaFree(ctx->d_cmap);
    cudaFree(ctx->d_cbits);
    cudaFree(ctx->d_atoms_c);
    cudaFree(ctx->d_exon_entries_c);
    ctx->d_cmap = nullptr;
    ctx->d_cbits = nullptr;
    ctx->d_atoms_c = ctx->d_exon_entries_c = nullptr;
    ctx->layout = RT_LAYOUT_DENSE;
    ctx->compact_elems = 0;
    ctx->d_atoms = nullptr;
    ctx->d_summaries = nullptr;
    ctx->n_atoms = 0;
    {
        std::vector<int32_t> lens((size_t)n_orf);
        for (int64_t o = 0; o < n_orf; ++o) lens[o] = (int32_t)(ctx->nt_prefix[o + 1] - ctx->nt_prefix[o]);
        RT_CUDA(ctx, cudaMalloc(&ctx->d_orf_len, sizeof(int32_t) * std::max<size_t>(1, lens.size())));
        if (!lens.empty())
            RT_CUDA(ctx, cudaMemcpy(ctx->d_orf_len, lens.data(), sizeof(int32_t) * lens.size(), cudaMemcpyHostToDevice));
    }
    RT_CUDA(ctx, cudaMalloc(&ctx->d_orf_desc, sizeof(uint64_t) * std::max<size_t>(1, desc.size())));
    RT_CUDA(ctx, cudaMalloc(&ctx->d_exon_entries, sizeof(uint64_t) * std::max<size_t>(1, entries.size())));
    if (!desc.empty())
        RT_CUDA(ctx, cudaMemcpy(ctx->d_orf_desc, desc.data(), sizeof(uint64_t) * desc.size(), cudaMemcpyHostToDevice));
    if (!entries.empty())
        RT_CUDA(ctx, cudaMemcpy(ctx->d_exon_entries, entries.data(), sizeof(uint64_t) * entries.size(),
                                cudaMemcpyHostToDevice));
    {
        const auto t_atoms = std::chrono::steady_clock::now();
        int rc = build_atoms(ctx, desc, entries);
        if (getenv("RT_HOST_TIMING"))
            fprintf(stderr, "rt_set_index: build_atoms %.1f ms (%zu ORFs, %zu exon entries, %zu atoms)\n",
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_atoms).count(), desc.size(), entries.size(),
                    ctx->h_atoms.size());
        if (rc != RT_OK) return rc;
    }
    ctx->n_orf = n_orf;
    return RT_OK;
}

int64_t rt_index_orfs(const rt_ctx* ctx) { return ctx ? ctx->n_orf : 0; }

int64_t rt_index_score_bytes(const rt_ctx* ctx, int64_t lo, int64_t hi) {
    if (!ctx || lo < 0 || hi > ctx->n_orf || lo > hi) return -1;
    return ctx->bytes_prefix[hi] - ctx->bytes_prefix[lo];
}

int64_t rt_index_total_nt(const rt_ctx* ctx, int64_t lo, int64_t hi) {
    if (!ctx || lo < 0 || hi > ctx->n_orf || lo > hi) return -1;
    return ctx->nt_prefix[hi] - ctx->nt_prefix[lo];
}

int rt_shard_bounds(const rt_ctx* ctx, int n_shards, int64_t* h_bounds) {
    if (!ctx || n_shards < 1 || !h_bounds) return RT_EINVAL;
    const int64_t total = ctx->bytes_prefix.empty() ? 0 : ctx->bytes_prefix.back();
    h_bounds[0] = 0;
    for (int s = 1; s < n_shards; ++s) {
        const int64_t target = (int64_t)((__int128)total * s / n_shards);
        auto it = std::lower_bound(ctx->bytes_prefix.begin(), ctx->bytes_prefix.end(), target);
        h_bounds[s] = std::max<int64_t>(h_bounds[s - 1], it - ctx->bytes_prefix.begin());
        if (h_bounds[s] > ctx->n_orf) h_bounds[s] = ctx->n_orf;
    }
    h_bounds[n_shards] = ctx->n_orf;
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
        std::vector<uint8_t> used((size_t)ctx->n_atoms, 0);
        for (int64_t o = lo; o < hi; ++o) {
            const uint64_t d = ctx->h_orf_refs_desc[o];
            const uint64_t b = d & rt::kBeginMask, c = (d >> 40) & rt::kMaxEntriesPerOrf;
            for (uint64_t k = b; k < b + c; ++k)
                if (ctx->h_ref_atom[k] != 0xffffffffu) used[ctx->h_ref_atom[k]] = 1;
        }
        std::vector<int32_t>& alist = ph.alist;
        for (int64_t a = 0; a < ctx->n_atoms; ++a)
            if (used[a]) alist.push_back((int32_t)a);
        {   // passes of the streamed phase A: consecutive atom ids are adjacent in the compact buffer
            std::vector<rt::PassDesc>& passes = ph.passes;
            const uint64_t* ac = ctx->h_atoms_c.data();
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
                return (ctx->h_atoms[x] & rt::kLenMask) > (ctx->h_atoms[y] & rt::kLenMask);
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
        refs.reserve((size_t)(ctx->h_ref_ent.size() / std::max<int64_t>(1, ctx->n_orf) * n * 3 / 4 + 64));
        const rt::RefRec pad_rec{0xffffffffu, 0u, 0u, -1};
        int& n_long = ph.n_long_b;
        auto pad_group = [&]() {
            while (refs.size() % 32) refs.push_back(pad_rec);
            warps.resize(refs.size() / 32, rt::RefWarp{-1, 0, -1, 0});
        };
        auto desc_of = [&](int64_t o, uint64_t& rb, uint64_t& cnt, uint32_t& rev) {
            const uint64_t d = ctx->h_orf_refs_desc[o];
            rb = d & rt::kBeginMask;
            cnt = (d >> 40) & (uint64_t)rt::kMaxEntriesPerOrf;
            rev = (uint32_t)(d >> 63);
        };
        // hash of a reference list, powers counted from its END, so that the hash of a suffix of a parent equals the
        // hash of the child that is that suffix
        const uint64_t kB = 0x9E3779B97F4A7C15ull;
        auto elem = [&](uint64_t k) {
            uint64_t x = ((uint64_t)ctx->h_ref_atom[k] << 25) ^ (ctx->h_ref_ent[k] & rt::kLenMask);
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
        auto refs_of = [&](int64_t o) { return (ctx->h_orf_refs_desc[o] >> 40) & (uint64_t)rt::kMaxEntriesPerOrf; };
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
                    if ((ctx->h_ref_ent[crb] & rt::kLenMask) < 2) continue;
                    bool same = true;
                    for (uint64_t j = 0; j < ccnt && same; ++j)
                        same = ctx->h_ref_atom[crb + j] == ctx->h_ref_atom[rb + k + j] &&
                               (ctx->h_ref_ent[crb + j] & rt::kLenMask) == (ctx->h_ref_ent[rb + k + j] & rt::kLenMask);
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
            const uint64_t L = (uint64_t)(ctx->nt_prefix[o + 1] - ctx->nt_prefix[o]);
            auto flags_of = [&](uint64_t len, uint64_t l_mod3) -> uint32_t {
                return ((uint32_t)(P % 3) << rt::kRefPmod3Shift) | (P >= 1 ? rt::kRefPge1 : 0u) | (P >= 2 ? rt::kRefPge2 : 0u) |
                       (P + len == L ? rt::kRefLast : 0u) | ((uint32_t)l_mod3 << rt::kRefLmod3Shift) | (rev ? rt::kRefRev : 0u);
            };
            for (uint64_t k = 0; k < cnt; ++k) {
                const uint32_t len = (uint32_t)(ctx->h_ref_ent[rb + k] & rt::kLenMask);
                // L mod 3 of the ORF that starts on this slot; a long ORF carries its own on every slot (its last
                // group applies the trailing partial codon itself)
                const uint64_t lm3 = (k == 0 || cnt > 32) ? L % 3 : 0;
                refs.push_back({ctx->h_ref_atom[rb + k], len | flags_of(len, lm3), (uint32_t)((len + P) % 3) | (k == 0 ? rt::kRefFamilyHead : 0u),
                                k == 0 ? (int32_t)o : -2});
                P += len;
            }
            if (cnt == 0) refs.push_back({0xffffffffu, flags_of(0, L % 3), rt::kRefFamilyHead, (int32_t)o});   // an ORF without intervals still gets its row
            for (const auto& ch : children[o - lo]) {
                rt::RefRec& r = refs[first_slot + (size_t)ch.first];
                const uint64_t Lc = (uint64_t)(ctx->nt_prefix[ch.second + 1] - ctx->nt_prefix[ch.second]);
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
    if (ctx->plans.size() >= 24) {   // bounded cache (rt_score_host keeps four part plans per range it is asked for)
        free_plan(ctx->plans.front());
        ctx->plans.erase(ctx->plans.begin());
    }
    rt_ctx::ScorePlan p;
    p.lo = lo;
    p.hi = hi;
    RT_CUDA(ctx, cudaMalloc(&p.d_fallback, sizeof(int32_t) * std::max<int64_t>(1, n)));
    p.n_passes = (int64_t)ph.passes.size();
    RT_CUDA(ctx, cudaMalloc(&p.d_passes, sizeof(rt::PassDesc) * std::max<size_t>(1, ph.passes.size())));
    if (!ph.passes.empty())
        RT_CUDA(ctx, cudaMemcpy(p.d_passes, ph.passes.data(), sizeof(rt::PassDesc) * ph.passes.size(), cudaMemcpyHostToDevice));
    p.n_atom_list = (int64_t)ph.alist.size();
    RT_CUDA(ctx, cudaMalloc(&p.d_atom_list, sizeof(int32_t) * std::max<size_t>(1, ph.alist.size())));
    if (!ph.alist.empty())
        RT_CUDA(ctx, cudaMemcpy(p.d_atom_list, ph.alist.data(), sizeof(int32_t) * ph.alist.size(), cudaMemcpyHostToDevice));
    const std::vector<rt::RefRec>& refs = ph.refs;
    const std::vector<rt::RefWarp>& warps = ph.warps;
    p.n_ref_warps = (int64_t)warps.size();
    RT_CUDA(ctx, cudaMalloc(&p.d_refs, sizeof(rt::RefRec) * std::max<size_t>(1, refs.size())));
    RT_CUDA(ctx, cudaMalloc(&p.d_ref_warps, sizeof(rt::RefWarp) * std::max<size_t>(1, warps.size())));
    if (!refs.empty()) {
        RT_CUDA(ctx, cudaMemcpy(p.d_refs, refs.data(), sizeof(rt::RefRec) * refs.size(), cudaMemcpyHostToDevice));
        RT_CUDA(ctx, cudaMemcpy(p.d_ref_warps, warps.data(), sizeof(rt::RefWarp) * warps.size(), cudaMemcpyHostToDevice));
    }
    std::vector<rt::LongAcc> acc((size_t)std::max(1, ph.n_long_b));
    memset(acc.data(), 0, sizeof(rt::LongAcc) * acc.size());
    for (auto& a : acc) a.mn = 0xffffffffu;
    RT_CUDA(ctx, cudaMalloc(&p.d_long_acc, sizeof(rt::LongAcc) * acc.size()));
    RT_CUDA(ctx, cudaMemcpy(p.d_long_acc, acc.data(), sizeof(rt::LongAcc) * acc.size(), cudaMemcpyHostToDevice));
    ctx->plans.push_back(p);
    *out = &ctx->plans.back();
    return RT_OK;
}

int get_plan(rt_ctx* ctx, int64_t lo, int64_t hi, rt_ctx::ScorePlan** out) {
    for (auto& p : ctx->plans)
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
        for (auto& p : ctx->plans) cached = cached || (p.lo == a && p.hi == b);
        if (!cached) {
            todo.emplace_back();
            todo.back().lo = a;
            todo.back().hi = b;
        }
    }
    if (todo.size() < 2) return RT_OK;           // get_plan does a single one just as well
    {
        std::vector<std::thread> pool;
        for (size_t k = 1; k < todo.size(); ++k)
            pool.emplace_back([ctx, &todo, k]() { build_plan_host(ctx, todo[k].lo, todo[k].hi, todo[k]); });
        build_plan_host(ctx, todo[0].lo, todo[0].hi, todo[0]);
        for (auto& th : pool) th.join();
    }
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
    if (orf_lo < 0 || orf_hi > ctx->n_orf || orf_lo > orf_hi)
        return fail(ctx, RT_EINVAL, "rt_score: ORF range [%lld,%lld) outside the index [0,%lld)", (long long)orf_lo,
                    (long long)orf_hi, (long long)ctx->n_orf);
    if (orf_lo == orf_hi) return RT_OK;
    if (!d_out->score || !d_out->valid || !d_out->count || !d_out->length)
        return fail(ctx, RT_EINVAL, "rt_score: score/valid/count/length columns are required");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    rt_ctx::ScorePlan* plan = nullptr;
    int rc = get_plan(ctx, orf_lo, orf_hi, &plan);
    if (rc != RT_OK) return rc;
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_work_counter, 0, 4 * sizeof(unsigned long long), st));
    rt::ScoreArgs a;
    a.cov = d_cov;
    a.orf_desc = ctx->d_orf_desc;
    const bool compact = ctx->layout == RT_LAYOUT_COMPACT;
    a.exon_entries = compact ? ctx->d_exon_entries_c : ctx->d_exon_entries;
    a.orf_len = ctx->d_orf_len;
    a.orf_lo = orf_lo;
    a.n_fallback = reinterpret_cast<unsigned*>(ctx->d_work_counter + 3);
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
            pa.atoms = ctx->d_atoms_c;
            pa.passes = plan->d_passes;
            pa.n_passes = (unsigned)plan->n_passes;
            pa.out = ctx->d_summaries;
            pa.nonzero = ctx->d_atom_nonzero;
            const size_t smem = rt::kUvEntries * sizeof(double2) + (size_t)rt::kPassWarps * rt::kPassStages * rt::kPassStageBytes;
            const auto kern = want_min ? rt::atom_pass_kernel<true> : rt::atom_pass_kernel<false>;
            RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const int64_t want = (plan->n_passes + rt::kPassWarps - 1) / rt::kPassWarps;
            const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, ctx->n_sm));
            kern<<<grid, rt::kPassWarps * 32, smem, st>>>(pa);
        } else {
            rt::AtomArgs aa;
            aa.cov = d_cov;
            aa.atoms = ctx->d_atoms;
            aa.list = plan->d_atom_list;
            aa.n_list = plan->n_atom_list;
            aa.work_counter = ctx->d_work_counter + 0;
            aa.out = ctx->d_summaries;
            aa.nonzero = ctx->d_atom_nonzero;
            const auto kern = want_min ? rt::atom_summary_kernel<true> : rt::atom_summary_kernel<false>;
            const int g = 32 / rt::kAtomLPO;
            kern<<<persistent_grid(ctx, kern, (plan->n_atom_list + g - 1) / g), threads, 0, st>>>(aa);
        }
        ctx->launches++;
    }
    // phase B: the ORFs of every family from the summaries of their atoms
    rt::RefComposeArgs ra;
    ra.refs = plan->d_refs;
    ra.warps = plan->d_ref_warps;
    ra.n_warps = plan->n_ref_warps;
    ra.summaries = ctx->d_summaries;
    ra.atom_nonzero = ctx->d_atom_nonzero;
    ra.uv_table = ctx->d_uv_table;
    ra.want_min = want_min ? 1 : 0;
    ra.orf_len = ctx->d_orf_len;
    ra.orf_lo = orf_lo;
    ra.fallback = plan->d_fallback;
    ra.n_fallback = a.n_fallback;
    ra.long_acc = plan->d_long_acc;
    ra.prm = *params;
    ra.out = *d_out;
    if (ra.n_warps > 0) {
        if (want_min) rt::compose_refs_kernel<true><<<(unsigned)((ra.n_warps + 7) / 8), 256, 0, st>>>(ra);
        else rt::compose_refs_kernel<false><<<(unsigned)((ra.n_warps + 7) / 8), 256, 0, st>>>(ra);
    }
    ctx->launches++;
    // ORFs holding counts >= 2^20: redone by the generic kernel (normally none)
    a.list = plan->d_fallback;
    a.n_list = 0;
    a.n_list_dev = a.n_fallback;
    a.work_counter = ctx->d_work_counter + 2;
    rt::score_orfs_kernel<<<(unsigned)ctx->n_sm, threads, 0, st>>>(a);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

int rt_score_host(rt_ctx* ctx, const int32_t* d_cov, int64_t orf_lo, int64_t orf_hi, const rt_score_params* params,
                  const rt_score_out* h_out) {
    if (!ctx) return fail(nullptr, RT_EINVAL, "rt_score_host: ctx is NULL");
    if (!h_out || !params) return fail(ctx, RT_EINVAL, "rt_score_host: NULL argument");
    if (orf_lo < 0 || orf_hi > ctx->n_orf || orf_lo > orf_hi) return fail(ctx, RT_EINVAL, "rt_score_host: bad ORF range");
    const int64_t n = orf_hi - orf_lo;
    if (n == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    // one scratch allocation, 8-byte columns first
    const size_t bytes = (size_t)n * (8 + 8 + 24 + 4 + 4 + 4 + 12 + 1) + 256;
    RT_CUDA(ctx, ctx->score_buf.reserve(bytes));
    char* p = static_cast<char*>(ctx->score_buf.p);
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
    const int64_t* bp = ctx->bytes_prefix.data();
    for (int i = 1; i < n_parts; ++i) {
        const int64_t target = bp[orf_lo] + (bp[orf_hi] - bp[orf_lo]) * i / n_parts;
        cut[(size_t)i] = std::max<int64_t>(cut[(size_t)i - 1], std::lower_bound(bp + orf_lo, bp + orf_hi, target) - bp);
    }
    if (n_parts > 1) {                 // the parts' plans that are not cached yet: host halves built side by side
        const int rc = prebuild_plans(ctx, cut);
        if (rc != RT_OK) return rc;
    }
    if (!ctx->slot_stream[0]) RT_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slot_stream[0], cudaStreamNonBlocking));
    cudaStream_t copy = n_parts > 1 ? ctx->slot_stream[0] : nullptr;
    if (n_parts > 1 && !ctx->ev_scored) RT_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_scored, cudaEventDisableTiming));
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
    double* d_vals = static_cast<double*>(ctx->score_buf.p);
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
    if (ctx->n_orf == 0 && n_sel > 0) return fail(ctx, RT_ESTATE, "rt_gather_profiles: no index");
    if (n_sel == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    rt::GatherArgs a;
    a.cov = d_cov;
    a.orf_desc = ctx->d_orf_desc;
    a.exon_entries = ctx->layout == RT_LAYOUT_COMPACT ? ctx->d_exon_entries_c : ctx->d_exon_entries;
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
    if (ctx->n_orf == 0 || !ctx->d_atoms_c) return fail(ctx, RT_ESTATE, "rt_compact_from_dense: call rt_set_index first");
    if (ctx->n_atoms == 0) return RT_OK;
    DeviceGuard guard(ctx->device);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((ctx->n_atoms + 7) / 8, (int64_t)ctx->n_sm * 16));
    rt::compact_from_dense_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ctx->d_atoms, ctx->d_atoms_c, ctx->n_atoms, d_dense, d_compact);
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
    if (ctx->layout != RT_LAYOUT_DENSE)
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
    DevBuf vals, idx, outb, scratch;
    auto cleanup = [&]() { vals.release(); idx.release(); outb.release(); scratch.release(); };
    cudaError_t e = vals.reserve(sizeof(double) * (size_t)n);
    if (e == cudaSuccess) e = idx.reserve(sizeof(int64_t) * (size_t)(n_sel * reps));
    if (e == cudaSuccess) e = outb.reserve(sizeof(double) * (size_t)reps);
    if (e == cudaSuccess && !in_smem) e = scratch.reserve(key_bytes * (size_t)reps);
    if (e == cudaSuccess) e = cudaMemcpy(vals.p, h_values, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(idx.p, h_idx, sizeof(int64_t) * (size_t)(n_sel * reps), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && in_smem)
        e = cudaFuncSetAttribute(rt::bootstrap_median_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)key_bytes);
    if (e == cudaSuccess) {
        rt::bootstrap_median_kernel<<<(unsigned)reps, 256, in_smem ? key_bytes : 0>>>(
            static_cast<const double*>(vals.p), static_cast<const long long*>(idx.p), n_sel, reps,
            static_cast<unsigned long long*>(scratch.p), in_smem ? 1 : 0, static_cast<double*>(outb.p));
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(h_out, outb.p, sizeof(double) * (size_t)reps, cudaMemcpyDeviceToHost);
    cleanup();
    if (e != cudaSuccess) return fail(ctx, e == cudaErrorMemoryAllocation ? RT_ENOMEM : RT_ECUDA, "rt_bootstrap_medians: %s", cudaGetErrorString(e));
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------ prepare-orfs
namespace {
enum OrfBuf { kCodes, kExSrc, kExDst, kExLen, kExRev, kTxSeq, kTxCds, kTxExon, kTxRev, kExStart, kExEnd, kExBefore, kSeq,
              kTxRows, kRowOff, kRowTx, kRowStart, kRowStop, kRowType, kRowCodon, kIvCount, kIvOff, kIvStart, kIvEnd,
              kClaim, kOrfBufs };
static_assert(kOrfBufs <= 32, "rt_ctx::orf_buf is too small");
}  // namespace

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
    DevBuf* B = ctx->orf_buf;
    auto reserve = [&](int k, size_t bytes) { return B[k].reserve(std::max<size_t>(bytes, 16)); };
    RT_CUDA(ctx, reserve(kCodes, (size_t)q->n_codes));
    RT_CUDA(ctx, reserve(kExSrc, 8 * (size_t)n_ex));
    RT_CUDA(ctx, reserve(kExDst, 8 * (size_t)n_ex));
    RT_CUDA(ctx, reserve(kExLen, 4 * (size_t)n_ex));
    RT_CUDA(ctx, reserve(kExRev, (size_t)n_ex));
    RT_CUDA(ctx, reserve(kTxSeq, 8 * (size_t)(n_tx + 1)));
    RT_CUDA(ctx, reserve(kTxCds, 8 * (size_t)n_tx));
    RT_CUDA(ctx, reserve(kTxExon, 8 * (size_t)(n_tx + 1)));
    RT_CUDA(ctx, reserve(kTxRev, (size_t)n_tx));
    RT_CUDA(ctx, reserve(kExStart, 4 * (size_t)n_ex));
    RT_CUDA(ctx, reserve(kExEnd, 4 * (size_t)n_ex));
    RT_CUDA(ctx, reserve(kExBefore, 4 * (size_t)n_ex));
    RT_CUDA(ctx, reserve(kSeq, (size_t)n_seq + 4));
    RT_CUDA(ctx, reserve(kTxRows, 8 * (size_t)n_tx));
    RT_CUDA(ctx, reserve(kRowOff, 8 * (size_t)n_tx));
    RT_CUDA(ctx, reserve(kClaim, 4));
    cudaStream_t st = 0;
    cudaEvent_t ev[RT_ORF_STAGES + 1];
    for (auto& e : ev) RT_CUDA(ctx, cudaEventCreate(&e));
    struct EvGuard { cudaEvent_t* ev; ~EvGuard() { for (int i = 0; i <= RT_ORF_STAGES; ++i) cudaEventDestroy(ev[i]); } } evg{ev};
    auto up = [&](int k, const void* src, size_t bytes) { return bytes ? cudaMemcpyAsync(B[k].p, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess; };
    RT_CUDA(ctx, cudaEventRecord(ev[0], st));
    // 1. upload: contig codes, the transcript and exon tables
    RT_CUDA(ctx, up(kCodes, q->codes, (size_t)q->n_codes));
    RT_CUDA(ctx, up(kExSrc, ex_src.data(), 8 * (size_t)n_ex));
    RT_CUDA(ctx, up(kExDst, ex_dst.data(), 8 * (size_t)n_ex));
    RT_CUDA(ctx, up(kExLen, ex_len.data(), 4 * (size_t)n_ex));
    RT_CUDA(ctx, up(kExRev, ex_rev.data(), (size_t)n_ex));
    RT_CUDA(ctx, up(kTxSeq, tx_seq.data(), 8 * (size_t)(n_tx + 1)));
    RT_CUDA(ctx, up(kTxCds, q->tx_cds, 8 * (size_t)n_tx));
    RT_CUDA(ctx, up(kTxExon, q->exon_ptr, 8 * (size_t)(n_tx + 1)));
    RT_CUDA(ctx, up(kTxRev, q->tx_strand, (size_t)n_tx));
    RT_CUDA(ctx, up(kExStart, q->exon_start, 4 * (size_t)n_ex));
    RT_CUDA(ctx, up(kExEnd, q->exon_end, 4 * (size_t)n_ex));
    RT_CUDA(ctx, up(kExBefore, ex_before.data(), 4 * (size_t)n_ex));
    RT_CUDA(ctx, cudaEventRecord(ev[1], st));
    const unsigned big = (unsigned)std::max(1, ctx->n_sm * 8);
    // 2. spliced, oriented sequences
    if (n_ex) {
        rt::orf_splice_kernel<<<(unsigned)std::min<int64_t>((n_ex + 7) / 8, big), 256, 0, st>>>(
            (const uint8_t*)B[kCodes].p, (const long long*)B[kExSrc].p, (const long long*)B[kExDst].p, (const int*)B[kExLen].p,
            (const uint8_t*)B[kExRev].p, n_ex, (uint8_t*)B[kSeq].p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(ev[2], st));
    // 3. rows per transcript
    rt::OrfArgs A{(const long long*)B[kTxSeq].p, (const int2*)B[kTxCds].p, (uint8_t*)B[kSeq].p, q->start_mask, q->stop_mask,
                  (int)n_tx, q->min_orf_length, q->longest ? 1 : 0, (unsigned*)B[kClaim].p};
    const unsigned walk_grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n_tx + 7) / 8, big));
    if (n_tx) {
        RT_CUDA(ctx, cudaMemsetAsync(B[kClaim].p, 0, 4, st));
        rt::orf_walk_kernel<false><<<walk_grid, 256, 0, st>>>(A, (long long*)B[kTxRows].p, nullptr, nullptr, nullptr, nullptr,
                                                                nullptr, nullptr);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(ev[3], st));
    // 4. exclusive scan of the row counts (host: one int64 per transcript)
    std::vector<int64_t> cnt((size_t)n_tx), off((size_t)n_tx + 1, 0);
    if (n_tx) RT_CUDA(ctx, cudaMemcpyAsync(cnt.data(), B[kTxRows].p, 8 * (size_t)n_tx, cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    for (int64_t t = 0; t < n_tx; ++t) off[(size_t)t + 1] = off[(size_t)t] + cnt[(size_t)t];
    const int64_t rows = off[(size_t)n_tx];
    RT_CUDA(ctx, reserve(kRowTx, 4 * (size_t)rows));
    RT_CUDA(ctx, reserve(kRowStart, 4 * (size_t)rows));
    RT_CUDA(ctx, reserve(kRowStop, 4 * (size_t)rows));
    RT_CUDA(ctx, reserve(kRowType, (size_t)rows));
    RT_CUDA(ctx, reserve(kRowCodon, (size_t)rows));
    RT_CUDA(ctx, reserve(kIvCount, 8 * (size_t)rows));
    RT_CUDA(ctx, reserve(kIvOff, 8 * (size_t)rows));
    RT_CUDA(ctx, up(kRowOff, off.data(), 8 * (size_t)n_tx));
    RT_CUDA(ctx, cudaEventRecord(ev[4], st));
    // 5. the rows
    if (rows) {
        RT_CUDA(ctx, cudaMemsetAsync(B[kClaim].p, 0, 4, st));
        rt::orf_walk_kernel<true><<<walk_grid, 256, 0, st>>>(A, (long long*)B[kTxRows].p, (const long long*)B[kRowOff].p,
                                                               (int*)B[kRowTx].p, (int*)B[kRowStart].p, (int*)B[kRowStop].p,
                                                               (uint8_t*)B[kRowType].p, (uint8_t*)B[kRowCodon].p);
        ctx->launches++;
        RT_CUDA(ctx, cudaGetLastError());
    }
    RT_CUDA(ctx, cudaEventRecord(ev[5], st));
    // 6. intervals per row, their exclusive scan (host)
    const unsigned row_grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((rows + 255) / 256, (int64_t)big * 4));
    auto intervals = [&](bool count) {
        if (count)
            rt::orf_interval_kernel<true><<<row_grid, 256, 0, st>>>(
                rows, (const int*)B[kRowTx].p, (const int*)B[kRowStart].p, (const int*)B[kRowStop].p, (const long long*)B[kTxExon].p,
                (const long long*)B[kTxSeq].p, (const uint8_t*)B[kTxRev].p, (const int*)B[kExStart].p, (const int*)B[kExEnd].p,
                (const int*)B[kExBefore].p, (long long*)B[kIvCount].p, nullptr, nullptr, nullptr);
        else
            rt::orf_interval_kernel<false><<<row_grid, 256, 0, st>>>(
                rows, (const int*)B[kRowTx].p, (const int*)B[kRowStart].p, (const int*)B[kRowStop].p, (const long long*)B[kTxExon].p,
                (const long long*)B[kTxSeq].p, (const uint8_t*)B[kTxRev].p, (const int*)B[kExStart].p, (const int*)B[kExEnd].p,
                (const int*)B[kExBefore].p, nullptr, (const long long*)B[kIvOff].p, (int*)B[kIvStart].p, (int*)B[kIvEnd].p);
        ctx->launches++;
        return cudaGetLastError();
    };
    std::vector<int64_t>& ivp = ctx->orf_iv_ptr;
    ivp.assign((size_t)rows + 1, 0);
    if (rows) {
        RT_CUDA(ctx, intervals(true));
        std::vector<int64_t> ivc((size_t)rows);
        RT_CUDA(ctx, cudaMemcpyAsync(ivc.data(), B[kIvCount].p, 8 * (size_t)rows, cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));
        for (int64_t r = 0; r < rows; ++r) ivp[(size_t)r + 1] = ivp[(size_t)r] + ivc[(size_t)r];
    }
    const int64_t ivs = ivp.back();
    RT_CUDA(ctx, reserve(kIvStart, 4 * (size_t)ivs));
    RT_CUDA(ctx, reserve(kIvEnd, 4 * (size_t)ivs));
    RT_CUDA(ctx, up(kIvOff, ivp.data(), 8 * (size_t)rows));
    RT_CUDA(ctx, cudaEventRecord(ev[6], st));
    // 7. the intervals
    if (rows) RT_CUDA(ctx, intervals(false));
    RT_CUDA(ctx, cudaEventRecord(ev[7], st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    if (stage_ms)
        for (int i = 0; i < RT_ORF_STAGES; ++i) RT_CUDA(ctx, cudaEventElapsedTime(&stage_ms[i], ev[i], ev[i + 1]));
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
    DevBuf* B = ctx->orf_buf;
    cudaStream_t st = 0;
    auto down = [&](void* dst, int k, size_t bytes) { return dst && bytes ? cudaMemcpyAsync(dst, B[k].p, bytes, cudaMemcpyDeviceToHost, st) : cudaSuccess; };
    RT_CUDA(ctx, down(row_tx, kRowTx, 4 * (size_t)rows));
    RT_CUDA(ctx, down(row_start, kRowStart, 4 * (size_t)rows));
    RT_CUDA(ctx, down(row_stop, kRowStop, 4 * (size_t)rows));
    RT_CUDA(ctx, down(row_type, kRowType, (size_t)rows));
    RT_CUDA(ctx, down(row_codon, kRowCodon, (size_t)rows));
    RT_CUDA(ctx, down(iv_start, kIvStart, 4 * (size_t)ivs));
    RT_CUDA(ctx, down(iv_end, kIvEnd, 4 * (size_t)ivs));
    if (iv_ptr) memcpy(iv_ptr, ctx->orf_iv_ptr.data(), 8 * (size_t)(rows + 1));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    return RT_OK;
}

}  // extern "C"
