// rt_kernels.cuh -- sm_100a kernels of the detect-orfs scoring path.
//
//   K1 bin_stream_kernel      bam.py:71-137 + detect_orfs.py:54-83 on the 4 B/read record stream of a coordinate-sorted
//                             library (persistent, per-warp cp.async.bulk rings; <Zoned>: every block writes its zone
//                             of the compact buffer before it adds into it), with zone_bounds / zone_carry / zone_spill
//      bin_psites_kernel      the same loop on the decoder's columns (any read order, dense planes with the sparse clear)
//   K2+K3 atom_pass_kernel    phase A: detect_orfs.py:134-203 + statistics.py:48-115 per atom of the exon union,
//                             streamed by cp.async.bulk (compact layout); atom_summary_kernel for the dense planes
//      compose_refs_kernel    phase B: per-ORF columns from the atom summaries (families of nested ORFs, suffix scan),
//                             detect_orfs.py:274-299 + common.py:164-180
//      score_orfs_kernel      the whole per-ORF loop in one kernel: fallback for counts >= 2^20
//   K4 gather_profiles_kernel detect_orfs.py:134-203 for the reported ORFs (:322)
//
// All "file:line" citations are relative to the reference tree.
#pragma once
#include <cuda_runtime.h>
#include <type_traits>
#include <stdint.h>

#include "ribotricer_b200.h"

namespace rt {

constexpr unsigned kFull = 0xffffffffu;

// ---- device-resident index encoding ------------------------------------------------------
// exon entry : (slot_offset << 24) | len      slot_offset relative to d_cov (strand plane
//              included), len in [1, 2^24); slot_offset == kZeroOff means "reads as zeros"
//              (unknown contig / strand, or the part of an exon outside the padded contig).
// ORF desc   : exon_begin (40 bits) | n_entries (23 bits) << 40 | reverse << 63
constexpr int kLenBits = 24;
constexpr uint64_t kLenMask = (1ull << kLenBits) - 1;
constexpr uint64_t kZeroOff = (1ull << 40) - 1;
constexpr uint64_t kBeginMask = (1ull << 40) - 1;
constexpr int kMaxEntriesPerOrf = (1 << 23) - 1;

// ---- K3 tiling ------------------------------------------------------------------------------
constexpr int kScoreWarps = 8;                 // warps per CTA
constexpr int kTileCodons = 256;               // codons per warp tile (8 rounds of 32 lanes)
constexpr int kTileNt = 3 * kTileCodons;       // window starts per tile
constexpr int kBufNt = kTileNt + 8;            // + 2 halo + zero pad, keeps 16 B multiples
constexpr int kFetchBatch = 8;                 // ORFs claimed per atomic
constexpr int kBigShift = 20;                  // a value >= 2^20 sends its tile down the 64-bit path
constexpr int kFlushTiles = 3;                 // packed 10-bit fields hold 3 tiles (<= 9 codons/lane/tile)

__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ long long warp_min_i64(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        long long t = __shfl_xor_sync(kFull, v, o);
        v = t < v ? t : v;
    }
    return v;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ int ld_cov(const int32_t* p) { return __ldg(p); }

// Per-lane accumulators of one frame.  w1 / w2 pack 10-bit counters and are flushed into the
// warp-uniform totals every kFlushTiles tiles; the fp64 sums live for the whole ORF.
//   w1 = n(a,0,0) | n(0,b,0) << 10 | n(0,0,c) << 20      unit vectors (1,0), (-1/2, +-sqrt3/2)
//   w2 = n(general) | n(uniform) << 10
struct FrameLane {
    unsigned w1 = 0, w2 = 0;
    double sre = 0.0;   // sum of A / sqrt(A^2 + 3 B^2),            A = 2a - b - c
    double sim = 0.0;   // sum of B / sqrt(A^2 + 3 B^2) (x sqrt3),  B = b - c
};

// One complete codon (a,b,c) of one frame: statistics.py:72-90 in closed form.  The reference
// normalises the triplet by |a + b w + c w^2| and SciPy's coherence then only sees the unit
// vector u = (a + b w + c w^2) / |.| of every non-uniform kept codon (SURVEY.md 8(a) A4);
// 2 Re = A, 2 Im = sqrt3 * B, 4 |.|^2 = A^2 + 3 B^2.  Codons with a single non-zero count map
// to three constant unit vectors and are only counted.
template <bool Big>
__device__ __forceinline__ void accumulate_codon(int a, int b, int c, FrameLane& f) {
    if ((a | b | c) == 0) return;                       // statistics.py:72-73
    if ((b | c) == 0) f.w1 += 1u;
    else if ((a | c) == 0) f.w1 += 1u << 10;
    else if ((a | b) == 0) f.w1 += 1u << 20;
    else if (a == b && b == c) f.w2 += 1u << 10;        // uniform: counts in K only
    else {
        f.w2 += 1u;
        double dA, dB, r;
        if (Big) {
            dA = (double)(2ll * a - b - c);
            dB = (double)((long long)b - c);
            r = rsqrt(fma(dA, dA, 3.0 * dB * dB));
        } else {
            // |A|, |B| < 2^22: D is exact; MUFU seed (2^-22) + one Newton step -> ~1e-13 relative
            dA = (double)(2 * a - b - c);
            dB = (double)(b - c);
            const double D = fma(dA, dA, (3.0 * dB) * dB);
            const double r0 = (double)rsqrt_approx((float)D);
            const double e = fma(-D * r0, r0, 1.0);
            r = fma(0.5 * r0, e, r0);
        }
        f.sre = fma(dA, r, f.sre);
        f.sim = fma(dB, r, f.sim);
    }
}

// Cursor over the concatenated exons of one ORF in PROFILE order (ascending genomic
// positions for '+', descending for '-': detect_orfs.py:176-187,201-202).  Warp-uniform.
struct ExonCursor {
    const uint64_t* entries;  // first entry of this ORF
    int n;                    // entries of this ORF
    bool rev;
    int next = 0;             // entries consumed
    int rem = 0;              // values left in the current entry
    long long pos = 0;        // slot of the next value (relative to cov)
    bool zero = false;
    uint64_t cached = 0;      // lane-private: entry (next & ~31) + lane

    __device__ __forceinline__ bool advance(int lane) {
        if (next == n) return false;
        if ((next & 31) == 0) {
            const int idx = next + lane;
            if (idx < n) cached = __ldg(entries + (rev ? n - 1 - idx : idx));
        }
        const uint64_t ent = __shfl_sync(kFull, cached, next & 31);
        rem = (int)(ent & kLenMask);
        const uint64_t off = ent >> kLenBits;
        zero = off == kZeroOff;
        pos = rev ? (long long)off + rem - 1 : (long long)off;
        ++next;
        return true;
    }
};

// Copy `take` coverage values of the current exon into the tile (4 loads in flight per lane).
template <int Dir>
__device__ __forceinline__ void stage_segment(int32_t* dst, const int32_t* src, int take, int lane, int& ormask) {
    for (int k = lane; k < take; k += 128) {
        int v0 = 0, v1 = 0, v2 = 0, v3 = 0;
        v0 = ld_cov(src + Dir * k);
        if (k + 32 < take) v1 = ld_cov(src + Dir * (k + 32));
        if (k + 64 < take) v2 = ld_cov(src + Dir * (k + 64));
        if (k + 96 < take) v3 = ld_cov(src + Dir * (k + 96));
        dst[k] = v0;
        if (k + 32 < take) dst[k + 32] = v1;
        if (k + 64 < take) dst[k + 64] = v2;
        if (k + 96 < take) dst[k + 96] = v3;
        ormask |= v0 | v1 | v2 | v3;
    }
}

// K3 over one staged tile: one lane per codon, so the three frames are three fixed register
// sets.  Codons [0, nfull) have all three windows complete; the (at most two) codons after them
// only exist in the last tile and are checked window by window (statistics.py:71).
template <bool Big, typename CountT>
__device__ __forceinline__ void score_tile(const int32_t* buf, int nvals, int ncod, int lane, FrameLane& f0,
                                           FrameLane& f1, FrameLane& f2, CountT& cnt, CountT& mn) {
    const int nfull = max(nvals - 2, 0) / 3;
    for (int c = lane; c < nfull; c += 32) {
        const int32_t* p = buf + 3 * c;
        const int v0 = p[0], v1 = p[1], v2 = p[2], v3 = p[3], v4 = p[4];
        const CountT cs = (CountT)(unsigned)v0 + (CountT)(unsigned)v1 + (CountT)(unsigned)v2;   // common.py:177-179
        cnt += cs;                                                           // detect_orfs.py:278
        mn = cs < mn ? cs : mn;
        if ((v0 | v1 | v2 | v3 | v4) != 0) {
            accumulate_codon<Big>(v0, v1, v2, f0);
            accumulate_codon<Big>(v1, v2, v3, f1);
            accumulate_codon<Big>(v2, v3, v4, f2);
        }
    }
    for (int c = nfull + lane; c < ncod; c += 32) {     // ragged end of the profile
        const int32_t* p = buf + 3 * c;
        const int v0 = p[0], v1 = p[1], v2 = p[2], v3 = p[3], v4 = p[4];   // zero padded past nvals
        const CountT cs = (CountT)(unsigned)v0 + (CountT)(unsigned)v1 + (CountT)(unsigned)v2;
        cnt += cs;
        mn = cs < mn ? cs : mn;
        if (3 * c + 2 < nvals) accumulate_codon<Big>(v0, v1, v2, f0);
        if (3 * c + 3 < nvals) accumulate_codon<Big>(v1, v2, v3, f1);
        if (3 * c + 4 < nvals) accumulate_codon<Big>(v2, v3, v4, f2);
    }
}

struct ScoreArgs {
    const int32_t* cov;
    const uint64_t* orf_desc;   // indexed by absolute ORF id
    const uint64_t* exon_entries;
    const int32_t* orf_len;     // profile length per ORF (absolute ORF id)
    long long orf_lo;           // output element k <-> ORF orf_lo + k
    const int32_t* list;        // ORF ids to score (absolute)
    long long n_list;           // entries of `list` ...
    const unsigned* n_list_dev; // ... or, when not NULL, read from the device (fallback queue)
    unsigned long long* work_counter;
    unsigned* n_fallback;
    rt_score_params prm;
    rt_score_out out;
};

// Warp-uniform totals of one frame.
struct TileTotals {
    int na = 0, nb = 0, nc = 0, ng = 0, nu = 0;
    __device__ __forceinline__ void flush(FrameLane& f) {
        const unsigned t1 = __reduce_add_sync(kFull, f.w1);
        const unsigned t2 = __reduce_add_sync(kFull, f.w2);
        na += t1 & 1023;
        nb += (t1 >> 10) & 1023;
        nc += t1 >> 20;
        ng += t2 & 1023;
        nu += t2 >> 10;
        f.w1 = f.w2 = 0;
    }
};

// Generic kernel: one warp per ORF, any length, any counts (64-bit path for huge values).
__global__ void __launch_bounds__(kScoreWarps * 32, 4)
score_orfs_kernel(const ScoreArgs args) {
    const long long n_list = args.n_list_dev ? (long long)*args.n_list_dev : args.n_list;
    __shared__ __align__(16) int32_t s_buf[kScoreWarps][kBufNt];
    const int lane = threadIdx.x & 31;
    int32_t* buf = s_buf[threadIdx.x >> 5];
    const double kSqrt3 = 1.7320508075688772;
    const double kNaN = __longlong_as_double(0x7ff8000000000000ll);

    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(args.work_counter, (unsigned long long)kFetchBatch);
        base = __shfl_sync(kFull, base, 0);
        if ((long long)base >= n_list) break;
        uint64_t my_desc = 0;
        int my_orf = 0;
        if (lane < kFetchBatch && (long long)base + lane < n_list) {
            my_orf = __ldg(args.list + base + lane);
            my_desc = __ldg(args.orf_desc + my_orf);
        }

        for (int bi = 0; bi < kFetchBatch; ++bi) {
            if ((long long)base + bi >= n_list) break;
            const long long k_out = (long long)__shfl_sync(kFull, my_orf, bi) - args.orf_lo;

            const uint64_t desc = __shfl_sync(kFull, my_desc, bi);
            ExonCursor cur;
            cur.entries = args.exon_entries + (desc & kBeginMask);
            cur.n = (int)((desc >> 40) & kMaxEntriesPerOrf);
            cur.rev = (desc >> 63) != 0;

            FrameLane f0, f1, f2;
            TileTotals t0, t1, t2;
            unsigned cnt32 = 0, mn32 = 0xffffffffu;    // per lane, flushed with the packed counters
            long long count = 0;                       // warp-uniform totals
            long long min_codon = 0x7fffffffffffffffll;
            long long total = 0;                       // profile length so far
            int fill = 0, ormask = 0, pending = 0;
            bool last = false;

            while (!last) {
                // ---- K2: stage the next profile tile into shared memory ----
                while (fill < kTileNt + 2) {
                    if (cur.rem == 0 && !cur.advance(lane)) { last = true; break; }
                    const int take = min(cur.rem, kTileNt + 2 - fill);
                    if (cur.zero) {
                        for (int k = lane; k < take; k += 32) buf[fill + k] = 0;
                    } else if (cur.rev) {
                        stage_segment<-1>(buf + fill, args.cov + cur.pos, take, lane, ormask);
                    } else {
                        stage_segment<1>(buf + fill, args.cov + cur.pos, take, lane, ormask);
                    }
                    fill += take;
                    total += take;
                    cur.rem -= take;
                    cur.pos += cur.rev ? -take : take;
                }
                const int nvals = fill;
                if (last && lane < 6) buf[nvals + lane] = 0;   // nvals + 5 < kBufNt
                __syncwarp();

                // ---- K3 ----
                const int ncod = last ? (nvals + 2) / 3 : kTileCodons;
                const bool big = __any_sync(kFull, (ormask >> kBigShift) != 0);
                if (!big) {
                    score_tile<false, unsigned>(buf, nvals, ncod, lane, f0, f1, f2, cnt32, mn32);
                } else {   // huge counts: 64-bit codon sums, reduced right away
                    long long c64 = 0, m64 = 0x7fffffffffffffffll;
                    score_tile<true, long long>(buf, nvals, ncod, lane, f0, f1, f2, c64, m64);
                    count += warp_sum_i64(c64);
                    const long long m = warp_min_i64(m64);
                    min_codon = m < min_codon ? m : min_codon;
                }
                if (++pending == kFlushTiles || last) {
                    t0.flush(f0);
                    t1.flush(f1);
                    t2.flush(f2);
                    count += __reduce_add_sync(kFull, cnt32);
                    const unsigned m = __reduce_min_sync(kFull, mn32);
                    if (m != 0xffffffffu && (long long)m < min_codon) min_codon = m;
                    cnt32 = 0;
                    mn32 = 0xffffffffu;
                    pending = 0;
                }
                __syncwarp();
                if (!last) {   // carry the 2-value halo to the front of the next tile
                    int t = 0;
                    if (lane < 2) t = buf[kTileNt + lane];
                    __syncwarp();
                    if (lane < 2) buf[lane] = t;
                    fill = 2;
                    __syncwarp();
                }
            }

            // ---- epilogue: statistics.py:92-115 + detect_orfs.py:278-299 ----
            const long long L = total;
            const long long n_codons = L / 3 > 1 ? L / 3 : 1;             // detect_orfs.py:281
            double score = 0.0, ratio = 0.0, density = 0.0;
            int valid = 0;
            int K0 = 0, K1 = 0, K2 = 0;
            double s0 = kNaN, s1 = kNaN, s2 = kNaN;
            if (L == 0) min_codon = 0;
            if (count != 0) {
                K0 = t0.na + t0.nb + t0.nc + t0.ng + t0.nu;
                K1 = t1.na + t1.nb + t1.nc + t1.ng + t1.nu;
                K2 = t2.na + t2.nb + t2.nc + t2.ng + t2.nu;
                double re0 = 0.0, im0 = 0.0, re1 = 0.0, im1 = 0.0, re2 = 0.0, im2 = 0.0;
                if ((t0.ng | t1.ng | t2.ng) != 0) {
                    re0 = warp_sum_f64(f0.sre); im0 = warp_sum_f64(f0.sim);
                    re1 = warp_sum_f64(f1.sre); im1 = warp_sum_f64(f1.sim);
                    re2 = warp_sum_f64(f2.sre); im2 = warp_sum_f64(f2.sim);
                }
                re0 += 0.5 * (double)(2 * t0.na - t0.nb - t0.nc); im0 = kSqrt3 * (im0 + 0.5 * (double)(t0.nb - t0.nc));
                re1 += 0.5 * (double)(2 * t1.na - t1.nb - t1.nc); im1 = kSqrt3 * (im1 + 0.5 * (double)(t1.nb - t1.nc));
                re2 += 0.5 * (double)(2 * t2.na - t2.nb - t2.nc); im2 = kSqrt3 * (im2 + 0.5 * (double)(t2.nb - t2.nc));
                // one fp64 division sequence for all seven quotients: lanes 0-2 the coherences
                // |sum u|^2 / (K * M), lane 3 the density, lanes 4-6 K_f / n_codons
                double nn, dd = (double)n_codons;
                if (lane == 0) { nn = re0 * re0 + im0 * im0; dd = (double)K0 * (double)(K0 - t0.nu); }
                else if (lane == 1) { nn = re1 * re1 + im1 * im1; dd = (double)K1 * (double)(K1 - t1.nu); }
                else if (lane == 2) { nn = re2 * re2 + im2 * im2; dd = (double)K2 * (double)(K2 - t2.nu); }
                else if (lane == 3) nn = (double)count;                  // detect_orfs.py:287
                else if (lane == 4) nn = (double)K0;                     // detect_orfs.py:285
                else if (lane == 5) nn = (double)K1;
                else nn = (double)K2;
                const double q = nn / dd;                                // 0/0 -> NaN never wins
                s0 = __shfl_sync(kFull, q, 0);
                s1 = __shfl_sync(kFull, q, 1);
                s2 = __shfl_sync(kFull, q, 2);
                density = __shfl_sync(kFull, q, 3);
                // statistics.py:64-66,92-115: running maximum with the K==0 reset quirk
                double coh = 0.0;
                int vf = -1;          // frame whose K is `valid`; -1: valid = 0
                bool unset = true;    // valid == -1 in the reference
                if (K0 == 0) { coh = 0.0; vf = -1; unset = false; s0 = kNaN; }
                else { if (s0 > coh) { coh = s0; vf = 0; unset = false; } if (unset) { vf = 0; unset = false; } }
                if (K1 == 0) { coh = 0.0; vf = -1; unset = false; s1 = kNaN; }
                else { if (s1 > coh) { coh = s1; vf = 1; unset = false; } if (unset) { vf = 1; unset = false; } }
                if (K2 == 0) { coh = 0.0; vf = -1; unset = false; s2 = kNaN; }
                else { if (s2 > coh) { coh = s2; vf = 2; unset = false; } if (unset) { vf = 2; unset = false; } }
                score = sqrt(coh);                                       // statistics.py:115
                valid = vf == 0 ? K0 : vf == 1 ? K1 : vf == 2 ? K2 : 0;
                ratio = __shfl_sync(kFull, q, vf >= 0 ? 4 + vf : 4);
                if (vf < 0) ratio = 0.0;
            }
            if (lane == 0) {
                const bool ok = score >= args.prm.phase_score_cutoff &&
                                (double)valid >= args.prm.min_valid_codons &&
                                (L == 0 || (double)min_codon >= args.prm.min_reads_per_codon) &&
                                ratio >= args.prm.min_valid_codons_ratio &&
                                density >= args.prm.min_density_over_orf;   // detect_orfs.py:289-299
                args.out.score[k_out] = score;
                args.out.valid[k_out] = valid;
                args.out.count[k_out] = count;
                args.out.length[k_out] = (int32_t)L;
                if (args.out.min_codon)
                    args.out.min_codon[k_out] = min_codon > 0x7fffffffll ? 0x7fffffff : (int32_t)min_codon;
                if (args.out.status) args.out.status[k_out] = ok ? 1 : 0;
                if (args.out.frame_K) {
                    args.out.frame_K[3 * k_out + 0] = K0;
                    args.out.frame_K[3 * k_out + 1] = K1;
                    args.out.frame_K[3 * k_out + 2] = K2;
                }
                if (args.out.frame_s) {
                    args.out.frame_s[3 * k_out + 0] = s0;
                    args.out.frame_s[3 * k_out + 1] = s1;
                    args.out.frame_s[3 * k_out + 2] = s2;
                }
            }
            __syncwarp();
        }
    }
}

template <int LPO>
__device__ __forceinline__ unsigned group_sum_u32(unsigned v) {
#pragma unroll
    for (int o = LPO / 2; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
template <int LPO>
__device__ __forceinline__ double group_sum_f64(double v) {
#pragma unroll
    for (int o = LPO / 2; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// ---- K3, two-phase: atom summaries + per-ORF composition -----------------------------------------
// Candidate ORFs overlap massively (nested ORFs share their 3' exons, isoforms share exons), so the
// index is cut at every exon boundary of every ORF into ATOMS: maximal coverage intervals that no
// ORF exon boundary splits.  Every ORF is a sequence of atoms (plus "reads-as-zero" stretches).
//   phase A (atom_pass_kernel on the compact layout, atom_summary_kernel on the dense planes): every
//            atom is scanned ONCE per library -- windows that lie fully inside the atom are classified
//            and summed by local frame (window start offset mod 3) into the atom's summary;
//   phase B (compose_refs_kernel): the summaries of an ORF's atoms are added with the frame rotation
//            that the atom's profile offset implies, the two windows that straddle every seam between
//            consecutive atoms are rebuilt from the edge values of the summaries, and the epilogue
//            runs (statistics.py:92-115, detect_orfs.py:278-299).
// The work per library is proportional to the UNION of the exons instead of the sum over ORFs.
// '-' strand: a profile window (v0,v1,v2) is the reversed genomic triple and u(v0,v1,v2) =
// w^2 conj(u(v2,v1,v0)), so |sum u| is what the '+'-oriented sums give; only the frame mapping of
// a local frame differs (see compose_refs_kernel).
constexpr int kPieceNt = 33;           // values per lane and pass of atom_pass_kernel (odd multiple of 3: frames stay
                                       //   static per window and consecutive pieces fall into distinct banks)
constexpr int kPassPieces = 32;        // pieces (= lanes) per pass
constexpr int kAtomMaxNt = kPieceNt * kPassPieces;   // 1,056: an atom never spans two passes; <= 352 windows per frame

struct AtomSummary {                   // 96 bytes, six 16-byte chunks
    long long re[3];                   // sum of unit vectors by local frame, '+' orientation, in units of 2^-42 (uv_grid:
    long long im[3];                   //   exact); imaginary part without its sqrt3 factor
    int edge[4];                       // first two and last two values of the atom, ascending slots
                                       //   (edge[1] = edge[2] = 0 for a one-value atom)
    unsigned kpack;                    // kept (non-all-zero) windows by local frame, 10 bits each;
                                       //   bit 31: a value >= 2^kBigShift (32-bit sums may have wrapped)
    unsigned upack;                    // uniform windows among them (count in K only), 10 bits each
    unsigned count;                    // sum of all values of the atom
    unsigned spare0;
    unsigned mn[3];                    // min window sum by local frame (0xffffffff: no window); only read
    unsigned spare1;                   //   when the minima are wanted (the first 80 bytes are enough otherwise)
};
static_assert(sizeof(AtomSummary) == 96, "AtomSummary layout");

struct AtomArgs {
    const int32_t* cov;
    const uint64_t* atoms;             // (slot offset << 24) | len, len <= kAtomMaxNt
    const int32_t* list;               // atom ids to summarise, similar lengths adjacent
    long long n_list;
    unsigned long long* work_counter;
    AtomSummary* out;                  // indexed by atom id; not written for an atom whose values are all zero
    uint8_t* nonzero;                  // indexed by atom id: 0 = every value of the atom is zero
};

// Unit vectors by table.  The unit vector of a codon (a,b,c) depends only on x = a - c and y = b - c
// (A = 2x - y, B = y); for counts below kUvMax every window of the lane indexes one shared-memory
// table of (A, B) / sqrt(A^2 + 3 B^2) -- all-zero and uniform codons hit the (0,0) entry -- so the
// three windows of a round are settled by three loads and six fp64 adds with every lane active,
// instead of a divergent classify / rsqrt sequence that few lanes take.
constexpr int kUvMax = 16;                         // table covers counts 0 .. kUvMax - 1
constexpr int kUvSide = 2 * kUvMax - 1;            // x, y in [-(kUvMax-1), kUvMax-1]
constexpr int kUvStride = 2 * kUvMax + 5;          // row stride 37 = 5 mod 8: the all-zero entry and the three entries of a single count
                                                   //   of 1 -- (1,0,0), (0,1,0), (0,0,1) -- fall into four different bank groups; with the
                                                   //   power of two of round 1 every (a,0,0) entry shared its banks with the all-zero one
constexpr int kUvEntries = kUvSide * kUvStride;
constexpr int kUvCenter = (kUvMax - 1) * kUvStride + (kUvMax - 1);

// The unit vector of a non-uniform codon, ROUNDED TO A GRID of 2^-42: (A, B) / sqrt(A^2 + 3 B^2) with the exactly
// rounded IEEE sqrt and divisions, then to the nearest multiple of 2^-42 (adding and subtracting 1.5 * 2^10, whose
// ulp is 2^-42).  Sums of up to 1,024 such values are EXACT in fp64 (every partial sum is a multiple of 2^-42 below
// 2^10), so the per-atom sums do not depend on the order of summation: any lane / tile / layout decomposition of
// phase A gives bit-identical summaries, and phase B adds them as 64-bit integers (units of 2^-42).  The rounding
// moves a unit vector by at most 2^-42 (2^-43 in A / n, sqrt(3) * 2^-43 in the sqrt(3) B / n it stands for), so a score
// |sum u| / sqrt(K * M) (M non-uniform codons) moves by at most M * 2^-42 / sqrt(K * M) <= 2^-42.
constexpr double kUvGridMagic = 1536.0;
constexpr double kUvGridScale = 4398046511104.0;      // 2^42
__device__ __forceinline__ double2 uv_grid(double A, double B) {     // (A, B) != (0, 0); |A|, |B| < 2^22: D is exact
    const double n = sqrt(fma(A, A, (3.0 * B) * B));
    const double re = __dadd_rn(__dadd_rn(A / n, kUvGridMagic), -kUvGridMagic);
    const double im = __dadd_rn(__dadd_rn(B / n, kUvGridMagic), -kUvGridMagic);
    return make_double2(re, im);
}
__device__ __forceinline__ void fill_uv_table(double2* tab) {
    for (int i = threadIdx.x; i < kUvEntries; i += blockDim.x) {
        const int x = i / kUvStride - (kUvMax - 1), y = i % kUvStride - (kUvMax - 1);
        const double A = (double)(2 * x - y), B = (double)y;
        tab[i] = (x | y) != 0 ? uv_grid(A, B) : make_double2(0.0, 0.0);
    }
}

// One complete window of local frame F outside the table's range (or at the ragged end of an atom).
template <int F>
__device__ __forceinline__ void slow_window(int x, int y, int z, unsigned& accK, unsigned& accM, FrameLane& f) {
    if ((x | y | z) == 0) return;                       // statistics.py:72-73
    accK += 1u << (10 * F);
    const int A = 2 * x - y - z, B = y - z;
    if ((A | B) == 0) return;                           // uniform: counts in K only
    accM += 1u << (10 * F);
    const double2 u = uv_grid((double)A, (double)B);
    f.sre += u.x;
    f.sim += u.y;
}

constexpr int kAtomLPO = 4;            // lanes per atom of atom_summary_kernel
// Packs of G atoms are handed out through an atomic counter (the atoms of a plan window are sorted
// by length, so a static split leaves warps idle).  The chain counter -> list[] -> atoms[] ->
// coverage is four dependent memory round trips; it is software pipelined ACROSS packs: while pack k
// is scanned the warp already holds the atom id of pack k+1, fetches its descriptor and the atom id
// of pack k+2, and has the counter bump for pack k+3 in flight; the first coverage loads of pack
// k+1 are issued before the reductions and the summary store of pack k.
template <bool WantMin>
__global__ void __launch_bounds__(kScoreWarps * 32, 4)
atom_summary_kernel(const AtomArgs args) {
    constexpr int LPO = kAtomLPO;
    constexpr int G = 32 / LPO;
    constexpr int RNT = 3 * LPO;
    __shared__ double2 s_uv[kUvEntries];
    fill_uv_table(s_uv);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int sl = lane % LPO;
    const int gb = lane - sl;
    const int grp = lane / LPO;
    const int nbr = sl + 1 == LPO ? gb : lane + 1;
    const unsigned n_list = (unsigned)args.n_list;        // < 2^32 atoms (rt_set_index)
    const unsigned n_packs = (n_list + G - 1) / G;
    auto load_atom = [&](unsigned pk) -> int {            // atom id of this lane's group in pack pk, -1: none
        const unsigned it = pk * G + grp;
        return (pk < n_packs && it < n_list) ? __ldg(args.list + it) : -1;
    };

    // lane's three values of round r sit at src + 3 sl + r RNT; `left` = values from there to the atom's end
    const int32_t* ptr = args.cov;
    int left = 0;
    auto load3 = [&](int& v0, int& v1, int& v2) {
        v0 = left > 0 ? ld_cov(ptr) : 0;
        v1 = left > 1 ? ld_cov(ptr + 1) : 0;
        v2 = left > 2 ? ld_cov(ptr + 2) : 0;
        ptr += RNT;
        left -= RNT;
    };

    // ---- pipeline prologue: packs k, k+1, k+2 of this warp ----
    unsigned long long raw = 0;
    if (lane == 0) raw = atomicAdd(args.work_counter, 3ull);
    raw = __shfl_sync(kFull, raw, 0);
    unsigned pack = (unsigned)min(raw, 0xfffffff0ull), pack1 = pack + 1;
    unsigned raw2 = pack + 2;                             // lane 0's copy is the one that is read
    int atom = load_atom(pack);
    int atom1 = load_atom(pack1);
    int len = 0;
    const int32_t* src = args.cov;
    if (atom >= 0) {
        const uint64_t ent = __ldg(args.atoms + atom);
        len = (int)(ent & kLenMask);
        src = args.cov + (ent >> kLenBits);
    }
    // Three register sets hold rounds r, r + 1, r + 2 and are refilled in turn (the round loop is unrolled
    // by three so that no register is ever copied: a copy would wait for its load).  A set is requested
    // right after it has been consumed, two rounds before its first two values are needed again.
    int a0, a1, a2, b0, b1, b2, c0, c1, c2;
    ptr = src + 3 * sl;
    left = len - 3 * sl;
    load3(a0, a1, a2);
    load3(b0, b1, b2);
    load3(c0, c1, c2);

    while (pack < n_packs) {
        // ---- descriptor of pack k+1, atom id of pack k+2, counter bump for pack k+3 ----
        uint64_t ent1 = 0;
        if (atom1 >= 0) ent1 = __ldg(args.atoms + atom1);
        const unsigned pack2 = __shfl_sync(kFull, raw2, 0);
        const int atom2 = load_atom(pack2);
        if (lane == 0) raw2 = (unsigned)min(atomicAdd(args.work_counter, 1ull), 0xfffffff0ull);

        FrameLane f0, f1, f2;                  // only the fp64 sums are used here
        unsigned accK = 0, accM = 0;           // 10-bit fields by local frame: kept windows, non-uniform windows
        unsigned cnt32 = 0, mn0 = 0xffffffffu, mn1 = 0xffffffffu, mn2 = 0xffffffffu;
        int ormask = 0;
        const int rounds = __reduce_max_sync(kFull, ((len + 2) / 3 + LPO - 1) / LPO);
        int p = 3 * sl;
        // one round: the lane's values (u0,u1,u2) at profile offsets p..p+2 of its atom, (w0,w1) = the same
        // lane's first two values of the next round (what the last lane of a group hands to the first)
        auto round = [&](int& u0, int& u1, int& u2, const int w0, const int w1) {
            const int v3 = __shfl_sync(kFull, sl == 0 ? w0 : u0, nbr);
            const int v4 = __shfl_sync(kFull, sl == 0 ? w1 : u1, nbr);
            if (p < len) {
                cnt32 += (unsigned)u0 + (unsigned)u1 + (unsigned)u2;
                const int o3 = u0 | u1 | u2;
                ormask |= o3;
                if (p + 4 < len) {                               // all three windows lie inside the atom
                    if (WantMin) {
                        const unsigned s0 = (unsigned)u0 + (unsigned)u1 + (unsigned)u2;
                        const unsigned s1 = (unsigned)u1 + (unsigned)u2 + (unsigned)v3;
                        const unsigned s2 = (unsigned)u2 + (unsigned)v3 + (unsigned)v4;
                        mn0 = min(mn0, s0); mn1 = min(mn1, s1); mn2 = min(mn2, s2);
                    }
                    const int o5 = o3 | v3 | v4;
                    if (o5 != 0) {
                        if ((unsigned)o5 < (unsigned)kUvMax) {
                            const int i0 = (u0 - u2) * kUvStride + (u1 - u2) + kUvCenter;
                            const int i1 = (u1 - v3) * kUvStride + (u2 - v3) + kUvCenter;
                            const int i2 = (u2 - v4) * kUvStride + (v3 - v4) + kUvCenter;
                            const double2 t0 = s_uv[i0], t1 = s_uv[i1], t2 = s_uv[i2];
                            f0.sre += t0.x; f0.sim += t0.y;
                            f1.sre += t1.x; f1.sim += t1.y;
                            f2.sre += t2.x; f2.sim += t2.y;
                            accK += min((unsigned)o3, 1u) + (min((unsigned)(u1 | u2 | v3), 1u) << 10) +
                                    (min((unsigned)(u2 | v3 | v4), 1u) << 20);
                            accM += min((unsigned)(i0 ^ kUvCenter), 1u) + (min((unsigned)(i1 ^ kUvCenter), 1u) << 10) +
                                    (min((unsigned)(i2 ^ kUvCenter), 1u) << 20);
                        } else {
                            slow_window<0>(u0, u1, u2, accK, accM, f0);
                            slow_window<1>(u1, u2, v3, accK, accM, f1);
                            slow_window<2>(u2, v3, v4, accK, accM, f2);
                        }
                    }
                } else {                                         // ragged end of the atom
                    if (p + 2 < len) { if (WantMin) mn0 = min(mn0, (unsigned)u0 + (unsigned)u1 + (unsigned)u2); slow_window<0>(u0, u1, u2, accK, accM, f0); }
                    if (p + 3 < len) { if (WantMin) mn1 = min(mn1, (unsigned)u1 + (unsigned)u2 + (unsigned)v3); slow_window<1>(u1, u2, v3, accK, accM, f1); }
                }
            }
            p += RNT;
            load3(u0, u1, u2);                                   // this set's next turn: three rounds on
        };
        for (int r = 0; r < rounds; r += 3) {
            round(a0, a1, a2, b0, b1);
            if (r + 1 < rounds) round(b0, b1, b2, c0, c1);
            if (r + 2 < rounds) round(c0, c1, c2, a0, a1);
        }

        // ---- pack k+1 becomes current: its first two rounds are requested before pack k is reduced ----
        const int atom_done = atom, len_done = len;
        const int32_t* src_done = src;
        atom = atom1;
        len = (int)(ent1 & kLenMask);
        src = args.cov + (ent1 >> kLenBits);
        ptr = src + 3 * sl;
        left = len - 3 * sl;
        load3(a0, a1, a2);
        load3(b0, b1, b2);
        load3(c0, c1, c2);
        atom1 = atom2;
        pack = pack1;
        pack1 = pack2;

        // ---- reductions and summary of the pack just scanned ----
        const unsigned K = group_sum_u32<LPO>(accK), M = group_sum_u32<LPO>(accM);
        const unsigned count = group_sum_u32<LPO>(cnt32);
#pragma unroll
        for (int o = LPO / 2; o > 0; o >>= 1) {
            if (WantMin) {
                mn0 = min(mn0, __shfl_xor_sync(kFull, mn0, o));
                mn1 = min(mn1, __shfl_xor_sync(kFull, mn1, o));
                mn2 = min(mn2, __shfl_xor_sync(kFull, mn2, o));
            }
            ormask |= __shfl_xor_sync(kFull, ormask, o);
        }
        double re0 = 0.0, im0 = 0.0, re1 = 0.0, im1 = 0.0, re2 = 0.0, im2 = 0.0;
        if (__any_sync(kFull, M != 0)) {
            re0 = group_sum_f64<LPO>(f0.sre); im0 = group_sum_f64<LPO>(f0.sim);
            re1 = group_sum_f64<LPO>(f1.sre); im1 = group_sum_f64<LPO>(f1.sim);
            re2 = group_sum_f64<LPO>(f2.sre); im2 = group_sum_f64<LPO>(f2.sim);
        }
        if (atom_done >= 0 && sl == 0) {
            args.nonzero[atom_done] = ormask != 0;
            if (ormask != 0) {
                AtomSummary s;
                s.kpack = K | ((ormask >> kBigShift) != 0 ? 0x80000000u : 0u);
                s.upack = K - M;                         // field-wise: no borrow, every M field <= its K field
                s.count = count;
                s.spare0 = s.spare1 = 0;
                s.re[0] = __double2ll_rn(re0 * kUvGridScale); s.im[0] = __double2ll_rn(im0 * kUvGridScale);
                s.re[1] = __double2ll_rn(re1 * kUvGridScale); s.im[1] = __double2ll_rn(im1 * kUvGridScale);
                s.re[2] = __double2ll_rn(re2 * kUvGridScale); s.im[2] = __double2ll_rn(im2 * kUvGridScale);
                s.mn[0] = mn0; s.mn[1] = mn1; s.mn[2] = mn2;
                s.edge[0] = ld_cov(src_done);
                s.edge[1] = len_done >= 2 ? ld_cov(src_done + 1) : 0;
                s.edge[2] = len_done >= 2 ? ld_cov(src_done + len_done - 2) : 0;
                s.edge[3] = ld_cov(src_done + len_done - 1);
                args.out[atom_done] = s;
            }
        }
        __syncwarp();
    }
}

// ---- phase A, streamed: atom_pass_kernel --------------------------------------------------------
// In the compact layout the atoms lie back to back, so phase A is one sequential read of the coverage buffer.
// The host cuts the atom list into PASSES: runs of consecutive atoms, adjacent in memory, of at most kPassPieces
// PIECES (a piece = kPieceNt consecutive values of ONE atom, starting a multiple of kPieceNt after the atom's
// first value).  Every warp owns a ring of shared-memory stages; one elected lane brings the coverage span of a
// pass (and its atom descriptors) in with cp.async.bulk (TMA, 1-D) completing on the stage's mbarrier, a few passes
// ahead of the one being scanned.  One lane per piece: the lane reads its kPieceNt + 2 values from shared memory
// (consecutive pieces are 33 words apart: conflict-free), zeroes what lies beyond its atom's end and settles its
// 33 windows in straight-line code -- window q is local frame q mod 3, a compile-time constant, and every window
// is one table lookup (see fill_uv_table) and two exact fp64 adds.  With the tail zeroed the only windows a lane
// gets wrong are the two that start on the atom's last two values; they depend on those two values alone, and
// because the sums are exact (uv_grid) the atom's head lane simply subtracts them again.  The pieces of an atom sit
// on consecutive lanes and are added up by a segmented shuffle reduction; the head lane writes the summary.
struct PassDesc {                      // 16 bytes, everything the elected lane needs to issue the two copies
    uint32_t atom0;                    // first atom of the pass
    uint32_t n_atoms_cov16;            // atoms of the pass (<= kPassPieces) | 16-byte units of coverage to copy << 8
    uint32_t slot0_q;                  // first coverage slot to copy (slot of atom0's first value, rounded down to 4) >> 2
    uint32_t slot0_r;                  // slot of atom0's first value minus that (0..3)
};
struct PassArgs {
    const int32_t* cov;
    const uint64_t* atoms;             // (slot offset << 24) | len; allocated with slack (descriptor pairs are copied)
    const PassDesc* passes;
    unsigned n_passes;
    AtomSummary* out;
    uint8_t* nonzero;
};
constexpr int kPassBufSlots = kAtomMaxNt + 4 + 36;                   // + alignment slack + the reads past a short tail
constexpr int kPassEntSlots = kPassPieces + 2;                       // atom descriptors of a pass (16-byte aligned copy)
constexpr int kPassStageBytes = kPassBufSlots * 4 + kPassEntSlots * 8 + 16 + 16;   // values | descriptors | PassDesc | mbarrier
static_assert(kPassStageBytes % 16 == 0 && (kPassBufSlots * 4) % 16 == 0, "stage layout");
constexpr int kGroupNt = kPieceNt / 3;                               // a lane settles its piece in three groups of 11 windows
static_assert(kGroupNt * 3 == kPieceNt, "piece = three groups");
// 16 warps x 2 stages measured best on C2 (profiles/README.md): more warps need the 64-register build, which spills, and
// a third stage buys nothing -- the kernel is bound by the shared-memory pipe, not by the copies
constexpr int kPassWarps = 16, kPassStages = 2;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// n += (x != 0) as one compare and one predicated add
__device__ __forceinline__ void count_nonzero(unsigned& n, int x) {
    asm("{\n.reg .pred p;\nsetp.ne.s32 p, %1, 0;\n@p add.u32 %0, %0, 1;\n}" : "+r"(n) : "r"(x));
}

template <bool WantMin>
__global__ void __launch_bounds__(kPassWarps * 32, 1) atom_pass_kernel(const PassArgs args) {
    constexpr int STAGES = kPassStages;
    extern __shared__ __align__(16) unsigned char s_raw[];
    double2* s_uv = reinterpret_cast<double2*>(s_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    unsigned char* my = s_raw + ((kUvEntries * sizeof(double2) + 15) & ~(size_t)15) + (size_t)warp * STAGES * kPassStageBytes;
    auto st_buf = [&](int s) { return reinterpret_cast<int32_t*>(my + (size_t)s * kPassStageBytes); };
    auto st_ent = [&](int s) { return reinterpret_cast<uint64_t*>(my + (size_t)s * kPassStageBytes + kPassBufSlots * 4); };
    auto st_desc = [&](int s) { return reinterpret_cast<uint4*>(my + (size_t)s * kPassStageBytes + kPassBufSlots * 4 + kPassEntSlots * 8); };
    auto st_bar = [&](int s) { return reinterpret_cast<uint64_t*>(my + (size_t)s * kPassStageBytes + kPassBufSlots * 4 + kPassEntSlots * 8 + 16); };
    fill_uv_table(s_uv);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(st_bar(s), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const unsigned G = gridDim.x * (unsigned)n_warps, g = blockIdx.x * (unsigned)n_warps + (unsigned)warp;
    const unsigned n_mine = g < args.n_passes ? (args.n_passes - g + G - 1) / G : 0u;     // passes g, g + G, ...
    // lane 0: bring pass number `it` of this warp into stage it % STAGES
    auto issue = [&](unsigned it, const uint4 d) {
        const int s = (int)(it % STAGES);
        const unsigned cov_bytes = (d.y >> 8) * 16u;
        const unsigned e0 = d.x & ~1u;
        const unsigned ent_bytes = ((d.x + (d.y & 255u) + 1u) & ~1u) * 8u - e0 * 8u;
        *st_desc(s) = d;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(st_bar(s), cov_bytes + ent_bytes);
        tma_load_1d(st_buf(s), args.cov + ((size_t)d.z << 2), cov_bytes, st_bar(s));
        tma_load_1d(st_ent(s), args.atoms + e0, ent_bytes, st_bar(s));
    };
    auto load_desc = [&](unsigned it) -> uint4 {
        return it < n_mine ? __ldg(reinterpret_cast<const uint4*>(args.passes) + (size_t)g + (size_t)it * G) : make_uint4(0, 0, 0, 0);
    };
    uint4 d_next = make_uint4(0, 0, 0, 0);      // lane 0: descriptor of the next pass to issue
    if (lane == 0) {
        for (unsigned it = 0; it + 1 < (unsigned)STAGES && it < n_mine; ++it) issue(it, load_desc(it));
        d_next = load_desc(STAGES - 1);
    }

    for (unsigned it = 0; it < n_mine; ++it) {
        const int s = (int)(it % STAGES);
        if (lane == 0) {       // the stage of pass it - 1 is free (the __syncwarp below): refill it with pass it + STAGES - 1
            const unsigned nx = it + STAGES - 1;
            if (nx < n_mine) issue(nx, d_next);
            d_next = load_desc(nx + 1);
        }
        __syncwarp();
        mbar_wait(st_bar(s), (it / STAGES) & 1u);
        const int32_t* buf = st_buf(s);
        const uint4 d = *st_desc(s);
        const int n_atoms = (int)(d.y & 255u);
        const uint64_t a0 = (uint64_t)d.z << 2;                                        // slot of buf[0]

        // ---- pieces -> lanes ----
        uint64_t ent = 0;
        int np = 0;
        if (lane < n_atoms) {
            ent = st_ent(s)[(d.x & 1u) + lane];
            np = ((int)(ent & kLenMask) + kPieceNt - 1) / kPieceNt;
        }
        int incl = np;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += t;
        }
        const int excl = incl - np;
        const unsigned heads = __reduce_or_sync(kFull, np > 0 ? 1u << excl : 0u);     // bit = first lane of an atom
        const int total = __shfl_sync(kFull, incl, 31);
        const int max_np = (int)__reduce_max_sync(kFull, (unsigned)np);
        const bool active = lane < total;
        const int k = __popc(heads & (0xffffffffu >> (31 - lane))) - 1;               // my atom (lane index of its descriptor)
        const uint64_t entk = __shfl_sync(kFull, ent, k);
        const int first_lane = __shfl_sync(kFull, excl, k);
        const int end_lane = __shfl_sync(kFull, incl, k);                              // pieces of my atom: [first_lane, end_lane)
        const int len = (int)(entk & kLenMask);
        const int off = (lane - first_lane) * kPieceNt;
        const int rem = active ? len - off : 0;                                        // values from my first one to the atom's end
        const int abase = (int)((entk >> kLenBits) - a0);                              // atom's first value in buf
        const int base = active ? abase + off : 0;
        const int32_t* mine = buf + base;

        unsigned cnt = 0;
        int orm = 0, e0v = 0, e1v = 0;
        double re0 = 0.0, im0 = 0.0, re1 = 0.0, im1 = 0.0, re2 = 0.0, im2 = 0.0;
        unsigned K0 = 0, K1 = 0, K2 = 0, M0 = 0, M1 = 0, M2 = 0;
        unsigned mn0 = 0xffffffffu, mn1 = 0xffffffffu, mn2 = 0xffffffffu;
        const char* center = reinterpret_cast<const char*>(s_uv + kUvCenter);
        int h0 = mine[0], h1 = mine[1];                                                // the two values a group inherits
        if (rem < 2) { if (rem < 1) h0 = 0; h1 = 0; }
        e0v = h0;
        e1v = h1;
#pragma unroll
        for (int gq = 0; gq < 3; ++gq) {
            // values gq * 11 .. gq * 11 + 12 of the piece; what lies beyond the atom's end reads as zero
            int v[kGroupNt + 2];
            v[0] = h0;
            v[1] = h1;
#pragma unroll
            for (int t = 2; t < kGroupNt + 2; ++t) v[t] = mine[gq * kGroupNt + t];
            const int left = rem - gq * kGroupNt;                                      // values from v[0] to the atom's end
            if (left < kGroupNt + 2) {
#pragma unroll
                for (int t = 2; t < kGroupNt + 2; ++t)
                    if (t >= left) v[t] = 0;
            }
            h0 = v[kGroupNt];
            h1 = v[kGroupNt + 1];
            int og = 0;
#pragma unroll
            for (int t = 0; t < kGroupNt; ++t) {
                cnt += (unsigned)v[t];
                og |= v[t];
            }
            orm |= og;
            if ((unsigned)(og | h0 | h1) < (unsigned)kUvMax) {
#pragma unroll
                for (int q = 0; q < kGroupNt; ++q) {
                    const int a = v[q], b = v[q + 1], c = v[q + 2];
                    const int i16 = (a * kUvStride + b - c * (kUvStride + 1)) * 16;
                    constexpr int kF0 = 0;
                    const int f = (gq * kGroupNt + q) % 3 + kF0;
                    // all-zero windows (most of them) neither load nor add: their lanes take no part in the table access,
                    // so they cannot collide with the lanes that look something up
                    if ((a | b | c) != 0) {
                        const double2 u = *reinterpret_cast<const double2*>(center + i16);
                        if (f == 0) { re0 += u.x; im0 += u.y; K0 += 1u; }
                        else if (f == 1) { re1 += u.x; im1 += u.y; K1 += 1u; }
                        else { re2 += u.x; im2 += u.y; K2 += 1u; }
                    }
                    if (f == 0) count_nonzero(M0, i16);
                    else if (f == 1) count_nonzero(M1, i16);
                    else count_nonzero(M2, i16);
                    if (WantMin) {
                        const unsigned sum = q + 2 < left ? (unsigned)a + (unsigned)b + (unsigned)c : 0xffffffffu;
                        if (f == 0) mn0 = min(mn0, sum);
                        else if (f == 1) mn1 = min(mn1, sum);
                        else mn2 = min(mn2, sum);
                    }
                }
            } else {
                // a count outside the table: the same windows through uv_grid (same values as the table holds)
#pragma unroll 1
                for (int q = 0; q < kGroupNt; ++q) {
                    const int p = gq * kGroupNt + q;
                    const int a = p < rem ? mine[p] : 0, b = p + 1 < rem ? mine[p + 1] : 0, c = p + 2 < rem ? mine[p + 2] : 0;
                    const unsigned kq = (a | b | c) != 0 ? 1u : 0u;
                    const int A = 2 * a - b - c, B = b - c;
                    const unsigned mq = (A | B) != 0 ? 1u : 0u;
                    double2 u = make_double2(0.0, 0.0);
                    if (mq) u = uv_grid((double)A, (double)B);
                    const unsigned sum = p + 2 < rem ? (unsigned)a + (unsigned)b + (unsigned)c : 0xffffffffu;
                    const int f = p % 3;
                    if (f == 0) { re0 += u.x; im0 += u.y; K0 += kq; M0 += mq; if (WantMin) mn0 = min(mn0, sum); }
                    else if (f == 1) { re1 += u.x; im1 += u.y; K1 += kq; M1 += mq; if (WantMin) mn1 = min(mn1, sum); }
                    else { re2 += u.x; im2 += u.y; K2 += kq; M2 += mq; if (WantMin) mn2 = min(mn2, sum); }
                }
            }
        }

        // ---- add up the pieces of every atom (consecutive lanes) ----
        unsigned Kp = K0 | (K1 << 10) | (K2 << 20), Mp = M0 | (M1 << 10) | (M2 << 20);
        for (int o = 1; o < max_np; o <<= 1) {
            const bool take = lane + o < end_lane;
            const double t0 = __shfl_down_sync(kFull, re0, o), t1 = __shfl_down_sync(kFull, im0, o);
            const double t2 = __shfl_down_sync(kFull, re1, o), t3 = __shfl_down_sync(kFull, im1, o);
            const double t4 = __shfl_down_sync(kFull, re2, o), t5 = __shfl_down_sync(kFull, im2, o);
            const unsigned tk = __shfl_down_sync(kFull, Kp, o), tm = __shfl_down_sync(kFull, Mp, o);
            const unsigned tc = __shfl_down_sync(kFull, cnt, o);
            const int to = __shfl_down_sync(kFull, orm, o);
            if (take) {
                re0 += t0; im0 += t1; re1 += t2; im1 += t3; re2 += t4; im2 += t5;
                Kp += tk; Mp += tm; cnt += tc; orm |= to;
            }
            if (WantMin) {
                const unsigned u0 = __shfl_down_sync(kFull, mn0, o), u1 = __shfl_down_sync(kFull, mn1, o);
                const unsigned u2 = __shfl_down_sync(kFull, mn2, o);
                if (take) { mn0 = min(mn0, u0); mn1 = min(mn1, u1); mn2 = min(mn2, u2); }
            }
        }

        // ---- head lane: take the two windows that run over the atom's end out again, write the summary ----
        if (active && lane == first_lane) {
            const unsigned atom = d.x + (unsigned)k;
            args.nonzero[atom] = orm != 0;
            if (orm != 0) {
                const int z1 = buf[abase + len - 1];                       // last value
                const int z0 = len >= 2 ? buf[abase + len - 2] : 0;        // the one before it
                if (z1 != 0) {                                             // window (z1, 0, 0) at len - 1: u = (1, 0)
                    const int f = (len - 1) % 3;
                    if (f == 0) re0 -= 1.0; else if (f == 1) re1 -= 1.0; else re2 -= 1.0;
                    Kp -= 1u << (10 * f);
                    Mp -= 1u << (10 * f);
                }
                if (len >= 2 && (z0 | z1) != 0) {                          // window (z0, z1, 0) at len - 2
                    const int f = (len - 2) % 3;
                    double2 u;
                    if ((unsigned)(z0 | z1) < (unsigned)kUvMax) u = s_uv[kUvCenter + z0 * kUvStride + z1];
                    else u = uv_grid((double)(2 * z0 - z1), (double)z1);
                    if (f == 0) { re0 -= u.x; im0 -= u.y; } else if (f == 1) { re1 -= u.x; im1 -= u.y; } else { re2 -= u.x; im2 -= u.y; }
                    Kp -= 1u << (10 * f);
                    Mp -= 1u << (10 * f);
                }
                AtomSummary sm;
                sm.re[0] = __double2ll_rn(re0 * kUvGridScale); sm.re[1] = __double2ll_rn(re1 * kUvGridScale);
                sm.re[2] = __double2ll_rn(re2 * kUvGridScale);
                sm.im[0] = __double2ll_rn(im0 * kUvGridScale); sm.im[1] = __double2ll_rn(im1 * kUvGridScale);
                sm.im[2] = __double2ll_rn(im2 * kUvGridScale);
                sm.edge[0] = e0v;
                sm.edge[1] = e1v;                                          // zero when len == 1
                sm.edge[2] = z0;
                sm.edge[3] = z1;
                sm.kpack = Kp | ((orm >> kBigShift) != 0 ? 0x80000000u : 0u);
                sm.upack = Kp - Mp;                                        // field-wise: every M field <= its K field
                sm.count = cnt;
                sm.spare0 = sm.spare1 = 0;
                sm.mn[0] = mn0; sm.mn[1] = mn1; sm.mn[2] = mn2;
                args.out[atom] = sm;
            }
        }
        __syncwarp();
    }
}

// ---- phase B, one lane per atom reference of a FAMILY of ORFs: compose_refs_kernel ------------------------
// Candidate ORFs that share their stop (nested ORFs of a transcript) are suffixes of the longest one: from some
// reference on they consist of the same atoms.  The host groups such ORFs into families and lays the references of
// the longest member (the parent) out, 16 bytes each, with everything the kernel needs of the reference's profile
// offset precomputed, padded so that a family never straddles a group of 32 slots.  A warp takes one group: every
// lane loads its reference and the summary of its atom (coalesced / independent loads, no serial walk), turns the
// summary into sums by the PARENT's profile frames and rebuilds the two windows that straddle the seam with the
// reference before it from the edge values of the neighbouring lanes.  A segmented SUFFIX scan over the lanes of a
// family then gives, on every lane, the sums from that reference to the end -- the sums are 64-bit integers
// (uv_grid), so the order of summation is immaterial and a suffix sum can lose its own seam windows again by
// subtraction.  Every lane on which an ORF starts (the parent on the first, a child anywhere) rotates the sums into
// that ORF's frames and scores it: a reference is visited once per family, not once per ORF.  ORFs with more than 32
// references stay alone and fill whole groups; each group adds its sums to the ORF's accumulator with integer
// atomics and the group that arrives last scores the ORF.
struct RefRec {                        // 16 bytes
    uint32_t atom;                     // atom id; 0xffffffff: a stretch that reads as zeros
    uint32_t len_flags;                // values of the reference (24 bits) and what the kernel needs of its profile offset P and
                                       //   of the ORF's length L, precomputed: see kRef* below
    uint32_t aux;                      // (len + P) mod 3 | kRefFamilyHead on the first reference of a family
    int32_t orf;                       // the ORF that STARTS on this reference (absolute id); -2: none; -1: padding slot
};
constexpr uint32_t kRefFamilyHead = 1u << 2;
constexpr uint32_t kRefLenMask = (1u << 24) - 1u;
constexpr int kRefPmod3Shift = 24;     // 2 bits: P mod 3
constexpr uint32_t kRefPge1 = 1u << 26, kRefPge2 = 1u << 27;
constexpr uint32_t kRefLast = 1u << 28;    // P + len == L
constexpr int kRefLmod3Shift = 29;     // 2 bits: L mod 3 of the ORF that starts here (of the ORF itself on every slot of a long one)
constexpr uint32_t kRefRev = 1u << 31;     // ORF on the '-' strand
struct RefWarp {                       // per group of 32 slots
    int32_t long_idx;                  // >= 0: the group belongs to long ORF number long_idx (more than 32 references)
    int32_t n_groups;                  //        ... which spans this many groups
    int32_t orf;                       //        ... its absolute id
    int32_t pad;
};
struct LongAcc {                       // accumulator of one long ORF; all-zero except mn = 0xffffffff between launches
    unsigned long long RE[3], IM[3];
    unsigned long long count;
    unsigned K[3], U[3];
    unsigned mn, big, done, pad;
};
static_assert(sizeof(LongAcc) == 96, "LongAcc layout");
struct RefComposeArgs {
    const RefRec* refs;
    const RefWarp* warps;
    long long n_warps;
    const AtomSummary* summaries;
    const uint8_t* atom_nonzero;
    const double2* uv_table;           // fill_uv_table in global memory (seam windows)
    int want_min;
    const int32_t* orf_len;
    long long orf_lo;
    int32_t* fallback;
    unsigned* n_fallback;
    LongAcc* long_acc;
    rt_score_params prm;
    rt_score_out out;
};
constexpr int kMaxExactCodons = 1 << 20;      // per frame: the 21-bit packed K / U fields of the reduction

__global__ void __launch_bounds__(256) fill_uv_table_kernel(double2* tab) { fill_uv_table(tab); }

// v[i] for i in {0, 1, 2} without indexing registers: p0 = (i == 0), p1 = (i == 1)
template <typename T>
__device__ __forceinline__ T sel3(bool p0, bool p1, T v0, T v1, T v2) { return p0 ? v0 : (p1 ? v1 : v2); }

// statistics.py:92-115 + detect_orfs.py:278-299 on the finished sums of one ORF; the two quotients of the filter
// predicate are only formed when their thresholds can reject anything
template <typename Args>
__device__ __forceinline__ void finish_orf_lean(const Args& args, int orf, int L, const unsigned* K, const unsigned* U,
                                                const long long* RE, const long long* IM, unsigned mn, long long count) {
    const double kSqrt3 = 1.7320508075688772;
    const double kNaN = __longlong_as_double(0x7ff8000000000000ll);
    const int n_codons = L / 3 > 1 ? L / 3 : 1;                          // detect_orfs.py:281
    double s3[3];
    double coh = 0.0;
    int valid = -1;
#pragma unroll
    for (int f = 0; f < 3; ++f) {
        double s = kNaN;
        if (K[f] == 0) { coh = 0.0; valid = 0; }                          // statistics.py:94-95
        else {
            const double re = (double)RE[f] * (1.0 / kUvGridScale);        // the sums are exact integers (units of 2^-42)
            const double im = kSqrt3 * ((double)IM[f] * (1.0 / kUvGridScale));
            s = (re * re + im * im) / ((double)K[f] * (double)(K[f] - U[f]));   // 0/0 -> NaN never wins
            if (s > coh) { coh = s; valid = (int)K[f]; }                  // statistics.py:109-111
            if (valid == -1) valid = (int)K[f];                           // statistics.py:112-113
        }
        s3[f] = s;
    }
    const double score = sqrt(coh);                                      // statistics.py:115
    bool ok = score >= args.prm.phase_score_cutoff && (double)valid >= args.prm.min_valid_codons &&
              (L == 0 || (double)(L == 0 ? 0u : mn) >= args.prm.min_reads_per_codon);
    if (args.prm.min_valid_codons_ratio > 0.0)                           // detect_orfs.py:285 (valid >= 0: a threshold <= 0 always passes)
        ok = ok && (double)valid / (double)n_codons >= args.prm.min_valid_codons_ratio;
    else ok = ok && !(args.prm.min_valid_codons_ratio != args.prm.min_valid_codons_ratio);
    if (args.prm.min_density_over_orf > 0.0)                             // detect_orfs.py:287
        ok = ok && (double)count / (double)n_codons >= args.prm.min_density_over_orf;
    else ok = ok && !(args.prm.min_density_over_orf != args.prm.min_density_over_orf);
    const unsigned min_codon = L == 0 ? 0u : mn;
    const long long k_out = (long long)orf - args.orf_lo;
    args.out.score[k_out] = score;
    args.out.valid[k_out] = valid;
    args.out.count[k_out] = count;
    args.out.length[k_out] = L;
    if (args.out.min_codon) args.out.min_codon[k_out] = (int32_t)min_codon;
    if (args.out.status) args.out.status[k_out] = ok ? 1 : 0;
    if (args.out.frame_K) {
        args.out.frame_K[3 * k_out + 0] = (int)K[0];
        args.out.frame_K[3 * k_out + 1] = (int)K[1];
        args.out.frame_K[3 * k_out + 2] = (int)K[2];
    }
    if (args.out.frame_s) {
        args.out.frame_s[3 * k_out + 0] = s3[0];
        args.out.frame_s[3 * k_out + 1] = s3[1];
        args.out.frame_s[3 * k_out + 2] = s3[2];
    }
}

template <bool WantMin>
__global__ void __launch_bounds__(256, 4) compose_refs_kernel(const RefComposeArgs args) {
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= args.n_warps) return;
    const int lane = threadIdx.x & 31;
    const long long slot = w * 32 + lane;
    const uint4 rr = __ldg(reinterpret_cast<const uint4*>(args.refs) + slot);
    const RefWarp rw = args.warps[w];
    const bool is_long = rw.long_idx >= 0;
    const int orf = (int)rr.w;                                            // the ORF that starts here (>= 0), -2, or -1 = padding
    const bool valid = orf != -1;
    const unsigned atom = rr.x;
    const int len = (int)(rr.y & kRefLenMask);
    const bool rev = (rr.y & kRefRev) != 0;
    const int pm3 = (int)((rr.y >> kRefPmod3Shift) & 3u);                 // P mod 3 (P: offset in the parent's profile)
    const bool p_ge1 = (rr.y & kRefPge1) != 0, p_ge2 = (rr.y & kRefPge2) != 0, last = (rr.y & kRefLast) != 0;
    const int lm3 = (int)((rr.y >> kRefLmod3Shift) & 3u);                 // L mod 3 of the ORF starting here
    // the summary is requested together with the atom's "holds a read" byte, not after it
    const bool has_atom = valid && atom != 0xffffffffu;
    const AtomSummary* s = args.summaries + (has_atom ? atom : 0u);
    const bool nz = has_atom && __ldg(args.atom_nonzero + atom) != 0;
    longlong2 r01 = make_longlong2(0, 0), r2i0 = r01, i12 = r01;
    int4 edge = make_int4(0, 0, 0, 0);
    uint4 ku = make_uint4(0, 0, 0, 0), mc = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0u);
    if (has_atom) {
        r01 = __ldg(reinterpret_cast<const longlong2*>(s));          // re[0], re[1]
        r2i0 = __ldg(reinterpret_cast<const longlong2*>(s) + 1);     // re[2], im[0]
        i12 = __ldg(reinterpret_cast<const longlong2*>(s) + 2);      // im[1], im[2]
        edge = __ldg(reinterpret_cast<const int4*>(s) + 3);
        ku = __ldg(reinterpret_cast<const uint4*>(s) + 4);           // kpack, upack, count
        if (WantMin) mc = __ldg(reinterpret_cast<const uint4*>(s) + 5);               // mn[0..2]
    }
    constexpr long long kOne = 1ll << 42, kHalf = 1ll << 41;

    // sums of this reference by the PARENT's profile frames: interior windows (from the summary) ...
    unsigned K[3] = {0, 0, 0}, U[3] = {0, 0, 0};
    long long RE[3] = {0, 0, 0}, IM[3] = {0, 0, 0};
    unsigned imn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};      // WantMin: minimum window sum by parent frame, interior
    long long count = 0;
    int ormask = 0;
    bool big = false;
    int a0 = 0, a1 = 0, z0 = 0, z1 = 0;         // first two / last two values of the reference in profile order
    if (nz) {
        big = (ku.x >> 31) != 0;
        count = ku.z;
        if (rev) { a0 = edge.w; a1 = edge.z; z0 = edge.y; z1 = edge.x; }
        else { a0 = edge.x; a1 = edge.y; z0 = edge.z; z1 = edge.w; }
        // local frame fl (window start offset inside the atom, mod 3) -> profile frame f:
        //   '+': f = (fl + P) mod 3, so profile frame q holds local frame (q - P) mod 3
        //   '-': f = (len + P - fl) mod 3, so profile frame q holds local frame (len + P - q) mod 3
        const int b = rev ? (int)(rr.z & 3u) : pm3;
        const int i0 = rev ? b : (b == 0 ? 0 : 3 - b);
        const int i1 = rev ? (i0 == 0 ? 2 : i0 - 1) : (i0 == 2 ? 0 : i0 + 1);
        const int i2 = 3 - i0 - i1;
        const bool p00 = i0 == 0, p01 = i0 == 1, p10 = i1 == 0, p11 = i1 == 1, p20 = i2 == 0, p21 = i2 == 1;
        RE[0] = sel3(p00, p01, r01.x, r01.y, r2i0.x); IM[0] = sel3(p00, p01, r2i0.y, i12.x, i12.y);
        RE[1] = sel3(p10, p11, r01.x, r01.y, r2i0.x); IM[1] = sel3(p10, p11, r2i0.y, i12.x, i12.y);
        RE[2] = sel3(p20, p21, r01.x, r01.y, r2i0.x); IM[2] = sel3(p20, p21, r2i0.y, i12.x, i12.y);
        K[0] = (ku.x >> (10 * i0)) & 1023u; K[1] = (ku.x >> (10 * i1)) & 1023u; K[2] = (ku.x >> (10 * i2)) & 1023u;
        U[0] = (ku.y >> (10 * i0)) & 1023u; U[1] = (ku.y >> (10 * i1)) & 1023u; U[2] = (ku.y >> (10 * i2)) & 1023u;
        if (WantMin) {
            imn[0] = sel3(p00, p01, mc.x, mc.y, mc.z);
            imn[1] = sel3(p10, p11, mc.x, mc.y, mc.z);
            imn[2] = sel3(p20, p21, mc.x, mc.y, mc.z);
        }
    } else if (WantMin && valid && len >= 3) {
        // a stretch without a read: frame q has a whole codon inside it when its first window start, (q - P) mod 3
        // values in, leaves room for three values
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const int d = q - pm3, first = d < 0 ? d + 3 : d;
            if (first <= len - 3) imn[q] = 0;
        }
    }

    // ---- the last two profile values before this reference: from the lanes to the left ----
    int p_z0 = __shfl_up_sync(kFull, z0, 1), p_z1 = __shfl_up_sync(kFull, z1, 1), p_len = __shfl_up_sync(kFull, len, 1);
    int pp_z1 = __shfl_up_sync(kFull, z1, 2);
    if (valid && p_ge1 && lane < 2) {
        // only in the groups of a long ORF: the references before this one sit in the group to the left
        auto fetch_tail = [&](long long sl, int& tz0, int& tz1, int& tlen) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(args.refs) + sl);
            tlen = (int)(q.y & kRefLenMask);
            tz0 = tz1 = 0;
            if (q.x != 0xffffffffu && __ldg(args.atom_nonzero + q.x) != 0) {
                const int4 e = __ldg(reinterpret_cast<const int4*>(args.summaries + q.x) + 3);
                if ((q.y & kRefRev) != 0) { tz0 = e.y; tz1 = e.x; } else { tz0 = e.z; tz1 = e.w; }
            }
        };
        int d0, dl;
        if (lane == 0) {
            fetch_tail(slot - 1, p_z0, p_z1, p_len);
            if (p_len < 2 && p_ge2) fetch_tail(slot - 2, d0, pp_z1, dl);
        } else if (p_len < 2 && p_ge2) {
            fetch_tail(slot - 2, d0, pp_z1, dl);
        }
    }
    // ... and the two seam windows: the one that ENDS on the first value of this reference (profile position P - 2)
    // and the one that ends on its second value (P - 1); statistics.py:72-90.  Kept apart: an ORF that STARTS on this
    // reference does not have them.
    unsigned sK[3] = {0, 0, 0}, sU[3] = {0, 0, 0};
    long long sRE[3] = {0, 0, 0}, sIM[3] = {0, 0, 0};
    unsigned smn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};
    if (valid) {
        const int y = p_z1, x = p_len >= 2 ? p_z0 : pp_z1;
#pragma unroll 1
        for (int k = 0; k < 2; ++k) {
            if (k == 0 ? !p_ge2 : !(len >= 2 && p_ge1)) continue;
            const int v0 = k == 0 ? x : y, v1 = k == 0 ? y : a0, v2 = k == 0 ? a0 : a1;
            const int f = k == 0 ? (pm3 == 2 ? 0 : pm3 + 1) : (pm3 == 0 ? 2 : pm3 - 1);     // (P - 2) mod 3, (P - 1) mod 3
            if (WantMin) {
                const unsigned sum = (unsigned)v0 + (unsigned)v1 + (unsigned)v2;
                if (f == 0) smn[0] = min(smn[0], sum); else if (f == 1) smn[1] = min(smn[1], sum); else smn[2] = min(smn[2], sum);
            }
            if ((v0 | v1 | v2) == 0) continue;
            ormask |= v0 | v1 | v2;
            // '+'-oriented triple (a,b,c): the profile of a '-' ORF runs against the plane
            const int a = rev ? v2 : v0, bb = v1, c = rev ? v0 : v2;
            long long re, im;
            unsigned uni = 0;
            if ((bb | c) == 0) { re = kOne; im = 0; }
            else if ((a | c) == 0) { re = -kHalf; im = kHalf; }
            else if ((a | bb) == 0) { re = -kHalf; im = -kHalf; }
            else if (a == bb && bb == c) { re = 0; im = 0; uni = 1; }
            else {
                double2 u;
                if ((unsigned)(a | bb | c) < (unsigned)kUvMax) u = __ldg(args.uv_table + kUvCenter + (a - c) * kUvStride + (bb - c));
                else u = uv_grid((double)(2ll * a - bb - c), (double)((long long)bb - c));
                re = __double2ll_rn(u.x * kUvGridScale);
                im = __double2ll_rn(u.y * kUvGridScale);
            }
            if (f == 0) { sK[0] += 1u; sU[0] += uni; sRE[0] += re; sIM[0] += im; }
            else if (f == 1) { sK[1] += 1u; sU[1] += uni; sRE[1] += re; sIM[1] += im; }
            else { sK[2] += 1u; sU[2] += uni; sRE[2] += re; sIM[2] += im; }
        }
    }
    // the last two values of the family's profile (the trailing partial codon of every member, common.py:177-179)
    const int ty = len >= 1 ? z1 : p_z1, tx = len >= 2 ? z0 : (len == 1 ? (p_ge1 ? p_z1 : 0) : (p_len >= 2 ? p_z0 : pp_z1));
    unsigned tail_mn = 0xffffffffu;
    if (is_long && valid && last) {          // a long ORF: its last group settles the trailing partial codon itself
        if (lm3 == 1) { tail_mn = (unsigned)ty; ormask |= ty; }
        else if (lm3 == 2) { tail_mn = (unsigned)tx + (unsigned)ty; ormask |= tx | ty; }
    }
    big |= (ormask >> kBigShift) != 0;

    // ---- suffix sums over the lanes of every family (consecutive lanes) ----
    const unsigned heads = __ballot_sync(kFull, lane == 0 || !valid || (rr.z & kRefFamilyHead) != 0);
    const unsigned after = lane == 31 ? 0u : heads >> (lane + 1);
    const int end_lane = after ? lane + __ffs(after) : 32;              // lanes [.., end_lane) belong to my family
    const bool head = ((heads >> lane) & 1u) != 0;
    const int max_run = (int)__reduce_max_sync(kFull, head ? (unsigned)(end_lane - lane) : 0u);
    long long TRE[3], TIM[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) { TRE[q] = RE[q] + sRE[q]; TIM[q] = IM[q] + sIM[q]; }
    unsigned long long Kp = (unsigned long long)(K[0] + sK[0]) | ((unsigned long long)(K[1] + sK[1]) << 21) | ((unsigned long long)(K[2] + sK[2]) << 42);
    unsigned long long Up = (unsigned long long)(U[0] + sU[0]) | ((unsigned long long)(U[1] + sU[1]) << 21) | ((unsigned long long)(U[2] + sU[2]) << 42);
    unsigned flags = big ? 1u : 0u;
    unsigned tmn[3] = {min(imn[0], smn[0]), min(imn[1], smn[1]), min(imn[2], smn[2])};
    if (WantMin && is_long) tmn[0] = min(tmn[0], tail_mn);              // a long ORF is its own parent: frame 0 is frame 0
    for (int o = 1; o < max_run; o <<= 1) {
        const bool take = lane + o < end_lane;
        const long long t0 = __shfl_down_sync(kFull, TRE[0], o), t1 = __shfl_down_sync(kFull, TRE[1], o);
        const long long t2 = __shfl_down_sync(kFull, TRE[2], o), t3 = __shfl_down_sync(kFull, TIM[0], o);
        const long long t4 = __shfl_down_sync(kFull, TIM[1], o), t5 = __shfl_down_sync(kFull, TIM[2], o);
        const unsigned long long tk = __shfl_down_sync(kFull, Kp, o), tu = __shfl_down_sync(kFull, Up, o);
        const long long tc = __shfl_down_sync(kFull, count, o);
        const unsigned tf = __shfl_down_sync(kFull, flags, o);
        if (take) {
            TRE[0] += t0; TRE[1] += t1; TRE[2] += t2; TIM[0] += t3; TIM[1] += t4; TIM[2] += t5;
            Kp += tk; Up += tu; count += tc; flags |= tf;
        }
        if (WantMin) {
            const unsigned m0 = __shfl_down_sync(kFull, tmn[0], o), m1 = __shfl_down_sync(kFull, tmn[1], o), m2 = __shfl_down_sync(kFull, tmn[2], o);
            if (take) { tmn[0] = min(tmn[0], m0); tmn[1] = min(tmn[1], m1); tmn[2] = min(tmn[2], m2); }
        }
    }
    // the family's last two values, for the members that start further left
    const int f_tx = __shfl_sync(kFull, tx, end_lane - 1), f_ty = __shfl_sync(kFull, ty, end_lane - 1);
    // minima of the lanes to the right of this one (an ORF starting here has its own interior windows, not its seam ones)
    unsigned xmn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};
    if (WantMin) {
        const unsigned m0 = __shfl_down_sync(kFull, tmn[0], 1), m1 = __shfl_down_sync(kFull, tmn[1], 1), m2 = __shfl_down_sync(kFull, tmn[2], 1);
        if (lane + 1 < end_lane) { xmn[0] = m0; xmn[1] = m1; xmn[2] = m2; }
    }
    const unsigned kMask = (1u << 21) - 1u;
    if (is_long) {
        // one group of a long ORF: integer atomics into the ORF's accumulator; the last group to arrive scores it
        if (lane != 0) return;
        unsigned Kt[3] = {(unsigned)Kp & kMask, (unsigned)(Kp >> 21) & kMask, (unsigned)(Kp >> 42) & kMask};
        unsigned Ut[3] = {(unsigned)Up & kMask, (unsigned)(Up >> 21) & kMask, (unsigned)(Up >> 42) & kMask};
        LongAcc* acc = args.long_acc + rw.long_idx;
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            atomicAdd(&acc->RE[f], (unsigned long long)TRE[f]);
            atomicAdd(&acc->IM[f], (unsigned long long)TIM[f]);
            atomicAdd(&acc->K[f], Kt[f]);
            atomicAdd(&acc->U[f], Ut[f]);
        }
        atomicAdd(&acc->count, (unsigned long long)count);
        if (WantMin) atomicMin(&acc->mn, tmn[0]);
        if (flags) atomicOr(&acc->big, 1u);
        __threadfence();
        if (atomicAdd(&acc->done, 1u) != (unsigned)(rw.n_groups - 1)) return;
        __threadfence();
        volatile LongAcc* va = acc;
        long long RE2[3], IM2[3];
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            RE2[f] = (long long)va->RE[f]; IM2[f] = (long long)va->IM[f]; Kt[f] = va->K[f]; Ut[f] = va->U[f];
            va->RE[f] = 0; va->IM[f] = 0; va->K[f] = 0; va->U[f] = 0;
        }
        const long long cnt2 = (long long)va->count;
        const unsigned mn2 = va->mn;
        const bool big2 = va->big != 0;
        va->count = 0; va->mn = 0xffffffffu; va->big = 0; va->done = 0;      // ready for the next launch
        const int L = __ldg(args.orf_len + rw.orf);
        if (big2 || L > 3 * kMaxExactCodons) {
            args.fallback[atomicAdd(args.n_fallback, 1u)] = rw.orf;
            return;
        }
        finish_orf_lean(args, rw.orf, L, Kt, Ut, RE2, IM2, mn2, cnt2);
        return;
    }
    if (orf < 0) return;                    // no ORF starts on this reference
    // ---- the ORF that starts here: suffix sums without this reference's seam windows, in the ORF's own frames ----
    const int L = __ldg(args.orf_len + orf);
    unsigned long long sKp = (unsigned long long)sK[0] | ((unsigned long long)sK[1] << 21) | ((unsigned long long)sK[2] << 42);
    unsigned long long sUp = (unsigned long long)sU[0] | ((unsigned long long)sU[1] << 21) | ((unsigned long long)sU[2] << 42);
    Kp -= sKp;                              // field-wise: the seam windows of this lane are part of its suffix sums
    Up -= sUp;
    unsigned Kq[3] = {(unsigned)Kp & kMask, (unsigned)(Kp >> 21) & kMask, (unsigned)(Kp >> 42) & kMask};
    unsigned Uq[3] = {(unsigned)Up & kMask, (unsigned)(Up >> 21) & kMask, (unsigned)(Up >> 42) & kMask};
#pragma unroll
    for (int q = 0; q < 3; ++q) { TRE[q] -= sRE[q]; TIM[q] -= sIM[q]; }
    // frame q of this ORF is frame (q + P) mod 3 of the parent
    const int j0 = pm3, j1 = pm3 == 2 ? 0 : pm3 + 1, j2 = 3 - j0 - j1;
    const bool q00 = j0 == 0, q01 = j0 == 1, q10 = j1 == 0, q11 = j1 == 1, q20 = j2 == 0, q21 = j2 == 1;
    unsigned Ko[3] = {sel3(q00, q01, Kq[0], Kq[1], Kq[2]), sel3(q10, q11, Kq[0], Kq[1], Kq[2]), sel3(q20, q21, Kq[0], Kq[1], Kq[2])};
    unsigned Uo[3] = {sel3(q00, q01, Uq[0], Uq[1], Uq[2]), sel3(q10, q11, Uq[0], Uq[1], Uq[2]), sel3(q20, q21, Uq[0], Uq[1], Uq[2])};
    long long REo[3] = {sel3(q00, q01, TRE[0], TRE[1], TRE[2]), sel3(q10, q11, TRE[0], TRE[1], TRE[2]), sel3(q20, q21, TRE[0], TRE[1], TRE[2])};
    long long IMo[3] = {sel3(q00, q01, TIM[0], TIM[1], TIM[2]), sel3(q10, q11, TIM[0], TIM[1], TIM[2]), sel3(q20, q21, TIM[0], TIM[1], TIM[2])};
    unsigned mn = 0xffffffffu;
    bool big_o = flags != 0 || L > 3 * kMaxExactCodons;
    if (WantMin) {
        mn = min(sel3(q00, q01, imn[0], imn[1], imn[2]), sel3(q00, q01, xmn[0], xmn[1], xmn[2]));       // this ORF's frame 0
        if (lm3 == 1) mn = min(mn, (unsigned)f_ty);
        else if (lm3 == 2) mn = min(mn, (unsigned)f_tx + (unsigned)f_ty);
    }
    if (lm3 == 1) big_o |= (f_ty >> kBigShift) != 0;
    else if (lm3 == 2) big_o |= ((f_tx | f_ty) >> kBigShift) != 0;
    if (big_o) {
        args.fallback[atomicAdd(args.n_fallback, 1u)] = orf;
        return;
    }
    finish_orf_lean(args, orf, L, Ko, Uo, REo, IMo, mn, count);
}

// ---- K4 -------------------------------------------------------------------------------------
struct GatherArgs {
    const int32_t* cov;
    const uint64_t* orf_desc;
    const uint64_t* exon_entries;
    const int64_t* orf_ids;
    const int64_t* out_ptr;
    int32_t* out;
    long long n_sel;
};

__global__ void __launch_bounds__(256) gather_profiles_kernel(const GatherArgs args) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp0; i < args.n_sel; i += nwarps) {
        const uint64_t desc = __ldg(args.orf_desc + args.orf_ids[i]);
        ExonCursor cur;
        cur.entries = args.exon_entries + (desc & kBeginMask);
        cur.n = (int)((desc >> 40) & kMaxEntriesPerOrf);
        cur.rev = (desc >> 63) != 0;
        int32_t* dst = args.out + args.out_ptr[i];
        while (cur.advance(lane)) {
            const int take = cur.rem;
            if (cur.zero) {
                for (int k = lane; k < take; k += 32) dst[k] = 0;
            } else if (cur.rev) {
                const int32_t* src = args.cov + cur.pos;
                for (int k = lane; k < take; k += 32) dst[k] = ld_cov(src - k);
            } else {
                const int32_t* src = args.cov + cur.pos;
                for (int k = lane; k < take; k += 32) dst[k] = ld_cov(src + k);
            }
            dst += take;
            cur.rem = 0;
        }
    }
}

// ---- interval sums (count_orfs.py:28-89 on device results) ------------------------------------
// One warp per interval of the dense planes: its coverage sum is added to the group (= gene) it belongs to.
__global__ void __launch_bounds__(256) interval_sum_kernel(const int32_t* __restrict__ cov, long long n_iv,
                                                            const long long* __restrict__ iv_off,
                                                            const int32_t* __restrict__ iv_len,
                                                            const int32_t* __restrict__ iv_group,
                                                            unsigned long long* sums) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp0; i < n_iv; i += nwarps) {
        const int32_t* src = cov + iv_off[i];
        const int len = iv_len[i];
        long long acc = 0;
        for (int k = lane; k < len; k += 32) acc += ld_cov(src + k);
        acc = warp_sum_i64(acc);
        if (lane == 0 && acc != 0) atomicAdd(sums + iv_group[i], (unsigned long long)acc);
    }
}

// ---- bootstrap medians (learn_cutoff.py:88-98) -------------------------------------------------
// np.median(values[idx], axis=0) for idx of shape (n_sel, reps): one block per replicate gathers its n_sel
// values as order-preserving 64-bit keys (shared memory when they fit, else a global scratch row) and finds
// the middle order statistic(s) by a 64-step bisection on the key bits -- no sort.
__device__ __forceinline__ unsigned long long f64_key(double v) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(unsigned long long k) {
    const unsigned long long u = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)u);
}
__global__ void __launch_bounds__(256) bootstrap_median_kernel(const double* __restrict__ values,
                                                                const long long* __restrict__ idx, long long n_sel,
                                                                long long reps, unsigned long long* scratch,
                                                                int keys_in_smem, double* out) {
    extern __shared__ unsigned long long s_keys[];
    __shared__ long long s_part[8];
    const long long r = blockIdx.x;
    unsigned long long* keys = keys_in_smem ? s_keys : scratch + r * n_sel;
    for (long long i = threadIdx.x; i < n_sel; i += blockDim.x) keys[i] = f64_key(values[idx[i * reps + r]]);
    __syncthreads();
    auto count_below = [&](unsigned long long cand) {      // block-wide number of keys < cand
        long long c = 0;
        for (long long i = threadIdx.x; i < n_sel; i += blockDim.x) c += keys[i] < cand;
        c = warp_sum_i64(c);
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = c;
        __syncthreads();
        long long tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) tot += s_part[w];
        __syncthreads();
        return tot;
    };
    auto kth = [&](long long k) {                          // k-th smallest key (0-based): largest R with count(< R) <= k
        unsigned long long res = 0;
        for (int bit = 63; bit >= 0; --bit) {
            const unsigned long long cand = res | (1ull << bit);
            if (count_below(cand) <= k) res = cand;
        }
        return res;
    };
    double med;
    if (n_sel & 1) med = key_f64(kth(n_sel / 2));
    else med = (key_f64(kth(n_sel / 2 - 1)) + key_f64(kth(n_sel / 2))) * 0.5;     // np.mean of the two middle values
    if (threadIdx.x == 0) out[r] = med;
}

// ---- K1 -------------------------------------------------------------------------------------
struct BinArgs {
    int32_t* cov;
    const int32_t* ref_id;
    const int32_t* first;
    const int32_t* last;
    const uint16_t* mlen;
    const uint16_t* flag;
    const uint8_t* mapq;
    const uint8_t* nh;
    long long n;
    int protocol;
    int weight;                    // +1 bin, -1 un-bin
    int len_base;                  // lengths [len_base, len_base + 16) are counted in registers
    unsigned long long* touched;   // optional: every 32 B sector (slot >> 3) that received an atomic (duplicates allowed)
    unsigned long long* n_touched;
    const uint2* cmap;             // compact layout: per 32 dense slots (member mask, compact index after the last member)
    const unsigned* cbits;         // compact layout: one bit per cmap word, set when the word has members (L2 resident)
    const int32_t* len_table;      // RT_LEN_TABLE
    const int2* contig_tab;        // n_contig x (length, first slot of the contig >> 5)
    int n_contig;
    int pad;
    unsigned plane_words;          // plane >> 5
    unsigned long long* stats;       // RT_N_STATS
    unsigned long long* len_counts;  // RT_LEN_TABLE
};

constexpr int kBinThreads = 256;
constexpr int kBinReadsPerThread = 8;
constexpr int kLenHist = 512;   // read lengths below this are histogrammed in shared memory

// Category of one read after the cascade of bam.py:77-91: one of RT_ST_QCFAIL .. RT_ST_VALID.
// The four flag tests are one lookup: index = unmapped | secondary << 1 | qcfail << 2 | duplicate << 3.
__host__ __device__ constexpr unsigned long long flag_cascade_lut() {
    unsigned long long t = 0;
    for (int i = 0; i < 16; ++i) {
        int cat = 0;
        if (i & 4) cat = RT_ST_QCFAIL;           // bam.py:77
        else if (i & 8) cat = RT_ST_DUPLICATE;   // bam.py:80
        else if (i & 2) cat = RT_ST_SECONDARY;   // bam.py:83
        else if (i & 1) cat = RT_ST_UNMAPPED;    // bam.py:86
        t |= (unsigned long long)cat << (4 * i);
    }
    return t;
}
__device__ __forceinline__ int classify_read(unsigned fl, unsigned mapq, unsigned nh) {
    constexpr unsigned long long kLut = flag_cascade_lut();
    const unsigned idx = ((fl >> 2) & 1u) | ((fl >> 7) & 0xeu);
    const int cat = (int)((kLut >> (4 * idx)) & 15ull);
    // is_read_uniq_mapping, common.py:33-69 (None is falsy -> counted as multi, bam.py:89):
    // NH present decides (common.py:54-56), else only MAPQ 255 is unique (common.py:59-69)
    const bool uniq = nh != 0 ? nh == 1 : mapq == 255;
    return cat ? cat : (uniq ? RT_ST_VALID : RT_ST_MULTI);
}

template <bool Compact>
__global__ void __launch_bounds__(kBinThreads) bin_psites_kernel(const BinArgs a) {
    __shared__ unsigned int s_stats[RT_N_STATS];
    __shared__ unsigned int s_len[kLenHist];
    __shared__ unsigned long long s_touch[Compact ? 1 : kBinThreads * kBinReadsPerThread];
    __shared__ unsigned int s_ntouch;
    __shared__ unsigned long long s_touch_base;
    if (threadIdx.x == 0) s_ntouch = 0;
    for (int i = threadIdx.x; i < kLenHist; i += kBinThreads) s_len[i] = 0;
    if (threadIdx.x < RT_N_STATS) s_stats[threadIdx.x] = 0;
    __syncthreads();

    using slot_t = typename std::conditional<Compact, unsigned, long long>::type;
    constexpr slot_t kNone = (slot_t)-1;
    const int lane = threadIdx.x & 31;
    const long long block_base = (long long)blockIdx.x * (kBinThreads * kBinReadsPerThread);
    // per-thread 4-bit counters of categories RT_ST_QCFAIL..RT_ST_BADREF (<= 8 reads per thread)
    unsigned packed = 0;
    unsigned long long len_packed = 0;
    constexpr int kBatch = 4;                // reads per thread whose columns are in flight together
#pragma unroll 1
    for (int it0 = 0; it0 < kBinReadsPerThread; it0 += kBatch) {
        // ---- all column loads of the batch first (7 x kBatch independent, coalesced loads) ----
        unsigned fl[kBatch], mq[kBatch], nh[kBatch], ml[kBatch];
        int fi[kBatch], la[kBatch], rid[kBatch];
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
            const long long i = block_base + (long long)(it0 + j) * kBinThreads + threadIdx.x;
            const bool in = i < a.n;
            fl[j] = in ? a.flag[i] : 0u;
            mq[j] = in ? a.mapq[i] : 0u;
            nh[j] = in ? a.nh[i] : 0u;
            rid[j] = in ? a.ref_id[i] : 0;
            ml[j] = in ? a.mlen[i] : 0u;
            fi[j] = in ? a.first[i] : 0;
            la[j] = in ? a.last[i] : 0;
        }
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
            const long long i = block_base + (long long)(it0 + j) * kBinThreads + threadIdx.x;
            int len = -1;            // >= 0: counts in read_length_counts
            slot_t slot = kNone;     // coverage slot to bump
            if (i < a.n) {
                int cat = classify_read(fl[j], mq[j], nh[j]);
                const bool rev = (fl[j] & 0x10) != 0;               // bam.py:94
                if (cat == RT_ST_VALID) {
                    const int l = (int)ml[j];                       // bam.py:99
                    const int mode = __ldg(a.len_table + l);
                    // forward protocol: '+' reads sit on their 5' end = first position (bam.py:105-117);
                    // reverse protocol swaps the strand and takes the other end (bam.py:118-131)
                    const bool minus = rev == (a.protocol == RT_PROTOCOL_FORWARD);
                    const int pos = minus ? la[j] : fi[j];
                    const int c = rid[j];
                    if (mode == RT_LEN_FILTERED || a.protocol > RT_PROTOCOL_REVERSE) {
                        cat = 0;                                    // bam.py:101 / no protocol branch: only `total`
                    } else if ((unsigned)c >= (unsigned)a.n_contig) {
                        cat = RT_ST_BADREF;                         // chrom is None, bam.py:133
                    } else {
                        len = l;                                    // bam.py:136
                        if (mode != RT_LEN_UNUSED) {                // detect_orfs.py:74 (the offset may be negative)
                            const int2 ct = __ldg(a.contig_tab + c);
                            // 1-based P-site p = pos + 1 +- offset (bam.py:135, detect_orfs.py:78-81);
                            // q = p + pad - 1 is its 0-based place in the padded contig
                            const unsigned q = (unsigned)(pos + (minus ? -mode : mode) + a.pad);
                            if (q >= (unsigned)(ct.x + 2 * a.pad)) {
                                atomicAdd(&s_stats[RT_ST_OOB], 1u);
                            } else {
                                const unsigned in_contig = q + 1u;                      // pad + p
                                const unsigned w = (minus ? a.plane_words : 0u) + (unsigned)ct.y + (in_contig >> 5);
                                const unsigned bit = in_contig & 31u;
                                if (Compact) {   // rank of the slot inside the exon union, or no slot at all
                                    if ((__ldg(a.cbits + (w >> 5)) >> (w & 31u)) & 1u) {
                                        const uint2 m = __ldg(a.cmap + w);
                                        const unsigned above = m.x >> bit;
                                        if (above & 1u) slot = (slot_t)(m.y - (unsigned)__popc(above));
                                    }
                                } else {
                                    slot = (slot_t)(((unsigned long long)w << 5) | bit);
                                }
                            }
                        }
                    }
                }
                if (cat) packed += 1u << (4 * (cat - 1));
            }
            // detect_orfs.py:82: duplicated 5' ends are the rule in Ribo-seq and adjacent in a
            // coordinate-sorted BAM: the first lane of every run of equal slots adds the run length
            const slot_t prev = __shfl_up_sync(kFull, slot, 1);
            const bool head = lane == 0 || slot != prev;
            const unsigned heads = __ballot_sync(kFull, head);
            if (head && slot != kNone) {
                const unsigned after = lane == 31 ? 0u : heads >> (lane + 1);
                const int run = after ? __ffs(after) : 32 - lane;
                atomicAdd(a.cov + slot, a.weight * run);
            }
            if (!Compact && a.touched) {   // remember the 32 B sector so the planes can be cleared sparsely afterwards
                const long long sec = slot != kNone ? (long long)(slot >> 3) : -1;
                const long long prev_sec = __shfl_up_sync(kFull, sec, 1);
                const bool shead = sec >= 0 && (lane == 0 || sec != prev_sec);
                const unsigned writers = __ballot_sync(kFull, shead);
                unsigned base = 0;
                if (lane == 0 && writers) base = atomicAdd(&s_ntouch, (unsigned)__popc(writers));
                base = __shfl_sync(kFull, base, 0);
                if (shead) s_touch[base + __popc(writers & ((1u << lane) - 1u))] = (unsigned long long)sec;
            }
            // bam.py:136: per-thread 4-bit counters for the 16 lengths from len_base on
            if (len >= 0) {
                const unsigned d = (unsigned)(len - a.len_base);
                if (d < 16u) len_packed += 1ull << (4 * d);
                else if (len < kLenHist) atomicAdd(&s_len[len], 1u);
                else atomicAdd(a.len_counts + len, (unsigned long long)(long long)a.weight);
            }
        }
    }
    {   // flush the register length counters: one REDUX per length, one shared atomic per lane
        unsigned mine_len = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const unsigned v = __reduce_add_sync(kFull, (unsigned)(len_packed >> (4 * k)) & 15u);
            if (lane == k) mine_len = v;
        }
        const int l = a.len_base + lane;
        if (lane < 16 && mine_len && l >= 0) {
            if (l < kLenHist) atomicAdd(&s_len[l], mine_len);
            else atomicAdd(a.len_counts + l, (unsigned long long)((long long)a.weight * mine_len));
        }
    }
    // bam.py:61,73-91,137: categories RT_ST_QCFAIL (slot 1) .. RT_ST_BADREF (slot 8), minus OOB
    unsigned mine = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const unsigned v = __reduce_add_sync(kFull, (packed >> (4 * k)) & 15u);
        if (lane == k) mine = v;
    }
    if (lane < 8 && mine) atomicAdd(&s_stats[1 + lane], mine);
    if (threadIdx.x == 0) {
        const long long left = a.n - block_base;
        s_stats[RT_ST_TOTAL] = (unsigned)(left < kBinThreads * kBinReadsPerThread ? left : kBinThreads * kBinReadsPerThread);
    }
    __syncthreads();
    if (!Compact && a.touched) {   // one global atomic per block, then a coalesced copy of the block's slots
        if (threadIdx.x == 0) s_touch_base = atomicAdd(a.n_touched, (unsigned long long)s_ntouch);
        __syncthreads();
        for (unsigned i = threadIdx.x; i < s_ntouch; i += kBinThreads) a.touched[s_touch_base + i] = s_touch[i];
    }
    // two's-complement wrap makes weight = -1 subtract
    if (threadIdx.x < RT_N_STATS && s_stats[threadIdx.x])
        atomicAdd(a.stats + threadIdx.x, (unsigned long long)((long long)a.weight * s_stats[threadIdx.x]));
    for (int i = threadIdx.x; i < kLenHist; i += kBinThreads)
        if (s_len[i]) atomicAdd(a.len_counts + i, (unsigned long long)((long long)a.weight * s_len[i]));
}

// ---- K1 on a record stream ----------------------------------------------------------------------------
// A coordinate-sorted library as 4-byte delta-coded records in blocks of RT_STREAM_BLOCK (format: ribotricer_b200.h).
// One warp per block: a lane takes 8 consecutive records (two 128-bit loads), positions come from a warp-wide
// prefix sum over the records' advances, the contig is a property of the block.  The filter cascade (bam.py:77-91,
// common.py:33-69) is one shared-memory lookup on the 7 raw bits the record carries; runs of equal slots are merged
// inside the thread's strip (duplicated 5' ends are adjacent in a sorted library) before the RED.
struct StreamArgs {
    int32_t* cov;
    const uint4* rec;              // n_blocks * RT_STREAM_BLOCK records
    const int4* hdr;               // per block: (ref_id, position the deltas start from, 0, 0)
    long long n_blocks;
    // zoned launch (rt_bin_stream_fresh): zone_bounds[s * (n_blocks + 1) + b] = first compact slot of block b's zone on
    // strand s; the block zero-fills [bounds[b], bounds[b + 1]) before it adds its own reads there, reads that fall
    // outside go to the spill list and are added once every zone has been written
    const unsigned* zone_bounds;
    const unsigned* zone_carry;    // per strand and tile of kZoneTile boundaries: the maximum of all boundaries before the tile
    long long zone_tiles;
    unsigned* spill;
    unsigned long long* n_spill;
    int protocol;
    int weight;
    int len_base;
    const uint2* cmap;
    const unsigned* cbits;
    const int32_t* len_table;
    const int2* contig_tab;
    int n_contig;
    int pad;
    unsigned plane_words;
    unsigned long long* stats;
    unsigned long long* len_counts;
};

constexpr int kStreamThreads = 256;
constexpr int kStreamWarps = kStreamThreads / 32;
constexpr int kStreamStrip = RT_STREAM_BLOCK / 32;                  // records per lane: one warp takes one block
static_assert(kStreamStrip == 8, "bin_stream_kernel loads a strip as two uint4");

__device__ __forceinline__ unsigned shl_clamp(unsigned v, unsigned s) {   // PTX shl: shift amounts above 31 give 0
    unsigned r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(s));
    return r;
}

constexpr int kStreamModes = 512;       // read lengths below this find their offset in shared memory
constexpr int kStreamFastLens = 256;    // a read without an extension record is shorter than this
constexpr unsigned kShValid = 4u * RT_ST_VALID - 4u;
constexpr int kFastCounted = 1, kFastBinned = 2, kFastNoCounter = 4;    // low bits of a fast-path entry's y

// Slots of the strip's records -> coverage.  detect_orfs.py:82 with duplicates merged: one RED per run of equal slots.
template <typename slot_t>
__device__ __forceinline__ void stream_scatter(int32_t* cov, const slot_t (&slot)[kStreamStrip], int weight) {
    constexpr slot_t kNone = (slot_t)-1;
    slot_t cur = kNone;
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kStreamStrip; ++j) {
        if (slot[j] != cur) {
            if (cur != kNone) atomicAdd(cov + cur, weight * cnt);
            cur = slot[j];
            cnt = 0;
        }
        ++cnt;
    }
    if (cur != kNone) atomicAdd(cov + cur, weight * cnt);
}

// (word, bit) of the dense slot -> slot of the current layout (compact: through the member bitmap and the rank word)
template <bool Compact, typename slot_t>
__device__ __forceinline__ void stream_slots(const StreamArgs& a, unsigned live, const unsigned (&wd)[kStreamStrip],
                                             const unsigned (&bit)[kStreamStrip], slot_t (&slot)[kStreamStrip]) {
    constexpr slot_t kNone = (slot_t)-1;
    if (Compact) {
        unsigned cb[kStreamStrip];
#pragma unroll
        for (int j = 0; j < kStreamStrip; ++j) cb[j] = (live >> j) & 1u ? __ldg(a.cbits + (wd[j] >> 5)) : 0u;
#pragma unroll
        for (int h = 0; h < kStreamStrip; h += 4) {      // the rank words of four records in flight together
            uint2 m[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                m[j] = ((cb[h + j] >> (wd[h + j] & 31u)) & 1u) ? __ldg(a.cmap + wd[h + j]) : make_uint2(0u, 0u);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const unsigned above = m[j].x >> bit[h + j];
                slot[h + j] = (above & 1u) ? (slot_t)(m[j].y - (unsigned)__popc(above)) : kNone;
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < kStreamStrip; ++j)
            slot[j] = (live >> j) & 1u ? (slot_t)(((unsigned long long)wd[j] << 5) | bit[j]) : kNone;
    }
}

constexpr int kStreamContigs = 256;     // contig table entries kept in shared memory
constexpr int kStreamCtasPerSm = 3;

// Zero the compact slots [z0, z1): 16-byte stores where the range is aligned, single slots at its two ends.
__device__ __forceinline__ void stream_zero_zone(int32_t* cov, unsigned z0, unsigned z1, int lane) {
    if (z1 <= z0) return;
    const unsigned a0 = min((z0 + 3u) & ~3u, z1), a1 = max(z1 & ~3u, a0);     // [a0, a1) is whole int4s
    if (z0 + (unsigned)lane < a0) cov[z0 + lane] = 0;
    int4* v = reinterpret_cast<int4*>(cov);
    for (unsigned i = (a0 >> 2) + lane; i < (a1 >> 2); i += 32) v[i] = make_int4(0, 0, 0, 0);
    if (a1 + (unsigned)lane < z1) cov[a1 + lane] = 0;
}

// Lower-bound rank: compact index of the first member slot at or after bit `bit` of dense word `w` (after
// fill_cmap_gaps an empty word carries the index its next member will get).
__device__ __forceinline__ unsigned cmap_rank(const uint2* cmap, unsigned w, unsigned bit) {
    const uint2 m = __ldg(cmap + w);
    return m.y - (unsigned)__popc(m.x >> bit);
}

// Zone boundaries of a stream: boundary of block b on strand s = rank of the first position a read of the block can
// put a P-site on (its header position + the smallest offset of the strand).  Blocks without a usable reference get the
// strand's first slot and inherit their predecessor's boundary through the prefix maximum.
struct ZoneArgs {
    const int4* hdr;
    long long n_blocks;
    unsigned* bounds;              // 2 x (n_blocks + 1)
    const uint2* cmap;
    const int2* contig_tab;
    int n_contig;
    int pad;
    unsigned plane_words;
    int delta_plus, delta_minus;   // smallest P-site displacement from `first` on either strand
    unsigned plus_end, minus_end;  // compact index after the last '+' / '-' slot
};
constexpr int kZoneTile = 256;      // boundaries per CTA of zone_bounds_kernel
static_assert(kZoneTile == 256, "bin_stream_kernel finds the tile of a boundary with >> 8");
// grid (tiles, 2 strands): raw boundaries clamped to the strand's range, then the prefix maximum inside the tile;
// tile_max[s * tiles + t] = the tile's maximum.  zone_carry_kernel turns those into the carry of every tile, and
// whoever reads boundary b takes max(bounds[b], tile_carry[tile of b]): monotone whatever the stream looks like.
__global__ void __launch_bounds__(kZoneTile) zone_bounds_kernel(const ZoneArgs z, unsigned* tile_max) {
    __shared__ unsigned s_w[kZoneTile / 32];
    const int s = blockIdx.y;
    const long long b = (long long)blockIdx.x * kZoneTile + threadIdx.x;
    const unsigned lo = s ? z.plus_end : 0u, hi = s ? z.minus_end : z.plus_end;
    unsigned r = lo;
    if (b >= z.n_blocks) r = b == z.n_blocks ? hi : lo;
    else if (b > 0) {
        const int4 hd = __ldg(z.hdr + b);
        if ((unsigned)hd.x < (unsigned)z.n_contig) {
            const int2 ct = __ldg(z.contig_tab + hd.x);
            long long q = (long long)hd.y + (s ? z.delta_minus : z.delta_plus) + z.pad + 1;    // in_contig of the first reachable P-site
            q = q < 0 ? 0 : (q > (long long)ct.x + 2 * z.pad ? (long long)ct.x + 2 * z.pad : q);
            const unsigned w = (s ? z.plane_words : 0u) + (unsigned)ct.y + (unsigned)(q >> 5);
            r = min(max(cmap_rank(z.cmap, w, (unsigned)(q & 31)), lo), hi);
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(kFull, r, o);
        if (lane >= o) r = max(r, t);
    }
    if (lane == 31) s_w[warp] = r;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kZoneTile / 32 - 1; ++k)
        if (k < warp) r = max(r, s_w[k]);
    if (b <= z.n_blocks) z.bounds[(size_t)s * (size_t)(z.n_blocks + 1) + (size_t)b] = r;
    if (threadIdx.x == kZoneTile - 1) tile_max[(size_t)s * gridDim.x + blockIdx.x] = r;
}
// One CTA per strand: exclusive prefix maximum over the tile maxima.
__global__ void __launch_bounds__(1024) zone_carry_kernel(const unsigned* __restrict__ tile_max, unsigned* tile_carry, long long tiles,
                                                          unsigned plus_end) {
    __shared__ unsigned s_max[1024];
    const unsigned* in = tile_max + (size_t)blockIdx.x * (size_t)tiles;
    unsigned* out = tile_carry + (size_t)blockIdx.x * (size_t)tiles;
    const unsigned lo = blockIdx.x ? plus_end : 0u;
    const long long per = (tiles + 1023) / 1024;
    const long long t0 = (long long)threadIdx.x * per, t1 = t0 + per < tiles ? t0 + per : tiles;
    unsigned m = lo;
    for (long long t = t0; t < t1; ++t) m = max(m, in[t]);
    s_max[threadIdx.x] = m;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const unsigned v = threadIdx.x >= o ? s_max[threadIdx.x - o] : 0u;
        __syncthreads();
        s_max[threadIdx.x] = max(s_max[threadIdx.x], v);
        __syncthreads();
    }
    m = threadIdx.x ? s_max[threadIdx.x - 1] : lo;
    for (long long t = t0; t < t1; ++t) {
        out[t] = m;
        m = max(m, in[t]);
    }
}
// The P-sites that fell outside their block's zone, once every zone has been written.
__global__ void __launch_bounds__(256) zone_spill_kernel(int32_t* cov, const unsigned* __restrict__ spill, const unsigned long long* n_spill) {
    const unsigned long long n = *n_spill;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
        atomicAdd(cov + spill[i], 1);
}

// Persistent: kStreamCtasPerSm CTAs per SM; every WARP walks blocks of the stream on its own (no CTA-wide barrier
// after start-up, so the warps of an SM drift apart and cover each other's load latencies).  A warp owns a ring of two
// shared-memory stages with one mbarrier each: an elected lane brings block i + 1 (1 KB of records and its header) in
// with a cp.async.bulk pair while the warp works on block i.  The lookup tables are built once per CTA and the
// per-thread 4-bit counters are drained into 8-bit ones every block.
template <bool Compact, bool Zoned>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm) bin_stream_kernel(const StreamArgs a) {
    static_assert(Compact || !Zoned, "zones are ranges of the compact buffer");
    __shared__ __align__(128) unsigned int s_rec[kStreamWarps][2][RT_STREAM_BLOCK];
    __shared__ __align__(16) int4 s_hdr[kStreamWarps][2];
    __shared__ __align__(8) uint64_t s_bar[kStreamWarps][2];
    __shared__ unsigned int s_stats[RT_N_STATS];
    __shared__ unsigned int s_len[kLenHist];
    __shared__ int s_mode[kStreamModes];
    // fast path, per read length: (offset of a '+' P-site from `first`, of a '-' one and flags, the length's 4-bit counter as two words)
    __shared__ int4 s_fast[kStreamFastLens];
    __shared__ int2 s_ctab[kStreamContigs];
    __shared__ uint8_t s_cat[128];
    __shared__ uint8_t s_sh[256];       // fast path: 4 * category - 4 of a record's meta byte
    if ((threadIdx.x & 31) == 0) {
        mbar_init(&s_bar[threadIdx.x >> 5][0], 1);
        mbar_init(&s_bar[threadIdx.x >> 5][1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < kLenHist; i += kStreamThreads) s_len[i] = 0;
    for (int i = threadIdx.x; i < kStreamModes; i += kStreamThreads) s_mode[i] = __ldg(a.len_table + i);
    for (int i = threadIdx.x; i < kStreamContigs && i < a.n_contig; i += kStreamThreads) s_ctab[i] = __ldg(a.contig_tab + i);
    if (threadIdx.x < RT_N_STATS) s_stats[threadIdx.x] = 0;
    {   // the cascade on the record's raw bits, once per CTA
        const unsigned m = threadIdx.x & 127u, st = (m >> 5) & 3u;
        int cat;
        if (m & RT_STREAM_QCFAIL) cat = RT_ST_QCFAIL;             // bam.py:77
        else if (m & RT_STREAM_DUPLICATE) cat = RT_ST_DUPLICATE;  // bam.py:80
        else if (m & RT_STREAM_SECONDARY) cat = RT_ST_SECONDARY;  // bam.py:83
        else if (m & RT_STREAM_UNMAPPED) cat = RT_ST_UNMAPPED;    // bam.py:86
        else cat = (st == RT_STREAM_NH_ONE || st == RT_STREAM_NH_ABSENT_MAPQ255) ? RT_ST_VALID : RT_ST_MULTI;   // common.py:53-69
        if (threadIdx.x < 128) s_cat[m] = (uint8_t)cat;
        s_sh[threadIdx.x] = (uint8_t)(4 * cat - 4);
    }
    {   // fast-path entry of read length l = threadIdx.x
        const int l = threadIdx.x;
        const int mode = __ldg(a.len_table + l);
        const unsigned dl = (unsigned)(l - a.len_base);
        const bool filtered = mode == RT_LEN_FILTERED;      // bam.py:101: counted nowhere
        const bool unused = mode == RT_LEN_UNUSED;          // detect_orfs.py:74: counted, not binned
        const bool plainlen = !filtered && !unused;
        int4 e;
        // pad + p of bam.py:135 / detect_orfs.py:78-81 relative to `first`: '+' reads first + x, '-' reads first + x + (y >> 3)
        e.x = plainlen ? mode + a.pad + 1 : 0;
        e.y = ((plainlen ? l - 1 - 2 * mode : 0) << 3) | (dl < 16u || filtered ? 0 : kFastNoCounter) | (plainlen ? kFastBinned : 0) |
              (filtered ? 0 : kFastCounted);
        e.z = filtered ? 0 : (int)shl_clamp(1u, dl < 16u ? 4u * dl : 255u);
        e.w = filtered ? 0 : (int)shl_clamp(1u, dl < 16u ? 4u * dl - 32u : 255u);
        s_fast[l] = e;
    }
    __syncthreads();

    using slot_t = typename std::conditional<Compact, unsigned, long long>::type;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool fwd = a.protocol == RT_PROTOCOL_FORWARD;
    const bool stores = a.protocol <= RT_PROTOCOL_REVERSE;
    const unsigned prot_bit = fwd ? 0u : 1u;
    const unsigned char* rec_bytes = reinterpret_cast<const unsigned char*>(a.rec);
    const unsigned char* hdr_bytes = reinterpret_cast<const unsigned char*>(a.hdr);
    auto issue = [&](long long blk, unsigned st) {     // lane 0: bring block `blk` into the warp's stage st
        mbar_expect_tx(&s_bar[warp][st], RT_STREAM_BLOCK * 4u + 16u);
        tma_load_1d(s_rec[warp][st], rec_bytes + (size_t)blk * (RT_STREAM_BLOCK * 4u), RT_STREAM_BLOCK * 4u, &s_bar[warp][st]);
        tma_load_1d(&s_hdr[warp][st], hdr_bytes + (size_t)blk * 16u, 16u, &s_bar[warp][st]);
    };
    const long long stride = (long long)gridDim.x * kStreamWarps;
    long long blk = (long long)blockIdx.x * kStreamWarps + warp;
    if (lane == 0 && blk < a.n_blocks) issue(blk, 0u);

    // 8-bit counters, four per word: categories RT_ST_QCFAIL.. (even / odd nibbles of `packed`), read lengths likewise
    unsigned cat_e = 0, cat_o = 0, len_e0 = 0, len_o0 = 0, len_e1 = 0, len_o1 = 0, total = 0;
    unsigned drained = 0;
    auto flush = [&]() {           // byte counters -> shared memory (one REDUX per counter)
        const unsigned cw[2] = {cat_e, cat_o};
        unsigned mine = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {          // nibble k of `packed` = byte k / 2 of the even or odd word
            const unsigned v = __reduce_add_sync(kFull, (cw[k & 1] >> (8 * (k >> 1))) & 255u);
            if (lane == k) mine = v;
        }
        if (lane < 8 && mine) atomicAdd(&s_stats[1 + lane], mine);
        const unsigned lw[4] = {len_e0, len_o0, len_e1, len_o1};
        unsigned mine_len = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {         // length len_base + k: word k / 8, nibble k % 8
            const unsigned v = __reduce_add_sync(kFull, (lw[2 * (k >> 3) + (k & 1)] >> (8 * ((k & 7) >> 1))) & 255u);
            if (lane == k) mine_len = v;
        }
        const int l = a.len_base + lane;
        if (lane < 16 && mine_len && l >= 0) {
            if (l < kLenHist) atomicAdd(&s_len[l], mine_len);
            else atomicAdd(a.len_counts + l, (unsigned long long)((long long)a.weight * mine_len));
        }
        const unsigned reads = __reduce_add_sync(kFull, total);
        if (lane == 0 && reads) atomicAdd(&s_stats[RT_ST_TOTAL], reads);
        cat_e = cat_o = len_e0 = len_o0 = len_e1 = len_o1 = total = 0;
        drained = 0;
    };

    for (unsigned it = 0; blk < a.n_blocks; ++it, blk += stride) {
        const unsigned st = it & 1u;
        __syncwarp();          // every lane has read stage st ^ 1 (previous block): it is free again
        if (lane == 0 && blk + stride < a.n_blocks) issue(blk + stride, st ^ 1u);
        mbar_wait(&s_bar[warp][st], (it >> 1) & 1u);
        const int4 hd = s_hdr[warp][st];
        unsigned z0p = 0, z1p = 0, z0m = 0, z1m = 0;
        if (Zoned) {
            // this block's zone on both strands: zero it with plain stores (whole sectors are written, none is fetched)
            unsigned zb = 0;
            if (lane < 4) {
                const long long zi = blk + (lane & 1);
                zb = max(__ldg(a.zone_bounds + (size_t)(lane >> 1) * (size_t)(a.n_blocks + 1) + (size_t)zi),
                         __ldg(a.zone_carry + (size_t)(lane >> 1) * (size_t)a.zone_tiles + (size_t)(zi >> 8)));
            }
            z0p = __shfl_sync(kFull, zb, 0); z1p = __shfl_sync(kFull, zb, 1);
            z0m = __shfl_sync(kFull, zb, 2); z1m = __shfl_sync(kFull, zb, 3);
            stream_zero_zone(a.cov, z0p, z1p, lane);
            stream_zero_zone(a.cov, z0m, z1m, lane);
        }
        unsigned w[kStreamStrip + 1];
        {
            const uint4* sp = reinterpret_cast<const uint4*>(s_rec[warp][st]) + 2 * lane;
            const uint4 r0 = sp[0], r1 = sp[1];
            w[0] = r0.x; w[1] = r0.y; w[2] = r0.z; w[3] = r0.w;
            w[4] = r1.x; w[5] = r1.y; w[6] = r1.z; w[7] = r1.w;
        }
        // the usual strip: eight reads, none with an extension record
        const bool plain = __all_sync(kFull, ((w[0] | w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7]) & (RT_STREAM_SPECIAL | (RT_STREAM_EXT << 24))) == 0u);
        // positions: sum of the advances inside the strip, exclusive prefix over the strips of the block; the
        // per-record positions are accumulated again where they are used (cheaper than eight live registers)
        auto advance = [](unsigned x) {
            const unsigned skip = (x & RT_STREAM_KIND_EXT) ? 0u : ((x >> 16) | ((x & 0x3fffu) << 16));
            return (x & RT_STREAM_SPECIAL) ? skip : (x & 0x7fffu);
        };
        unsigned run = 0;
        if (plain) {
#pragma unroll
            for (int j = 0; j < kStreamStrip; ++j) run += w[j] & 0x7fffu;
        } else {
            // an extension record follows its read, possibly in the next thread's strip (never in the next block)
            w[8] = lane == 31 ? (unsigned)RT_STREAM_NULL : s_rec[warp][st][kStreamStrip * (lane + 1)];
#pragma unroll
            for (int j = 0; j < kStreamStrip; ++j) run += advance(w[j]);
        }
        unsigned incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += t;
        }
        unsigned at_first = (unsigned)hd.y + incl - run;      // position the strip's deltas start from

        const int c = hd.x;
        const bool known = (unsigned)c < (unsigned)a.n_contig;
        int2 ct = make_int2(0, 0);
        if (known) ct = c < kStreamContigs ? s_ctab[c] : __ldg(a.contig_tab + c);
        const unsigned span = (unsigned)(ct.x + 2 * a.pad);

        unsigned packed = 0, len_lo = 0, len_hi = 0, n_reads = 0;
        unsigned wd[kStreamStrip], bit[kStreamStrip];
        unsigned live = 0;              // bit j: record j bumps a slot
        if (plain && known && stores) {
            // ---- eight plain reads of a known reference: two shared-memory lookups per read, conditions as bit masks ----
            unsigned odd = 0;           // != 0: some counted read has a length without a register counter
            unsigned oob = 0;
#pragma unroll
            for (int j = 0; j < kStreamStrip; ++j) {
                const unsigned x = w[j];
                const unsigned t = s_sh[x >> 24];
                const int4 e = s_fast[__byte_perm(x, 0u, 0x4442)];
                const unsigned pm = t == kShValid ? 0xffffffffu : 0u;                 // passed the cascade
                const unsigned cm = pm & (0u - ((unsigned)e.y & 1u));                 // counted (bam.py:101,136)
                const unsigned bm = pm & (0u - (((unsigned)e.y >> 1) & 1u));          // binned (detect_orfs.py:74)
                const unsigned mbit = ((x >> 28) ^ prot_bit) & 1u;                    // '-' strand (bam.py:105-131)
                at_first += x & 0x7fffu;
                const unsigned in_contig = at_first + (unsigned)e.x + ((unsigned)(e.y >> 3) & (0u - mbit));
                const unsigned im = in_contig - 1u < span ? 0xffffffffu : 0u;
                oob += bm & ~im & 1u;
                wd[j] = (mbit ? a.plane_words : 0u) + (unsigned)ct.y + (in_contig >> 5);
                bit[j] = in_contig & 31u;
                live |= bm & im & (1u << j);
                packed += shl_clamp(1u, t | (pm & ~cm & 0xe0u));                      // a filtered length counts in `total` only
                len_lo += (unsigned)e.z & cm;
                len_hi += (unsigned)e.w & cm;
                odd |= cm & (unsigned)e.y & (unsigned)kFastNoCounter;
            }
            n_reads = kStreamStrip;
            if (oob) atomicAdd(&s_stats[RT_ST_OOB], oob);
            if (odd) {                  // rare: a length outside the 16 register counters
#pragma unroll
                for (int j = 0; j < kStreamStrip; ++j) {
                    const int l = (int)__byte_perm(w[j], 0u, 0x4442);
                    const int4 e = s_fast[l];
                    if (s_sh[w[j] >> 24] == kShValid && (e.y & kFastCounted) && (e.y & kFastNoCounter)) atomicAdd(&s_len[l], 1u);
                }
            }
        } else {
            // ---- any record: specials, extensions, unknown reference, protocol without a branch in bam.py:105-131 ----
            const unsigned sh_passed = known ? kShValid : 4u * RT_ST_BADREF - 4u;   // where a read that passed is counted
#pragma unroll
            for (int j = 0; j < kStreamStrip; ++j) {
                const unsigned x = w[j];
                const bool normal = !(x & RT_STREAM_SPECIAL);
                const unsigned meta = x >> 24;
                int l = (int)__byte_perm(x, 0u, 0x4442);                  // bits 16-23
                int last_off = l - 1;                                     // last - first
                if (normal && (meta & RT_STREAM_EXT)) {
                    const unsigned e = w[j + 1];
                    l |= (int)((e & 0xffu) << 8);
                    last_off = l - 1 + (int)((e >> 16) | (((e >> 8) & 0x3fu) << 16));
                }
                const int cat = normal ? (int)s_cat[meta & 0x7fu] : 0;
                n_reads += normal ? 1u : 0u;
                int mode = s_mode[l & (kStreamModes - 1)];
                if (l >= kStreamModes) mode = __ldg(a.len_table + l);     // rare: not a Ribo-seq read length
                const bool passed = cat == RT_ST_VALID;
                // bam.py:101 and protocols without a branch in bam.py:105-131 count the read in `total` only
                const bool kept = passed && mode != RT_LEN_FILTERED && stores;
                const bool counted = kept && known;                       // bam.py:136 (a read without a reference name is dropped, :133)
                const bool minus = ((meta & RT_STREAM_REVERSE) != 0) == fwd;           // bam.py:105-131
                at_first += advance(x);
                const int at = (int)at_first + (minus ? last_off : 0);
                const unsigned q = (unsigned)(at + (minus ? -mode : mode) + a.pad);    // detect_orfs.py:78-81
                const bool binned = counted && mode != RT_LEN_UNUSED;                  // detect_orfs.py:74
                const bool inside = q < span;
                if (binned && !inside) atomicAdd(&s_stats[RT_ST_OOB], 1u);
                const unsigned in_contig = q + 1u;
                wd[j] = (minus ? a.plane_words : 0u) + (unsigned)ct.y + (in_contig >> 5);
                bit[j] = in_contig & 31u;
                live |= (binned && inside) ? 1u << j : 0u;
                // categories: what the cascade said, except that a read that passed is counted as valid / badref / nothing
                const unsigned sh_cat = passed ? (kept ? sh_passed : 255u) : 4u * (unsigned)cat - 4u;
                packed += shl_clamp(1u, sh_cat);
                const unsigned dl = (unsigned)(l - a.len_base);
                const unsigned sh = counted ? 4u * dl : 255u;
                len_lo += shl_clamp(1u, sh);
                len_hi += shl_clamp(1u, sh - 32u);
                if (counted && dl >= 16u) {
                    if (l < kLenHist) atomicAdd(&s_len[l], 1u);
                    else atomicAdd(a.len_counts + l, (unsigned long long)(long long)a.weight);
                }
            }
        }
        slot_t slot[kStreamStrip];
        stream_slots<Compact, slot_t>(a, live, wd, bit, slot);
        if (Zoned) {
            // the zones were zeroed at the top of the iteration: their lines are still in L2, so adding the block's
            // own reads fetches nothing from DRAM.  P-sites beyond the zones (rare) wait in the spill list.
            __syncwarp();
            unsigned out[kStreamStrip];
            unsigned n_out = 0;
#pragma unroll
            for (int j = 0; j < kStreamStrip; ++j) {
                const unsigned sl = (unsigned)slot[j];
                const bool mine = (sl - z0p < z1p - z0p) || (sl - z0m < z1m - z0m);
                const bool spills = sl != 0xffffffffu && !mine;
                out[j] = spills ? sl : 0xffffffffu;
                if (spills) {
                    ++n_out;
                    slot[j] = (slot_t)-1;
                }
            }
            stream_scatter<slot_t>(a.cov, slot, 1);
            if (__any_sync(kFull, n_out != 0u)) {
                unsigned incl_out = n_out;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned t = __shfl_up_sync(kFull, incl_out, o);
                    if (lane >= o) incl_out += t;
                }
                unsigned long long base = 0;
                if (lane == 31) base = atomicAdd(a.n_spill, (unsigned long long)incl_out);
                base = __shfl_sync(kFull, base, 31) + incl_out - n_out;
#pragma unroll
                for (int j = 0; j < kStreamStrip; ++j)
                    if (out[j] != 0xffffffffu) a.spill[base++] = out[j];
            }
        } else {
            stream_scatter<slot_t>(a.cov, slot, a.weight);
        }
        // drain the 4-bit counters (at most 8 each) into the 8-bit ones; those hold 31 blocks of the warp
        cat_e += packed & 0x0f0f0f0fu;
        cat_o += (packed >> 4) & 0x0f0f0f0fu;
        len_e0 += len_lo & 0x0f0f0f0fu;
        len_o0 += (len_lo >> 4) & 0x0f0f0f0fu;
        len_e1 += len_hi & 0x0f0f0f0fu;
        len_o1 += (len_hi >> 4) & 0x0f0f0f0fu;
        total += n_reads;
        if (++drained == 31u) flush();
    }
    flush();
    __syncthreads();
    if (threadIdx.x < RT_N_STATS && s_stats[threadIdx.x])
        atomicAdd(a.stats + threadIdx.x, (unsigned long long)((long long)a.weight * s_stats[threadIdx.x]));
    for (int i = threadIdx.x; i < kLenHist; i += kStreamThreads)
        if (s_len[i]) atomicAdd(a.len_counts + i, (unsigned long long)((long long)a.weight * s_len[i]));
}

// Compact layout: one (mask, top) word per 32 dense slots.  A member slot with bit b maps to
// top - popc(mask >> b): members keep their genome order and sit back to back in the compact buffer.
__global__ void __launch_bounds__(256) build_cmap_kernel(const uint64_t* __restrict__ atoms, const uint64_t* __restrict__ atoms_c,
                                                          long long n_atoms, uint2* cmap) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp; i < n_atoms; i += n_warps) {
        const unsigned long long off = atoms[i] >> kLenBits, len = atoms[i] & kLenMask, cb = atoms_c[i] >> kLenBits;
        const unsigned long long w0 = off >> 5, w1 = (off + len - 1) >> 5;
        for (unsigned long long w = w0 + lane; w <= w1; w += 32) {
            const unsigned long long lo = max(off, w << 5), hi = min(off + len, (w << 5) + 32);   // [lo, hi)
            const unsigned nbits = (unsigned)(hi - lo);
            const unsigned mask = (nbits == 32 ? 0xffffffffu : ((1u << nbits) - 1u)) << (unsigned)(lo & 31);
            atomicOr(&cmap[w].x, mask);
            atomicMax(&cmap[w].y, (unsigned)(cb + (hi - off)));
        }
    }
}

__global__ void __launch_bounds__(256) build_cbits_kernel(const uint2* __restrict__ cmap, long long n_words, unsigned* cbits) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool member = w < n_words && cmap[w].x != 0u;
    const unsigned bits = __ballot_sync(kFull, member);
    if ((threadIdx.x & 31) == 0 && w < n_words) cbits[w >> 5] = bits;
}

// Empty cmap words (no member slot) get the compact index of the next member in .y, so that cmap_rank() answers
// "how many member slots lie before this position" for every position of the genome.  Tiles of kGapTile words:
// tile_last = .y of the tile's last word with members (0 if none); the host turns that into a carry per tile.
constexpr int kGapTile = 2048;
__global__ void __launch_bounds__(256) cmap_tile_last_kernel(const uint2* __restrict__ cmap, long long n_words, unsigned* tile_last) {
    __shared__ unsigned s_m[256];
    const long long w0 = (long long)blockIdx.x * kGapTile + (long long)threadIdx.x * (kGapTile / 256);
    unsigned m = 0;
    for (int k = 0; k < kGapTile / 256; ++k)
        if (w0 + k < n_words) {
            const uint2 e = cmap[w0 + k];
            if (e.x) m = e.y;          // .y grows along the genome: the last one seen is the largest
        }
    s_m[threadIdx.x] = m;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s_m[threadIdx.x] = max(s_m[threadIdx.x], s_m[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_last[blockIdx.x] = s_m[0];
}
__global__ void __launch_bounds__(256) cmap_fill_gaps_kernel(uint2* cmap, long long n_words, const unsigned* __restrict__ tile_carry) {
    __shared__ unsigned s_m[256];
    constexpr int kPer = kGapTile / 256;
    const long long w0 = (long long)blockIdx.x * kGapTile + (long long)threadIdx.x * kPer;
    uint2 e[kPer];
    unsigned m = 0;
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        e[k] = w0 + k < n_words ? cmap[w0 + k] : make_uint2(0u, 0u);
        if (e[k].x) m = e[k].y;
    }
    s_m[threadIdx.x] = m;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        const unsigned t = threadIdx.x >= o ? s_m[threadIdx.x - o] : 0u;
        __syncthreads();
        s_m[threadIdx.x] = max(s_m[threadIdx.x], t);
        __syncthreads();
    }
    unsigned carry = max(tile_carry[blockIdx.x], threadIdx.x ? s_m[threadIdx.x - 1] : 0u);
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        if (e[k].x) carry = e[k].y;
        else if (w0 + k < n_words) cmap[w0 + k].y = carry;
    }
}

// Sparse clear: zero the 32-byte sectors (8 slots) K1 touched since the last clear.  Whole sectors
// are safe to zero because only K1 writes the planes and they started from zero; duplicates in the
// list are harmless.
__global__ void __launch_bounds__(256) clear_touched_kernel(int32_t* cov, const unsigned long long* __restrict__ touched,
                                                             const unsigned long long* __restrict__ n_touched) {
    const unsigned long long n = *n_touched;
    int4* sectors = reinterpret_cast<int4*>(cov);
    const int4 z = make_int4(0, 0, 0, 0);
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n; i += 4 * stride) {       // four independent list loads in flight
        const unsigned long long s0 = touched[i], s1 = touched[i + stride], s2 = touched[i + 2 * stride],
                                 s3 = touched[i + 3 * stride];
        sectors[2 * s0] = z; sectors[2 * s0 + 1] = z;
        sectors[2 * s1] = z; sectors[2 * s1 + 1] = z;
        sectors[2 * s2] = z; sectors[2 * s2 + 1] = z;
        sectors[2 * s3] = z; sectors[2 * s3 + 1] = z;
    }
    for (; i < n; i += stride) {
        const unsigned long long sec = touched[i];
        sectors[2 * sec] = z;
        sectors[2 * sec + 1] = z;
    }
}

// ---- dense planes -> compact buffer ---------------------------------------------------------------
// The compact layout is the atoms laid end to end: one warp copies one atom.  Lets a library that was binned
// into the genome-wide planes (the WIG export and the metagene windows need those) be scored by the streamed
// kernels without binning it a second time.
__global__ void __launch_bounds__(256) compact_from_dense_kernel(const uint64_t* __restrict__ atoms, const uint64_t* __restrict__ atoms_c,
                                                                  long long n_atoms, const int32_t* __restrict__ dense,
                                                                  int32_t* __restrict__ compact) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp0; i < n_atoms; i += n_warps) {
        const uint64_t a = __ldg(atoms + i), c = __ldg(atoms_c + i);
        const int32_t* src = dense + (a >> kLenBits);
        int32_t* dst = compact + (c >> kLenBits);
        const int len = (int)(a & kLenMask);
        for (int k = lane; k < len; k += 32) dst[k] = ld_cov(src + k);
    }
}

// ---- export_wig (detect_orfs.py:327-351): the covered positions of a stretch of the dense planes, in order ----
// Two passes over tiles of kWigTile slots: count the non-zero slots of every tile; then, with the exclusive prefix
// of the counts, every thread writes the non-zero ones among its 16 consecutive slots behind those of the threads
// before it (block-wide exclusive scan), so the output is in slot order.
constexpr int kWigPerThread = 16;
constexpr int kWigTile = 256 * kWigPerThread;
__device__ __forceinline__ int wig_load(const int32_t* __restrict__ cov, long long n, long long at, int (&v)[kWigPerThread]) {
    int c = 0;
    if (at + kWigPerThread <= n && (reinterpret_cast<uintptr_t>(cov + at) & 15) == 0) {
#pragma unroll
        for (int q = 0; q < kWigPerThread / 4; ++q) {
            const int4 x = __ldg(reinterpret_cast<const int4*>(cov + at) + q);
            v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < kWigPerThread; ++k) v[k] = at + k < n ? ld_cov(cov + at + k) : 0;
    }
#pragma unroll
    for (int k = 0; k < kWigPerThread; ++k) c += v[k] != 0;
    return c;
}
__global__ void __launch_bounds__(256) wig_count_kernel(const int32_t* __restrict__ cov, long long n, unsigned* tile_counts) {
    int v[kWigPerThread];
    const long long at = (long long)blockIdx.x * kWigTile + (long long)threadIdx.x * kWigPerThread;
    int c = wig_load(cov, n, at, v);
    c = (int)__reduce_add_sync(kFull, (unsigned)c);
    __shared__ unsigned s_part[8];
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = (unsigned)c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += s_part[w];
        tile_counts[blockIdx.x] = t;
    }
}
__global__ void __launch_bounds__(256) wig_fill_kernel(const int32_t* __restrict__ cov, long long n,
                                                        const long long* __restrict__ tile_offsets, long long* out_slot,
                                                        int32_t* out_count) {
    int v[kWigPerThread];
    const long long at = (long long)blockIdx.x * kWigTile + (long long)threadIdx.x * kWigPerThread;
    const int c = wig_load(cov, n, at, v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += t;
    }
    __shared__ int s_warp[8];
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int before = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) before += w < warp ? s_warp[w] : 0;
    long long o = tile_offsets[blockIdx.x] + before + incl - c;
#pragma unroll
    for (int k = 0; k < kWigPerThread; ++k)
        if (v[k] != 0) {
            out_slot[o] = at + k;
            out_count[o] = v[k];
            ++o;
        }
}

// ---- phasescore of one arbitrary (float) profile --------------------------------------------
// statistics.py:48-115 for a single sequence of doubles (the metagene profiles are floats,
// metagene.py:243-244).  One warp; frames in turn; same closed form as accumulate_codon.
__global__ void __launch_bounds__(32) phasescore_values_kernel(const double* __restrict__ v, long long n,
                                                                 double* score_out, int* valid_out) {
    const int lane = threadIdx.x;
    const double kNaN = __longlong_as_double(0x7ff8000000000000ll);
    double coh = 0.0;
    int valid = -1;
    for (int f = 0; f < 3; ++f) {
        int K = 0, M = 0;
        double sre = 0.0, sim = 0.0;
        for (long long i = f + 3ll * lane; i + 2 < n; i += 96) {     // statistics.py:68,71
            const double a = v[i], b = v[i + 1], c = v[i + 2];
            if (a == 0.0 && b == 0.0 && c == 0.0) continue;          // statistics.py:72-73
            ++K;
            const double A = 2.0 * a - b - c, B = b - c;
            if (A == 0.0 && B == 0.0) continue;                      // uniform codon: K only
            const double r = rsqrt(fma(A, A, 3.0 * B * B));
            sre = fma(A, r, sre);
            sim = fma(B, r, sim);
            ++M;
        }
        K = __reduce_add_sync(kFull, K);
        M = __reduce_add_sync(kFull, M);
        sre = warp_sum_f64(sre);
        sim = warp_sum_f64(sim);
        if (K == 0) { coh = 0.0; valid = 0; continue; }              // statistics.py:94-95
        const double s = M == 0 ? kNaN : (sre * sre + 3.0 * sim * sim) / ((double)K * (double)M);
        if (s > coh) { coh = s; valid = K; }                         // statistics.py:109-111
        if (valid == -1) valid = K;                                  // statistics.py:112-113
    }
    if (lane == 0) {
        *score_out = sqrt(coh);                                      // statistics.py:115
        *valid_out = valid;
    }
}


// ------------------------------------------------------------------------------------------------- prepare-orfs
// Candidate ORFs of every transcript (DESIGN.md section 9).  orf_splice_kernel writes each transcript's spliced,
// strand-oriented sequence (codes 0-3 = ACGT, 4 = anything else; '-' transcripts reverse-complemented).  The count and
// fill kernels give one warp to a transcript, claimed dynamically (lengths run from 100 nt to more than 100 knt), and
// walk it in windows of 32 codon positions, one per lane: ballots of the start and stop positions, and per frame the
// nearest stop to the right carried from window to window (3' -> 5').  With `longest`, a 5' -> 3' walk first marks the
// first start of every stop segment (bit 7 of its code byte).  Rows come out in ascending start order per transcript.
enum : uint8_t { kOrfAnnotated = 0, kOrfU = 1, kOrfOverlapU = 2, kOrfSuperU = 3, kOrfOverlapD = 4, kOrfD = 5,
                 kOrfNovel = 6, kOrfInternal = 7 };

struct OrfArgs {
    const long long* tx_seq;          // n_tx + 1: offset of each transcript's spliced sequence
    const int2* tx_cds;               // oriented first / last CDS nt, (-1, -1) without a CDS
    uint8_t* seq;                     // spliced sequences (bit 7: first start of its stop segment, longest only)
    unsigned long long start_mask, stop_mask;
    int n_tx, min_len, longest;
    unsigned* claim;                  // work counter, zeroed before the launch
};

__global__ void orf_splice_kernel(const uint8_t* __restrict__ codes, const long long* __restrict__ ex_src,
                                  const long long* __restrict__ ex_dst, const int* __restrict__ ex_len,
                                  const uint8_t* __restrict__ ex_rev, long long n_exon, uint8_t* __restrict__ seq) {
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long e = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < n_exon; e += warps) {
        const uint8_t* src = codes + ex_src[e];
        const int len = ex_len[e];
        if (ex_rev[e]) {            // '-': ex_dst is the oriented position of the exon's last genomic nt
            uint8_t* dst = seq + ex_dst[e];
            for (int k = lane; k < len; k += 32) {
                const uint8_t c = src[k];
                dst[len - 1 - k] = c < 4 ? (uint8_t)(3 - c) : (uint8_t)4;
            }
        } else {
            uint8_t* dst = seq + ex_dst[e];
            for (int k = lane; k < len; k += 32) dst[k] = src[k];
        }
    }
}

__device__ __forceinline__ uint8_t orf_classify(int a, int b, int2 cds) {
    const int c = cds.x, d = cds.y;
    if (c < 0) return kOrfNovel;
    if (b < c) return kOrfU;
    if (a < c) return b < d ? kOrfOverlapU : kOrfSuperU;
    if (a > d) return kOrfD;
    if (b > d) return kOrfOverlapD;
    return (a == c && b == d) ? kOrfAnnotated : kOrfInternal;
}

// 6-bit codon code at i (16 c0 + 4 c1 + c2), or -1 when a base is not ACGT
__device__ __forceinline__ int orf_codon(const uint8_t* s, long long i) {
    const int a = s[i] & 7, b = s[i + 1] & 7, c = s[i + 2] & 7;
    return (a | b | c) & 4 ? -1 : (a << 4) | (b << 2) | c;
}

template <bool FILL>
__global__ void __launch_bounds__(256) orf_walk_kernel(OrfArgs A, long long* __restrict__ tx_rows,
                                                       const long long* __restrict__ row_off, int* __restrict__ row_tx,
                                                       int* __restrict__ row_start, int* __restrict__ row_stop,
                                                       uint8_t* __restrict__ row_type, uint8_t* __restrict__ row_codon) {
    const int lane = threadIdx.x & 31;
    const unsigned full = 0xffffffffu;
    const unsigned below = (1u << lane) - 1u, above = lane == 31 ? 0u : ~0u << (lane + 1);
    for (;;) {
        int t = 0;
        if (lane == 0) t = (int)atomicAdd(A.claim, 1u);
        t = __shfl_sync(full, t, 0);
        if (t >= A.n_tx) return;
        uint8_t* s = A.seq + A.tx_seq[t];
        const long long n = A.tx_seq[t + 1] - A.tx_seq[t];
        if (n < 3) { if (!FILL && lane == 0) tx_rows[t] = 0; continue; }
        const long long last = n - 3;                   // last codon position
        const int2 cds = A.tx_cds[t];
        if (!FILL && A.longest) {                       // 5' -> 3': mark the first start of every stop segment
            unsigned open = 0;                          // bit g: frame g has a start since its last stop
            for (long long base = 0; base <= last; base += 32) {
                const long long i = base + lane;
                const int cc = i <= last ? orf_codon(s, i) : -1;
                const bool st = cc >= 0 && ((A.stop_mask >> cc) & 1ull), sa = cc >= 0 && ((A.start_mask >> cc) & 1ull);
                const unsigned bst = __ballot_sync(full, st), bsa = __ballot_sync(full, sa);
                const int f = (int)(i % 3);
                const unsigned fm0 = __ballot_sync(full, f == 0), fm1 = __ballot_sync(full, f == 1), fm2 = ~(fm0 | fm1);
                if (sa) {
                    const unsigned fm = f == 0 ? fm0 : f == 1 ? fm1 : fm2;
                    const unsigned stops_le = bst & fm & (below | (1u << lane));
                    bool first;
                    if (stops_le) {
                        const int lst = 31 - __clz(stops_le);
                        first = (bsa & fm & below & ~((1u << lst) - 1u)) == 0u;   // a start at the stop itself opens the segment
                    } else {
                        first = (bsa & fm & below) == 0u && !((open >> f) & 1u);
                    }
                    if (first) s[i] |= 0x80;
                }
#pragma unroll
                for (int g = 0; g < 3; ++g) {
                    const unsigned fm = g == 0 ? fm0 : g == 1 ? fm1 : fm2;
                    const unsigned ms = bst & fm, ma = bsa & fm;
                    const bool o = ms ? (ma >> (31 - __clz(ms))) != 0u : (((open >> g) & 1u) || ma != 0u);
                    open = (open & ~(1u << g)) | ((unsigned)o << g);
                }
            }
            __syncwarp();
        }
        // 3' -> 5': the nearest in-frame stop of every start, the rules, the rows
        int next0 = -1, next1 = -1, next2 = -1;           // per frame: nearest stop right of the window
        long long done = 0;                             // rows of this transcript at positions right of the window
        const long long total = FILL ? tx_rows[t] : 0;
        const long long out0 = FILL ? row_off[t] : 0;
        for (long long base = (last / 32) * 32; base >= 0; base -= 32) {
            const long long i = base + lane;
            const int cc = i <= last ? orf_codon(s, i) : -1;
            const bool st = cc >= 0 && ((A.stop_mask >> cc) & 1ull), sa = cc >= 0 && ((A.start_mask >> cc) & 1ull);
            const unsigned bst = __ballot_sync(full, st);
            const int f = (int)(i % 3);
            const unsigned fm0 = __ballot_sync(full, f == 0), fm1 = __ballot_sync(full, f == 1), fm2 = ~(fm0 | fm1);
            bool keep = false;
            int p = -1;
            uint8_t type = 0;
            if (sa) {
                const unsigned right = bst & (f == 0 ? fm0 : f == 1 ? fm1 : fm2) & above;
                p = right ? (int)base + __ffs(right) - 1 : f == 0 ? next0 : f == 1 ? next1 : next2;
                if (p >= 0 && p - (int)i >= A.min_len && (!A.longest || (s[i] & 0x80))) {
                    type = orf_classify((int)i, p - 1, cds);
                    keep = type != kOrfAnnotated && type != kOrfInternal;
                }
            }
            const unsigned bkeep = __ballot_sync(full, keep);
            if (FILL && keep) {
                const long long r = out0 + total - 1 - (done + __popc(bkeep & above));
                row_tx[r] = t;
                row_start[r] = (int)i;
                row_stop[r] = p;
                row_type[r] = type;
                row_codon[r] = (uint8_t)cc;
            }
            done += __popc(bkeep);
            if (bst & fm0) next0 = (int)base + __ffs(bst & fm0) - 1;
            if (bst & fm1) next1 = (int)base + __ffs(bst & fm1) - 1;
            if (bst & fm2) next2 = (int)base + __ffs(bst & fm2) - 1;
        }
        if (!FILL && lane == 0) tx_rows[t] = done;
    }
}

// Genomic intervals of every row: the oriented range [start, stop) of transcript t as ascending 1-based closed
// intervals of its merged exons.  COUNT writes the number per row, otherwise the intervals at iv_off[row].
template <bool COUNT>
__global__ void orf_interval_kernel(long long n_rows, const int* __restrict__ row_tx, const int* __restrict__ row_start,
                                    const int* __restrict__ row_stop, const long long* __restrict__ tx_exon,
                                    const long long* __restrict__ tx_seq, const uint8_t* __restrict__ tx_rev,
                                    const int* __restrict__ ex_start, const int* __restrict__ ex_end,
                                    const int* __restrict__ ex_before, long long* __restrict__ iv_count,
                                    const long long* __restrict__ iv_off, int* __restrict__ iv_start, int* __restrict__ iv_end) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (long long)gridDim.x * blockDim.x) {
        const int t = row_tx[r];
        const int n = (int)(tx_seq[t + 1] - tx_seq[t]);
        const int lo = tx_rev[t] ? n - row_stop[r] : row_start[r];
        const int hi = tx_rev[t] ? n - row_start[r] : row_stop[r];
        const long long e0 = tx_exon[t], e1 = tx_exon[t + 1];
        auto find = [&](int x) {                        // last exon whose first nt is at or before x
            long long a = e0, b = e1 - 1;
            while (a < b) {
                const long long m = (a + b + 1) >> 1;
                if (ex_before[m] <= x) a = m; else b = m - 1;
            }
            return a;
        };
        const long long ea = find(lo), eb = find(hi - 1);
        if (COUNT) {
            iv_count[r] = eb - ea + 1;
        } else {
            long long o = iv_off[r];
            for (long long e = ea; e <= eb; ++e, ++o) {
                iv_start[o] = e == ea ? ex_start[e] + (lo - ex_before[e]) : ex_start[e];
                iv_end[o] = e == eb ? ex_start[e] + (hi - 1 - ex_before[e]) : ex_end[e];
            }
        }
    }
}

// ----------------------------------------------------------------------------------------------------- orfs-seq
// The output lines of index rows [row_lo, row_lo + n_rows) (DESIGN.md section 10): "ORF_ID\tsequence\n" at
// line_off[row] - line_off[row_lo] of `out`.  One warp per row, claimed dynamically (rows run from 3 nt to more than
// 100 knt).  Nucleotides go straight from the contig codes to their oriented place.  For protein the warp stages the
// oriented codes in a shared-memory window of kSeqWindow nt (a multiple of 3, so a codon never straddles two windows)
// and each lane translates codons of it through a 64-entry table.
struct SeqArgs {
    const uint8_t* codes;
    const long long* exon_ptr;
    const int* ex_start;
    const int* ex_end;
    const int* contig;
    const uint8_t* strand;            // 1: reverse complement
    const long long* contig_base;
    const long long* id_off;
    const char* ids;
    const long long* line_off;        // n_orf + 1: offset of every line after the header
    unsigned* claim;                  // work counter, zeroed before every launch
};

// The warp's next item t < n from a work counter (lane 0 claims it, the warp shares it); false when none is left.
__device__ __forceinline__ bool warp_claim(unsigned* counter, long long n, unsigned& t) {
    t = 0;
    if ((threadIdx.x & 31) == 0) t = atomicAdd(counter, 1u);
    t = __shfl_sync(kFull, t, 0);
    return (long long)t < n;
}

constexpr int kSeqWarps = 8;
constexpr int kSeqWindow = 3 * 32 * 8;

template <bool Protein>
__global__ void __launch_bounds__(kSeqWarps * 32) orf_seq_kernel(SeqArgs A, long long row_lo, long long n_rows,
                                                                 char* __restrict__ out) {
    __shared__ uint8_t window[Protein ? kSeqWarps : 1][Protein ? kSeqWindow : 1];
    __shared__ char amino[64];
    const int lane = threadIdx.x & 31;
    if (Protein) {
        // NCBI table 1, codon code 16 b0 + 4 b1 + b2 with A C G T = 0 1 2 3
        if (threadIdx.x < 64) amino[threadIdx.x] = "KNKNTTTTRSRSIIMIQHQHPPPPRRRRLLLLEDEDAAAAGGGGVVVV*Y*YSSSS*CWCLFLF"[threadIdx.x];
        __syncthreads();
    }
    uint8_t* win = window[Protein ? threadIdx.x >> 5 : 0];
    const long long base = A.line_off[row_lo];
    for (unsigned t; warp_claim(A.claim, n_rows, t);) {
        const long long r = row_lo + t;
        char* o = out + (A.line_off[r] - base);
        const long long i0 = A.id_off[r], n_id = A.id_off[r + 1] - i0;
        for (long long k = lane; k < n_id; k += 32) o[k] = A.ids[i0 + k];
        o += n_id;
        if (lane == 0) *o = '\t';
        ++o;
        const long long e0 = A.exon_ptr[r], e1 = A.exon_ptr[r + 1];
        const uint8_t* g = A.codes + A.contig_base[A.contig[r]];
        const bool rev = A.strand[r] == 1;
        long long n_out;
        if (!Protein) {
            long long L = 0;
            for (long long e = e0; e < e1; ++e) L += A.ex_end[e] - A.ex_start[e] + 1;
            long long before = 0;                     // nt of the row's intervals left of interval e
            for (long long e = e0; e < e1; ++e) {
                const uint8_t* src = g + A.ex_start[e] - 1;
                const int len = A.ex_end[e] - A.ex_start[e] + 1;
                if (rev) {
                    char* dst = o + (L - 1 - before);
                    for (int k = lane; k < len; k += 32) {
                        const uint8_t c = src[k];
                        dst[-k] = c < 4 ? "TGCA"[c] : 'N';
                    }
                } else {
                    char* dst = o + before;
                    for (int k = lane; k < len; k += 32) {
                        const uint8_t c = src[k];
                        dst[k] = c < 4 ? "ACGT"[c] : 'N';
                    }
                }
                before += len;
            }
            n_out = L;
        } else {
            int fill = 0;                             // oriented nt staged in the window
            long long done = 0;                       // amino acids written
            auto emit = [&](int n_codon) {
                __syncwarp();
                for (int c = lane; c < n_codon; c += 32) {
                    const int a = win[3 * c], b = win[3 * c + 1], d = win[3 * c + 2];
                    o[done + c] = (a | b | d) & 4 ? 'X' : amino[(a << 4) | (b << 2) | d];
                }
                __syncwarp();
                done += n_codon;
            };
            for (long long j = 0; j < e1 - e0; ++j) {
                const long long e = rev ? e1 - 1 - j : e0 + j;
                const uint8_t* src = g + A.ex_start[e] - 1;
                const int len = A.ex_end[e] - A.ex_start[e] + 1;
                for (int k0 = 0; k0 < len;) {
                    const int n = min(len - k0, kSeqWindow - fill);
                    for (int k = lane; k < n; k += 32) {
                        const uint8_t c = rev ? src[len - 1 - (k0 + k)] : src[k0 + k];
                        win[fill + k] = c < 4 ? (rev ? (uint8_t)(3 - c) : c) : (uint8_t)4;
                    }
                    fill += n;
                    k0 += n;
                    if (fill == kSeqWindow) {
                        emit(kSeqWindow / 3);
                        fill = 0;
                    }
                }
            }
            emit(fill / 3);
            n_out = done;
        }
        if (lane == 0) o[n_out] = '\n';
    }
}

// ---------------------------------------------------------------------------------- selected detected-ORF rows
// The selected rows of a detected-ORFs TSV as codon_emit_kernel and count_emit_kernel read them: one warp per row,
// claimed dynamically (profiles run from "[]" to more than 100 knt).
struct RowArgs {
    const char* prof;                 // profile text of the selected rows, back to back
    const long long* prof_base;       // n_sel + 1
    const long long* len_base;        // n_sel + 1: row lengths in nt, scanned
    const long long* row;             // index row of each selected row
    const long long* exon_ptr;
    const int* ex_start;
    const int* ex_end;
    const uint8_t* strand;            // per index row, 1: reverse
    const int* gene;
    uint8_t* flag;                    // per selected row: its refusal bits (1 malformed, 2 value above 2^31 - 1, ...)
    long long n_sel;
    unsigned* claim;                  // work counter, zeroed before the launch
};

// Refuses selected row t with `bits`: sets its flag and takes part in the atomicMin of the first refused row, *first.
__device__ __forceinline__ void refuse_row(uint8_t* flag, unsigned long long* first, unsigned t, unsigned bits) {
    flag[t] = (uint8_t)bits;
    atomicMin(first, (unsigned long long)t);
}

// Per lane: the genomic coordinate of oriented nt k of a row of L nt, through the row's intervals.  The cursor keeps
// interval e and the nt of the intervals left of it, `before` (ascending order); '-' rows walk the intervals from the
// right.  A lane asks for ascending k.
struct IntervalCursor {
    const int* ex_start;
    const int* ex_end;
    long long L, e, before;
    bool rev;
    __device__ __forceinline__ IntervalCursor(const RowArgs& A, long long r, long long L_)
        : ex_start(A.ex_start), ex_end(A.ex_end), L(L_) {
        const long long e0 = A.exon_ptr[r], e1 = A.exon_ptr[r + 1];
        rev = A.strand[r] == 1;
        e = rev ? e1 - 1 : e0;
        before = 0;
        if (rev)
            for (long long x = e0; x < e1 - 1; ++x) before += ex_end[x] - ex_start[x] + 1;
    }
    __device__ __forceinline__ int coord(long long k) {
        const long long a = rev ? L - 1 - k : k;       // ascending index of oriented nt k
        if (rev) {
            while (a < before) { --e; before -= ex_end[e] - ex_start[e] + 1; }
        } else {
            while (a >= before + (ex_end[e] - ex_start[e] + 1)) { before += ex_end[e] - ex_start[e] + 1; ++e; }
        }
        return ex_start[e] + (int)(a - before);
    }
};

// ---------------------------------------------------------------------------------------------- count-orfs-codon
// codon_emit_kernel: one warp per selected TSV row, claimed dynamically (profiles run from "[]" to more than 100 knt).
// The warp reads the profile text in 32-byte windows: every byte is checked against the grammar "[" (D(", "D)*)? "]"
// with D = 0 | [1-9][0-9]*, a ballot of the digits that follow a non-digit finds the values, and each lane parses the
// value it starts and adds it to the count of its codon (a zero adds nothing).  Then codon k < min(values, length) / 3
// is named from the row's letters (6-bit code 16 b0 + 4 b1 + b2, A C G T = 0 1 2 3) and placed on the genome: its first
// oriented nt, through the row's intervals ('-' rows walk them from the right).  Slot k of the row gets the place key
// gseq << 32 | first nt and the value (gene * 64 + code) << 32 | count; a codon with N, or past the profile, gets the key
// ~0 (dropped).
struct CodonArgs {
    RowArgs rows;                     // flag 4: a codon count above 2^32 - 1
    const char* seq;                  // the rows' letters, back to back (at len_base)
    const long long* slot_base;       // n_sel + 1: floor(length / 3) slots per row
    const int* gseq;
    unsigned long long* cnt;          // per slot: codon count, zeroed before the launch
    unsigned long long* pos_key;      // per slot: place key
    unsigned long long* val;          // per slot: (gene * 64 + codon) << 32 | count
    unsigned long long* counters;     // [0] codons named, [1] with N, [2] first refused row (atomicMin), zeroed / ~0
};

constexpr int kCodonWarps = 8;

__device__ __forceinline__ bool is_digit(char c) { return c >= '0' && c <= '9'; }

// The profile grammar walk shared by codon_emit_kernel and count_emit_kernel, called by the whole warp on the profile
// text s[0, n) of one row.  Every byte is checked against "[" (D(", "D)*)? "]" with D = 0 | [1-9][0-9]*, 32 bytes a
// window; a ballot of the digits that follow a non-digit finds the values, and the lane that starts value j calls
// on_value(j, v) while it has seen nothing wrong.  Returns this lane's refusal bits (1 malformed, 2 a value above
// 2^31 - 1; the caller reduces them over the warp) and sets P to the number of values.
template <class OnValue>
__device__ __forceinline__ unsigned profile_walk(const char* s, long long n, int lane, long long& P, OnValue&& on_value) {
    const unsigned below = (1u << lane) - 1u;
    unsigned bad = 0;
    P = 0;
    if (n < 2 || s[0] != '[' || s[n - 1] != ']') return 1;
    const char* b = s + 1;
    const long long nb = n - 2;
    for (long long w = 0; w < nb; w += 32) {
        const long long i = w + lane;
        bool start = false;
        unsigned long long v = 0;
        if (i < nb) {
            const char c = b[i], p = i > 0 ? b[i - 1] : ' ', q = i + 1 < nb ? b[i + 1] : ',';
            if (is_digit(c)) {                             // the defaults of p and q refuse a separator at either end
                start = !is_digit(p);
            } else if (c == ',') {
                if (!is_digit(p) || q != ' ') bad |= 1;
            } else if (c == ' ') {
                if (p != ',' || !is_digit(q)) bad |= 1;
            } else {
                bad |= 1;
            }
            if (start) {
                if (c == '0' && i + 1 < nb && is_digit(b[i + 1])) bad |= 1;   // a leading zero
                int d = 0;
                for (long long j = i; j < nb && is_digit(b[j]) && d < 11; ++j, ++d) v = v * 10 + (b[j] - '0');
                if (d > 10 || v > 2147483647ull) bad |= 2;
            }
        }
        const unsigned starts = __ballot_sync(kFull, start);
        if (start && !bad) on_value(P + __popc(starts & below), v);
        P += __popc(starts);
    }
    return bad;
}

__global__ void __launch_bounds__(kCodonWarps * 32) codon_emit_kernel(const CodonArgs A) {
    const RowArgs& R = A.rows;
    const int lane = threadIdx.x & 31;
    for (unsigned t; warp_claim(R.claim, R.n_sel, t);) {
        const char* s = R.prof + R.prof_base[t];
        const long long n = R.prof_base[t + 1] - R.prof_base[t];
        const long long L = R.len_base[t + 1] - R.len_base[t];
        const long long s0 = A.slot_base[t], n_slot = A.slot_base[t + 1] - s0;
        long long P;                                       // values parsed
        unsigned bad = profile_walk(s, n, lane, P, [&](long long j, unsigned long long v) {
            if (v && j / 3 < n_slot) atomicAdd(A.cnt + s0 + j / 3, v);
        });
        bad = __reduce_or_sync(kFull, bad);
        __syncwarp();                                      // the counts of this row are in place (read through L2 below)
        if (bad) {
            if (lane == 0) refuse_row(R.flag, A.counters + 2, t, bad);
            continue;
        }
        const long long n_cod = min(P, L) / 3;
        IntervalCursor cur(R, R.row[t], L);
        const char* letters = A.seq + R.len_base[t];
        const unsigned long long hi_gene = (unsigned long long)R.gene[t] * 64ull;
        const unsigned long long hi_place = (unsigned long long)(unsigned)A.gseq[t] << 32;
        unsigned named = 0, with_n = 0, over = 0;
        for (long long k = lane; k < n_slot; k += 32) {
            unsigned long long key = ~0ull, value = 0;
            if (k < n_cod) {
                const unsigned long long c = __ldcg(A.cnt + s0 + k);
                over |= c > 0xffffffffull;
                const char* l3 = letters + 3 * k;
                int code = 0;
                bool has_n = false;
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const char x = l3[u];
                    has_n |= x == 'N';
                    code = code * 4 + (x == 'C' ? 1 : x == 'G' ? 2 : x == 'T' ? 3 : 0);
                }
                ++named;
                if (has_n) {
                    ++with_n;
                } else {
                    key = hi_place | (unsigned)cur.coord(3 * k);
                    value = (hi_gene + (unsigned long long)code) << 32 | (c & 0xffffffffull);
                }
            }
            A.pos_key[s0 + k] = key;
            A.val[s0 + k] = value;
        }
        named = __reduce_add_sync(kFull, named);
        with_n = __reduce_add_sync(kFull, with_n);
        over = __reduce_or_sync(kFull, over);
        if (lane == 0) {
            if (named) atomicAdd(A.counters + 0, (unsigned long long)named);
            if (with_n) atomicAdd(A.counters + 1, (unsigned long long)with_n);
            if (over) refuse_row(R.flag, A.counters + 2, t, 4);
        }
    }
}

// After the stable sort by place key: the first slot of every place is kept.  Appends its value to `kept` and its
// pooled key (codon << 32 | count) to `pooled`; the order of the appends does not matter (both are sorted next).
__global__ void __launch_bounds__(256) codon_keep_kernel(const unsigned long long* __restrict__ key,
                                                         const unsigned long long* __restrict__ val, long long n,
                                                         unsigned long long* kept, unsigned long long* pooled,
                                                         unsigned long long* n_kept) {
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long w = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); w < n; w += stride) {
        const long long i = w + lane;
        bool keep = false;
        if (i < n) {
            const unsigned long long k = key[i];
            keep = k != ~0ull && (i == 0 || key[i - 1] != k);
        }
        const unsigned b = __ballot_sync(kFull, keep);
        unsigned long long at = 0;
        if (lane == 0 && b) at = atomicAdd(n_kept, (unsigned long long)__popc(b));
        at = __shfl_sync(kFull, at, 0);
        if (keep) {
            const unsigned long long v = val[i], o = at + __popc(b & ((1u << lane) - 1u));
            kept[o] = v;
            pooled[o] = ((v >> 32) & 63ull) << 32 | (v & 0xffffffffull);
        }
    }
}

// One warp per cell (the keys whose high 32 bits equal the cell, counts in the low 32 bits, sorted): n, S1, S2 (two
// 64-bit halves) and the sum of the middle two counts (twice the middle one for odd n).  Exact integers: the result
// does not depend on the order of the additions.
__global__ void __launch_bounds__(256) codon_stats_kernel(const unsigned long long* __restrict__ keys, long long n,
                                                          long long n_cells, unsigned long long* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    auto lower = [&](unsigned long long x) {              // first key >= x (every lane searches the same addresses)
        long long a = 0, b = n;
        while (a < b) {
            const long long m = (a + b) >> 1;
            if (keys[m] < x) a = m + 1; else b = m;
        }
        return a;
    };
    for (long long c = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < n_cells; c += warps) {
        const long long lo = lower((unsigned long long)c << 32), hi = lower((unsigned long long)(c + 1) << 32);
        unsigned long long s1 = 0, s2_lo = 0, s2_hi = 0;
        for (long long i = lo + lane; i < hi; i += 32) {
            const unsigned long long x = keys[i] & 0xffffffffull, sq = x * x;
            s1 += x;
            s2_lo += sq;
            s2_hi += s2_lo < sq;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            s1 += __shfl_xor_sync(kFull, s1, d);
            const unsigned long long o_lo = __shfl_xor_sync(kFull, s2_lo, d), o_hi = __shfl_xor_sync(kFull, s2_hi, d);
            s2_lo += o_lo;
            s2_hi += o_hi + (s2_lo < o_lo);
        }
        if (lane == 0) {
            const long long m = hi - lo;
            unsigned long long mid = 0;
            if (m) {
                const unsigned long long x1 = keys[lo + m / 2] & 0xffffffffull;
                mid = m & 1 ? 2 * x1 : x1 + (keys[lo + m / 2 - 1] & 0xffffffffull);
            }
            unsigned long long* o = out + 5 * c;
            o[0] = (unsigned long long)m;
            o[1] = s1;
            o[2] = s2_lo;
            o[3] = s2_hi;
            o[4] = mid;
        }
    }
}

// ---------------------------------------------------------------------------------------------------- count-orfs
// count_emit_kernel (DESIGN.md section 13): one warp per selected TSV line, claimed dynamically.  The warp checks the
// profile grammar (profile_walk) and stores value j < L of the row's L nt as val[s0 + j].  Then oriented nt k < m =
// min(values, L) gets the key gene << 32 | (uint32) its genomic coordinate, found through the row's intervals with a
// per-lane cursor ('-' rows walk them from the right); slots k in [m, L) get the key ~0 (dropped).  A refused line sets
// its flag and takes part in an atomicMin of the first refused line.
struct CountArgs {
    RowArgs rows;                     // flag: 1 malformed, 2 value above 2^31 - 1
    unsigned long long* key;          // per slot (len_base)
    unsigned* val;                    // per slot
    unsigned long long* counters;     // [0] positions named (sum of m), [1] first refused line (atomicMin), zeroed / ~0
};

__global__ void __launch_bounds__(kCodonWarps * 32) count_emit_kernel(const CountArgs A) {
    const RowArgs& R = A.rows;
    const int lane = threadIdx.x & 31;
    for (unsigned t; warp_claim(R.claim, R.n_sel, t);) {
        const long long s0 = R.len_base[t], L = R.len_base[t + 1] - s0;
        long long P;
        unsigned bad = profile_walk(R.prof + R.prof_base[t], R.prof_base[t + 1] - R.prof_base[t], lane, P,
                                    [&](long long j, unsigned long long v) {
            if (j < L) A.val[s0 + j] = (unsigned)v;
        });
        bad = __reduce_or_sync(kFull, bad);
        if (bad) {
            if (lane == 0) refuse_row(R.flag, A.counters + 1, t, bad);
            continue;
        }
        const long long m = min(P, L);
        IntervalCursor cur(R, R.row[t], L);
        const unsigned long long hi = (unsigned long long)(unsigned)R.gene[t] << 32;
        for (long long k = lane; k < L; k += 32)
            A.key[s0 + k] = k < m ? hi | (unsigned)cur.coord(k) : ~0ull;
        if (lane == 0 && m) atomicAdd(A.counters + 0, (unsigned long long)m);
    }
}

// After the stable sort by key: the first slot of every key is kept (TSV order survives a stable sort, so it is the
// first line's value), and adds its value to total[gene] and 1 to length[gene].  Keys are sorted, so the gene of the
// slots, key >> 32 (0xffffffff for dropped slots and past the end), never decreases across a warp: a segmented scan over
// runs of equal gene leaves each run's sums with its last lane, which alone issues the two atomics.
__global__ void __launch_bounds__(256) count_keep_kernel(const unsigned long long* __restrict__ key,
                                                         const unsigned* __restrict__ val, long long n,
                                                         unsigned long long* total, unsigned long long* length) {
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long w = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); w < n; w += stride) {
        const long long i = w + lane;
        unsigned gene = 0xffffffffu;
        unsigned long long sum = 0, cnt = 0;
        if (i < n) {
            const unsigned long long k = key[i];
            gene = (unsigned)(k >> 32);
            if (k != ~0ull && (i == 0 || key[i - 1] != k)) {
                sum = val[i];
                cnt = 1;
            }
        }
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned g_up = __shfl_up_sync(kFull, gene, d);
            const unsigned long long s_up = __shfl_up_sync(kFull, sum, d), c_up = __shfl_up_sync(kFull, cnt, d);
            if (lane >= d && g_up == gene) {
                sum += s_up;
                cnt += c_up;
            }
        }
        const unsigned g_next = __shfl_down_sync(kFull, gene, 1);
        if ((lane == 31 || g_next != gene) && cnt) {
            atomicAdd(total + gene, sum);
            atomicAdd(length + gene, cnt);
        }
    }
}


// ---------------------------------------------------------------------------------------------------- BGZF inflate
// bgzf_inflate_kernel (DESIGN.md section 12): one warp per BGZF member, claimed dynamically.  Lane 0 walks the DEFLATE
// bit stream (RFC 1951) and writes the literals; the back-references it meets go to a queue of kInfQueue entries in
// shared memory, which the whole warp then copies in order, one byte per lane (a copy that overlaps its own output reads
// source byte k mod distance).  The Huffman decode tables of every DEFLATE block are built by the warp in shared memory:
// code lengths counted and ranked with __match_any_sync, then a kInfLitFast-bit (literal/length) or kInfDistFast-bit
// (distance) lookup table of (symbol << 4 | code length); longer codes take the canonical walk over the per-length counts.
// Every read stays inside the member's payload and every write inside [out_off, out_off + ISIZE).  Then each lane takes
// the CRC-32 of a 32nd of the output and the lanes combine theirs by multiplication with x^(8n) mod P (zlib's
// crc32_combine).  status[b] = kInfOk when member b inflated to exactly ISIZE bytes with the CRC-32 of its footer.
struct BgzfBlock {
    unsigned long long in_off, out_off;   // DEFLATE payload in the compressed file; first byte in the text
    unsigned in_len, out_len, crc, pad;
};

constexpr int kInflateWarps = 8;
constexpr int kInfLitFast = 10, kInfDistFast = 8, kInfQueue = 32;
enum : int { kInfOk = 0, kInfBadBlock = 1, kInfBadCode = 2, kInfBadSymbol = 3, kInfOverrun = 4, kInfSize = 5, kInfCrc = 6 };

__constant__ uint16_t kInfLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99,
                                         115, 131, 163, 195, 227, 258};
__constant__ uint8_t kInfLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t kInfDistBase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025,
                                          1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t kInfDistExtra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12,
                                          12, 13, 13};
__constant__ uint8_t kInfClOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct InflateWarp {                              // the shared memory of one warp
    uint16_t lit_fast[1 << kInfLitFast];          // (symbol << 4) | code length; 0: a longer code, or none
    uint16_t dist_fast[1 << kInfDistFast];
    uint16_t lit_sorted[288], dist_sorted[32];    // symbols in canonical order (code length, then symbol)
    uint16_t lit_count[16], dist_count[16];       // codes of each length
    uint16_t run[16], code0[16];                  // table build: next rank of each length; first code minus first rank
    uint8_t lens[320];                            // code lengths: literal/length 0..287, distance 288..319
    uint8_t cl_lens[20];                          // the code length code of a dynamic block
    unsigned q_pos[kInfQueue];                    // back-references waiting for the warp: output offset, length, distance
    uint16_t q_len[kInfQueue], q_dist[kInfQueue];
};

// Lane 0's view of the member's bits, least significant first; bytes past the payload read as 0 and are caught by the
// callers (pos > n + 8 means bits past the end have been consumed).
struct InflateBits {
    const uint8_t* in;
    unsigned n, pos;
    unsigned long long bb;
    int bc;
    __device__ __forceinline__ void refill() {
        while (bc <= 56) {
            const unsigned long long b = pos < n ? in[pos] : 0u;
            ++pos;
            bb |= b << bc;
            bc += 8;
        }
    }
    __device__ __forceinline__ unsigned take(int k) {
        const unsigned v = (unsigned)(bb & ((1ull << k) - 1));
        bb >>= k;
        bc -= k;
        return v;
    }
};

// The decode table of one canonical code, built by the whole warp.  false when the lengths over-subscribe the code, or
// leave it incomplete with a longest code above 1 bit (zlib accepts a lone 1-bit code), or, for the code length code,
// leave it incomplete at all.
__device__ bool inflate_build(const uint8_t* lens, int n, int fast_bits, uint16_t* fast, uint16_t* sorted, uint16_t* count,
                              InflateWarp& w, bool cl_code, int lane) {
    if (lane < 16) count[lane] = 0;
    for (int i = lane; i < (1 << fast_bits); i += 32) fast[i] = 0;
    __syncwarp();
    for (int c = 0; c < n; c += 32) {
        const int L = c + lane < n ? lens[c + lane] : 0;
        const unsigned m = __match_any_sync(kFull, L);
        if (L && lane == __ffs(m) - 1) count[L] += (uint16_t)__popc(m);
        __syncwarp();
    }
    int left = 1, longest = 0, offs = 0, code = 0;
    for (int L = 1; L < 16; ++L) {
        const int k = count[L];
        left = (left << 1) - k;
        if (left < 0) return false;
        if (k) longest = L;
        if (lane == 0) {
            w.run[L] = (uint16_t)offs;
            w.code0[L] = (uint16_t)(code - offs);
        }
        offs += k;
        code = (code + k) << 1;
    }
    if (left > 0 && (longest > 1 || cl_code)) return false;
    __syncwarp();
    for (int c = 0; c < n; c += 32) {
        const int s = c + lane;
        const int L = s < n ? lens[s] : 0;
        const unsigned m = __match_any_sync(kFull, L);
        const int idx = w.run[L] + __popc(m & ((1u << lane) - 1u));
        __syncwarp();
        if (L) {
            if (lane == __ffs(m) - 1) w.run[L] += (uint16_t)__popc(m);
            sorted[idx] = (uint16_t)s;
            if (L <= fast_bits) {
                const unsigned rev = __brev((unsigned)(w.code0[L] + idx)) >> (32 - L);
                for (unsigned k = rev; k < (1u << fast_bits); k += 1u << L) fast[k] = (uint16_t)(s << 4 | L);
            }
        }
        __syncwarp();
    }
    return true;
}

// One symbol (lane 0; at least 15 bits in the buffer): the table entry, else the canonical walk bit by bit.  -1: no code.
__device__ __forceinline__ int inflate_symbol(InflateBits& br, const uint16_t* fast, int fast_bits, const uint16_t* count,
                                              const uint16_t* sorted) {
    const unsigned e = fast[br.bb & ((1u << fast_bits) - 1)];
    if (e & 15) {
        br.bb >>= e & 15;
        br.bc -= (int)(e & 15);
        return (int)(e >> 4);
    }
    int code = 0, first = 0, index = 0;
    for (int len = 1; len < 16; ++len) {
        code |= (int)((br.bb >> (len - 1)) & 1);
        const int k = count[len];
        if (code - k < first) {
            br.bb >>= len;
            br.bc -= len;
            return sorted[index + (code - first)];
        }
        index += k;
        first = (first + k) << 1;
        code <<= 1;
    }
    return -1;
}

// The DEFLATE stream of one member into out[0, out_len), by the whole warp; returns the same status in every lane.
__device__ int inflate_member(InflateWarp& w, const uint8_t* __restrict__ in, unsigned in_len, uint8_t* out,
                              unsigned out_len, int lane) {
    InflateBits br{in, in_len, 0u, 0ull, 0};
    unsigned op = 0;                                  // bytes written; lane 0's count is the one that matters
    int err = kInfOk, last = 0;
    while (!last) {
        int type = 0;
        if (lane == 0) {
            br.refill();
            if (br.pos > in_len + 8) err = kInfOverrun;
            last = (int)br.take(1);
            type = (int)br.take(2);
        }
        err = __shfl_sync(kFull, err, 0);
        if (err) return err;
        type = __shfl_sync(kFull, type, 0);
        last = __shfl_sync(kFull, last, 0);
        if (type == 0) {                              // stored: LEN, NLEN, then LEN bytes from the next byte boundary
            unsigned src = 0, n = 0;
            if (lane == 0) {
                br.take(br.bc & 7);
                src = br.pos - (unsigned)(br.bc >> 3);
                br.bb = 0;
                br.bc = 0;
                if (src + 4 > in_len) {
                    err = kInfOverrun;
                } else {
                    n = in[src] | (unsigned)in[src + 1] << 8;
                    const unsigned nn = in[src + 2] | (unsigned)in[src + 3] << 8;
                    if (n != (~nn & 0xffffu)) err = kInfBadBlock;
                    else if (src + 4 + n > in_len) err = kInfOverrun;
                    else if (n > out_len - op) err = kInfSize;
                }
                br.pos = src + 4 + n;
            }
            err = __shfl_sync(kFull, err, 0);
            if (err) return err;
            src = __shfl_sync(kFull, src, 0) + 4;
            n = __shfl_sync(kFull, n, 0);
            op = __shfl_sync(kFull, op, 0);
            for (unsigned k = lane; k < n; k += 32) out[op + k] = in[src + k];
            op += n;
            continue;
        }
        if (type == 3) return kInfBadBlock;
        if (type == 1) {                              // fixed codes (RFC 1951 3.2.6); symbols 286, 287, 30, 31 are refused
            for (int i = lane; i < 320; i += 32) w.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
            __syncwarp();
        } else {                                      // dynamic: HLIT, HDIST, HCLEN, the code length code, the lengths
            int nlit = 0, ndist = 0;
            for (int i = lane; i < 320; i += 32) w.lens[i] = 0;
            if (lane == 0) {
                br.refill();
                nlit = (int)br.take(5) + 257;
                ndist = (int)br.take(5) + 1;
                const int ncl = (int)br.take(4) + 4;
                for (int i = 0; i < 19; ++i) {
                    if (br.bc < 3) br.refill();
                    w.cl_lens[kInfClOrder[i]] = (uint8_t)(i < ncl ? br.take(3) : 0);
                }
                if (nlit > 286 || ndist > 30) err = kInfBadBlock;
            }
            err = __shfl_sync(kFull, err, 0);
            if (err) return err;
            __syncwarp();
            if (!inflate_build(w.cl_lens, 19, 7, w.lit_fast, w.dist_sorted, w.dist_count, w, true, lane)) return kInfBadCode;
            if (lane == 0) {
                const int total = nlit + ndist;
                int prev = -1;
                for (int i = 0; i < total;) {
                    if (br.bc < 16) {
                        br.refill();
                        if (br.pos > in_len + 8) { err = kInfOverrun; break; }
                    }
                    const int sym = inflate_symbol(br, w.lit_fast, 7, w.dist_count, w.dist_sorted);
                    int len = 0, rep = 1;
                    if (sym < 0) { err = kInfBadSymbol; break; }
                    if (sym < 16) {
                        len = sym;
                    } else if (sym == 16) {
                        if (prev < 0) { err = kInfBadBlock; break; }
                        len = prev;
                        rep = 3 + (int)br.take(2);
                    } else {
                        rep = sym == 17 ? 3 + (int)br.take(3) : 11 + (int)br.take(7);
                    }
                    if (rep > total - i) { err = kInfBadBlock; break; }
                    prev = len;
                    for (; rep > 0; --rep, ++i) w.lens[i < nlit ? i : 288 + i - nlit] = (uint8_t)len;
                }
                if (!err && w.lens[256] == 0) err = kInfBadCode;   // no end-of-block code
            }
            err = __shfl_sync(kFull, err, 0);
            if (err) return err;
            __syncwarp();
        }
        if (!inflate_build(w.lens, 288, kInfLitFast, w.lit_fast, w.lit_sorted, w.lit_count, w, false, lane)) return kInfBadCode;
        if (!inflate_build(w.lens + 288, 32, kInfDistFast, w.dist_fast, w.dist_sorted, w.dist_count, w, false, lane))
            return kInfBadCode;
        for (;;) {                                    // batches: lane 0 decodes up to kInfQueue back-references, the warp copies
            int nq = 0, eob = 0;
            if (lane == 0) {
                while (nq < kInfQueue) {
                    if (br.bc < 48) {                 // a length and a distance with their extra bits take at most 48
                        br.refill();
                        if (br.pos > in_len + 8) { err = kInfOverrun; break; }
                    }
                    int sym = inflate_symbol(br, w.lit_fast, kInfLitFast, w.lit_count, w.lit_sorted);
                    if (sym < 256) {
                        if (sym < 0) { err = kInfBadSymbol; break; }
                        if (op >= out_len) { err = kInfSize; break; }
                        out[op++] = (uint8_t)sym;
                        continue;
                    }
                    if (sym == 256) { eob = 1; break; }
                    sym -= 257;
                    if (sym >= 29) { err = kInfBadSymbol; break; }
                    const unsigned len = kInfLenBase[sym] + br.take(kInfLenExtra[sym]);
                    const int ds = inflate_symbol(br, w.dist_fast, kInfDistFast, w.dist_count, w.dist_sorted);
                    if (ds < 0 || ds >= 30) { err = kInfBadSymbol; break; }
                    const unsigned dist = kInfDistBase[ds] + br.take(kInfDistExtra[ds]);
                    if (dist > op) { err = kInfBadSymbol; break; }
                    if (len > out_len - op) { err = kInfSize; break; }
                    w.q_pos[nq] = op;
                    w.q_len[nq] = (uint16_t)len;
                    w.q_dist[nq] = (uint16_t)dist;
                    ++nq;
                    op += len;
                }
            }
            err = __shfl_sync(kFull, err, 0);
            if (err) return err;
            nq = __shfl_sync(kFull, nq, 0);
            eob = __shfl_sync(kFull, eob, 0);
            __syncwarp();
            for (int q = 0; q < nq; ++q) {
                const unsigned len = w.q_len[q], dist = w.q_dist[q];
                uint8_t* dst = out + w.q_pos[q];
                const uint8_t* src = dst - dist;
                if (dist >= len) {
                    for (unsigned k = lane; k < len; k += 32) dst[k] = src[k];
                } else {
                    unsigned s = (unsigned)lane % dist;
                    const unsigned step = 32u % dist;
                    for (unsigned k = lane; k < len; k += 32) {
                        dst[k] = src[s];
                        s += step;
                        if (s >= dist) s -= dist;
                    }
                }
                __syncwarp();
            }
            if (eob) break;
        }
    }
    if (lane == 0) {
        if ((unsigned long long)br.pos * 8 - (unsigned long long)br.bc > (unsigned long long)in_len * 8) err = kInfOverrun;
        else if (op != out_len) err = kInfSize;
    }
    return __shfl_sync(kFull, err, 0);
}

// a * b mod P over GF(2), bit-reflected (zlib's multmodp)
__device__ __forceinline__ unsigned crc_multmodp(unsigned a, unsigned b) {
    unsigned p = 0;
    for (unsigned m = 1u << 31; m; m >>= 1) {
        if (a & m) p ^= b;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}

// x^(8n) mod P from x2n[k] = x^(2^k) mod P
__device__ __forceinline__ unsigned crc_x8n(unsigned n, const unsigned* x2n) {
    unsigned p = 1u << 31;
    for (int k = 3; n; n >>= 1, ++k)
        if (n & 1) p = crc_multmodp(x2n[k & 31], p);
    return p;
}

__global__ void __launch_bounds__(kInflateWarps * 32) bgzf_inflate_kernel(const uint8_t* __restrict__ comp,
                                                                          const BgzfBlock* __restrict__ blocks,
                                                                          long long n_blocks, uint8_t* text,
                                                                          uint8_t* __restrict__ status, unsigned* claim) {
    __shared__ InflateWarp warps[kInflateWarps];
    __shared__ unsigned crc_tab[256], x2n[32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        unsigned c = (unsigned)i;
        for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
        crc_tab[i] = c;
    }
    if (threadIdx.x == 0) {
        unsigned p = 1u << 30;                        // x^1
        for (int k = 0; k < 32; ++k) {
            x2n[k] = p;
            p = crc_multmodp(p, p);
        }
    }
    __syncthreads();
    InflateWarp& w = warps[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    for (;;) {
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(claim, 1u);
        t = __shfl_sync(kFull, t, 0);
        if ((long long)t >= n_blocks) return;
        const BgzfBlock B = blocks[t];
        uint8_t* out = text + B.out_off;
        int err = inflate_member(w, comp + B.in_off, B.in_len, out, B.out_len, lane);
        if (err == kInfOk) {
            __syncwarp();
            const unsigned L = B.out_len, S = (L + 31) >> 5;
            const unsigned lo = min(lane * S, L), hi = min(lo + S, L);
            unsigned c = ~0u;
            for (unsigned k = lo; k < hi; ++k) c = crc_tab[(c ^ out[k]) & 255u] ^ (c >> 8);
            c = ~c;
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned other = __shfl_down_sync(kFull, c, d);
                if ((lane & (2 * d - 1)) == 0) {
                    const unsigned b0 = min((lane + d) * S, L), b1 = min((lane + 2 * d) * S, L);
                    c = crc_multmodp(crc_x8n(b1 - b0, x2n), c) ^ other;
                }
            }
            if (__shfl_sync(kFull, c, 0) != B.crc) err = kInfCrc;
        }
        if (lane == 0) status[t] = (uint8_t)err;
    }
}

}  // namespace rt
