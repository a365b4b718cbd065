/*
 * ribotricer_b200.h -- C ABI of the B200-native detect-orfs scoring path.
 *
 * The reference (smithlabcode/ribotricer v1.5.0) is pure Python and has no
 * FFI; the boundary it offers for this path is its function surface
 * (SURVEY.md 8(b)).  Each entry point below names the reference function it
 * replaces (paths relative to the reference tree).  The ctypes binding a
 * maintainer would add on the reference side is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C, no torch types; every function returns 0 on success or a
 *     negative RT_E* code, and rt_last_error() gives the message;
 *   - one rt_ctx per (process, device); a ctx is not thread-safe;
 *   - "d_" pointers are DEVICE pointers owned by the caller (e.g. torch
 *     tensors), "h_" pointers are HOST pointers; `stream` is a cudaStream_t
 *     (NULL = default stream); device-pointer calls only enqueue work;
 *   - there is no CPU fallback anywhere: without a CUDA device rt_create fails.
 *
 * Data layout in HBM
 *   coverage   int32 [2][plane]   plane 0 = '+' strand, plane 1 = '-' strand,
 *              slot(contig c, 1-based pos) = contig_base[c] + pad + pos,
 *              contig strides rounded up to 32 elements (128 B), `pad` slots
 *              of slack on both sides of every contig so that P-sites shifted
 *              off a contig end (pos <= 0 or > len) keep a private slot.
 *              This is the default, dense layout; rt_set_layout(ctx, RT_LAYOUT_COMPACT)
 *              switches to a buffer that holds only the slots the index reads (see
 *              below) -- same arguments, same results, 13x smaller for a human index.
 *   reads      structure of arrays, one element per alignment record:
 *              ref_id i32 | first i32 | last i32 | mlen u16 | flag u16 |
 *              mapq u8 | nh u8          (18 B / read)
 *              first/last = 0-based first/last matched reference position
 *              (pysam get_reference_positions()[0] / [-1], bam.py:95),
 *              mlen = number of matched positions (bam.py:99), flag = SAM flag,
 *              nh = the NH tag as common.py:53-56 tests it: 0 = absent, 1 = present and equal
 *              to 1, any other value = present and different from 1 (rt_bam_* stores 2..254 as
 *              is and 255 for values <= 0, > 254 or of a non-numeric type).
 *   index      CSR over candidate ORFs in index-file order: exon_ptr[n+1],
 *              exon_start/exon_end (1-based closed, ascending, orf.py:100),
 *              orf_contig (-1 = contig unknown to the genome table),
 *              orf_strand (0 '+', 1 '-', anything else = no coverage).
 */
#ifndef RIBOTRICER_B200_H
#define RIBOTRICER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 3

/* read-length table: one int32 per matched length = the P-site offset of that length (may be negative:
 * align_metagenes returns lag + 12 with lag in [-min(base, length), ...), metagene.py:319-324; |offset| <=
 * RT_MAX_OFFSET) or one of two sentinels that lie outside the range of offsets */
#define RT_LEN_TABLE 65536
#define RT_MAX_OFFSET 65535
#define RT_LEN_UNUSED (-2147483647 - 1)  /* length kept by split_bam but absent from psite_offsets
                                            (dropped by merge_read_lengths, detect_orfs.py:74) */
#define RT_LEN_FILTERED (-2147483647)    /* length not in --read_lengths (bam.py:101) */

/* protocol (bam.py:105,118); any other value stores no read, like the reference */
#define RT_PROTOCOL_FORWARD 0
#define RT_PROTOCOL_REVERSE 1
#define RT_PROTOCOL_NONE 2

/* stats[] slots written by rt_bin_reads (bam.py:61,141-146) */
enum {
    RT_ST_TOTAL = 0, RT_ST_QCFAIL, RT_ST_DUPLICATE, RT_ST_SECONDARY, RT_ST_UNMAPPED,
    RT_ST_MULTI, RT_ST_VALID,
    RT_ST_OOB,     /* valid reads whose P-site falls outside the padded contig */
    RT_ST_BADREF,  /* ref_id outside the contig table (reference_name is None) */
    RT_N_STATS
};

enum {
    RT_OK = 0, RT_EINVAL = -1, RT_ECUDA = -2, RT_ENOMEM = -3, RT_ESTATE = -4
};

typedef struct rt_ctx rt_ctx;

/* filter thresholds of export_orf_coverages (detect_orfs.py:209-215,289-299) */
typedef struct rt_score_params {
    double phase_score_cutoff;
    double min_valid_codons;
    double min_reads_per_codon;
    double min_valid_codons_ratio;
    double min_density_over_orf;
} rt_score_params;

/* per-ORF result columns (any pointer except score/valid/count/length may be NULL) */
typedef struct rt_score_out {
    double*  score;      /* phase score, statistics.py:115                      */
    int32_t* valid;      /* valid codons of the winning frame, statistics.py:110 */
    int64_t* count;      /* read_count, detect_orfs.py:278                      */
    int32_t* length;     /* profile length, detect_orfs.py:279                  */
    int32_t* min_codon;  /* min over codon sums (common.py:177-179), saturated  */
    uint8_t* status;     /* 1 = translating, detect_orfs.py:289-299             */
    int32_t* frame_K;    /* optional diagnostics [n][3]: kept codons per frame  */
    double*  frame_s;    /* optional diagnostics [n][3]: coherence per frame (NaN if undefined) */
} rt_score_out;

int rt_abi_version(void);
const char* rt_last_error(const rt_ctx* ctx);   /* ctx may be NULL (creation errors) */

int rt_create(int device, rt_ctx** out);
void rt_destroy(rt_ctx* ctx);
int rt_device_count(void);

/* ---- genome table: replaces the (chrom, pos) dict keys of AlignmentDict (bam.py:29) ---- */
int rt_set_genome(rt_ctx* ctx, int n_contig, const int64_t* h_contig_len, int pad);
int64_t rt_plane_elems(const rt_ctx* ctx);                 /* int32 elements per strand plane */
int rt_get_contig_base(const rt_ctx* ctx, int64_t* h_out); /* n_contig values */

/* ---- read-length table: --read_lengths (bam.py:101) + psite_offsets (detect_orfs.py:74-81) ---- */
int rt_set_length_table(rt_ctx* ctx, const int32_t* h_len_table /* RT_LEN_TABLE */);

/*
 * ---- K1: split_bam per-read loop (bam.py:71-137) fused with merge_read_lengths
 *      (detect_orfs.py:54-83) on decoded read columns.
 * Adds into d_cov (2*plane int32; clear it first for a fresh library),
 * accumulates into d_stats[RT_N_STATS] and d_len_counts[RT_LEN_TABLE] (int64).
 * `sorted_hint` != 0 promises reads grouped by reference (a coordinate-sorted BAM); the device-pointer
 * entry ignores it, the host-pointer entry uses it to ship packed records (below).  Results are identical
 * either way.
 * `weight` is +1 to add a library, or -1 to take the same reads out again
 * (coverage, stats and length counts all return to their previous values),
 * which recycles a resident coverage buffer without a multi-GB memset.
 */
int rt_bin_reads(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* d_ref_id,
                 const int32_t* d_first, const int32_t* d_last, const uint16_t* d_mlen,
                 const uint16_t* d_flag, const uint8_t* d_mapq, const uint8_t* d_nh,
                 int protocol, int sorted_hint, int weight, int64_t* d_stats,
                 int64_t* d_len_counts, void* stream);

/* Same with HOST columns (what a BAM decoder produces, 18 B/read): chunked, double-buffered H2D overlapped with the
 * kernel; h_stats / h_len_counts receive the totals (they are overwritten, not added to).  With `sorted_hint` every
 * chunk crosses PCIe as a 4 B/read record stream (rt_stream_pack below): host threads delta-code chunk k+1 while
 * chunk k is on the wire and K1 runs on the stream; a chunk that cannot be coded (not sorted after all) is sent as
 * plain columns.  Returns after the work has completed. */
int rt_bin_reads_host(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* h_ref_id,
                      const int32_t* h_first, const int32_t* h_last, const uint16_t* h_mlen,
                      const uint16_t* h_flag, const uint8_t* h_mapq, const uint8_t* h_nh,
                      int protocol, int sorted_hint, int64_t* h_stats, int64_t* h_len_counts);

/*
 * ---- K1 on PACKED read records: 11 B/read over PCIe instead of 18.  `first`, `last`, `mlen` are the
 * columns above; `meta` (u8) replaces flag, mapq and nh -- bits 0-2 hold the outcome of the filter
 * cascade (bam.py:77-91 + common.py:33-69), decided on the host: 0 = passed, else RT_ST_QCFAIL ..
 * RT_ST_MULTI; bit 3 = is_reverse -- and ref_id is run-length coded: reads [run_start[r],
 * run_start[r+1]) belong to reference run_ref[r] (a coordinate-sorted BAM has one run per reference).
 * rt_pack_read_meta builds meta and the run table from the columns (RT_ESTATE if there are more than
 * run_cap runs: the input is not grouped by reference, use rt_bin_reads_host).  Results are identical
 * to rt_bin_reads on the same reads.  `read_base` = number of the launch's first read in the run table.
 */
int rt_pack_read_meta(int64_t n, const int32_t* h_ref_id, const uint16_t* h_flag, const uint8_t* h_mapq,
                      const uint8_t* h_nh, uint8_t* h_meta, int64_t run_cap, int64_t* h_run_start /* run_cap+1 */,
                      int32_t* h_run_ref /* run_cap */, int64_t* n_runs);
int rt_bin_reads_packed(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* d_first, const int32_t* d_last,
                        const uint16_t* d_mlen, const uint8_t* d_meta, int64_t read_base, int64_t n_runs,
                        const int64_t* d_run_start, const int32_t* d_run_ref, int protocol, int weight,
                        int64_t* d_stats, int64_t* d_len_counts, void* stream);
int rt_bin_reads_packed_host(rt_ctx* ctx, int32_t* d_cov, int64_t n, const int32_t* h_first, const int32_t* h_last,
                             const uint16_t* h_mlen, const uint8_t* h_meta, int64_t n_runs,
                             const int64_t* h_run_start, const int32_t* h_run_ref, int protocol,
                             int64_t* h_stats, int64_t* h_len_counts);

/*
 * ---- K1 on a RECORD STREAM: a coordinate-sorted library as 4-byte delta-coded records (a quarter of the 18 B/read
 *      columns over PCIe and out of HBM).  Same loop as above (bam.py:71-137 + detect_orfs.py:54-83), identical results.
 * Records come in blocks of RT_STREAM_BLOCK; block b has the 16-byte header h_hdr[4b] = ref_id of all its reads,
 * h_hdr[4b+1] = the position its deltas start from, h_hdr[4b+2] = h_hdr[4b+3] = 0 (reserved).  One warp takes one
 * block: K1 runs a few persistent CTAs per SM whose warps walk the blocks independently, each with its own
 * shared-memory ring filled by cp.async.bulk (TMA) one block ahead.  A record is one little-endian u32:
 *   read       bits 0-14 delta = first - first of the previous read (or the header position), bit 15 = 0,
 *              bits 16-23 mlen & 255, bits 24-31 the RAW bits the filter cascade reads (it is evaluated on the
 *              device): RT_STREAM_UNMAPPED / SECONDARY / QCFAIL / DUPLICATE / REVERSE = SAM flags 0x4 / 0x100 /
 *              0x200 / 0x400 / 0x10, bits 5-6 = what common.py:33-69 looks at (RT_STREAM_NH_*: NH absent and
 *              MAPQ != 255, NH absent and MAPQ == 255, NH == 1, NH present and != 1), bit 7 RT_STREAM_EXT = an
 *              extension record follows (never in another block);
 *   extension  bits 15,14 = 1,1: bits 0-7 = mlen >> 8, bits 16-31 | bits 8-13 << 16 = last - first + 1 - mlen
 *              (the reference positions a spliced or deleted-from read skips; < 2^22);
 *   skip       bits 15,14 = 1,0: advances the position by bits 16-31 | bits 0-13 << 16 without being a read
 *              (gaps above 32767 nt; RT_STREAM_NULL = skip 0 pads the last block of a range).
 * Reads whose category the flags decide (unmapped, secondary, qcfail, duplicate) carry delta 0 and mlen 0: the
 * reference never looks at their position.  rt_stream_pack builds the stream from the decoder's columns with
 * `n_threads` host threads (<= 0: all cores), every RT_STREAM_RANGE reads starting a fresh block.  A read that
 * starts before its predecessor (a CIGAR that opens with D or N) starts a block of its own; the call returns
 * RT_ESTATE when the stream would be more than half padding (the library is not coordinate-sorted) or when a read
 * spans 2^22 nt more than it matches -- use rt_bin_reads / rt_bin_reads_host then.  With h_records == NULL it only
 * counts: *n_blocks = the capacity the real call needs.
 */
#define RT_STREAM_BLOCK 256
#define RT_STREAM_RANGE (1 << 20)
#define RT_STREAM_SPECIAL 0x8000u
#define RT_STREAM_KIND_EXT 0x4000u
#define RT_STREAM_NULL 0x8000u
#define RT_STREAM_UNMAPPED 0x01u
#define RT_STREAM_SECONDARY 0x02u
#define RT_STREAM_QCFAIL 0x04u
#define RT_STREAM_DUPLICATE 0x08u
#define RT_STREAM_REVERSE 0x10u
#define RT_STREAM_NH_ABSENT 0u
#define RT_STREAM_NH_ABSENT_MAPQ255 1u
#define RT_STREAM_NH_ONE 2u
#define RT_STREAM_NH_OTHER 3u
#define RT_STREAM_EXT 0x80u
int rt_stream_pack(int64_t n, const int32_t* h_ref_id, const int32_t* h_first, const int32_t* h_last,
                   const uint16_t* h_mlen, const uint16_t* h_flag, const uint8_t* h_mapq, const uint8_t* h_nh,
                   int n_threads, int64_t cap_blocks, uint32_t* h_records /* cap_blocks * RT_STREAM_BLOCK */,
                   int32_t* h_hdr /* 4 * cap_blocks */, int64_t* n_blocks);
int rt_bin_stream(rt_ctx* ctx, int32_t* d_cov, int64_t n_blocks, const uint32_t* d_records /* 16-byte aligned */,
                  const int32_t* d_hdr /* 16-byte aligned */, int protocol, int weight, int64_t* d_stats, int64_t* d_len_counts,
                  void* stream);
int rt_bin_stream_host(rt_ctx* ctx, int32_t* d_cov, int64_t n_blocks, const uint32_t* h_records, const int32_t* h_hdr,
                       int protocol, int64_t* h_stats, int64_t* h_len_counts);
/* A whole library into a coverage buffer of the COMPACT layout that need NOT be cleared first: the call overwrites
 * every slot.  The compact buffer is cut into one zone per stream block and strand (from the rank of the block's header
 * position to that of the next block's); a block zeroes its zones with plain stores and adds its own reads into the
 * lines it has just written, so neither the clear of the buffer nor the read half of the scatter's read-modify-write
 * reaches DRAM.  Reads whose P-site falls outside their block's zone (a few per thousand at block edges; any read of
 * a stream that is not sorted) are added afterwards from a spill list.  Same results as rt_clear_coverage +
 * rt_bin_stream(weight 1); the stats and length counts are added to, as everywhere. */
int rt_bin_stream_fresh(rt_ctx* ctx, int32_t* d_cov, int64_t n_blocks, const uint32_t* d_records /* 16-byte aligned */,
                        const int32_t* d_hdr /* 16-byte aligned */, int protocol, int64_t* d_stats,
                        int64_t* d_len_counts, void* stream);

int rt_clear_coverage(rt_ctx* ctx, int32_t* d_cov, void* stream);

/*
 * Coverage layout.  RT_LAYOUT_DENSE (default): the genome-wide planes described at the top, needed
 * by the WIG export and the metagene windows.  RT_LAYOUT_COMPACT (after rt_set_index): the buffer
 * holds only the slots some candidate ORF reads -- the union of all exon intervals, in genome order,
 * back to back (human GENCODE index: 1.8 GB instead of 24.7 GB).  K1 maps a P-site to its compact
 * slot through a bitmap+rank table and drops P-sites no ORF can see; scoring and rt_gather_profiles
 * return exactly what they return on the dense planes.  The layout applies to every later call that
 * takes d_cov; rt_coverage_elems gives the int32 element count a buffer of the current layout needs.
 * In the compact layout rt_clear_touched is a plain memset of that buffer.
 */
#define RT_LAYOUT_DENSE 0
#define RT_LAYOUT_COMPACT 1
int rt_set_layout(rt_ctx* ctx, int layout);
int64_t rt_coverage_elems(const rt_ctx* ctx);

/* Sparse clear for a resident coverage buffer that is recycled library after library: with tracking
 * on, K1 (weight +1) appends every slot it bumps to a ctx-owned list (8 B per read at most) and
 * rt_clear_touched zeroes exactly those slots -- a fraction of a millisecond instead of a
 * 2 * plane * 4 B memset (24.7 GB for the human genome) or a second K1 pass with weight -1. */
int rt_track_touched(rt_ctx* ctx, int enable);
int rt_clear_touched(rt_ctx* ctx, int32_t* d_cov, void* stream);

/* ---- index: ORF.from_string rows (orf.py:121-182) packed as CSR; kept resident on the device ---- */
int rt_set_index(rt_ctx* ctx, int64_t n_orf, const int64_t* h_exon_ptr, const int32_t* h_exon_start,
                 const int32_t* h_exon_end, const int32_t* h_orf_contig, const uint8_t* h_orf_strand);
int64_t rt_index_orfs(const rt_ctx* ctx);
/* algorithmic bytes of scoring ORFs [lo, hi): sum of 4L + 8E + 42 (BASELINE.md 4.5) */
int64_t rt_index_score_bytes(const rt_ctx* ctx, int64_t orf_lo, int64_t orf_hi);
/* total profile length (nt) of ORFs [lo, hi) */
int64_t rt_index_total_nt(const rt_ctx* ctx, int64_t orf_lo, int64_t orf_hi);
/* cut [0, n_orf) into n_shards contiguous, byte-balanced ranges; h_bounds has n_shards+1 entries */
int rt_shard_bounds(const rt_ctx* ctx, int n_shards, int64_t* h_bounds);

/*
 * ---- K2+K3: per-ORF body of export_orf_coverages (detect_orfs.py:274-299):
 *      orf_coverage (:134-203) + phasescore (statistics.py:48-115) +
 *      collapse_coverage_to_codon (common.py:164-180) + status predicate.
 * Scores ORFs [orf_lo, orf_hi); output element k belongs to ORF orf_lo + k.
 */
int rt_score(rt_ctx* ctx, const int32_t* d_cov, int64_t orf_lo, int64_t orf_hi,
             const rt_score_params* params, const rt_score_out* d_out, void* stream);
/* Same with HOST result columns (device scratch is owned by the ctx; D2H inside).  A range of a million ORFs or more is
 * scored in four byte-balanced parts, the columns of one part crossing PCIe while the next is scored. */
int rt_score_host(rt_ctx* ctx, const int32_t* d_cov, int64_t orf_lo, int64_t orf_hi,
                  const rt_score_params* params, const rt_score_out* h_out);

/*
 * ---- K4: the `profile` column (detect_orfs.py:322): orf_coverage of selected ORFs,
 *      written at d_out[d_out_ptr[i] ...] (lengths as reported by rt_score).
 */
int rt_gather_profiles(rt_ctx* ctx, const int32_t* d_cov, int64_t n_sel, const int64_t* d_orf_ids,
                       const int64_t* d_out_ptr, int32_t* d_out, void* stream);

/*
 * ---- a library binned into the DENSE planes, copied into a buffer of the COMPACT layout (after rt_set_index; the
 *      layout setting of the ctx does not matter): lets export_orf_coverages (detect_orfs.py:206-324) score with the
 *      compact-layout kernels a coverage that export_wig (detect_orfs.py:327-351) needed genome-wide.
 */
int rt_compact_from_dense(rt_ctx* ctx, const int32_t* d_dense, int32_t* d_compact, void* stream);

/*
 * ---- export_wig (detect_orfs.py:327-351), device side: the non-zero slots of d_cov[0, n_slots) in slot order.
 *      rt_wig_count writes the number of non-zero slots of every tile (rt_wig_tiles(n_slots) tiles); the caller
 *      turns the counts into exclusive offsets (int64) and rt_wig_fill writes slot numbers (relative to d_cov) and
 *      counts at those offsets.  Replaces the sorted (chrom, pos) key walk of the reference.
 */
int64_t rt_wig_tiles(int64_t n_slots);
int rt_wig_count(rt_ctx* ctx, const int32_t* d_cov, int64_t n_slots, uint32_t* d_tile_counts, void* stream);
int rt_wig_fill(rt_ctx* ctx, const int32_t* d_cov, int64_t n_slots, const int64_t* d_tile_offsets, int64_t* d_out_slot,
                int32_t* d_out_count, void* stream);

/*
 * ---- count_orfs (count_orfs.py:28-89) on device results: coverage sums over intervals of the DENSE planes,
 *      added per group (gene).  d_iv_off = slot offset of the interval's first position (strand * plane +
 *      contig_base + pad + start), d_sums[n_group] int64 is added to (zero it first).  SURVEY.md 8(f) #4.
 */
int rt_interval_sums(rt_ctx* ctx, const int32_t* d_cov, int64_t n_iv, const int64_t* d_iv_off, const int32_t* d_iv_len,
                     const int32_t* d_iv_group, int64_t* d_sums, void* stream);

/*
 * ---- learn-cutoff bootstrap (learn_cutoff.py:88-98): out[r] = np.median(values[idx[:, r]]) for a row-major
 *      index matrix idx[n_sel][reps] (the caller draws it with NumPy's legacy generator, as the reference
 *      does, so that the replicates are the same).  Host pointers; synchronous.  SURVEY.md 8(f) #4.
 */
int rt_bootstrap_medians(rt_ctx* ctx, const double* h_values, int64_t n, const int64_t* h_idx, int64_t n_sel,
                         int64_t reps, double* h_out);

/*
 * ---- phasescore(values) (statistics.py:48-115) of ONE sequence of doubles, e.g. a metagene
 *      profile (metagene.py:243-244).  Host pointers; synchronous.
 */
int rt_phasescore_values(rt_ctx* ctx, const double* h_values, int64_t n, double* h_score, int32_t* h_valid);

/*
 * ---- native host I/O (no GPU involved; SURVEY.md 8(f) "next #3") -------------------------------
 * rt_index_load parses a prepare-orfs index (prepare_orfs.py:370-404) with the rules of
 * ORF.from_string (orf.py:121-182): 11 tab-separated columns (otherwise RT_ESTATE and the
 * reference's "unexpected number of columns" message in rt_io_last_error), intervals sorted by
 * start (orf.py:100), leading rows containing "annotated" counted (detect_orfs.py:104-118).
 * rt_tsv_* write {prefix}_translating_ORFs.tsv rows exactly as detect_orfs.py:304-323 formats them.
 */
typedef struct rt_index rt_index;
typedef struct rt_tsv rt_tsv;
const char* rt_io_last_error(void);
int rt_index_load(const char* path, rt_index** out);
void rt_index_free(rt_index* ix);
int64_t rt_index_n_orf(const rt_index* ix);
int64_t rt_index_n_exon(const rt_index* ix);
int64_t rt_index_n_annotated_prefix(const rt_index* ix);
int rt_index_n_chrom(const rt_index* ix);                    /* distinct chrom names, first-appearance order */
const char* rt_index_chrom_name(const rt_index* ix, int i);
/* copy the columns out (any pointer may be NULL): exon_ptr[n+1], exon_start/end[E], orf_chrom[n], orf_strand[n] */
int rt_index_copy(const rt_index* ix, int64_t* exon_ptr, int32_t* exon_start, int32_t* exon_end,
                  int32_t* orf_chrom, uint8_t* orf_strand);
/* raw text of column k (1 = ORF_type .. 9 = start_codon) of row `orf`; not NUL terminated */
const char* rt_index_field(const rt_index* ix, int64_t orf, int k, int* len);
int rt_tsv_open(const char* path, int write_header, rt_tsv** out);
int rt_tsv_write(rt_tsv* t, const rt_index* ix, int64_t n_sel, const int64_t* orf_ids, int64_t orf_lo,
                 const double* score, const int32_t* valid, const int64_t* count, const int32_t* length,
                 const uint8_t* status, const int64_t* prof_ptr, const int32_t* prof);
int rt_tsv_close(rt_tsv* t);
int rt_repr_double(double x, char* buf, int cap);            /* Python float repr (shortest round trip) */
/* WIG side output (detect_orfs.py:327-351): one "variableStep chrom=" block per call */
int rt_wig_open(const char* path, rt_tsv** out);
int rt_wig_block(rt_tsv* t, const char* chrom, int64_t n, const int64_t* pos, const int32_t* count);
int rt_wig_close(rt_tsv* t);

/*
 * ---- native BAM/BGZF decode to read columns (no GPU involved; SURVEY.md 8(f) "next #2") -------
 * Replaces the pysam passes of split_bam (bam.py:65-71) on the host: per record ref_id, flag,
 * mapq, the first/last/count of matched reference positions (get_reference_positions() semantics of
 * bam.py:95-99: M, = and X operations only) and the NH tag (see `nh` above, common.py:53-56).
 * Records whose fields run past their block_size are rejected ("corrupt BAM record").
 * The file is cut into batches of BGZF blocks; `n_threads` threads (<= 0: all cores) each inflate a batch (the DEFLATE
 * decoder of csrc/rt_inflate.cpp; every block is checked against the CRC-32 of its footer, and a block the decoder
 * refuses goes to zlib), walk its records in file order and decode them, so the load scales with the cores.
 * RT_BAM_ZLIB=1 in the environment uses zlib for every block (A/B timing).
 */
typedef struct rt_bam rt_bam;
const char* rt_bam_last_error(void);
int rt_bam_load(const char* path, int n_threads, rt_bam** out);
void rt_bam_free(rt_bam* b);
int64_t rt_bam_n_reads(const rt_bam* b);
int rt_bam_n_ref(const rt_bam* b);
const char* rt_bam_ref_name(const rt_bam* b, int i);
int64_t rt_bam_ref_len(const rt_bam* b, int i);
int rt_bam_sorted(const rt_bam* b);                          /* @HD SO:coordinate */
int rt_bam_copy(const rt_bam* b, int32_t* ref_id, int32_t* first, int32_t* last, uint16_t* mlen,
                uint16_t* flag, uint8_t* mapq, uint8_t* nh); /* any pointer may be NULL */
/* reference_start / reference_end of every record as infer_protocol.py:84-85 reads them (host-side protocol
 * inference only; ref_end = -1 where pysam gives None: unmapped flag or no CIGAR) */
int rt_bam_copy_span(const rt_bam* b, int32_t* pos, int32_t* ref_end);
/* the decoded reads as packed records (rt_pack_read_meta on the decoder's own columns): meta[n_reads] and the
 * run table; first / last / mlen come from rt_bam_copy */
int rt_bam_pack(const rt_bam* b, uint8_t* meta, int64_t run_cap, int64_t* run_start, int32_t* run_ref, int64_t* n_runs);
/* the decoded reads as a record stream (rt_stream_pack on the decoder's own columns; same arguments, same two-call
 * pattern: records == NULL counts the blocks).  RT_ESTATE when the BAM is not coordinate-sorted after all */
int rt_bam_stream(const rt_bam* b, int n_threads, int64_t cap_blocks, uint32_t* records, int32_t* hdr, int64_t* n_blocks);

/* Metagene sums (metagene.py:204-252, host side of the P-site offset inference): row i of the ragged matrix
 * flat[ptr[i], ptr[i+1]) holds the coverage of one annotated ORF over its first <= width positions (K4 over the truncated
 * windows).  Every row that holds a read is divided by its mean and added to the start-aligned sums and, shifted to end
 * at the last column, to the stop-aligned sums; *_cnt[k] = rows that reach column k.  All four outputs have `width`
 * entries and are overwritten.  The result does not depend on the number of host threads. */
int rt_metagene_sums(const int32_t* flat, const int64_t* ptr, int64_t n_rows, int64_t width, double* start_sum,
                     int64_t* start_cnt, double* stop_sum, int64_t* stop_cnt);

/* One raw DEFLATE stream (RFC 1951; the payload of a BGZF block, htslib's bgzf.c under pysam.AlignmentFile, bam.py:65)
 * that must inflate to exactly n_dst bytes: RT_OK, or RT_EINVAL for anything else (corrupt, truncated, a different
 * size, or a stream shape the decoder leaves to zlib).  Never writes outside dst[0, n_dst).  rt_crc32 is the gzip CRC-32
 * of a buffer (PCLMULQDQ folding where the host has it). */
int rt_inflate_raw(const uint8_t* src, int64_t n_src, uint8_t* dst, int64_t n_dst);
uint32_t rt_crc32(const uint8_t* p, int64_t n);

/*
 * ---- prepare-orfs: the candidate-ORF index from a GTF and a genome FASTA (DESIGN.md section 9) ----------------
 * Host side (no GPU involved; errors in rt_io_last_error):
 * rt_gtf_load parses the exon and CDS lines of a plain-text GTF in chunks on all cores (RT_GTF_THREADS overrides the
 * number of chunks).  Comment and blank lines are skipped; any other line must have 9 tab-separated columns and
 * integer start <= end, else RT_EINVAL with the line number.  Per kept line: 1-based line number, feature (0 exon,
 * 1 CDS), chrom, start, end, strand (0 '+', 1 '-', 2 other) and 5 attribute string ids (gene_id, transcript_id,
 * gene_name or else gene_id, gene_type or else gene_biotype, transcript_type or else transcript_biotype; -1 absent).
 * Strings are NUL-terminated, back to back, in order of first appearance (rt_gtf_string_bytes bytes in all).
 */
typedef struct rt_gtf rt_gtf;
int rt_gtf_load(const char* path, rt_gtf** out);
void rt_gtf_free(rt_gtf* g);
int64_t rt_gtf_n_lines(const rt_gtf* g);
int64_t rt_gtf_n_strings(const rt_gtf* g);
int64_t rt_gtf_string_bytes(const rt_gtf* g);
int rt_gtf_copy(const rt_gtf* g, int64_t* line_no, uint8_t* feature, int32_t* chrom, int32_t* start, int32_t* end,
                uint8_t* strand, int32_t* attr, char* strings);   /* any pointer may be NULL; attr: 5 per line */
/* rt_fasta_load reads and indexes a plain-text FASTA on all cores (contig name = header up to the first blank; '\n' and
 * '\r' are dropped; a duplicate name is RT_EINVAL).  rt_fasta_codes writes the listed contigs back to back as 1-byte
 * codes (A C G T in either case -> 0-3, anything else -> 4).  Nothing is written next to the input. */
typedef struct rt_fasta rt_fasta;
int rt_fasta_load(const char* path, rt_fasta** out);
void rt_fasta_free(rt_fasta* fa);
int rt_fasta_n_contig(const rt_fasta* fa);
const char* rt_fasta_contig_name(const rt_fasta* fa, int i);
int64_t rt_fasta_contig_len(const rt_fasta* fa, int i);
int rt_fasta_codes(const rt_fasta* fa, int n_sel, const int32_t* contigs, uint8_t* out);
/* rt_orf_write writes {prefix}_candidate_orfs.tsv: the header, then one row per entry.  tx_text[tx_text_off[t],
 * tx_text_off[t+1]) is "transcript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand" of transcript t,
 * whose first tx_id_len[t] bytes are the transcript id.  row_type: 0 annotated, 1 uORF, 2 overlap_uORF, 3 super_uORF,
 * 4 overlap_dORF, 5 dORF, 6 novel; row_codon: 6-bit codon code (16 b0 + 4 b1 + b2); intervals CSR, 1-based closed. */
int rt_orf_write(const char* path, int64_t n_tx, const char* tx_text, const int64_t* tx_text_off, const int32_t* tx_id_len,
                 int64_t n_rows, const int32_t* row_tx, const uint8_t* row_type, const uint8_t* row_codon,
                 const int64_t* iv_ptr, const int32_t* iv_start, const int32_t* iv_end);
/* Device side: rt_orf_search uploads the contig codes and the transcript table (merged exons, strand, oriented CDS
 * bounds), splices and orients every transcript (orf_splice_kernel), counts and fills its candidate rows
 * (orf_walk_kernel<false> / <true>: codon masks over the 6-bit codes, nearest in-frame stop, min length, longest, type;
 * annotated and internal ORFs are not rows) and their genomic intervals (orf_interval_kernel<true> / <false>).  Rows are
 * ordered by transcript, then start.  Returns the row and interval counts; the columns stay on the device until
 * rt_orf_fetch copies them (any pointer may be NULL; iv_ptr has n_rows + 1 entries).  stage_ms (optional) receives the
 * device time of RT_ORF_STAGES stages: upload, splice, count, row scan, fill, interval count + scan, interval fill. */
#define RT_ORF_STAGES 7
typedef struct rt_orf_query {
    int64_t n_tx;
    const int64_t* exon_ptr;        /* n_tx + 1 */
    const int32_t* exon_start;      /* merged exons, 1-based closed, ascending within a transcript */
    const int32_t* exon_end;
    const int64_t* tx_base;         /* offset of the transcript's contig in codes */
    const uint8_t* tx_strand;       /* 0 '+', 1 '-' */
    const int32_t* tx_cds;          /* 2 per transcript: oriented first / last CDS nt, or -1 -1 */
    const uint8_t* codes;           /* contig codes (rt_fasta_codes) */
    int64_t n_codes;
    uint64_t start_mask, stop_mask; /* bit c set: 6-bit codon code c is a start / stop codon */
    int32_t min_orf_length;
    int32_t longest;                /* of the starts that share a stop, keep the first only */
} rt_orf_query;
int rt_orf_search(rt_ctx* ctx, const rt_orf_query* q, int64_t* n_rows, int64_t* n_iv, float* stage_ms);
int rt_orf_fetch(rt_ctx* ctx, int32_t* row_tx, int32_t* row_start, int32_t* row_stop, uint8_t* row_type, uint8_t* row_codon,
                 int64_t* iv_ptr, int32_t* iv_start, int32_t* iv_end);

/* number of kernel launches issued through this ctx so far (bench.py's gpu_launches) */
int64_t rt_launch_count(const rt_ctx* ctx);
/* bytes of read data the host-buffer entry points (rt_bin_reads_host, rt_bin_stream_host, rt_bin_reads_packed_host) have
 * copied to the device through this ctx so far (bench.py's e2e.h2d_bytes_per_step) */
int64_t rt_h2d_bytes(const rt_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* RIBOTRICER_B200_H */
