"""ctypes binding of libribotricer_b200.so (C ABI: include/ribotricer_b200.h).

There is no CPU fallback: if the shared library is missing or no B200 is
visible, the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RT_LIB_PATH") or os.path.join(HERE, "libribotricer_b200.so")   # override: kernel A/B runs

RT_LEN_TABLE = 65536
RT_MAX_OFFSET = 65535
RT_LEN_UNUSED = -2147483648
RT_LEN_FILTERED = -2147483647
RT_PROTOCOL_FORWARD, RT_PROTOCOL_REVERSE, RT_PROTOCOL_NONE = 0, 1, 2
ST_NAMES = ("total", "qcfail", "duplicate", "secondary", "unmapped", "multi", "valid", "oob", "badref")
RT_N_STATS = len(ST_NAMES)
RT_STREAM_BLOCK = 256

EXPORTS = (
    "rt_abi_version", "rt_last_error", "rt_create", "rt_destroy", "rt_device_count",
    "rt_set_genome", "rt_plane_elems", "rt_get_contig_base", "rt_set_length_table",
    "rt_bin_reads", "rt_bin_reads_host", "rt_pack_read_meta", "rt_bin_reads_packed", "rt_bin_reads_packed_host", "rt_stream_pack", "rt_bin_stream", "rt_bin_stream_host", "rt_bin_stream_fresh", "rt_clear_coverage", "rt_set_layout", "rt_coverage_elems", "rt_track_touched", "rt_clear_touched", "rt_set_index", "rt_index_orfs",
    "rt_index_score_bytes", "rt_index_total_nt", "rt_shard_bounds", "rt_score", "rt_score_host",
    "rt_gather_profiles", "rt_compact_from_dense", "rt_wig_tiles", "rt_wig_count", "rt_wig_fill", "rt_interval_sums", "rt_bootstrap_medians", "rt_launch_count", "rt_h2d_bytes", "rt_phasescore_values", "rt_io_last_error", "rt_index_load",
    "rt_index_free", "rt_index_n_orf", "rt_index_n_exon", "rt_index_n_annotated_prefix", "rt_index_n_chrom",
    "rt_index_chrom_name", "rt_index_copy", "rt_index_field", "rt_tsv_open", "rt_tsv_write", "rt_tsv_close",
    "rt_repr_double", "rt_wig_open", "rt_wig_block", "rt_wig_close", "rt_bam_last_error", "rt_bam_load", "rt_bam_free", "rt_bam_n_reads", "rt_bam_n_ref",
    "rt_bam_ref_name", "rt_bam_ref_len", "rt_bam_sorted", "rt_bam_copy", "rt_bam_copy_span", "rt_bam_pack", "rt_bam_stream",
    "rt_inflate_raw", "rt_crc32", "rt_metagene_sums",
    "rt_gtf_load", "rt_gtf_free", "rt_gtf_n_lines", "rt_gtf_n_strings", "rt_gtf_string_bytes", "rt_gtf_copy",
    "rt_fasta_load", "rt_fasta_free", "rt_fasta_n_contig", "rt_fasta_contig_name", "rt_fasta_contig_len", "rt_fasta_codes",
    "rt_orf_write", "rt_orf_search", "rt_orf_fetch",
)
RT_ORF_STAGES = 7


class ScoreParams(C.Structure):
    _fields_ = [("phase_score_cutoff", C.c_double), ("min_valid_codons", C.c_double),
                ("min_reads_per_codon", C.c_double), ("min_valid_codons_ratio", C.c_double),
                ("min_density_over_orf", C.c_double)]


class ScoreOut(C.Structure):
    _fields_ = [("score", C.c_void_p), ("valid", C.c_void_p), ("count", C.c_void_p),
                ("length", C.c_void_p), ("min_codon", C.c_void_p), ("status", C.c_void_p),
                ("frame_K", C.c_void_p), ("frame_s", C.c_void_p)]


class OrfQuery(C.Structure):
    _fields_ = [("n_tx", C.c_int64), ("exon_ptr", C.c_void_p), ("exon_start", C.c_void_p), ("exon_end", C.c_void_p),
                ("tx_base", C.c_void_p), ("tx_strand", C.c_void_p), ("tx_cds", C.c_void_p), ("codes", C.c_void_p),
                ("n_codes", C.c_int64), ("start_mask", C.c_uint64), ("stop_mask", C.c_uint64),
                ("min_orf_length", C.c_int32), ("longest", C.c_int32)]


class RtError(RuntimeError):
    pass


_lib = None


def load():
    """Load the C-ABI library; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RtError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C ribotricer_b200/csrc`. ribotricer_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    lib.rt_abi_version.restype = i32
    lib.rt_last_error.restype = C.c_char_p
    lib.rt_last_error.argtypes = [vp]
    lib.rt_create.argtypes = [i32, C.POINTER(vp)]
    lib.rt_destroy.argtypes = [vp]
    lib.rt_destroy.restype = None
    lib.rt_set_genome.argtypes = [vp, i32, vp, i32]
    lib.rt_plane_elems.argtypes = [vp]
    lib.rt_plane_elems.restype = i64
    lib.rt_get_contig_base.argtypes = [vp, vp]
    lib.rt_set_length_table.argtypes = [vp, vp]
    lib.rt_bin_reads.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp]
    lib.rt_bin_reads_host.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp]
    lib.rt_pack_read_meta.argtypes = [i64, vp, vp, vp, vp, vp, i64, vp, vp, C.POINTER(i64)]
    lib.rt_bin_reads_packed.argtypes = [vp, vp, i64, vp, vp, vp, vp, i64, i64, vp, vp, i32, i32, vp, vp, vp]
    lib.rt_bin_reads_packed_host.argtypes = [vp, vp, i64, vp, vp, vp, vp, i64, vp, vp, i32, vp, vp]
    lib.rt_stream_pack.argtypes = [i64, vp, vp, vp, vp, vp, vp, vp, i32, i64, vp, vp, C.POINTER(i64)]
    lib.rt_bin_stream.argtypes = [vp, vp, i64, vp, vp, i32, i32, vp, vp, vp]
    lib.rt_bin_stream_host.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp]
    lib.rt_bin_stream_fresh.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp, vp]
    lib.rt_clear_coverage.argtypes = [vp, vp, vp]
    lib.rt_track_touched.argtypes = [vp, i32]
    lib.rt_set_layout.argtypes = [vp, i32]
    lib.rt_coverage_elems.argtypes = [vp]
    lib.rt_coverage_elems.restype = i64
    lib.rt_clear_touched.argtypes = [vp, vp, vp]
    lib.rt_set_index.argtypes = [vp, i64, vp, vp, vp, vp, vp]
    lib.rt_index_orfs.argtypes = [vp]
    lib.rt_index_orfs.restype = i64
    lib.rt_index_score_bytes.argtypes = [vp, i64, i64]
    lib.rt_index_score_bytes.restype = i64
    lib.rt_index_total_nt.argtypes = [vp, i64, i64]
    lib.rt_index_total_nt.restype = i64
    lib.rt_shard_bounds.argtypes = [vp, i32, vp]
    lib.rt_score.argtypes = [vp, vp, i64, i64, C.POINTER(ScoreParams), C.POINTER(ScoreOut), vp]
    lib.rt_score_host.argtypes = [vp, vp, i64, i64, C.POINTER(ScoreParams), C.POINTER(ScoreOut)]
    lib.rt_gather_profiles.argtypes = [vp, vp, i64, vp, vp, vp, vp]
    lib.rt_compact_from_dense.argtypes = [vp, vp, vp, vp]
    lib.rt_wig_tiles.argtypes = [i64]
    lib.rt_wig_tiles.restype = i64
    lib.rt_wig_count.argtypes = [vp, vp, i64, vp, vp]
    lib.rt_wig_fill.argtypes = [vp, vp, i64, vp, vp, vp, vp]
    lib.rt_interval_sums.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp]
    lib.rt_bootstrap_medians.argtypes = [vp, vp, i64, vp, i64, i64, vp]
    lib.rt_phasescore_values.argtypes = [vp, vp, i64, C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    lib.rt_launch_count.argtypes = [vp]
    lib.rt_io_last_error.restype = C.c_char_p
    lib.rt_index_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.rt_index_free.argtypes = [vp]
    lib.rt_index_free.restype = None
    for name in ("rt_index_n_orf", "rt_index_n_exon", "rt_index_n_annotated_prefix"):
        getattr(lib, name).argtypes = [vp]
        getattr(lib, name).restype = i64
    lib.rt_index_n_chrom.argtypes = [vp]
    lib.rt_index_chrom_name.argtypes = [vp, i32]
    lib.rt_index_chrom_name.restype = C.c_char_p
    lib.rt_index_copy.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.rt_index_field.argtypes = [vp, i64, i32, C.POINTER(C.c_int)]
    lib.rt_index_field.restype = vp
    lib.rt_tsv_open.argtypes = [C.c_char_p, i32, C.POINTER(vp)]
    lib.rt_tsv_write.argtypes = [vp, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.rt_tsv_close.argtypes = [vp]
    lib.rt_repr_double.argtypes = [C.c_double, C.c_char_p, i32]
    lib.rt_wig_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.rt_wig_block.argtypes = [vp, C.c_char_p, i64, vp, vp]
    lib.rt_wig_close.argtypes = [vp]
    lib.rt_bam_last_error.restype = C.c_char_p
    lib.rt_bam_load.argtypes = [C.c_char_p, i32, C.POINTER(vp)]
    lib.rt_bam_free.argtypes = [vp]
    lib.rt_bam_free.restype = None
    lib.rt_bam_n_reads.argtypes = [vp]
    lib.rt_bam_n_reads.restype = i64
    lib.rt_bam_n_ref.argtypes = [vp]
    lib.rt_bam_ref_name.argtypes = [vp, i32]
    lib.rt_bam_ref_name.restype = C.c_char_p
    lib.rt_bam_ref_len.argtypes = [vp, i32]
    lib.rt_bam_ref_len.restype = i64
    lib.rt_bam_sorted.argtypes = [vp]
    lib.rt_bam_copy.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.rt_bam_copy_span.argtypes = [vp, vp, vp]
    lib.rt_bam_pack.argtypes = [vp, vp, i64, vp, vp, C.POINTER(i64)]
    lib.rt_bam_stream.argtypes = [vp, i32, i64, vp, vp, C.POINTER(i64)]
    lib.rt_inflate_raw.argtypes = [vp, i64, vp, i64]
    lib.rt_metagene_sums.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp]
    lib.rt_crc32.argtypes = [vp, i64]
    lib.rt_crc32.restype = C.c_uint32
    lib.rt_launch_count.restype = i64
    lib.rt_h2d_bytes.argtypes = [vp]
    lib.rt_h2d_bytes.restype = i64
    lib.rt_gtf_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.rt_gtf_free.argtypes = [vp]
    lib.rt_gtf_free.restype = None
    for name in ("rt_gtf_n_lines", "rt_gtf_n_strings", "rt_gtf_string_bytes"):
        getattr(lib, name).argtypes = [vp]
        getattr(lib, name).restype = i64
    lib.rt_gtf_copy.argtypes = [vp] * 9
    lib.rt_fasta_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.rt_fasta_free.argtypes = [vp]
    lib.rt_fasta_free.restype = None
    lib.rt_fasta_n_contig.argtypes = [vp]
    lib.rt_fasta_contig_name.argtypes = [vp, i32]
    lib.rt_fasta_contig_name.restype = C.c_char_p
    lib.rt_fasta_contig_len.argtypes = [vp, i32]
    lib.rt_fasta_contig_len.restype = i64
    lib.rt_fasta_codes.argtypes = [vp, i32, vp, vp]
    lib.rt_orf_write.argtypes = [C.c_char_p, i64, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    lib.rt_orf_search.argtypes = [vp, C.POINTER(OrfQuery), C.POINTER(i64), C.POINTER(i64), vp]
    lib.rt_orf_fetch.argtypes = [vp] * 9
    if lib.rt_abi_version() != 3:
        raise RtError(f"ABI mismatch: library reports {lib.rt_abi_version()}, binding expects 3")
    _lib = lib
    return lib


def check(rc: int, ctx=None):
    if rc != 0:
        msg = load().rt_last_error(ctx)
        raise RtError(f"ribotricer_b200 error {rc}: {msg.decode() if msg else '?'}")
