"""``split_bam`` on the GPU (mirror of ribotricer/bam.py:33-153).

The host keeps the BAM decode (pysam, as the north star prescribes) and turns
every alignment record into seven small columns; the read filter cascade, the
strand / 5'-end rule, the per-length totals and the binning itself run in the
K1 kernel (``bin_psites_kernel``).  Because pysam is not installable in every
environment, the same columns can also be loaded from a ``.npz`` file
(``save_read_columns``) -- that is what the tests and the benchmark use.
"""
from __future__ import annotations

from collections import Counter, defaultdict
from dataclasses import dataclass

import numpy as np

from . import _lib
from .const import DEFAULT_PAD
from .engine import READ_COLUMNS, Engine, make_len_table


@dataclass
class ReadColumns:
    """Decoded alignment records (structure of arrays) + the BAM header's contig table."""
    contig_names: list
    contig_len: np.ndarray
    cols: dict              # name -> numpy array, see engine.READ_COLUMNS; optional host-only extras "pos" and
                            # "ref_end" (reference_start / reference_end, -1 = None) for infer_protocol
    sorted_by_coordinate: bool = False

    def __len__(self) -> int:
        return len(self.cols["ref_id"])


def save_read_columns(path: str, reads: ReadColumns) -> None:
    np.savez(path, contig_names=np.array(reads.contig_names), contig_len=reads.contig_len,
             sorted_by_coordinate=np.array(reads.sorted_by_coordinate), **reads.cols)


def encode_nh(tags: dict) -> int:
    """The ``nh`` column: how ``dict(read.get_tags())["NH"] == 1`` (common.py:53-56) turns out.
    0 = no NH tag, 1 = equal to 1, anything else = present and different from 1."""
    if "NH" not in tags:
        return 0
    v = tags["NH"]
    if isinstance(v, (int, float)) and not isinstance(v, bool):
        if v == 1:
            return 1
        if isinstance(v, int) and 2 <= v <= 254:
            return int(v)
    return 255


def _matched_span(read):
    """first/last matched reference position and their count, i.e. what
    ``read.get_reference_positions()`` (bam.py:95) would give for [0], [-1] and len():
    only M, = and X operations contribute positions."""
    first, last, n = 0, 0, 0
    pos = read.reference_start
    for op, length in read.cigartuples or ():
        if op in (0, 7, 8):          # M, =, X
            if n == 0:
                first = pos
            last = pos + length - 1
            n += length
            pos += length
        elif op in (2, 3):           # D, N consume the reference only
            pos += length
    return first, last, n


def read_bam_columns(bam_path: str) -> ReadColumns:
    """Decode a BAM into read columns with pysam (host I/O; not on the measured path)."""
    try:
        import pysam
    except ImportError as exc:
        raise RuntimeError(
            "pysam is required to decode BAM files and is not installed here; pass decoded read columns "
            "as a .npz file instead (ribotricer_b200.bam.save_read_columns)") from exc
    bam = pysam.AlignmentFile(bam_path, "rb")
    names = list(bam.references)
    lens = np.array(bam.lengths, np.int64)
    acc = {name: [] for name, _ in READ_COLUMNS}
    acc["pos"], acc["ref_end"] = [], []
    for read in bam.fetch(until_eof=True):      # bam.py:71
        first, last, n = _matched_span(read)
        acc["ref_id"].append(read.reference_id if read.reference_id is not None else -1)
        acc["first"].append(first)
        acc["last"].append(last)
        acc["mlen"].append(min(n, 65535))
        acc["flag"].append(read.flag)
        acc["mapq"].append(read.mapping_quality)
        acc["nh"].append(encode_nh(dict(read.get_tags())))     # common.py:53-56
        acc["pos"].append(read.reference_start)
        acc["ref_end"].append(-1 if read.reference_end is None else read.reference_end)
    so = bam.header.to_dict().get("HD", {}).get("SO", "") == "coordinate"
    bam.close()
    cols = {k: np.asarray(acc[k], dt) for k, dt in READ_COLUMNS}
    cols["pos"], cols["ref_end"] = np.asarray(acc["pos"], np.int32), np.asarray(acc["ref_end"], np.int32)
    return ReadColumns(names, lens, cols, so)


def read_bam_columns_native(bam_path: str, n_threads: int = 0) -> ReadColumns:
    """Decode a BAM with the native BGZF/BAM reader (csrc/rt_bam.cpp, multi-threaded inflate);
    same columns as ``read_bam_columns``, no pysam needed."""
    import ctypes as C

    lib = _lib.load()
    handle = C.c_void_p()
    if lib.rt_bam_load(str(bam_path).encode(), int(n_threads), C.byref(handle)) != 0:
        raise OSError(f"cannot decode {bam_path}: {lib.rt_bam_last_error().decode()}")
    try:
        n = int(lib.rt_bam_n_reads(handle))
        cols = {name: np.empty(n, dt) for name, dt in READ_COLUMNS}
        lib.rt_bam_copy(handle, *[cols[name].ctypes.data_as(C.c_void_p) for name, _ in READ_COLUMNS])
        cols["pos"], cols["ref_end"] = np.empty(n, np.int32), np.empty(n, np.int32)
        lib.rt_bam_copy_span(handle, cols["pos"].ctypes.data_as(C.c_void_p), cols["ref_end"].ctypes.data_as(C.c_void_p))
        n_ref = lib.rt_bam_n_ref(handle)
        names = [lib.rt_bam_ref_name(handle, i).decode() for i in range(n_ref)]
        lens = np.array([lib.rt_bam_ref_len(handle, i) for i in range(n_ref)], np.int64)
        return ReadColumns(names, lens, cols, bool(lib.rt_bam_sorted(handle)))
    finally:
        lib.rt_bam_free(handle)


def load_reads(path) -> ReadColumns:
    """BAM (native decoder; ``RIBOTRICER_B200_PYSAM=1`` forces pysam) or ``.npz`` of decoded columns."""
    import os

    if isinstance(path, ReadColumns):
        return path
    if str(path).endswith(".npz"):
        z = np.load(path, allow_pickle=False)
        cols = {name: np.ascontiguousarray(z[name], dt) for name, dt in READ_COLUMNS}
        for extra in ("pos", "ref_end"):
            if extra in z:
                cols[extra] = np.ascontiguousarray(z[extra], np.int32)
        so = bool(z["sorted_by_coordinate"]) if "sorted_by_coordinate" in z else False
        return ReadColumns([str(c) for c in z["contig_names"]], np.asarray(z["contig_len"], np.int64), cols, so)
    if os.environ.get("RIBOTRICER_B200_PYSAM") == "1":
        return read_bam_columns(path)
    return read_bam_columns_native(path)


class Alignments:
    """What ``split_bam`` returns: the library's reads, resident on the GPU.

    The reference returns ``alignments[length][strand][(chrom, pos)] -> count``
    (bam.py:29,135); here the same information stays in HBM -- as the 4 B/read record stream of
    ``rt_stream_pack`` when the library is coordinate-sorted, else as the decoder's 18 B/read columns -- and is
    binned on demand (per length for the metagene step, merged for scoring)."""

    def __init__(self, engine: Engine, reads: ReadColumns, protocol: str, read_lengths=None):
        self.engine = engine
        self.reads = reads
        self.protocol = protocol
        self.read_lengths = None if read_lengths is None else [int(x) for x in read_lengths]
        self.n = len(reads)
        self.sorted = reads.sorted_by_coordinate
        self.dcols = self.dstream = None
        if self.sorted and self.n:
            try:
                self.dstream = engine.upload_stream(engine.stream_reads(reads.cols))
            except _lib.RtError:       # "sorted" in the header, but the positions descend somewhere: plain columns
                self.dstream = None
        if self.dstream is None:
            self.dcols = engine.upload_reads(reads.cols)
        self.stats: dict = {}
        self.read_length_counts: dict = {}

    def count(self):
        """Filter cascade + per-length totals (bam.py:73-91,136) without storing coverage."""
        eng = self.engine
        eng.set_length_table(None, self.read_lengths)     # no offsets: nothing is binned
        cov = eng.torch.zeros(1, dtype=eng.torch.int32, device=eng.device)
        stats, lc = eng.new_bin_accumulators()
        self._bin(cov, stats, lc, 1)
        st = stats.cpu().numpy()
        lcn = lc.cpu().numpy()
        self.stats = dict(zip(_lib.ST_NAMES, st.tolist()))
        rlc = defaultdict(int)
        for length in np.flatnonzero(lcn):
            rlc[int(length)] = int(lcn[length])
        self.read_length_counts = rlc
        return self.stats, rlc

    def bin_into(self, cov, psite_offsets: dict, weight: int = 1):
        """merge_read_lengths (detect_orfs.py:54-83): bin P-sites of the lengths in
        ``psite_offsets`` into ``cov``."""
        eng = self.engine
        eng.set_length_table(psite_offsets, self.read_lengths)
        stats, lc = eng.new_bin_accumulators()
        self._bin(cov, stats, lc, weight)
        return stats

    def _bin(self, cov, stats, lc, weight):
        """K1 on the resident library: the stream kernel or the column kernel, same results."""
        if self.dstream is not None:
            self.engine.bin_stream_device(cov, self.dstream, self.protocol, stats, lc, weight=weight)
        else:
            self.engine.bin_reads_device(cov, self.dcols, self.protocol, stats, lc, self.sorted, n=self.n, weight=weight)


    def to_dict(self):
        """The reference's ``alignments[length][strand][(chrom, pos)] -> count`` view (bam.py:29,135),
        rebuilt by binning one read length at a time with offset 0.  Small libraries / tests only."""
        from .detect_orfs import MergedAlignments

        if not self.read_length_counts:
            self.count()
        eng = self.engine
        out = defaultdict(lambda: defaultdict(Counter))
        for length in sorted(self.read_length_counts):
            cov = eng.new_coverage()
            self.bin_into(cov, {length: 0})
            for strand, ctr in MergedAlignments(eng, cov).to_dict().items():
                out[length][strand] = ctr
        return out


def bam_summary_text(stats: dict, read_length_counts: dict) -> str:
    """Text of ``{prefix}_bam_summary.txt`` exactly as bam.py:141-148 formats it."""
    summary = (
        f"summary:\n\ttotal_reads: {stats['total']}\n\tunique_mapped: {stats['valid']}\n"
        f"\tqcfail: {stats['qcfail']}\n\tduplicate: {stats['duplicate']}\n\tsecondary: {stats['secondary']}\n"
        f"\tunmapped:{stats['unmapped']}\n\tmulti:{stats['multi']}\n\nlength dist:\n"
    )
    for length in sorted(read_length_counts):
        summary += f"\t{length}: {read_length_counts[length]}\n"
    return summary


def split_bam(bam_path, protocol: str, prefix: str, read_lengths=None, engine: Engine | None = None):
    """Mirror of ``split_bam(bam_path, protocol, prefix, read_lengths=None)`` (bam.py:33-38).

    Returns ``(alignments, read_length_counts)``; writes ``{prefix}_bam_summary.txt``.
    ``bam_path`` may be a BAM, a ``.npz`` of decoded columns or a ``ReadColumns``.
    """
    from .detect_orfs import get_engine

    reads = load_reads(bam_path)
    eng = engine or get_engine()
    if (list(eng.contig_names) != list(reads.contig_names) or eng.pad != DEFAULT_PAD
            or not np.array_equal(eng.contig_len, reads.contig_len)):
        eng.set_genome(reads.contig_names, reads.contig_len, DEFAULT_PAD)
    eng.ensure_dense()
    alignments = Alignments(eng, reads, protocol, read_lengths)
    stats, rlc = alignments.count()
    with open(f"{prefix}_bam_summary.txt", "w") as output:
        output.write(bam_summary_text(stats, rlc))
    return alignments, rlc


__all__ = ["ReadColumns", "Alignments", "split_bam", "load_reads", "save_read_columns", "read_bam_columns",
           "bam_summary_text", "make_len_table"]
