"""Candidate-ORF index (``prepare-orfs`` output) -> CSR-packed exon intervals.

Mirrors ``ORF.from_string`` (ribotricer/orf.py:121-182), the interval sort of
``ORF.__init__`` (orf.py:100) and the ``oid`` derivation (orf.py:103), but
produces columnar arrays for the device instead of one Python object per row.
"""
from __future__ import annotations

import sys
from dataclasses import dataclass

import numpy as np

INDEX_COLUMNS = ("ORF_ID", "ORF_type", "transcript_id", "transcript_type", "gene_id", "gene_name",
                 "gene_type", "chrom", "strand", "start_codon", "coordinate")


@dataclass
class ORF:
    """One index row (same attribute names as ribotricer/orf.py:28-113)."""
    category: str
    tid: str
    ttype: str
    gid: str
    gname: str
    gtype: str
    chrom: str
    strand: str
    intervals: list      # [(start, end)], 1-based closed, sorted by start
    start_codon: str

    @property
    def oid(self) -> str:   # orf.py:101-103
        length = sum(e - s + 1 for s, e in self.intervals)
        return f"{self.tid}_{self.intervals[0][0]}_{self.intervals[-1][1]}_{length}"

    @classmethod
    def from_string(cls, line: str):
        """orf.py:121-182, same fail-fast behaviour."""
        if not line:
            print("annotation line cannot be empty")
            return None
        fields = line.split("\t")
        if len(fields) != 11:
            sys.exit("{}\n{}".format("Error: unexpected number of columns found for index file",
                                     "please run ribotricer prepare-orfs to regenerate"))
        intervals = []
        for group in fields[10].split(","):
            start, end = group.split("-")
            intervals.append((int(start), int(end)))
        intervals.sort(key=lambda iv: iv[0])   # orf.py:100
        return cls(fields[1], fields[2], fields[3], fields[4], fields[5], fields[6], fields[7],
                   fields[8], intervals, fields[9])


@dataclass
class PackedIndex:
    """The whole index in columns.  Row order = file order = output order."""
    exon_ptr: np.ndarray      # int64 [n+1]
    exon_start: np.ndarray    # int32 [E]
    exon_end: np.ndarray      # int32 [E]
    chrom: list               # str per ORF
    strand: list              # str per ORF
    fields: list              # per ORF: (category, tid, ttype, gid, gname, gtype, start_codon)
    n_annotated_prefix: int   # leading rows whose line contains 'annotated' (detect_orfs.py:104-118)

    @property
    def n_orf(self) -> int:
        return len(self.chrom)

    def lengths(self) -> np.ndarray:
        exlen = self.exon_end.astype(np.int64) - self.exon_start + 1
        cs = np.concatenate([[0], np.cumsum(exlen)])
        return cs[self.exon_ptr[1:]] - cs[self.exon_ptr[:-1]]

    def oid(self, o: int) -> str:
        a, b = self.exon_ptr[o], self.exon_ptr[o + 1]
        length = int((self.exon_end[a:b].astype(np.int64) - self.exon_start[a:b] + 1).sum())
        return f"{self.fields[o][1]}_{self.exon_start[a]}_{self.exon_end[b - 1]}_{length}"

    def contig_table(self) -> list:
        """Chromosome names in order of first appearance."""
        return list(dict.fromkeys(self.chrom))

    def device_columns(self, contig_lut: dict) -> dict:
        """CSR arrays for ``Engine.set_index``; unknown chromosomes get contig -1 and unknown
        strands code 2 (both read as zero coverage, detect_orfs.py:160-187)."""
        contig = np.fromiter((contig_lut.get(c, -1) for c in self.chrom), np.int32, self.n_orf)
        strand = np.fromiter((0 if s == "+" else 1 if s == "-" else 2 for s in self.strand), np.uint8, self.n_orf)
        return dict(exon_ptr=self.exon_ptr, exon_start=self.exon_start, exon_end=self.exon_end,
                    orf_contig=contig, orf_strand=strand)


def parse_index(path: str) -> PackedIndex:
    """Parse a ribotricer index TSV (prepare_orfs.py:370-404 layout)."""
    exon_ptr = [0]
    starts, ends = [], []
    chrom, strand, fields = [], [], []
    n_annot, in_prefix = 0, True
    with open(path) as fh:
        fh.readline()   # header (detect_orfs.py:273)
        for line in fh:
            if not line:
                continue
            f = line.split("\t")
            if len(f) != 11:   # orf.py:145-151
                sys.exit("{}\n{}".format("Error: unexpected number of columns found for index file",
                                         "please run ribotricer prepare-orfs to regenerate"))
            if in_prefix:
                if "annotated" in line:   # detect_orfs.py:104-105 tests the whole line
                    n_annot += 1
                else:
                    in_prefix = False
            ivs = []
            for group in f[10].split(","):
                s, e = group.split("-")
                ivs.append((int(s), int(e)))
            if len(ivs) > 1:
                ivs.sort(key=lambda iv: iv[0])   # orf.py:100
            for s, e in ivs:
                starts.append(s)
                ends.append(e)
            exon_ptr.append(len(starts))
            chrom.append(f[7])
            strand.append(f[8])
            fields.append((f[1], f[2], f[3], f[4], f[5], f[6], f[9]))
    return PackedIndex(np.asarray(exon_ptr, np.int64), np.asarray(starts, np.int32), np.asarray(ends, np.int32),
                       chrom, strand, fields, n_annot)


# --------------------------------------------------------------------------------------------
# Native loader (csrc/rt_host_io.cpp): same rules, no Python object per row.
# --------------------------------------------------------------------------------------------
class _RowView:
    """Indexable per-row view backed by the native index (rows are decoded on demand)."""

    def __init__(self, getter, n):
        self._get, self._n = getter, n

    def __len__(self):
        return self._n

    def __getitem__(self, o):
        if o < 0:
            o += self._n
        if not 0 <= o < self._n:
            raise IndexError(o)
        return self._get(int(o))


class NativeIndex:
    """The whole index in columns, parsed by ``rt_index_load``.  Duck-types ``PackedIndex``.  ``src`` is a path or a
    ``bgzf.NativeText`` (``rt_index_load_text``)."""

    def __init__(self, src):
        import ctypes as C

        from . import _lib
        from .bgzf import NativeText

        self._lib = lib = _lib.load()
        handle = C.c_void_p()
        if isinstance(src, NativeText):
            path = src.path
            rc = lib.rt_index_load_text(src.take(), path.encode(), C.byref(handle))
        else:
            path = src
            rc = lib.rt_index_load(path.encode(), C.byref(handle))
        if rc != 0:
            msg = lib.rt_io_last_error().decode()
            if msg.startswith("Error: unexpected number of columns"):
                sys.exit(msg)          # orf.py:145-151
            raise ValueError(f"cannot load index {path}: {msg}")
        self.handle = handle
        n = int(lib.rt_index_n_orf(handle))
        e = int(lib.rt_index_n_exon(handle))
        self.exon_ptr = np.empty(n + 1, np.int64)
        self.exon_start = np.empty(e, np.int32)
        self.exon_end = np.empty(e, np.int32)
        self.orf_chrom_id = np.empty(n, np.int32)
        self.orf_strand_code = np.empty(n, np.uint8)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        lib.rt_index_copy(handle, p(self.exon_ptr), p(self.exon_start), p(self.exon_end), p(self.orf_chrom_id),
                          p(self.orf_strand_code))
        self.chrom_names = [lib.rt_index_chrom_name(handle, i).decode() for i in range(lib.rt_index_n_chrom(handle))]
        self.n_annotated_prefix = int(lib.rt_index_n_annotated_prefix(handle))
        self._n = n
        self.fields = _RowView(self._row_fields, n)
        self.chrom = _RowView(lambda o: self.chrom_names[self.orf_chrom_id[o]], n)
        self.strand = _RowView(lambda o: self.field(o, 8), n)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.rt_index_free(self.handle)
                self.handle = None
        except Exception:
            pass

    @property
    def n_orf(self) -> int:
        return self._n

    def field(self, o: int, k: int) -> str:
        import ctypes as C

        n = C.c_int()
        ptr = self._lib.rt_index_field(self.handle, int(o), int(k), C.byref(n))
        return C.string_at(ptr, n.value).decode()

    def _row_fields(self, o: int):
        return (self.field(o, 1), self.field(o, 2), self.field(o, 3), self.field(o, 4), self.field(o, 5),
                self.field(o, 6), self.field(o, 9))

    def ids(self):
        """The ORF_ID column byte for byte (``rt_index_ids``): row o is ``blob[off[o]:off[o + 1]]`` (uint8)."""
        import ctypes as C

        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        off = np.empty(self._n + 1, np.int64)
        self._lib.rt_index_ids(self.handle, p(off), None)
        blob = np.empty(max(1, int(off[-1])), np.uint8)
        self._lib.rt_index_ids(self.handle, p(off), p(blob))
        return off, blob[:int(off[-1])]

    def lengths(self) -> np.ndarray:
        exlen = self.exon_end.astype(np.int64) - self.exon_start + 1
        cs = np.concatenate([[0], np.cumsum(exlen)])
        return cs[self.exon_ptr[1:]] - cs[self.exon_ptr[:-1]]

    def oid(self, o: int) -> str:
        a, b = self.exon_ptr[o], self.exon_ptr[o + 1]
        length = int((self.exon_end[a:b].astype(np.int64) - self.exon_start[a:b] + 1).sum())
        return f"{self.field(o, 2)}_{self.exon_start[a]}_{self.exon_end[b - 1]}_{length}"

    def contig_table(self) -> list:
        return list(self.chrom_names)

    def device_columns(self, contig_lut: dict) -> dict:
        table = np.fromiter((contig_lut.get(c, -1) for c in self.chrom_names), np.int32, len(self.chrom_names))
        contig = table[self.orf_chrom_id] if len(table) else np.zeros(0, np.int32)
        return dict(exon_ptr=self.exon_ptr, exon_start=self.exon_start, exon_end=self.exon_end,
                    orf_contig=np.ascontiguousarray(contig, np.int32), orf_strand=self.orf_strand_code)


def load_native_index(src) -> NativeIndex:
    return NativeIndex(src)
