"""count-orfs on the results of the GPU path (SURVEY.md 8(f) #4).

The reference's ``count_orfs`` (count_orfs.py:28-89) re-reads ``{prefix}_translating_ORFs.tsv``, parses
the ``profile`` text of every selected ORF and, per ``(gene_id, gene_name)``, keeps the first coverage seen
at every position: the union of the positions of the gene's selected ORFs, each counted once.  Two entry
points give the same table:

* ``count_orfs_device``  works on what ``detect_orfs`` already holds in HBM -- the dense P-site planes, the
  packed index and the status column -- so no profile is ever turned into text: the union intervals of every
  gene are merged on the host (a sort over exon intervals) and summed by ``rt_interval_sums``;
* ``count_orfs_gpu``     keeps the reference's signature (index path, TSV path) and reads the TSV text on the GPU
  (DESIGN.md section 13); the index and the TSV may be plain text or BGZF.  The ``count-orfs`` command runs it:

    TSV            rt_codon_load_tsv (all cores): fields, selection, ORF_ID -> index row, gene keys
    counts         Engine.orf_counts: count_emit_kernel, a stable radix sort on (gene, coordinate), count_keep_kernel
    table          write_counts

* ``count_orfs``         the same table in plain Python, from plain-text files: the statement the GPU path is
  checked against.

``count_orfs_codon`` gives the same selection at codon level (DESIGN.md section 11): per gene and pooled over all
genes, the occurrences, total, mean, median and variance of the read count of every codon.

    TSV            rt_codon_load_tsv (all cores): fields, selection, ORF_ID -> index row, gene keys
    sequences      rt_codon_load_seq (all cores): the orfs-seq nucleotide file checked against the index
    codons         Engine.codon_counts: codon_emit_kernel, radix sorts (place dedup, counts in order),
                   codon_stats_kernel
    tables         rt_codon_write: formatted on all cores, written by a write-behind thread
"""
from __future__ import annotations

import ctypes as C
import os
import pathlib
from collections import defaultdict

import numpy as np

from . import _lib
from .bgzf import NativeText, StageClock, open_texts
from .index import load_native_index

_POS_BITS = 33          # positions are int32: gene * 2^33 + (pos + 2^31) orders intervals by (gene, pos)


def _gene_groups(idx, rows):
    """Group the selected index rows by (gene_id, gene_name) (count_orfs.py:67,71)."""
    keys, lut, group = [], {}, np.empty(len(rows), np.int64)
    for k, o in enumerate(rows):
        key = (idx.field(int(o), 4), idx.field(int(o), 5))
        g = lut.get(key)
        if g is None:
            g = lut[key] = len(keys)
            keys.append(key)
        group[k] = g
    return keys, group


def _union_intervals(group, seq, start, end):
    """Merge the closed intervals of every (group, seq) into disjoint ones; inputs are flat arrays."""
    if len(group) == 0:
        z = np.zeros(0, np.int64)
        return z, z, z, z
    order = np.lexsort((start, seq, group))
    g, q, s, e = group[order], seq[order], start[order].astype(np.int64), end[order].astype(np.int64)
    key = g * 4 + q                                   # seq < 4 per group here (callers renumber)
    shift = key << _POS_BITS
    run_end = np.maximum.accumulate(shift + e + (1 << 31))
    new = np.ones(len(g), bool)
    new[1:] = (shift[1:] + s[1:] + (1 << 31)) > run_end[:-1]      # starts after everything seen so far
    first = np.flatnonzero(new)
    last_end = np.maximum.reduceat(e, first)
    return g[first], q[first], s[first], last_end


def gene_union_counts(engine, cov, idx, rows):
    """Per (gene_id, gene_name) of the selected ``rows``: (sum of coverage over the union of the positions of
    its ORFs, number of positions).  ``cov`` = dense planes of ``engine`` (``MergedAlignments.cov``)."""
    t = engine.torch
    rows = np.asarray(rows, np.int64)
    keys, group = _gene_groups(idx, rows)
    n_exon = (idx.exon_ptr[rows + 1] - idx.exon_ptr[rows]).astype(np.int64)
    ex = np.repeat(idx.exon_ptr[rows], n_exon) + (np.arange(int(n_exon.sum())) - np.repeat(np.cumsum(n_exon) - n_exon, n_exon))
    g = np.repeat(group, n_exon)
    lut = {c: i for i, c in enumerate(engine.contig_names)}
    contig_of_chrom = np.fromiter((lut.get(c, -1) for c in idx.chrom_names), np.int64, len(idx.chrom_names))
    chrom = np.repeat(idx.orf_chrom_id[rows].astype(np.int64), n_exon)
    strand = np.repeat(idx.orf_strand_code[rows].astype(np.int64), n_exon)
    # the reference keys positions by `pos` alone (count_orfs.py:80-82): a gene whose ORFs sit on one
    # (chrom, strand) -- every real gene -- is a plain interval union; anything else is redone exactly below
    seq = chrom * 4 + np.minimum(strand, 3)
    n_gene = len(keys)
    first_seq = np.full(n_gene, -1, np.int64)
    first_seq[g[::-1]] = seq[::-1]
    mixed = np.zeros(n_gene, bool)
    np.logical_or.at(mixed, g, seq != first_seq[g])
    plain = ~mixed[g]
    ug, _, us, ue = _union_intervals(g[plain], np.zeros(int(plain.sum()), np.int64), idx.exon_start[ex][plain],
                                     idx.exon_end[ex][plain])
    length = np.zeros(n_gene, np.int64)
    np.add.at(length, ug, ue - us + 1)
    total = np.zeros(n_gene, np.int64)
    if len(ug):
        contig = contig_of_chrom[first_seq[ug] // 4]
        strand_u = first_seq[ug] % 4
        ok = (contig >= 0) & (strand_u <= 1)                      # anything else reads as zeros (detect_orfs.py:188-199)
        clen = np.where(ok, engine.contig_len[np.maximum(contig, 0)], 0)
        a = np.maximum(us, 1 - engine.pad)
        b = np.minimum(ue, clen + engine.pad)                     # outside the padded contig: no slot, reads 0
        ok &= a <= b
        off = strand_u * engine.plane + engine.contig_base[np.maximum(contig, 0)] + engine.pad + a
        d_off = t.from_numpy(np.ascontiguousarray(off[ok], np.int64)).to(engine.device)
        d_len = t.from_numpy(np.ascontiguousarray((b - a + 1)[ok], np.int32)).to(engine.device)
        d_grp = t.from_numpy(np.ascontiguousarray(ug[ok], np.int32)).to(engine.device)
        d_sum = t.zeros(n_gene, dtype=t.int64, device=engine.device)
        engine._check(engine.lib.rt_interval_sums(engine.ctx, C.c_void_p(cov.data_ptr()), int(ok.sum()),
                                                  C.c_void_p(d_off.data_ptr()), C.c_void_p(d_len.data_ptr()),
                                                  C.c_void_p(d_grp.data_ptr()), C.c_void_p(d_sum.data_ptr()),
                                                  engine._stream()))
        total = d_sum.cpu().numpy()
    for gi in np.flatnonzero(mixed):       # ORFs of one gene on several sequences: first value per `pos` wins
        seen = {}
        for o in rows[group == gi]:
            contig = int(contig_of_chrom[idx.orf_chrom_id[o]])
            s_code = int(idx.orf_strand_code[o])
            coor, vals = [], []
            for a0, b0 in zip(idx.exon_start[idx.exon_ptr[o]:idx.exon_ptr[o + 1]].tolist(),
                              idx.exon_end[idx.exon_ptr[o]:idx.exon_ptr[o + 1]].tolist()):
                coor.append(np.arange(a0, b0 + 1))
                v = np.zeros(b0 - a0 + 1, np.int64)
                if contig >= 0 and s_code <= 1:
                    lo, hi = max(a0, 1 - engine.pad), min(b0, int(engine.contig_len[contig]) + engine.pad)
                    if lo <= hi:
                        at = s_code * engine.plane + int(engine.contig_base[contig]) + engine.pad
                        v[lo - a0:hi - a0 + 1] = cov[at + lo:at + hi + 1].cpu().numpy()
                vals.append(v)
            coor, vals = np.concatenate(coor), np.concatenate(vals)
            if s_code == 1:
                coor, vals = coor[::-1], vals[::-1]
            for pos, c in zip(coor.tolist(), vals.tolist()):
                seen.setdefault(pos, c)
        total[gi], length[gi] = sum(seen.values()), len(seen)
    return keys, total, length


def write_counts(outfile, keys, total, length):
    """count_orfs.py:84-89: rows sorted by (gene_id, gene_name), only the id is printed."""
    with open(outfile, "w") as fout:
        fout.write("gene_id\tcount\tlength\n")
        for k in sorted(range(len(keys)), key=lambda i: keys[i]):
            fout.write(f"{keys[k][0]}\t{int(total[k])}\t{int(length[k])}\n")


def count_orfs_device(engine, cov, idx, status, features, outfile, report_all=False, rows_written="all"):
    """``count_orfs`` without the text round trip.  ``status`` = the status column of the scoring step
    (1 = translating) for every index row; ``rows_written`` says which rows the TSV would have held:
    "all" (detect-orfs ran with --report_all) or "translating"."""
    status = np.asarray(status).astype(bool)
    otype = np.fromiter((idx.field(o, 1) in features for o in range(idx.n_orf)), bool, idx.n_orf)
    present = np.ones(idx.n_orf, bool) if rows_written == "all" else status
    rows = np.flatnonzero(otype & present & (status | bool(report_all)))      # count_orfs.py:73-75
    keys, total, length = gene_union_counts(engine, cov, idx, rows)
    write_counts(outfile, keys, total, length)


def count_orfs(ribotricer_index, detected_orfs, features, outfile, report_all=False):
    """Same signature and output as the reference's ``count_orfs`` (count_orfs.py:28-34), from the TSV text."""
    idx = load_native_index(ribotricer_index)
    row_of = {}
    for o in range(idx.n_orf):
        if idx.field(o, 1) in features:
            row_of[idx.oid(o)] = o                    # later duplicates replace earlier ones, like the dict at :59
    pos_parts, cov_parts, keys, lut = defaultdict(list), defaultdict(list), [], {}
    with open(detected_orfs) as fin:
        fin.readline()
        for line in fin:
            f = line.strip().split("\t")
            if f[1] not in features or (f[2] == "nontranslating" and not report_all):
                continue
            o = row_of[f[0]]
            a, b = idx.exon_ptr[o], idx.exon_ptr[o + 1]
            coor = np.concatenate([np.arange(s, e + 1, dtype=np.int64) for s, e in zip(idx.exon_start[a:b], idx.exon_end[a:b])])
            if f[15] == "-":
                coor = coor[::-1]
            body = f[17].strip()[1:-1]
            prof = np.array(body.split(", "), np.int64) if body else np.zeros(0, np.int64)
            m = min(len(coor), len(prof))
            if m == 0:
                continue
            key = (f[11], f[12])
            if key not in lut:
                lut[key] = len(keys)
                keys.append(key)
            pos_parts[lut[key]].append(coor[:m])
            cov_parts[lut[key]].append(prof[:m])
    total, length = np.zeros(len(keys), np.int64), np.zeros(len(keys), np.int64)
    for g in range(len(keys)):
        pos, cov = np.concatenate(pos_parts[g]), np.concatenate(cov_parts[g])
        _, first = np.unique(pos, return_index=True)              # first coverage seen at a position wins (:80-82)
        total[g], length[g] = cov[first].sum(), len(first)
    write_counts(outfile, keys, total, length)


def count_orfs_gpu(ribotricer_index, detected_orfs, features, outfile, report_all=False, stage_ms: dict | None = None):
    """``count_orfs`` on the GPU (DESIGN.md section 13): the same table, byte for byte, on every input ``count_orfs``
    accepts.  Every check runs before ``outfile`` is opened, so a refused input leaves no file; the refusals (a plain
    gzip input, a line without 18 fields, an unknown ORF_ID, a malformed profile) raise ValueError naming the file and
    the line.  ``stage_ms``, when given, receives the time of every stage in milliseconds.  Returns a summary dict."""
    from .detect_orfs import get_engine

    clock = StageClock(stage_ms)
    idx, inp, _ = _open_selection(clock, "count-orfs", ribotricer_index, detected_orfs, features, report_all)
    dev_ms = np.zeros(_lib.RT_COUNT_STAGES, np.float32)
    total, length, summary = get_engine().orf_counts(inp.sel, inp.text(0), idx.exon_ptr, idx.exon_start, idx.exon_end,
                                                     idx.orf_strand_code, inp.n_gene, stage_ms=dev_ms)
    clock.lap("orf_counts")
    clock.device(("host_gather", "upload", "count_emit_kernel", "sort", "count_keep_kernel", "copy_back"), dev_ms)
    _raise_refused(detected_orfs, inp, summary[2:4])
    genes = np.flatnonzero(length)
    keys = [tuple(part.decode("utf-8") for part in inp.gene(int(g))) for g in genes]
    write_counts(outfile, keys, total[genes], length[genes])
    clock.lap("write")
    return dict(rows=inp.n_sel, genes=len(keys), positions=int(summary[1]), duplicates=int(summary[0] - summary[1]))


class CodonInput:
    """The selected rows of a detected-ORFs TSV matched to the index (``rt_codon_load_tsv``) and, after
    ``load_seq``, the checked orfs-seq nucleotide file (``rt_codon_load_seq``).  Rule violations raise ValueError."""

    def __init__(self, idx, detected_orfs, features, report_all: bool = False):
        self._lib = lib = _lib.load()
        self.idx = idx
        feats = [f.encode() for f in features]
        arr = (C.c_char_p * max(1, len(feats)))(*feats)
        handle = C.c_void_p()
        if isinstance(detected_orfs, NativeText):
            path = detected_orfs.path.encode()
            rc = lib.rt_codon_load_tsv_text(idx.handle, detected_orfs.take(), path, len(feats), arr, int(bool(report_all)),
                                            C.byref(handle))
        else:
            rc = lib.rt_codon_load_tsv(idx.handle, str(detected_orfs).encode(), len(feats), arr, int(bool(report_all)),
                                       C.byref(handle))
        if rc != 0:
            raise ValueError(lib.rt_io_last_error().decode())
        self.handle = handle
        sizes = np.zeros(4, np.int64)
        lib.rt_codon_sizes(handle, sizes.ctypes.data_as(C.c_void_p))
        self.n_sel, self.n_gene, self.n_gseq, self.n_lines = (int(v) for v in sizes)
        n = self.n_sel
        self.sel = dict(row=np.empty(n, np.int64), gene=np.empty(n, np.int32), gseq=np.empty(n, np.int32),
                        line=np.empty(n, np.int64), prof_off=np.empty(n, np.int64), prof_len=np.empty(n, np.int64),
                        seq_off=np.zeros(idx.n_orf, np.int64))
        self._copy()

    def _copy(self):
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        s = self.sel
        self._lib.rt_codon_copy(self.handle, p(s["row"]), p(s["gene"]), p(s["gseq"]), p(s["line"]), p(s["prof_off"]),
                                p(s["prof_len"]), p(s["seq_off"]))

    def load_seq(self, src) -> None:
        """The orfs-seq nucleotide file: a path or a ``bgzf.NativeText``."""
        if isinstance(src, NativeText):
            rc = self._lib.rt_codon_load_seq_text(self.handle, self.idx.handle, src.take(), src.path.encode())
        else:
            rc = self._lib.rt_codon_load_seq(self.handle, self.idx.handle, str(src).encode())
        if rc != 0:
            raise ValueError(self._lib.rt_io_last_error().decode())
        self._copy()

    def text(self, which: int) -> np.ndarray:
        """The TSV (0) or sequence file (1) text as a uint8 view of the native buffer."""
        n = C.c_int64()
        ptr = self._lib.rt_codon_text(self.handle, int(which), C.byref(n))
        if not n.value:
            return np.zeros(1, np.uint8)[:0]
        return np.ctypeslib.as_array((C.c_uint8 * n.value).from_address(ptr))

    def gene(self, g: int) -> tuple:
        """(gene_id, gene_name) of gene g as bytes."""
        il, nl = C.c_int(), C.c_int()
        ptr = self._lib.rt_codon_gene(self.handle, int(g), C.byref(il), C.byref(nl))
        raw = C.string_at(ptr, il.value + 1 + nl.value)
        return raw[:il.value], raw[il.value + 1:]

    def write(self, gene_tab, pooled_tab, gene_path: str, pooled_path: str) -> None:
        p = lambda a: np.ascontiguousarray(a, np.uint64).ctypes.data_as(C.c_void_p)  # noqa: E731
        gene_tab, pooled_tab = np.ascontiguousarray(gene_tab, np.uint64), np.ascontiguousarray(pooled_tab, np.uint64)
        if self._lib.rt_codon_write(self.handle, p(gene_tab), p(pooled_tab), str(gene_path).encode(),
                                    str(pooled_path).encode()) != 0:
            raise ValueError(self._lib.rt_io_last_error().decode())

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.rt_codon_free(self.handle)
                self.handle = None
        except Exception:
            pass


_PROFILE_REFUSALS = ((1, "the profile is not a list of integers written as str(list) writes it"),
                     (2, "a profile value lies outside 0..2147483647"),
                     (4, "a codon count exceeds 4294967295"))


def _open_selection(clock, command, ribotricer_index, detected_orfs, features, report_all, *more):
    """The input stage of count-orfs and count-orfs-codon: every input opened (``bgzf.open_texts``), the index loaded
    and the selected TSV rows matched to it.  Returns (index, ``CodonInput``, the opened ``more`` inputs)."""
    index_src, tsv_src, *more_src = open_texts([ribotricer_index, detected_orfs, *more], command)
    clock.lap("inflate")
    idx = load_native_index(index_src)
    clock.lap("index_load")
    inp = CodonInput(idx, tsv_src, features, report_all)
    clock.lap("tsv_load")
    return idx, inp, more_src


def _raise_refused(detected_orfs, inp, refusal):
    """A ValueError naming the TSV line of the first refused profile, when ``refusal`` (the first refused selected row,
    -1 for none, and its reasons: the two summary fields of the emit kernel) names one."""
    bad, bits = int(refusal[0]), int(refusal[1])
    if bad >= 0:
        reason = next(text for bit, text in _PROFILE_REFUSALS if bits & bit)
        raise ValueError(f"{detected_orfs} line {int(inp.sel['line'][bad])}: {reason}")


def count_orfs_codon(ribotricer_index, detected_orfs, features, ribotricer_index_fasta, prefix, report_all=False,
                     stage_ms: dict | None = None):
    """Write ``{prefix}_codon_counts_by_gene.tsv`` and ``{prefix}_codon_counts.tsv`` (DESIGN.md section 11) from the
    index, a detected-ORFs TSV and the orfs-seq nucleotide file of the same index.  ``features`` is a set of ORF types.
    Every check runs before either file is opened.  ``stage_ms``, when given, receives the time of every stage in
    milliseconds.  Returns a summary dict."""
    from .detect_orfs import get_engine

    clock = StageClock(stage_ms)
    idx, inp, (seq_src,) = _open_selection(clock, "count-orfs-codon", ribotricer_index, detected_orfs, features,
                                           report_all, ribotricer_index_fasta)
    inp.load_seq(seq_src)
    clock.lap("seq_check")
    dev_ms = np.zeros(_lib.RT_CODON_STAGES, np.float32)
    gene_tab, pooled_tab, summary = get_engine().codon_counts(
        inp.sel, inp.text(0), inp.text(1), idx.exon_ptr, idx.exon_start, idx.exon_end, idx.orf_strand_code,
        inp.n_gene, inp.n_gseq, stage_ms=dev_ms)
    clock.lap("codon_counts")
    clock.device(("host_gather", "upload", "codon_emit_kernel", "dedup", "count_sorts", "codon_stats_kernel",
                  "copy_back"), dev_ms)
    _raise_refused(detected_orfs, inp, summary[4:6])
    gene_path, pooled_path = f"{prefix}_codon_counts_by_gene.tsv", f"{prefix}_codon_counts.tsv"
    pathlib.Path(os.path.dirname(os.path.abspath(gene_path))).mkdir(parents=True, exist_ok=True)
    inp.write(gene_tab, pooled_tab, gene_path, pooled_path)
    clock.lap("write")
    genes = int(np.count_nonzero(gene_tab[:, 0].reshape(-1, 64).any(axis=1))) if inp.n_gene else 0
    result = dict(rows=inp.n_sel, genes=genes, codons=int(summary[3]), duplicates=int(summary[2]),
                  codons_with_n=int(summary[1]), gene_table=gene_path, codon_table=pooled_path)
    print(f"count-orfs-codon: {inp.n_sel} rows selected, {genes} genes, {result['codons']} codons kept, "
          f"{result['duplicates']} duplicates skipped, {result['codons_with_n']} codons with N")
    return result
