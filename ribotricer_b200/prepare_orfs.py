"""``prepare-orfs``: the candidate-ORF index ``{prefix}_candidate_orfs.tsv`` from a GTF and a genome FASTA.

    GTF, FASTA          rt_gtf_load / rt_fasta_load (csrc/rt_prepare.cpp, all cores)
    transcripts         exon / CDS lines grouped by (gene_id, transcript_id) and merged here, in numpy
    candidate ORFs      Engine.orf_search: orf_splice_kernel, orf_walk_kernel (count, fill), orf_interval_kernel
    annotated rows      the first codon of every CDS, read from the host copy of the contig codes
    index file          rt_orf_write (all cores, write-behind)

The rules are those of DESIGN.md section 9.  Same name and argument order as the reference's ``prepare_orfs``
(prepare_orfs.py:278).  Inputs are plain text or BGZF (inflated on the GPU, ``bgzf.open_texts``); other gzip files are
refused.
"""
from __future__ import annotations

import ctypes as C
import os
import pathlib

import numpy as np

from . import _lib
from .bgzf import NativeText, StageClock, open_text, open_texts

TYPES = ("annotated", "uORF", "overlap_uORF", "super_uORF", "overlap_dORF", "dORF", "novel", "internal")
BASES = "ACGT"
_SHIFT = np.int64(1) << np.int64(32)


def codon_code(codon: str) -> int:
    """6-bit code of a codon of ACGT (16 b0 + 4 b1 + b2)."""
    if len(codon) != 3 or any(b not in BASES for b in codon):
        raise ValueError(f"codon {codon!r} is not three letters of ACGT")
    return 16 * BASES.index(codon[0]) + 4 * BASES.index(codon[1]) + BASES.index(codon[2])


def codon_mask(codons) -> int:
    mask = 0
    for codon in codons:
        mask |= 1 << codon_code(codon)
    return mask


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _io_error(what: str):
    return ValueError(f"{what}: {_lib.load().rt_io_last_error().decode()}")


class Genome:
    """A FASTA indexed by ``rt_fasta_load``; ``codes`` translates contigs to 1-byte codes on demand.  ``src`` is a path
    (plain text or BGZF) or a ``NativeText``."""

    def __init__(self, src):
        self.handle = None
        src = open_text(src, "prepare-orfs") if isinstance(src, str) else src
        self._lib = lib = _lib.load()
        h = C.c_void_p()
        if isinstance(src, NativeText):
            path = src.path
            rc = lib.rt_fasta_load_text(src.take(), path.encode(), C.byref(h))
        else:
            path = src
            rc = lib.rt_fasta_load(path.encode(), C.byref(h))
        if rc != 0:
            raise _io_error(f"cannot load FASTA {path}")
        self.handle = h
        n = lib.rt_fasta_n_contig(h)
        self.names = [lib.rt_fasta_contig_name(h, i).decode() for i in range(n)]
        self.lengths = np.array([lib.rt_fasta_contig_len(h, i) for i in range(n)], np.int64)

    def codes(self, contigs) -> np.ndarray:
        """The listed contigs back to back (A C G T -> 0-3, anything else -> 4)."""
        contigs = np.ascontiguousarray(contigs, np.int32)
        out = np.empty(int(self.lengths[contigs].sum()), np.uint8)
        if self._lib.rt_fasta_codes(self.handle, len(contigs), _np_ptr(contigs), _np_ptr(out)) != 0:
            raise _io_error("FASTA codes")
        return out

    def close(self):
        if getattr(self, "handle", None):
            self._lib.rt_fasta_free(self.handle)
            self.handle = None

    __del__ = close


def load_gtf(src) -> dict:
    """The exon and CDS lines of a GTF (``rt_gtf_load``) as columns; ``attr`` holds 5 string ids per line (gene_id,
    transcript_id, gene_name, gene_type, transcript_type with their fallbacks; -1 absent) into ``strings``.  ``src`` is
    a path (plain text or BGZF) or a ``NativeText``."""
    src = open_text(src, "prepare-orfs") if isinstance(src, str) else src
    lib = _lib.load()
    h = C.c_void_p()
    if isinstance(src, NativeText):
        path = src.path
        rc = lib.rt_gtf_load_text(src.take(), path.encode(), C.byref(h))
    else:
        path = src
        rc = lib.rt_gtf_load(path.encode(), C.byref(h))
    if rc != 0:
        raise _io_error(f"cannot load GTF {path}")
    try:
        n = int(lib.rt_gtf_n_lines(h))
        cols = dict(line=np.empty(n, np.int64), feature=np.empty(n, np.uint8), chrom=np.empty(n, np.int32),
                    start=np.empty(n, np.int32), end=np.empty(n, np.int32), strand=np.empty(n, np.uint8),
                    attr=np.empty((n, 5), np.int32))
        blob = C.create_string_buffer(max(1, int(lib.rt_gtf_string_bytes(h))))
        lib.rt_gtf_copy(h, *[_np_ptr(cols[k]) for k in ("line", "feature", "chrom", "start", "end", "strand", "attr")],
                        blob)
        n_str = int(lib.rt_gtf_n_strings(h))
        cols["strings"] = blob.raw.decode().split("\0")[:n_str]
    finally:
        lib.rt_gtf_free(h)
    return cols


def _group(g: dict, sel: np.ndarray, key: np.ndarray) -> dict:
    """Lines ``sel`` (file order) grouped by ``key``, groups in order of first appearance, intervals sorted by start
    and merged (overlapping or book-ended)."""
    k = key[sel]
    uk, first, inv = np.unique(k, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    gid = rank[inv]
    n_groups = len(uk)
    members = sel[np.lexsort((g["start"][sel], gid))]
    gm = np.sort(gid, kind="stable")
    out = dict(key=uk[order], first=sel[first[order]], n=n_groups)
    if n_groups == 0:
        z = np.zeros(0, np.int64)
        out.update(consistent=np.zeros(0, bool), ptr=np.zeros(1, np.int64), start=z, end=z)
        return out
    cnt = np.bincount(gm, minlength=n_groups)
    gptr = np.concatenate([[0], np.cumsum(cnt)])[:-1]
    ch, st = g["chrom"][members], g["strand"][members]
    out["consistent"] = (np.minimum.reduceat(ch, gptr) == np.maximum.reduceat(ch, gptr)) & \
        (np.minimum.reduceat(st, gptr) == np.maximum.reduceat(st, gptr))
    off = gm.astype(np.int64) * _SHIFT
    s = g["start"][members].astype(np.int64) + off
    cm = np.maximum.accumulate(g["end"][members].astype(np.int64) + off)
    new = np.ones(len(s), bool)
    new[1:] = s[1:] > cm[:-1] + 1
    at = np.flatnonzero(new)
    last = np.append(at[1:] - 1, len(s) - 1)
    out["start"] = s[at] - off[at]
    out["end"] = cm[last] - off[at]
    out["ptr"] = np.concatenate([[0], np.cumsum(np.bincount(gm[at], minlength=n_groups))])
    return out


def _rank(grp: dict, owner: np.ndarray, x: np.ndarray) -> np.ndarray:
    """Position of nt ``x`` in the ascending concatenation of group ``owner``'s intervals, -1 where x is not in one."""
    gof = np.repeat(np.arange(grp["n"]), np.diff(grp["ptr"])).astype(np.int64)
    length = grp["end"] - grp["start"] + 1
    cum = np.concatenate([[0], np.cumsum(length)])
    before = cum[:-1] - cum[grp["ptr"][gof]]
    i = np.searchsorted(gof * _SHIFT + grp["start"], owner.astype(np.int64) * _SHIFT + x, side="right") - 1
    hit = (i >= grp["ptr"][owner]) & (i < grp["ptr"][owner + 1])
    i = np.where(hit, i, 0)
    hit &= x <= grp["end"][i]
    return np.where(hit, before[i] + x - grp["start"][i], -1)


def _gene_order(gene: np.ndarray, line: np.ndarray) -> np.ndarray:
    """Order: genes by their first line (the smallest of their transcripts'), transcripts of a gene by their first line."""
    by_line = np.argsort(line, kind="stable")
    _, first, inv = np.unique(gene[by_line], return_index=True, return_inverse=True)
    return by_line[np.argsort(first[inv], kind="stable")]


def build_transcripts(g: dict, genome: Genome) -> dict:
    """Rule 1 of DESIGN.md section 9: kept transcripts in candidate order, with their merged exons and CDS."""
    attr = g["attr"]
    strings = g["strings"]
    key = attr[:, 0].astype(np.int64) * max(1, len(strings)) + attr[:, 1]
    named = (attr[:, 0] >= 0) & (attr[:, 1] >= 0)
    E = _group(g, np.flatnonzero(named & (g["feature"] == 0)), key)
    D = _group(g, np.flatnonzero(named & (g["feature"] == 1)), key)
    n = E["n"]
    # contig of every transcript (-1: absent from the FASTA)
    lut = {name: i for i, name in enumerate(genome.names)}
    chrom_id = g["chrom"][E["first"]]
    ids = np.unique(chrom_id)
    fa_of = dict(zip(ids.tolist(), (lut.get(strings[c], -1) for c in ids.tolist())))
    contig = np.array([fa_of[c] for c in chrom_id.tolist()], np.int64) if n else np.zeros(0, np.int64)
    strand = g["strand"][E["first"]]
    last_end = E["end"][E["ptr"][1:] - 1] if n else np.zeros(0, np.int64)
    bad = ~E["consistent"] | (strand > 1) | (contig < 0)
    bad |= last_end > np.where(contig >= 0, genome.lengths[np.maximum(contig, 0)] if len(genome.lengths) else 0, 0)
    # the CDS of every transcript: its group, consistent with the exons, first and last nt exonic
    cds = np.full(n, -1, np.int64)
    if D["n"] and n:
        ek = np.argsort(E["key"])
        j = np.minimum(np.searchsorted(E["key"][ek], D["key"]), n - 1)
        hit = E["key"][ek[j]] == D["key"]
        cds[ek[j[hit]]] = np.flatnonzero(hit)
    has = cds >= 0
    t_cds = np.flatnonzero(has)
    c = cds[t_cds]
    same = D["consistent"][c] & (g["chrom"][D["first"][c]] == chrom_id[t_cds]) & \
        (g["strand"][D["first"][c]] == strand[t_cds])
    lo, hi = D["start"][D["ptr"][c]], D["end"][D["ptr"][c + 1] - 1]
    r_lo, r_hi = _rank(E, t_cds, lo), _rank(E, t_cds, hi)
    bad[t_cds] |= ~same | (r_lo < 0) | (r_hi < 0)
    tx_len = np.diff(np.concatenate([[0], np.cumsum(E["end"] - E["start"] + 1)])[E["ptr"]]) if n else np.zeros(0, np.int64)
    cds_bounds = np.full((n, 2), -1, np.int32)
    minus = strand[t_cds] == 1
    cds_bounds[t_cds, 0] = np.where(minus, tx_len[t_cds] - 1 - r_hi, r_lo)
    cds_bounds[t_cds, 1] = np.where(minus, tx_len[t_cds] - 1 - r_lo, r_hi)
    kept = np.flatnonzero(~bad)
    first_line = g["line"][E["first"]]
    gene = attr[E["first"], 0]
    kept = kept[_gene_order(gene[kept], first_line[kept])]
    # candidate-order table
    ex_cnt = np.diff(E["ptr"])[kept]
    ex_ptr = np.concatenate([[0], np.cumsum(ex_cnt)]).astype(np.int64)
    src = np.repeat(E["ptr"][kept], ex_cnt) + (np.arange(int(ex_ptr[-1])) - np.repeat(ex_ptr[:-1], ex_cnt))
    kc = cds[kept]
    return dict(n=len(kept), n_skipped=int(n - len(kept)), exon_ptr=ex_ptr, exon_start=E["start"][src].astype(np.int32),
                exon_end=E["end"][src].astype(np.int32), contig=contig[kept], strand=strand[kept],
                cds_bounds=cds_bounds[kept], attr=attr[E["first"][kept]], chrom=chrom_id[kept],
                cds_group=kc, cds_first_line=np.where(kc >= 0, g["line"][D["first"][np.maximum(kc, 0)]] if D["n"] else 0, -1),
                cds=D)


def _annotated(tx: dict, codes: np.ndarray, tx_base: np.ndarray, start_mask: int) -> dict:
    """Rule 5: one row per transcript with a CDS whose first oriented codon is a start codon, in CDS order."""
    D = tx["cds"]
    t = np.flatnonzero(tx["cds_group"] >= 0)
    t = t[_gene_order(tx["attr"][t, 0], tx["cds_first_line"][t])]
    c = tx["cds_group"][t]
    length = (D["end"] - D["start"] + 1)
    cum = np.concatenate([[0], np.cumsum(length)])
    total = cum[D["ptr"][c + 1]] - cum[D["ptr"][c]] if len(c) else np.zeros(0, np.int64)
    minus = tx["strand"][t] == 1
    codon = np.zeros(len(t), np.int64)
    valid = total >= 3
    gof = np.repeat(np.arange(D["n"]), np.diff(D["ptr"])).astype(np.int64)
    before = cum[:-1] - cum[D["ptr"][gof]]
    for k in range(3):                                  # oriented nt k of the CDS -> genomic nt -> code
        r = np.clip(np.where(minus, total - 1 - k, k), 0, np.maximum(total - 1, 0))
        i = np.searchsorted(gof * _SHIFT + before, c * _SHIFT + r, side="right") - 1
        pos = D["start"][i] + r - before[i]
        b = codes[tx_base[t] + pos - 1].astype(np.int64)
        b = np.where(minus & (b < 4), 3 - b, b)
        valid &= b < 4
        codon = codon * 4 + np.minimum(b, 3)
    keep = valid & (((np.uint64(start_mask) >> codon.astype(np.uint64)) & np.uint64(1)) == 1)
    t, c, codon = t[keep], c[keep], codon[keep]
    n_iv = np.diff(D["ptr"])[c]
    iv_ptr = np.concatenate([[0], np.cumsum(n_iv)]).astype(np.int64)
    src = np.repeat(D["ptr"][c], n_iv) + (np.arange(int(iv_ptr[-1])) - np.repeat(iv_ptr[:-1], n_iv))
    return dict(row_tx=t.astype(np.int32), row_type=np.zeros(len(t), np.uint8), row_codon=codon.astype(np.uint8),
                iv_ptr=iv_ptr, iv_start=D["start"][src].astype(np.int32), iv_end=D["end"][src].astype(np.int32))


def _tx_text(tx: dict, strings: list):
    """Per transcript: "transcript_id\\ttranscript_type\\tgene_id\\tgene_name\\tgene_type\\tchrom\\tstrand" as one blob."""
    get = lambda i: "NA" if i < 0 else strings[i]  # noqa: E731
    texts, id_len = [], []
    for (gid, tid, gname, gtype, ttype), chrom, strand in zip(tx["attr"].tolist(), tx["chrom"].tolist(),
                                                              tx["strand"].tolist()):
        tid_b = strings[tid].encode()
        texts.append(b"\t".join((tid_b, get(ttype).encode(), strings[gid].encode(), get(gname).encode(),
                                 get(gtype).encode(), strings[chrom].encode(), b"+" if strand == 0 else b"-")))
        id_len.append(len(tid_b))
    off = np.concatenate([[0], np.cumsum([len(t) for t in texts])]).astype(np.int64)
    return b"".join(texts), off, np.asarray(id_len, np.int32)


def prepare_orfs(gtf, fasta, prefix, min_orf_length=60, start_codons={"ATG"}, stop_codons={"TAG", "TAA", "TGA"},
                 longest=False, stage_ms: dict | None = None):
    """Write ``{prefix}_candidate_orfs.tsv`` (DESIGN.md section 9).  ``stage_ms``, when given, receives the time of
    every stage in milliseconds."""
    from .detect_orfs import get_engine

    if min_orf_length < 0:
        raise ValueError("min_orf_length must be >= 0")
    if not start_codons or not stop_codons:
        raise ValueError("the start and stop codon lists must not be empty")
    start_mask, stop_mask = codon_mask(start_codons), codon_mask(stop_codons)
    pathlib.Path(os.path.dirname(prefix) or ".").mkdir(parents=True, exist_ok=True)
    clock = StageClock(stage_ms)
    fasta_src, gtf_src = open_texts([fasta, gtf], "prepare-orfs")
    clock.lap("inflate")
    genome = Genome(fasta_src)
    clock.lap("fasta_load")
    g = load_gtf(gtf_src)
    clock.lap("gtf_load")
    tx = build_transcripts(g, genome)
    used = np.unique(tx["contig"]).astype(np.int32)
    codes = genome.codes(used)
    base = np.zeros(len(genome.names), np.int64)
    base[used] = np.concatenate([[0], np.cumsum(genome.lengths[used])[:-1]]) if len(used) else 0
    tx_base = base[tx["contig"]] if tx["n"] else np.zeros(0, np.int64)
    clock.lap("transcripts")
    ann = _annotated(tx, codes, tx_base, start_mask)
    clock.lap("annotated")
    dev_ms = np.zeros(_lib.RT_ORF_STAGES, np.float32)
    cand = get_engine().orf_search(codes, tx_base, tx["exon_ptr"], tx["exon_start"], tx["exon_end"], tx["strand"],
                                   tx["cds_bounds"], start_mask, stop_mask, int(min_orf_length), bool(longest),
                                   stage_ms=dev_ms)
    clock.lap("orf_search")
    clock.device(("upload", "orf_splice_kernel", "orf_walk_kernel<count>", "row_scan", "orf_walk_kernel<fill>",
                  "orf_interval_kernel<count>+scan", "orf_interval_kernel<fill>"), dev_ms)
    text, text_off, id_len = _tx_text(tx, g["strings"])
    n_ann = len(ann["row_tx"])
    rows = {k: np.concatenate([ann[k], cand[k]]) for k in ("row_tx", "row_type", "row_codon", "iv_start", "iv_end")}
    rows["iv_ptr"] = np.concatenate([ann["iv_ptr"], cand["iv_ptr"][1:] + ann["iv_ptr"][-1]])
    n_rows = len(rows["row_tx"])
    rc = _lib.load().rt_orf_write(
        f"{prefix}_candidate_orfs.tsv".encode(), tx["n"], text, _np_ptr(text_off), _np_ptr(id_len), n_rows,
        *[_np_ptr(np.ascontiguousarray(rows[k])) for k in ("row_tx", "row_type", "row_codon", "iv_ptr", "iv_start",
                                                            "iv_end")])
    if rc != 0:
        raise _io_error("cannot write the index")
    clock.lap("write")
    genome.close()
    print(f"prepare-orfs: {tx['n']} transcripts ({tx['n_skipped']} skipped), {n_ann} annotated and "
          f"{n_rows - n_ann} candidate ORFs written to {prefix}_candidate_orfs.tsv")
    return dict(n_tx=tx["n"], n_skipped=tx["n_skipped"], n_annotated=n_ann, n_candidates=n_rows - n_ann)
