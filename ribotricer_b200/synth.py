"""Synthetic inputs for the BASELINE.json configurations (SURVEY.md 8(d)).

No real data can be fetched in this environment, so every parity test and
benchmark runs on seeded synthetic libraries: a genome (contig table), a
candidate-ORF index in ``prepare-orfs`` layout (prepare_orfs.py:370-404) and
Ribo-seq read columns as a coordinate-sorted BAM would decode to.

The index is built with numpy (it is at most a few 10^7 exons); reads are built
with torch ops so that 10^8-read libraries can be generated on the GPU in
milliseconds (plumbing only -- nothing here is on the measured path).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

R64_CONTIGS = [
    ("chrI", 230218), ("chrII", 813184), ("chrIII", 316620), ("chrIV", 1531933), ("chrV", 576874),
    ("chrVI", 270161), ("chrVII", 1090940), ("chrVIII", 562643), ("chrIX", 439888), ("chrX", 745751),
    ("chrXI", 666816), ("chrXII", 1078177), ("chrXIII", 924431), ("chrXIV", 784333), ("chrXV", 1091291),
    ("chrXVI", 948066), ("chrMito", 85779),
]
GRCH38_CONTIGS = [
    ("chr1", 248956422), ("chr2", 242193529), ("chr3", 198295559), ("chr4", 190214555),
    ("chr5", 181538259), ("chr6", 170805979), ("chr7", 159345973), ("chr8", 145138636),
    ("chr9", 138394717), ("chr10", 133797422), ("chr11", 135086622), ("chr12", 133275309),
    ("chr13", 114364328), ("chr14", 107043718), ("chr15", 101991189), ("chr16", 90338345),
    ("chr17", 83257441), ("chr18", 80373285), ("chr19", 58617616), ("chr20", 64444167),
    ("chr21", 46709983), ("chr22", 50818468), ("chrX", 156040895), ("chrY", 57227415), ("chrM", 16569),
]

READ_LENGTHS = np.array([26, 27, 28, 29, 30, 31, 32])
READ_LENGTH_P = np.array([0.03, 0.07, 0.20, 0.30, 0.20, 0.12, 0.08])
TRUE_OFFSETS = {26: 12, 27: 12, 28: 12, 29: 12, 30: 13, 31: 13, 32: 13}


@dataclass
class SynthConfig:
    name: str
    contigs: list
    n_orf: int
    n_reads: int
    seed: int
    single_exon_frac: float = 0.0      # C1: 0.95
    mean_exons: float = 4.0
    n_giant: int = 0                   # C5: ORFs of `giant_codons`
    giant_codons: int = 100_000
    n_micro: int = 0                   # C5: ORFs of exactly 20 codons
    expr_shape: float = 0.5            # gamma shape of per-ORF expression (smaller = more skew)
    annotated_rows: int = 0
    genome_order: bool = True          # rows in transcript order along the genome inside the annotated block and after it,
                                       # as prepare-orfs writes them from a sorted GTF (prepare_orfs.py:322-365)


def config(name: str, scale: float = 1.0, contig_scale: float = 1.0) -> SynthConfig:
    """The five BASELINE.json configurations; ``scale`` shrinks ORF and read counts and
    ``contig_scale`` the contig lengths (CPU tests cannot hold a 24.8 GB human coverage array)."""
    cfg = _config(name, scale)
    if contig_scale != 1.0:
        cfg.contigs = [(n, max(400_000, int(length * contig_scale))) for n, length in cfg.contigs]
    return cfg


def _config(name: str, scale: float) -> SynthConfig:
    s = lambda n: max(1, int(round(n * scale)))  # noqa: E731
    if name == "C1":
        return SynthConfig("C1", R64_CONTIGS, s(100_000), s(10_000_000), 1001, single_exon_frac=0.95,
                           annotated_rows=s(6000))
    if name == "C2":
        return SynthConfig("C2", GRCH38_CONTIGS, s(2_500_000), s(100_000_000), 1002, annotated_rows=s(60_000))
    if name == "C3":
        return SynthConfig("C3", GRCH38_CONTIGS, s(10_000_000), s(500_000_000), 1003, annotated_rows=s(60_000))
    if name == "C4":   # one of the 64 libraries; the index is C2's
        return SynthConfig("C4", GRCH38_CONTIGS, s(2_500_000), s(100_000_000), 1004, annotated_rows=s(60_000))
    if name == "C5":
        return SynthConfig("C5", GRCH38_CONTIGS, s(7_500_000), s(100_000_000), 1005, n_giant=max(1, s(100)),
                           n_micro=s(5_000_000), expr_shape=0.2, annotated_rows=s(60_000))
    if name == "tiny":
        return SynthConfig("tiny", [("c1", 300_000), ("c2", 150_000), ("c3", 40_000)], s(3000), s(200_000), 7,
                           mean_exons=3.0, annotated_rows=s(200))
    raise ValueError(f"unknown config {name}")


@dataclass
class SynthIndex:
    contig_names: list
    contig_len: np.ndarray
    exon_ptr: np.ndarray
    exon_start: np.ndarray
    exon_end: np.ndarray
    orf_contig: np.ndarray
    orf_strand: np.ndarray
    orf_len: np.ndarray
    orf_tx: np.ndarray
    annotated_rows: int
    meta: dict = field(default_factory=dict)

    @property
    def n_orf(self) -> int:
        return len(self.orf_contig)

    def as_dict(self) -> dict:
        return dict(exon_ptr=self.exon_ptr, exon_start=self.exon_start, exon_end=self.exon_end,
                    orf_contig=self.orf_contig, orf_strand=self.orf_strand)

    def write_tsv(self, path: str, lo: int = 0, hi: int | None = None):
        """11-column index as prepare-orfs writes it (prepare_orfs.py:370-404)."""
        hi = self.n_orf if hi is None else hi
        cats = ["uORF", "dORF", "novel", "super_uORF", "overlap_uORF", "overlap_dORF"]
        codons = ["ATG", "CTG", "GTG", "TTG"]
        with open(path, "w") as fh:
            fh.write("ORF_ID\tORF_type\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\t"
                     "chrom\tstrand\tstart_codon\tcoordinate\n")
            for o in range(lo, hi):
                a, b = self.exon_ptr[o], self.exon_ptr[o + 1]
                coord = ",".join(f"{s}-{e}" for s, e in zip(self.exon_start[a:b], self.exon_end[a:b]))
                t = int(self.orf_tx[o])
                cat = "annotated" if o < self.annotated_rows else cats[o % len(cats)]
                chrom = self.contig_names[self.orf_contig[o]]
                strand = "+" if self.orf_strand[o] == 0 else "-"
                fh.write(f"ORF{o}\t{cat}\tTX{t:07d}\tprotein_coding\tG{t:07d}\tgene{t}\tprotein_coding\t"
                         f"{chrom}\t{strand}\t{codons[o % 4]}\t{coord}\n")


def make_index(cfg: SynthConfig) -> SynthIndex:
    rng = np.random.default_rng(cfg.seed)
    names = [c[0] for c in cfg.contigs]
    clen = np.array([c[1] for c in cfg.contigs], dtype=np.int64)
    n_orf = cfg.n_orf
    n_special = cfg.n_giant + cfg.n_micro
    n_regular = max(0, n_orf - n_special)
    # transcripts carry ~3 nested ORFs sharing the stop (prepare_orfs.py:216-227 without --longest)
    n_tx = max(1, n_regular // 3) if n_regular else 0
    codons = np.maximum(20, np.rint(rng.lognormal(np.log(110.0), 1.0, n_tx))).astype(np.int64)
    codons = np.minimum(codons, 100_000)
    tx_codons = np.concatenate([codons, np.full(cfg.n_giant, cfg.giant_codons, np.int64),
                                np.full(cfg.n_micro, 20, np.int64)])
    n_tx_all = len(tx_codons)
    tx_len = tx_codons * 3
    # exon structure per transcript
    if cfg.single_exon_frac > 0:
        n_ex = np.where(rng.random(n_tx_all) < cfg.single_exon_frac, 1, 1 + rng.geometric(0.5, n_tx_all))
    else:
        n_ex = rng.geometric(1.0 / cfg.mean_exons, n_tx_all)
    n_ex = np.minimum(np.minimum(n_ex, 64), np.maximum(1, tx_len // 30)).astype(np.int64)
    n_ex[n_tx + cfg.n_giant:] = np.minimum(n_ex[n_tx + cfg.n_giant:], 2)   # micro ORFs: 1-2 exons
    tx_eptr = np.zeros(n_tx_all + 1, np.int64)
    np.cumsum(n_ex, out=tx_eptr[1:])
    n_exon_tx = int(tx_eptr[-1])
    ex_tx = np.repeat(np.arange(n_tx_all), n_ex)
    ex_rank = np.arange(n_exon_tx) - tx_eptr[ex_tx]
    # split tx_len into n_ex parts >= 1: n_ex - 1 sorted cut points, made strictly increasing by rank
    u = rng.random(n_exon_tx)
    cut = np.floor(u * (tx_len[ex_tx] - n_ex[ex_tx] + 1)).astype(np.int64)   # in [0, L - n_ex]
    order = np.argsort(ex_tx.astype(np.float64) * 4e6 + cut, kind="stable")
    ex_end_in_tx = cut[order] + ex_rank + 1
    last = tx_eptr[1:] - 1
    ex_end_in_tx[last] = tx_len            # the last exon ends at L
    ex_begin_in_tx = np.empty_like(ex_end_in_tx)
    ex_begin_in_tx[1:] = ex_end_in_tx[:-1]
    ex_begin_in_tx[tx_eptr[:-1]] = 0
    ex_len = ex_end_in_tx - ex_begin_in_tx
    assert (ex_len >= 1).all()
    introns = rng.integers(100, 5001, n_exon_tx)
    introns[tx_eptr[:-1]] = 0
    span_step = ex_len + introns
    ex_off_in_span = np.cumsum(span_step) - ex_len      # start offset incl. introns (global cumsum)
    tx_span_base = ex_off_in_span[tx_eptr[:-1]]
    ex_off_in_span = ex_off_in_span - tx_span_base[ex_tx]
    tx_span = ex_off_in_span[last] + ex_len[last]
    # place transcripts: contig by length, start uniform where it fits
    p = clen / clen.sum()
    tx_contig = rng.choice(len(clen), n_tx_all, p=p)
    too_long = tx_span >= clen[tx_contig] - 2
    if too_long.any():
        tx_contig[too_long] = int(np.argmax(clen))
    room = np.maximum(1, clen[tx_contig] - tx_span - 1)
    tx_start = 1 + np.floor(rng.random(n_tx_all) * room).astype(np.int64)
    tx_strand = (rng.random(n_tx_all) < 0.5).astype(np.uint8)
    # Transcripts that overlap an annotated transcript are isoforms of that gene: they take its strand.  (Randomly
    # placed transcripts overlap far more often than real genes do; with independent strands the reads of a highly
    # expressed overlapping transcript make the first-20,000-reads heuristic of infer_protocol.py:75-105 a coin
    # flip, which no real stranded library does.)
    n_annot_tx = min(cfg.annotated_rows, n_tx_all)
    if n_annot_tx:
        tx_end = tx_start + tx_span - 1
        for c in np.unique(tx_contig[:n_annot_tx]):
            ann = np.flatnonzero(tx_contig[:n_annot_tx] == c)
            ann = ann[np.argsort(tx_start[ann], kind="stable")]
            a_start, a_end, a_strand = tx_start[ann], tx_end[ann], tx_strand[ann]
            other = n_annot_tx + np.flatnonzero(tx_contig[n_annot_tx:] == c)
            j = np.searchsorted(a_start, tx_end[other], side="right") - 1      # last annotated span starting at or before my end
            for back in range(3):
                jj = j - back
                hit = (jj >= 0) & (a_end[np.maximum(jj, 0)] >= tx_start[other])
                tx_strand[other[hit]] = a_strand[jj[hit]]
                other, j = other[~hit], j[~hit]
    ex_start_g = tx_start[ex_tx] + ex_off_in_span
    ex_end_g = ex_start_g + ex_len - 1
    # ORFs: regular transcripts get nested ORFs (trim multiples of 3 from the 5' end)
    nested = np.full(n_tx_all, 1, np.int64)
    if n_tx:
        base = n_regular // n_tx
        nested[:n_tx] = base
        nested[: n_regular - base * n_tx] += 1
    orf_tx = np.repeat(np.arange(n_tx_all), nested)
    o_rank = np.arange(len(orf_tx)) - np.repeat(np.cumsum(nested) - nested, nested)
    max_trim_codons = np.maximum(0, tx_codons[orf_tx] - 20)
    trim = np.where(o_rank == 0, 0, np.floor(rng.random(len(orf_tx)) * (max_trim_codons + 1)).astype(np.int64)) * 3
    # annotated rows first: the untrimmed ORF of the first `annotated_rows` transcripts
    n_total = len(orf_tx)
    first_rows = np.flatnonzero((o_rank == 0))[: cfg.annotated_rows]
    mask = np.ones(n_total, bool)
    mask[first_rows] = False
    rest = np.flatnonzero(mask)
    if cfg.genome_order:
        key = lambda rows: np.lexsort((rows, tx_start[orf_tx[rows]], tx_contig[orf_tx[rows]]))  # noqa: E731
        first_rows, rest = first_rows[key(first_rows)], rest[key(rest)]
    perm = np.concatenate([first_rows, rest])
    orf_tx, trim = orf_tx[perm], trim[perm]
    # kept genomic-concat range of the transcript: '+' [trim, L), '-' [0, L - trim)
    L_tx = tx_len[orf_tx]
    strand = tx_strand[orf_tx]
    keep_lo = np.where(strand == 0, trim, 0)
    keep_hi = np.where(strand == 0, L_tx, L_tx - trim)
    a_t = tx_eptr[orf_tx]
    # exon containing keep_lo (first kept) and keep_hi - 1 (last kept), via global cumulative ends
    g_end = np.cumsum(ex_len)
    g_begin = g_end - ex_len
    tx_g0 = g_begin[tx_eptr[:-1]]
    e_first = np.searchsorted(g_end, tx_g0[orf_tx] + keep_lo, side="right")
    e_last = np.searchsorted(g_end, tx_g0[orf_tx] + keep_hi - 1, side="right")
    cnt = e_last - e_first + 1
    exon_ptr = np.zeros(n_total + 1, np.int64)
    np.cumsum(cnt, out=exon_ptr[1:])
    src = np.repeat(e_first, cnt) + (np.arange(int(exon_ptr[-1])) - np.repeat(exon_ptr[:-1], cnt))
    exon_start = ex_start_g[src].copy()
    exon_end = ex_end_g[src].copy()
    first_pos = exon_ptr[:-1]
    last_pos = exon_ptr[1:] - 1
    exon_start[first_pos] += (tx_g0[orf_tx] + keep_lo) - g_begin[e_first]
    exon_end[last_pos] -= g_end[e_last] - (tx_g0[orf_tx] + keep_hi)
    del a_t
    return SynthIndex(names, clen, exon_ptr, exon_start.astype(np.int32), exon_end.astype(np.int32),
                      tx_contig[orf_tx].astype(np.int32), strand.astype(np.uint8),
                      (keep_hi - keep_lo).astype(np.int64), orf_tx.astype(np.int64),
                      min(cfg.annotated_rows, n_total), meta=dict(config=cfg.name, seed=cfg.seed))


def make_reads(cfg: SynthConfig, idx: SynthIndex, device="cpu", n_reads: int | None = None,
               sort: bool = True, dirty_frac: float = 0.02, seed_offset: int = 0) -> dict:
    """Read columns (torch tensors on ``device``), forward-stranded protocol.

    70 % of the reads sit in "expressed" ORFs (gamma expression x length) with
    their P-site on a codon position with frame probabilities (0.70, 0.15,
    0.15); 30 % are uniform background on both strands.  The 5' end is the
    P-site -/+ the true offset of the read's length.  ``dirty_frac`` of the
    reads each carry qcfail / duplicate / secondary / multi-mapper marks so the
    filter cascade of bam.py:77-91 is exercised.
    """
    import torch

    n = cfg.n_reads if n_reads is None else int(n_reads)
    dev = torch.device(device)
    g = torch.Generator(device=dev)
    g.manual_seed(cfg.seed * 7919 + 13 + seed_offset)
    rng = np.random.default_rng(cfg.seed + 99)
    T = lambda a, dt=None: torch.as_tensor(np.ascontiguousarray(a), device=dev, dtype=dt)  # noqa: E731
    rand = lambda m: torch.rand(m, generator=g, device=dev, dtype=torch.float64)  # noqa: E731

    n_expr = int(n * 0.7)
    n_bg = n - n_expr
    expr = rng.gamma(cfg.expr_shape, 1.0, idx.n_orf) * (rng.random(idx.n_orf) < 0.6)
    w = expr * idx.orf_len
    if w.sum() <= 0:
        w = idx.orf_len.astype(np.float64)
    cw = T(np.cumsum(w) / w.sum())
    orf = torch.searchsorted(cw, rand(n_expr)).clamp_(max=idx.n_orf - 1)
    orf_len = T(idx.orf_len)[orf]
    codon = (rand(n_expr) * (orf_len // 3).to(torch.float64)).floor().to(torch.int64)
    fr = rand(n_expr)
    frame = (fr > 0.70).to(torch.int64) + (fr > 0.85).to(torch.int64)
    p = torch.minimum(codon * 3 + frame, orf_len - 1)
    strand_o = T(idx.orf_strand, torch.int64)[orf]
    q = torch.where(strand_o == 0, p, orf_len - 1 - p)           # position in genomic-ascending concat
    exlen = idx.exon_end.astype(np.int64) - idx.exon_start + 1
    gend = T(np.cumsum(exlen))
    gbeg = gend - T(exlen)
    target = gbeg[T(idx.exon_ptr[:-1])[orf]] + q
    e = torch.searchsorted(gend, target, right=True)
    psite = T(idx.exon_start, torch.int64)[e] + (target - gbeg[e])
    contig_e = T(idx.orf_contig, torch.int64)[orf]
    # background
    clen = T(idx.contig_len)
    ccw = torch.cumsum(clen.to(torch.float64), 0) / float(idx.contig_len.sum())
    contig_b = torch.searchsorted(ccw, rand(n_bg)).clamp_(max=len(idx.contig_len) - 1)
    psite_b = 1 + (rand(n_bg) * clen[contig_b].to(torch.float64)).floor().to(torch.int64)
    strand_b = (rand(n_bg) < 0.5).to(torch.int64)
    contig = torch.cat([contig_e, contig_b])
    psite = torch.cat([psite, psite_b])
    strand = torch.cat([strand_o, strand_b])
    del contig_e, contig_b, psite_b, strand_b, orf, codon, fr, frame, p, q, target, e
    # read length and 5' end
    lcw = T(np.cumsum(READ_LENGTH_P))
    li = torch.searchsorted(lcw, rand(n)).clamp_(max=len(READ_LENGTHS) - 1)
    length = T(READ_LENGTHS)[li]
    off = T(np.array([TRUE_OFFSETS[int(x)] for x in READ_LENGTHS]))[li]
    pos5 = torch.where(strand == 0, psite - off, psite + off)            # 1-based 5' end
    first = torch.where(strand == 0, pos5 - 1, pos5 - length)           # 0-based matched range
    cl = clen[contig]
    first = torch.minimum(torch.clamp(first, min=0), cl - length)
    first = torch.clamp(first, min=0)
    last = first + length - 1
    flag = torch.where(strand == 0, 0, 16)
    # dirt
    r = rand(n)
    d = dirty_frac
    flag = flag | torch.where(r < d, 0x200, 0) | torch.where((r >= d) & (r < 2 * d), 0x400, 0) \
        | torch.where((r >= 2 * d) & (r < 3 * d), 0x100, 0)
    multi = (r >= 3 * d) & (r < 4 * d)
    star = (r >= 4 * d) & (r < 4 * d + 0.10)          # no NH tag, MAPQ 255 (STAR)
    lowq = (r >= 4 * d + 0.10) & (r < 4 * d + 0.11)   # no NH tag, MAPQ 3 -> "None" -> dropped
    nh = torch.ones(n, dtype=torch.int64, device=dev)
    nh = torch.where(multi, 3, nh)
    nh = torch.where(star | lowq, 0, nh)
    mapq = torch.full((n,), 255, dtype=torch.int64, device=dev)
    mapq = torch.where(multi, 1, mapq)
    mapq = torch.where(lowq, 3, mapq)
    if sort:   # coordinate-sorted like a real BAM (reference_id, reference_start)
        key = contig * (1 << 32) + first
        order = torch.argsort(key, stable=True)
        contig, first, last, length, flag, mapq, nh = (x[order] for x in (contig, first, last, length, flag, mapq, nh))
    return dict(ref_id=contig.to(torch.int32), first=first.to(torch.int32), last=last.to(torch.int32),
                mlen=length.to(torch.int16), flag=flag.to(torch.int16), mapq=mapq.to(torch.uint8),
                nh=nh.to(torch.uint8))


def reads_to_numpy(cols: dict) -> dict:
    out = {}
    for k, v in cols.items():
        a = v.cpu().numpy()
        if k in ("mlen", "flag"):
            a = a.view(np.uint16)
        out[k] = a
    return out


# --------------------------------------------------------------------------------------------------------------
# Annotation + genome for prepare-orfs: a seeded FASTA and GTF with planted coding sequences.
# --------------------------------------------------------------------------------------------------------------
_STOPS = (b"TAA", b"TAG", b"TGA")
_COMPLEMENT = np.frombuffer(bytes.maketrans(b"ACGTNacgtn", b"TGCANtgcan"), np.uint8)


def _sense_codons(rng, k: int) -> bytes:
    """k random codons, none of them a stop."""
    out = rng.choice(np.frombuffer(b"ACGT", np.uint8), 3 * k + 96).tobytes()
    codons = [out[i:i + 3] for i in range(0, len(out) - 2, 3)]
    codons = [c for c in codons if c not in _STOPS]
    while len(codons) < k:
        codons.append(b"GCT")
    return b"".join(codons[:k])


def make_annotation(out_dir: str, n_genes: int = 40, tx_per_gene: float = 2.0, genome_size: int = 400_000,
                    seed: int = 11, contigs: list | None = None, edge_cases: bool = True) -> dict:
    """Write ``genome.fa`` and ``annotation.gtf`` under ``out_dir``.

    Every gene sits in its own slot of a contig (``contigs`` or ``genome_size`` split over three contigs), on a random
    strand, with 1-12 exons.  Its first transcript carries a planted CDS (ATG, sense codons, a stop that the CDS lines
    exclude); the other isoforms skip inner exons and carry the same CDS when they keep every exon it touches, or none.
    ``edge_cases`` (the small test configurations) adds: non-ATG CDS, lowercase and N bases, CRLF line ends,
    overlapping and book-ended exon lines, shuffled attribute order, Ensembl ``*_biotype`` keys, missing
    ``gene_name``, start / stop codons split across an exon junction, a uORF with a nested in-frame start, and
    transcripts that must be skipped (contig absent from the FASTA, past a contig end, exons on both strands).
    Returns the two paths, the contig table and the planted CDS per transcript id."""
    import os

    rng = np.random.default_rng(seed)
    if contigs is None:
        contigs = [(f"chr{k + 1}", int(genome_size * w)) for k, w in enumerate((0.5, 0.3, 0.2))]
    acgt = np.frombuffer(b"ACGT", np.uint8)
    seqs = {name: acgt[rng.integers(0, 4, length, dtype=np.uint8)] for name, length in contigs}
    clen = np.array([length for _, length in contigs], np.int64)
    gene_contig = rng.choice(len(contigs), n_genes, p=clen / clen.sum())
    lines, planted = [], {}
    crlf = edge_cases
    slot_of = {}
    for g in range(n_genes):
        ci = int(gene_contig[g])
        slot_of.setdefault(ci, []).append(g)
    for ci, genes in slot_of.items():
        name, length = contigs[ci]
        seq = seqs[name]
        slot = length // len(genes)
        for k, g in enumerate(genes):
            lo = k * slot + 1
            span = slot - 2
            if span < 400:
                continue
            strand = "+" if rng.random() < 0.5 else "-"
            n_ex = int(rng.integers(1, 13))
            ex_len = rng.integers(60, 700, n_ex)
            intron = rng.integers(60, 3000, n_ex)
            total = int(ex_len.sum() + intron[:-1].sum())
            while total > span and n_ex > 1:
                n_ex -= 1
                ex_len, intron = ex_len[:n_ex], intron[:n_ex]
                total = int(ex_len.sum() + intron[:-1].sum())
            if total > span:
                ex_len = np.array([span // 2])
                total = int(ex_len[0])
            start = lo + int(rng.integers(0, span - total + 1))
            exons, at = [], start
            for e in range(n_ex):
                exons.append((at, at + int(ex_len[e]) - 1))
                at += int(ex_len[e]) + int(intron[e])
            # genomic position (0-based) of every transcript nt, in transcript (oriented) order
            pos = np.concatenate([np.arange(s - 1, e) for s, e in exons])
            if strand == "-":
                pos = pos[::-1]
            n = len(pos)
            # plant the CDS: [c0, c0 + 3k) is ATG + sense codons, the stop follows and is not part of the CDS
            k_cod = int(rng.integers(2, max(3, (n - 6) // 3)))
            c0 = int(rng.integers(0, n - 3 * k_cod - 3 + 1))
            if edge_cases and g % 7 == 3 and n_ex >= 3:     # start and stop codons split across exon junctions
                j0 = int(ex_len[0]) if strand == "+" else int(ex_len[-1])
                j1 = n - (int(ex_len[-1]) if strand == "+" else int(ex_len[0]))
                for a, b in ((j0 - 1, j1 - 1), (j0 - 1, j1 - 2), (j0 - 2, j1 - 1), (j0 - 2, j1 - 2)):
                    if (b - a) % 3 == 0 and b - a >= 6:
                        c0, k_cod = a, (b - a) // 3
                        break
            body = bytearray(_sense_codons(rng, k_cod))
            body[:3] = b"CTG" if edge_cases and g % 5 == 2 else b"ATG"
            body += _STOPS[int(rng.integers(0, 3))]
            codes = np.frombuffer(bytes(body), np.uint8)
            if strand == "-":
                codes = _COMPLEMENT[codes]
            seq[pos[c0:c0 + len(codes)]] = codes
            if edge_cases and g % 6 == 1 and c0 >= 100:     # uORF with a nested in-frame start sharing its stop
                u = bytearray(b"ATG" + _sense_codons(rng, 4) + b"ATG" + _sense_codons(rng, 18) + b"TAA")
                ucodes = np.frombuffer(bytes(u), np.uint8)
                seq[pos[2:2 + len(ucodes)]] = _COMPLEMENT[ucodes] if strand == "-" else ucodes
            cds_lo, cds_hi = sorted((int(pos[c0]) + 1, int(pos[c0 + 3 * k_cod - 1]) + 1))
            gid, gname = f"G{seed}_{g:06d}", f"GENE{g}"
            style = int(rng.integers(0, 3)) if edge_cases else 0
            n_tx = max(1, int(rng.poisson(tx_per_gene - 1)) + 1)
            for t in range(n_tx):
                tid = f"T{seed}_{g:06d}_{t}"
                keep = [True] * n_ex
                if t > 0 and n_ex > 2:
                    keep = [e in (0, n_ex - 1) or rng.random() < 0.6 for e in range(n_ex)]
                tex = [ex for ex, kp in zip(exons, keep) if kp]
                coding = all(kp for (s0, e0), kp in zip(exons, keep) if e0 >= cds_lo and s0 <= cds_hi)
                ttype = "protein_coding" if coding else "processed_transcript"
                attrs = [("gene_id", gid), ("transcript_id", tid), ("gene_name", gname),
                         ("gene_type", "protein_coding"), ("transcript_type", ttype)]
                if style == 1:                                          # Ensembl keys, shuffled order
                    attrs = [(kk.replace("_type", "_biotype"), v) for kk, v in attrs]
                    attrs = [attrs[i] for i in rng.permutation(len(attrs))]
                elif style == 2:                                        # no gene_name
                    attrs = [a for a in attrs if a[0] != "gene_name"] + [("tag", "basic"), ("tag", "CCDS")]
                attr = " ".join(f'{kk} "{v}";' for kk, v in attrs)
                rows = [(s, e, "exon") for s, e in tex]
                if edge_cases and t == 0 and g % 4 == 0 and tex[0][1] - tex[0][0] > 20:
                    s, e = tex[0]                                       # one exon as overlapping + book-ended pieces
                    m = (s + e) // 2
                    rows[0:1] = [(s, m, "exon"), (m - 5, m + 3, "exon"), (m + 1, e, "exon")]
                if coding:
                    cds_iv = [(max(s, cds_lo), min(e, cds_hi)) for s, e in tex if s <= cds_hi and e >= cds_lo]
                    rows += [(s, e, "CDS") for s, e in cds_iv]
                    planted[tid] = dict(gene_id=gid, chrom=name, strand=strand, cds=cds_iv)
                for s, e, feat in rows:
                    lines.append(f"{name}\tsynth\t{feat}\t{s}\t{e}\t.\t{strand}\t{'.' if feat == 'exon' else '0'}\t{attr}")
    if edge_cases:
        name0, len0 = contigs[0]
        base = f'gene_type "protein_coding"; transcript_type "protein_coding";'
        lines += [f"chrAbsent\tsynth\texon\t100\t400\t.\t+\t.\tgene_id \"GX1\"; transcript_id \"TX_absent\"; {base}",
                  f"{name0}\tsynth\texon\t{len0 - 50}\t{len0 + 20}\t.\t+\t.\tgene_id \"GX2\"; transcript_id \"TX_pastend\"; {base}",
                  f"{name0}\tsynth\texon\t100\t200\t.\t+\t.\tgene_id \"GX3\"; transcript_id \"TX_twostrands\"; {base}",
                  f"{name0}\tsynth\texon\t300\t400\t.\t-\t.\tgene_id \"GX3\"; transcript_id \"TX_twostrands\"; {base}",
                  f"{name0}\tsynth\tgene\t100\t400\t.\t+\t.\tgene_id \"GX3\";",
                  f"{name0}\tsynth\texon\t500\t600\t.\t+\t.\ttranscript_id \"TX_nogene\";"]
        for name, _ in contigs:                                         # soft-masked stretches and N runs
            seq = seqs[name]
            for _ in range(max(1, len(seq) // 20_000)):
                a = int(rng.integers(0, len(seq) - 200))
                seq[a:a + int(rng.integers(20, 200))] += 32
                b = int(rng.integers(0, len(seq) - 50))
                seq[b:b + int(rng.integers(1, 50))] = ord("N") + (32 if rng.random() < 0.3 else 0)
    os.makedirs(out_dir, exist_ok=True)
    eol = "\r\n" if crlf else "\n"
    gtf = os.path.join(out_dir, "annotation.gtf")
    with open(gtf, "w", newline="") as fh:
        fh.write("#!genome-build synthetic" + eol + "##seed " + str(seed) + "\n")
        for i, line in enumerate(lines):
            fh.write(line + (eol if i % 2 else "\n"))
        fh.write("\n")
    fasta = os.path.join(out_dir, "genome.fa")
    with open(fasta, "wb") as fh:
        for name, length in contigs:
            fh.write(f">{name} synthetic contig{eol}".encode())
            seq = seqs[name]
            width = 60 if not crlf else 61
            full = (length // width) * width
            if full:
                block = np.empty((full // width, width + len(eol)), np.uint8)
                block[:, :width] = seq[:full].reshape(-1, width)
                block[:, width:] = np.frombuffer(eol.encode(), np.uint8)
                fh.write(block.tobytes())
            if full < length:
                fh.write(seq[full:].tobytes() + eol.encode())
    return dict(fasta=fasta, gtf=gtf, contigs=list(contigs), planted=planted)
