"""Binning, scoring and detect-orfs on a genome of ~1,900 small contigs, against the C oracle.

Assemblies with unplaced scaffolds (Drosophila dm6 has 1,870 references) take paths that a genome of a few chromosomes
never reaches:
- the stream kernel keeps only the first 256 entries of the contig table in shared memory and reads later ones from
  global memory;
- the packer opens a block at every reference change, and refuses a stream that would be mostly padding, so a sparse
  library falls back to the column kernel;
- fresh (zoned) binning must also clear the compact slots of contigs that have ORFs but no reads, at every join;
- contigs shorter than a word or than the pad sit next to each other in the planes, where an off-by-one in a P-site
  bounds test moves a count into the neighbour;
- the WIG writer orders chromosomes by name, and ``scaffold_1010`` sorts before ``scaffold_3``.

The genome has contigs of 500-20,000 nt, one of 3 Mb, and a set of edge lengths (1, 2, 31-33, pad - 1 .. pad + 1,
2 pad, 255-257, 511-513 for pads 16 and 64) twice: at ids 247-264, across 255/256, and again among the last ids.
Some contigs carry ORFs but no reads (before the first read, in the middle, after the last one), some reads but no ORFs.
"""
from __future__ import annotations

import ctypes as C
import functools

import numpy as np
import pytest

from helpers import DEFAULT_PARAMS, compare_scores, compare_tsv, decode_stream

N_CONTIG = 1900
PADS = (16, 64)
EDGE_LENS = (1, 2, 15, 16, 17, 31, 32, 33, 63, 64, 65, 128, 255, 256, 257, 511, 512, 513)
FIRST_EDGE = 247                                   # ids 247 .. 264: the edge lengths straddle 255 / 256
N_TAIL_NOREAD = 7                                  # the last ids: ORFs, no reads
LAST_EDGE = N_CONTIG - N_TAIL_NOREAD - len(EDGE_LENS)
BIG = 3                                            # the 3 Mb contig
EDGE_IDS = tuple(range(FIRST_EDGE, FIRST_EDGE + len(EDGE_LENS))) + tuple(range(LAST_EDGE, LAST_EDGE + len(EDGE_LENS)))
NOREAD_IDS = (0, 1, 2) + tuple(range(900, 906)) + tuple(range(N_CONTIG - N_TAIL_NOREAD, N_CONTIG))
NOORF_IDS = tuple(range(1000, 1010))
# negative offsets, offsets beyond either pad, and the two long lengths of the extension records
OFFSETS = {26: -1, 27: -2, 28: 12, 29: -5, 30: 0, 31: 300, 150: 40, 300: -7}
DENSE_READS, SPARSE_READS = 300_000, 40_000
ABSENT_CHROMS = ("chrAbsent", "scaffold_99999")
RT_ESTATE = -4                                     # include/ribotricer_b200.h: the call cannot be done in this state
RT_STREAM_RANGE = 1 << 20                          # include/ribotricer_b200.h: reads per range the packer codes alone
RT_STREAM_BLOCK = 256


def _oracle():
    from oracle import c_oracle
    return c_oracle


# ---------------------------------------------------------------------------------------------------- the genome
@functools.lru_cache(maxsize=None)
def genome():
    rng = np.random.default_rng(1870)
    lens = rng.integers(500, 20_001, N_CONTIG).astype(np.int64)
    lens[BIG] = 3_000_000
    lens[FIRST_EDGE:FIRST_EDGE + len(EDGE_LENS)] = EDGE_LENS
    lens[LAST_EDGE:LAST_EDGE + len(EDGE_LENS)] = EDGE_LENS
    return [f"scaffold_{i}" for i in range(N_CONTIG)], lens


def _hand_orfs():
    """(contig, strand, [(start, end)]) ORFs on every edge-length and reads-free contig: whole-contig single exons on
    both strands, exons that hang into both pads (and past pad 16), and a two-exon ORF on the contig's ends."""
    _, lens = genome()
    out = []
    for c in sorted(set(EDGE_IDS) | set(NOREAD_IDS)):
        L = int(lens[c])
        for s in (0, 1):
            out.append((c, s, [(1, L)]))
            out.append((c, s, [(-20, L + 20)]))
            out.append((c, s, [(-3, min(L, 2))]))
            out.append((c, s, [(max(1, L - 1), L + 5)]))
            if L >= 4:
                out.append((c, s, [(1, 1), (L - 1, L)]))
    return out


def _csr(orfs):
    ptr, st, en, contig, strand = [0], [], [], [], []
    for c, s, ivs in orfs:
        for a, b in ivs:
            st.append(a)
            en.append(b)
        ptr.append(len(st))
        contig.append(c)
        strand.append(s)
    return dict(exon_ptr=np.array(ptr, np.int64), exon_start=np.array(st, np.int32), exon_end=np.array(en, np.int32),
                orf_contig=np.array(contig, np.int32), orf_strand=np.array(strand, np.uint8))


def _cat(a, b):
    n_ex = len(a["exon_start"])
    return dict(exon_ptr=np.concatenate([a["exon_ptr"], b["exon_ptr"][1:] + n_ex]),
                **{k: np.concatenate([a[k], b[k]]) for k in ("exon_start", "exon_end", "orf_contig", "orf_strand")})


@functools.lru_cache(maxsize=None)
def synth_index():
    """synth's index on the genome, without the rows on the contigs that must have no ORFs."""
    import dataclasses

    from ribotricer_b200 import synth

    names, lens = genome()
    cfg = synth.SynthConfig("many", list(zip(names, lens.tolist())), 20_000, DENSE_READS, 1870, annotated_rows=300)
    idx = synth.make_index(cfg)
    keep = ~np.isin(idx.orf_contig, NOORF_IDS)
    rows = np.flatnonzero(keep)
    n_ex = np.diff(idx.exon_ptr)[rows]
    ex = np.concatenate([np.arange(idx.exon_ptr[o], idx.exon_ptr[o + 1]) for o in rows])
    ptr = np.zeros(len(rows) + 1, np.int64)
    np.cumsum(n_ex, out=ptr[1:])
    return cfg, dataclasses.replace(idx, exon_ptr=ptr, exon_start=idx.exon_start[ex], exon_end=idx.exon_end[ex],
                                    orf_contig=idx.orf_contig[rows], orf_strand=idx.orf_strand[rows],
                                    orf_len=idx.orf_len[rows], orf_tx=idx.orf_tx[rows],
                                    annotated_rows=int(keep[:idx.annotated_rows].sum()))


@functools.lru_cache(maxsize=None)
def index():
    """The device index: synth's rows, then the hand-built ones."""
    _, idx = synth_index()
    return _cat(idx.as_dict(), _csr(_hand_orfs()))


# ---------------------------------------------------------------------------------------------------- the libraries
@functools.lru_cache(maxsize=None)
def library(kind):
    """A coordinate-sorted library over the genome.  ``dense`` streams, ``sparse`` (fewer reads on as many contigs) is
    refused by the packer.  Besides synth's reads: hand reads at the first and last positions of every edge-length
    contig (and of the contigs without ORFs) on both strands, long and spliced reads, every filter category, reads on
    reference ``N_CONTIG`` (no such contig) and an unmapped tail."""
    from ribotricer_b200 import synth

    cfg, idx = synth_index()
    _, lens = genome()
    n, seed = (DENSE_READS, 1) if kind == "dense" else (SPARSE_READS, 2)
    r = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=n, sort=True, seed_offset=seed))
    keep = ~np.isin(r["ref_id"], NOREAD_IDS)
    r = {k: v[keep] for k, v in r.items()}
    hand = {k: [] for k in r}
    for c in EDGE_IDS + NOORF_IDS:
        L = int(lens[c])
        for first in sorted({max(0, p) for p in (0, 1, 2, L - 3, L - 2, L - 1)}):
            for length in (26, 27, 28, 29, 30, 31):
                for flag in (0, 16):
                    hand["ref_id"].append(c)
                    hand["first"].append(first)
                    hand["last"].append(first + length - 1)
                    hand["mlen"].append(length)
                    hand["flag"].append(flag)
                    hand["mapq"].append(255)
                    hand["nh"].append(1)
    r = {k: np.concatenate([v, np.array(hand[k], v.dtype)]) for k, v in r.items()}
    order = np.lexsort((r["first"], r["ref_id"]))
    r = {k: v[order] for k, v in r.items()}
    rng = np.random.default_rng(seed)
    m = len(r["ref_id"])
    first = r["first"].astype(np.int64)
    mlen = np.where(rng.random(m) < 0.02, rng.choice([150, 255, 256, 300, 700], m), r["mlen"].astype(np.int64))
    extra = np.where(rng.random(m) < 0.05, rng.choice([1, 3, 85, 6_000, 70_000], m), 0)
    r["mlen"] = mlen.astype(np.uint16)
    r["last"] = (first + mlen - 1 + extra).astype(np.int32)
    flag = r["flag"].astype(np.int64)
    flag = np.where(rng.random(m) < 0.1, flag | rng.choice([4, 256, 512, 1024, 2048, 0x704], m), flag)
    r["flag"] = flag.astype(np.uint16)
    r["nh"] = rng.choice([0, 1, 1, 1, 2, 255], m).astype(np.uint8)
    r["mapq"] = rng.choice([255, 255, 3, 0], m).astype(np.uint8)
    junk = (flag & 0x704) != 0
    r["first"] = np.where(junk & (rng.random(m) < 0.5), -1, r["first"]).astype(np.int32)
    # reads on reference N_CONTIG (sorted after every real one), then the unmapped tail
    k_bad, k_tail = 300, 500
    pos = np.sort(rng.integers(0, 5_000, k_bad)).astype(np.int32)
    bad = dict(ref_id=np.full(k_bad, N_CONTIG, np.int32), first=pos, last=pos + 27, mlen=np.full(k_bad, 28, np.uint16),
               flag=rng.choice([0, 16], k_bad).astype(np.uint16), mapq=np.full(k_bad, 255, np.uint8),
               nh=np.ones(k_bad, np.uint8))
    tail = dict(ref_id=np.full(k_tail, -1, np.int32), first=np.full(k_tail, -1, np.int32), last=np.full(k_tail, 27, np.int32),
                mlen=np.full(k_tail, 29, np.uint16), flag=np.full(k_tail, 4, np.uint16), mapq=np.zeros(k_tail, np.uint8),
                nh=np.zeros(k_tail, np.uint8))
    return {k: np.ascontiguousarray(np.concatenate([r[k], bad[k], tail[k]])) for k in r}


def _contigs_with_reads(reads):
    """Contigs that carry a read whose flags leave its position to the packer."""
    ref = reads["ref_id"][(reads["flag"] & 0x704) == 0]
    return np.unique(ref[(ref >= 0) & (ref < N_CONTIG)])


def _pack(cols, n_threads=0):
    """rt_stream_pack on host columns: (rc, records, headers, n_blocks)."""
    from ribotricer_b200 import _lib

    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    cols = {k: np.ascontiguousarray(cols[k], dt) for k, dt in (("ref_id", np.int32), ("first", np.int32), ("last", np.int32),
                                                               ("mlen", np.uint16), ("flag", np.uint16), ("mapq", np.uint8),
                                                               ("nh", np.uint8))}
    args = [p(cols[k]) for k in ("ref_id", "first", "last", "mlen", "flag", "mapq", "nh")]
    n = len(cols["ref_id"])
    nb = C.c_int64(0)
    rc = lib.rt_stream_pack(n, *args, n_threads, 0, None, None, C.byref(nb))
    if rc != 0:
        return rc, None, None, 0
    rec = np.zeros(max(1, nb.value) * RT_STREAM_BLOCK, np.uint32)
    hdr = np.zeros(max(1, nb.value) * 4, np.int32)
    rc = lib.rt_stream_pack(n, *args, n_threads, nb.value, p(rec), p(hdr), C.byref(nb))
    return rc, rec, hdr, nb.value


# ---------------------------------------------------------------------------------------------------- files
def write_bam(path, reads):
    """The library as a BAM with every reference in its (coordinate-sorted) header."""
    import bam_writer as W

    names, lens = genome()
    recs = []
    for i in range(len(reads["ref_id"])):
        first, last, mlen = int(reads["first"][i]), int(reads["last"][i]), int(reads["mlen"][i])
        extra = last - first + 1 - mlen
        cigar = [("M", mlen)] if extra == 0 else [("M", 1), ("N", extra), ("M", mlen - 1)]
        nh = int(reads["nh"][i])
        aux = b"" if nh == 0 else W.aux_field("NH", "S", 300 if nh == 255 else nh)
        recs.append(W.record(int(reads["ref_id"][i]), first, int(reads["mapq"][i]), int(reads["flag"][i]), cigar,
                             name=b"r%d" % i, aux=aux))
    W.write_bam(str(path), list(zip(names, lens.tolist())), recs, sorted_header=True)


def write_index(path):
    """synth's rows (SynthIndex.write_tsv), the hand rows an index file can hold (start >= 1), and rows on chromosomes
    the BAM does not have."""
    names, _ = genome()
    _, idx = synth_index()
    idx.write_tsv(str(path))
    lines = []
    for k, (c, s, ivs) in enumerate(_hand_orfs()):
        if ivs[0][0] < 1:
            continue
        coord = ",".join(f"{a}-{b}" for a, b in ivs)
        lines.append(f"HAND{k}\tnovel\tHTX{k:05d}\tprotein_coding\tHG{k:05d}\thand{k}\tprotein_coding\t{names[c]}\t"
                     f"{'+-'[s]}\tATG\t{coord}\n")
    for j, chrom in enumerate(ABSENT_CHROMS):
        for s in "+-":
            lines.append(f"ABS{j}{s}\tnovel\tATX{j}\tprotein_coding\tAG{j}\tabs{j}\tprotein_coding\t{chrom}\t{s}\tATG\t"
                         f"100-400,500-{600 + j}\n")
    with open(path, "a") as fh:
        fh.writelines(lines)


# ======================================================================================================== CPU tests
def test_genome_and_libraries_hold_what_they_target(built):
    names, lens = genome()
    idx = index()
    assert len(names) == N_CONTIG and sorted(names)[:3] == ["scaffold_0", "scaffold_1", "scaffold_10"]
    has_orf = np.zeros(N_CONTIG, bool)
    has_orf[idx["orf_contig"]] = True
    assert has_orf[list(NOREAD_IDS)].all() and not has_orf[list(NOORF_IDS)].any()
    assert 1400 < has_orf.sum() < N_CONTIG - 200       # and hundreds without ORFs: long runs of empty map words
    assert min(EDGE_IDS[:len(EDGE_LENS)]) < 256 <= max(EDGE_IDS[:len(EDGE_LENS)])
    for kind in ("dense", "sparse"):
        reads = library(kind)
        with_reads = _contigs_with_reads(reads)
        assert not np.isin(with_reads, NOREAD_IDS).any() and np.isin(NOORF_IDS, with_reads).all()
        assert np.isin(EDGE_IDS, with_reads).all()
        # reads-free contigs before the first read, in the middle and after the last one
        assert with_reads.min() > 2 and with_reads.max() == LAST_EDGE + len(EDGE_LENS) - 1
        assert len(with_reads) > 1700
        assert (reads["mlen"] > 255).any() and (reads["last"] - reads["first"] + 1 > reads["mlen"]).any()
        for bit in (4, 256, 512, 1024):
            assert (reads["flag"] & bit).any()
        assert (reads["ref_id"] == N_CONTIG).sum() == 300 and (reads["ref_id"][-500:] == -1).all()


def _decode_blocks(rec, hdr, nb):
    """decode_stream block by block: (ref_id, first, last, mlen, meta) per read, and the index of every block's first
    read."""
    rows, starts = [], []
    for b in range(nb):
        starts.append(len(rows))
        rows += decode_stream(rec[b * RT_STREAM_BLOCK:(b + 1) * RT_STREAM_BLOCK], hdr[4 * b:4 * b + 4], 1)
    return np.array(rows, np.int64).reshape(-1, 5), np.array(starts, np.int64)


@pytest.mark.parametrize("kind", ["dense", "dense_x4", "sparse"])
def test_packer_on_many_contigs(built, kind):
    """rt_stream_pack on the libraries: the dense one codes, with a block per reference (every block's reads on its
    header's reference, references above 255 among them), and decodes back to its columns; one thread and many give the
    same bytes.  ``dense_x4`` (every read four times) is more than one range of RT_STREAM_RANGE reads: the ranges are
    coded on different threads, and the first read of every range after the first opens a block, in the middle of a
    contig.  The sparse one would be more than half padding and is refused."""
    reads = library(kind.split("_")[0])
    if kind == "dense_x4":
        reads = {k: np.repeat(v, 4) for k, v in reads.items()}
    n = len(reads["ref_id"])
    n_ranges = (n + RT_STREAM_RANGE - 1) // RT_STREAM_RANGE
    assert n_ranges == (2 if kind == "dense_x4" else 1)
    rc, rec, hdr, nb = _pack(reads)
    if kind == "sparse":
        assert rc == RT_ESTATE
        return
    assert rc == 0
    with_reads = _contigs_with_reads(reads)
    assert nb >= len(with_reads)
    refs = hdr.reshape(-1, 4)[:nb, 0]
    assert (refs >= 256).sum() > 1000
    assert refs[refs < N_CONTIG].max() == with_reads.max()
    got, starts = _decode_blocks(rec, hdr, nb)
    assert len(got) == n
    # the decoder takes every read's reference from its block's header: a read the flags do not decide must sit in a
    # block of its own reference, at its own position
    plain = (reads["flag"] & 0x704) == 0
    for j, k in enumerate(("ref_id", "first", "last", "mlen")):
        assert (got[plain, j] == reads[k][plain]).all(), k
    assert np.isin(np.arange(n_ranges) * RT_STREAM_RANGE, starts).all()
    if n_ranges > 1:
        b = int(np.searchsorted(starts, RT_STREAM_RANGE))
        assert refs[b] == refs[b - 1] and refs[b] == reads["ref_id"][RT_STREAM_RANGE]      # mid-contig
    rc1, rec1, hdr1, nb1 = _pack(reads, n_threads=1)
    rcm, recm, hdrm, nbm = _pack(reads, n_threads=16)
    assert rc1 == rcm == 0 and nb1 == nbm == nb
    assert (rec1 == rec).all() and (hdr1 == hdr).all() and (recm == rec).all() and (hdrm == hdr).all()


@pytest.mark.parametrize("k,ok", [(1032, True), (1033, False)])
def test_packer_refusal_threshold(built, k, ok):
    """One read on each of k contigs is k blocks for n = k reads.  The packer refuses a stream whose records (256 per
    block, padding included) number more than 2 n plus 1,024 blocks' worth per range of RT_STREAM_RANGE reads; with one
    range that is 256 k > 2 k + 262,144, so 1,032 contigs are coded and 1,033 are refused."""
    pos = np.arange(k, dtype=np.int32) * 7 % 5000
    cols = dict(ref_id=np.arange(k, dtype=np.int32), first=pos, last=pos + 27, mlen=np.full(k, 28, np.uint16),
                flag=np.where(np.arange(k) % 2, 16, 0).astype(np.uint16), mapq=np.full(k, 255, np.uint8),
                nh=np.ones(k, np.uint8))
    rc, rec, hdr, nb = _pack(cols)
    if not ok:
        assert rc == RT_ESTATE
        return
    assert rc == 0 and nb == k
    assert (hdr.reshape(-1, 4)[:, 0] == np.arange(k)).all()
    got = decode_stream(rec, hdr, nb)
    assert [g[:4] for g in got] == [(i, int(pos[i]), int(pos[i]) + 27, 28) for i in range(k)]


def test_bam_decoder_reads_a_header_of_many_references(built, tmp_path):
    """The native decoder on a BAM whose header holds all 1,900 references: names, lengths and the reference count, and
    every record -- on ids above 255 too, spliced, long, unmapped, on reference N_CONTIG -- decodes to its columns."""
    from ribotricer_b200.bam import read_bam_columns_native

    names, lens = genome()
    reads = library("sparse")
    path = tmp_path / "many.bam"
    write_bam(path, reads)
    got = read_bam_columns_native(str(path), 4)
    assert got.contig_names == names and (got.contig_len == lens).all() and got.sorted_by_coordinate
    for k in ("ref_id", "first", "last", "mlen", "flag", "mapq", "nh"):
        assert (got.cols[k] == reads[k]).all(), k
    assert (got.cols["ref_id"] >= 256).sum() > 0.5 * len(reads["ref_id"])


def test_wig_chromosomes_in_name_order_on_cpu_twin(built, tmp_path, monkeypatch):
    """detect_orfs() on the CPU twin: the variableStep blocks of both WIG files come in lexicographic order of the names
    (scaffold_1010 before scaffold_3), one per covered contig, and the reads-free contigs have none."""
    from oracle_engine import install
    from ribotricer_b200 import detect_orfs as D

    install(monkeypatch)
    reads = library("sparse")
    bam, idx_path = tmp_path / "lib.bam", tmp_path / "index.tsv"
    write_bam(bam, reads)
    write_index(idx_path)
    prefix = str(tmp_path / "twin")
    D.detect_orfs(str(bam), str(idx_path), prefix, "forward", None, dict(OFFSETS), *DEFAULT_PARAMS, False,
                  meta_min_reads=10 ** 9)
    names, _ = genome()
    for tag in ("pos", "neg"):
        chroms = [line.split("chrom=")[1].split()[0] for line in open(f"{prefix}_{tag}.wig") if line.startswith("variableStep")]
        assert chroms == sorted(chroms) and len(set(chroms)) == len(chroms) > 1000
        assert chroms.index("scaffold_1010") < chroms.index("scaffold_3")
        assert not {names[c] for c in NOREAD_IDS} & set(chroms)


# ======================================================================================================== GPU tests
def _setup(engine, pad):
    names, lens = genome()
    engine.set_genome(names, lens, pad=pad)
    engine.set_length_table(OFFSETS, None)
    engine.set_index(**index())
    CO = _oracle()
    base, plane = CO.genome_layout(lens, pad)
    assert plane == engine.plane and (base == engine.contig_base).all()
    return CO.make_len_table(OFFSETS, None), base, plane


def _compact_of(engine, dense_np):
    """compact_from_dense of oracle planes: what a compact-layout buffer must hold."""
    t = engine.torch
    engine.set_layout("compact")
    out = engine.new_coverage()
    engine.compact_from_dense(t.from_numpy(dense_np).to(engine.device), out)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("protocol", ["forward", "reverse"])
def test_column_kernel_matches_oracle(engine, pad, protocol):
    """bin_psites_kernel through both entry points, in the dense and compact layouts: stats, length counts and every
    dense slot equal the oracle's; the compact buffer holds compact_from_dense of the oracle's planes.  The host entry
    with sorted_hint (which streams a library that codes) must give the same."""
    CO = _oracle()
    t = engine.torch
    _, lens = genome()
    lt, base, plane = _setup(engine, pad)
    code = {"forward": 0, "reverse": 1}[protocol]
    try:
        for kind in ("dense", "sparse"):
            reads = library(kind)
            ref_cov, ref_stats, ref_len = CO.bin_reads(reads, code, lt, base, lens, pad, plane)
            assert ref_stats["badref"] > 0 and ref_stats["oob"] > 0
            engine.set_layout("dense")
            cov = engine.new_coverage()
            stats, lc = engine.bin_reads_host(cov, reads, protocol)
            assert stats == ref_stats and (lc == ref_len).all()
            assert (cov.cpu().numpy() == ref_cov).all(), kind
            st, lcd = engine.new_bin_accumulators()
            engine.bin_reads_device(cov, engine.upload_reads(reads), protocol, st, lcd)
            assert (cov.cpu().numpy() == 2 * ref_cov).all(), kind
            assert dict(zip(ref_stats, st.cpu().tolist())) == ref_stats and (lcd.cpu().numpy() == ref_len).all()
            want = _compact_of(engine, ref_cov)
            got = engine.new_coverage()
            stats_c, lc_c = engine.bin_reads_host(got, reads, protocol)
            assert stats_c == ref_stats and (lc_c == ref_len).all()
            assert t.equal(got, want), kind
            st, lcd = engine.new_bin_accumulators()
            engine.bin_reads_device(got, engine.upload_reads(reads), protocol, st, lcd, weight=-1)
            assert int(got.abs().max().item()) == 0
            stats_h, lc_h = engine.bin_reads_host(got, reads, protocol, sorted_hint=True)
            assert stats_h == ref_stats and (lc_h == ref_len).all() and t.equal(got, want), kind
    finally:
        engine.set_layout("dense")


@pytest.mark.gpu
@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("protocol", ["forward", "reverse"])
def test_stream_kernel_matches_oracle(engine, pad, protocol):
    """bin_stream_kernel on the dense library: headers on references above 255 (read from global memory) and on the last
    contig with reads; host and device entry points in both layouts equal the oracle and the column kernel; weight -1
    returns the buffer to zero; fresh (zoned) binning over garbage, in order and with the blocks shuffled, gives the same
    buffer -- the zones must clear the compact slots of the reads-free contigs at every join."""
    CO = _oracle()
    t = engine.torch
    _, lens = genome()
    lt, base, plane = _setup(engine, pad)
    code = {"forward": 0, "reverse": 1}[protocol]
    reads = library("dense")
    stream = engine.stream_reads(reads)
    refs = np.asarray(stream["hdr"]).reshape(-1, 4)[:stream["n_blocks"], 0]
    assert (refs >= 256).any() and refs[refs < N_CONTIG].max() == _contigs_with_reads(reads).max()
    ref_cov, ref_stats, ref_len = CO.bin_reads(reads, code, lt, base, lens, pad, plane)
    dstream = engine.upload_stream(stream)
    try:
        engine.set_layout("dense")
        got = engine.new_coverage()
        stats, lc = engine.bin_stream_host(got, stream, protocol)
        assert stats == ref_stats and (lc == ref_len).all()
        assert (got.cpu().numpy() == ref_cov).all()
        cols = engine.new_coverage()
        st0, lc0 = engine.new_bin_accumulators()
        engine.bin_reads_device(cols, engine.upload_reads(reads), protocol, st0, lc0)
        st, lcd = engine.new_bin_accumulators()
        engine.bin_stream_device(got, dstream, protocol, st, lcd)
        assert t.equal(got, 2 * cols) and t.equal(st, st0) and t.equal(lcd, lc0)
        engine.bin_stream_device(got, dstream, protocol, st, lcd, weight=-1)
        engine.bin_stream_device(got, dstream, protocol, st, lcd, weight=-1)
        assert int(got.abs().max().item()) == 0 and t.equal(st, -st0) and t.equal(lcd, -lc0)
        del got, cols
        want = _compact_of(engine, ref_cov)
        got = engine.new_coverage()
        stats, lc = engine.bin_stream_host(got, stream, protocol)
        assert stats == ref_stats and (lc == ref_len).all() and t.equal(got, want)
        st, lcd = engine.new_bin_accumulators()
        engine.bin_stream_device(got, dstream, protocol, st, lcd, weight=-1)
        assert int(got.abs().max().item()) == 0
        fresh = t.full_like(want, 12345)
        st, lcd = engine.new_bin_accumulators()
        engine.bin_stream_device(fresh, dstream, protocol, st, lcd, fresh=True)
        assert t.equal(fresh, want)
        assert dict(zip(ref_stats, st.cpu().tolist())) == ref_stats and (lcd.cpu().numpy() == ref_len).all()
        perm = np.random.default_rng(pad).permutation(stream["n_blocks"])
        rec = np.asarray(stream["records"]).reshape(-1, 256)[perm].reshape(-1)
        hdr = np.asarray(stream["hdr"]).reshape(-1, 4)[perm].reshape(-1)
        shuffled = engine.upload_stream(dict(records=rec, hdr=hdr, n_blocks=stream["n_blocks"], n=stream["n"]))
        fresh.fill_(-3)
        st, lcd = engine.new_bin_accumulators()
        engine.bin_stream_device(fresh, shuffled, protocol, st, lcd, fresh=True)
        assert t.equal(fresh, want)
        assert dict(zip(ref_stats, st.cpu().tolist())) == ref_stats
    finally:
        engine.set_layout("dense")


@pytest.mark.gpu
def test_sparse_library_falls_back_to_columns(engine):
    """The packer refuses the sparse library; bam.Alignments then keeps its columns and bins them with the column
    kernel, to the oracle's coverage."""
    from ribotricer_b200 import _lib
    from ribotricer_b200.bam import Alignments, ReadColumns

    CO = _oracle()
    names, lens = genome()
    lt, base, plane = _setup(engine, 64)
    reads = library("sparse")
    with pytest.raises(_lib.RtError):
        engine.stream_reads(reads)
    al = Alignments(engine, ReadColumns(names, lens, dict(reads), True), "forward")
    assert al.dstream is None and al.dcols is not None
    cov = engine.new_coverage()
    stats = al.bin_into(cov, OFFSETS)
    ref_cov, ref_stats, _ = CO.bin_reads(reads, 0, lt, base, lens, 64, plane)
    assert dict(zip(ref_stats, stats.cpu().tolist())) == ref_stats
    assert (cov.cpu().numpy() == ref_cov).all()


@pytest.mark.gpu
@pytest.mark.parametrize("pad", PADS)
def test_scores_and_profiles_match_oracle(engine, pad):
    """Scores of every ORF in both layouts against the oracle (frame_K equal), score_device once, and the profiles of
    every ORF on a contig above 255 or on an edge-length contig plus a sample of the rest."""
    CO = _oracle()
    t = engine.torch
    _, lens = genome()
    lt, base, plane = _setup(engine, pad)
    idx = index()
    ref_cov, _, _ = CO.bin_reads(library("dense"), 0, lt, base, lens, pad, plane)
    ref = CO.score(idx, ref_cov, base, lens, pad, plane, DEFAULT_PARAMS)
    tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
    n_orf = len(idx["orf_contig"])
    assert tie.sum() < 0.05 * n_orf and (ref["count"] > 0).sum() > n_orf // 3
    dense = t.from_numpy(ref_cov).to(engine.device)
    edge = np.isin(idx["orf_contig"], EDGE_IDS)
    rng = np.random.default_rng(pad)
    sel = np.flatnonzero(edge | (idx["orf_contig"] >= 256) | (rng.random(n_orf) < 0.1))
    assert edge.sum() > 300 and (idx["orf_contig"][sel] >= 256).sum() > 10_000 and len(sel) < n_orf
    rptr, rprof = CO.gather_profiles(idx, sel, ref_cov, base, lens, pad, plane)
    try:
        for layout in ("dense", "compact"):
            engine.set_layout(layout)
            cov = dense if layout == "dense" else _compact_of(engine, ref_cov)
            got = engine.score_host(cov, diagnostics=True)
            compare_scores(got, ref, tie, what=f"{layout}: ")
            assert (got["frame_K"] == ref["frame_K"]).all()
            ptr, prof = engine.gather_profiles(cov, sel, got["length"][sel])
            assert (ptr == rptr).all() and (prof == rprof).all()
            if layout == "compact":
                out = engine.new_score_columns(n_orf, diagnostics=True)
                engine.score_device(cov, out)
                dev = {k: v.cpu().numpy() for k, v in out.items()}
                for k in got:
                    assert np.array_equal(dev[k], got[k], equal_nan=True), k
    finally:
        engine.set_layout("dense")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dense", "sparse"])
def test_detect_orfs_from_bam_matches_cpu_twin(engine, tmp_path, monkeypatch, kind):
    """detect_orfs() from a BAM of all 1,900 references and an index with rows on chromosomes the BAM lacks, once on the
    GPU and once on the CPU twin: the BAM summary and both WIG files are byte-identical, the TSV agrees row by row under helpers.compare_tsv.  The
    dense library takes the stream kernel, the sparse one the column kernel."""
    from oracle_engine import install
    from ribotricer_b200 import detect_orfs as D

    reads = library(kind)
    bam, idx_path = tmp_path / "lib.bam", tmp_path / "index.tsv"
    write_bam(bam, reads)
    write_index(idx_path)
    paths = {}
    for who in ("gpu", "twin"):
        with monkeypatch.context() as m:
            m.setattr(D, "_INDEX_CACHE", {})
            if who == "gpu":
                m.setattr(D, "_ENGINE", engine)
                seen = []
                orig = engine.bin_stream_device
                m.setattr(engine, "bin_stream_device", lambda *a, **k: (seen.append(1), orig(*a, **k))[1])
            else:
                install(m)
            prefix = str(tmp_path / who / "run")
            D.detect_orfs(str(bam), str(idx_path), prefix, "forward", None, dict(OFFSETS), *DEFAULT_PARAMS, True,
                          meta_min_reads=10 ** 9)
            if who == "gpu":
                assert bool(seen) == (kind == "dense")
            paths[who] = prefix
    for suffix in ("_bam_summary.txt", "_pos.wig", "_neg.wig"):
        assert open(paths["gpu"] + suffix, "rb").read() == open(paths["twin"] + suffix, "rb").read(), suffix
    got = open(paths["gpu"] + "_translating_ORFs.tsv").read()
    want = open(paths["twin"] + "_translating_ORFs.tsv").read()
    n_rows = compare_tsv(got, want, DEFAULT_PARAMS[0])
    assert n_rows > 15_000
    assert sum(1 for line in want.split("\n") if "\tscaffold_99999\t" in line or "\tchrAbsent\t" in line) == 4
