"""prepare-orfs: GTF + FASTA -> candidate-ORF index (DESIGN.md section 9).

CPU tests drive the whole host flow (native GTF / FASTA loaders, transcript table, annotated rows, native writer) with
``Engine.orf_search`` answered by the plain-Python statement of the rules (``oracle/prepare_py.py``); the GPU tests run
the same comparisons through the real kernels.
"""
from __future__ import annotations

import os

import numpy as np
import pytest

from oracle import prepare_py as P

PARAM_SETS = {
    "defaults": dict(min_orf_length=60, start_codons={"ATG"}, stop_codons={"TAG", "TAA", "TGA"}, longest=False),
    "longest": dict(min_orf_length=60, start_codons={"ATG"}, stop_codons={"TAG", "TAA", "TGA"}, longest=True),
    "near_cognate_min30": dict(min_orf_length=30, start_codons={"ATG", "CTG", "GTG"},
                               stop_codons={"TAG", "TAA", "TGA"}, longest=False),
    "min0_taa": dict(min_orf_length=0, start_codons={"ATG"}, stop_codons={"TAA"}, longest=False),
}


class StatementEngine:
    """``Engine.orf_search`` answered by the plain-Python rules (str.find over the spliced transcript strings)."""

    def __init__(self):
        self.device_index, self.ctx, self.calls = 0, object(), 0

    def orf_search(self, codes, tx_base, exon_ptr, exon_start, exon_end, tx_strand, tx_cds, start_mask, stop_mask,
                   min_orf_length, longest, stage_ms=None):
        self.calls += 1
        letters = np.frombuffer(b"ACGTN", np.uint8)
        codons = [a + b + c for a in "ACGT" for b in "ACGT" for c in "ACGT"]
        starts = {codons[i] for i in range(64) if (start_mask >> i) & 1}
        stops = {codons[i] for i in range(64) if (stop_mask >> i) & 1}
        out = {k: [] for k in ("row_tx", "row_start", "row_stop", "row_type", "row_codon", "iv_start", "iv_end")}
        iv_ptr = [0]
        for t in range(len(tx_base)):
            exons = [(int(exon_start[e]), int(exon_end[e])) for e in range(exon_ptr[t], exon_ptr[t + 1])]
            strand = "+" if tx_strand[t] == 0 else "-"
            genome = {"c": letters[codes].tobytes().decode()[int(tx_base[t]):int(tx_base[t]) + exons[-1][1]]}
            seq = P.spliced(genome, "c", strand, exons)
            cds = None if tx_cds[t][0] < 0 else (int(tx_cds[t][0]), int(tx_cds[t][1]))
            for s, p, kind in P.candidates(seq, cds, starts, stops, min_orf_length, longest):
                out["row_tx"].append(t)
                out["row_start"].append(s)
                out["row_stop"].append(p)
                out["row_type"].append(P.TYPES.index(kind))
                out["row_codon"].append(codons.index(seq[s:s + 3]))
                for a, b in P.to_genomic(exons, strand, s, p):
                    out["iv_start"].append(a)
                    out["iv_end"].append(b)
                iv_ptr.append(len(out["iv_start"]))
        dt = dict(row_tx=np.int32, row_start=np.int32, row_stop=np.int32, row_type=np.uint8, row_codon=np.uint8,
                  iv_start=np.int32, iv_end=np.int32)
        res = {k: np.asarray(v, dt[k]) for k, v in out.items()}
        res["iv_ptr"] = np.asarray(iv_ptr, np.int64)
        return res


@pytest.fixture
def statement_engine(built, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    eng = StatementEngine()
    monkeypatch.setattr(D, "_ENGINE", eng)
    return eng


@pytest.fixture(scope="module")
def annotation(tmp_path_factory):
    from ribotricer_b200 import synth

    return synth.make_annotation(str(tmp_path_factory.mktemp("annot")), n_genes=40, genome_size=400_000, seed=11)


def _run(tmp_path, ann, params, name="idx"):
    from ribotricer_b200.prepare_orfs import prepare_orfs

    prefix = os.path.join(str(tmp_path), "out", name)
    prepare_orfs(ann["gtf"], ann["fasta"], prefix, **params)
    return open(prefix + "_candidate_orfs.tsv").read()


def _expected(ann, params):
    return P.prepare_orfs_text(ann["gtf"], ann["fasta"], params["min_orf_length"], params["start_codons"],
                               params["stop_codons"], params["longest"])


# ------------------------------------------------------------------------------------------------ known answer
KNOWN_FASTA = ">k1 known\nCCATGAAATAAGGATGATGCCCTGATT\nAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA\n>k2\n" \
              "TTAGGGCATCATTTTT\n"
# k1 1-27: C C A T G A A A T A A G G A T G A T G C C C T G A T T
#          1 2 3 4 5 6 7 8 9 ...
# T1 (+, exons 1-11 and 14-27): spliced CCATGAAATAA|ATGATGCCCTGATT (25 nt, spliced = genomic - 3 in exon 2), CDS 17-22
# T2 (-, k2 1-16): reverse complement of TTAGGGCATCATTTTT is AAAAATGATGCCCTAA
KNOWN_GTF = "\n".join([
    'k1\tt\texon\t1\t11\t.\t+\t.\tgene_id "GA"; transcript_id "T1"; gene_name "A"; gene_type "pc"; transcript_type "pc";',
    'k1\tt\texon\t14\t27\t.\t+\t.\tgene_id "GA"; transcript_id "T1";',
    'k1\tt\tCDS\t17\t22\t.\t+\t0\tgene_id "GA"; transcript_id "T1";',
    'k2\tt\texon\t1\t16\t.\t-\t.\ttranscript_id "T2"; gene_id "GB"; gene_biotype "lnc";',
]) + "\n"


def test_known_answer(tmp_path, statement_engine):
    """Expected rows written out by hand from the rules (min length 0).
    T1 spliced (+): CCATGAAATAAATGATGCCCTGATT; positions 0-based; starts ATG at 2, 11, 14; stops TAA at 8, TGA at 20.
      s=2 (frame 2): next in-frame stop 8 -> [2, 8) genomic 3-8; CDS = nt 17-22 -> oriented 14..19 (c=14, d=19).
        b=7 < c -> uORF.
      (TGA at 3 and 12 are in frame 0 and stop nothing.)
      s=11 (frame 2): stops in frame 2 after 11: 20 -> [11, 20) = nt 14-22, a=11 < c=14 <= b=19 = d -> super_uORF.
      s=14 (frame 2): stop 20 -> [14, 20): a=c, b=d -> annotated (not written).
      With --longest, s=11 and s=14 share stop 20: only s=11 is kept (s=14 was annotated anyway).
    Annotated row: CDS 17-22, first codon ATG.
    T2 (-): AAAAATGATGCCCTAA; starts 4 (frame 1), 7 (frame 1); stop TAA at 13 (frame 1), TGA at 5 (frame 2); no CDS
      -> novel; transcript_type absent -> NA, gene_name absent -> gene_id, gene_type from gene_biotype.
      s=4 -> [4, 13) genomic: n=16, ascending [16-13, 16-4) = [3, 12) -> nt 4-12.
      s=7 -> [7, 13) -> ascending [3, 9) -> nt 4-9.  --longest keeps s=4 only.
    """
    fa, gtf = tmp_path / "k.fa", tmp_path / "k.gtf"
    fa.write_text(KNOWN_FASTA)
    gtf.write_text(KNOWN_GTF)
    ann = dict(fasta=str(fa), gtf=str(gtf))
    head = P.HEADER
    a_row = "T1_17_22_6\tannotated\tT1\tpc\tGA\tA\tpc\tk1\t+\tATG\t17-22\n"
    u_row = "T1_3_8_6\tuORF\tT1\tpc\tGA\tA\tpc\tk1\t+\tATG\t3-8\n"
    s_row = "T1_14_22_9\tsuper_uORF\tT1\tpc\tGA\tA\tpc\tk1\t+\tATG\t14-22\n"
    n4 = "T2_4_12_9\tnovel\tT2\tNA\tGB\tGB\tlnc\tk2\t-\tATG\t4-12\n"
    n7 = "T2_4_9_6\tnovel\tT2\tNA\tGB\tGB\tlnc\tk2\t-\tATG\t4-9\n"
    base = dict(min_orf_length=0, start_codons={"ATG"}, stop_codons={"TAG", "TAA", "TGA"})
    assert _run(tmp_path, ann, dict(base, longest=False)) == head + a_row + u_row + s_row + n4 + n7
    assert _run(tmp_path, ann, dict(base, longest=True)) == head + a_row + u_row + s_row + n4
    assert P.prepare_orfs_text(ann["gtf"], ann["fasta"], 0) == head + a_row + u_row + s_row + n4 + n7


# ------------------------------------------------------------------------------------------------ loaders
def test_gtf_loader_matches_the_statement(annotation, monkeypatch, built):
    from ribotricer_b200.prepare_orfs import load_gtf

    ref = P.parse_gtf(annotation["gtf"])
    results = []
    for threads in ("1", "3", "8"):
        monkeypatch.setenv("RT_GTF_THREADS", threads)
        g = load_gtf(annotation["gtf"])
        s = g["strings"]
        get = lambda i: None if i < 0 else s[i]  # noqa: E731
        rows = [(int(g["line"][i]), "exon" if g["feature"][i] == 0 else "CDS", s[g["chrom"][i]], int(g["start"][i]),
                 int(g["end"][i]), "+-."[min(2, g["strand"][i])], *[get(a) for a in g["attr"][i].tolist()])
                for i in range(len(g["line"]))]
        results.append(rows)
    assert results[0] == results[1] == results[2]
    want = [(r["line"], r["feature"], r["chrom"], r["start"], r["end"], r["strand"] if r["strand"] in "+-" else ".",
             r["gene_id"], r["transcript_id"], r["gene_name"],
             None if r["gene_type"] == "NA" else r["gene_type"],
             None if r["transcript_type"] == "NA" else r["transcript_type"]) for r in ref]
    assert results[0] == want


def test_fasta_loader_matches_the_statement(annotation, built):
    from ribotricer_b200.prepare_orfs import Genome

    ref = P.parse_fasta(annotation["fasta"])
    g = Genome(annotation["fasta"])
    assert g.names == list(ref) and g.lengths.tolist() == [len(v) for v in ref.values()]
    codes = g.codes(np.arange(len(g.names)))
    assert np.frombuffer(b"ACGTN", np.uint8)[codes].tobytes().decode() == "".join(ref.values())
    assert not os.path.exists(annotation["fasta"] + ".fai")


@pytest.fixture(scope="module")
def big_fasta(tmp_path_factory):
    """Contigs of a few bases up to one of 9 Mb (several 8 MB pieces), 60- and 61-column lines, one with CRLF ends."""
    rng = np.random.default_rng(5)
    path = tmp_path_factory.mktemp("fa") / "g.fa"
    parts = []
    for i, (n, width, eol) in enumerate([(5, 60, "\n"), (9_000_000, 60, "\n"), (130_001, 61, "\r\n"), (1, 60, "\n")]):
        seq = np.frombuffer(b"ACGTNacgt", np.uint8)[rng.integers(0, 9, n)].tobytes().decode()
        parts.append(f">c{i} contig {i}{eol}" + "".join(seq[j:j + width] + eol for j in range(0, n, width)))
    path.write_text("".join(parts), newline="")
    return str(path)


@pytest.mark.parametrize("threads", ["1", "2", "7"])
def test_fasta_loader_thread_count_does_not_change_the_codes(big_fasta, built, monkeypatch, threads):
    from ribotricer_b200.prepare_orfs import Genome

    ref = P.parse_fasta(big_fasta)
    monkeypatch.setenv("RT_FASTA_THREADS", threads)
    g = Genome(big_fasta)
    assert g.names == list(ref) and g.lengths.tolist() == [len(v) for v in ref.values()]
    codes = g.codes(np.arange(len(g.names))[::-1].copy())
    assert np.frombuffer(b"ACGTN", np.uint8)[codes].tobytes().decode() == "".join(reversed(ref.values()))


def _orf_rows(n_rows, seed=9):
    """Arguments of rt_orf_write for n_rows rows of two transcripts, and the text the rows must become."""
    rng = np.random.default_rng(seed)
    tx = ["T1\tpc\tGA\tA\tpc\tk1\t+", "TX22\tNA\tGB\tGB\tlnc\tk2\t-"]
    tx_text = "".join(tx).encode()
    tx_off = np.array([0, len(tx[0]), len(tx[0]) + len(tx[1])], np.int64)
    tx_id_len = np.array([2, 4], np.int32)
    row_tx = rng.integers(0, 2, n_rows).astype(np.int32)
    row_type = rng.integers(0, 8, n_rows).astype(np.uint8)
    row_codon = rng.integers(0, 64, n_rows).astype(np.uint8)
    n_iv = rng.integers(1, 4, n_rows)
    iv_ptr = np.zeros(n_rows + 1, np.int64)
    np.cumsum(n_iv, out=iv_ptr[1:])
    iv_start = rng.integers(1, 10**9, iv_ptr[-1]).astype(np.int32)
    iv_end = (iv_start + rng.integers(0, 5000, iv_ptr[-1])).astype(np.int32)
    args = (len(tx), tx_text, tx_off, tx_id_len, n_rows, row_tx, row_type, row_codon, iv_ptr, iv_start, iv_end)
    acgt = "ACGT"
    lines = [P.HEADER]
    for r in range(n_rows):
        t, a, b = int(row_tx[r]), int(iv_ptr[r]), int(iv_ptr[r + 1])
        ivs = list(zip(iv_start[a:b].tolist(), iv_end[a:b].tolist()))
        c = int(row_codon[r])
        lines.append(f"{tx[t][:tx_id_len[t]]}_{ivs[0][0]}_{ivs[-1][1]}_{sum(e - s + 1 for s, e in ivs)}\t"
                     f"{P.TYPES[row_type[r]]}\t{tx[t]}\t{acgt[c >> 4 & 3]}{acgt[c >> 2 & 3]}{acgt[c & 3]}\t"
                     + ",".join(f"{s}-{e}" for s, e in ivs) + "\n")
    return args, "".join(lines)


def _orf_write(path, args):
    import ctypes as C

    from ribotricer_b200 import _lib

    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    n_tx, tx_text, tx_off, tx_id_len, n_rows, *cols = args
    return _lib.load().rt_orf_write(str(path).encode(), n_tx, tx_text, p(tx_off), p(tx_id_len), n_rows, *map(p, cols))


@pytest.mark.parametrize("threads", ["1", "3"])
def test_index_writer_thread_count_does_not_change_the_bytes(tmp_path, built, monkeypatch, threads):
    args, want = _orf_rows(450_000)                     # 7 rounds of 64 Ki rows on one thread, 3 on three
    monkeypatch.setenv("RT_WRITE_THREADS", threads)
    assert _orf_write(tmp_path / "idx.tsv", args) == 0
    assert (tmp_path / "idx.tsv").read_text() == want


@pytest.mark.parametrize("n_rows", [0, 200_000])
def test_index_writer_reports_a_refused_write(tmp_path, built, n_rows):
    """The header alone fails when the file is closed; megabytes of rows fail in the write-behind thread."""
    from ribotricer_b200 import _lib

    if not os.path.exists("/dev/full"):
        pytest.skip("no /dev/full")
    lib = _lib.load()
    args, _ = _orf_rows(n_rows)
    assert _orf_write(tmp_path / "missing" / "idx.tsv", args) != 0
    assert lib.rt_io_last_error().decode().startswith("cannot open")
    assert _orf_write("/dev/full", args) != 0
    assert lib.rt_io_last_error().decode() == "write failed: /dev/full"


@pytest.mark.parametrize("text,message", [
    ("c\tt\texon\t1\t10\t.\t+\t.\n", "GTF line 2: expected 9 tab-separated columns, found 8"),
    ("c\tt\texon\tx1\t10\t.\t+\t.\tgene_id \"g\";\n", "GTF line 2: start is not a positive integer"),
    ("c\tt\tgene\t1\t1e3\t.\t+\t.\tgene_id \"g\";\n", "GTF line 2: end is not a positive integer"),
    ("c\tt\tCDS\t20\t10\t.\t+\t.\tgene_id \"g\";\n", "GTF line 2: start > end"),
])
def test_gtf_errors_name_the_line(tmp_path, built, monkeypatch, text, message):
    from ribotricer_b200.prepare_orfs import load_gtf

    path = tmp_path / "bad.gtf"
    path.write_text("# comment\n" + text + "c\tt\texon\t1\t10\t.\t+\t.\tgene_id \"g\"; transcript_id \"t\";\n")
    for threads in ("1", "2"):
        monkeypatch.setenv("RT_GTF_THREADS", threads)
        with pytest.raises(ValueError, match=message):
            load_gtf(str(path))
    with pytest.raises(P.GtfError, match=message):
        P.parse_gtf(str(path))


def test_fasta_and_gzip_errors(tmp_path, built):
    import gzip

    from ribotricer_b200.prepare_orfs import Genome, load_gtf

    dup = tmp_path / "dup.fa"
    dup.write_text(">a x\nACGT\n>b\nAC\n>a\nGG\n")
    with pytest.raises(ValueError, match="duplicate FASTA contig a"):
        Genome(str(dup))
    with pytest.raises(P.FastaError, match="duplicate FASTA contig a"):
        P.parse_fasta(str(dup))
    gz = tmp_path / "a.gtf.gz"
    with gzip.open(gz, "wt") as fh:
        fh.write("c\tt\texon\t1\t10\t.\t+\t.\tgene_id \"g\";\n")
    with pytest.raises(ValueError, match="gzip"):
        load_gtf(str(gz))


# ------------------------------------------------------------------------------------------------ host flow
@pytest.mark.parametrize("which", list(PARAM_SETS))
def test_host_flow_matches_the_statement(tmp_path, annotation, statement_engine, which):
    params = PARAM_SETS[which]
    got = _run(tmp_path, annotation, params)
    assert statement_engine.calls == 1
    assert got == _expected(annotation, params)


def test_generated_annotation_covers_the_cases(tmp_path, annotation, statement_engine):
    text = _run(tmp_path, annotation, PARAM_SETS["near_cognate_min30"])
    kinds = {line.split("\t")[1] for line in text.splitlines()[1:]}
    assert kinds == set(P.TYPES) - {"internal"}
    codons = {line.split("\t")[9] for line in text.splitlines()[1:] if "\tannotated\t" in line}
    assert codons == {"ATG", "CTG"}                     # the non-ATG CDS is written when CTG is a start codon
    _, skipped = P.transcripts(P.parse_gtf(annotation["gtf"]), P.parse_fasta(annotation["fasta"]))
    assert skipped == 3                                 # contig absent, past the contig end, two strands
    assert "-" in {line.split("\t")[8] for line in text.splitlines()[1:]}
    assert "\r\n" in open(annotation["gtf"], newline="").read()


def test_round_trip_through_the_index_loaders(tmp_path, annotation, statement_engine):
    from ribotricer_b200.index import load_native_index, parse_index

    _run(tmp_path, annotation, PARAM_SETS["defaults"])
    path = os.path.join(str(tmp_path), "out", "idx_candidate_orfs.tsv")
    lines = open(path).read().splitlines()[1:]
    native, packed = load_native_index(path), parse_index(path)
    assert native.n_orf == packed.n_orf == len(lines)
    n_ann = sum(1 for line in lines if line.split("\t")[1] == "annotated")
    assert native.n_annotated_prefix == packed.n_annotated_prefix == n_ann
    for o, line in enumerate(lines):
        assert line.split("\t")[0] == native.oid(o) == packed.oid(o)


def test_cli_writes_the_same_file_and_rejects_bad_codons(tmp_path, annotation, statement_engine):
    from click.testing import CliRunner

    from ribotricer_b200.cli import cli

    want = _run(tmp_path, annotation, PARAM_SETS["near_cognate_min30"], name="py")
    prefix = os.path.join(str(tmp_path), "cli", "idx")
    args = ["prepare-orfs", "--gtf", annotation["gtf"], "--fasta", annotation["fasta"], "--prefix", prefix]
    res = CliRunner().invoke(cli, args + ["--min_orf_length", "30", "--start_codons", " atg, CTG ,GTG"])
    assert res.exit_code == 0, res.output
    assert open(prefix + "_candidate_orfs.tsv").read() == want
    for bad in (["--start_codons", "ATGA"], ["--stop_codons", "TNA"], ["--start_codons", ""],
                ["--min_orf_length", "-1"], ["--gtf", annotation["gtf"] + ".missing"]):
        res = CliRunner().invoke(cli, args + bad)
        assert res.exit_code != 0 and "Error" in str(res.exception if res.exception else res.output), bad
    gz = os.path.join(str(tmp_path), "a.gtf.gz")
    open(gz, "wb").write(b"\x1f\x8b")
    res = CliRunner().invoke(cli, ["prepare-orfs", "--gtf", gz, "--fasta", annotation["fasta"], "--prefix", prefix])
    assert res.exit_code != 0


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("which", list(PARAM_SETS))
def test_gpu_matches_the_statement(tmp_path, annotation, engine, monkeypatch, which):
    from ribotricer_b200 import detect_orfs as D

    monkeypatch.setattr(D, "_ENGINE", engine)
    params = PARAM_SETS[which]
    assert _run(tmp_path, annotation, params) == _expected(annotation, params)


@pytest.mark.gpu
def test_gpu_codon_sets_that_overlap(tmp_path, annotation, engine, monkeypatch):
    """A codon in both sets (a start at a stop opens the next stop segment), with and without --longest."""
    from ribotricer_b200 import detect_orfs as D

    monkeypatch.setattr(D, "_ENGINE", engine)
    for longest in (False, True):
        params = dict(min_orf_length=0, start_codons={"ATG", "TAA", "CTG"}, stop_codons={"TAA", "TGA", "CTG"},
                      longest=longest)
        assert _run(tmp_path, annotation, params) == _expected(annotation, params), longest


@pytest.mark.gpu
def test_gpu_large_random_case(tmp_path, engine, monkeypatch):
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import synth

    monkeypatch.setattr(D, "_ENGINE", engine)
    ann = synth.make_annotation(str(tmp_path / "big"), n_genes=6_000, tx_per_gene=3.4, genome_size=50_000_000, seed=5)
    for which in ("defaults", "longest"):
        params = PARAM_SETS[which]
        got = _run(tmp_path, ann, params, name=which)
        assert got.count("\n") > 20_000
        assert got == _expected(ann, params), which


@pytest.mark.gpu
def test_gpu_chain_prepare_then_detect(tmp_path, engine, monkeypatch):
    """Index built here -> reads on the planted CDS -> detect_orfs: the planted CDS rows are annotated and
    translating, and the scores meet the C checker."""
    import helpers
    from oracle import c_oracle
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import synth
    from ribotricer_b200.bam import ReadColumns, save_read_columns
    from ribotricer_b200.index import parse_index

    monkeypatch.setattr(D, "_ENGINE", engine)
    ann = synth.make_annotation(str(tmp_path / "chain"), n_genes=60, genome_size=1_500_000, seed=23, edge_cases=False)
    prefix = str(tmp_path / "idx" / "chain")
    from ribotricer_b200.prepare_orfs import prepare_orfs
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    idx = parse_index(ipath)
    names = [c for c, _ in ann["contigs"]]
    clen = np.array([n for _, n in ann["contigs"]], np.int64)
    n_ann = idx.n_annotated_prefix
    assert n_ann == len(ann["planted"]) > 0
    # the annotated rows as the synthetic index make_reads expects (reads only on the planted CDS, no background)
    sub = slice(0, n_ann)
    eptr = idx.exon_ptr[:n_ann + 1]
    sidx = synth.SynthIndex(names, clen, eptr, idx.exon_start[:eptr[-1]], idx.exon_end[:eptr[-1]],
                            np.array([names.index(c) for c in idx.chrom[sub]], np.int32),
                            np.array([0 if s == "+" else 1 for s in idx.strand[sub]], np.uint8),
                            idx.lengths()[:n_ann], np.arange(n_ann), n_ann)
    cfg = synth.SynthConfig("chain", ann["contigs"], n_ann, 200_000, 31, expr_shape=5.0)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, sidx, device="cpu"))
    bam = str(tmp_path / "reads.npz")
    save_read_columns(bam, ReadColumns(names, clen, reads, True))
    out = str(tmp_path / "det" / "chain")
    D.detect_orfs(bam, ipath, out, "forward", sorted(synth.TRUE_OFFSETS), dict(synth.TRUE_OFFSETS), *helpers.DEFAULT_PARAMS,
                  report_all=True)
    rows = [line.rstrip("\n").split("\t") for line in open(out + "_translating_ORFs.tsv")][1:]
    ann_rows = {r[9]: r for r in rows if r[1] == "annotated"}
    assert set(ann["planted"]) == set(ann_rows)
    for tid, p in ann["planted"].items():       # the row is the planted CDS
        assert ann_rows[tid][0] == f"{tid}_{p['cds'][0][0]}_{p['cds'][-1][1]}_{sum(e - s + 1 for s, e in p['cds'])}"
    # make_reads expresses ~60 % of the ORFs; a planted CDS can be as short as 2 codons, and a row with fewer than
    # min_valid_codons (5) covered codons is nontranslating by the filters whatever its phase score
    expressed = [r for r in ann_rows.values() if float(r[8]) >= 1.0 and int(r[6]) >= helpers.DEFAULT_PARAMS[1]]
    assert len(expressed) >= len(ann_rows) // 3
    assert all(r[2] == "translating" for r in expressed)
    # scores of every index row against the C checker
    eng = D.get_engine()
    eng.set_genome(names, clen)
    eng.set_length_table(dict(synth.TRUE_OFFSETS), None)
    eng.set_index(**idx.device_columns({n: i for i, n in enumerate(names)}))
    cov = eng.new_coverage()
    eng.bin_reads_host(cov, reads, "forward")
    got = eng.score_host(cov, diagnostics=True)
    base, plane = c_oracle.genome_layout(clen, eng.pad)
    ref_cov, _, _ = c_oracle.bin_reads(reads, 0, c_oracle.make_len_table(dict(synth.TRUE_OFFSETS), None), base, clen,
                                       eng.pad, plane)
    ref = c_oracle.score(idx.device_columns({n: i for i, n in enumerate(names)}), ref_cov, base, clen, eng.pad, plane,
                         list(helpers.DEFAULT_PARAMS))
    helpers.compare_scores(got, ref, c_oracle.tie_mask(ref["frame_K"], ref["frame_s"]))
