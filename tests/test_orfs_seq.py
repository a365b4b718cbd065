"""orfs-seq: the nucleotide or protein sequence of every index row (DESIGN.md section 10).

CPU tests drive the host flow (native index loader and ``rt_index_ids``, native FASTA loader, contig mapping, the
CLI) with ``Engine.orf_seq_write`` answered by the plain-Python statement of the rules (``oracle/seq_py.py``); the GPU
tests run the same comparisons through ``orf_seq_kernel``.
"""
from __future__ import annotations

import os

import numpy as np
import pytest

from oracle import prepare_py as P
from oracle import seq_py as S

PARAM_SETS = {
    "defaults": dict(min_orf_length=60, start_codons={"ATG"}, stop_codons={"TAG", "TAA", "TGA"}, longest=False),
    "longest": dict(min_orf_length=60, start_codons={"ATG"}, stop_codons={"TAG", "TAA", "TGA"}, longest=True),
    "near_cognate_min30": dict(min_orf_length=30, start_codons={"ATG", "CTG", "GTG"},
                               stop_codons={"TAG", "TAA", "TGA"}, longest=False),
}


class StatementEngine:
    """``Engine.orf_seq_write`` answered by the plain-Python rules."""

    def __init__(self):
        self.device_index, self.ctx, self.calls = 0, object(), 0

    def orf_seq_write(self, path, exon_ptr, exon_start, exon_end, orf_contig, orf_strand, contig_base, contig_len,
                      codes, id_off, ids, protein, chunk_bytes=0, stage_ms=None):
        self.calls += 1
        assert len(contig_base) == len(contig_len) and len(id_off) == len(exon_ptr)
        letters = np.frombuffer(b"ACGTN", np.uint8)[codes].tobytes().decode()
        genome = {c: letters[int(b):int(b) + int(n)] for c, (b, n) in enumerate(zip(contig_base, contig_len))}
        blob = bytes(np.asarray(ids, np.uint8)).decode("latin-1")
        rows = []
        for o in range(len(exon_ptr) - 1):
            ivs = list(zip(exon_start[exon_ptr[o]:exon_ptr[o + 1]].tolist(), exon_end[exon_ptr[o]:exon_ptr[o + 1]].tolist()))
            rows.append((blob[id_off[o]:id_off[o + 1]], int(orf_contig[o]), "-" if orf_strand[o] == 1 else "+", ivs))
        text = S.lines_text(rows, genome, protein)          # raises before anything is written
        with open(path, "wb") as fh:
            fh.write(text.encode("latin-1"))


@pytest.fixture
def statement_engine(built, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    eng = StatementEngine()
    monkeypatch.setattr(D, "_ENGINE", eng)
    return eng


@pytest.fixture
def gpu_engine(engine, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    monkeypatch.setattr(D, "_ENGINE", engine)
    return engine


@pytest.fixture(scope="module")
def annotation(tmp_path_factory):
    from ribotricer_b200 import synth

    return synth.make_annotation(str(tmp_path_factory.mktemp("annot")), n_genes=40, genome_size=400_000, seed=11)


def _run(tmp_path, index, fasta, protein, name="seq.tsv", **kw):
    from ribotricer_b200.orf_seq import orf_seq

    out = os.path.join(str(tmp_path), "out", name)
    orf_seq(index, fasta, out, protein, **kw)
    with open(out, "rb") as fh:
        return fh.read().decode("latin-1")


def _index_file(tmp_path, ann, params, name="idx.tsv"):
    path = os.path.join(str(tmp_path), name)
    with open(path, "w") as fh:
        fh.write(P.prepare_orfs_text(ann["gtf"], ann["fasta"], params["min_orf_length"], params["start_codons"],
                                     params["stop_codons"], params["longest"]))
    return path


# ------------------------------------------------------------------------------------------------ known answer
KNOWN_FASTA = ">c1 first\nATGaaaTGAnCC\nGGGTAA\n>c2\nCCCATGGTTTAG\n>unused\nACGT\n"
# c1 1-18: A T G a a a T G A n C C G G G T A A   (upper case, n -> N: ATGAAATGANCCGGGTAA)
# c2 1-12: C C C A T G G T T T A G
KNOWN_INDEX_ROWS = [
    # + row, intervals listed unsorted: 13-18 then 1-6 -> ATGAAA + GGGTAA
    ("R1", "c1", "+", "13-18,1-6"),
    # - row over two intervals: c2 1-3 and 7-12 = CCC + GTTTAG, reverse complement CTAAACGGG
    ("R2", "c2", "-", "7-12,1-3"),
    # lowercase and N bases, a length not divisible by 3, a codon holding N: c1 5-12 = AATGANCC (8 nt)
    ("R3", "c1", "+", "5-12"),
    # strand "." reads as +: c2 4-9 = ATGGTT
    ("R4", "c2", ".", "4-9"),
    # a duplicate ORF_ID, kept as is
    ("R1", "c2", "-", "4-12"),
]
KNOWN_NT = ["ATGAAAGGGTAA", "CTAAACGGG", "AATGANCC", "ATGGTT", "CTAAACCAT"]
KNOWN_AA = ["MKG*", "LNG", "NX", "MV", "LNH"]   # R2: CTA AAC GGG; R3: AAT GAN, CC dropped


def _known(tmp_path):
    fa, idx = tmp_path / "k.fa", tmp_path / "k_candidate_orfs.tsv"
    fa.write_text(KNOWN_FASTA)
    idx.write_text(P.HEADER + "".join(
        f"{oid}\tuORF\tT\tpc\tG\tG\tpc\t{chrom}\t{strand}\tATG\t{coord}\n"
        for oid, chrom, strand, coord in KNOWN_INDEX_ROWS))
    return str(idx), str(fa)


def _known_text(seqs):
    return S.HEADER + "".join(f"{r[0]}\t{s}\n" for r, s in zip(KNOWN_INDEX_ROWS, seqs))


def test_known_answer(tmp_path, statement_engine):
    idx, fa = _known(tmp_path)
    for protein, seqs in ((False, KNOWN_NT), (True, KNOWN_AA)):
        want = _known_text(seqs)
        assert S.orfs_seq_text(idx, fa, protein) == want
        assert _run(tmp_path, idx, fa, protein) == want
    assert statement_engine.calls == 2


def test_oracle_codon_table_is_the_standard_code():
    assert len(S.CODON_TABLE) == 64 and sorted(c for c, a in S.CODON_TABLE.items() if a == "*") == ["TAA", "TAG", "TGA"]
    assert S.translate("ATGTGGTTTAAAGGCCCTX") == "MWFKGP"
    assert S.translate("ATGNAATTTAC") == "MXF"


# ------------------------------------------------------------------------------------------------ ids, host flow
def test_index_ids_are_the_first_column(tmp_path, annotation, built):
    from ribotricer_b200.index import load_native_index

    path = _index_file(tmp_path, annotation, PARAM_SETS["near_cognate_min30"])
    with open(path, "a") as fh:                     # a duplicate id and an empty id
        fh.write("T_dup\tuORF\tT\tpc\tG\tG\tpc\tchr1\t+\tATG\t1-9\n" * 2)
        fh.write("\tuORF\tT\tpc\tG\tG\tpc\tchr1\t+\tATG\t1-9\n")
    want = [line.split("\t", 1)[0] for line in open(path).read().splitlines()[1:]]
    off, blob = load_native_index(path).ids()
    got = [bytes(blob[off[o]:off[o + 1]]).decode() for o in range(len(off) - 1)]
    assert got == want and len(got) > 100


@pytest.mark.parametrize("which", list(PARAM_SETS))
def test_host_flow_matches_the_statement(tmp_path, annotation, statement_engine, which):
    idx = _index_file(tmp_path, annotation, PARAM_SETS[which])
    for protein in (False, True):
        assert _run(tmp_path, idx, annotation["fasta"], protein) == S.orfs_seq_text(idx, annotation["fasta"], protein)


def test_header_only_index(tmp_path, statement_engine):
    _, fa = _known(tmp_path)
    idx = tmp_path / "empty.tsv"
    idx.write_text(P.HEADER)
    assert _run(tmp_path, str(idx), fa, False) == S.HEADER


# ------------------------------------------------------------------------------------------------ errors
BAD_ROWS = [
    ("c9\t+\tATG\t1-9", "chrom c9 of the index \\(2 rows\\) is absent from the FASTA"),
    ("c1\t+\tATG\t0-9", "ORF BAD: interval 0-9 is outside its contig of 18 nt"),
    ("c1\t-\tATG\t1-3,9-6", "ORF BAD: interval 9-6 ends before it starts"),
    ("c2\t+\tATG\t1-3,10-13", "ORF BAD: interval 10-13 is outside its contig of 12 nt"),
]


def _bad_index(tmp_path, row):
    idx, fa = _known(tmp_path)
    bad = tmp_path / "bad.tsv"
    text = open(idx).read() + f"BAD\tuORF\tT\tpc\tG\tG\tpc\t{row}\n"
    if row.startswith("c9"):
        text += f"BAD2\tuORF\tT\tpc\tG\tG\tpc\t{row}\n"
    bad.write_text(text)
    return str(bad), fa


@pytest.mark.parametrize("row,message", BAD_ROWS)
def test_errors_leave_no_file(tmp_path, statement_engine, row, message):
    idx, fa = _bad_index(tmp_path, row)
    out = tmp_path / "out" / "seq.tsv"
    with pytest.raises(ValueError, match=message):
        S.orfs_seq_text(idx, fa)
    with pytest.raises(ValueError, match=message):
        _run(tmp_path, idx, fa, False)
    assert not out.exists()


def test_gzip_and_column_count(tmp_path, statement_engine):
    import gzip

    idx, fa = _known(tmp_path)
    gz_fa, gz_idx = tmp_path / "k.fa.gz", tmp_path / "idx.tsv.gz"
    with gzip.open(gz_fa, "wt") as fh:
        fh.write(KNOWN_FASTA)
    with gzip.open(gz_idx, "wt") as fh:
        fh.write(open(idx).read())
    for args in ((idx, str(gz_fa)), (str(gz_idx), fa)):
        with pytest.raises(ValueError, match="gzip-compressed; orfs-seq reads plain text only"):
            _run(tmp_path, *args, False)
    short = tmp_path / "short.tsv"
    short.write_text(P.HEADER + "R1\tuORF\tc1\t+\tATG\t1-9\n")
    with pytest.raises(SystemExit, match="unexpected number of columns"):
        _run(tmp_path, str(short), fa, False)
    with pytest.raises(SystemExit, match="unexpected number of columns"):
        S.orfs_seq_text(str(short), fa)
    assert not (tmp_path / "out" / "seq.tsv").exists()


# ------------------------------------------------------------------------------------------------ CLI
def test_cli_writes_the_same_bytes(tmp_path, annotation, statement_engine):
    from click.testing import CliRunner

    from ribotricer_b200.cli import cli

    idx = _index_file(tmp_path, annotation, PARAM_SETS["defaults"])
    for protein in (False, True):
        want = _run(tmp_path, idx, annotation["fasta"], protein, name="py.tsv")
        out = os.path.join(str(tmp_path), "cli", "seq.tsv")
        args = ["orfs-seq", "--ribotricer_index", idx, "--fasta", annotation["fasta"], "--saveto", out]
        res = CliRunner().invoke(cli, args + (["--protein"] if protein else []))
        assert res.exit_code == 0, res.output
        assert open(out, "rb").read().decode("latin-1") == want
    for bad, what in ((["--fasta", annotation["fasta"] + ".missing"], "FASTA file not found"),
                      (["--ribotricer_index", idx + ".missing"], "ribotricer index file not found")):
        res = CliRunner().invoke(cli, args + bad)
        assert res.exit_code != 0 and what in str(res.exception), bad
    bad_idx, fa = _bad_index(tmp_path, BAD_ROWS[1][0])
    res = CliRunner().invoke(cli, ["orfs-seq", "--ribotricer_index", bad_idx, "--fasta", fa, "--saveto", out + "2"])
    assert res.exit_code != 0 and "interval 0-9" in str(res.exception) and not os.path.exists(out + "2")


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_known_answer_and_errors(tmp_path, gpu_engine):
    idx, fa = _known(tmp_path)
    assert _run(tmp_path, idx, fa, False) == _known_text(KNOWN_NT)
    assert _run(tmp_path, idx, fa, True) == _known_text(KNOWN_AA)
    empty = tmp_path / "empty.tsv"
    empty.write_text(P.HEADER)
    assert _run(tmp_path, str(empty), fa, True) == S.HEADER
    for row, message in BAD_ROWS:
        bad, _ = _bad_index(tmp_path, row)
        with pytest.raises(ValueError, match=message):
            _run(tmp_path, bad, fa, False, name="bad.tsv")
        assert not (tmp_path / "out" / "bad.tsv").exists()


@pytest.mark.gpu
@pytest.mark.parametrize("which", list(PARAM_SETS))
def test_gpu_matches_the_statement(tmp_path, annotation, gpu_engine, which):
    idx = _index_file(tmp_path, annotation, PARAM_SETS[which])
    for protein in (False, True):
        assert _run(tmp_path, idx, annotation["fasta"], protein) == S.orfs_seq_text(idx, annotation["fasta"], protein)


@pytest.mark.gpu
def test_gpu_chunking_gives_the_same_file(tmp_path, annotation, gpu_engine):
    idx = _index_file(tmp_path, annotation, PARAM_SETS["near_cognate_min30"])
    for protein in (False, True):
        want = _run(tmp_path, idx, annotation["fasta"], protein, name="default.tsv")
        assert len(want) > 3 * 4096
        for chunk in (4096, 1):
            assert _run(tmp_path, idx, annotation["fasta"], protein, name=f"c{chunk}.tsv", chunk_bytes=chunk) == want


@pytest.mark.gpu
def test_gpu_chain_prepare_then_seq(tmp_path, gpu_engine):
    """prepare_orfs on the GPU, then orf_seq: lengths, first codons and proteins of every row."""
    from ribotricer_b200 import synth
    from ribotricer_b200.index import parse_index
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    ann = synth.make_annotation(str(tmp_path / "chain"), n_genes=300, genome_size=6_000_000, seed=29, edge_cases=False)
    prefix = str(tmp_path / "idx" / "chain")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    idx = parse_index(ipath)
    nt_path, aa_path = str(tmp_path / "nt.tsv"), str(tmp_path / "aa.tsv")
    orf_seq(ipath, ann["fasta"], nt_path)
    orf_seq(ipath, ann["fasta"], aa_path, translate=True)
    nt = [line.split("\t") for line in open(nt_path).read().splitlines()[1:]]
    aa = [line.split("\t") for line in open(aa_path).read().splitlines()[1:]]
    ids = [line.split("\t", 1)[0] for line in open(ipath).read().splitlines()[1:]]
    assert len(nt) == len(aa) == idx.n_orf > 1000
    lengths = idx.lengths()
    for o in range(idx.n_orf):
        assert nt[o][0] == aa[o][0] == ids[o]
        assert len(nt[o][1]) == lengths[o] and len(aa[o][1]) == lengths[o] // 3
        assert nt[o][1][:3] == idx.fields[o][6] == "ATG"
        assert "*" not in aa[o][1]
    by_id = {a[0]: a[1] for a in aa}
    for tid, p in ann["planted"].items():
        oid = f"{tid}_{p['cds'][0][0]}_{p['cds'][-1][1]}_{sum(e - s + 1 for s, e in p['cds'])}"
        assert by_id[oid].startswith("M"), tid


@pytest.mark.gpu
def test_gpu_large_random_case(tmp_path, gpu_engine):
    from ribotricer_b200 import synth
    from ribotricer_b200.prepare_orfs import prepare_orfs

    ann = synth.make_annotation(str(tmp_path / "big"), n_genes=6_000, tx_per_gene=3.4, genome_size=50_000_000, seed=5)
    prefix = str(tmp_path / "idx" / "big")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    rows = S.parse_rows(ipath)
    genome = P.parse_fasta(ann["fasta"])
    assert len(rows) > 20_000
    for protein in (False, True):
        assert _run(tmp_path, ipath, ann["fasta"], protein) == S.lines_text(rows, genome, protein), protein
