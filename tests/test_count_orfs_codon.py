"""count-orfs-codon: per-gene and pooled codon tables of detected ORFs (DESIGN.md section 11).

CPU tests drive the host flow (native index, TSV and sequence-file loaders, the table writer, the CLI) with
``Engine.codon_counts`` answered by the plain-Python statement of the rules (``oracle/codon_py.py``); the GPU tests run
the same comparisons through ``codon_emit_kernel``, the radix sorts and ``codon_stats_kernel``.
"""
from __future__ import annotations

import gzip
import os

import numpy as np
import pytest

from oracle import codon_py as CP

INDEX_HEADER = ("ORF_ID\tORF_type\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\t"
                "start_codon\tcoordinate\n")
TSV_HEADER = ("ORF_ID\tORF_type\tstatus\tphase_score\tread_count\tlength\tvalid_codons\tvalid_codons_ratio\t"
              "read_density\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\t"
              "start_codon\tprofile\n")
FEATURES = {"annotated", "uORF"}


class StatementEngine:
    """``Engine.codon_counts`` answered by the plain-Python rules, from the columns the native loaders hand over."""

    def __init__(self):
        self.device_index, self.ctx, self.calls = 0, object(), 0

    def codon_counts(self, sel, tsv, seq, exon_ptr, exon_start, exon_end, orf_strand, n_gene, n_gseq, stage_ms=None):
        self.calls += 1
        tsv, seq = bytes(tsv), bytes(seq)
        items = []
        for i in range(len(sel["row"])):
            o = int(sel["row"][i])
            ivs = list(zip(exon_start[exon_ptr[o]:exon_ptr[o + 1]].tolist(), exon_end[exon_ptr[o]:exon_ptr[o + 1]].tolist()))
            coor = [p for s, e in ivs for p in range(s, e + 1)]
            if orf_strand[o] == 1:
                coor = coor[::-1]
            a, n = int(sel["prof_off"][i]), int(sel["prof_len"][i])
            s0 = int(sel["seq_off"][o])
            assert 0 <= int(sel["gene"][i]) < n_gene and 0 <= int(sel["gseq"][i]) < n_gseq
            items.append((i, int(sel["gene"][i]), int(sel["gseq"][i]), tsv[a:a + n], seq[s0:s0 + len(coor)], coor))
        res = CP.codons(items)
        gene_tab = np.zeros((64 * n_gene, 5), np.uint64)
        pooled_tab = np.zeros((64, 5), np.uint64)
        if res[0] == "refused":
            return gene_tab, pooled_tab, np.array([0, 0, 0, 0, res[1], res[2]], np.int64)
        by_gene, pooled, s = res
        code = {a + b + c: 16 * i + 4 * j + k for i, a in enumerate("ACGT") for j, b in enumerate("ACGT")
                for k, c in enumerate("ACGT")}
        for (g, name), xs in by_gene.items():
            gene_tab[64 * g + code[name]] = CP.stat_cell(xs)
        for name, xs in pooled.items():
            pooled_tab[code[name]] = CP.stat_cell(xs)
        return gene_tab, pooled_tab, np.array([s["codons"], s["with_n"], s["duplicates"], s["kept"], -1, 0], np.int64)


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


def _run(tmp_path, index, tsv, seq, features=FEATURES, report_all=False, name="out"):
    from ribotricer_b200.count_orfs import count_orfs_codon

    prefix = os.path.join(str(tmp_path), name, "run")
    summary = count_orfs_codon(index, tsv, features, seq, prefix, report_all)
    texts = []
    for suffix in ("_codon_counts_by_gene.tsv", "_codon_counts.tsv"):
        with open(prefix + suffix, "rb") as fh:
            texts.append(fh.read().decode("latin-1"))
    return texts[0], texts[1], summary


def _files(tmp_path, index_rows, seqs, tsv_rows, tag="k"):
    """Index, orfs-seq file and detected-ORFs TSV from row tuples."""
    idx, seq, tsv = tmp_path / f"{tag}_index.tsv", tmp_path / f"{tag}_seq.tsv", tmp_path / f"{tag}_orfs.tsv"
    idx.write_text(INDEX_HEADER + "".join("\t".join(r) + "\n" for r in index_rows))
    seq.write_text("ORF_ID\tsequence\n" + "".join(f"{r[0]}\t{s}\n" for r, s in zip(index_rows, seqs)))
    tsv.write_text(TSV_HEADER + "".join("\t".join(r) + "\n" for r in tsv_rows))
    return str(idx), str(tsv), str(seq)


def _tsv_row(oid, otype, status, tid, gid, gname, chrom, strand, profile):
    return (oid, otype, status, "0.9", "10", "9", "3", "1.0", "1.1", tid, "protein_coding", gid, gname, "protein_coding",
            chrom, strand, "ATG", profile)


# ------------------------------------------------------------------------------------------------ known answer
def _irow(oid, otype, tid, gid, gname, chrom, strand, coord):
    return (oid, otype, tid, "protein_coding", gid, gname, "protein_coding", chrom, strand, "ATG", coord)


KNOWN_INDEX = [
    _irow("T1_1_9_9", "uORF", "T1", "G1", "g1", "chr1", "+", "1-9"),
    _irow("T2_4_12_9", "uORF", "T2", "G1", "g1", "chr1", "+", "4-12"),           # shares AAA@4 and CCC@7 with T1
    _irow("T4_2_7_6", "uORF", "T4", "G1", "g1", "chr1", "+", "2-7"),             # another frame: kept
    _irow("T3_10_32_9", "uORF", "T3", "G2", "g2", "chr2", "-", "30-32,10-15"),   # '-' over two intervals
    _irow("T5_100_107_8", "annotated", "T5", "G3", "g3", "chr1", "+", "100-107"),  # ANG, CCC, trailing TT
    _irow("T6_200_211_12", "uORF", "T6", "G3", "g3", "chr1", "+", "200-211"),    # profile of 7 values
    _irow("T7_1_6_6", "uORF", "T7", "G4", "g4", "chr3", "+", "1-6"),             # nontranslating
    _irow("T8_10_15_6", "novel", "T8", "G4", "g4", "chr3", "+", "10-15"),        # type not in the features
    _irow("T9_50_55_6", "uORF", "T9", "G1", "g1b", "chr1", "+", "50-55"),        # same gene_id, other name
]
KNOWN_SEQS = ["ATGAAACCC", "AAACCCGGG", "TGAAAC", "ATGCCCAAA", "ANGCCCTT", "AAAAAACCCGGG", "GGGTTT", "CCCCCC", "ATGATG"]
KNOWN_TSV = [
    _tsv_row("T1_1_9_9", "uORF", "translating", "T1", "G1", "g1", "chr1", "+", "[1, 2, 3, 4, 5, 6, 7, 8, 9]"),
    _tsv_row("T2_4_12_9", "uORF", "translating", "T2", "G1", "g1", "chr1", "+", "[100, 0, 0, 200, 0, 0, 1, 1, 1]"),
    _tsv_row("T4_2_7_6", "uORF", "translating", "T4", "G1", "g1", "chr1", "+", "[0, 0, 5, 0, 0, 2]"),
    _tsv_row("T3_10_32_9", "uORF", "translating", "T3", "G2", "g2", "chr2", "-", "[10, 0, 0, 3, 3, 3, 0, 0, 1]"),
    _tsv_row("T5_100_107_8", "annotated", "translating", "T5", "G3", "g3", "chr1", "+", "[1, 1, 1, 2, 2, 2, 9, 9]"),
    _tsv_row("T6_200_211_12", "uORF", "translating", "T6", "G3", "g3", "chr1", "+", "[4, 0, 0, 1, 1, 1, 7]"),
    _tsv_row("T7_1_6_6", "uORF", "nontranslating", "T7", "G4", "g4", "chr3", "+", "[5, 5, 5, 6, 6, 6]"),
    _tsv_row("T8_10_15_6", "novel", "translating", "T8", "G4", "g4", "chr3", "+", "[1, 1, 1, 1, 1, 1]"),
    _tsv_row("T9_50_55_6", "uORF", "translating", "T9", "G1", "g1b", "chr1", "+", "[2, 2, 2, 0, 0, 0]"),
]
# worked out by hand: T2's AAA and CCC repeat T1's places and are skipped; ANG holds an N; T6 has 7 values -> 2 codons
KNOWN_GENE = CP.GENE_HEADER + """\
G1\tAAA\t1\t15\t15.0\t15.0\t0.0
G1\tAAC\t1\t2\t2.0\t2.0\t0.0
G1\tATG\t1\t6\t6.0\t6.0\t0.0
G1\tCCC\t1\t24\t24.0\t24.0\t0.0
G1\tGGG\t1\t3\t3.0\t3.0\t0.0
G1\tTGA\t1\t5\t5.0\t5.0\t0.0
G1\tATG\t2\t6\t3.0\t3.0\t9.0
G2\tAAA\t1\t1\t1.0\t1.0\t0.0
G2\tATG\t1\t10\t10.0\t10.0\t0.0
G2\tCCC\t1\t9\t9.0\t9.0\t0.0
G3\tAAA\t2\t7\t3.5\t3.5\t0.25
G3\tCCC\t1\t6\t6.0\t6.0\t0.0
"""
KNOWN_CODON = CP.CODON_HEADER + """\
AAA\t4\t23\t5.75\t3.5\t29.6875
AAC\t1\t2\t2.0\t2.0\t0.0
ATG\t4\t22\t5.5\t6.0\t12.75
CCC\t3\t39\t13.0\t9.0\t62.0
GGG\t1\t3\t3.0\t3.0\t0.0
TGA\t1\t5\t5.0\t5.0\t0.0
"""
# --report_all adds T7 (G4): GGG 15, TTT 18
KNOWN_GENE_ALL = KNOWN_GENE + "G4\tGGG\t1\t15\t15.0\t15.0\t0.0\nG4\tTTT\t1\t18\t18.0\t18.0\t0.0\n"
KNOWN_CODON_ALL = KNOWN_CODON.replace("GGG\t1\t3\t3.0\t3.0\t0.0\n", "GGG\t2\t18\t9.0\t9.0\t36.0\n") + \
    "TTT\t1\t18\t18.0\t18.0\t0.0\n"
KNOWN_SUMMARY = dict(rows=7, genes=4, codons=14, duplicates=2, codons_with_n=1)


def _known(tmp_path, tsv_rows=None, seqs=None, tag="k"):
    return _files(tmp_path, KNOWN_INDEX, KNOWN_SEQS if seqs is None else seqs,
                  KNOWN_TSV if tsv_rows is None else tsv_rows, tag)


def _check_known(tmp_path):
    idx, tsv, seq = _known(tmp_path)
    for report_all, gene, codon in ((False, KNOWN_GENE, KNOWN_CODON), (True, KNOWN_GENE_ALL, KNOWN_CODON_ALL)):
        g, c, s = CP.count_orfs_codon_text(idx, tsv, FEATURES, seq, report_all)
        assert (g, c) == (gene, codon)
        got = _run(tmp_path, idx, tsv, seq, report_all=report_all)
        assert got[:2] == (gene, codon)
        assert {k: got[2][k] for k in s} == s
    assert s == dict(KNOWN_SUMMARY, rows=8, genes=5, codons=16)
    assert CP.count_orfs_codon_text(idx, tsv, FEATURES, seq)[2] == KNOWN_SUMMARY


def test_known_answer(tmp_path, statement_engine):
    _check_known(tmp_path)
    assert statement_engine.calls == 2


def test_empty_selection_gives_header_only_files(tmp_path, statement_engine):
    idx, tsv, seq = _known(tmp_path)
    gene, codon, summary = _run(tmp_path, idx, tsv, seq, features={"dORF"})
    assert (gene, codon) == (CP.GENE_HEADER, CP.CODON_HEADER) and summary["rows"] == 0
    empty = tmp_path / "empty.tsv"
    empty.write_text("")
    assert _run(tmp_path, idx, str(empty), seq, name="e")[:2] == (CP.GENE_HEADER, CP.CODON_HEADER)


# ------------------------------------------------------------------------------------------------ random cases
def random_case(tmp_path, seed, n_rows=300, n_genes=25, big=False, long_rows=0, tag="r"):
    """A random index, its sequence file and a shuffled detected-ORFs TSV with repeated lines.  Rows of one gene
    overlap often, so codons are shared; ``big`` puts maximal values into some codons (counts up to 2^32 - 1)."""
    rng = np.random.default_rng(seed)
    genes = [(f"G{g % (n_genes - 3)}", f"n{g}") for g in range(n_genes)]     # a few ids carry two names
    irows, seqs, trows = [], [], []
    for o in range(n_rows):
        gid, gname = genes[int(rng.integers(n_genes))]
        chrom = ("chr1", "chr2")[int(rng.integers(2))]
        strand = "+-."[int(rng.choice(3, p=[0.45, 0.45, 0.1]))]
        ivs, at = [], int(rng.integers(1, 400))
        for _ in range(int(rng.integers(1, 4))):
            n = int(rng.integers(1, 60))
            ivs.append((at, at + n - 1))
            at += n + int(rng.integers(0, 40))
        if o < long_rows:
            ivs = [(5, 5 + 100_500 + o)]
        length = sum(e - s + 1 for s, e in ivs)
        tid = f"T{o}"
        coord = ",".join(f"{s}-{e}" for s, e in (ivs[::-1] if rng.random() < 0.3 else ivs))
        otype = ("uORF", "annotated", "novel")[int(rng.choice(3, p=[0.5, 0.3, 0.2]))]
        irows.append(_irow(f"{tid}_{ivs[0][0]}_{ivs[-1][1]}_{length}", otype, tid, gid, gname, chrom, strand, coord))
        seqs.append("".join(rng.choice(list("ACGTN"), size=length, p=[0.24, 0.24, 0.24, 0.24, 0.04])))
        n_val = max(0, length + int(rng.integers(-6, 7))) if rng.random() < 0.9 else int(rng.integers(0, 2))
        vals = rng.poisson(1.5, n_val) * (rng.random(n_val) < 0.5) + (rng.random(n_val) < 0.05) * rng.integers(10, 100000, n_val)
        vals = vals.astype(np.int64)
        if big and n_val >= 3:
            for k in rng.choice(n_val // 3, size=min(3, n_val // 3), replace=False) if n_val // 3 else []:
                vals[3 * k:3 * k + 3] = [2 ** 31 - 1, 2 ** 31 - 1, 1] if rng.random() < 0.5 else [2 ** 31 - 1, 0, 5]
        status = "translating" if rng.random() < 0.7 else "nontranslating"
        trows.append(_tsv_row(irows[-1][0], otype, status, tid, gid, gname, chrom, strand, str(vals.tolist())))
    trows += [trows[int(k)] for k in rng.integers(0, n_rows, n_rows // 10)]
    order = rng.permutation(len(trows))
    return _files(tmp_path, irows, seqs, [trows[int(k)] for k in order], tag)


@pytest.mark.parametrize("threads", ["1", "2", "7"])
def test_loaders_match_the_statement(tmp_path, built, monkeypatch, threads):
    from ribotricer_b200.count_orfs import CodonInput
    from ribotricer_b200.index import load_native_index

    idx, tsv, seq = random_case(tmp_path, 3, n_rows=400)
    monkeypatch.setenv("RT_CODON_THREADS", threads)
    rows = CP.index_rows(idx)
    for report_all in (False, True):
        want = CP.select(tsv, rows, FEATURES, report_all)
        inp = CodonInput(load_native_index(idx), tsv, FEATURES, report_all)
        inp.load_seq(seq)
        assert inp.n_sel == len(want) > 100 and inp.n_lines == 440
        text = bytes(inp.text(0))
        keys, places = [], {}
        for i, (line_no, o, key, prof) in enumerate(want):
            assert int(inp.sel["line"][i]) == line_no and int(inp.sel["row"][i]) == o
            a = int(inp.sel["prof_off"][i])
            assert text[a:a + int(inp.sel["prof_len"][i])] == prof
            if key not in keys:
                keys.append(key)
            assert int(inp.sel["gene"][i]) == keys.index(key) and inp.gene(keys.index(key)) == key
            place = (key, rows[o].chrom, rows[o].strand)
            assert places.setdefault(place, int(inp.sel["gseq"][i])) == int(inp.sel["gseq"][i])
        assert inp.n_gene == len(keys) and inp.n_gseq == len(places) == len(set(places.values()))
        seqs = CP.sequences(seq, rows)
        letters = bytes(inp.text(1))
        for o, s in enumerate(seqs):
            assert letters[int(inp.sel["seq_off"][o]):int(inp.sel["seq_off"][o]) + len(s)] == s


def test_random_case_host_flow(tmp_path, statement_engine):
    idx, tsv, seq = random_case(tmp_path, 5, big=True)
    for report_all in (False, True):
        g, c, s = CP.count_orfs_codon_text(idx, tsv, FEATURES, seq, report_all)
        got = _run(tmp_path, idx, tsv, seq, report_all=report_all)
        assert got[:2] == (g, c) and {k: got[2][k] for k in s} == s
        assert s["duplicates"] > 0 and s["codons_with_n"] > 0


# ------------------------------------------------------------------------------------------------ errors
def _bad_cases(tmp_path):
    """(name, files, message) per refused input; every case is the known answer with one thing broken."""
    cases = []
    short = list(KNOWN_TSV)
    short[2] = short[2][:-1]
    cases.append(("fields", _known(tmp_path, short, tag="b1"), r"line 4: 17 tab-separated fields, 18 expected"))
    unknown = list(KNOWN_TSV)
    unknown[3] = ("T3_10_32_10",) + unknown[3][1:]
    cases.append(("unknown", _known(tmp_path, unknown, tag="b2"), r"line 5: ORF_ID T3_10_32_10 is not in the index"))
    for k, (prof, why) in enumerate((("[1,2, 3]", "not a list of integers"), ("[1, 02, 3]", "not a list of integers"),
                                     ("[1, 2147483648]", "outside 0..2147483647"),
                                     ("[2147483647, 2147483647, 2, 0, 0, 0]", "codon count exceeds 4294967295"))):
        bad = list(KNOWN_TSV)
        bad[5] = bad[5][:-1] + (prof,)
        cases.append((f"profile{k}", _known(tmp_path, bad, tag=f"b3{k}"), rf"line 7: .*{why}"))
    protein = ["MKP", "KPG", "*N", "MPK", "XP", "KKPG", "GF", "PP", "MM"]
    cases.append(("protein", _known(tmp_path, seqs=protein, tag="b4"),
                  r"line 2: the sequence of T1_1_9_9 has 3 letters, the index row has 9 nt.*without --protein"))
    idx, tsv, seq = _known(tmp_path, tag="b5")
    text = open(seq).read().replace("T4_2_7_6\t", "T4_2_7_7\t")
    open(seq, "w").write(text)
    cases.append(("other_index", (idx, tsv, seq), r"line 4: ORF_ID T4_2_7_7 is not T4_2_7_6"))
    return cases


def _check_errors(tmp_path):
    for name, (idx, tsv, seq), message in _bad_cases(tmp_path):
        with pytest.raises(ValueError, match=message) as want:
            CP.count_orfs_codon_text(idx, tsv, FEATURES, seq)
        with pytest.raises(ValueError) as got:
            _run(tmp_path, idx, tsv, seq, name=name)
        assert str(got.value) == str(want.value), name
        assert not os.path.exists(os.path.join(str(tmp_path), name)), name
    idx, tsv, seq = _known(tmp_path)
    for k in range(3):
        args = [idx, tsv, seq]
        gz = str(tmp_path / f"in{k}.gz")
        with gzip.open(gz, "wb") as fh:
            fh.write(open(args[k], "rb").read())
        args[k] = gz
        with pytest.raises(ValueError, match="gzip-compressed; count-orfs-codon reads plain text only"):
            _run(tmp_path, *args, name="gz")
        assert not os.path.exists(os.path.join(str(tmp_path), "gz"))


def test_errors_leave_no_file(tmp_path, statement_engine):
    _check_errors(tmp_path)


# ------------------------------------------------------------------------------------------------ CLI
def test_cli_writes_the_same_bytes(tmp_path, statement_engine):
    from click.testing import CliRunner

    from ribotricer_b200.cli import cli

    idx, tsv, seq = random_case(tmp_path, 9)
    want = _run(tmp_path, idx, tsv, seq, features={"uORF", "annotated"}, report_all=True)
    prefix = str(tmp_path / "cli" / "run")
    args = ["count-orfs-codon", "--ribotricer_index", idx, "--detected_orfs", tsv, "--features", "uORF, annotated",
            "--ribotricer_index_fasta", seq, "--prefix", prefix, "--report_all"]
    res = CliRunner().invoke(cli, args)
    assert res.exit_code == 0, res.output
    assert open(prefix + "_codon_counts_by_gene.tsv", "rb").read().decode("latin-1") == want[0]
    assert open(prefix + "_codon_counts.tsv", "rb").read().decode("latin-1") == want[1]
    res = CliRunner().invoke(cli, [seq + ".missing" if a == seq else a for a in args])
    assert res.exit_code != 0 and "ribotricer index fasta file not found" in str(res.exception)
    _, (bidx, btsv, bseq), message = _bad_cases(tmp_path)[1]
    res = CliRunner().invoke(cli, ["count-orfs-codon", "--ribotricer_index", bidx, "--detected_orfs", btsv, "--features",
                                   "uORF,annotated", "--ribotricer_index_fasta", bseq, "--prefix", prefix + "2"])
    assert res.exit_code != 0 and "is not in the index" in str(res.exception)
    assert not os.path.exists(prefix + "2_codon_counts.tsv")


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_known_answer_and_errors(tmp_path, gpu_engine):
    _check_known(tmp_path)
    _check_errors(tmp_path)
    idx, tsv, seq = _known(tmp_path)
    assert _run(tmp_path, idx, tsv, seq, features={"dORF"}, name="e")[:2] == (CP.GENE_HEADER, CP.CODON_HEADER)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,big,long_rows", [(1, False, 0), (2, True, 0), (4, True, 3)])
def test_gpu_random_cases(tmp_path, gpu_engine, seed, big, long_rows):
    idx, tsv, seq = random_case(tmp_path, seed, n_rows=500, big=big, long_rows=long_rows)
    for report_all in (False, True):
        g, c, s = CP.count_orfs_codon_text(idx, tsv, FEATURES, seq, report_all)
        got = _run(tmp_path, idx, tsv, seq, report_all=report_all)
        assert got[:2] == (g, c) and {k: got[2][k] for k in s} == s, (seed, report_all)
    if big:
        assert "4294967295" in open(tsv).read() or "2147483647" in open(tsv).read()


@pytest.mark.gpu
def test_gpu_chain_prepare_seq_detect_then_codons(tmp_path, gpu_engine):
    """prepare_orfs -> orf_seq -> detect_orfs(report_all) on reads over the planted CDS -> count_orfs_codon."""
    import helpers
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import synth
    from ribotricer_b200.bam import ReadColumns, save_read_columns
    from ribotricer_b200.index import parse_index
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    ann = synth.make_annotation(str(tmp_path / "chain"), n_genes=60, genome_size=1_500_000, seed=23, edge_cases=False)
    prefix = str(tmp_path / "idx" / "chain")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    spath = str(tmp_path / "idx" / "chain_seq.tsv")
    orf_seq(ipath, ann["fasta"], spath)
    idx = parse_index(ipath)
    names = [c for c, _ in ann["contigs"]]
    clen = np.array([n for _, n in ann["contigs"]], np.int64)
    n_ann = idx.n_annotated_prefix
    eptr = idx.exon_ptr[:n_ann + 1]
    sidx = synth.SynthIndex(names, clen, eptr, idx.exon_start[:eptr[-1]], idx.exon_end[:eptr[-1]],
                            np.array([names.index(c) for c in idx.chrom[:n_ann]], np.int32),
                            np.array([0 if s == "+" else 1 for s in idx.strand[:n_ann]], np.uint8),
                            idx.lengths()[:n_ann], np.arange(n_ann), n_ann)
    cfg = synth.SynthConfig("chain", ann["contigs"], n_ann, 200_000, 31, expr_shape=5.0)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, sidx, device="cpu"))
    bam = str(tmp_path / "reads.npz")
    save_read_columns(bam, ReadColumns(names, clen, reads, True))
    det = str(tmp_path / "det" / "chain")
    D.detect_orfs(bam, ipath, det, "forward", sorted(synth.TRUE_OFFSETS), dict(synth.TRUE_OFFSETS), *helpers.DEFAULT_PARAMS,
                  report_all=True)
    tsv = det + "_translating_ORFs.tsv"
    features = {"annotated", "uORF", "dORF"}
    for report_all in (False, True):
        g, c, s = CP.count_orfs_codon_text(ipath, tsv, features, spath, report_all)
        got = _run(tmp_path, ipath, tsv, spath, features=features, report_all=report_all)
        assert got[:2] == (g, c) and {k: got[2][k] for k in s} == s
    gene_rows = [line.split("\t") for line in got[0].splitlines()]
    codon_rows = [line.split("\t") for line in got[1].splitlines()]
    assert gene_rows[0] == CP.GENE_HEADER.rstrip("\n").split("\t") and all(len(r) == 7 for r in gene_rows)
    assert codon_rows[0] == CP.CODON_HEADER.rstrip("\n").split("\t") and all(len(r) == 6 for r in codon_rows)
    assert s["codons"] > 1000
    planted_genes = {line.split("\t")[4] for line in open(ipath).read().splitlines()[1:]
                     if line.split("\t")[2] in ann["planted"]}
    assert planted_genes and planted_genes <= {r[0] for r in gene_rows[1:]}


@pytest.mark.gpu
def test_gpu_large_case(tmp_path, gpu_engine):
    idx, tsv, seq = random_case(tmp_path, 17, n_rows=20_000, n_genes=2_000, big=True)
    g, c, s = CP.count_orfs_codon_text(idx, tsv, FEATURES | {"novel"}, seq, True)
    got = _run(tmp_path, idx, tsv, seq, features=FEATURES | {"novel"}, report_all=True)
    assert got[:2] == (g, c) and {k: got[2][k] for k in s} == s
    assert s["rows"] > 20_000
