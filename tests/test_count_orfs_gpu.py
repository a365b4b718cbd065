"""count-orfs on the GPU from the detected-ORFs TSV text (DESIGN.md section 13).

CPU tests drive the host flow (index and TSV loaders, BGZF inputs, the CLI, the table writer) with
``Engine.orf_counts`` answered by a plain-Python restatement of rules 4-6; the GPU tests run the same comparisons through
``count_emit_kernel``, the radix sort and ``count_keep_kernel``.  Every table is compared with ``count_orfs``, the
plain-Python path, or with the tables the unmodified reference wrote (``tests/golden/count_orfs_cases.json.gz``).
"""
from __future__ import annotations

import numpy as np
import pytest

import test_bgzf_inputs as TB
from oracle import codon_py as CP

INDEX_HEADER = ("ORF_ID\tORF_type\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\t"
                "start_codon\tcoordinate\n")
TSV_HEADER = ("ORF_ID\tORF_type\tstatus\tphase_score\tread_count\tlength\tvalid_codons\tvalid_codons_ratio\t"
              "read_density\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\t"
              "start_codon\tprofile\n")
FEATURES = {"annotated", "uORF"}


def statement_counts(sel, tsv, exon_ptr, exon_start, exon_end, orf_strand, n_gene):
    """Rules 3-6 in plain Python over the columns the loader hands over: (total, length, summary[4])."""
    tsv = bytes(tsv)
    total, length = np.zeros(n_gene, np.uint64), np.zeros(n_gene, np.uint64)
    profiles = []
    for i in range(len(sel["row"])):
        a = int(sel["prof_off"][i])
        reason, vals = CP.profile_values(tsv[a:a + int(sel["prof_len"][i])])
        if reason:
            return total, length, np.array([0, 0, i, reason], np.int64)
        profiles.append(vals)
    seen = [dict() for _ in range(n_gene)]
    named = 0
    for i, vals in enumerate(profiles):
        o, g = int(sel["row"][i]), int(sel["gene"][i])
        ivs = sorted(zip(exon_start[exon_ptr[o]:exon_ptr[o + 1]].tolist(), exon_end[exon_ptr[o]:exon_ptr[o + 1]].tolist()))
        coor = [p for s, e in ivs for p in range(s, e + 1)]
        if orf_strand[o] == 1:
            coor = coor[::-1]
        for pos, v in zip(coor, vals):                  # the first m pairs; the first value at a coordinate wins
            named += 1
            seen[g].setdefault(pos, v)
    for g in range(n_gene):
        total[g], length[g] = sum(seen[g].values()), len(seen[g])
    return total, length, np.array([named, int(length.sum()), -1, 0], np.int64)


class StatementEngine:
    """``Engine.orf_counts`` answered by ``statement_counts``."""

    def __init__(self):
        self.device_index, self.ctx, self.counts = 0, object(), 0

    def orf_counts(self, sel, tsv, exon_ptr, exon_start, exon_end, orf_strand, n_gene, stage_ms=None):
        self.counts += 1
        return statement_counts(sel, tsv, exon_ptr, exon_start, exon_end, orf_strand, n_gene)


class ZlibCountEngine(TB.ZlibEngine, StatementEngine):
    """``inflate_bgzf`` answered by zlib and ``orf_counts`` by the statement, for BGZF inputs on the CPU."""

    def __init__(self):
        TB.ZlibEngine.__init__(self)
        self.counts = 0


@pytest.fixture
def statement_engine(built, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    eng = ZlibCountEngine()
    monkeypatch.setattr(D, "_ENGINE", eng)
    return eng


@pytest.fixture
def gpu_engine(engine, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    monkeypatch.setattr(D, "_ENGINE", engine)
    return engine


def _gpu_run(idx, tsv, features, out, report_all=False):
    from ribotricer_b200.count_orfs import count_orfs_gpu

    summary = count_orfs_gpu(idx, tsv, features, out, report_all)
    return open(out, "rb").read(), summary


def _py_run(idx, tsv, features, out, report_all=False):
    from ribotricer_b200.count_orfs import count_orfs

    count_orfs(idx, tsv, features, out, report_all)
    return open(out, "rb").read()


# ------------------------------------------------------------------------------------------------ golden cases
def _golden_cases(tmp_path):
    """(index path, TSV path, features, report_all, the reference's table) of every golden count_orfs case."""
    from helpers import load_golden

    pipe = {c["name"]: c for c in load_golden("pipeline_cases.json.gz")["cases"]}
    for k, c in enumerate(load_golden("count_orfs_cases.json.gz")["cases"]):
        case = pipe[c["case"]]
        idx, tsv = tmp_path / f"g{k}_idx.tsv", tmp_path / f"g{k}_orfs.tsv"
        idx.write_text("\n".join(case["index"]) + "\n")
        tsv.write_text(case["tsv"][c["tsv"]]["text"])
        yield str(idx), str(tsv), set(c["features"]), c["report_all"], c["text"]


def _check_golden(tmp_path):
    n = 0
    for idx, tsv, features, report_all, text in _golden_cases(tmp_path):
        got, summary = _gpu_run(idx, tsv, features, str(tmp_path / "out.tsv"), report_all)
        assert got.decode() == text, (idx, features, report_all)
        assert summary["genes"] == text.count("\n") - 1
        n += 1
    assert n == 72


def test_golden_cases(tmp_path, statement_engine):
    _check_golden(tmp_path)
    assert statement_engine.counts == 72


# ------------------------------------------------------------------------------------------------ random cases
def _irow(oid, otype, tid, gid, gname, chrom, strand, coord):
    return (oid, otype, tid, "protein_coding", gid, gname, "protein_coding", chrom, strand, "ATG", coord)


def _tsv_row(oid, otype, status, tid, gid, gname, chrom, strand, profile):
    return (oid, otype, status, "0.9", "10", "9", "3", "1.0", "1.1", tid, "protein_coding", gid, gname, "protein_coding",
            chrom, strand, "ATG", profile)


def _write(tmp_path, tag, irows, trows):
    idx, tsv = tmp_path / f"{tag}_index.tsv", tmp_path / f"{tag}_orfs.tsv"
    idx.write_text(INDEX_HEADER + "".join("\t".join(r) + "\n" for r in irows))
    tsv.write_text(TSV_HEADER + "".join("\t".join(r) + "\n" for r in trows))
    return str(idx), str(tsv)


def random_case(tmp_path, seed, n_rows=300, n_genes=25, long_rows=0, max_len=60, tag="r"):
    """A random index and a shuffled detected-ORFs TSV with repeated lines.  Genes have ORFs on both chroms at shared
    coordinates; rows run on '+', '-' and '.', some with overlapping intervals; profiles are shorter or longer
    than their row, or "[]"; gene "Gempty" has only "[]" profiles; a few index rows repeat the oid of another row."""
    rng = np.random.default_rng(seed)
    genes = [(f"G{g % (n_genes - 3)}", f"n{g}") for g in range(n_genes)]     # a few ids carry two names
    irows, trows = [], []
    for o in range(n_rows):
        gid, gname = genes[int(rng.integers(n_genes))] if o % 50 else ("Gempty", "e")
        chrom = ("chr1", "chr2")[int(rng.integers(2))]
        strand = "+-."[int(rng.choice(3, p=[0.45, 0.45, 0.1]))]
        ivs, at = [], int(rng.integers(1, 400))
        for _ in range(int(rng.integers(1, 4))):
            n = int(rng.integers(1, max_len))
            ivs.append((at, at + n - 1))
            at += n + int(rng.integers(-n // 2 if rng.random() < 0.1 else 0, 40))      # sometimes overlapping
        if o < long_rows:
            ivs = [(5, 5 + 100_500 + o)]
        ivs.sort()
        tid = f"T{o}"
        otype = ("uORF", "annotated", "novel")[int(rng.choice(3, p=[0.5, 0.3, 0.2]))]
        prev = irows[-1] if irows else None
        if o % 20 == 7 and "," not in prev[10] and int(prev[10].split("-")[1]) - int(prev[10].split("-")[0]) >= 3:
            # the oid, strand and gene of the previous row over other coordinates: the later row is the one matched
            s, e = map(int, prev[10].split("-"))
            otype, tid, gid, gname, chrom, strand = prev[1], prev[2], prev[4], prev[5], prev[7], prev[8]
            ivs = [(s, s + 1), (s + 1, s + 1), (s + 3, e)]
        length = sum(e - s + 1 for s, e in ivs)
        coord = ",".join(f"{s}-{e}" for s, e in (ivs[::-1] if rng.random() < 0.3 else ivs))
        irows.append(_irow(f"{tid}_{ivs[0][0]}_{ivs[-1][1]}_{length}", otype, tid, gid, gname, chrom, strand, coord))
        n_val = max(0, length + int(rng.integers(-6, 7))) if rng.random() < 0.9 else int(rng.integers(0, 2))
        if gid == "Gempty":
            n_val = 0
        vals = rng.poisson(1.5, n_val) * (rng.random(n_val) < 0.5) + (rng.random(n_val) < 0.05) * rng.integers(10, 100000, n_val)
        if n_val and rng.random() < 0.1:
            vals[int(rng.integers(n_val))] = 2 ** 31 - 1
        status = "translating" if rng.random() < 0.7 else "nontranslating"
        trows.append(_tsv_row(irows[-1][0], otype, status, tid, gid, gname, chrom, strand, str(vals.tolist())))
    trows += [trows[int(k)] for k in rng.integers(0, n_rows, n_rows // 10)]
    order = rng.permutation(len(trows))
    return _write(tmp_path, tag, irows, [trows[int(k)] for k in order])


def _check_random(tmp_path, seed, **kw):
    from ribotricer_b200.count_orfs import CodonInput
    from ribotricer_b200.index import load_native_index

    idx, tsv = random_case(tmp_path, seed, tag=f"r{seed}", **kw)
    feats = FEATURES | {"novel"} if seed % 2 else FEATURES
    slots = 0
    for report_all in (False, True):
        want = _py_run(idx, tsv, feats, str(tmp_path / "want.tsv"), report_all)
        got, summary = _gpu_run(idx, tsv, feats, str(tmp_path / "got.tsv"), report_all)
        assert got == want, (seed, report_all)
        assert summary["duplicates"] > 0 and summary["genes"] == want.count(b"\n") - 1
        assert b"Gempty" not in got
        inp = CodonInput(load_native_index(idx), tsv, feats, report_all)
        assert any(inp.gene(g)[0] == b"Gempty" for g in range(inp.n_gene))
        lengths = load_native_index(idx).lengths()
        slots = int(lengths[inp.sel["row"]].sum())
    ids = [line.split("\t", 1)[0] for line in open(idx).read().splitlines()[1:]]
    assert len(ids) > len(set(ids))
    return slots


@pytest.mark.parametrize("seed", [1, 2])
def test_random_cases_match_count_orfs(tmp_path, statement_engine, seed):
    _check_random(tmp_path, seed)


# ------------------------------------------------------------------------------------------------ refusals
KNOWN_INDEX = [
    _irow("T1_1_9_9", "uORF", "T1", "G1", "g1", "chr1", "+", "1-9"),
    _irow("T2_4_12_9", "uORF", "T2", "G1", "g1", "chr1", "-", "4-12"),
    _irow("T3_10_32_9", "annotated", "T3", "G2", "g2", "chr2", "-", "30-32,10-15"),
]
KNOWN_TSV = [
    _tsv_row("T1_1_9_9", "uORF", "translating", "T1", "G1", "g1", "chr1", "+", "[1, 2, 3, 4, 5, 6, 7, 8, 9]"),
    _tsv_row("T2_4_12_9", "uORF", "translating", "T2", "G1", "g1", "chr1", "-", "[100, 0, 0, 200]"),
    _tsv_row("T3_10_32_9", "annotated", "translating", "T3", "G2", "g2", "chr2", "-", "[10, 0, 0, 3, 3, 3, 0, 0, 1]"),
]
# worked out by hand: T2 on '-' puts 100 on 12 and 200 on 9, which T1 already holds
KNOWN_TABLE = b"gene_id\tcount\tlength\nG1\t145\t12\nG2\t20\t9\n"


def _bad_cases(tmp_path):
    """(name, index, TSV, message) per refused input: the known case with line 3 broken."""
    cases = []
    short = list(KNOWN_TSV)
    short[1] = short[1][:-1]
    unknown = list(KNOWN_TSV)
    unknown[1] = ("T2_4_12_8",) + unknown[1][1:]
    for name, rows, why in (("fields", short, "17 tab-separated fields, 18 expected"),
                            ("unknown", unknown, "ORF_ID T2_4_12_8 is not in the index with an ORF_type of the features")):
        idx, tsv = _write(tmp_path, name, KNOWN_INDEX, rows)
        cases.append((name, idx, tsv, f"{tsv} line 3: {why}"))
    for name, prof, bit in (("leading_zero", "[1, 02, 3]", 1), ("sign", "[1, -2, 3]", 1), ("no_space", "[1,2, 3]", 1),
                            ("plus", "[+1, 2]", 1), ("too_big", "[1, 2147483648]", 2)):
        rows = list(KNOWN_TSV)
        rows[1] = rows[1][:-1] + (prof,)
        idx, tsv = _write(tmp_path, name, KNOWN_INDEX, rows)
        cases.append((name, idx, tsv, f"{tsv} line 3: {CP.PROFILE_REASONS[bit]}"))
    return cases


def _check_refusals(tmp_path):
    idx, tsv = _write(tmp_path, "known", KNOWN_INDEX, KNOWN_TSV)
    assert _gpu_run(idx, tsv, FEATURES, str(tmp_path / "known.out"))[0] == KNOWN_TABLE
    assert _py_run(idx, tsv, FEATURES, str(tmp_path / "known_py.out")) == KNOWN_TABLE
    for name, idx, tsv, message in _bad_cases(tmp_path):
        out = tmp_path / f"{name}.out"
        with pytest.raises(ValueError) as err:
            _gpu_run(idx, tsv, FEATURES, str(out))
        assert str(err.value) == message, name
        assert not out.exists(), name


def test_refusals_leave_no_file(tmp_path, statement_engine):
    _check_refusals(tmp_path)


# ------------------------------------------------------------------------------------------------ CLI and BGZF
def _cli(idx, tsv, out, features="annotated, uORF", report_all=False):
    from click.testing import CliRunner

    from ribotricer_b200.cli import cli

    args = ["count-orfs", "--ribotricer_index", idx, "--detected_orfs", tsv, "--features", features, "--out", out]
    return CliRunner().invoke(cli, args + (["--report_all"] if report_all else []))


def _check_cli(tmp_path):
    n = 0
    for k, (idx, tsv, features, report_all, text) in enumerate(_golden_cases(tmp_path)):
        if k % 6:
            continue
        out = str(tmp_path / f"cli{k}.tsv")
        res = _cli(idx, tsv, out, ",".join(sorted(features)), report_all)
        assert res.exit_code == 0, res.output
        assert open(out).read() == text
        b_out = str(tmp_path / f"cli{k}_bgzf.tsv")
        res = _cli(TB._bgz(idx, tmp_path, block=300), TB._bgz(tsv, tmp_path, block=700), b_out, ",".join(sorted(features)),
                   report_all)
        assert res.exit_code == 0, res.output
        assert open(b_out).read() == text
        n += 1
    assert n == 12
    idx, tsv = random_case(tmp_path, 3, tag="cli")
    want = _py_run(idx, tsv, FEATURES, str(tmp_path / "cli_want.tsv"), True)
    out = str(tmp_path / "cli_bgzf.tsv")
    res = _cli(TB._bgz(idx, tmp_path, level=9), TB._bgz(tsv, tmp_path, block=4000), out, report_all=True)
    assert res.exit_code == 0, res.output
    assert open(out, "rb").read() == want
    for k in range(2):
        args = [idx, tsv]
        args[k] = TB._plain_gzip(args[k], tmp_path)
        res = _cli(*args, str(tmp_path / "gz.tsv"))
        assert res.exit_code != 0
        assert str(res.exception) == f"Error: {args[k]} is gzip-compressed; count-orfs reads plain text only"
        assert not (tmp_path / "gz.tsv").exists()
    _, bidx, btsv, message = _bad_cases(tmp_path)[1]
    res = _cli(bidx, btsv, str(tmp_path / "bad.tsv"))
    assert res.exit_code != 0 and str(res.exception) == "Error: " + message
    assert not (tmp_path / "bad.tsv").exists()


def test_cli_writes_the_same_bytes_from_plain_and_bgzf(tmp_path, statement_engine):
    _check_cli(tmp_path)
    assert len(statement_engine.inflated) == 26


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_golden_cases(tmp_path, gpu_engine):
    _check_golden(tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,kw", [(11, {}), (12, dict(long_rows=3)),
                                     (13, dict(n_rows=4000, n_genes=300, max_len=1000))])
def test_gpu_random_cases(tmp_path, gpu_engine, seed, kw):
    slots = _check_random(tmp_path, seed, **kw)
    if seed == 13:
        assert slots > 4_000_000
    if seed == 12:
        assert slots > 300_000


@pytest.mark.gpu
def test_gpu_refusals_leave_no_file(tmp_path, gpu_engine):
    _check_refusals(tmp_path)


@pytest.mark.gpu
def test_gpu_cli_and_bgzf(tmp_path, gpu_engine):
    _check_cli(tmp_path)


@pytest.mark.gpu
def test_gpu_chain_prepare_detect_count(tmp_path, gpu_engine):
    """prepare_orfs -> detect_orfs(report_all) on reads over the planted CDS -> count_orfs_gpu, from plain and BGZF."""
    import helpers
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import synth
    from ribotricer_b200.bam import ReadColumns, save_read_columns
    from ribotricer_b200.index import parse_index
    from ribotricer_b200.prepare_orfs import prepare_orfs

    ann = synth.make_annotation(str(tmp_path / "chain"), n_genes=60, genome_size=1_500_000, seed=29, edge_cases=False)
    prefix = str(tmp_path / "idx" / "chain")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    idx = parse_index(ipath)
    names = [c for c, _ in ann["contigs"]]
    clen = np.array([n for _, n in ann["contigs"]], np.int64)
    n_ann = idx.n_annotated_prefix
    eptr = idx.exon_ptr[:n_ann + 1]
    sidx = synth.SynthIndex(names, clen, eptr, idx.exon_start[:eptr[-1]], idx.exon_end[:eptr[-1]],
                            np.array([names.index(c) for c in idx.chrom[:n_ann]], np.int32),
                            np.array([0 if s == "+" else 1 for s in idx.strand[:n_ann]], np.uint8),
                            idx.lengths()[:n_ann], np.arange(n_ann), n_ann)
    cfg = synth.SynthConfig("chain", ann["contigs"], n_ann, 200_000, 37, expr_shape=5.0)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, sidx, device="cpu"))
    bam = str(tmp_path / "reads.npz")
    save_read_columns(bam, ReadColumns(names, clen, reads, True))
    det = str(tmp_path / "det" / "chain")
    D.detect_orfs(bam, ipath, det, "forward", sorted(synth.TRUE_OFFSETS), dict(synth.TRUE_OFFSETS), *helpers.DEFAULT_PARAMS,
                  report_all=True)
    tsv = det + "_translating_ORFs.tsv"
    features = {"annotated", "uORF", "dORF"}
    b_idx, b_tsv = TB._bgz(ipath, tmp_path), TB._bgz(tsv, tmp_path, block=20_000)
    for report_all in (False, True):
        want = _py_run(ipath, tsv, features, str(tmp_path / "want.tsv"), report_all)
        assert want.count(b"\n") > 20
        for k, (i, t) in enumerate(((ipath, tsv), (b_idx, tsv), (ipath, b_tsv), (b_idx, b_tsv))):
            got, summary = _gpu_run(i, t, features, str(tmp_path / f"got{k}.tsv"), report_all)
            assert got == want, (report_all, k)
        assert summary["positions"] > 10_000
