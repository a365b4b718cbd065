"""The reference-facing Python surface (detect_orfs(), its inner seams, phasescore, the metagene
step) on the GPU, against files and values produced by the unmodified reference."""
import os

import numpy as np
import pytest

from helpers import SCORE_TOL, alignments_to_reads, compare_tsv, load_golden

pytestmark = pytest.mark.gpu


def _read_columns(case, by_length=False):
    from ribotricer_b200.bam import ReadColumns

    names = [c[0] for c in case["contigs"]]
    lens = np.array([c[1] for c in case["contigs"]], np.int64)
    if by_length:   # reads grouped by ascending length: read_length_counts insertion order (bam.py:136)
        case = dict(case, alignments=sorted(case["alignments"], key=lambda a: a[0]))
    return ReadColumns(names, lens, alignments_to_reads(case, names))


def test_phasescore_function(engine):
    """statistics.phasescore mirror: int and float sequences, quirk KATs of SURVEY.md 8(a)."""
    from oracle import oracle_py as O
    from ribotricer_b200.statistics import phasescore

    assert phasescore([], engine) == (0.0, 0)
    assert phasescore([1] + [0] * 29, engine) == (0.0, 0)
    assert phasescore([0, 0, 0, 1] + [0] * 26, engine) == (1.0, 1)
    assert phasescore([1, 1, 1] * 5, engine) == (0.0, 5)
    s, v = phasescore([3, 1, 2, 0, 0, 0, 5, 0, 1, 2, 2, 2, 0, 4, 0, 1], engine)
    assert abs(s - 0.39247762314783674) < 1e-12 and v == 4 and isinstance(s, np.float64)
    cases = load_golden("phasescore_cases.json.gz")["cases"]
    for c in cases[30:400:3]:
        fr = O.frame_spectra(c["cov"])
        s, v = phasescore(c["cov"], engine)
        assert abs(s - float.fromhex(c["score"])) <= SCORE_TOL
        if not O.is_frame_tie(fr):
            assert v == c["valid"]
    rng = np.random.default_rng(3)
    for _ in range(40):   # float profiles, as the metagene step produces
        vals = [x if rng.random() < 0.8 else 0.0 for x in rng.gamma(0.7, 1.0, int(rng.integers(3, 700))).tolist()]
        s, v = phasescore(vals, engine)
        rs, rv = O.select_frame(O.frame_spectra(vals))
        assert abs(s - rs) <= SCORE_TOL and v == rv


def test_detect_orfs_end_to_end(engine, tmp_path):
    """detect_orfs() with explicit read lengths and offsets: TSV, WIG and bam summary against the
    files written by the reference's export_orf_coverages / export_wig (golden)."""
    from ribotricer_b200 import detect_orfs as D

    D._ENGINE = engine
    for case in load_golden("pipeline_cases.json.gz")["cases"]:
        reads = _read_columns(case)
        idx_path = tmp_path / f"{case['name']}_index.tsv"
        idx_path.write_text("\n".join(case["index"]) + "\n")
        offsets = {int(k): v for k, v in case["psite_offsets"].items()}
        for run in case["tsv"]:
            prm = run["params"]
            prefix = str(tmp_path / "out" / case["name"])
            D.detect_orfs(reads, str(idx_path), prefix, "forward", None, dict(offsets), prm["phase_score_cutoff"],
                          prm["min_valid_codons"], prm["min_reads_per_codon"], prm["min_valid_codons_ratio"],
                          prm["min_density_over_orf"], prm["report_all"], meta_min_reads=10 ** 9)
            compare_tsv(open(f"{prefix}_translating_ORFs.tsv").read(), run["text"], prm["phase_score_cutoff"],
                        what=case["name"] + ": ")
        # WIG: every P-site the reference wrote, except those shifted beyond the contig pad
        for tag, text in case["wig"].items():
            assert open(f"{prefix}_{tag}.wig").read() == text
        summary = open(f"{prefix}_bam_summary.txt").read()
        assert summary.startswith(f"summary:\n\ttotal_reads: {len(reads)}\n\tunique_mapped: {len(reads)}\n")


def test_inner_seams(engine, tmp_path):
    """split_bam -> merge_read_lengths -> orf_coverage, the reference's own seam order."""
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200.bam import split_bam
    from ribotricer_b200.index import ORF

    D._ENGINE = engine
    case = load_golden("pipeline_cases.json.gz")["cases"][1]
    reads = _read_columns(case)
    alignments, rlc = split_bam(reads, "forward", str(tmp_path / "s"), None, engine=engine)
    want = {}
    for length, _, _, _, n in case["alignments"]:
        want[length] = want.get(length, 0) + n
    assert dict(rlc) == want
    offsets = {int(k): v for k, v in case["psite_offsets"].items()}
    merged = D.merge_read_lengths(alignments, offsets)
    got = sorted([s, c, p, n] for s, t in merged.to_dict().items() for (c, p), n in t.items())
    assert got == [m for m in case["merged"]]
    for line, (oid, prof) in list(zip(case["index"][1:], case["profiles"]))[:25]:
        orf = ORF.from_string(line + "\n")
        assert orf.oid == oid
        assert D.orf_coverage(orf, merged) == prof
    # leader / trailer extension (detect_orfs.py:158-199), checked against the dict semantics
    table = merged.to_dict()
    orf = ORF.from_string(case["index"][3] + "\n")
    ext = D.orf_coverage(orf, merged, offset_5p=7, offset_3p=3)
    o5, o3 = (3, 7) if orf.strand == "-" else (7, 3)
    pos = list(range(orf.intervals[0][0] - o5, orf.intervals[0][0]))
    for s, e in orf.intervals:
        pos += list(range(s, e + 1))
    pos += list(range(orf.intervals[-1][1] + 1, orf.intervals[-1][1] + o3 + 1))
    ref = [table[orf.strand].get((orf.chrom, p), 0) for p in pos]
    assert ext == (ref[::-1] if orf.strand == "-" else ref)


def test_metagene_and_offset_inference(engine, tmp_path):
    """metagene_coverage + align_metagenes against the reference's own output (golden)."""
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import metagene as mg
    from ribotricer_b200.bam import split_bam

    D._ENGINE = engine
    case = load_golden("metagene_case.json.gz")["case"]
    reads = _read_columns(case, by_length=True)
    idx_path = tmp_path / "mg_index.tsv"
    idx_path.write_text("\n".join(case["index"]) + "\n")
    prefix = str(tmp_path / "mg")
    annotated, _ = D.parse_ribotricer_index(str(idx_path))
    assert len(annotated) == len(case["index"]) - 1
    alignments, rlc = split_bam(reads, "forward", prefix, None, engine=engine)
    assert {str(k): v for k, v in rlc.items()} == case["read_length_counts_in"]
    rlc = dict(sorted(rlc.items()))
    metagenes = mg.metagene_coverage(annotated, alignments, rlc, prefix, meta_min_reads=case["meta_min_reads"])
    assert list(rlc) == case["kept_lengths"]
    for length, ref in case["metagenes"].items():
        m = metagenes[int(length)]
        assert m[0][0] == ref["idx5"] and m[1][0] == ref["idx3"]
        assert np.allclose(m[0][1], ref["prof5"], rtol=0, atol=1e-9)
        assert np.allclose(m[1][1], ref["prof3"], rtol=0, atol=1e-9)
        assert abs(m[2] - ref["ps5"]) <= SCORE_TOL and m[3] == ref["v5"]
        assert abs(m[4] - ref["ps3"]) <= SCORE_TOL and m[5] == ref["v3"]
    offsets = mg.align_metagenes(metagenes, rlc, prefix, 0.428571428571, True)
    assert {str(k): v for k, v in offsets.items()} == case["psite_offsets"]
    assert open(f"{prefix}_psite_offsets.txt").read() == case["psite_offsets_txt"]
    # and the whole default-flag path: no read lengths, no offsets given
    D.detect_orfs(reads, str(idx_path), prefix, None, None, None, 0.428571428571, 5, 0, 0, 0.0, True,
                  meta_min_reads=case["meta_min_reads"])
    assert os.path.exists(f"{prefix}_translating_ORFs.tsv")
    assert open(f"{prefix}_protocol.txt").read().startswith("In total")
    rows = open(f"{prefix}_translating_ORFs.tsv").read().split("\n")
    assert len(rows) == len(case["index"]) + 1
    n_tr = sum(1 for r in rows[1:] if r.split("\t")[2:3] == ["translating"])
    assert n_tr > 0.5 * (len(case["index"]) - 1)


@pytest.mark.gpu
def test_split_bam_matches_reference(engine, tmp_path):
    """A1 end to end on the GPU path: native BAM decode -> K1, against what the UNMODIFIED reference
    split_bam (bam.py:33-153, run over oracle/pysam_restated.py) returned for the same BAM bytes."""
    import base64

    from ribotricer_b200 import bam as B
    from ribotricer_b200.detect_orfs import merge_read_lengths

    case = load_golden("split_bam_case.json.gz")["case"]
    path = tmp_path / "golden.bam"
    path.write_bytes(base64.b64decode(case["bam_b64"]))
    for run in case["runs"]:
        prefix = str(tmp_path / "out")
        alignments, rlc = B.split_bam(str(path), run["protocol"], prefix, run["read_lengths"], engine=engine)
        assert {str(k): int(v) for k, v in rlc.items()} == run["read_length_counts"]
        assert open(prefix + "_bam_summary.txt").read() == run["summary"]
        flat = sorted([int(length), strand, chrom, int(pos), int(n)] for length, by in alignments.to_dict().items()
                      for strand, ctr in by.items() for (chrom, pos), n in ctr.items())
        assert flat == run["alignments"], (run["protocol"], run["read_lengths"])
        # merged over lengths with offsets (detect_orfs.py:54-83) == the same merge of the reference's dict
        offsets = {int(k): 12 + (int(k) % 3) for k in run["read_length_counts"]}
        merged = merge_read_lengths(alignments, offsets).to_dict()
        want = {"+": {}, "-": {}}
        for length, strand, chrom, pos, n in run["alignments"]:
            key = (chrom, pos + offsets[length] if strand == "+" else pos - offsets[length])
            want[strand][key] = want[strand].get(key, 0) + n
        for strand in "+-":
            assert dict(merged.get(strand, {})) == want[strand]


@pytest.mark.gpu
def test_count_orfs_device_matches_reference(engine, tmp_path):
    """count_orfs on device results (coverage planes + status column, no profile text) against the table
    the reference's count_orfs (count_orfs.py:28-89) wrote from the corresponding TSV."""
    from helpers import case_to_arrays, merged_to_dense
    from oracle import c_oracle as CO
    from ribotricer_b200.count_orfs import count_orfs_device
    from ribotricer_b200.index import load_native_index

    pipe = {c["name"]: c for c in load_golden("pipeline_cases.json.gz")["cases"]}
    state = {}
    for c in load_golden("count_orfs_cases.json.gz")["cases"]:
        case = pipe[c["case"]]
        if c["case"] not in state:
            names, lens, _, _ = case_to_arrays(case)
            pad = 64
            base, plane = CO.genome_layout(lens, pad)
            dense, dropped = merged_to_dense(case, names, base, pad, plane)
            assert dropped == 0
            path = tmp_path / f"{c['case']}.tsv"
            path.write_text("\n".join(case["index"]) + "\n")
            idx = load_native_index(str(path))
            oid_row = {idx.oid(o): o for o in range(idx.n_orf)}
            state[c["case"]] = (names, lens, pad, dense, idx, oid_row)
        names, lens, pad, dense, idx, oid_row = state[c["case"]]
        engine.set_genome(names, lens, pad=pad)
        cov = engine.torch.from_numpy(dense).to(engine.device)
        run = case["tsv"][c["tsv"]]
        status = np.zeros(idx.n_orf, bool)
        for line in run["text"].splitlines()[1:]:
            f = line.split("\t")
            status[oid_row[f[0]]] = f[2] == "translating"
        out = tmp_path / "counts.tsv"
        count_orfs_device(engine, cov, idx, status, set(c["features"]), str(out), c["report_all"],
                          rows_written="all" if run["params"]["report_all"] else "translating")
        assert out.read_text() == c["text"], (c["case"], c["tsv"], c["features"], c["report_all"])


@pytest.mark.gpu
def test_learn_cutoff_matches_reference(engine, tmp_path, capsys):
    """determine_cutoff_tsv: same replicates (NumPy legacy generator, seed 42), medians from the GPU, same
    printed report as the reference's learn_cutoff.py:35-144; plus the median kernel against np.median."""
    from ribotricer_b200 import learn_cutoff as L

    pipe = {c["name"]: c for c in load_golden("pipeline_cases.json.gz")["cases"]}
    for c in load_golden("learn_cutoff_cases.json.gz")["cases"]:
        ribo, rna = [], []
        for k in range(c["n_files"]):
            a, b = tmp_path / f"ribo{k}.tsv", tmp_path / f"rna{k}.tsv"
            a.write_text(pipe[c["case"]]["tsv"][0]["text"])
            b.write_text(c["rna_texts"][k])
            ribo.append(str(a))
            rna.append(str(b))
        capsys.readouterr()
        L.determine_cutoff_tsv(ribo, rna, c["filter_by"], c["sampling_ratio"], c["reps"], engine=engine)
        assert capsys.readouterr().out == c["stdout"]
    rng = np.random.default_rng(9)
    for n, n_sel, reps in ((50, 1, 7), (1000, 333, 40), (4000, 2000, 9), (30000, 25001, 3)):   # the last one: global scratch
        vals = np.where(rng.random(n) < 0.3, 0.0, rng.random(n)) * rng.choice([1.0, -1.0, 1e-300, 1e300], n)
        idx = rng.integers(0, n, (n_sel, reps))
        got = L._bootstrap_medians(engine, vals, idx)
        assert np.array_equal(got, np.median(vals[idx], axis=0))


@pytest.mark.gpu
def test_default_flags_on_full_config1(engine, tmp_path):
    """detect_orfs() with NOTHING given (protocol, read lengths and P-site offsets all inferred) on the full
    BASELINE configs[0] library (100 k ORFs, 10 M reads).  The unmodified reference's infer_protocol says
    "forward" on this library (profiles/r2_protocol_heuristic.txt) and its metagene_coverage /
    align_metagenes recover the planted offsets {26-29: 12, 30-32: 13} (VERDICT round 1, measured with the
    reference); the inferred run must find the same and write the very TSV of the run with explicit offsets."""
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import synth
    from ribotricer_b200.bam import ReadColumns

    D._ENGINE = engine
    cfg = synth.config("C1")
    idx = synth.make_index(cfg)
    index_path = str(tmp_path / "index.tsv")
    idx.write_tsv(index_path)
    cols = synth.reads_to_numpy(synth.make_reads(cfg, idx, device=engine.device))
    reads = ReadColumns(idx.contig_names, idx.contig_len, cols, True)
    inferred, explicit = str(tmp_path / "inferred"), str(tmp_path / "explicit")
    D.detect_orfs(reads, index_path, inferred, None, None, None, 0.428571428571, 5, 0, 0, 0.0, False)
    assert open(f"{inferred}_protocol.txt").read().startswith("In total 20005 reads checked")
    lags = dict(line.strip().replace("lag of ", "").split(": ") for line in open(f"{inferred}_psite_offsets.txt").read().split("\n")[1:] if line)
    assert {int(k): int(v) + 12 for k, v in lags.items()} == synth.TRUE_OFFSETS
    D.detect_orfs(reads, index_path, explicit, "forward", None, dict(synth.TRUE_OFFSETS), 0.428571428571, 5, 0, 0, 0.0, False)
    a, b = open(f"{inferred}_translating_ORFs.tsv", "rb").read(), open(f"{explicit}_translating_ORFs.tsv", "rb").read()
    assert a == b
    assert a.count(b"\n") > 20_000      # header + the translating rows
    for tag in ("pos", "neg"):
        assert open(f"{inferred}_{tag}.wig", "rb").read() == open(f"{explicit}_{tag}.wig", "rb").read()


@pytest.mark.gpu
def test_genomic_shards_reproduce_the_single_run(engine, tmp_path):
    """The N-rank driver's per-rank work (multi_gpu.score_shard: sub-index of a genomic block in the compact layout,
    scored from the block's slice of the reads, one TSV part per run of rows) run for every block of a 3-way and a
    5-way plan on this one GPU: the joined parts must be the single run's TSV byte for byte."""
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import multi_gpu, synth
    from ribotricer_b200.bam import ReadColumns, split_bam
    from ribotricer_b200.engine import ScoreParams

    D._ENGINE = engine
    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    index_path = str(tmp_path / "index.tsv")
    idx.write_tsv(index_path)
    cols = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=300_000))
    reads = ReadColumns(idx.contig_names, idx.contig_len, cols, True)
    offsets = {28: 12, 29: 12, 30: 13, 31: 13}
    single = str(tmp_path / "single")
    D.detect_orfs(reads, index_path, single, "forward", None, dict(offsets), 0.428571428571, 5, 0, 0, 0.0, True)
    want = open(f"{single}_translating_ORFs.tsv", "rb").read()
    nidx = D.load_index(index_path)
    lut = {n: i for i, n in enumerate(engine.contig_names)}
    dc = nidx.device_columns(lut)
    for n in (3, 5):
        prefix = str(tmp_path / f"sharded{n}")
        plan = multi_gpu.shard_plan(dc["exon_ptr"], dc["exon_start"], dc["exon_end"], dc["orf_contig"], n)
        with open(f"{prefix}_translating_ORFs.tsv.header", "w") as fh:
            fh.write("\t".join(D.TSV_COLUMNS) + "\n")
        seen = 0
        for sh in plan:
            _, n_reads = multi_gpu.score_shard(engine, nidx, sh, reads, "forward", None, offsets, ScoreParams(), prefix, True)
            seen += n_reads
        assert seen < 2 * len(reads)          # the blocks' slices overlap at their borders only
        multi_gpu.join_runs(prefix, plan)
        assert open(f"{prefix}_translating_ORFs.tsv", "rb").read() == want, n


@pytest.mark.gpu
def test_two_rank_job_is_byte_identical(tmp_path):
    """tests/multi_gpu_check.py under torchrun on 2 GPUs (skipped on a single-GPU box)."""
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, MGPU_TMP=str(tmp_path), MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29641", os.path.join(root, "tests", "multi_gpu_check.py")],
                         capture_output=True, text=True, env=env, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert out.stdout.count("MULTI_GPU_OK") == 2


@pytest.mark.gpu
def test_batch_of_libraries_matches_single_runs(engine, tmp_path):
    """BASELINE configs[3] in small: eight libraries against one resident index through detect_orfs_batch (index and
    compact slot map set once, copy / kernels / text pipelined over two coverage buffers).  Every library's TSV and
    BAM summary must be the bytes detect_orfs() writes for that library alone.  Then the same on the genome of 1,900
    contigs of test_many_contigs.py (edge-length contigs, contigs with ORFs but no reads at either end and in the
    middle): a streamed library, one the packer refuses and an unsorted one."""
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import synth
    from ribotricer_b200.bam import ReadColumns, save_read_columns

    D._ENGINE = engine
    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    index_path = str(tmp_path / "index.tsv")
    idx.write_tsv(index_path)
    offsets = {27: 12, 28: 12, 29: 12, 30: 13, 31: 13}
    lengths = [27, 28, 29, 30, 31]
    libs = []
    for k in range(8):
        cols = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=40_000 + 15_000 * k, seed_offset=100 + k, sort=k != 5))
        path = str(tmp_path / f"lib{k}.npz")
        save_read_columns(path, ReadColumns(idx.contig_names, idx.contig_len, cols, k != 5))
        libs.append(path)
    params = (0.3, 3, 0, 0.1, 0.25)
    _batch_matches_single_runs(engine, tmp_path / "tiny", libs, index_path, lengths, offsets, params)

    import test_many_contigs as M

    names, lens = M.genome()
    index_path = str(tmp_path / "many_index.tsv")
    M.write_index(index_path)
    libs = []
    for k, kind in enumerate(("dense", "sparse", "dense")):
        cols = M.library(kind)
        if k == 2:                      # not coordinate-sorted: the column kernel after a clear
            cols = {c: v[np.random.default_rng(k).permutation(len(v))] for c, v in cols.items()}
        path = str(tmp_path / f"many{k}.npz")
        save_read_columns(path, ReadColumns(names, lens, cols, k != 2))
        libs.append(path)
    _batch_matches_single_runs(engine, tmp_path / "many", libs, index_path, None, M.OFFSETS, params)


def _batch_matches_single_runs(engine, out_dir, libs, index_path, lengths, offsets, params):
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200.batch import detect_orfs_batch

    singles = [str(out_dir / f"single{k}") for k in range(len(libs))]
    batched = [str(out_dir / "batch" / f"lib{k}") for k in range(len(libs))]
    for report_all in (False, True):
        for k in range(len(libs)):
            D.detect_orfs(libs[k], index_path, singles[k], "forward", lengths, dict(offsets), *params, report_all)
        done = detect_orfs_batch(libs, index_path, batched, "forward", lengths, offsets, *params, report_all=report_all,
                                 engine=engine)
        assert [k for k, _ in done] == list(range(len(libs)))
        for k in range(len(libs)):
            for suffix in ("_translating_ORFs.tsv", "_bam_summary.txt"):
                assert open(batched[k] + suffix, "rb").read() == open(singles[k] + suffix, "rb").read(), (k, suffix)
    assert engine.layout == "dense"
