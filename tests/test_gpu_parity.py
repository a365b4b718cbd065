"""Parity of the CUDA path (through the C ABI) with the oracle -- the tests proper.

Bar (BASELINE.json north_star): bit-exact P-site counts, read counts, lengths, valid codons and
ordering; phase score within 1e-9 absolute; status bit-exact except near the cutoff.  ORFs whose
best frame is an exact-arithmetic tie (hazard H1: the reference's valid_codons is then decided by
SciPy rounding noise) are excluded from the valid_codons/status comparison and counted.
"""
import numpy as np
import pytest

from helpers import (DEFAULT_PARAMS, SCORE_TOL, alignments_to_reads, case_to_arrays, compare_scores,
                     load_golden, merged_to_dense)

pytestmark = pytest.mark.gpu


def _oracle():
    from oracle import c_oracle
    return c_oracle


def _setup(engine, names, lens, idx, offsets, read_lengths=None, pad=64):
    engine.set_genome(names, lens, pad=pad)
    engine.set_length_table(offsets, read_lengths)
    engine.set_index(**idx)
    CO = _oracle()
    base, plane = CO.genome_layout(lens, pad)
    assert plane == engine.plane and (base == engine.contig_base).all()
    return base, plane


def test_phasescore_golden_profiles(engine):
    """Every golden phasescore profile as a one-exon ORF on its own stretch of a contig."""
    CO = _oracle()
    cases = load_golden("phasescore_cases.json.gz")["cases"]
    cases = [c for c in cases if len(c["cov"]) > 0]
    pad = 64
    starts, ends, pos = [], [], 1
    for c in cases:
        starts.append(pos)
        ends.append(pos + len(c["cov"]) - 1)
        pos += len(c["cov"]) + 7
    lens = np.array([pos + 10], np.int64)
    n = len(cases)
    for strand in (0, 1):
        idx = dict(exon_ptr=np.arange(n + 1, dtype=np.int64), exon_start=np.array(starts, np.int32),
                   exon_end=np.array(ends, np.int32), orf_contig=np.zeros(n, np.int32),
                   orf_strand=np.full(n, strand, np.uint8))
        base, plane = _setup(engine, ["c"], lens, idx, {28: 12}, pad=pad)
        cov = np.zeros(2 * plane, np.int32)
        for c, s in zip(cases, starts):
            v = np.array(c["cov"], np.int32)
            if strand == 1:
                v = v[::-1]
            cov[strand * plane + base[0] + pad + s: strand * plane + base[0] + pad + s + len(v)] = v
        d_cov = engine.torch.from_numpy(cov).to(engine.device)
        got = engine.score_host(d_cov, diagnostics=True)
        ref = CO.score(idx, cov, base, lens, pad, plane, DEFAULT_PARAMS)
        tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
        compare_scores(got, ref, tie)
        assert (got["frame_K"] == ref["frame_K"]).all()
        # and directly against the reference's own numbers
        ref_s = np.array([float.fromhex(c["score"]) for c in cases])
        ref_v = np.array([c["valid"] for c in cases])
        assert np.abs(got["score"] - ref_s).max() <= SCORE_TOL
        assert (got["valid"] == ref_v)[~tie].all()
        assert tie.sum() < 0.02 * n


def test_golden_pipeline_end_to_end(engine):
    """reads -> K1 -> K3 -> K4 against merge_read_lengths / orf_coverage / export_orf_coverages
    outputs of the reference (tests/golden/pipeline_cases.json.gz)."""
    CO = _oracle()
    for case in load_golden("pipeline_cases.json.gz")["cases"]:
        names, lens, idx, rows = case_to_arrays(case)
        offsets = {int(k): v for k, v in case["psite_offsets"].items()}
        pad = 64
        base, plane = _setup(engine, names, lens, idx, offsets, pad=pad)
        reads = alignments_to_reads(case, names)
        cov = engine.new_coverage()
        stats, len_counts = engine.bin_reads_host(cov, reads, "forward")
        ref_cov, dropped = merged_to_dense(case, names, base, pad, plane)
        assert (cov.cpu().numpy() == ref_cov).all(), case["name"]
        assert stats["oob"] == dropped and stats["valid"] == len(reads["ref_id"])
        got = engine.score_host(cov, diagnostics=True)
        ref = CO.score(idx, ref_cov, base, lens, pad, plane, DEFAULT_PARAMS)
        tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
        compare_scores(got, ref, tie, what=case["name"] + ": ")
        ptr, prof = engine.gather_profiles(cov, np.arange(len(rows)), got["length"])
        for i, (oid, p) in enumerate(case["profiles"]):
            assert prof[ptr[i]:ptr[i + 1]].tolist() == p, oid
        ref_rows = [r.split("\t") for r in case["tsv"][0]["text"].split("\n")[1:] if r]
        for i, r in enumerate(ref_rows):
            assert abs(got["score"][i] - float(r[3])) <= SCORE_TOL
            assert got["count"][i] == int(r[4]) and got["length"][i] == int(r[5])
            if not tie[i]:
                assert got["valid"][i] == int(r[6])


NEGATIVE_OFFSETS = {26: -1, 27: -2, 28: 12, 29: -5, 30: 0, 31: 300}   # what align_metagenes may return (lag + 12 < 0)


@pytest.mark.parametrize("protocol,read_lengths,sort,offsets", [
    ("forward", None, True, None), ("reverse", None, False, None), ("forward", [28, 29, 30], False, None),
    ("no", None, True, None), ("forward", None, True, NEGATIVE_OFFSETS), ("reverse", [26, 27, 29, 31], False, NEGATIVE_OFFSETS)])
def test_bin_psites_matches_oracle(engine, protocol, read_lengths, sort, offsets):
    CO = _oracle()
    from ribotricer_b200 import synth

    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=300_000, sort=sort))
    reads["ref_id"][:7] = -1
    reads["ref_id"][7:9] = 99
    reads["flag"][9:20] = 4
    reads["nh"][20:40] = 0
    reads["mapq"][20:30] = 0
    reads["mlen"][40:45] = 700      # beyond the shared-memory histogram
    reads["first"][45:50] = 0       # P-sites shifted off the contig start stay in the pad
    reads["last"][45:50] = 27
    offsets = offsets or {26: 12, 27: 12, 28: 12, 29: 12, 30: 13, 31: 13}
    pad = 16                        # small pad: some shifted P-sites fall outside -> oob
    base, plane = _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), offsets, read_lengths, pad=pad)
    code = {"forward": 0, "reverse": 1}.get(protocol, 2)
    lt = CO.make_len_table(offsets, read_lengths)
    ref_cov, ref_stats, ref_len = CO.bin_reads(reads, code, lt, base, idx.contig_len, pad, plane)
    cov = engine.new_coverage()
    stats, len_counts = engine.bin_reads_host(cov, reads, protocol, sorted_hint=sort)
    assert stats == ref_stats
    assert (len_counts == ref_len).all()
    assert (cov.cpu().numpy() == ref_cov).all()
    # device-pointer entry gives the same and accumulates
    dcols = engine.upload_reads(reads)
    st, lc = engine.new_bin_accumulators()
    engine.bin_reads_device(cov, dcols, protocol, st, lc, sorted_hint=sort)
    engine.torch.cuda.synchronize()
    assert (cov.cpu().numpy() == 2 * ref_cov).all()
    assert dict(zip(ref_stats.keys(), st.cpu().tolist())) == ref_stats


@pytest.mark.parametrize("name,scale,contig_scale", [("tiny", 1.0, 1.0), ("C1", 0.2, 1.0), ("C5", 0.004, 0.01),
                                                     ("C5", 0.1, 0.1)])      # 750 k ORFs, ten 100 k-codon ones, 310 Mb
def test_score_matches_oracle(engine, name, scale, contig_scale):
    CO = _oracle()
    from ribotricer_b200 import synth

    cfg = synth.config(name, scale, contig_scale)
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=min(cfg.n_reads, 2_000_000 if scale < 0.05 else 10_000_000),
                                                  device=engine.device if scale >= 0.05 else "cpu"))
    pad = 256
    base, plane = _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, pad=pad)
    cov = engine.new_coverage()
    engine.bin_reads_host(cov, reads, "forward", sorted_hint=True)
    ref_cov, _, _ = CO.bin_reads(reads, 0, CO.make_len_table(synth.TRUE_OFFSETS), base, idx.contig_len, pad, plane)
    assert (cov.cpu().numpy() == ref_cov).all()
    for params in (DEFAULT_PARAMS, [0.3, 3, 1, 0.1, 0.25]):
        from ribotricer_b200.engine import ScoreParams
        got = engine.score_host(cov, params=ScoreParams(*params), diagnostics=True)
        ref = CO.score(idx.as_dict(), ref_cov, base, idx.contig_len, pad, plane, params)
        tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
        n_tie, n_near = compare_scores(got, ref, tie, params, what=f"{name}: ")
        assert (got["frame_K"] == ref["frame_K"]).all()
        assert n_tie < 0.05 * idx.n_orf
    # sub-range scoring (what a shard does) returns the same rows
    lo, hi = idx.n_orf // 3, idx.n_orf // 3 + 1000
    part = engine.score_host(cov, lo, min(hi, idx.n_orf))
    full = engine.score_host(cov)
    for k in part:
        assert (part[k] == full[k][lo:hi]).all()
    # K4 on a sample of ORFs, both strands, long and short
    sel = np.unique(np.concatenate([np.arange(0, idx.n_orf, max(1, idx.n_orf // 300)),
                                    np.argsort(idx.orf_len)[-3:]]))
    ptr, prof = engine.gather_profiles(cov, sel, full["length"][sel])
    rptr, rprof = CO.gather_profiles(idx.as_dict(), sel, ref_cov, base, idx.contig_len, pad, plane)
    assert (ptr == rptr).all() and (prof == rprof).all()


def test_edge_cases(engine):
    """Empty / ragged inputs: unknown contig, unknown strand, exons hanging off the contig,
    length-1 and length-2 ORFs, 1-nt exons, lengths not a multiple of 3, tile-boundary lengths."""
    CO = _oracle()
    rng = np.random.default_rng(5)
    lens = np.array([5000, 300], np.int64)
    pad = 16
    orfs = [
        (0, 0, [(1, 1)]), (0, 1, [(10, 11)]), (0, 0, [(20, 22)]), (0, 1, [(30, 33)]),
        (0, 0, [(40, 40), (42, 42), (44, 44), (46, 60)]),            # 1-nt exons
        (-1, 0, [(1, 90)]), (0, 2, [(1, 90)]),                        # unknown contig / strand
        (1, 0, [(-30, 30)]), (1, 1, [(280, 340)]), (1, 0, [(-50, -20)]), (1, 1, [(400, 450)]),
        (0, 0, [(100, 100 + 767)]), (0, 1, [(100, 100 + 768)]), (0, 0, [(100, 100 + 769)]),
        (0, 1, [(100, 100 + 770)]), (0, 0, [(100, 100 + 771)]), (0, 0, [(100, 100 + 1535)]),
        (0, 1, [(100, 100 + 1537)]), (0, 0, [(1, 4999)]), (0, 1, [(2, 5000)]),
        (0, 0, [(s, s + 9) for s in range(1000, 1000 + 40 * 20, 20)]),   # 40 exons > 32-entry cache
        (0, 1, [(s, s + 6) for s in range(2000, 2000 + 70 * 9, 9)]),     # 70 exons
    ]
    ptr, st, en, contig, strand = [0], [], [], [], []
    for c, s, ivs in orfs:
        for a, b in ivs:
            st.append(a)
            en.append(b)
        ptr.append(len(st))
        contig.append(c)
        strand.append(s)
    idx = dict(exon_ptr=np.array(ptr, np.int64), exon_start=np.array(st, np.int32), exon_end=np.array(en, np.int32),
               orf_contig=np.array(contig, np.int32), orf_strand=np.array(strand, np.uint8))
    base, plane = _setup(engine, ["a", "b"], lens, idx, {28: 12}, pad=pad)
    cov = np.zeros(2 * plane, np.int32)
    for c in range(2):
        for s in range(2):
            lo = s * plane + base[c]
            span = lens[c] + 2 * pad + 1
            cov[lo:lo + span] = rng.poisson(0.4, span) * (rng.random(span) < 0.5)
    cov[base[0] + pad + 200] = 2_000_000_000     # near-int32-max counts: 64-bit sums, fp64 path
    cov[base[0] + pad + 201] = 2_000_000_000
    cov[base[0] + pad + 203] = 1_999_999_999
    d_cov = engine.torch.from_numpy(cov).to(engine.device)
    got = engine.score_host(d_cov, diagnostics=True)
    ref = CO.score(idx, cov, base, lens, pad, plane, DEFAULT_PARAMS)
    tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
    compare_scores(got, ref, tie)
    assert (got["frame_K"] == ref["frame_K"]).all()
    p, prof = engine.gather_profiles(d_cov, np.arange(len(orfs)), got["length"])
    rp, rprof = CO.gather_profiles(idx, np.arange(len(orfs)), cov, base, lens, pad, plane)
    assert (prof == rprof).all()
    # empty inputs
    engine.set_index(np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int32),
                     np.zeros(0, np.int32), np.zeros(0, np.uint8))
    assert len(engine.score_host(d_cov)["score"]) == 0
    empty = {k: np.zeros(0, dt) for k, dt in (("ref_id", np.int32), ("first", np.int32), ("last", np.int32),
             ("mlen", np.uint16), ("flag", np.uint16), ("mapq", np.uint8), ("nh", np.uint8))}
    stats, _ = engine.bin_reads_host(d_cov, empty, "forward")
    assert stats["total"] == 0


def test_errors_are_loud(engine):
    from ribotricer_b200 import _lib

    engine.set_genome(["a"], [1000], pad=8)
    engine.set_length_table({28: 12, 40: 30, 41: -7})   # offsets beyond the pad or below zero are offsets like any other
    with pytest.raises(_lib.RtError):   # ... up to RT_MAX_OFFSET
        engine.set_length_table({28: 12, 40: _lib.RT_MAX_OFFSET + 1})
    with pytest.raises(_lib.RtError):
        engine.set_length_table({28: -_lib.RT_MAX_OFFSET - 1})
    with pytest.raises(_lib.RtError):   # empty interval
        engine.set_index(np.array([0, 1], np.int64), np.array([10], np.int32), np.array([5], np.int32),
                         np.array([0], np.int32), np.array([0], np.uint8))
    engine.set_index(np.array([0, 1], np.int64), np.array([10], np.int32), np.array([50], np.int32),
                     np.array([0], np.int32), np.array([0], np.uint8))
    cov = engine.new_coverage()
    with pytest.raises(_lib.RtError):   # ORF range outside the index
        engine.score_host(cov, 0, 5)


def test_full_config1_against_oracle(engine):
    """BASELINE.json configs[0] at full size (yeast R64 scale: 100 k ORFs, 10 M reads): every ORF
    against the C oracle (seconds on the CPU)."""
    CO = _oracle()
    from ribotricer_b200 import synth

    cfg = synth.config("C1")
    idx = synth.make_index(cfg)
    dreads = synth.make_reads(cfg, idx, device=engine.device)
    reads = synth.reads_to_numpy(dreads)
    pad = 256
    base, plane = _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, pad=pad)
    cov = engine.new_coverage()
    stats, lens = engine.bin_reads_host(cov, reads, "forward", sorted_hint=True)
    ref_cov, ref_stats, ref_len = CO.bin_reads(reads, 0, CO.make_len_table(synth.TRUE_OFFSETS), base, idx.contig_len,
                                               pad, plane)
    assert stats == ref_stats and (lens == ref_len).all()
    assert (cov.cpu().numpy() == ref_cov).all()
    got = engine.score_host(cov, diagnostics=True)
    ref = CO.score(idx.as_dict(), ref_cov, base, idx.contig_len, pad, plane, DEFAULT_PARAMS)
    tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
    n_tie, n_near = compare_scores(got, ref, tie, what="C1: ")
    assert (got["frame_K"] == ref["frame_K"]).all()
    assert n_tie < 0.02 * idx.n_orf
    assert np.abs(got["score"] - ref["score"]).max() < 1e-11



def _oracle_on_subgenome(engine, idx, dreads, contigs, got, what):
    """The C oracle (bin + score, OpenMP) on the contigs ``contigs`` of a full-size configuration -- their reads,
    their ORFs, a coverage array of just those contigs on the host -- against the rows the GPU produced for the
    same ORFs while it scored the WHOLE configuration.  Returns the number of ORFs compared."""
    CO = _oracle()
    from ribotricer_b200 import synth

    t = engine.torch
    contigs = np.asarray(sorted(contigs), np.int64)
    remap = np.full(len(idx.contig_len), -1, np.int64)
    remap[contigs] = np.arange(len(contigs))
    on = np.isin(idx.orf_contig, contigs)
    rows = np.flatnonzero(on)
    from ribotricer_b200 import multi_gpu
    sub = multi_gpu.sub_index(idx.as_dict(), rows)
    sub["orf_contig"] = remap[sub["orf_contig"]].astype(np.int32)
    keep = t.isin(dreads["ref_id"], t.as_tensor(contigs, device=dreads["ref_id"].device).to(dreads["ref_id"].dtype))
    reads = synth.reads_to_numpy({k: v[keep] for k, v in dreads.items()})
    reads["ref_id"] = remap[reads["ref_id"]].astype(np.int32)
    sub_len = idx.contig_len[contigs]
    pad = engine.pad
    base, plane = CO.genome_layout(sub_len, pad)
    ref_cov, _, _ = CO.bin_reads(reads, 0, CO.make_len_table(synth.TRUE_OFFSETS), base, sub_len, pad, plane)
    ref = CO.score(sub, ref_cov, base, sub_len, pad, plane, DEFAULT_PARAMS)
    tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
    mine = {k: v[rows] for k, v in got.items()}
    n_tie, _ = compare_scores(mine, ref, tie, what=what)
    if "frame_K" in mine:
        assert (mine["frame_K"] == ref["frame_K"]).all(), f"{what}frame_K differs"
    assert n_tie < 0.02 * len(rows)
    return len(rows)


def test_full_config2_properties(engine):
    """BASELINE.json configs[1] at full size (2.5 M ORFs, 100 M reads, 24.7 GB coverage) through
    size-independent properties: un-binning returns the planes to zero; binning the library
    twice doubles every count and leaves score and valid codons unchanged (the phase score is
    scale invariant); shard results concatenate to the full result; a 20 k-ORF sample agrees
    with the oracle run on the gathered profiles."""
    CO = _oracle()
    from ribotricer_b200 import synth

    t = engine.torch
    cfg = synth.config("C2")
    idx = synth.make_index(cfg)
    dreads = synth.make_reads(cfg, idx, device=engine.device)
    engine.set_genome(idx.contig_names, idx.contig_len)
    engine.set_length_table(synth.TRUE_OFFSETS, None)
    engine.set_index(**idx.as_dict())
    cov = engine.new_coverage()
    st, lc = engine.new_bin_accumulators()
    engine.bin_reads_device(cov, dreads, "forward", st, lc, sorted_hint=True)
    one = engine.score_host(cov, min_codon=True, diagnostics=True)
    stats1 = st.cpu().numpy().copy()
    assert stats1[0] == cfg.n_reads and stats1[6] + stats1[1:6].sum() == cfg.n_reads
    assert int(cov.sum(dtype=t.int64).item()) == int(stats1[6] - stats1[7])      # every valid in-range read is one count
    engine.bin_reads_device(cov, dreads, "forward", st, lc, sorted_hint=True)
    two = engine.score_host(cov, min_codon=True)
    assert (two["count"] == 2 * one["count"]).all() and (two["min_codon"] == 2 * one["min_codon"]).all()
    assert (two["valid"] == one["valid"]).all() and (two["length"] == one["length"]).all()
    assert np.abs(two["score"] - one["score"]).max() <= 1e-12
    assert (two["status"] == one["status"])[np.abs(one["score"] - 0.428571428571) > 1e-9].all()
    engine.bin_reads_device(cov, dreads, "forward", st, lc, sorted_hint=True, weight=-1)
    engine.bin_reads_device(cov, dreads, "forward", st, lc, sorted_hint=True, weight=-1)
    assert int(cov.abs().max().item()) == 0 and int(st.abs().max().item()) == 0 and int(lc.abs().max().item()) == 0
    # shards
    engine.bin_reads_device(cov, dreads, "forward", st, lc, sorted_hint=True)
    bounds = engine.shard_bounds(8)
    assert bounds[0] == 0 and bounds[-1] == idx.n_orf and (np.diff(bounds) > 0).all()
    parts = [engine.score_host(cov, int(bounds[i]), int(bounds[i + 1]), min_codon=True, diagnostics=True) for i in range(8)]
    for k in one:
        assert np.array_equal(np.concatenate([p[k] for p in parts]), one[k], equal_nan=True), k
    # chr16 .. chrM (15 % of the genome, ~375 k ORFs) against the C oracle: every column of every one of those ORFs
    n_cmp = _oracle_on_subgenome(engine, idx, dreads, range(15, 25), one, "C2 chr16-chrM: ")
    assert n_cmp >= 200_000
    # sample against the oracle, through the gathered profiles (bit-exact integers, score 1e-9)
    rng = np.random.default_rng(11)
    sel = np.sort(np.concatenate([rng.choice(idx.n_orf, 20000, replace=False), np.argsort(idx.orf_len)[-20:]]))
    sel = np.unique(sel)
    ptr, prof = engine.gather_profiles(cov, sel, one["length"][sel])
    for j in range(0, len(sel), 7):
        o = sel[j]
        p = prof[ptr[j]:ptr[j + 1]]
        assert len(p) == idx.orf_len[o] and int(p.sum()) == one["count"][o]
        K, s3 = CO.frame_spectra(p)
        s, v = CO.phasescore(p)
        assert abs(s - one["score"][o]) <= SCORE_TOL
        if not CO.tie_mask(K[None, :], s3[None, :])[0]:
            assert v == one["valid"][o]



def test_full_config3_against_oracle(engine):
    """BASELINE.json configs[2] at full size (10 M candidate ORFs, 500 M reads) in the compact layout, as the
    benchmark runs it, and as two genomic blocks (what two ranks would hold): every ORF of chr13 .. chrM (a third of
    the genome, > 3 M ORFs) against the C oracle, the per-block results identical to the single run, and the
    size-independent books (every valid read inside the exon union is one count)."""
    import psutil

    from ribotricer_b200 import multi_gpu, synth

    if psutil.virtual_memory().available < 80 * 2 ** 30:
        pytest.skip("needs 80 GB of host memory for the oracle's copy of a third of the genome")
    t = engine.torch
    cfg = synth.config("C3")
    idx = synth.make_index(cfg)
    dreads = synth.make_reads(cfg, idx, device=engine.device)
    engine.set_genome(idx.contig_names, idx.contig_len)
    engine.set_length_table(synth.TRUE_OFFSETS, None)
    engine.set_index(**idx.as_dict())
    engine.set_layout("compact")
    cov = engine.new_coverage()
    st, lc = engine.new_bin_accumulators()
    engine.bin_reads_device(cov, dreads, "forward", st, lc, sorted_hint=True)
    got = engine.score_host(cov, diagnostics=True)
    assert len(got["score"]) == 10_000_000 and int(st[0].item()) == cfg.n_reads
    assert int(got["count"].sum()) >= int(cov.sum(dtype=t.int64).item())         # ORFs overlap: every count is seen at least once
    n_cmp = _oracle_on_subgenome(engine, idx, dreads, range(12, 25), got, "C3 chr13-chrM: ")
    assert n_cmp >= 3_000_000
    # the library as a record stream (2 M blocks), binned zone by zone over a buffer full of garbage: the same coverage
    dstream = engine.upload_stream(engine.stream_reads({k: v.cpu() for k, v in dreads.items()}))
    assert dstream["n"] == cfg.n_reads
    fresh = t.full_like(cov, -1)
    st2, lc2 = engine.new_bin_accumulators()
    engine.bin_stream_device(fresh, dstream, "forward", st2, lc2, fresh=True)
    assert t.equal(fresh, cov) and t.equal(st2, st) and t.equal(lc2, lc)
    del cov, fresh, dstream
    # two genomic blocks, each from its own slice of the reads
    plan = multi_gpu.shard_plan(idx.exon_ptr, idx.exon_start, idx.exon_end, idx.orf_contig, 2)
    reach = max(synth.TRUE_OFFSETS.values()) + int((dreads["last"].long() - dreads["first"].long()).max().item())
    key = dreads["ref_id"].long() * (1 << 32) + dreads["first"].long()
    for sh in plan:
        keep = t.zeros(len(key), dtype=t.bool, device=key.device)
        for c, lo, hi in sh.spans:
            a = int(t.searchsorted(key, t.tensor(c * (1 << 32) + max(lo - 1 - reach, 0), device=key.device)))
            b = int(t.searchsorted(key, t.tensor(c * (1 << 32) + hi + reach, device=key.device), right=True))
            keep[a:b] = True
        assert int(keep.sum().item()) < 0.55 * len(key)
        engine.set_index(**multi_gpu.sub_index(idx.as_dict(), sh.rows))
        engine.set_layout("compact")
        bcov = engine.new_coverage()
        st, lc = engine.new_bin_accumulators()
        engine.bin_reads_device(bcov, {k: v[keep].contiguous() for k, v in dreads.items()}, "forward", st, lc, sorted_hint=True)
        part = engine.score_host(bcov, diagnostics=True)
        for k in got:
            assert np.array_equal(part[k], got[k][sh.rows], equal_nan=True), k
        del bcov
    engine.set_layout("dense")


def test_sparse_clear(engine):
    """rt_track_touched / rt_clear_touched: after binning through both entry points the sparse
    clear must leave the planes exactly zero, and a second library must bin as if freshly cleared."""
    CO = _oracle()
    from ribotricer_b200 import synth

    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    pad = 64
    base, plane = _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, pad=pad)
    lt = CO.make_len_table(synth.TRUE_OFFSETS)
    cov = engine.new_coverage()
    engine.track_touched(True)
    try:
        for rep, (n, sort) in enumerate(((250_000, True), (90_000, False), (400_000, True))):
            reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=n, sort=sort, seed_offset=rep))
            ref_cov, ref_stats, _ = CO.bin_reads(reads, 0, lt, base, idx.contig_len, pad, plane)
            if rep % 2 == 0:
                stats, _ = engine.bin_reads_host(cov, reads, "forward", sorted_hint=sort)
                assert stats == ref_stats
            else:
                st, lc = engine.new_bin_accumulators()
                half = n // 2
                for part in (slice(0, half), slice(half, n)):     # two launches accumulate one list
                    d = engine.upload_reads({k: v[part] for k, v in reads.items()})
                    engine.bin_reads_device(cov, d, "forward", st, lc, sorted_hint=sort)
            assert (cov.cpu().numpy() == ref_cov).all()
            engine.clear_touched(cov)
            assert int(cov.abs().max().item()) == 0
    finally:
        engine.track_touched(False)


@pytest.mark.parametrize("name,scale,contig_scale,sort", [("tiny", 1.0, 1.0, True), ("C1", 0.2, 1.0, True),
                                                         ("C5", 0.004, 0.01, False)])
def test_compact_layout_matches_dense_and_oracle(engine, name, scale, contig_scale, sort):
    """RT_LAYOUT_COMPACT (coverage over the exon union only): stats and length counts are those of the
    dense planes, every compact slot holds the dense slot's count, and scores / gathered profiles are
    bit-identical to the dense layout's (and so to the oracle's)."""
    CO = _oracle()
    from ribotricer_b200 import synth
    from ribotricer_b200.engine import ScoreParams

    cfg = synth.config(name, scale, contig_scale)
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=min(cfg.n_reads, 1_000_000), sort=sort))
    pad = 256
    base, plane = _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, pad=pad)
    dense = engine.new_coverage()
    stats_d, len_d = engine.bin_reads_host(dense, reads, "forward", sorted_hint=sort)
    ref_d = engine.score_host(dense, diagnostics=True, min_codon=True)
    sel = np.unique(np.concatenate([np.arange(0, idx.n_orf, max(1, idx.n_orf // 200)), np.argsort(idx.orf_len)[-3:]]))
    ptr_d, prof_d = engine.gather_profiles(dense, sel, ref_d["length"][sel])
    engine.set_layout("compact")
    try:
        n_c = engine.coverage_elems()
        assert n_c < 2 * plane + 64
        cov = engine.new_coverage()
        assert cov.numel() == n_c
        stats_c, len_c = engine.bin_reads_host(cov, reads, "forward", sorted_hint=sort)
        assert stats_c == stats_d and (len_c == len_d).all()
        # every read that lands in the exon union is kept, nothing else
        ref_cov, _, _ = CO.bin_reads(reads, 0, CO.make_len_table(synth.TRUE_OFFSETS), base, idx.contig_len, pad, plane)
        member = np.zeros(2 * plane, bool)
        d = idx.as_dict()
        for o in range(idx.n_orf):
            c, s = int(d["orf_contig"][o]), int(d["orf_strand"][o])
            if c < 0 or s > 1:
                continue
            for e in range(d["exon_ptr"][o], d["exon_ptr"][o + 1]):
                a = max(int(d["exon_start"][e]), 1 - pad)
                b = min(int(d["exon_end"][e]), int(idx.contig_len[c]) + pad)
                if a <= b:
                    member[s * plane + base[c] + pad + a: s * plane + base[c] + pad + b + 1] = True
        got = cov.cpu().numpy()
        n_member = int(member.sum())
        assert n_member <= n_c <= n_member + 64
        assert (got[:n_member] == ref_cov[member]).all() and not got[n_member:].any()
        for params in (DEFAULT_PARAMS, [0.3, 3, 1, 0.1, 0.25]):
            one = engine.score_host(cov, params=ScoreParams(*params), diagnostics=True, min_codon=True)
            engine.set_layout("dense")
            two = engine.score_host(dense, params=ScoreParams(*params), diagnostics=True, min_codon=True)
            engine.set_layout("compact")
            for k in one:
                assert np.array_equal(one[k], two[k], equal_nan=True), k
        ptr_c, prof_c = engine.gather_profiles(cov, sel, ref_d["length"][sel])
        assert (ptr_c == ptr_d).all() and (prof_c == prof_d).all()
        # recycling: the sparse clear of a compact buffer is a memset
        engine.clear_touched(cov)
        assert int(cov.abs().max().item()) == 0
        st, lc = engine.new_bin_accumulators()
        engine.bin_reads_device(cov, engine.upload_reads(reads), "forward", st, lc, sorted_hint=sort)
        assert (cov.cpu().numpy() == got).all()
    finally:
        engine.set_layout("dense")


def test_compact_layout_needs_an_index(engine):
    from ribotricer_b200._lib import RtError

    engine.set_genome(["c"], [1000], pad=32)
    with pytest.raises(RtError, match="rt_set_index first"):
        engine.set_layout("compact")


def test_edge_cases_compact_layout(engine):
    """The ragged index of test_edge_cases (unknown contig / strand, exons hanging off the contig ends,
    1-nt exons, 70-exon ORFs, whole-contig ORFs) in the compact layout, with reads that land in the
    pads, off the contigs and on unknown references: K1 keeps exactly the P-sites some ORF reads,
    scores and profiles equal the dense layout's and the oracle's, and weight -1 undoes a library."""
    CO = _oracle()
    rng = np.random.default_rng(11)
    lens = np.array([5000, 300], np.int64)
    pad = 16
    orfs = [
        (0, 0, [(1, 1)]), (0, 1, [(10, 11)]), (0, 0, [(20, 22)]), (0, 1, [(30, 33)]),
        (0, 0, [(40, 40), (42, 42), (44, 44), (46, 60)]),
        (-1, 0, [(1, 90)]), (0, 2, [(1, 90)]),
        (1, 0, [(-30, 30)]), (1, 1, [(280, 340)]), (1, 0, [(-50, -20)]), (1, 1, [(400, 450)]),
        (0, 0, [(100, 100 + 767)]), (0, 1, [(100, 100 + 770)]), (0, 0, [(1, 4999)]), (0, 1, [(2, 5000)]),
        (0, 0, [(s, s + 9) for s in range(1000, 1000 + 40 * 20, 20)]),
        (0, 1, [(s, s + 6) for s in range(2000, 2000 + 70 * 9, 9)]),
        (1, 0, [(5, 7), (9, 9), (11, 40)]), (1, 1, [(250, 300)]),
    ]
    ptr, st, en, contig, strand = [0], [], [], [], []
    for c, s, ivs in orfs:
        for a, b in ivs:
            st.append(a)
            en.append(b)
        ptr.append(len(st))
        contig.append(c)
        strand.append(s)
    idx = dict(exon_ptr=np.array(ptr, np.int64), exon_start=np.array(st, np.int32), exon_end=np.array(en, np.int32),
               orf_contig=np.array(contig, np.int32), orf_strand=np.array(strand, np.uint8))
    offsets = {27: 11, 28: 12, 29: 12, 30: 13}
    base, plane = _setup(engine, ["a", "b"], lens, idx, offsets, pad=pad)
    n = 60_000
    ref_id = rng.choice([0, 0, 0, 1, 1, -1, 5], n).astype(np.int32)
    mlen = rng.integers(26, 32, n).astype(np.uint16)
    first = np.where(ref_id == 1, rng.integers(-40, 340, n), rng.integers(-40, 5040, n)).astype(np.int32)
    reads = dict(ref_id=ref_id, first=first, last=(first + mlen - 1).astype(np.int32), mlen=mlen,
                 flag=rng.choice([0, 16, 0, 16, 4, 256, 1024], n).astype(np.uint16),
                 mapq=rng.choice([255, 255, 3], n).astype(np.uint8), nh=rng.choice([0, 1, 1, 2], n).astype(np.uint8))
    lt = CO.make_len_table(offsets)
    for protocol, code in (("forward", 0), ("reverse", 1)):
        ref_cov, ref_stats, ref_len = CO.bin_reads(reads, code, lt, base, lens, pad, plane)
        ref = CO.score(idx, ref_cov, base, lens, pad, plane, DEFAULT_PARAMS)
        tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
        _, rprof = CO.gather_profiles(idx, np.arange(len(orfs)), ref_cov, base, lens, pad, plane)
        engine.set_layout("dense")
        dense = engine.new_coverage()
        stats_d, _ = engine.bin_reads_host(dense, reads, protocol)
        assert stats_d == ref_stats and (dense.cpu().numpy() == ref_cov).all()
        got_d = engine.score_host(dense, diagnostics=True, min_codon=True)
        engine.set_layout("compact")
        try:
            cov = engine.new_coverage()
            stats_c, len_c = engine.bin_reads_host(cov, reads, protocol)
            assert stats_c == ref_stats and (len_c == ref_len).all()
            got = engine.score_host(cov, diagnostics=True, min_codon=True)
            compare_scores(got, ref, tie)
            for k in got:
                assert np.array_equal(got[k], got_d[k], equal_nan=True), k
            _, prof = engine.gather_profiles(cov, np.arange(len(orfs)), got["length"])
            assert (prof == rprof).all()
            assert int(cov.sum().item()) <= int(ref_cov.sum()) and int(cov.sum().item()) > 0
            st, lc = engine.new_bin_accumulators()           # take the library out again
            engine.bin_reads_device(cov, engine.upload_reads(reads), protocol, st, lc, weight=-1)
            assert int(cov.abs().max().item()) == 0
        finally:
            engine.set_layout("dense")


@pytest.mark.parametrize("layout", ["dense", "compact"])
def test_packed_records_match_columns(engine, layout):
    """rt_pack_read_meta + rt_bin_reads_packed_host (11 B/read) against rt_bin_reads_host (18 B/read) on
    the same reads: stats, length totals and every coverage slot; reads of unknown references and all
    filter categories included; several launches (chunks) and runs that end inside a block."""
    from ribotricer_b200 import synth
    from ribotricer_b200._lib import RtError

    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=700_000))
    rng = np.random.default_rng(3)
    n = len(reads["ref_id"])
    reads["flag"] = np.where(rng.random(n) < 0.1, rng.choice([4, 256, 512, 1024, 2048, 272], n), reads["flag"]).astype(np.uint16)
    reads["nh"] = rng.choice([0, 1, 1, 1, 2], n).astype(np.uint8)
    reads["mapq"] = rng.choice([255, 255, 3, 0], n).astype(np.uint8)
    tail = slice(n - 5000, n)                      # a last run of reads without a reference, like unmapped BAM tails
    reads["ref_id"][tail] = -1
    _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, pad=64)
    engine.set_layout(layout)
    try:
        for protocol in ("forward", "reverse"):
            want = engine.new_coverage()
            stats_w, len_w = engine.bin_reads_host(want, reads, protocol, sorted_hint=True)
            packed = engine.pack_reads(reads)
            assert len(packed["run_ref"]) <= len(idx.contig_names) + 1 and packed["run_start"][-1] == n
            got = engine.new_coverage()
            stats_g, len_g = engine.bin_reads_packed_host(got, packed, protocol)
            assert stats_g == stats_w and (len_g == len_w).all()
            assert engine.torch.equal(got, want)
            dev = engine.new_coverage()                    # the same records resident on the device
            st, lc = engine.new_bin_accumulators()
            engine.bin_reads_packed_device(dev, engine.upload_packed(packed), protocol, st, lc)
            assert engine.torch.equal(dev, want) and dict(zip(stats_w.keys(), st.cpu().tolist())) == stats_w
        empty = engine.pack_reads({k: v[:0] for k, v in reads.items()})        # no reads at all
        stats_e, len_e = engine.bin_reads_packed_host(engine.new_coverage(), empty, "forward")
        assert stats_e["total"] == 0 and not len_e.any()
        # unsorted input has one run per read, far more than the table holds: refused, not mis-binned
        shuffled = {k: v[rng.permutation(n)] for k, v in reads.items()}
        with pytest.raises(RtError, match="not grouped by reference"):
            engine.pack_reads(shuffled)
        # ... unless the caller sizes the run table for it; results are still the same
        small = {k: v[:30_000] for k, v in shuffled.items()}
        packed = engine.pack_reads(small, max_runs=30_000)
        want = engine.new_coverage()
        stats_w, _ = engine.bin_reads_host(want, small, "forward")
        got = engine.new_coverage()
        stats_g, _ = engine.bin_reads_packed_host(got, packed, "forward")
        assert stats_g == stats_w and engine.torch.equal(got, want)
    finally:
        engine.set_layout("dense")


def test_random_many_exon_orfs_both_layouts(engine):
    """Randomised soak (fixed seed): ORFs of up to 200 exons of 1-40 nt with gaps of 0-7 nt, nested ORFs that
    share their tails, both strands, coverage densities from 0.02 to 30 per nt (table path, slow path,
    segmented phase B, one-value atoms at segment cuts) against the C oracle; the compact layout must return
    bit-identical columns."""
    CO = _oracle()
    from helpers import compare_scores as _cmp
    n_bad = 0
    rng = np.random.default_rng(12345)
    n_bad = 0
    for trial in range(16):
        L = int(rng.integers(3000, 20000))
        lens = np.array([L, int(rng.integers(500, 3000))], np.int64)
        pad = int(rng.choice([8, 16, 64]))
        orfs = []
        for _ in range(int(rng.integers(5, 40))):
            c = int(rng.integers(0, 2)); s = int(rng.integers(0, 2))
            n_ex = int(rng.choice([1, 2, 5, 30, 60, 120, 200]))
            pos = int(rng.integers(1, max(2, lens[c] // 3)))
            ivs = []
            for _ in range(n_ex):
                ln = int(rng.choice([1, 1, 2, 3, 5, 9, 40]))
                if pos + ln - 1 > lens[c] + pad - 1:
                    break
                ivs.append((pos, pos + ln - 1))
                pos += ln + int(rng.choice([0, 0, 1, 2, 7]))   # gap 0 = adjacent exons (separate entries)
            if not ivs:
                continue
            orfs.append((c, s, ivs))
            for k in range(int(rng.integers(0, 3))):            # nested ORFs sharing the tail
                cut = int(rng.integers(0, len(ivs)))
                a, b = ivs[cut]
                a2 = int(rng.integers(a, b + 1))
                orfs.append((c, s, [(a2, b)] + ivs[cut + 1:]))
        ptr, st, en, contig, strand = [0], [], [], [], []
        for c, s, ivs in orfs:
            for a, b in ivs:
                st.append(a); en.append(b)
            ptr.append(len(st)); contig.append(c); strand.append(s)
        idx = dict(exon_ptr=np.array(ptr, np.int64), exon_start=np.array(st, np.int32), exon_end=np.array(en, np.int32),
                   orf_contig=np.array(contig, np.int32), orf_strand=np.array(strand, np.uint8))
        engine.set_genome(["a", "b"], lens, pad=pad)
        engine.set_length_table({28: min(12, pad)}, None)
        engine.set_index(**idx)
        base, plane = CO.genome_layout(lens, pad)
        cov = np.zeros(2 * plane, np.int32)
        dens = float(rng.choice([0.02, 0.3, 2.0, 30.0]))
        for c in range(2):
            for s in range(2):
                lo = s * plane + base[c]; span = lens[c] + 2 * pad + 1
                cov[lo:lo + span] = rng.poisson(dens, span) * (rng.random(span) < rng.choice([0.1, 0.5, 1.0]))
        d_cov = engine.torch.from_numpy(cov).to(engine.device)
        got = engine.score_host(d_cov, diagnostics=True, min_codon=True)
        ref = CO.score(idx, cov, base, lens, pad, plane, DEFAULT_PARAMS)
        tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
        try:
            _cmp(got, ref, tie)
            assert (got["frame_K"] == ref["frame_K"]).all()
            # compact layout through K1-free path: copy dense values of member slots
            engine.set_layout("compact")
            ccov = engine.new_coverage()
            member = np.zeros(2 * plane, bool)
            for o in range(len(contig)):
                for e in range(ptr[o], ptr[o + 1]):
                    a = max(st[e], 1 - pad); b = min(en[e], int(lens[contig[o]]) + pad)
                    if a <= b:
                        member[strand[o] * plane + base[contig[o]] + pad + a: strand[o] * plane + base[contig[o]] + pad + b + 1] = True
            ccov[:int(member.sum())] = engine.torch.from_numpy(cov[member]).to(engine.device)
            got_c = engine.score_host(ccov, diagnostics=True, min_codon=True)
            for k in got:
                assert np.array_equal(got[k], got_c[k], equal_nan=True), ("compact", k)
            engine.set_layout("dense")
        except AssertionError as exc:
            n_bad += 1
            print("trial", trial, "FAILED:", exc, "orfs", len(orfs), "max exons", max(len(i) for _, _, i in orfs))
            engine.set_layout("dense")
    assert n_bad == 0


def _stream_library(idx, n_reads, seed):
    """A coordinate-sorted library over the synthetic genome with everything the record stream has to code: spliced
    reads, reads longer than 255, long gaps, all filter categories, reads without NH, an unknown reference, an
    unmapped tail with junk positions."""
    from ribotricer_b200 import synth

    cfg = synth.config("tiny")
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=n_reads, sort=True, seed_offset=seed))
    rng = np.random.default_rng(seed)
    n = len(reads["ref_id"])
    first = reads["first"].astype(np.int64)
    mlen = reads["mlen"].astype(np.int64)
    mlen = np.where(rng.random(n) < 0.02, rng.choice([1, 150, 255, 256, 300, 700], n), mlen)
    extra = np.where(rng.random(n) < 0.2, rng.choice([1, 3, 85, 6_000, 70_000], n), 0)
    reads["mlen"] = mlen.astype(np.uint16)
    reads["last"] = (first + mlen - 1 + extra).astype(np.int32)
    flag = reads["flag"].astype(np.int64)
    flag = np.where(rng.random(n) < 0.1, flag | rng.choice([4, 256, 512, 1024, 2048, 0x704], n), flag)
    reads["flag"] = flag.astype(np.uint16)
    reads["nh"] = rng.choice([0, 1, 1, 1, 2, 255], n).astype(np.uint8)
    reads["mapq"] = rng.choice([255, 255, 3, 0], n).astype(np.uint8)
    junk = (flag & 0x704) != 0
    reads["first"] = np.where(junk & (rng.random(n) < 0.5), -1, reads["first"]).astype(np.int32)
    last_contig = int(reads["ref_id"].max())
    reads["ref_id"][reads["ref_id"] == last_contig] = 99          # sorted, but no such reference
    tail = slice(n - 3000, n)
    reads["ref_id"][tail] = -1
    reads["flag"][tail] |= 4
    return reads


@pytest.mark.parametrize("layout", ["dense", "compact"])
def test_record_stream_matches_oracle_and_columns(engine, layout):
    """rt_stream_pack + rt_bin_stream(_host) (4 B/read delta-coded records, cascade on the device) against the C
    oracle's split_bam + merge_read_lengths and against rt_bin_reads on the columns the stream was made from: stats,
    length totals, every coverage slot; both protocols; weight -1 takes the library out again; a sparse library
    (gaps above 32,767 nt between neighbours) and the sorted_hint path of rt_bin_reads_host ride along."""
    CO = _oracle()
    from ribotricer_b200 import synth

    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    offsets = dict(synth.TRUE_OFFSETS)
    offsets[150] = 40
    offsets[300] = -7
    pad = 64
    base, plane = _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), offsets, None, pad=pad)
    lt = CO.make_len_table(offsets, None)
    engine.set_layout(layout)
    try:
        for n_reads, seed in ((400_000, 1), (900, 2)):
            reads = _stream_library(idx, n_reads, seed)
            stream = engine.stream_reads(reads, n_threads=3)
            assert stream["n"] == len(reads["ref_id"]) and stream["n_blocks"] >= 1
            for protocol, code in (("forward", 0), ("reverse", 1)):
                ref_cov, ref_stats, ref_len = CO.bin_reads(reads, code, lt, base, idx.contig_len, pad, plane)
                want = engine.new_coverage()
                st_w, lc_w = engine.new_bin_accumulators()
                engine.bin_reads_device(want, engine.upload_reads(reads), protocol, st_w, lc_w)
                stats_w = dict(zip(ref_stats.keys(), st_w.cpu().tolist()))
                assert stats_w == ref_stats and (lc_w.cpu().numpy() == ref_len).all()
                if layout == "dense":
                    assert (want.cpu().numpy() == ref_cov).all()
                got = engine.new_coverage()
                stats_g, len_g = engine.bin_stream_host(got, stream, protocol)
                assert stats_g == ref_stats and (len_g == ref_len).all()
                assert engine.torch.equal(got, want)
                hinted = engine.new_coverage()                     # the same through rt_bin_reads_host(sorted_hint=1)
                stats_h, len_h = engine.bin_reads_host(hinted, reads, protocol, sorted_hint=True)
                assert stats_h == ref_stats and (len_h == ref_len).all() and engine.torch.equal(hinted, want)
                dstream = engine.upload_stream(stream)             # resident stream, then taken out again
                st, lc = engine.new_bin_accumulators()
                engine.bin_stream_device(got, dstream, protocol, st, lc)
                assert engine.torch.equal(got, 2 * want)
                engine.bin_stream_device(got, dstream, protocol, st, lc, weight=-1)
                assert engine.torch.equal(got, want) and int(st.abs().sum().item()) == 0 and int(lc.abs().sum().item()) == 0
                if layout == "compact":      # rt_bin_stream_fresh: zones instead of a cleared buffer; any previous content goes
                    fresh = engine.torch.full_like(want, 12345)
                    st, lc = engine.new_bin_accumulators()
                    engine.bin_stream_device(fresh, dstream, protocol, st, lc, fresh=True)
                    assert engine.torch.equal(fresh, want)
                    assert dict(zip(ref_stats.keys(), st.cpu().tolist())) == ref_stats and (lc.cpu().numpy() == ref_len).all()
                    # the blocks of the stream in any order: the zone boundaries are made monotone, whatever then falls
                    # outside its block's zone goes through the spill list -- the coverage is the same
                    perm = np.random.default_rng(seed).permutation(stream["n_blocks"])
                    rec = np.asarray(stream["records"]).reshape(-1, 256)[perm].reshape(-1)
                    hdr = np.asarray(stream["hdr"]).reshape(-1, 4)[perm].reshape(-1)
                    shuffled = engine.upload_stream(dict(records=rec, hdr=hdr, n_blocks=stream["n_blocks"], n=stream["n"]))
                    fresh.fill_(-3)
                    st, lc = engine.new_bin_accumulators()
                    engine.bin_stream_device(fresh, shuffled, protocol, st, lc, fresh=True)
                    assert engine.torch.equal(fresh, want)
                    assert dict(zip(ref_stats.keys(), st.cpu().tolist())) == ref_stats
        empty = engine.stream_reads({k: v[:0] for k, v in reads.items()})
        stats_e, len_e = engine.bin_stream_host(engine.new_coverage(), empty, "forward")
        assert stats_e["total"] == 0 and not len_e.any()
        # protocol "no": reads are counted, nothing is stored (bam.py:105-131 has no branch for it)
        none = engine.new_coverage()
        stats_n, _ = engine.bin_stream_host(none, stream, "no")
        ref_cov, ref_stats, _ = CO.bin_reads(reads, 2, lt, base, idx.contig_len, pad, plane)
        assert stats_n == ref_stats and int(none.abs().max().item()) == 0
    finally:
        engine.set_layout("dense")


def test_zone_binning_soak(engine):
    """rt_bin_stream_fresh against rt_bin_stream into a cleared buffer (fixed seed): random length tables (negative
    offsets, unused and filtered lengths: the zone boundaries move with the smallest displacement), both protocols,
    piles of reads on few positions (empty zones, long spill lists), sparse and dense libraries, spliced and long reads."""
    from ribotricer_b200 import synth

    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, None, pad=64)
    engine.set_layout("compact")
    t = engine.torch
    rng = np.random.default_rng(11)
    binned = 0
    try:
        for trial in range(24):
            n = int(rng.choice([300, 5_000, 80_000, 300_000]))
            if trial % 2:
                reads = _stream_library(idx, n, trial)
            else:
                reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, n_reads=n, seed_offset=trial))
                if trial % 4 == 0:
                    keep = np.sort(rng.choice(len(reads["first"]), size=max(50, n // 50), replace=False))
                    reads = {k: np.repeat(v[keep], 50)[:n] for k, v in reads.items()}
            if trial % 3 == 1:          # a few reads that start before their predecessor: each opens a block of its own
                back = rng.random(len(reads["first"])) < 0.01
                shift = rng.integers(1, 40, len(back))
                reads["first"] = np.where(back, np.maximum(reads["first"] - shift, 0), reads["first"]).astype(np.int32)
                reads["last"] = np.maximum(reads["last"], reads["first"]).astype(np.int32)
            lengths = rng.choice(np.arange(24, 36), size=int(rng.integers(2, 10)), replace=False)
            offs = {int(length): int(rng.integers(-40, 60)) for length in lengths}
            rl = None if trial % 3 else [int(x) for x in rng.choice(np.arange(24, 36), size=8, replace=False)]
            engine.set_length_table(offs, rl)
            stream = engine.upload_stream(engine.stream_reads(reads))
            for protocol in ("forward", "reverse"):
                want = engine.new_coverage()
                st, lc = engine.new_bin_accumulators()
                engine.bin_stream_device(want, stream, protocol, st, lc)
                cols = engine.new_coverage()           # the column kernel on the reads the stream was made from
                st0, lc0 = engine.new_bin_accumulators()
                engine.bin_reads_device(cols, engine.upload_reads(reads), protocol, st0, lc0)
                assert t.equal(cols, want) and t.equal(st0, st) and t.equal(lc0, lc), (trial, protocol, "stream vs columns")
                got = t.full_like(want, 99)
                st2, lc2 = engine.new_bin_accumulators()
                engine.bin_stream_device(got, stream, protocol, st2, lc2, fresh=True)
                assert t.equal(got, want) and t.equal(st, st2) and t.equal(lc, lc2), (trial, protocol, offs, rl)
                binned += int(want.sum().item())
        assert binned > 100_000
    finally:
        engine.set_layout("dense")


def test_score_host_in_parts(engine, monkeypatch):
    """rt_score_host scores a large range in parts (own plan each) so that result copies overlap scoring: the columns
    are those of the single-range call, bit for bit."""
    from ribotricer_b200 import synth
    from ribotricer_b200.engine import ScoreParams

    cfg = synth.config("C1", 0.3)
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx))
    _setup(engine, idx.contig_names, idx.contig_len, idx.as_dict(), synth.TRUE_OFFSETS, None, pad=64)
    engine.set_layout("compact")
    try:
        cov = engine.new_coverage()
        engine.bin_reads_host(cov, reads, "forward", sorted_hint=True)
        monkeypatch.setenv("RT_SCORE_HOST_PARTS", "1")
        whole = engine.score_host(cov, params=ScoreParams(min_reads_per_codon=1), diagnostics=True)
        for parts in ("2", "5", "16"):
            monkeypatch.setenv("RT_SCORE_HOST_PARTS", parts)
            got = engine.score_host(cov, params=ScoreParams(min_reads_per_codon=1), diagnostics=True)
            for k in whole:
                assert np.array_equal(got[k], whole[k], equal_nan=True), (parts, k)
            sub = engine.score_host(cov, 1000, idx.n_orf - 777, params=ScoreParams(min_reads_per_codon=1), diagnostics=True)
            for k in whole:
                assert np.array_equal(sub[k], whole[k][1000:idx.n_orf - 777], equal_nan=True), (parts, k)
    finally:
        engine.set_layout("dense")
