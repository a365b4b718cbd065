"""One engine (one rt_ctx) through many calls on the GPU: a second index, a new genome, an index that is refused, more
ORF ranges than the score-plan cache holds, command buffers kept from a larger call, an empty index, and the device
memory a closed engine gives back.  Every result is compared with what a fresh Engine computes from the same inputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def case():
    from ribotricer_b200 import synth

    cfg = synth.config("tiny")
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, device="cpu", n_reads=60_000))
    return idx, reads


def _csr(idx, rows):
    """The index rows `rows` (in that order) as set_index arguments."""
    ptr = np.asarray(idx.exon_ptr, np.int64)
    lens = ptr[np.asarray(rows) + 1] - ptr[rows]
    take = np.concatenate([np.arange(ptr[r], ptr[r + 1]) for r in rows]) if len(rows) else np.zeros(0, np.int64)
    return dict(exon_ptr=np.concatenate([[0], np.cumsum(lens)]).astype(np.int64),
                exon_start=np.asarray(idx.exon_start)[take], exon_end=np.asarray(idx.exon_end)[take],
                orf_contig=np.asarray(idx.orf_contig)[rows], orf_strand=np.asarray(idx.orf_strand)[rows])


def _refused(ix):
    """`ix` with the last interval of its last ORF ending before it starts: rt_set_index refuses it."""
    bad = {k: np.array(v, copy=True) for k, v in ix.items()}
    bad["exon_start"][-1], bad["exon_end"][-1] = bad["exon_end"][-1] + 5, bad["exon_start"][-1]
    return bad


def _engine(names, clen, ix=None):
    from ribotricer_b200 import synth
    from ribotricer_b200.engine import Engine

    eng = Engine(0)
    eng.set_genome(names, clen)
    eng.set_length_table(synth.TRUE_OFFSETS, None)
    if ix is not None:
        eng.set_index(**ix)
    return eng


def _score(eng, reads, layout, lo=0, hi=None):
    if layout == "compact":
        eng.set_layout("compact")
    else:
        eng.ensure_dense()
    cov = eng.new_coverage()
    eng.bin_reads_host(cov, reads, "forward", sorted_hint=True)
    return eng.score_host(cov, lo, hi, diagnostics=True)


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def _fresh(names, clen, ix, reads, ranges):
    """Dense, then compact columns of a fresh engine for every (lo, hi) of `ranges`, and its index sizes."""
    eng = _engine(names, clen, ix)
    try:
        out = {lay: [_score(eng, reads, lay, lo, hi) for lo, hi in ranges] for lay in ("dense", "compact")}
        sizes = (eng.score_bytes(), eng.total_nt(), eng.score_bytes(3, 11), eng.total_nt(3, 11), eng.shard_bounds(4))
        return out, sizes
    finally:
        eng.close()


def _check(eng, names, clen, ix, reads, ranges):
    want, sizes = _fresh(names, clen, ix, reads, ranges)
    for lay in ("dense", "compact"):
        for (lo, hi), w in zip(ranges, want[lay]):
            _same(_score(eng, reads, lay, lo, hi), w)
    got = (eng.score_bytes(), eng.total_nt(), eng.score_bytes(3, 11), eng.total_nt(3, 11), eng.shard_bounds(4))
    assert got[:4] == sizes[:4] and np.array_equal(got[4], sizes[4])


def test_reindex_one_engine(case):
    """Index A, then index B, then a new genome, then indexes that are refused: each state scores as a fresh engine."""
    from ribotricer_b200 import _lib

    idx, reads = case
    names, clen = idx.contig_names, np.asarray(idx.contig_len, np.int64)
    n = idx.n_orf
    a = idx.as_dict()
    b = _csr(idx, np.concatenate([np.arange(n - 1, 0, -3), np.arange(0, n, 7)]))
    nb = len(b["orf_contig"])
    eng = _engine(names, clen, a)
    try:
        _score(eng, reads, "compact")
        eng.set_index(**b)
        _check(eng, names, clen, b, reads, [(0, nb)])
        # another contig table: every slot moves, the index is encoded anew
        clen2 = clen + np.array([1000, 77, 3], np.int64)[:len(clen)]
        eng.set_genome(names, clen2)
        eng.set_index(**b)
        _check(eng, names, clen2, b, reads, [(0, nb)])
        # a refused index leaves B as it was: a range not scored yet, after a refused index with more ORFs than B ...
        with pytest.raises(_lib.RtError):
            eng.set_index(**_refused(a))
        _check(eng, names, clen2, b, reads, [(0, nb), (7, nb - 3)])
        # ... and after one with fewer
        with pytest.raises(_lib.RtError):
            eng.set_index(**_refused(_csr(idx, np.arange(0, n, 11))))
        _check(eng, names, clen2, b, reads, [(0, nb), (5, nb - 1), (nb // 2, nb)])
    finally:
        eng.close()


def test_plan_cache_eviction(case, monkeypatch):
    """More ORF ranges than the plan cache holds (24), then the first ones again: the same columns."""
    idx, reads = case
    n = idx.n_orf
    eng = _engine(idx.contig_names, np.asarray(idx.contig_len, np.int64), idx.as_dict())
    try:
        eng.set_layout("compact")
        cov = eng.new_coverage()
        eng.bin_reads_host(cov, reads, "forward", sorted_hint=True)
        ranges = [(k * 61, min(n, k * 61 + 400 + 13 * k)) for k in range(30)]
        monkeypatch.setenv("RT_SCORE_HOST_PARTS", "4")
        first_all = eng.score_host(cov, diagnostics=True)
        monkeypatch.delenv("RT_SCORE_HOST_PARTS")
        first = [eng.score_host(cov, lo, hi, diagnostics=True) for lo, hi in ranges]
        for (lo, hi), f in zip(ranges[:8], first[:8]):
            _same(eng.score_host(cov, lo, hi, diagnostics=True), f)
        monkeypatch.setenv("RT_SCORE_HOST_PARTS", "4")
        _same(eng.score_host(cov, diagnostics=True), first_all)
        for (lo, hi), f in zip(ranges[:3], first[:3]):
            _same(eng.score_host(cov, lo, hi, diagnostics=True), f)
    finally:
        eng.close()


def _orf_query(rng, n_tx, genome=300_000):
    from ribotricer_b200.prepare_orfs import codon_mask

    codes = rng.choice(5, genome, p=[0.24, 0.24, 0.24, 0.24, 0.04]).astype(np.uint8)
    ptr, starts, ends = [0], [], []
    for _ in range(n_tx):
        at = int(rng.integers(1, genome - 4000))
        for _ in range(int(rng.integers(1, 4))):
            m = int(rng.integers(30, 900))
            starts.append(at)
            ends.append(at + m - 1)
            at += m + int(rng.integers(1, 300))
        ptr.append(len(starts))
    cds = np.full((n_tx, 2), -1, np.int32)
    return dict(codes=codes, tx_base=np.zeros(n_tx, np.int64), exon_ptr=np.array(ptr, np.int64),
                exon_start=np.array(starts, np.int32), exon_end=np.array(ends, np.int32),
                tx_strand=rng.integers(0, 2, n_tx).astype(np.uint8), tx_cds=cds,
                start_mask=codon_mask(["ATG", "CTG"]), stop_mask=codon_mask(["TAA", "TAG", "TGA"]), min_orf_length=0,
                longest=False)


def _rows(rng, n, genome):
    ptr, starts, ends = [0], [], []
    for _ in range(n):
        at = int(rng.integers(1, genome - 4000))
        for _ in range(int(rng.integers(1, 4))):
            m = int(rng.integers(1, 700))
            starts.append(at)
            ends.append(at + m - 1)
            at += m + int(rng.integers(0, 200))
        ptr.append(len(starts))
    return np.array(ptr, np.int64), np.array(starts, np.int32), np.array(ends, np.int32)


def _seq_query(rng, n, genome=300_000):
    ptr, starts, ends = _rows(rng, n, genome)
    ids = [b"orf%d_%d" % (r, int(rng.integers(1 << 20))) for r in range(n)]
    return dict(exon_ptr=ptr, exon_start=starts, exon_end=ends, orf_contig=np.zeros(n, np.int32),
                orf_strand=rng.integers(0, 2, n).astype(np.uint8), contig_base=np.zeros(1, np.int64),
                contig_len=np.array([genome], np.int64),
                codes=rng.choice(5, genome, p=[0.24, 0.24, 0.24, 0.24, 0.04]).astype(np.uint8),
                id_off=np.concatenate([[0], np.cumsum([len(i) for i in ids])]).astype(np.int64),
                ids=np.frombuffer(b"".join(ids), np.uint8))


def _codon_query(rng, n_orf, n_sel, n_gene=40, genome=300_000):
    ptr, starts, ends = _rows(rng, n_orf, genome)
    lengths = np.add.reduceat(ends.astype(np.int64) - starts + 1, ptr[:-1])
    seq = rng.choice(np.frombuffer(b"ACGTN", np.uint8), int(lengths.sum()), p=[0.24, 0.24, 0.24, 0.24, 0.04])
    seq_off = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    row = rng.integers(0, n_orf, n_sel).astype(np.int64)
    texts = [("[" + ", ".join(map(str, rng.poisson(1.2, int(lengths[r])).tolist())) + "]").encode() for r in row]
    prof_len = np.array([len(t) for t in texts], np.int64)
    sel = dict(row=row, gene=rng.integers(0, n_gene, n_sel).astype(np.int32),
               gseq=rng.integers(0, 2 * n_gene, n_sel).astype(np.int32), prof_len=prof_len,
               prof_off=np.concatenate([[0], np.cumsum(prof_len)[:-1]]).astype(np.int64), seq_off=seq_off)
    return dict(sel=sel, tsv=np.frombuffer(b"".join(texts), np.uint8), seq=seq, exon_ptr=ptr, exon_start=starts,
                exon_end=ends, orf_strand=rng.integers(0, 2, n_orf).astype(np.uint8), n_gene=n_gene, n_gseq=2 * n_gene)


def _bytes(path):
    with open(path, "rb") as fh:
        return fh.read()


def test_command_buffers_kept_between_calls(case, tmp_path):
    """A large orf_search, then a small one, and a large orf_seq_write, then a small one in small chunks: the small
    calls reuse the larger buffers and return what a fresh engine returns."""
    idx, _ = case
    rng = np.random.default_rng(11)
    names, clen = idx.contig_names, np.asarray(idx.contig_len, np.int64)
    big_q, small_q = _orf_query(rng, 6000), _orf_query(rng, 40)
    big_s, small_s = _seq_query(rng, 8000), _seq_query(rng, 60)
    eng = _engine(names, clen)
    try:
        got = [eng.orf_search(**big_q), eng.orf_search(**small_q)]
        eng.orf_seq_write(tmp_path / "big.tsv", **big_s, protein=False)
        eng.orf_seq_write(tmp_path / "small.tsv", **small_s, protein=True, chunk_bytes=512)
    finally:
        eng.close()
    assert len(got[0]["row_tx"]) > 10 * len(got[1]["row_tx"]) > 0

    def fresh(call):
        eng = _engine(names, clen)
        try:
            return call(eng)
        finally:
            eng.close()

    _same(got[0], fresh(lambda e: e.orf_search(**big_q)))
    _same(got[1], fresh(lambda e: e.orf_search(**small_q)))
    fresh(lambda e: e.orf_seq_write(tmp_path / "big_fresh.tsv", **big_s, protein=False))
    fresh(lambda e: e.orf_seq_write(tmp_path / "small_fresh.tsv", **small_s, protein=True, chunk_bytes=512))
    assert _bytes(tmp_path / "big.tsv") == _bytes(tmp_path / "big_fresh.tsv")
    assert _bytes(tmp_path / "small.tsv") == _bytes(tmp_path / "small_fresh.tsv")
    assert _bytes(tmp_path / "small.tsv").count(b"\n") == 61


def test_empty_index_sizes(case):
    """No index yet, and an index dropped by a new genome: the byte and length sums of the empty range are 0."""
    idx, _ = case
    from ribotricer_b200.engine import Engine

    eng = Engine(0)
    try:
        assert eng.score_bytes(0, 0) == 0 and eng.total_nt(0, 0) == 0
        eng.set_genome(idx.contig_names, idx.contig_len)
        eng.set_index(**idx.as_dict())
        assert eng.score_bytes(0, idx.n_orf) > 0
        eng.set_genome(idx.contig_names, np.asarray(idx.contig_len, np.int64) + 5)
        assert eng.score_bytes(0, 0) == 0 and eng.total_nt(0, 0) == 0
    finally:
        eng.close()


def test_closed_engines_give_their_device_memory_back(case, tmp_path):
    """Five engines, one after another, each through every command with a ctx of several hundred MB (a 600 Mnt
    contig without ORFs, whose compact-layout map alone is 300 MB; host-column and record-stream binning of 4.8 M
    reads): after each is closed, the free device memory is what it was after the first.

    The check sees device memory only, in the 2 MiB pages the driver hands out: page-locked host buffers, and a
    buffer below 2 MiB that shares its page with others, can leak without changing the number."""
    import torch

    from ribotricer_b200 import learn_cutoff, synth
    from ribotricer_b200.engine import Engine

    idx, reads = case
    names = list(idx.contig_names) + ["empty"]
    clen = np.concatenate([np.asarray(idx.contig_len, np.int64), [600_000_000]])
    many = {k: np.repeat(v, 80) for k, v in reads.items()}        # stays coordinate-sorted
    rng = np.random.default_rng(5)
    orf_q, seq_q, codon_q = _orf_query(rng, 3000), _seq_query(rng, 3000), _codon_query(rng, 2000, 2500)
    count_q = {k: v for k, v in codon_q.items() if k not in ("seq", "n_gseq")}
    scores = rng.random(50_000)
    boot = rng.integers(0, len(scores), (30_000, 6)).astype(np.int64)   # 240 KB of keys per replicate: global scratch
    free = []
    for cycle in range(5):
        eng = Engine(0)
        eng.set_genome(names, clen)
        eng.set_length_table(synth.TRUE_OFFSETS, None)
        eng.set_index(**idx.as_dict())
        eng.set_layout("compact")
        cov = eng.new_coverage()
        s1, _ = eng.bin_reads_host(cov, many, "forward", sorted_hint=True)
        eng.clear_coverage(cov)
        s2, _ = eng.bin_reads_host(cov, many, "forward", sorted_hint=False)
        eng.clear_coverage(cov)
        s3, _ = eng.bin_stream_host(cov, eng.stream_reads(many), "forward")
        assert s1 == s2 == s3 and s1["valid"] > 0
        cols = eng.score_host(cov, diagnostics=True)
        rows = eng.orf_search(**orf_q)
        for protein in (False, True):
            eng.orf_seq_write(tmp_path / f"seq{cycle}.tsv", **seq_q, protein=protein, chunk_bytes=1 << 16)
        tabs = eng.codon_counts(**codon_q)
        counts = eng.orf_counts(**count_q)
        med = learn_cutoff._bootstrap_medians(eng, scores, boot)
        if cycle == 0:
            first = (cols, rows, tabs, med, counts)
        else:
            _same(cols, first[0])
            _same(rows, first[1])
            for x, y in zip(tabs, first[2]):
                assert np.array_equal(x, y)
            assert np.array_equal(med, first[3])
            for x, y in zip(counts, first[4]):
                assert np.array_equal(x, y)
        eng.close()
        del cov
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free.append(torch.cuda.mem_get_info()[0])
    assert first[2][2][4] == -1, "a profile of the codon query was refused"
    assert first[4][2][2] == -1, "a profile of the count query was refused"
    drift = [f - free[0] for f in free[1:]]
    assert all(abs(d) <= 4 << 20 for d in drift), drift
