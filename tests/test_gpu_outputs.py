"""The device entry points behind the output files other than the scoring columns -- the WIG compaction
(``rt_wig_count`` / ``rt_wig_fill``), the count-orfs interval sums (``rt_interval_sums``), the dense-to-compact copy
(``rt_compact_from_dense``), the window gathers on the auxiliary index and ``rt_phasescore_values`` -- against plain
references (NumPy, the C oracle, oracle/oracle_py.py) at tile edges, unaligned bases, extreme counts and genome scale.

Integers must match bit for bit, phase scores within SCORE_TOL.  The cases on the human contig table (C2) hold a
coverage buffer of about 25 GB and are skipped when the GPU has less than about 40 GB free."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from helpers import SCORE_TOL

pytestmark = pytest.mark.gpu

INT32_MAX = 2 ** 31 - 1
RT_ESTATE = -4                      # include/ribotricer_b200.h
WIG_TILE = 4096                     # slots per block of wig_count_kernel / wig_fill_kernel (256 threads x 16 slots)
C2_FREE_GB = 40
# 26 nt reads shift by -20 and 31 nt reads by +40: P-sites land in the pads below position 1 and past the contig end
C1_OFFSETS = {26: -20, 27: 12, 28: 12, 29: 12, 30: 13, 31: 40, 32: 13}


def _oracle():
    from oracle import c_oracle
    return c_oracle


def _need_free_gpu_memory(engine, gb=C2_FREE_GB):
    free, _ = engine.torch.cuda.mem_get_info(engine.device)
    if free < gb * 2 ** 30:
        pytest.skip(f"needs about {gb} GB of free GPU memory for coverage planes of the human genome")


def _release(engine):
    engine.torch.cuda.synchronize()
    engine.torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------- reference helpers
def _nonzero_ref(a):
    """What Engine.nonzero_slots returns for a host array: slots in order and their counts."""
    s = np.flatnonzero(a).astype(np.int64)
    return s, np.asarray(a[s], np.int32)


def _tile_pattern(n, rng, shift=0):
    """n counts whose 4,096-slot tiles take turns being empty, full, non-zero on the first slot only, on the last
    slot only, non-zero on both sides of every 16-slot thread edge, and sparse at random.  Counts include negative
    values and +-INT32_MAX (the kernels keep every count != 0)."""
    special = np.array([1, -1, 2, INT32_MAX, -INT32_MAX, -2 ** 31, 12345], np.int32)
    v = np.zeros(n, np.int32)
    for t0 in range(0, n, WIG_TILE):
        t1 = min(n, t0 + WIG_TILE)
        kind = (t0 // WIG_TILE + shift) % 6
        if kind == 1:
            v[t0:t1] = rng.choice(special, t1 - t0)
        elif kind == 2:
            v[t0] = -3
        elif kind == 3:
            v[t1 - 1] = INT32_MAX
        elif kind == 4:
            v[t0 + 15:t1:16] = -5
            v[t0 + 16:t1:16] = 5
        elif kind == 5:
            m = rng.random(t1 - t0) < 0.1
            v[t0:t1][m] = rng.choice(special, int(m.sum()))
    return v


def _interval_sums_ref(cov, off, length, group, n_group):
    """np.add.at of every interval's coverage sum (from a prefix sum) onto its group."""
    cs = np.zeros(len(cov) + 1, np.int64)
    np.cumsum(cov, dtype=np.int64, out=cs[1:])
    out = np.zeros(n_group, np.int64)
    off = np.asarray(off, np.int64)
    np.add.at(out, np.asarray(group, np.int64), cs[off + length] - cs[off])
    return out


def _sparse_interval_sums_ref(slots, vals, off, length, group, n_group):
    """The same over a buffer that is zero except at the sorted ``slots``."""
    cs = np.zeros(len(slots) + 1, np.int64)
    np.cumsum(vals, dtype=np.int64, out=cs[1:])
    off = np.asarray(off, np.int64)
    a = np.searchsorted(slots, off)
    b = np.searchsorted(slots, off + np.asarray(length, np.int64))
    out = np.zeros(n_group, np.int64)
    np.add.at(out, np.asarray(group, np.int64), cs[b] - cs[a])
    return out


def _member_mask(idx, lens, base, pad, plane):
    """The dense slots some ORF of the index reads, i.e. the compact layout's slots in order (as in
    test_compact_layout_matches_dense_and_oracle)."""
    member = np.zeros(2 * plane, bool)
    for o in range(len(idx["orf_contig"])):
        c, s = int(idx["orf_contig"][o]), int(idx["orf_strand"][o])
        if c < 0 or s > 1:
            continue
        for e in range(idx["exon_ptr"][o], idx["exon_ptr"][o + 1]):
            a = max(int(idx["exon_start"][e]), 1 - pad)
            b = min(int(idx["exon_end"][e]), int(lens[c]) + pad)
            if a <= b:
                member[s * plane + base[c] + pad + a: s * plane + base[c] + pad + b + 1] = True
    return member


def _member_count(idx, lens, base, pad, plane):
    """Number of slots of _member_mask without the mask (a union of intervals), for indexes of the human genome."""
    n_ex = np.diff(idx["exon_ptr"])
    c = np.repeat(np.asarray(idx["orf_contig"], np.int64), n_ex)
    s = np.repeat(np.asarray(idx["orf_strand"], np.int64), n_ex)
    ok = (c >= 0) & (s <= 1)
    cc = np.maximum(c, 0)
    a = np.maximum(np.asarray(idx["exon_start"], np.int64), 1 - pad)
    b = np.minimum(np.asarray(idx["exon_end"], np.int64), np.asarray(lens, np.int64)[cc] + pad)
    ok &= a <= b
    at = s * plane + np.asarray(base, np.int64)[cc] + pad
    lo, hi = (at + a)[ok], (at + b)[ok]
    if len(lo) == 0:
        return 0
    order = np.argsort(lo, kind="stable")
    lo, hi = lo[order], hi[order]
    reach = np.maximum.accumulate(hi)
    new = np.ones(len(lo), bool)
    new[1:] = lo[1:] > reach[:-1]
    first = np.flatnonzero(new)
    last = np.append(first[1:], len(lo)) - 1
    return int((reach[last] - lo[first] + 1).sum())


def _dense_to_merged(dense, names, base, pad, plane):
    """The reference's ``merged[strand][(chrom, pos)] -> count`` dict of dense planes (positions in the pads included)."""
    merged = {}
    for strand, tag in ((0, "+"), (1, "-")):
        slots = np.flatnonzero(dense[strand * plane:(strand + 1) * plane])
        c = np.searchsorted(base, slots, side="right") - 1
        pos = slots - base[c] - pad
        vals = dense[strand * plane + slots]
        merged[tag] = {(names[ci], p): v for ci, p, v in zip(c.tolist(), pos.tolist(), vals.tolist())}
    return merged


def _extended(orf, offset_5p, offset_3p):
    """The intervals orf_coverage reads (detect_orfs.py:158-199): the leader joins the first interval, the trailer
    the last, and on '-' the two offsets trade places."""
    o_lo, o_hi = (offset_3p, offset_5p) if orf.strand == "-" else (offset_5p, offset_3p)
    ivs = [list(iv) for iv in orf.intervals]
    ivs[0][0] -= o_lo
    ivs[-1][1] += o_hi
    return [tuple(iv) for iv in ivs]


def _count_orfs_ref(index, rows, genes, dense, base, lens, pad, plane):
    """count_orfs.py:59-89 restated over the selected ``rows``: per (gene_id, gene_name), the first count seen at a
    position wins (rows in order, each profile in transcript order), every position counted once.  Returns the text
    of the counts table."""
    CO = _oracle()
    rows = np.asarray(rows, np.int64)
    ptr, prof = CO.gather_profiles(index, rows, dense, base, lens, pad, plane)
    nt = np.diff(ptr)
    ep = index["exon_ptr"]
    n_ex = ep[rows + 1] - ep[rows]
    ex = np.repeat(ep[rows], n_ex) + (np.arange(int(n_ex.sum())) - np.repeat(np.cumsum(n_ex) - n_ex, n_ex))
    ex_len = (index["exon_end"][ex].astype(np.int64) - index["exon_start"][ex] + 1)
    at = np.repeat(np.cumsum(ex_len) - ex_len, ex_len)
    pos_up = np.repeat(index["exon_start"][ex].astype(np.int64), ex_len) + (np.arange(int(ex_len.sum())) - at)
    row_of = np.repeat(np.arange(len(rows)), nt)
    j = np.arange(len(prof)) - ptr[row_of]
    minus = index["orf_strand"][rows][row_of] == 1
    pos = pos_up[np.where(minus, ptr[row_of] + nt[row_of] - 1 - j, ptr[row_of] + j)]
    keys = sorted(set(genes[int(o)] for o in rows))
    lut = {k: i for i, k in enumerate(keys)}
    g = np.fromiter((lut[genes[int(o)]] for o in rows), np.int64, len(rows))[row_of]
    order = np.lexsort((np.arange(len(pos)), pos, g))
    gs, ps = g[order], pos[order]
    first = np.ones(len(gs), bool)
    first[1:] = (gs[1:] != gs[:-1]) | (ps[1:] != ps[:-1])
    total = np.zeros(len(keys), np.int64)
    np.add.at(total, gs[first], prof[order][first].astype(np.int64))
    length = np.bincount(gs[first], minlength=len(keys))
    text = "gene_id\tcount\tlength\n"
    for i, k in enumerate(keys):
        text += f"{k[0]}\t{int(total[i])}\t{int(length[i])}\n"
    return text


def _phasescore_ref(values):
    from oracle import oracle_py as O

    frames = O.frame_spectra(np.asarray(values, np.float64).tolist())
    return O.select_frame(frames), O.is_frame_tie(frames)


# ----------------------------------------------------------------------------------------------- device helpers
def _interval_sums(engine, cov, off, length, group, n_group, init=0):
    """rt_interval_sums called the way count_orfs.gene_union_counts calls it; returns (rc, sums)."""
    t = engine.torch
    dev = lambda a, dt: t.from_numpy(np.ascontiguousarray(a, dt)).to(engine.device)  # noqa: E731
    d_off, d_len, d_grp = dev(off, np.int64), dev(length, np.int32), dev(group, np.int32)
    d_sum = t.full((max(n_group, 1),), init, dtype=t.int64, device=engine.device)
    p = lambda x: C.c_void_p(x.data_ptr()) if x.numel() else None  # noqa: E731
    rc = engine.lib.rt_interval_sums(engine.ctx, C.c_void_p(cov.data_ptr()), len(off), p(d_off), p(d_len), p(d_grp),
                                     C.c_void_p(d_sum.data_ptr()), engine._stream())
    return rc, d_sum.cpu().numpy()[:n_group]


def _random_reads(rng, lens, n, refs=None):
    """Read columns over the contigs ``lens`` with every filter case and reads that hang off the contig ends."""
    refs = list(range(len(lens))) * 3 + [-1, len(lens) + 3] if refs is None else refs
    ref_id = rng.choice(refs, n).astype(np.int32)
    mlen = rng.integers(26, 32, n).astype(np.uint16)
    span = np.asarray(lens, np.int64)[np.clip(ref_id, 0, len(lens) - 1)]
    first = (rng.random(n) * (span + 80)).astype(np.int64) - 40
    return dict(ref_id=ref_id, first=first.astype(np.int32), last=(first + mlen - 1).astype(np.int32), mlen=mlen,
                flag=rng.choice([0, 16, 0, 16, 4, 256, 1024], n).astype(np.uint16),
                mapq=rng.choice([255, 255, 3], n).astype(np.uint8), nh=rng.choice([0, 1, 1, 2], n).astype(np.uint8))


def _check_compact_copy(engine, names, lens, idx, reads, offsets, pad, sorted_hint=False):
    """Bin ``reads`` into the dense planes, copy them into a compact buffer full of garbage (rt_compact_from_dense) and
    check the copy slot by slot against the dense slots the index reads, against binning the same reads straight into
    the compact layout, and through the scores."""
    CO = _oracle()
    t = engine.torch
    engine.set_genome(names, lens, pad=pad)
    engine.set_length_table(offsets)
    engine.set_index(**idx)
    base, plane = CO.genome_layout(lens, pad)
    assert plane == engine.plane and (base == engine.contig_base).all()
    dense = engine.new_coverage()
    engine.bin_reads_host(dense, reads, "forward", sorted_hint=sorted_hint)
    dense_np = dense.cpu().numpy()
    member = _member_mask(idx, lens, base, pad, plane)
    n_m = int(member.sum())
    assert _member_count(idx, lens, base, pad, plane) == n_m
    one = engine.score_host(dense, diagnostics=True, min_codon=True)
    engine.set_layout("compact")
    try:
        n_c = engine.coverage_elems()
        assert n_m <= n_c <= n_m + 64
        ccov = t.full((n_c,), -7, dtype=t.int32, device=engine.device)
        engine.compact_from_dense(dense, ccov)
        got = ccov.cpu().numpy()
        bad = np.flatnonzero(got[:n_m] != dense_np[member])
        assert len(bad) == 0, f"{len(bad)} compact slots differ from the dense slots, first at {bad[:5]}"
        assert (got[n_m:] == -7).all(), "the copy wrote behind the last atom"
        direct = engine.new_coverage()
        engine.bin_reads_host(direct, reads, "forward", sorted_hint=sorted_hint)
        assert not direct[n_m:].any()
        ccov[n_m:] = 0
        assert t.equal(ccov, direct)
        two = engine.score_host(ccov, diagnostics=True, min_codon=True)
        for k in one:
            assert np.array_equal(one[k], two[k], equal_nan=True), k
    finally:
        engine.set_layout("dense")
    return n_m


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


@pytest.fixture(scope="module")
def c1(engine):
    return _c1_library(engine.device)


def _c1_library(device):
    """The full C1 library (R64 contig table, 100 k ORFs, 10 M reads) plus reads at both ends of every contig, and the
    C oracle's dense P-site planes of it for C1_OFFSETS."""
    from ribotricer_b200 import synth
    from ribotricer_b200.const import DEFAULT_PAD

    CO = _oracle()
    cfg = synth.config("C1")
    idx = synth.make_index(cfg)
    cols = synth.reads_to_numpy(synth.make_reads(cfg, idx, device=device))
    ext = {k: [] for k in cols}
    for ci, L in enumerate(idx.contig_len.tolist()):
        for first, mlen, flag in ((0, 26, 0), (0, 31, 16), (L - 31, 31, 0), (L - 26, 26, 16)):
            for _ in range(3):
                for k, v in (("ref_id", ci), ("first", first), ("last", first + mlen - 1), ("mlen", mlen),
                             ("flag", flag), ("mapq", 255), ("nh", 1)):
                    ext[k].append(v)
    cols = {k: np.concatenate([v, np.array(ext[k], v.dtype)]) for k, v in cols.items()}
    order = np.lexsort((cols["first"], cols["ref_id"]))
    cols = {k: np.ascontiguousarray(v[order]) for k, v in cols.items()}
    pad = DEFAULT_PAD
    base, plane = CO.genome_layout(idx.contig_len, pad)
    dense, _, _ = CO.bin_reads(cols, 0, CO.make_len_table(C1_OFFSETS), base, idx.contig_len, pad, plane)
    return SimpleNamespace(idx=idx, cols=cols, pad=pad, base=base, plane=plane, dense=dense)


# --------------------------------------------------------------------------------- 1. ordered non-zero compaction
@pytest.mark.parametrize("lo", [0, 3, 4])
def test_nonzero_slots_at_tile_and_thread_edges(engine, lo):
    """Engine.nonzero_slots against np.flatnonzero for stretches of 0 .. 1 M slots around the 4,096-slot tile and the
    16-slot thread edges, on a 16-byte aligned base (int4 loads, lo = 0, 4) and an unaligned one (scalar loads, lo = 3).
    The slots around the stretch are non-zero: nothing outside [lo, lo + n) may show up."""
    t = engine.torch
    rng = np.random.default_rng(100 + lo)
    sizes = [0, 1, 15, 16, 17, 4095, 4096, 4097, 2 * WIG_TILE - 1, 2 * WIG_TILE + 1, 7 * WIG_TILE - 1,
             7 * WIG_TILE + 1, 1_000_003]
    for n in sizes:
        for shift in range(6 if n <= 8 * WIG_TILE else 1):
            v = _tile_pattern(n, rng, shift)
            buf = np.full(lo + n + 40, 9, np.int32)
            buf[lo:lo + n] = v
            d = t.from_numpy(buf).to(engine.device)
            assert (d.data_ptr() + 4 * lo) % 16 == (12 if lo == 3 else 0)
            slots, vals = engine.nonzero_slots(d, lo, n)
            ref_s, ref_v = _nonzero_ref(v)
            assert slots.dtype == np.int64 and vals.dtype == np.int32
            assert np.array_equal(slots, ref_s), (n, lo, shift)
            assert np.array_equal(vals, ref_v), (n, lo, shift)
    # a stretch with nothing in it, and one that is non-zero everywhere
    for fill in (0, -1):
        d = t.full((3 * WIG_TILE + 5,), fill, dtype=t.int32, device=engine.device)
        slots, vals = engine.nonzero_slots(d, lo, 3 * WIG_TILE)
        assert len(slots) == (0 if fill == 0 else 3 * WIG_TILE)
        assert np.array_equal(slots, np.arange(len(slots))) and (vals == fill).all()


def test_nonzero_slots_and_interval_sums_above_2_32(engine):
    """The dense planes of the human contig table (2 x 3.1 G slots): known slots around 2^31, 2^32, the plane ends and
    tile edges, found by nonzero_slots on each strand plane, on the whole buffer and from an unaligned base; then
    rt_interval_sums over stretches at offsets above 2^32, with counts near INT32_MAX."""
    from ribotricer_b200 import synth

    _need_free_gpu_memory(engine)
    t = engine.torch
    rng = np.random.default_rng(7)
    cfg = synth.config("C2")
    engine.set_genome([c[0] for c in cfg.contigs], [c[1] for c in cfg.contigs])
    plane = engine.plane
    assert plane > 2 ** 31 and 2 * plane > 2 ** 32
    cov = engine.new_coverage()
    try:
        edge = (2 ** 32 // WIG_TILE + 3) * WIG_TILE
        edge_m = plane + 1000 * WIG_TILE
        slots = np.unique(np.array([
            0, 1, 15, 16, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, edge - 1, edge, edge + 15, edge + 16,
            plane - 1, plane, plane + 1, edge_m - 1, edge_m, plane + 2 ** 31 - 1, plane + 2 ** 31, 2 * plane - 17,
            2 * plane - 16, 2 * plane - 1], np.int64))
        vals = rng.choice(np.array([1, -1, 3, INT32_MAX, -INT32_MAX, -2 ** 31], np.int32), len(slots))
        cov[t.from_numpy(slots).to(engine.device)] = t.from_numpy(vals).to(engine.device)
        for lo, n in ((0, plane), (plane, plane), (0, 2 * plane), (1, 2 * plane - 1)):
            got_s, got_v = engine.nonzero_slots(cov, lo, n)
            m = (slots >= lo) & (slots < lo + n)
            assert np.array_equal(got_s, slots[m] - lo), (lo, n)
            assert np.array_equal(got_v, vals[m]), (lo, n)
        # interval sums: a stretch across 2^32 and one at the end of the '-' plane, each with a run near INT32_MAX
        seg = [(slots, vals)]
        for start, n in ((2 ** 32 - 60_000, 120_000), (2 * plane - 150_000, 150_000)):
            v = rng.poisson(4.0, n).astype(np.int32)
            v[n // 3:n // 3 + 300] = INT32_MAX - rng.integers(0, 100, 300).astype(np.int32)
            cov[start:start + n] = t.from_numpy(v).to(engine.device)
            seg.append((np.arange(start, start + n, dtype=np.int64), v))
        s_all = np.concatenate([s for s, _ in seg])[::-1]
        v_all = np.concatenate([v for _, v in seg])[::-1]
        sp, first = np.unique(s_all, return_index=True)           # the last write of a slot wins
        sv = v_all[first]
        n_iv = 3000
        length = rng.integers(1, 100_001, n_iv)
        anchor = rng.choice(np.array([2 ** 32 - 60_000, 2 ** 32, 2 * plane - 150_000, plane + 2 ** 31 - 50_000,
                                      2 ** 32 - 1, edge - 40]), n_iv)
        off = np.minimum(anchor + rng.integers(0, 100_000, n_iv), 2 * plane - length)
        group = rng.integers(0, 16, n_iv)
        assert (off > 2 ** 32).sum() > n_iv // 2
        rc, got = _interval_sums(engine, cov, off, length, group, 16)
        assert rc == 0
        ref = _sparse_interval_sums_ref(sp, sv, off, length, group, 16)
        assert np.array_equal(got, ref)
        assert (np.abs(ref) > 2 ** 32).any()
    finally:
        del cov
        _release(engine)


# ------------------------------------------------------------------------------------------ 2. WIG files at C1 scale
def test_wig_files_full_config1(engine, tmp_path, c1):
    """split_bam -> merge_read_lengths -> export_wig on the full C1 library against oracle_py.export_wig fed with the C
    oracle's coverage: contigs in lexicographic order (not R64's header order), positions in the pads included; and
    MergedAlignments.nonzero() against the same planes."""
    from oracle import oracle_py as O
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200.bam import ReadColumns, split_bam

    idx, names = c1.idx, c1.idx.contig_names
    assert sorted(names) != list(names)
    reads = ReadColumns(names, idx.contig_len, c1.cols, True)
    alignments, _ = split_bam(reads, "forward", str(tmp_path / "s"), None, engine=engine)
    merged = D.merge_read_lengths(alignments, dict(C1_OFFSETS))
    assert engine.pad == c1.pad and engine.plane == c1.plane
    assert np.array_equal(merged.cov.cpu().numpy(), c1.dense)
    D.export_wig(merged, str(tmp_path / "gpu"))
    ref = _dense_to_merged(c1.dense, names, c1.base, c1.pad, c1.plane)
    lens = dict(zip(names, idx.contig_len.tolist()))
    for tag in "+-":
        assert any(p < 1 for _, p in ref[tag]) and any(p > lens[c] for c, p in ref[tag])
    O.export_wig(ref, str(tmp_path / "ref"))
    for tag in ("pos", "neg"):
        got = (tmp_path / f"gpu_{tag}.wig").read_bytes()
        want = (tmp_path / f"ref_{tag}.wig").read_bytes()
        assert got == want, tag
    s, c, p, n = merged.nonzero()
    parts = []
    for strand in (0, 1):
        slots, vals = _nonzero_ref(c1.dense[strand * c1.plane:(strand + 1) * c1.plane])
        ci = np.searchsorted(c1.base, slots, side="right") - 1
        parts.append((np.full(len(slots), strand), ci, slots - c1.base[ci] - c1.pad, vals))
    for got, want in zip((s, c, p, n), (np.concatenate(x) for x in zip(*parts))):
        assert np.array_equal(got, want)
    slots, vals = engine.nonzero_slots(merged.cov, 0, 2 * c1.plane)
    ref_s, ref_v = _nonzero_ref(c1.dense)
    assert np.array_equal(slots, ref_s) and np.array_equal(vals, ref_v)


# -------------------------------------------------------------------------------------------------- 3. interval sums
def test_interval_sums_against_prefix_sums(engine):
    """rt_interval_sums against np.add.at over a cumsum: random intervals of 1 .. 100,000 slots, thousands of intervals
    in one group, counts near INT32_MAX (one interval's sum and one group's sum above 2^32), no interval at all, and the
    refusal in the compact layout."""
    t = engine.torch
    rng = np.random.default_rng(21)
    engine.set_genome(["c"], [3_000_000], pad=16)
    n = engine.coverage_elems()
    cov = (rng.poisson(3.0, n) * (rng.random(n) < 0.6)).astype(np.int32)
    hot = 1_500_000
    cov[hot:hot + 5000] = INT32_MAX - rng.integers(0, 1000, 5000).astype(np.int32)
    d = t.from_numpy(cov).to(engine.device)
    cases = []
    m = 20_000                                                      # random intervals, 500 groups
    length = rng.integers(1, 100_001, m)
    cases.append((rng.integers(0, n - length + 1), length, rng.integers(0, 500, m), 500))
    m = 8000                                                        # nearly all of them in group 0
    length = rng.integers(1, 2000, m)
    cases.append((rng.integers(0, n - length + 1), length, np.where(rng.random(m) < 0.97, 0, rng.integers(1, 4, m)), 4))
    m = 3000                                                        # around the counts near INT32_MAX
    length = rng.integers(1, 6000, m)
    cases.append((hot - 500 + rng.integers(0, 5000, m), length, rng.integers(0, 3, m), 3))
    cases.append((np.array([hot]), np.array([5000]), np.array([0]), 1))
    for off, length, group, n_group in cases:
        rc, got = _interval_sums(engine, d, off, length, group, n_group)
        assert rc == 0
        ref = _interval_sums_ref(cov, off, length, group, n_group)
        assert np.array_equal(got, ref)
    assert ref[0] > 2 ** 32
    rc, got = _interval_sums(engine, d, np.zeros(0), np.zeros(0), np.zeros(0), 3, init=5)
    assert rc == 0 and (got == 5).all()
    engine.set_index(np.array([0, 1], np.int64), np.array([10], np.int32), np.array([50], np.int32),
                     np.array([0], np.int32), np.array([0], np.uint8))
    engine.set_layout("compact")
    try:
        rc, got = _interval_sums(engine, d, np.array([0]), np.array([10]), np.array([0]), 1, init=5)
        assert rc == RT_ESTATE and got[0] == 5
        assert b"dense planes" in engine.lib.rt_last_error(engine.ctx)
    finally:
        engine.set_layout("dense")


def test_count_orfs_device_full_config1(engine, tmp_path, c1):
    """count_orfs_device / gene_union_counts on the full C1 library against a NumPy restatement of count_orfs.py:59-89,
    with genes whose ORFs lie on two chromosomes or on both strands (the first value seen at a position wins)."""
    from ribotricer_b200.count_orfs import count_orfs_device
    from ribotricer_b200.index import load_native_index

    idx = c1.idx
    path = tmp_path / "index.tsv"
    idx.write_tsv(str(path))
    lines = path.read_text().split("\n")
    rows = [line.split("\t") for line in lines[1:] if line]
    rng = np.random.default_rng(5)
    # three annotated rows take the gene of row 0: one on another chromosome, one on the other strand, one on both
    c0, s0 = int(idx.orf_contig[0]), int(idx.orf_strand[0])
    ann = np.arange(idx.annotated_rows)
    other_chrom = ann[(idx.orf_contig[ann] != c0)][:1]
    other_strand = ann[(idx.orf_contig[ann] == c0) & (idx.orf_strand[ann] != s0)][:1]
    both = ann[(idx.orf_contig[ann] != c0) & (idx.orf_strand[ann] != s0)][1:2]
    mixed = np.concatenate([other_chrom, other_strand, both])
    assert len(np.unique(mixed)) == 3
    # and two genes share a name with different ids (keys are (gene_id, gene_name))
    for o in mixed:
        rows[o][4], rows[o][5] = rows[0][4], rows[0][5]
    rows[1][5] = rows[2][5]
    path.write_text("\n".join([lines[0]] + ["\t".join(r) for r in rows]) + "\n")
    nidx = load_native_index(str(path))
    assert nidx.n_orf == idx.n_orf
    genes = [(r[4], r[5]) for r in rows]
    types = np.array([r[1] for r in rows])
    features = {"annotated", "uORF", "novel"}
    engine.set_genome(idx.contig_names, idx.contig_len, pad=c1.pad)
    cov = engine.torch.from_numpy(c1.dense).to(engine.device)
    status = rng.random(idx.n_orf) < 0.5
    status[0] = status[mixed] = True
    for report_all, written in ((False, "translating"), (True, "all")):
        out = tmp_path / "counts.tsv"
        count_orfs_device(engine, cov, nidx, status, features, str(out), report_all, rows_written=written)
        sel = np.flatnonzero(np.isin(types, list(features)) & (status | report_all))
        want = _count_orfs_ref(idx.as_dict(), sel, genes, c1.dense, c1.base, idx.contig_len, c1.pad, c1.plane)
        assert out.read_text() == want, (report_all, written)
        assert want.count("\n") > 5000


# --------------------------------------------------------------------------------------- 4. dense-to-compact copy
RAGGED_ORFS = [            # the index of test_edge_cases_compact_layout
    (0, 0, [(1, 1)]), (0, 1, [(10, 11)]), (0, 0, [(20, 22)]), (0, 1, [(30, 33)]),
    (0, 0, [(40, 40), (42, 42), (44, 44), (46, 60)]),
    (-1, 0, [(1, 90)]), (0, 2, [(1, 90)]),
    (1, 0, [(-30, 30)]), (1, 1, [(280, 340)]), (1, 0, [(-50, -20)]), (1, 1, [(400, 450)]),
    (0, 0, [(100, 100 + 767)]), (0, 1, [(100, 100 + 770)]), (0, 0, [(1, 4999)]), (0, 1, [(2, 5000)]),
    (0, 0, [(s, s + 9) for s in range(1000, 1000 + 40 * 20, 20)]),
    (0, 1, [(s, s + 6) for s in range(2000, 2000 + 70 * 9, 9)]),
    (1, 0, [(5, 7), (9, 9), (11, 40)]), (1, 1, [(250, 300)]),
]


def test_compact_from_dense_ragged_and_random_indexes(engine):
    """rt_compact_from_dense slot by slot on the ragged index (exons off the contig ends, unknown contig and strand,
    1-nt exons, 70-exon ORFs) and on random many-exon indexes of nested ORFs."""
    rng = np.random.default_rng(41)
    lens = np.array([5000, 300], np.int64)
    reads = _random_reads(rng, lens, 60_000)
    offsets = {27: 11, 28: 12, 29: 12, 30: 13}
    assert _check_compact_copy(engine, ["a", "b"], lens, _csr(RAGGED_ORFS), reads, offsets, pad=16) > 0
    for trial in range(6):
        lens = np.array([int(rng.integers(3000, 20000)), int(rng.integers(500, 3000))], np.int64)
        pad = int(rng.choice([8, 16, 64]))
        orfs = []
        for _ in range(int(rng.integers(5, 40))):
            c, s = int(rng.integers(0, 2)), int(rng.integers(0, 2))
            pos = int(rng.integers(1 - pad, max(2, lens[c] // 3)))
            ivs = []
            for _ in range(int(rng.choice([1, 2, 5, 30, 60, 120, 200]))):
                ln = int(rng.choice([1, 1, 2, 3, 5, 9, 33, 40]))
                if pos + ln - 1 > lens[c] + pad + 5:
                    break
                ivs.append((pos, pos + ln - 1))
                pos += ln + int(rng.choice([0, 0, 1, 2, 7]))
            if not ivs:
                continue
            orfs.append((c, s, ivs))
            for _ in range(int(rng.integers(0, 3))):             # nested ORFs sharing the tail
                cut = int(rng.integers(0, len(ivs)))
                a, b = ivs[cut]
                orfs.append((c, s, [(int(rng.integers(a, b + 1)), b)] + ivs[cut + 1:]))
        reads = _random_reads(rng, lens, int(rng.integers(5_000, 200_000)), refs=[0, 0, 1])
        _check_compact_copy(engine, ["a", "b"], lens, _csr(orfs), reads, {28: min(12, pad), 29: -3}, pad=pad)


def test_compact_from_dense_full_config1(engine, c1):
    """rt_compact_from_dense on the full C1 index and library: slot by slot, against direct compact binning, and
    through the scores."""
    idx = c1.idx
    n_m = _check_compact_copy(engine, idx.contig_names, idx.contig_len, idx.as_dict(), c1.cols, C1_OFFSETS, c1.pad,
                              sorted_hint=True)
    assert n_m > 10_000_000


def test_compact_from_dense_full_config2(engine):
    """rt_compact_from_dense on the full C2 index and library (dense planes of 24.8 GB, slots above 2^32) against
    binning the same reads straight into the compact layout."""
    from ribotricer_b200 import synth

    _need_free_gpu_memory(engine)
    t = engine.torch
    cfg = synth.config("C2")
    idx = synth.make_index(cfg)
    dreads = synth.make_reads(cfg, idx, device=engine.device)
    engine.set_genome(idx.contig_names, idx.contig_len)
    engine.set_length_table(synth.TRUE_OFFSETS, None)
    engine.set_index(**idx.as_dict())
    n_m = _member_count(idx.as_dict(), idx.contig_len, engine.contig_base, engine.pad, engine.plane)
    dense = engine.new_coverage()
    try:
        st, lc = engine.new_bin_accumulators()
        engine.bin_reads_device(dense, dreads, "forward", st, lc, sorted_hint=True)
        engine.set_layout("compact")
        n_c = engine.coverage_elems()
        assert n_m <= n_c <= n_m + 64
        ccov = t.full((n_c,), -7, dtype=t.int32, device=engine.device)
        engine.compact_from_dense(dense, ccov)
        del dense
        direct = engine.new_coverage()
        st, lc = engine.new_bin_accumulators()
        engine.bin_reads_device(direct, dreads, "forward", st, lc, sorted_hint=True)
        assert t.equal(ccov[:n_m], direct[:n_m])
        assert bool((ccov[n_m:] == -7).all()) and not bool(direct[n_m:].any())
        assert int(direct.sum(dtype=t.int64).item()) > 0.5 * cfg.n_reads
    finally:
        engine.set_layout("dense")
        dense = ccov = direct = None
        _release(engine)


# ----------------------------------------------------------------------------- 5. window gathers on the aux index
def test_windows_and_extended_orfs_at_contig_ends(engine):
    """The metagene windows (_metagene_windows on the auxiliary index) and orf_coverage with leader / trailer offsets
    larger than the pad, for ORFs that start within 20 nt of position 1 or end within 20 nt of the contig end, on both
    strands: aux.gather_profiles against CO.gather_profiles and against oracle_py.orf_profile of the extended ORF."""
    from oracle import oracle_py as O
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import metagene as mg
    from ribotricer_b200.index import ORF

    CO = _oracle()
    rng = np.random.default_rng(31)
    names = ["chrB", "chrA", "chrC"]
    lens = np.array([5000, 3001, 777], np.int64)
    pad = 16
    engine.set_genome(names, lens, pad=pad)
    base, plane = CO.genome_layout(lens, pad)
    assert plane == engine.plane
    cov = (rng.integers(1, 50, 2 * plane) * (rng.random(2 * plane) < 0.7)).astype(np.int32)
    inside = np.zeros(2 * plane, bool)        # slots of positions 1 - pad .. len + pad
    for s in (0, 1):
        for c in range(len(lens)):
            inside[s * plane + base[c] + 1: s * plane + base[c] + lens[c] + 2 * pad + 1] = True
    cov[~inside] = 1_000_000                  # slots of no padded contig: a gather that strays there shows it
    d_cov = engine.torch.from_numpy(cov).to(engine.device)
    orfs = []
    for ci, L in enumerate(lens.tolist()):
        for strand in "+-":
            for k in range(40):
                kind = k % 3
                n_nt = int(rng.integers(1, 900 if L > 1000 else 300))
                if kind == 0:       # starts within 20 nt of position 1
                    a = 1 + int(rng.integers(0, 21))
                    b = min(L, a + n_nt)
                elif kind == 1:     # ends within 20 nt of the contig end
                    b = L - int(rng.integers(0, 21))
                    a = max(1, b - n_nt)
                else:               # both
                    a, b = 1 + int(rng.integers(0, 21)), L - int(rng.integers(0, 21))
                cuts = np.sort(rng.choice(np.arange(a, b + 1), min(b - a + 1, int(rng.integers(0, 4))), replace=False))
                ivs, s0 = [], a
                for x in cuts.tolist():
                    if x > s0:
                        ivs.append((s0, x - 1))
                        s0 = x + int(rng.integers(0, 30))
                if s0 <= b:
                    ivs.append((s0, b))
                orfs.append(ORF("annotated", f"T{len(orfs)}", "protein_coding", "G", "g", "protein_coding", names[ci],
                                strand, ivs, "ATG"))
    orfs.append(ORF("annotated", "Tx", "protein_coding", "G", "g", "protein_coding", "chrZ", "+", [(1, 90)], "ATG"))
    merged = _dense_to_merged(cov * inside, names, base, pad, plane)
    aux = D._aux_engine(engine)
    sel = np.arange(len(orfs), dtype=np.int64)
    for o5, o3, max_positions in ((40, 30, 600), (20, 0, 600), (300, 100, 50), (17, 17, 3000)):
        ptr, st, en, contig, strand, wlen = mg._metagene_windows(orfs, engine, max_positions, o5, o3)
        aux.set_index(ptr, st, en, contig, strand)
        got_ptr, got = aux.gather_profiles(d_cov, sel, wlen)
        window = dict(exon_ptr=ptr, exon_start=st, exon_end=en, orf_contig=contig, orf_strand=strand)
        ref_ptr, ref = CO.gather_profiles(window, sel, cov, base, lens, pad, plane)
        assert np.array_equal(got_ptr, ref_ptr) and np.array_equal(got, ref), (o5, o3, max_positions)
        for i, orf in enumerate(orfs):
            want = O.orf_profile(orf.chrom, orf.strand, _extended(orf, o5, o3), merged)[:max_positions]
            assert got[got_ptr[i]:got_ptr[i + 1]].tolist() == want, (o5, o3, max_positions, i)
    alignments = D.MergedAlignments(engine, d_cov)
    for i, orf in enumerate(orfs):
        o5, o3 = ((40, 30), (30, 0), (0, 25), (300, 300))[i % 4]
        want = O.orf_profile(orf.chrom, orf.strand, _extended(orf, o5, o3), merged)
        assert D.orf_coverage(orf, alignments, o5, o3) == want, (i, o5, o3)


# ------------------------------------------------------------------------------------------------ 6. phasescore
def _metagene_like(rng, n_rows, width):
    """Means over rows of a Ribo-seq-like count matrix, every row divided by its mean (metagene.py:140-155)."""
    frame = np.tile([1.0, 0.35, 0.25], width // 3 + 1)[:width]
    lam = rng.gamma(0.6, 2.0, (n_rows, 1)) * frame[None, :] * (rng.random((n_rows, width)) < 0.8)
    m = rng.poisson(lam).astype(np.float64)
    mean = m.mean(axis=1)
    m = m[mean > 0] / mean[mean > 0, None]
    return m.mean(axis=0)


def test_phasescore_values_against_oracle(engine):
    """rt_phasescore_values (one warp, 32 codons per 96-value stride) against oracle_py.select_frame(frame_spectra(v)):
    every length 0 .. 200, long profiles, exact zeros, uniform codons (counted in K, not in M; a frame of only uniform
    codons has a NaN coherence, which never wins), a zero frame between two non-zero ones (the K == 0 reset) and
    metagene-like profiles.  valid_codons must match outside the frame-tie class."""
    from ribotricer_b200.statistics import phasescore

    rng = np.random.default_rng(61)
    profiles = []
    for n in range(0, 201):
        profiles.append(np.where(rng.random(n) < 0.3, 0.0, rng.gamma(0.7, 1.0, n)))
        profiles.append(rng.poisson(0.4, n).astype(np.float64))
    for n in (10_000, 10_001, 100_000):
        profiles.append(np.where(rng.random(n) < 0.5, 0.0, rng.gamma(0.5, 3.0, n)))
        profiles.append(rng.poisson(0.05, n).astype(np.float64))
    for n in (0, 2, 3, 97, 300):
        profiles.append(np.zeros(n))
    for n in (3, 4, 5, 96, 97, 98, 290, 10_000):                 # only uniform codons in every frame
        profiles.append(np.full(n, 2.5))
        profiles.append(np.full(n, 1.0))
    for n in (30, 95, 301):                                       # uniform codons among others
        v = np.repeat(rng.gamma(1.0, 1.0, n // 3 + 1), 3)[:n]
        m = rng.random(len(v)) < 0.2
        v[m] = rng.gamma(1.0, 1.0, int(m.sum()))
        profiles.append(v)
        profiles.append(np.repeat(rng.gamma(1.0, 1.0, n // 3 + 1), 3)[:n])
    for k in range(1, 40, 3):                                     # frame 1 empty between non-zero frames 0 and 2
        for a, b in ((1.0, 1.0), (0.25, 3.5), (7.0, 0.0)):
            v = np.zeros(3 * k + 2)
            v[0], v[-1] = a, b
            profiles.append(v)
    for width in (600, 601, 602, 620):
        profiles.append(_metagene_like(rng, 300, width))
    n_tie = 0
    for i, v in enumerate(profiles):
        s, k = phasescore(v, engine)
        (rs, rk), tie = _phasescore_ref(v)
        assert abs(s - rs) <= SCORE_TOL, (i, len(v), s, rs)
        n_tie += tie
        if not tie:
            assert k == rk, (i, len(v), k, rk)
    assert n_tie < 0.05 * len(profiles)
