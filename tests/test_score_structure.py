"""The two-phase scoring path (atom summaries, then families of ORFs composed from them) at its seams.

Phase A summarises every atom once: a stretch of coverage no ORF exon boundary cuts, chopped at 1,056 nt, read in
pieces of 33 values and passes of 32 pieces.  Phase B rebuilds every ORF from its atoms: the two windows across each
seam, suffix sums over a family of nested ORFs that share their stop, and group sums of 32 references added through
an accumulator for ORFs with more than 32 references.  Each case below is built by hand so that it holds the
structures it is about, re-derives those structures in plain Python and asserts that they are there, and then compares
both coverage layouts, with and without the per-frame minima, against the C oracle (integer columns exactly, score
within 1e-9) and against a high-precision restatement of the statistic (score within 1e-11).

Every value stays below 2^20 and every ORF below 3 * 2^20 nt, so no row takes the 64-bit fallback kernel.
"""
from __future__ import annotations

import math
from functools import lru_cache

import numpy as np
import pytest

from helpers import DEFAULT_PARAMS, SCORE_TOL, load_golden

ATOM_MAX = 1056          # kAtomMaxNt
PIECE = 33               # kPieceNt
PASS_PIECES = 32         # kPassPieces
GROUP = 32               # references per group of phase B
BIG = (1 << 20) - 1      # the largest value of the fast path
HP_TOL = 1e-11           # GPU vs the high-precision reference
MP_MAX_NT = 3000         # profiles up to 1,000 codons are judged by mpmath, longer ones by the fsum form


# ----------------------------------------------------------------------------------------------------------------
# case builder
class Case:
    """Contigs, ORFs given by contig / strand / 1-based inclusive exons, and dense coverage planes."""

    def __init__(self, contig_len, pad=16):
        self.lens = np.asarray(contig_len, np.int64)
        self.pad = int(pad)
        stride = (self.lens + 2 * self.pad + 1 + 31) // 32 * 32
        self.base = np.concatenate([[0], np.cumsum(stride)[:-1]]).astype(np.int64)
        self.plane = int(stride.sum())
        self.cov = np.zeros(2 * self.plane, np.int32)
        self.orfs = []

    def orf(self, contig, strand, exons):
        self.orfs.append((int(contig), int(strand), [(int(a), int(b)) for a, b in exons]))
        return len(self.orfs) - 1

    def slot(self, contig, strand, pos):
        return strand * self.plane + int(self.base[contig]) + self.pad + pos

    def put(self, contig, strand, pos, values):
        """Coverage of genomic positions pos, pos + 1, ... of one strand."""
        values = np.asarray(values, np.int64)
        assert 1 - self.pad <= pos and pos + len(values) - 1 <= self.lens[contig] + self.pad
        s = self.slot(contig, strand, pos)
        self.cov[s:s + len(values)] = values

    def put_profile(self, o, values):
        """Coverage along ORF o in PROFILE order (reversed on '-'); positions off the padded contig are skipped."""
        c, s, exons = self.orfs[o]
        pos = [p for a, b in exons for p in range(a, b + 1)]
        if s == 1:
            pos = pos[::-1]
        assert len(values) == len(pos)
        for p, v in zip(pos, values):
            if 1 - self.pad <= p <= self.lens[c] + self.pad:
                self.cov[self.slot(c, s, p)] = v

    def index(self):
        ptr, st, en = [0], [], []
        for _, _, exons in self.orfs:
            for a, b in exons:
                st.append(a)
                en.append(b)
            ptr.append(len(st))
        return dict(exon_ptr=np.array(ptr, np.int64), exon_start=np.array(st, np.int32),
                    exon_end=np.array(en, np.int32), orf_contig=np.array([o[0] for o in self.orfs], np.int32),
                    orf_strand=np.array([o[1] for o in self.orfs], np.uint8))

    # ---- the entries, atoms, references, passes and families the library derives (rt_set_index, build_atoms,
    # build_plan_host), restated in plain Python
    def entries(self, o):
        """(slot or None, length) pieces of ORF o in genomic order; None reads as zeros."""
        c, s, exons = self.orfs[o]
        out = []
        for a, b in exons:
            if not (0 <= c < len(self.lens) and s in (0, 1)):
                out.append((None, b - a + 1))
                continue
            lo, hi = 1 - self.pad, int(self.lens[c]) + self.pad
            x, y = max(a, lo), min(b, hi)
            if x > y:
                out.append((None, b - a + 1))
                continue
            if a < x:
                out.append((None, x - a))
            out.append((self.slot(c, s, x), y - x + 1))
            if y < b:
                out.append((None, b - y))
        return out

    def structure(self):
        if getattr(self, "_structure", None) is None:
            self._structure = _derive(self)
        return self._structure


def _derive(case):
    ents = [case.entries(o) for o in range(len(case.orfs))]
    pts = sorted({p for es in ents for off, ln in es if off is not None for p in (off, off + ln)})
    where = {p: i for i, p in enumerate(pts)}
    diff = np.zeros(len(pts) + 1, np.int64)
    for es in ents:
        for off, ln in es:
            if off is not None:
                diff[where[off]] += 1
                diff[where[off + ln]] -= 1
    atoms, begin, cover = [], [0] * (len(pts) + 1), 0
    for i in range(len(pts) - 1):
        cover += diff[i]
        begin[i] = len(atoms)
        if cover > 0:
            at = pts[i]
            while at < pts[i + 1]:
                piece = min(pts[i + 1] - at, ATOM_MAX)
                atoms.append((at, piece))
                at += piece
    if pts:
        begin[len(pts) - 1] = begin[len(pts)] = len(atoms)
    refs = []                                  # per ORF: [(atom id or None, length)] in profile order
    for o, es in enumerate(ents):
        rev = case.orfs[o][1] == 1
        r = []
        for off, ln in (es[::-1] if rev else es):
            if off is None:
                r.append((None, ln))
                continue
            ids = list(range(begin[where[off]], begin[where[off + ln]]))
            r += [(a, atoms[a][1]) for a in (ids[::-1] if rev else ids)]
        refs.append(r)
    # passes of the compact layout over the full range: consecutive atoms, at most 32 atoms and 32 pieces
    comp = np.concatenate([[0], np.cumsum([ln for _, ln in atoms])]).astype(np.int64)
    passes, i = [], 0
    while i < len(atoms):
        n = pieces = 0
        while i < len(atoms) and n < PASS_PIECES:
            np_ = -(-atoms[i][1] // PIECE)
            if pieces + np_ > PASS_PIECES:
                break
            pieces += np_
            n += 1
            i += 1
        first = i - n
        passes.append(dict(atoms=list(range(first, i)), pieces=pieces, r=int(comp[first] % 4)))
    # families: a child's reference list is a proper suffix of its parent's (<= 32 references), the child has at most
    # 31 references and its first one holds at least two values; longest ORFs first, one child per starting slot
    order = sorted(range(len(refs)), key=lambda o: -len(refs[o]))
    rev = [case.orfs[o][1] == 1 for o in range(len(refs))]
    parent = [-1] * len(refs)
    children = [[] for _ in refs]
    by_list = {}
    for o in range(len(refs)):
        if 1 <= len(refs[o]) <= 31:
            by_list.setdefault((rev[o], tuple(refs[o])), []).append(o)
    for o in order:
        cnt = len(refs[o])
        if parent[o] >= 0 or cnt < 2 or cnt > 32:
            continue
        for k in range(cnt - 1, 0, -1):
            for c in by_list.get((rev[o], tuple(refs[o][k:])), []):
                if c == o or parent[c] >= 0 or children[c] or refs[c][0][1] < 2:
                    continue
                parent[c] = o
                children[o].append((k, c))
                break
    return dict(atoms=atoms, refs=refs, passes=passes, parent=parent, children=children)


def family_sizes(st):
    """(slots of the family, number of children) of every family head with at least one child."""
    return [(len(st["refs"][o]), len(ch)) for o, ch in enumerate(st["children"]) if ch]


# ----------------------------------------------------------------------------------------------------------------
# the statistic in high precision (statistics.py:48-115 as orc_frame_spectra / orc_select state it)
def _windows(prof, f):
    p = np.asarray(prof, np.int64)
    n = (len(p) - f) // 3
    if n <= 0:
        return np.zeros((0, 3), np.int64)
    w = p[f:f + 3 * n].reshape(n, 3)
    return w[(w != 0).any(axis=1)]


def _frame_mp(w):
    """(K, s) of one frame: normalised triplet, detrend, DFT bin 1, Welch means, at 40 digits."""
    import mpmath as mp

    with mp.workdps(40):
        half, r3h = mp.mpf(1) / 2, mp.sqrt(3) / 2
        pxx = pre = pim = mp.mpf(0)
        for a, b, c in w.tolist():
            # |DFT bin 1|^2 of (a, b, c) is an integer over 4: its zero test is exact
            norm = mp.sqrt(mp.mpf((2 * a - b - c) ** 2 + 3 * (b - c) ** 2) / 4) if (a, b) != (c, c) else mp.mpf(1)
            x0, x1, x2 = a / norm, b / norm, c / norm
            m = (x0 + x1 + x2) / 3
            x0, x1, x2 = x0 - m, x1 - m, x2 - m
            xr, xi = x0 - half * (x1 + x2), r3h * (x2 - x1)
            pxx += xr * xr + xi * xi
            pre += xr
            pim -= xi
        K = len(w)
        if K == 0:
            return 0, math.nan
        pxx, pre, pim = pxx / K, pre / K, pim / K
        if pxx == 0:
            return K, math.nan
        return K, float((pre * pre + pim * pim) / pxx)


def _frame_fsum(w):
    """(K, s) of one frame from per-codon float64 unit vectors (A, B) / sqrt(A^2 + 3 B^2), summed exactly."""
    K = len(w)
    if K == 0:
        return 0, math.nan
    A = (2 * w[:, 0] - w[:, 1] - w[:, 2]).astype(np.float64)
    B = (w[:, 1] - w[:, 2]).astype(np.float64)
    keep = (A != 0) | (B != 0)
    n = np.sqrt(A[keep] ** 2 + 3 * B[keep] ** 2)
    M = int(keep.sum())
    if M == 0:
        return K, math.nan
    re, im = math.fsum((A[keep] / n).tolist()), math.fsum((B[keep] / n).tolist())
    return K, (re * re + 3 * im * im) / (K * M)


def _select(K3, s3):
    coh, valid = 0.0, -1
    for K, s in zip(K3, s3):
        if K == 0:
            coh, valid = 0.0, 0
            continue
        if s > coh:
            coh, valid = s, K
        if valid == -1:
            valid = K
    return math.sqrt(coh), valid


@lru_cache(maxsize=None)
def _reference_cached(key, mp):
    prof = np.frombuffer(key, np.int32)
    fr = [(_frame_mp if mp else _frame_fsum)(_windows(prof, f)) for f in range(3)]
    K3, s3 = [k for k, _ in fr], [s for _, s in fr]
    return _select(K3, s3) + (tuple(K3),)


def reference(prof, mp=None):
    """(score, valid_codons, K per frame) of one profile; mpmath for short profiles, the fsum form for long ones."""
    prof = np.ascontiguousarray(prof, np.int32)
    return _reference_cached(prof.tobytes(), len(prof) <= MP_MAX_NT if mp is None else mp)


# ----------------------------------------------------------------------------------------------------------------
# CPU checks of the builder and the reference
@pytest.fixture(scope="module")
def ps_cases():
    return load_golden("phasescore_cases.json.gz")["cases"]


def test_reference_matches_reference_tool(ps_cases):
    """Both forms of the high-precision statistic against the scores ribotricer itself wrote (mpmath on a sample)."""
    for i, c in enumerate(ps_cases):
        want = float.fromhex(c["score"])
        s_fs, _, _ = reference(c["cov"], mp=False)
        assert abs(s_fs - want) <= 1e-12, c["cov"]
        if i % 12 == 0:
            s_mp, _, _ = reference(c["cov"], mp=True)
            assert abs(s_mp - want) <= 1e-12, c["cov"]
            assert abs(s_fs - s_mp) <= 1e-14, c["cov"]


def test_reference_matches_c_oracle(built, ps_cases):
    from oracle import c_oracle as CO

    rng = np.random.default_rng(7)
    profiles = [c["cov"] for c in ps_cases[1::25]]
    profiles += [rng.poisson(lam, n) * (rng.random(n) < 0.6) for lam, n in ((0.3, 300), (3, 301), (20, 302), (400, 450))]
    profiles += [[0, 0, 14, 15, 16, 17, 16, 16, 16, 15, 15, 15, 0, 17, 0] * 7, [BIG, 0, 0, BIG, BIG, 0, 1, BIG, 2] * 11]
    for p in profiles:
        K, s3 = CO.frame_spectra(p)
        ref_s, _, ref_K = reference(p, mp=True)
        fs_s, _, fs_K = reference(p, mp=False)
        assert tuple(K) == ref_K == fs_K
        assert abs(CO.phasescore(p)[0] - ref_s) <= 1e-12
        assert abs(fs_s - ref_s) <= 1e-14


def test_builder_rederives_atoms_and_families():
    """The plain-Python derivation on a case small enough to check by hand."""
    c = Case([3000], pad=8)
    p = c.orf(0, 0, [(10, 20), (30, 40)])              # parent
    ch = c.orf(0, 0, [(14, 20), (30, 40)])             # child: first reference [14, 20] holds 7 values
    one = c.orf(0, 0, [(20, 20), (30, 40)])            # first reference holds 1 value: laid out alone
    lng = c.orf(0, 0, [(100, 100 + 2 * ATOM_MAX)])     # chopped into three atoms
    off = c.orf(0, 0, [(-20, -5), (1, 4)])             # starts off the padded contig
    st = c.structure()
    assert [ln for _, ln in st["refs"][p]] == [4, 6, 1, 11]
    assert [ln for _, ln in st["refs"][lng]] == [ATOM_MAX, ATOM_MAX, 1]
    assert st["refs"][off][:2] == [(None, 13), st["refs"][off][1]] and st["refs"][off][1][1] == 3
    assert st["parent"][ch] == p and st["parent"][one] == -1
    assert st["children"][p] == [(1, ch)]
    assert [ps["pieces"] for ps in st["passes"]] == [6, 32, 32, 1]       # slot order: the atoms of `off` come first


# ----------------------------------------------------------------------------------------------------------------
# GPU runs
@pytest.fixture
def eng(request):
    """The session's engine; the tests below skip cleanly on a machine without a CUDA device."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return request.getfixturevalue("engine")


def _oracle():
    from oracle import c_oracle as CO

    return CO


CONFIGS = [(False, 0), (True, 0), (False, 1), (True, 1)]      # (min_codon column, min_reads_per_codon)


def run_case(eng, case, params=None, configs=CONFIGS):
    """Score every ORF of `case` in both layouts and every config; compare with the oracle and the high-precision
    reference, and the compact layout bit for bit with the dense one.  Returns the columns of the first config."""
    from ribotricer_b200.engine import ScoreParams

    CO = _oracle()
    idx = case.index()
    eng.set_genome([f"c{i}" for i in range(len(case.lens))], case.lens, pad=case.pad)
    eng.set_index(**idx)
    assert eng.plane == case.plane and (eng.contig_base == case.base).all()
    d_dense = eng.torch.from_numpy(case.cov).to(eng.device)
    n = len(case.orfs)
    ptr, flat = CO.gather_profiles(idx, np.arange(n), case.cov, case.base, case.lens, case.pad, case.plane)
    hp = [reference(flat[ptr[o]:ptr[o + 1]]) for o in range(n)]
    hs, hK = np.array([h[0] for h in hp]), np.array([h[2] for h in hp]).reshape(n, 3)
    dense, worst_hp, worst_oracle = {}, 0.0, 0.0
    for layout in ("dense", "compact"):
        eng.set_layout(layout)
        if layout == "dense":
            d_cov = d_dense
        else:
            d_cov = eng.new_coverage()
            eng.compact_from_dense(d_dense, d_cov)
        for want_col, mrpc in configs:
            prm = list(params or DEFAULT_PARAMS)
            if params is None:
                prm[2] = mrpc
            got = eng.score_host(d_cov, params=ScoreParams(*prm), diagnostics=True, min_codon=want_col)
            ref = CO.score(idx, case.cov, case.base, case.lens, case.pad, case.plane, prm)
            what = f"[{layout}, min_codon={want_col}, params={prm}] "
            compare(got, ref, prm, what)
            assert ("min_codon" in got) == want_col
            assert (hK == ref["frame_K"]).all(), what + "reference K"
            d = np.abs(got["score"] - hs)
            worst = int(np.argmax(d))
            worst_hp = max(worst_hp, float(d.max()))
            worst_oracle = max(worst_oracle, float(np.abs(ref["score"] - hs).max()))
            assert d.max() <= HP_TOL, what + f"ORF {worst}: GPU {got['score'][worst]!r} vs reference {hs[worst]!r}"
            if layout == "dense":
                dense[want_col, mrpc] = got
            else:
                for k in got:
                    assert np.array_equal(got[k], dense[want_col, mrpc][k], equal_nan=True), what + k
    eng.set_layout("dense")
    print(f"\n{n} ORFs: largest |GPU - reference| {worst_hp:.3g}, largest |oracle - reference| {worst_oracle:.3g}")
    return dense[configs[0]]


def compare(got, ref, prm, what):
    CO = _oracle()
    for key in ("count", "length", "min_codon"):
        if key in got:
            assert (got[key] == ref[key]).all(), what + key
    assert (got["frame_K"] == ref["frame_K"]).all(), what + "frame_K"
    d = np.abs(got["score"] - ref["score"])
    assert not len(d) or d.max() <= SCORE_TOL, what + f"score differs from the oracle by {d.max()}"
    tie = CO.tie_mask(ref["frame_K"], ref["frame_s"])
    assert (got["valid"] == ref["valid"])[~tie].all(), what + "valid"
    near = np.abs(ref["score"] - prm[0]) <= SCORE_TOL
    assert (got["status"] == ref["status"])[~tie & ~near].all(), what + "status"


def _dense_random(rng, n, hi=40):
    return (rng.integers(0, hi, n) * (rng.random(n) < 0.7)).astype(np.int64)


# ---- phase A: atom lengths --------------------------------------------------------------------------------------
ATOM_LENGTHS = [1, 2, 3, 4, 5, 6, 32, 33, 34, 35, 36, 65, 66, 67, 98, 99, 100, 1054, 1055, 1056, 1057, 1058,
                2111, 2112, 2113, 3168, 3169]


def atom_length_case():
    rng = np.random.default_rng(1)
    total = sum(ATOM_LENGTHS) * 6 + 40 * len(ATOM_LENGTHS) * 6
    c = Case([total + 100], pad=16)
    pos = 20
    for L in ATOM_LENGTHS:
        for pattern in ("zero", "first", "second", "second_last", "last", "dense"):
            v = np.zeros(L, np.int64)
            nz = 1 + L % 20                                   # below and above the table's range of 16
            at = dict(first=0, second=1, second_last=L - 2, last=L - 1).get(pattern)
            if at is not None and 0 <= at < L:
                v[at] = nz
            if pattern == "dense":
                v = _dense_random(rng, L)
            for strand in (0, 1):                              # the two planes: same positions, separate atoms
                o = c.orf(0, strand, [(pos, pos + L - 1)])
                c.put_profile(o, v)
            pos += L + 40
    return c


@pytest.mark.gpu
def test_atom_lengths(eng):
    c = atom_length_case()
    st = c.structure()
    lens = {ln for _, ln in st["atoms"]}
    assert {1, 2, 3, 33, 34, 66, 67, 99, 100, 1055, ATOM_MAX} <= lens
    assert any(len(r) == 4 and r[-1][1] == 1 for r in st["refs"])      # 3169 = 3 * 1056 + 1
    run_case(eng, c)


# ---- phase A: pass packing and alignment ------------------------------------------------------------------------
def pass_case():
    rng = np.random.default_rng(2)
    c = Case([60000], pad=16)
    pos = 10

    def spliced(lengths, gap=3):
        nonlocal pos
        ex = []
        for ln in lengths:
            ex.append((pos, pos + ln - 1))
            pos += ln + gap
        pos += 50
        return ex

    # runs of adjacent atoms whose pieces total 31, 32 and 33, between full-length atoms
    for run in ([33] * 31, [33] * 32, [33] * 33, [34] * 15 + [33], [66] * 16, [34] * 15 + [33, 1], [67] * 11):
        c.orf(0, 0, spliced([ATOM_MAX] + run + [ATOM_MAX]))
        c.orf(0, 1, spliced(run[::-1]))
    # first slots at every residue mod 4 of the compact buffer: a full pass, then a short atom that shifts the next one
    for r in (1, 2, 3, 5, 6, 7):
        c.orf(0, 0, spliced([ATOM_MAX]))
        c.orf(0, 0, spliced([r]))
    # atoms of one and two values between long ones
    c.orf(0, 0, spliced([500, 1, 700, 2, ATOM_MAX, 1, 2, 1, 1000, 2, 2, 1, 33], gap=1))
    c.orf(0, 1, spliced([1, 2, 1, ATOM_MAX, 2, 1, ATOM_MAX, 1], gap=2))
    c.put(0, 0, 1, _dense_random(rng, pos))
    c.put(0, 1, 1, _dense_random(rng, pos, hi=20))
    return c


@pytest.mark.gpu
def test_pass_packing_and_alignment(eng):
    c = pass_case()
    passes = c.structure()["passes"]
    assert {p["r"] for p in passes} == {0, 1, 2, 3}
    assert any(p["pieces"] == 32 and len(p["atoms"]) > 1 for p in passes)
    assert any(p["pieces"] == 31 for p in passes)
    assert any(len(p["atoms"]) == 32 for p in passes)                 # cut by the atom limit
    assert any(p["pieces"] == 32 and len(p["atoms"]) == 17 for p in passes)   # 16 two-piece atoms and a one-value one
    run_case(eng, c)


# ---- table / slow path boundary ---------------------------------------------------------------------------------
def table_case():
    rng = np.random.default_rng(3)
    c = Case([40000], pad=16)
    pos = 10
    for trial in range(60):
        L = int(rng.integers(20, 400))
        vals = rng.choice([0, 0, 14, 15, 16, 17], L)
        for k in range(0, L - 2, 9):                          # uniform triplets on either side of 16
            vals[k:k + 3] = rng.choice([14, 15, 16, 17])
        strand = trial % 2
        if trial % 3 == 0:                                    # spliced: seam windows mix values of two atoms
            ex, p, left = [], pos, L
            while left:
                ln = min(left, int(rng.choice([1, 2, 4, 5, 31])))
                ex.append((p, p + ln - 1))
                p += ln + 2
                left -= ln
            pos = p + 10
        else:
            ex = [(pos, pos + L - 1)]
            pos += L + 10
        o = c.orf(0, strand, ex)
        c.put_profile(o, vals)
        if trial % 4 == 0 and min(ex[0][1] - ex[0][0], ex[-1][1] - ex[-1][0]) > 3:   # a nested ORF of the same stop
            c.orf(0, strand, [(ex[0][0] + 3, ex[0][1])] + ex[1:] if strand == 0 else ex[:-1] + [(ex[-1][0], ex[-1][1] - 3)])
    return c


@pytest.mark.gpu
def test_table_slow_boundary(eng):
    c = table_case()
    assert (c.cov == 16).any() and (c.cov == 15).any()
    run_case(eng, c)


# ---- largest fast-path values -----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_largest_fast_path_values(eng):
    rng = np.random.default_rng(4)
    c = Case([30000], pad=16)
    full = c.orf(0, 0, [(10, 10 + ATOM_MAX - 1)])
    c.put_profile(full, np.full(ATOM_MAX, BIG))
    multi = c.orf(0, 1, [(2000, 2000 + 4 * ATOM_MAX + 50)])
    c.put_profile(multi, np.full(4 * ATOM_MAX + 51, BIG))
    mixed = c.orf(0, 0, [(2000, 3999), (4100, 6300)])
    c.put_profile(mixed, rng.choice([0, 1, BIG, BIG - 1, 1 << 19], 4201))
    periodic = c.orf(0, 1, [(8000, 8000 + 4 * ATOM_MAX + 2)])
    c.put_profile(periodic, np.tile([BIG, 0, 0], 4 * ATOM_MAX // 3 + 1))
    child = c.orf(0, 0, [(3000, 3999), (4100, 6300)])
    st = c.structure()
    assert st["atoms"][st["refs"][full][0][0]][1] == ATOM_MAX
    assert ATOM_MAX * BIG > 2 ** 30 and c.cov.max() == BIG
    got = run_case(eng, c)
    assert got["count"][multi] > 2 ** 32 and got["count"][full] == ATOM_MAX * BIG
    assert st["parent"][child] == mixed


# ---- families ---------------------------------------------------------------------------------------------------
def family_case():
    rng = np.random.default_rng(5)
    c = Case([40000, 3000], pad=8)
    info = {}

    def family(strand, exons, starts, dup=False):
        """A parent and children that start at `starts` (offsets into its profile); returns the ids."""
        p = c.orf(0, strand, exons)
        ids = [p]
        pos = [q for a, b in exons for q in range(a, b + 1)]
        if strand == 1:
            pos = pos[::-1]
        for s in starts:
            g = pos[s]
            if strand == 0:
                ex = [(max(a, g), b) for a, b in exons if b >= g]
            else:
                ex = [(a, min(b, g)) for a, b in exons if a <= g]
            ids.append(c.orf(0, strand, ex))
        if dup:
            ids.append(c.orf(0, strand, exons))
            ids.append(c.orf(0, strand, c.orfs[ids[1]][2]))
        return ids

    def exons_at(start, lengths, gap=4):
        ex, p = [], start
        for ln in lengths:
            ex.append((p, p + ln - 1))
            p += ln + gap
        return ex

    # children every two values through the first two exons: P mod 3 of 0, 1, 2, children of every L mod 3
    info["even"] = family(0, exons_at(100, [20, 13, 7, 9, 30]), list(range(2, 20, 2)) + [21, 23, 28], dup=True)
    info["even_minus"] = family(1, exons_at(400, [30, 9, 7, 13, 20]), list(range(2, 20, 2)) + [21, 23, 28], dup=True)
    # children one value apart: all but the last have a one-value first reference and are laid out alone
    info["ones"] = family(0, exons_at(700, [12, 10, 8]), list(range(1, 9)))
    info["ones_minus"] = family(1, exons_at(900, [12, 10, 8]), list(range(1, 9)))
    # families of 31, 32 and 33 references (33: the smallest long ORF, children stay alone)
    for nref, start, strand in ((31, 1100, 0), (32, 2000, 1), (33, 3000, 0), (32, 4000, 0), (31, 5000, 1),
                                (33, 6000, 1)):
        lengths = [int(x) for x in rng.integers(2, 9, nref)]
        ex = exons_at(start, lengths, gap=2)
        starts = list(np.cumsum(lengths)[:-1][::-1][:5]) + [int(lengths[0]) // 2 if lengths[0] >= 4 else 0]
        if strand == 1:
            starts = [sum(lengths) - s for s in starts[:5]]
        info[f"n{nref}_{strand}_{start}"] = family(strand, ex, sorted({s for s in starts if s > 0}))
    # a reads-as-zero stretch inside a family: exons off the padded contig, then children after it
    info["off_left"] = family(0, [(-40, -30), (-12, -10), (-9, 3), (6, 20), (24, 30)], [11 + 3 + 2, 11 + 3 + 13 + 4, 11 + 3 + 13 + 15 + 2])
    end = 3000
    info["off_right"] = family(1, [(end - 30, end - 20), (end - 15, end + 3), (end + 7, end + 9), (end + 20, end + 40)],
                               [21 + 3 + 2, 21 + 3 + 11 + 4, 21 + 3 + 19 + 5])
    # ... and at the END of the profile, so that the trailing partial codon comes from a reference without an atom:
    # a '+' ORF that runs past the end of the padded contig, a '-' ORF that starts before it; the last child holds
    # nothing but reads-as-zero references
    info["off_end"] = family(0, [(end - 50, end - 40), (end - 35, end - 20), (end - 10, end + 15), (end + 20, end + 25)],
                             [2, 13, 15, 29, 46])
    info["off_start_minus"] = family(1, [(-30, -20), (-15, 10), (20, 30), (40, 50)], [2, 13, 25, 31, 40])
    for k in ("off_left", "off_right", "off_end", "off_start_minus"):   # on the second contig
        for o in info[k]:
            c.orfs[o] = (1, c.orfs[o][1], c.orfs[o][2])
    # unknown contig, unknown strand
    info["unknown"] = [c.orf(-1, 0, [(10, 20), (30, 40)]), c.orf(-1, 0, [(30, 40)]), c.orf(0, 2, [(10, 20), (30, 40)]),
                       c.orf(0, 2, [(35, 40)]), c.orf(-1, 1, [(50, 60)])]
    for contig in (0, 1):
        for strand in (0, 1):
            c.put(contig, strand, 1 - c.pad, _dense_random(rng, int(c.lens[contig]) + 2 * c.pad, hi=12))
    return c, info


@pytest.mark.gpu
def test_families(eng):
    c, info = family_case()
    st = c.structure()
    par, refs = st["parent"], st["refs"]
    for f in ("even", "even_minus"):                       # children at P mod 3 of 0, 1, 2 and of every L mod 3
        p = info[f][0]
        L = sum(ln for _, ln in refs[p])
        P = [sum(ln for _, ln in refs[p][:k]) for k, _ in st["children"][p]]
        assert {x % 3 for x in P} == {0, 1, 2} and {(L - x) % 3 for x in P} == {0, 1, 2}, f
    lone = [o for o in info["ones"][1:] + info["ones_minus"][1:] if par[o] < 0]
    assert len(lone) >= 14 and all(refs[o][0][1] == 1 for o in lone)
    sizes = family_sizes(st)
    assert {31, 32} <= {s for s, _ in sizes}
    assert any(len(refs[o]) == 33 for o in range(len(refs)))
    assert any(ch for o, ch in enumerate(st["children"]) if c.orfs[o][1] == 1)
    assert any(None in [a for a, _ in refs[o]] and st["children"][o] for o in range(len(refs)))
    for f in ("off_end", "off_start_minus"):                # a zero stretch ends the family, one child is all zeros
        p = info[f][0]
        assert refs[p][-1][0] is None and {c for _, c in st["children"][p]} >= set(info[f][1:]), f
        assert sum(ln for _, ln in refs[p]) % 3 == 2 and refs[info[f][-1]] == refs[p][-2:], f
    assert refs[info["even"][-2]] == refs[info["even"][0]]                  # exact duplicates
    run_case(eng, c)


# ---- long ORFs --------------------------------------------------------------------------------------------------
def long_case(seed=6):
    rng = np.random.default_rng(seed)
    c = Case([30000], pad=16)
    pos, info = 10, []
    for groups, strand in ((2, 0), (3, 1), (5, 0), (8, 1), (13, 0), (21, 1), (30, 0), (2, 1)):
        nref = 32 * groups - int(rng.integers(0, 31))
        lengths = [int(x) for x in rng.integers(1, 9, nref)]
        for g in range(1, groups):                            # one- and two-value references around every boundary
            for j, ln in zip((32 * g - 2, 32 * g - 1, 32 * g, 32 * g + 1), rng.choice([1, 2], 4)):
                if j < nref:
                    lengths[j] = int(ln)
            if g % 2:
                lengths[32 * g - 1] = 1                       # fetch_tail of a one-value reference
        prof_lengths = lengths if strand == 0 else lengths[::-1]
        ex, p = [], pos
        for ln in prof_lengths:
            ex.append((p, p + ln - 1))
            p += ln + 1
        pos = p + 30
        info.append(c.orf(0, strand, ex))
    for strand in (0, 1):
        c.put(0, strand, 1 - c.pad, _dense_random(rng, int(c.lens[0]) + 2 * c.pad, hi=25))
    return c, info


@pytest.mark.gpu
def test_long_orfs(eng):
    c, info = long_case()
    refs = c.structure()["refs"]
    groups = [-(-len(refs[o]) // GROUP) for o in info]
    assert min(groups) == 2 and max(groups) == 30
    for o in info:
        r = refs[o]
        for g in range(1, -(-len(r) // GROUP)):
            assert r[32 * g - 1][1] <= 2 and r[32 * g - 2][1] <= 2
    assert any(refs[o][32 * g - 1][1] == 1 for o in info for g in range(1, -(-len(refs[o]) // GROUP)))
    run_case(eng, c)


@pytest.mark.gpu
def test_300000_codon_orf(eng):
    rng = np.random.default_rng(8)
    L = 900_000
    c = Case([L + 1000], pad=16)
    o = c.orf(0, 0, [(100, 100 + L - 1)])
    om = c.orf(0, 1, [(50, 50 + L + 1)])
    c.put_profile(o, rng.poisson(0.8, L) * (rng.random(L) < 0.5) + np.tile([1, 0, 0], L // 3) * (rng.random(L) < 0.3))
    c.put_profile(om, rng.poisson(0.3, L + 2))
    assert len(c.structure()["refs"][o]) > 26 * GROUP
    run_case(eng, c, configs=[(True, 0), (False, 0)])
    CO = _oracle()
    ptr, flat = CO.gather_profiles(c.index(), np.arange(2), c.cov, c.base, c.lens, c.pad, c.plane)
    ref = CO.score(c.index(), c.cov, c.base, c.lens, c.pad, c.plane, DEFAULT_PARAMS)
    drift = [abs(ref["score"][k] - reference(flat[ptr[k]:ptr[k + 1]])[0]) for k in range(2)]
    print(f"\n300,000-codon ORFs: oracle drift from the fsum reference {drift}")


# ---- ranges and the plan cache ----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ranges_cut_through_families(eng):
    c, info = family_case()
    st = c.structure()
    n = len(c.orfs)
    full = run_case(eng, c, configs=[(True, 1)])
    cuts = []
    for f in ("even", "even_minus", "n31_0_1100", "off_left"):
        kids = [ch for _, ch in st["children"][info[f][0]]]
        assert kids and all(k > info[f][0] for k in kids)
        cuts.append((min(kids), min(kids) + 4))              # a child in the range, its parent not
    cuts += [(1, n - 1), (info["ones"][3], info["n33_0_3000"][0] + 1)]
    CO = _oracle()
    from ribotricer_b200.engine import ScoreParams
    d_cov = eng.torch.from_numpy(c.cov).to(eng.device)
    prm = list(DEFAULT_PARAMS)
    prm[2] = 1
    for lo, hi in cuts:
        got = eng.score_host(d_cov, lo, hi, params=ScoreParams(*prm), diagnostics=True, min_codon=True)
        ref = CO.score(c.index(), c.cov, c.base, c.lens, c.pad, c.plane, prm, lo, hi)
        compare(got, ref, prm, f"range {lo}:{hi} ")
        for k in got:                                         # the sums are exact: the same bits as the full range
            assert np.array_equal(got[k], full[k][lo:hi], equal_nan=True), (lo, hi, k)


@pytest.mark.gpu
def test_long_accumulators_reset_between_calls(eng):
    CO = _oracle()
    from ribotricer_b200.engine import ScoreParams
    c, info = long_case()
    idx = c.index()
    n = len(c.orfs)
    eng.set_genome(["c0"], c.lens, pad=c.pad)
    eng.set_index(**idx)
    rng = np.random.default_rng(9)
    for layout in ("dense", "compact"):
        eng.set_layout(layout)
        for rep, want in enumerate((True, True, False, False)):
            cov = (c.cov * (rep + 1) + rng.integers(0, 3, len(c.cov)) * (rep % 2)).astype(np.int32)
            d_dense = eng.torch.from_numpy(cov).to(eng.device)
            if layout == "compact":
                d_cov = eng.new_coverage()
                eng.compact_from_dense(d_dense, d_cov)
            else:
                d_cov = d_dense
            got = eng.score_host(d_cov, 0, n, params=ScoreParams(*DEFAULT_PARAMS), diagnostics=True, min_codon=want)
            ref = CO.score(idx, cov, c.base, c.lens, c.pad, c.plane, DEFAULT_PARAMS)
            compare(got, ref, DEFAULT_PARAMS, f"[{layout} call {rep}] ")
    eng.set_layout("dense")


@pytest.mark.gpu
def test_score_device_on_side_stream(eng):
    t = eng.torch
    from ribotricer_b200.engine import ScoreParams
    c, info = family_case()
    lc, _ = long_case(seed=10)
    base = len(c.orfs)
    for o in lc.orfs:                                         # the long ORFs onto contig 0 of the family case
        c.orfs.append((0, o[1], [(a + 7000, b + 7000) for a, b in o[2]]))
    c._structure = None
    eng.set_genome(["c0", "c1"], c.lens, pad=c.pad)
    eng.set_index(**c.index())
    n = len(c.orfs)
    prm = ScoreParams(*DEFAULT_PARAMS)
    d_cov = t.from_numpy(c.cov).to(eng.device)
    for lo, hi in ((0, n), (3, base + 4)):
        want = eng.score_host(d_cov, lo, hi, params=prm, diagnostics=True, min_codon=True)
        side = t.cuda.Stream(device=eng.device)
        side.wait_stream(t.cuda.current_stream(eng.device))
        with t.cuda.stream(side):
            out = eng.new_score_columns(hi - lo, diagnostics=True, min_codon=True)
            eng.score_device(d_cov, out, lo, hi, params=prm)
        side.synchronize()
        for k in want:
            assert np.array_equal(out[k].cpu().numpy(), want[k], equal_nan=True), (lo, hi, k)


# ---- thresholds at equality -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_thresholds_at_equality(eng):
    """Rows of 16 codons (valid / n_codons and count / n_codons exact in binary) whose valid codons, ratio, density
    and minimum codon sum sit exactly on the thresholds; status must match the oracle on every row outside frame
    ties, with the cutoff at 0 so that only score-0 rows are excluded as near the cutoff."""
    CO = _oracle()
    rng = np.random.default_rng(11)
    c = Case([60000], pad=16)
    pos = 10
    for k in range(600):
        L = 48 + k % 3
        strand = (k // 3) % 2
        if k % 5 == 0:
            ex = [(pos, pos + 20), (pos + 24, pos + L + 2)]
        else:
            ex = [(pos, pos + L - 1)]
        o = c.orf(0, strand, ex)
        vals = np.zeros(L, np.int64)
        kind = k % 4
        if kind == 0:                                         # sparse: valid codons near 6
            for j in rng.choice(16, int(rng.integers(4, 9)), replace=False):
                vals[3 * j + int(rng.integers(0, 3))] = int(rng.integers(1, 4))
        elif kind == 1:                                       # count near 32
            hits = rng.choice(L, 10, replace=False)
            vals[hits] = 1
            vals[hits[0]] += 32 - 10 + int(rng.integers(-1, 2))
        else:                                                 # every codon non-empty: minimum codon sum near 2
            vals = rng.integers(1, 4, L)
            j = int(rng.integers(0, 16))
            vals[3 * j:3 * j + 3] = [int(rng.integers(1, 3)), 0, 0]
            if L % 3:
                vals[-(L % 3):] = rng.integers(1, 3, L % 3)
        c.put_profile(o, vals)
        pos += L + 12
    idx = c.index()
    kind = np.arange(600) % 4
    ref0 = CO.score(idx, c.cov, c.base, c.lens, c.pad, c.plane, [0.0, 0, 0, 0, 0.0])
    tie = CO.tie_mask(ref0["frame_K"], ref0["frame_s"])
    assert (np.maximum(ref0["length"] // 3, 1) == 16).all()

    def mode(a):
        v, k = np.unique(a, return_counts=True)
        return int(v[np.argmax(k)])

    T_valid = mode(ref0["valid"][(kind == 0) & ~tie])
    T_count = mode(ref0["count"][kind == 1])
    T_min = mode(ref0["min_codon"][kind >= 2])
    param_sets = [[0.0, T_valid, 0, 0, 0.0], [0.0, 0, 0, T_valid / 16, 0.0], [0.0, 0, 0, 0, T_count / 16],
                  [0.0, 0, T_min, 0, 0.0]]
    on = [(ref0["valid"] == T_valid) & ~tie, (ref0["valid"] == T_valid) & ~tie, ref0["count"] == T_count,
          ref0["min_codon"] == T_min]
    for prm, rows in zip(param_sets, on):
        assert rows.sum() >= 20, (prm, int(rows.sum()))
        ref = CO.score(idx, c.cov, c.base, c.lens, c.pad, c.plane, prm)
        assert 0 < ref["status"][~tie].sum() < (~tie).sum(), prm           # the threshold splits the rows
    param_sets.append([0.0, T_valid - 1, T_min, (T_valid + 1) / 16, T_count / 16])
    for prm in param_sets:
        run_case(eng, c, params=prm, configs=[(False, None), (True, None)])
