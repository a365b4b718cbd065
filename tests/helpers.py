"""Shared helpers for the parity tests (checker side only)."""
from __future__ import annotations

import gzip
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
DEFAULT_PARAMS = [0.428571428571, 5, 0, 0, 0.0]
SCORE_TOL = 1e-9   # BASELINE.json north_star: phase score within 1e-9 absolute


def load_golden(name):
    with gzip.open(os.path.join(GOLDEN, name), "rt") as fh:
        return json.load(fh)


def case_to_arrays(case):
    """Golden pipeline case -> (contig names, lengths, CSR index dict, rows meta)."""
    from oracle import oracle_py as O

    names = [c[0] for c in case["contigs"]]
    lens = np.array([c[1] for c in case["contigs"]], np.int64)
    lut = {n: i for i, n in enumerate(names)}
    ptr, st, en, contig, strand, rows = [0], [], [], [], [], []
    for line in case["index"][1:]:
        orf = O.parse_index_line(line + "\n")
        rows.append(orf)
        for s, e in orf["intervals"]:
            st.append(s)
            en.append(e)
        ptr.append(len(st))
        contig.append(lut.get(orf["chrom"], -1))
        strand.append({"+": 0, "-": 1}.get(orf["strand"], 2))
    idx = dict(exon_ptr=np.array(ptr, np.int64), exon_start=np.array(st, np.int32),
               exon_end=np.array(en, np.int32), orf_contig=np.array(contig, np.int32),
               orf_strand=np.array(strand, np.uint8))
    return names, lens, idx, rows


def alignments_to_reads(case, names):
    """Expand a golden ``alignments[length][strand][(chrom,pos)] = n`` table into read columns
    (forward protocol): '+' reads have first = pos-1, '-' reads have last = pos-1."""
    lut = {n: i for i, n in enumerate(names)}
    cols = {k: [] for k in ("ref_id", "first", "last", "mlen", "flag", "mapq", "nh")}
    for length, strand, chrom, pos, n in case["alignments"]:
        for _ in range(n):
            cols["ref_id"].append(lut[chrom])
            if strand == "+":
                cols["first"].append(pos - 1)
                cols["last"].append(pos - 1 + length - 1)
                cols["flag"].append(0)
            else:
                cols["last"].append(pos - 1)
                cols["first"].append(pos - 1 - length + 1)
                cols["flag"].append(16)
            cols["mlen"].append(length)
            cols["mapq"].append(255)
            cols["nh"].append(1)
    dts = dict(ref_id=np.int32, first=np.int32, last=np.int32, mlen=np.uint16, flag=np.uint16,
               mapq=np.uint8, nh=np.uint8)
    return {k: np.array(v, dts[k]) for k, v in cols.items()}


def merged_to_dense(case, names, base, pad, plane):
    lut = {n: i for i, n in enumerate(names)}
    cov = np.zeros(2 * plane, np.int32)
    dropped = 0
    lens = {c[0]: c[1] for c in case["contigs"]}
    for strand, chrom, pos, n in case["merged"]:
        if pos < 1 - pad or pos > lens[chrom] + pad:
            dropped += n
            continue
        cov[(0 if strand == "+" else 1) * plane + base[lut[chrom]] + pad + pos] += n
    return cov, dropped


def compare_scores(got, ref, tie, params=DEFAULT_PARAMS, what=""):
    """The parity bar of BASELINE.json: integers bit-exact, score within 1e-9, valid/status
    bit-exact outside the frame-tie (H1) and near-cutoff classes."""
    for key in ("count", "length", "min_codon"):
        if key in got:
            assert (got[key] == ref[key]).all(), f"{what}{key} differs"
    d = np.abs(got["score"] - ref["score"])
    assert np.nanmax(d) <= SCORE_TOL if len(d) else True, f"{what}score differs by {np.nanmax(d)}"
    assert (got["valid"] == ref["valid"])[~tie].all(), f"{what}valid_codons differs outside frame ties"
    near = np.abs(ref["score"] - params[0]) <= SCORE_TOL
    assert (got["status"] == ref["status"])[~tie & ~near].all(), f"{what}status differs"
    return int(tie.sum()), int(near.sum())


def compare_tsv(got_text, want_text, phase_score_cutoff, what=""):
    """Two translating-ORFs TSV texts under the parity bar: same header and row order, phase score within SCORE_TOL,
    every other column equal except valid codons / ratio / status on frame ties (H1) and status near the cutoff.  A row
    only one side reports must be a tie or near the cutoff; at most max(2, 5 %) rows differ so.  Returns the number of
    rows of ``want_text``."""
    from oracle import oracle_py as O

    split = lambda text: {r.split("\t")[0]: r.split("\t") for r in text.split("\n")[1:] if r}     # noqa: E731
    assert got_text.split("\n")[0] == want_text.split("\n")[0], f"{what}header differs"
    got, ref = split(got_text), split(want_text)
    assert [k for k in got if k in ref] == [k for k in ref if k in got], f"{what}ORF ordering differs"
    n_exc = 0
    for oid, r in ref.items():
        tie = O.is_frame_tie(O.frame_spectra(eval(r[17])))
        near = abs(float(r[3]) - phase_score_cutoff) <= SCORE_TOL
        if oid not in got:
            assert tie or near, (what, oid)
            n_exc += 1
            continue
        g = got[oid]
        assert abs(float(g[3]) - float(r[3])) <= SCORE_TOL, (what, oid)
        cols = [0, 1, 4, 5, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17]
        if not tie:
            cols += [6, 7] + ([2] if not near else [])
        for c in cols:
            assert g[c] == r[c], (what, oid, c, g[c], r[c])
    n_exc += sum(1 for oid in got if oid not in ref)
    assert n_exc <= max(2, len(ref) // 20), f"{what}{n_exc} rows differ"
    return len(ref)


def decode_stream(records, hdr, n_blocks, block=256):
    """Checker-side decoder of the record stream of include/ribotricer_b200.h (rt_stream_pack): returns one tuple
    (ref_id, first, last, mlen, meta7) per read record, in order.  Plain Python: small cases only."""
    out = []
    rec = np.asarray(records, np.uint32).reshape(-1)
    hdr = np.asarray(hdr, np.int32).reshape(-1)
    for b in range(n_blocks):
        ref, pos = int(hdr[4 * b]), int(hdr[4 * b + 1])
        assert hdr[4 * b + 2] == 0 and hdr[4 * b + 3] == 0
        words = rec[b * block:(b + 1) * block].tolist()
        assert len(words) == block
        k = 0
        while k < block:
            w = words[k]
            k += 1
            if w & 0x8000:
                assert not (w & 0x4000), "extension record without a read in front of it"
                pos += (w >> 16) | ((w & 0x3fff) << 16)
                continue
            pos += w & 0x7fff
            mlen, meta, extra = (w >> 16) & 0xff, w >> 24, 0
            if meta & 0x80:
                assert k < block, "extension record in another block"
                e = words[k]
                k += 1
                assert (e & 0xc000) == 0xc000
                mlen |= (e & 0xff) << 8
                extra = (e >> 16) | (((e >> 8) & 0x3f) << 16)
            out.append((ref, pos, pos + mlen - 1 + extra, mlen, meta & 0x7f))
    return out
