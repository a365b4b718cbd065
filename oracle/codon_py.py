"""Plain-Python statement of ``count-orfs-codon`` (DESIGN.md section 11, rules 1-10): the checker of
``rt_codon_load_tsv``, ``rt_codon_load_seq``, ``codon_emit_kernel``, the radix sorts, ``codon_stats_kernel`` and
``rt_codon_write``.

Written for clarity, not speed: files are read as bytes and split line by line, every codon is a Python tuple, and S1,
S2 and the variance numerator are Python integers.  Parity with a run of the reference has NOT been verified (the
reference is not available here); these rules are this project's statement of them.
"""
from __future__ import annotations

import re
import sys

GENE_HEADER = ("gene_id\tcodon\tcodon_occurrences\ttotal_codon_coverage\tmean_codon_coverage\tmedian_codon_coverage\t"
               "var_codon_coverage\n")
CODON_HEADER = ("codon\tcodon_occurrences\ttotal_codon_coverage\tmean_codon_coverage\tmedian_codon_coverage\t"
                "var_codon_coverage\n")
SEQ_HINT = "; was it written by orfs-seq from this index, without --protein?"
PROFILE_RE = re.compile(rb"\[(?:(?:0|[1-9][0-9]*)(?:, (?:0|[1-9][0-9]*))*)?\]\Z")
PROFILE_REASONS = {1: "the profile is not a list of integers written as str(list) writes it",
                   2: "a profile value lies outside 0..2147483647",
                   4: "a codon count exceeds 4294967295"}
MAX_VALUE, MAX_COUNT = 2 ** 31 - 1, 2 ** 32 - 1


class Row:
    """One index row: its first column, ORF_type, re-derived oid, chrom, strand code and sorted intervals."""

    def __init__(self, fields: list):
        self.id, self.type, self.chrom = fields[0], fields[1], fields[7]
        self.strand = 0 if fields[8] == b"+" else 1 if fields[8] == b"-" else 2
        ivs = []
        for group in fields[10].split(b","):
            s, e = group.split(b"-")
            ivs.append((int(s), int(e)))
        ivs.sort(key=lambda iv: iv[0])
        self.ivs = ivs
        self.length = sum(e - s + 1 for s, e in ivs)
        self.oid = b"%s_%d_%d_%d" % (fields[2], ivs[0][0], ivs[-1][1], self.length)

    def coords(self) -> list:
        """Genomic coordinate of every nt in ORF orientation (reversed for '-', as count_orfs builds ``coor``)."""
        c = [p for s, e in self.ivs for p in range(s, e + 1)]
        return c[::-1] if self.strand == 1 else c


def index_rows(path: str) -> list:
    """Rule 1 (the column-count exit of rt_index_load)."""
    with open(path, "rb") as fh:
        lines = fh.read().split(b"\n")
    rows = []
    for line in lines[1:]:
        if not line:
            continue
        f = line.split(b"\t")
        if len(f) != 11:
            sys.exit("Error: unexpected number of columns found for index file\n"
                     "please run ribotricer prepare-orfs to regenerate")
        rows.append(Row(f))
    return rows


def _lines(data: bytes) -> list:
    lines = data.split(b"\n")
    return lines[:-1] if data.endswith(b"\n") else lines


def select(tsv_path: str, rows: list, features, report_all: bool) -> list:
    """Rule 2: (line number, index row, (gene_id, gene_name), profile text) of every selected line, in file order."""
    feats = {f.encode() if isinstance(f, str) else f for f in features}
    cand = {}
    for o, r in enumerate(rows):
        if r.type in feats:
            cand[r.oid] = o                            # a later duplicate replaces an earlier one
    with open(tsv_path, "rb") as fh:
        lines = _lines(fh.read())
    out = []
    for n, raw in enumerate(lines[1:], start=2):
        f = raw.strip().split(b"\t")
        if len(f) != 18:
            raise ValueError(f"{tsv_path} line {n}: {len(f)} tab-separated fields, 18 expected")
        if f[1] not in feats or (f[2] == b"nontranslating" and not report_all):
            continue
        if f[0] not in cand:
            raise ValueError(f"{tsv_path} line {n}: ORF_ID {f[0][:200].decode('latin-1')} is not in the index with an "
                             f"ORF_type of the features")
        out.append((n, cand[f[0]], (f[11], f[12]), f[17]))
    return out


def sequences(path: str, rows: list) -> list:
    """Rule 4: the letters of every index row, checked line by line."""
    with open(path, "rb") as fh:
        data = fh.read()
    nl = data.find(b"\n")
    head_end = nl if nl >= 0 else len(data)
    if data[:head_end] != b"ORF_ID\tsequence":
        raise ValueError(f"{path} line 1: the header is not ORF_ID<tab>sequence{SEQ_HINT}")
    pos, out = head_end + 1, []
    for k, r in enumerate(rows):
        if pos >= len(data):
            raise ValueError(f"{path}: the file ends after line {k + 1}, the index has {len(rows)} rows{SEQ_HINT}")
        e = data.find(b"\n", pos)
        stop = e if e >= 0 else len(data)
        line = data[pos:stop]
        tab = line.find(b"\t")
        got = line[:tab] if tab >= 0 else line
        want = r.id.decode("latin-1")
        if tab < 0 or got != r.id:
            raise ValueError(f"{path} line {k + 2}: ORF_ID {got[:200].decode('latin-1')} is not {want}, the ORF_ID of "
                             f"index row {k + 1}{SEQ_HINT}")
        s = line[tab + 1:]
        if len(s) != r.length:
            raise ValueError(f"{path} line {k + 2}: the sequence of {want} has {len(s)} letters, the index row has "
                             f"{r.length} nt{SEQ_HINT}")
        bad = next((i for i, c in enumerate(s) if c not in b"ACGTN"), None)
        if bad is not None:
            raise ValueError(f"{path} line {k + 2}: the sequence of {want} holds a letter other than A, C, G, T and N "
                             f"at position {bad + 1}{SEQ_HINT}")
        out.append(s)
        pos = stop + 1
    if pos < len(data):
        raise ValueError(f"{path} line {len(rows) + 2}: the file has more lines than the index has rows "
                         f"({len(rows)}){SEQ_HINT}")
    return out


def profile_values(text: bytes):
    """Rule 3: (0, values), or (reason bit, None)."""
    if not PROFILE_RE.match(text):
        return 1, None
    body = text[1:-1]
    vals = [int(x) for x in body.split(b", ")] if body else []
    if any(v > MAX_VALUE for v in vals):
        return 2, None
    return 0, vals


def codons(items: list):
    """Rules 3, 5 and 6 over ``items`` = (line number, gene, place group, profile text, letters, oriented coordinates)
    in file order.  Returns ("refused", line number, reason bit) for the first refused profile, else
    (counts per (gene, codon), counts per codon, summary dict)."""
    parsed = []
    for line_no, gene, group, prof, seq, coor in items:
        reason, vals = profile_values(prof)
        if reason == 0:
            m = min(len(vals), len(seq))
            counts = [vals[3 * k] + vals[3 * k + 1] + vals[3 * k + 2] for k in range(m // 3)]
            if any(c > MAX_COUNT for c in counts):
                reason = 4
        if reason:
            return "refused", line_no, reason
        parsed.append((gene, group, seq, coor, counts))
    seen, by_gene, pooled = set(), {}, {}
    summary = dict(codons=0, with_n=0, duplicates=0, kept=0)
    for gene, group, seq, coor, counts in parsed:
        for k, c in enumerate(counts):
            name = seq[3 * k:3 * k + 3].decode()
            summary["codons"] += 1
            if "N" in name:
                summary["with_n"] += 1
                continue
            place = (group, coor[3 * k])
            if place in seen:
                summary["duplicates"] += 1
                continue
            seen.add(place)
            summary["kept"] += 1
            by_gene.setdefault((gene, name), []).append(c)
            pooled.setdefault(name, []).append(c)
    return by_gene, pooled, summary


def stats(xs: list) -> tuple:
    """Rule 9: occurrences, total, mean, median, var with exact integers."""
    xs = sorted(xs)
    n, s1, s2 = len(xs), sum(xs), sum(x * x for x in xs)
    median = float(xs[n // 2]) if n % 2 else (xs[n // 2 - 1] + xs[n // 2]) / 2
    return n, s1, s1 / n, median, float(n * s2 - s1 * s1) / float(n * n)


def stat_cell(xs: list) -> list:
    """The cell values of codon_stats_kernel: n, S1, S2 low / high 64 bits, sum of the middle two (twice the middle)."""
    xs = sorted(xs)
    n, s1, s2 = len(xs), sum(xs), sum(x * x for x in xs)
    mid = 2 * xs[n // 2] if n % 2 else xs[n // 2 - 1] + xs[n // 2]
    return [n, s1, s2 & (2 ** 64 - 1), s2 >> 64, mid]


def _row(n, s1, mean, median, var) -> str:
    return f"{n}\t{s1}\t{mean!r}\t{median!r}\t{var!r}\n"


def tables_text(by_gene: dict, pooled: dict, gene_keys: list) -> tuple:
    """Rules 7 and 8: the two output texts.  ``gene_keys[g]`` = (gene_id, gene_name) bytes."""
    gene_text = [GENE_HEADER]
    for g in sorted(range(len(gene_keys)), key=lambda i: gene_keys[i]):
        for name in sorted(c for gg, c in by_gene if gg == g):
            gene_text.append(f"{gene_keys[g][0].decode('latin-1')}\t{name}\t" + _row(*stats(by_gene[(g, name)])))
    codon_text = [CODON_HEADER] + [f"{name}\t" + _row(*stats(pooled[name])) for name in sorted(pooled)]
    return "".join(gene_text), "".join(codon_text)


def count_orfs_codon_text(index_path: str, tsv_path: str, features, seq_path: str, report_all: bool = False):
    """The two output files as strings and the summary (rows, genes, codons kept, duplicates, codons with N)."""
    rows = index_rows(index_path)
    sel = select(tsv_path, rows, features, report_all)
    seqs = sequences(seq_path, rows)
    keys, gene_of = [], {}
    items = []
    for line_no, o, key, prof in sel:
        g = gene_of.setdefault(key, len(keys))
        if g == len(keys):
            keys.append(key)
        items.append((line_no, g, (key, rows[o].chrom, rows[o].strand), prof, seqs[o], rows[o].coords()))
    res = codons(items)
    if res[0] == "refused":
        raise ValueError(f"{tsv_path} line {res[1]}: {PROFILE_REASONS[res[2]]}")
    by_gene, pooled, s = res
    gene_text, codon_text = tables_text(by_gene, pooled, keys)
    summary = dict(rows=len(sel), genes=len({g for g, _ in by_gene}), codons=s["kept"], duplicates=s["duplicates"],
                   codons_with_n=s["with_n"])
    return gene_text, codon_text, summary
