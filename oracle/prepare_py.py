"""Plain-Python statement of ``prepare-orfs`` (DESIGN.md section 9, rules 1-7): the checker of the native loaders,
the ORF kernels and the index writer.

Everything here is written for clarity, not speed: the GTF and FASTA are read line by line into Python objects,
codons are found with ``str.find`` loops over the spliced transcript string (the way the reference searches), and the
file is assembled as one string.  Parity of ORF typing and row order with a run of the reference has NOT been
verified (the reference is not available here); these rules are this project's statement of them.
"""
from __future__ import annotations

import bisect

TYPES = ("annotated", "uORF", "overlap_uORF", "super_uORF", "overlap_dORF", "dORF", "novel", "internal")
HEADER = ("ORF_ID\tORF_type\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\t"
          "chrom\tstrand\tstart_codon\tcoordinate\n")
INT_MAX = 2147483647
_COMP = str.maketrans("ACGTN", "TGCAN")


class GtfError(ValueError):
    pass


class FastaError(ValueError):
    pass


# ------------------------------------------------------------------------------------------------ GTF (rule 1)
def parse_attributes(text: str) -> dict:
    """``key "value";`` pairs in any order; the first occurrence of a key wins."""
    out = {}
    for piece in text.split(";"):
        piece = piece.strip(" ")
        if not piece:
            continue
        key, _, value = piece.partition(" ")
        value = value.strip(" ")
        if len(value) >= 2 and value[0] == '"' and value[-1] == '"':
            value = value[1:-1]
        out.setdefault(key, value)
    return out


def _coord(text: str, line_no: int, what: str) -> int:
    if not text or len(text) > 10 or any(ch not in "0123456789" for ch in text) or not 1 <= int(text) <= INT_MAX:
        raise GtfError(f"GTF line {line_no}: {what} is not a positive integer")
    return int(text)


def parse_gtf(path: str) -> list:
    """The ``exon`` and ``CDS`` lines as dicts, in file order.  Comment (``#``) and blank lines are skipped; any other
    line must have 9 tab-separated columns and integer start <= end (checked on every line, kept or not)."""
    records = []
    with open(path, "rb") as fh:
        data = fh.read().decode()
    for line_no, line in enumerate(data.split("\n"), 1):
        if line.endswith("\r"):
            line = line[:-1]
        if not line or line.startswith("#"):
            continue
        f = line.split("\t")
        if len(f) != 9:
            raise GtfError(f"GTF line {line_no}: expected 9 tab-separated columns, found {len(f)}")
        start, end = _coord(f[3], line_no, "start"), _coord(f[4], line_no, "end")
        if start > end:
            raise GtfError(f"GTF line {line_no}: start > end")
        if f[2] not in ("exon", "CDS"):
            continue
        a = parse_attributes(f[8])
        gene_type = a.get("gene_type", a.get("gene_biotype"))
        tx_type = a.get("transcript_type", a.get("transcript_biotype"))
        records.append(dict(line=line_no, chrom=f[0], feature=f[2], start=start, end=end, strand=f[6],
                            gene_id=a.get("gene_id"), transcript_id=a.get("transcript_id"),
                            gene_name=a.get("gene_name", a.get("gene_id")),
                            gene_type="NA" if gene_type is None else gene_type,
                            transcript_type="NA" if tx_type is None else tx_type))
    return records


# ---------------------------------------------------------------------------------------------------- FASTA
def parse_fasta(path: str) -> dict:
    """contig name (header up to the first whitespace) -> sequence, upper case, every base other than ACGT as N."""
    genome, name, parts = {}, None, []

    def close():
        if name is not None:
            seq = "".join(parts).upper()
            genome[name] = "".join(ch if ch in "ACGT" else "N" for ch in seq)

    with open(path, "rb") as fh:
        data = fh.read().decode("latin-1")
    for line in data.split("\n"):
        line = line.replace("\r", "")
        if line.startswith(">"):
            close()
            name = line[1:].split()[0] if line[1:].split() else ""
            if name in genome:
                raise FastaError(f"duplicate FASTA contig {name}")
            parts = []
        elif name is None:
            if line.strip():
                raise FastaError("FASTA: sequence before the first header")
        else:
            parts.append(line)
    close()
    return genome


# ------------------------------------------------------------------------------------------ transcripts (rule 1)
def merge(intervals: list) -> list:
    """Sort by start, merge overlapping and book-ended intervals."""
    out = []
    for s, e in sorted(intervals):
        if out and s <= out[-1][1] + 1:
            out[-1][1] = max(out[-1][1], e)
        else:
            out.append([s, e])
    return [tuple(iv) for iv in out]


def rank(exons: list, x: int):
    """0-based position of genomic nt x in the ascending exon concatenation, None when x is not exonic."""
    before = 0
    for s, e in exons:
        if s <= x <= e:
            return before + x - s
        before += e - s + 1
    return None


def transcripts(records: list, genome: dict):
    """Kept transcripts (dicts) in candidate order, and the number of skipped ones."""
    groups, cds = {}, {}
    for r in records:
        if r["gene_id"] is None or r["transcript_id"] is None:
            continue
        key = (r["gene_id"], r["transcript_id"])
        (groups if r["feature"] == "exon" else cds).setdefault(key, []).append(r)
    kept, skipped = [], 0
    for key, lines in groups.items():
        first = lines[0]
        chroms, strands = {r["chrom"] for r in lines}, {r["strand"] for r in lines}
        cl = cds.get(key, [])
        exons = merge([(r["start"], r["end"]) for r in lines])
        chrom, strand = first["chrom"], first["strand"]
        bad = len(chroms) > 1 or len(strands) > 1 or strand not in ("+", "-") or chrom not in genome \
            or exons[-1][1] > len(genome[chrom])
        cds_iv = None
        if not bad and cl:
            if {r["chrom"] for r in cl} != {chrom} or {r["strand"] for r in cl} != {strand}:
                bad = True
            else:
                cds_iv = merge([(r["start"], r["end"]) for r in cl])
                if rank(exons, cds_iv[0][0]) is None or rank(exons, cds_iv[-1][1]) is None:
                    bad = True
        if bad:
            skipped += 1
            continue
        kept.append(dict(gene_id=first["gene_id"], transcript_id=first["transcript_id"],
                         gene_name=first["gene_name"], gene_type=first["gene_type"],
                         transcript_type=first["transcript_type"], chrom=chrom, strand=strand, exons=exons,
                         cds=cds_iv, first_exon=first["line"], first_cds=cl[0]["line"] if cl else None))
    return order_by(kept, "first_exon"), skipped


def order_by(txs: list, key: str) -> list:
    """Genes by their first line (the smallest of their transcripts'), transcripts of a gene by their first line."""
    gene_first = {}
    for t in txs:
        gene_first[t["gene_id"]] = min(gene_first.get(t["gene_id"], t[key]), t[key])
    return sorted(txs, key=lambda t: (gene_first[t["gene_id"]], t[key]))


# ------------------------------------------------------------------------------------------- sequence (rule 2)
def spliced(genome: dict, chrom: str, strand: str, intervals: list) -> str:
    seq = "".join(genome[chrom][s - 1:e] for s, e in intervals)
    return seq[::-1].translate(_COMP) if strand == "-" else seq


def cds_bounds(t: dict):
    """Oriented first / last CDS nt in transcript positions, or None."""
    if t["cds"] is None:
        return None
    n = sum(e - s + 1 for s, e in t["exons"])
    lo, hi = rank(t["exons"], t["cds"][0][0]), rank(t["exons"], t["cds"][-1][1])
    return (lo, hi) if t["strand"] == "+" else (n - 1 - hi, n - 1 - lo)


# ------------------------------------------------------------------------------------ candidates (rules 3 and 4)
def find_all(seq: str, codons) -> list:
    out = set()
    for codon in codons:
        i = seq.find(codon)
        while i != -1:
            out.add(i)
            i = seq.find(codon, i + 1)
    return sorted(out)


def orf_type(a: int, b: int, cds) -> str:
    if cds is None:
        return "novel"
    c, d = cds
    if b < c:
        return "uORF"
    if a < c:
        return "overlap_uORF" if b < d else "super_uORF"
    if a > d:
        return "dORF"
    if b > d:
        return "overlap_dORF"
    return "annotated" if (a, b) == (c, d) else "internal"


def candidates(seq: str, cds, start_codons, stop_codons, min_orf_length: int, longest: bool) -> list:
    """(s, p, type) of every written candidate ORF [s, p) of one oriented transcript sequence, s ascending."""
    stops = [[], [], []]
    for p in find_all(seq, stop_codons):
        stops[p % 3].append(p)
    found = []
    for s in find_all(seq, start_codons):
        frame = stops[s % 3]
        k = bisect.bisect_right(frame, s)
        if k < len(frame):
            found.append((s, frame[k]))
    if longest:
        first = {}
        for s, p in found:
            first.setdefault(p, s)
        found = [(s, p) for s, p in found if first[p] == s]
    out = []
    for s, p in found:
        if p - s < min_orf_length:
            continue
        kind = orf_type(s, p - 1, cds)
        if kind not in ("annotated", "internal"):
            out.append((s, p, kind))
    return out


def to_genomic(exons: list, strand: str, s: int, p: int) -> list:
    """Oriented transcript range [s, p) -> ascending 1-based closed genomic intervals."""
    n = sum(e - b + 1 for b, e in exons)
    lo, hi = (s, p) if strand == "+" else (n - p, n - s)
    out, before = [], 0
    for b, e in exons:
        a0, a1 = max(lo, before), min(hi, before + e - b + 1)
        if a0 < a1:
            out.append((b + a0 - before, b + a1 - 1 - before))
        before += e - b + 1
    return out


# ------------------------------------------------------------------------------------------ rows (rules 5-7)
def row_text(t: dict, kind: str, codon: str, ivs: list) -> str:
    length = sum(e - s + 1 for s, e in ivs)
    oid = f"{t['transcript_id']}_{ivs[0][0]}_{ivs[-1][1]}_{length}"
    coord = ",".join(f"{s}-{e}" for s, e in ivs)
    return "\t".join([oid, kind, t["transcript_id"], t["transcript_type"], t["gene_id"], t["gene_name"],
                      t["gene_type"], t["chrom"], t["strand"], codon, coord]) + "\n"


def annotated_rows(txs: list, genome: dict, start_codons) -> list:
    out = []
    for t in order_by([t for t in txs if t["cds"] is not None], "first_cds"):
        codon = spliced(genome, t["chrom"], t["strand"], t["cds"])[:3]
        if len(codon) == 3 and codon in start_codons:
            out.append(row_text(t, "annotated", codon, t["cds"]))
    return out


def candidate_rows(txs: list, genome: dict, start_codons, stop_codons, min_orf_length: int, longest: bool) -> list:
    out = []
    for t in txs:
        seq = spliced(genome, t["chrom"], t["strand"], t["exons"])
        for s, p, kind in candidates(seq, cds_bounds(t), start_codons, stop_codons, min_orf_length, longest):
            out.append(row_text(t, kind, seq[s:s + 3], to_genomic(t["exons"], t["strand"], s, p)))
    return out


def prepare_orfs_text(gtf: str, fasta: str, min_orf_length: int = 60, start_codons=("ATG",),
                      stop_codons=("TAG", "TAA", "TGA"), longest: bool = False) -> str:
    """The whole ``{prefix}_candidate_orfs.tsv`` as a string."""
    genome = parse_fasta(fasta)
    txs, _ = transcripts(parse_gtf(gtf), genome)
    starts, stops = set(start_codons), set(stop_codons)
    return HEADER + "".join(annotated_rows(txs, genome, starts)) + \
        "".join(candidate_rows(txs, genome, starts, stops, min_orf_length, longest))
