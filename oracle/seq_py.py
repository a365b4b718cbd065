"""Plain-Python statement of ``orfs-seq`` (DESIGN.md section 10, rules 1-6): the checker of ``rt_index_ids``,
``orf_seq_kernel`` and the sequence writer.

Written for clarity, not speed: the index is split line by line, every row's sequence is sliced out of the FASTA string
and, for protein, translated codon by codon through a dict.  Parity with a run of the reference has NOT been verified
(the reference is not available here); these rules are this project's statement of them.
"""
from __future__ import annotations

import sys

from oracle.prepare_py import parse_fasta, spliced

HEADER = "ORF_ID\tsequence\n"
_BASES = "TCAG"
_AMINO = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"   # NCBI table 1 in TCAG order
CODON_TABLE = {a + b + c: _AMINO[16 * i + 4 * j + k] for i, a in enumerate(_BASES) for j, b in enumerate(_BASES)
               for k, c in enumerate(_BASES)}


def parse_rows(index_path: str) -> list:
    """(ORF_ID, chrom, strand, intervals sorted by start) per row, in file order (rule 1)."""
    rows = []
    with open(index_path, "rb") as fh:
        lines = fh.read().decode("latin-1").split("\n")
    for line in lines[1:]:
        if not line:
            continue
        f = line.split("\t")
        if len(f) != 11:
            sys.exit("{}\n{}".format("Error: unexpected number of columns found for index file",
                                     "please run ribotricer prepare-orfs to regenerate"))
        ivs = []
        for group in f[10].split(","):
            s, e = group.split("-")
            ivs.append((int(s), int(e)))
        ivs.sort(key=lambda iv: iv[0])
        rows.append((f[0], f[7], f[8], ivs))
    return rows


def check_chroms(rows: list, genome: dict, fasta: str) -> None:
    """Rule 6: the first index chrom (in order of first appearance) absent from the FASTA."""
    counts = {}
    for _, chrom, _, _ in rows:
        counts[chrom] = counts.get(chrom, 0) + 1
    for chrom, n in counts.items():
        if chrom not in genome:
            raise ValueError(f"chrom {chrom} of the index ({n} rows) is absent from the FASTA {fasta}")


def check_intervals(oid: str, ivs: list, contig_len: int) -> None:
    """Rule 6: the first bad interval of a row."""
    for s, e in ivs:
        if e < s:
            raise ValueError(f"ORF {oid}: interval {s}-{e} ends before it starts")
        if s < 1 or e > contig_len:
            raise ValueError(f"ORF {oid}: interval {s}-{e} is outside its contig of {contig_len} nt")


def translate(seq: str) -> str:
    """Rule 5: codons from the first nt, table 1, X for a codon holding an N, a trailing 1-2 nt dropped."""
    return "".join(CODON_TABLE.get(seq[i:i + 3], "X") for i in range(0, len(seq) - 2, 3))


def sequence(genome: dict, chrom: str, strand: str, ivs: list, protein: bool) -> str:
    """Rules 3 and 4 (``parse_fasta`` already writes A C G T in upper case and every other byte as N)."""
    seq = spliced(genome, chrom, "-" if strand == "-" else "+", ivs)
    return translate(seq) if protein else seq


def lines_text(rows: list, genome: dict, protein: bool) -> str:
    for oid, chrom, _, ivs in rows:
        check_intervals(oid, ivs, len(genome[chrom]))
    return HEADER + "".join(f"{oid}\t{sequence(genome, chrom, strand, ivs, protein)}\n"
                            for oid, chrom, strand, ivs in rows)


def orfs_seq_text(index_path: str, fasta: str, protein: bool = False) -> str:
    """The whole output file as a string."""
    rows = parse_rows(index_path)
    genome = parse_fasta(fasta)
    check_chroms(rows, genome, fasta)
    return lines_text(rows, genome, protein)
