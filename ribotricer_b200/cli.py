"""Command line of the B200 path: ``prepare-orfs``, ``detect-orfs``, ``count-orfs`` and ``learn-cutoff``.

The flag names, defaults, flag -> argument renames (``--min_read_density`` -> ``min_density_over_orf``,
``--stranded yes`` -> ``forward``, ``--meta-min-reads``) and every validation message are those of the
reference command line (ribotricer/cli.py:127-289, 292-339, 435-560), so existing invocations keep working.
``prepare-orfs`` takes the reference's flags (ribotricer/cli.py) and reads plain-text GTF and FASTA files only.
The commands are assembled from option tables below.  ``--bam`` also accepts a ``.npz`` of decoded columns.
"""
from __future__ import annotations

import os
import sys

import click

from . import __version__
from . import const as K

CONTEXT_SETTINGS = {"help_option_names": ["-h", "--help"]}
_INDEX_HELP = "Path to the index file of ribotricer\nThis file should be generated using ribotricer prepare-orfs"
_REPORT_ALL_HELP = "Whether output all ORFs including those non-translating ones"

try:   # colours are cosmetic; the package is absent in some environments
    from click_help_colors import HelpColorsGroup
    _GROUP_KW = dict(cls=HelpColorsGroup, help_headers_color="yellow", help_options_color="green")
except ImportError:
    _GROUP_KW = {}


@click.group(**_GROUP_KW)
@click.version_option(version=__version__)
def cli() -> None:
    """ribotricer: Tool for detecting translating ORF from Ribo-seq data (B200-native prepare-orfs and detect-orfs)"""


def _register(name: str, summary: str, options, handler) -> None:
    """One sub-command from a table of (flag, click.Option keyword arguments)."""
    params = [click.Option([flag], **kw) for flag, kw in options]
    cli.add_command(click.Command(name, params=params, callback=handler, help=summary,
                                  context_settings=CONTEXT_SETTINGS))


def _fail(message: str):
    sys.exit("Error: " + message)


def _need_file(path, what: str) -> None:
    if not os.path.isfile(path):
        _fail(f"{what} not found")


def _csv(text: str) -> list:
    """Comma separated option value -> items with surrounding blanks removed (common.py:148-161)."""
    return [item.strip(" ") for item in text.split(",")]


def _int_list(text, name: str):
    if text is None:
        return None
    try:
        return [int(item.strip()) for item in text.strip().split(",")]
    except Exception:
        _fail(f"cannot convert {name} into integers")


# ------------------------------------------------------------------------------------ prepare-orfs
def _codons(text: str, name: str) -> set:
    """Comma separated codons, stripped and upper-cased; each must be three letters of ACGT."""
    items = [item.strip().upper() for item in text.split(",")]
    items = [item for item in items if item]
    if not items:
        _fail(f"{name} must list at least one codon")
    for item in items:
        if len(item) != 3 or any(b not in "ACGT" for b in item):
            _fail(f"{name}: {item!r} is not a codon of three letters of ACGT")
    return set(items)


def _prepare(gtf, fasta, prefix, min_orf_length, start_codons, stop_codons, longest) -> None:
    from .prepare_orfs import prepare_orfs

    _need_file(gtf, "GTF file")
    _need_file(fasta, "FASTA file")
    for path, what in ((gtf, "GTF"), (fasta, "FASTA")):
        if path.endswith((".gz", ".bgz")):
            _fail(f"{what} file {path} is compressed; prepare-orfs reads plain text only (decompress it first)")
    if min_orf_length < 0:
        _fail("min_orf_length must be >= 0")
    starts, stops = _codons(start_codons, "start_codons"), _codons(stop_codons, "stop_codons")
    try:
        prepare_orfs(gtf, fasta, prefix, min_orf_length, starts, stops, longest)
    except ValueError as exc:
        _fail(str(exc))


_register("prepare-orfs", "Extract candidate ORFs based on GTF and FASTA files", [
    ("--gtf", dict(help="Path to GTF file", required=True)),
    ("--fasta", dict(help="Path to FASTA file", required=True)),
    ("--prefix", dict(help="Prefix to output file", required=True)),
    ("--min_orf_length", dict(type=int, default=60, show_default=True, help="The minimum length (nts) of ORF to include")),
    ("--start_codons", dict(default="ATG", show_default=True, help="Comma separated list of start codons")),
    ("--stop_codons", dict(default="TAG,TAA,TGA", show_default=True, help="Comma separated list of stop codons")),
    ("--longest", dict(is_flag=True, help="Choose the most upstream start codon if multiple in frame ones exist")),
], _prepare)


# ------------------------------------------------------------------------------------ detect-orfs
def _detect(bam, ribotricer_index, prefix, stranded, read_lengths, psite_offsets, phase_score_cutoff,
            min_valid_codons, min_reads_per_codon, min_valid_codons_ratio, min_read_density, report_all,
            meta_min_reads) -> None:
    from .detect_orfs import detect_orfs

    _need_file(bam, "BAM file")
    _need_file(ribotricer_index, "ribotricer index file")
    lengths = _int_list(read_lengths, "read_lengths")
    if lengths is not None and min(lengths) <= 0:
        _fail("read length must be positive")
    offsets = None
    if psite_offsets is not None:
        if lengths is None:
            _fail("psite_offsets only allowed when read_lengths is provided")
        values = _int_list(psite_offsets, "psite_offsets")
        if len(values) != len(lengths):
            _fail("psite_offsets must match read_lengths")
        if min(values) < 0:
            _fail("P-site offset must be >= 0")
        if any(off >= length for length, off in zip(lengths, values)):
            _fail("P-site offset must be smaller than read length")
        offsets = dict(zip(lengths, values))
    protocol = "forward" if stranded == "yes" else stranded
    detect_orfs(bam, ribotricer_index, prefix, protocol, lengths, offsets, phase_score_cutoff, min_valid_codons,
                min_reads_per_codon, min_valid_codons_ratio, min_read_density, report_all, meta_min_reads)


_register("detect-orfs", "Detect translating ORFs from BAM file", [
    ("--bam", dict(help="Path to BAM file", required=True)),
    ("--ribotricer_index", dict(help=_INDEX_HELP, required=True)),
    ("--prefix", dict(help="Prefix to output file", required=True)),
    ("--stranded", dict(type=click.Choice(["yes", "no", "reverse"]), default=None, show_default=True,
                        help="whether the data is from a strand-specific assay If not provided, the experimental "
                             "protocol will be automatically inferred")),
    ("--read_lengths", dict(default=None, show_default=True,
                            help="Comma separated read lengths to be used, such as 28,29,30\nIf not provided, it will "
                                 "be automatically determined by assessing the metagene periodicity")),
    ("--psite_offsets", dict(default=None, show_default=True,
                             help="Comma separated P-site offsets for each read length matching the read lengths "
                                  "provided.\nIf not provided, reads from different read lengths will be "
                                  "automatically aligned using cross-correlation")),
    ("--phase_score_cutoff", dict(type=float, default=K.CUTOFF, show_default=True,
                                  help="Phase score cutoff for determining active translation")),
    ("--min_valid_codons", dict(type=int, default=K.MINIMUM_VALID_CODONS, show_default=True,
                                help="Minimum number of codons with non-zero reads for determining active translation")),
    ("--min_reads_per_codon", dict(type=int, default=K.MINIMUM_READS_PER_CODON, show_default=True,
                                   help="Minimum number of reads per codon for determining active translation")),
    ("--min_valid_codons_ratio", dict(type=float, default=K.MINIMUM_VALID_CODONS_RATIO, show_default=True,
                                      help="Minimum ratio of codons with non-zero reads to total codons for "
                                           "determining active translation")),
    ("--min_read_density", dict(type=float, default=K.MINIMUM_DENSITY_OVER_ORF, show_default=True,
                                help="Minimum read density (total_reads/length) over an ORF total codons for "
                                     "determining active translation")),
    ("--report_all", dict(is_flag=True, help=_REPORT_ALL_HELP)),
    ("--meta-min-reads", dict(type=int, default=K.META_MIN_READS, show_default=True,
                              help="Minimum number of reads for a read length to be considered")),
], _detect)


# ------------------------------------------------------------------------------------ count-orfs
def _count(ribotricer_index, detected_orfs, features, out, report_all) -> None:
    from .count_orfs import count_orfs

    _need_file(ribotricer_index, "ribotricer index file")
    _need_file(detected_orfs, "detected orfs file")
    count_orfs(ribotricer_index, detected_orfs, {item.strip() for item in features.strip().split(",")}, out, report_all)


_register("count-orfs", "Count reads for detected ORFs at gene level", [
    ("--ribotricer_index", dict(help=_INDEX_HELP, required=True)),
    ("--detected_orfs", dict(required=True, help="Path to the detected orfs file\nThis file should be generated "
                                                 "using ribotricer detect-orfs")),
    ("--features", dict(help="ORF types separated with comma", required=True)),
    ("--out", dict(help="Path to output file", required=True)),
    ("--report_all", dict(is_flag=True, help=_REPORT_ALL_HELP)),
], _count)


# ------------------------------------------------------------------------------------ learn-cutoff
def _learn(ribo_bams, rna_bams, ribo_tsvs, rna_tsvs, ribotricer_index, prefix, filter_by_tx_annotation,
           phase_score_cutoff, min_valid_codons, sampling_ratio, n_bootstraps) -> None:
    from .learn_cutoff import determine_cutoff_bam, determine_cutoff_tsv

    wanted_types = _csv(filter_by_tx_annotation)
    if ribo_bams and ribo_tsvs:
        _fail("--ribo-bams and --rna_bams cannot be specified together")
    if rna_bams and rna_tsvs:
        _fail("--rna-bams and --rna_tsvs cannot be specified together")
    if (ribo_bams and rna_tsvs) or (rna_bams and ribo_tsvs):
        _fail("BAM and TSV inputs cannot be specified together")
    if ribotricer_index:
        _need_file(ribotricer_index, "ribotricer index file")
    ribo_b = _csv(ribo_bams) if ribo_bams else []
    rna_b = _csv(rna_bams) if ribo_bams and rna_bams else []
    if ribo_b and rna_b:
        if not prefix:
            _fail("--prefix required with BAM inputs")
        if not ribotricer_index:
            _fail("--ribotricer_index required with BAM inputs")
        determine_cutoff_bam(ribo_b, rna_b, ribotricer_index, prefix, [], [], wanted_types, sampling_ratio,
                             n_bootstraps, phase_score_cutoff, min_valid_codons, report_all=True)
        return
    ribo_t = _csv(ribo_tsvs) if ribo_tsvs and not ribo_bams else []
    rna_t = _csv(rna_tsvs) if rna_tsvs and not ribo_bams else []
    determine_cutoff_tsv(ribo_t, rna_t, wanted_types, sampling_ratio, n_bootstraps)


_register("learn-cutoff", "Learn phase score cutoff from BAM/TSV file", [
    ("--ribo_bams", dict(help="Path(s) to Ribo-seq BAM file separated by comma")),
    ("--rna_bams", dict(help="Path(s) to RNA-seq BAM file separated by comma")),
    ("--ribo_tsvs", dict(help="Path(s) to Ribo-seq *_translating_ORFs.tsv file separated by comma")),
    ("--rna_tsvs", dict(help="Path(s) to RNA-seq *_translating_ORFs.tsv file separated by comma")),
    ("--ribotricer_index", dict(help=_INDEX_HELP + " (required for BAM input)")),
    ("--prefix", dict(help="Prefix to output file")),
    ("--filter_by_tx_annotation", dict(type=str, default="protein_coding", show_default=True,
                                       help="transcript_type to filter regions by")),
    ("--phase_score_cutoff", dict(type=float, default=K.CUTOFF, show_default=True,
                                  help="Phase score cutoff for determining active translation (required for BAM input)")),
    ("--min_valid_codons", dict(type=int, default=K.MINIMUM_VALID_CODONS, show_default=True,
                                help="Minimum number of codons with non-zero reads for determining active translation "
                                     "(required for BAM input)")),
    ("--sampling_ratio", dict(type=float, default=0.33, show_default=True,
                              help="Number of protein coding regions to sample per bootstrap")),
    ("--n_bootstraps", dict(type=int, default=20000, show_default=True, help="Number of bootstraps")),
], _learn)


if __name__ == "__main__":
    cli()
