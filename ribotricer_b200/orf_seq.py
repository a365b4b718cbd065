"""``orfs-seq``: the nucleotide or protein sequence of every row of a candidate-ORF index.

    index          rt_index_load (all cores), rt_index_ids (the ORF_ID column byte for byte)
    FASTA          rt_fasta_load / rt_fasta_codes (only the contigs the index uses)
    sequences      Engine.orf_seq_write: orf_seq_kernel<nt|protein> per chunk of lines, two device buffers, copy-back
                   overlapped with the next chunk's kernel, a writer thread

The rules are those of DESIGN.md section 10.  Same name and argument order as the reference's ``orf_seq``
(orf_seq.py:128-179).  Inputs are plain text or BGZF (inflated on the GPU, ``bgzf.open_texts``); other gzip files are
refused.
"""
from __future__ import annotations

import os
import pathlib

import numpy as np

from . import _lib
from .bgzf import StageClock, open_texts
from .index import load_native_index
from .prepare_orfs import Genome


def orf_seq(ribotricer_index, genome_fasta, saveto, translate=False, chunk_bytes: int = 0,
            stage_ms: dict | None = None):
    """Write ``saveto``: ``ORF_ID\\tsequence`` and one line per index row, in file order.  ``translate`` writes the
    protein instead of the nucleotides.  ``stage_ms``, when given, receives the time of every stage in milliseconds."""
    from .detect_orfs import get_engine

    clock = StageClock(stage_ms)
    index_src, fasta_src = open_texts([ribotricer_index, genome_fasta], "orfs-seq")
    clock.lap("inflate")
    idx = load_native_index(index_src)
    id_off, ids = idx.ids()
    clock.lap("index_load")
    genome = Genome(fasta_src)
    clock.lap("fasta_load")
    lut = {name: i for i, name in enumerate(genome.names)}
    table = np.array([lut.get(c, -1) for c in idx.chrom_names], np.int64)
    for k in np.flatnonzero(table < 0).tolist():
        n_rows = int(np.count_nonzero(idx.orf_chrom_id == k))
        raise ValueError(f"chrom {idx.chrom_names[k]} of the index ({n_rows} rows) is absent from the FASTA "
                         f"{genome_fasta}")
    used = np.unique(table).astype(np.int32)
    codes = genome.codes(used)
    contig_len = genome.lengths[used]
    contig_base = np.cumsum(contig_len) - contig_len
    orf_contig = np.searchsorted(used, table)[idx.orf_chrom_id] if idx.n_orf else np.zeros(0, np.int64)
    genome.close()
    clock.lap("codes")
    pathlib.Path(os.path.dirname(os.path.abspath(saveto))).mkdir(parents=True, exist_ok=True)
    dev_ms = np.zeros(_lib.RT_SEQ_STAGES, np.float32)
    get_engine().orf_seq_write(saveto, idx.exon_ptr, idx.exon_start, idx.exon_end, orf_contig,
                               idx.orf_strand_code == 1, contig_base, contig_len, codes, id_off, ids, bool(translate),
                               chunk_bytes, stage_ms=dev_ms)
    clock.lap("write")
    clock.device(("upload", "orf_seq_kernel", "copy_back"), dev_ms)
    n_orf = idx.n_orf
    residues = os.path.getsize(saveto) - len("ORF_ID\tsequence\n") - int(id_off[-1]) - 2 * n_orf
    unit = "aa" if translate else "nt"
    print(f"orfs-seq: {n_orf} ORF sequences ({residues} {unit}) written to {saveto} "
          f"({os.path.getsize(saveto)} bytes)")
    return dict(n_orf=n_orf, residues=residues, unit=unit, bytes=os.path.getsize(saveto))
