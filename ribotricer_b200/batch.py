"""Many libraries against one resident index (BASELINE.json configs[3]; the reference's analogue is the serial
loop over BAMs of learn_cutoff.py:228-264, one full detect_orfs() per library).

The index, its atoms and the compact slot map are set up once and stay on the GPU.  Libraries are dealt to the
ranks of a torchrun job round-robin; inside a rank they run through a three-stage software pipeline:

    stage(i)     decode / pack library i on the host, start its host-to-device copy on the copy stream
    compute(i-1) K1 on the record stream (rt_bin_stream_fresh: overwrites a coverage buffer, no clear) or, for a library
                 that cannot be streamed, a clear and K1 on its read columns; phase A + B, start the device-to-host
                 copy of the result columns -- all enqueued on the compute stream behind the copy of library i-1
    finalize(i-2) wait for library i-2, write its _bam_summary.txt and its TSV (K4 gathers the profiles of the
                 reported ORFs from the library's coverage buffer, which the pipeline keeps alive until then)

so the PCIe copy of the next library, the kernels of the current one and the host-side text of the previous one
overlap.  Two compact coverage buffers alternate (1.8 GB each for a human index).  No WIG files and no metagene
step: both need the genome-wide planes (use detect_orfs() for a library that wants them), so protocol and P-site
offsets have to be given.
"""
from __future__ import annotations

import os

import numpy as np

from .bam import bam_summary_text, load_reads
from .const import (CUTOFF, DEFAULT_PAD, MINIMUM_DENSITY_OVER_ORF, MINIMUM_READS_PER_CODON, MINIMUM_VALID_CODONS,
                    MINIMUM_VALID_CODONS_RATIO)
from .engine import READ_COLUMNS, ScoreParams


class LibraryPipeline:
    """The per-rank pipeline.  ``submit`` libraries one by one, ``drain`` at the end; results come back through
    ``on_result(tag, stats, read_length_counts, columns, coverage)`` (called in submission order)."""

    def __init__(self, engine, protocol, on_result=None):
        t = engine.torch
        self.eng, self.protocol, self.on_result = engine, protocol, on_result
        self.copy_stream = t.cuda.Stream(device=engine.device)
        self.compute_stream = t.cuda.Stream(device=engine.device)
        self.cov = [engine.new_coverage(), engine.new_coverage()]
        self.params = ScoreParams()
        self.want_min = False
        self._staged, self._running = None, None
        self._count = 0
        self._host_cols = [None, None]

    # -- the three stages ------------------------------------------------------------------------------------
    def _stage(self, tag, packed):
        t, eng = self.eng.torch, self.eng
        with t.cuda.stream(self.copy_stream):
            dev = {}
            if "records" in packed:       # a record stream (Engine.stream_reads): 4 B/read
                for k in ("records", "hdr"):
                    a = packed[k]
                    a = a if hasattr(a, "data_ptr") else t.from_numpy(np.ascontiguousarray(a).view(np.int32))
                    dev[k] = a.to(eng.device, non_blocking=True)
                dev["n_blocks"], dev["n"] = int(packed["n_blocks"]), int(packed["n"])
                ev = t.cuda.Event()
                ev.record(self.copy_stream)
                return dict(tag=tag, dev=dev, copied=ev, keep=packed)
            for name, _ in READ_COLUMNS:   # the read columns of _host_records: 18 B/read
                dev[name] = packed[name].to(eng.device, non_blocking=True)
            ev = t.cuda.Event()
            ev.record(self.copy_stream)
        return dict(tag=tag, dev=dev, copied=ev, keep=packed)

    def _compute(self, job):
        t, eng = self.eng.torch, self.eng
        slot = self._count % 2
        self._count += 1
        n_orf = eng.n_orf
        with t.cuda.stream(self.compute_stream):
            self.compute_stream.wait_event(job["copied"])
            cov = self.cov[slot]
            stats, len_counts = eng.new_bin_accumulators()
            if "records" in job["dev"]:      # overwrites the buffer zone by zone: no clear
                eng.bin_stream_device(cov, job["dev"], self.protocol, stats, len_counts, fresh=True)
            else:
                eng.clear_coverage(cov)
                eng.bin_reads_device(cov, job["dev"], self.protocol, stats, len_counts)
            out = eng.new_score_columns(n_orf, min_codon=self.want_min)
            eng.score_device(cov, out, 0, n_orf, self.params)
            if self._host_cols[slot] is None:
                self._host_cols[slot] = {k: t.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items()}
                self._host_cols[slot]["stats"] = t.empty(stats.shape, dtype=stats.dtype).pin_memory()
                self._host_cols[slot]["len_counts"] = t.empty(len_counts.shape, dtype=len_counts.dtype).pin_memory()
            host = self._host_cols[slot]
            for k, v in out.items():
                host[k].copy_(v, non_blocking=True)
            host["stats"].copy_(stats, non_blocking=True)
            host["len_counts"].copy_(len_counts, non_blocking=True)
            done = t.cuda.Event()
            done.record(self.compute_stream)
        # the device records and the result columns stay referenced until finalize(): their memory belongs to the
        # copy / compute stream pools and must not be handed out again while these kernels run
        job.update(slot=slot, done=done, _hold=(out, stats, len_counts, job["dev"], job["keep"]), dev=None, keep=None)
        return job

    def _finalize(self, job):
        from . import _lib

        job["done"].synchronize()
        host = self._host_cols[job["slot"]]
        cols = {k: host[k].numpy() for k in host if k not in ("stats", "len_counts")}
        stats = dict(zip(_lib.ST_NAMES, host["stats"].numpy().tolist()))
        lcn = host["len_counts"].numpy()
        rlc = {int(length): int(lcn[length]) for length in np.flatnonzero(lcn)}
        if self.on_result is not None:
            # K4 work of the callback goes behind this library's kernels, before the buffer's next clear
            with self.eng.torch.cuda.stream(self.compute_stream):
                self.on_result(job["tag"], stats, rlc, cols, self.cov[job["slot"]])
        job["_hold"] = None

    # -- driver ------------------------------------------------------------------------------------------------
    def submit(self, tag, packed):
        """``packed``: what ``Engine.stream_reads(cols, pinned=True)`` (a coordinate-sorted library as 4 B/read records)
        returns for one library, or its seven read columns as page-locked tensors (18 B/read, any order; 16-bit
        columns viewed as int16), as ``_host_records`` makes them."""
        nxt = self._stage(tag, packed)
        run = self._compute(self._staged) if self._staged is not None else None
        if self._running is not None:
            self._finalize(self._running)
        self._staged, self._running = nxt, run

    def drain(self):
        run = self._compute(self._staged) if self._staged is not None else None
        if self._running is not None:
            self._finalize(self._running)
        if run is not None:
            self._finalize(run)
        self._staged = self._running = None
        self.compute_stream.synchronize()


def _host_records(eng, reads):
    """The library as page-locked host records: the 4 B/read record stream when it is coordinate-sorted (and codes),
    else its 18 B/read columns."""
    from ._lib import RtError

    if reads.sorted_by_coordinate:
        try:
            return eng.stream_reads(reads.cols, pinned=True)
        except RtError:
            pass
    t = eng.torch
    cols = {}
    for name, dt in READ_COLUMNS:
        a = np.ascontiguousarray(reads.cols[name], dtype=dt)
        # torch has no uint16 arithmetic but can hold the bytes; view as int16 for transport, as Engine.upload_reads does
        cols[name] = t.from_numpy(a.view(np.int16) if dt == np.uint16 else a).pin_memory()
    return cols


def detect_orfs_batch(bams, ribotricer_index: str, prefixes, protocol: str, read_lengths, psite_offsets: dict,
                      phase_score_cutoff: float = CUTOFF, min_valid_codons: int = MINIMUM_VALID_CODONS,
                      min_reads_per_codon: float = MINIMUM_READS_PER_CODON,
                      min_valid_codons_ratio: float = MINIMUM_VALID_CODONS_RATIO,
                      min_density_over_orf: float = MINIMUM_DENSITY_OVER_ORF, report_all: bool = False, engine=None):
    """detect-orfs for every library of ``bams`` (BAM paths, ``.npz`` column files or ``ReadColumns``) against one
    index: ``{prefix}_translating_ORFs.tsv`` and ``{prefix}_bam_summary.txt`` per library, byte for byte what
    ``detect_orfs(bam, index, prefix, protocol, read_lengths, psite_offsets, ...)`` writes.  Under torchrun the
    libraries are dealt to the ranks round-robin (rank r takes libraries r, r + world, ...).  Returns the list of
    (library number, stats) this rank processed."""
    from .detect_orfs import MergedAlignments, get_engine, load_index, write_tsv
    from .multi_gpu import world

    if protocol is None or psite_offsets is None:
        raise ValueError("detect_orfs_batch needs the protocol and the P-site offsets (it keeps no genome-wide planes "
                         "for the metagene step); run detect_orfs() on one library to infer them")
    if len(bams) != len(prefixes):
        raise ValueError("one prefix per library")
    rank, size, local = world()
    eng = engine or get_engine(local)
    mine = list(range(rank, len(bams), size))
    if not mine:
        return []
    idx = load_index(ribotricer_index)
    first = load_reads(bams[mine[0]])
    if (list(eng.contig_names) != list(first.contig_names) or eng.pad != DEFAULT_PAD
            or not np.array_equal(eng.contig_len, first.contig_len)):
        eng.set_genome(first.contig_names, first.contig_len, DEFAULT_PAD)
    eng.set_length_table(psite_offsets, read_lengths)
    lut = {n: i for i, n in enumerate(eng.contig_names)}
    eng.set_index(**idx.device_columns(lut))
    eng._resident_index = idx
    eng.set_layout("compact")
    done = []

    def on_result(k, stats, rlc, cols, cov):
        prefix = prefixes[k]
        os.makedirs(os.path.dirname(prefix) or ".", exist_ok=True)
        with open(f"{prefix}_bam_summary.txt", "w") as fh:
            fh.write(bam_summary_text(stats, rlc))
        write_tsv(f"{prefix}_translating_ORFs.tsv", idx, cols, MergedAlignments(eng, cov), 0, idx.n_orf, report_all)
        done.append((k, stats))

    pipe = LibraryPipeline(eng, protocol, on_result)
    pipe.params = ScoreParams(phase_score_cutoff, min_valid_codons, min_reads_per_codon, min_valid_codons_ratio,
                              min_density_over_orf)
    try:
        for k in mine:
            reads = first if k == mine[0] else load_reads(bams[k])
            if list(reads.contig_names) != list(eng.contig_names) or not np.array_equal(reads.contig_len, eng.contig_len):
                raise ValueError(f"library {k}: its reference sequences differ from those of the first library")
            pipe.submit(k, _host_records(eng, reads))
        pipe.drain()
    finally:
        eng.set_layout("dense")
        eng._resident_index = None
    return done


__all__ = ["LibraryPipeline", "detect_orfs_batch"]
