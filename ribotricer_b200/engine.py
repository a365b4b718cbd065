"""Device-side engine: one ``Engine`` per (process, GPU).

Thin host layer over the C ABI (``include/ribotricer_b200.h``).  PyTorch is
used only as plumbing: it owns the device buffers (coverage planes, read
columns, result columns) and the CUDA stream; every computation on the path is
one of the hand-written sm_100a kernels in ``csrc/rt_kernels.cuh``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from .const import (CUTOFF, DEFAULT_PAD, MINIMUM_DENSITY_OVER_ORF, MINIMUM_READS_PER_CODON,
                    MINIMUM_VALID_CODONS, MINIMUM_VALID_CODONS_RATIO)

READ_COLUMNS = (("ref_id", np.int32), ("first", np.int32), ("last", np.int32), ("mlen", np.uint16),
                ("flag", np.uint16), ("mapq", np.uint8), ("nh", np.uint8))
READ_BYTES = sum(np.dtype(dt).itemsize for _, dt in READ_COLUMNS)   # 18 B / read

PROTOCOLS = {"forward": _lib.RT_PROTOCOL_FORWARD, "reverse": _lib.RT_PROTOCOL_REVERSE}


def protocol_code(protocol) -> int:
    """bam.py:105,118 only know 'forward' and 'reverse'; anything else stores no read."""
    if isinstance(protocol, (int, np.integer)):
        return int(protocol)
    return PROTOCOLS.get(protocol, _lib.RT_PROTOCOL_NONE)


def make_len_table(psite_offsets=None, read_lengths=None) -> np.ndarray:
    """length -> P-site offset / RT_LEN_UNUSED / RT_LEN_FILTERED.

    ``read_lengths`` is split_bam's filter (bam.py:101); ``psite_offsets`` are
    the lengths merge_read_lengths keeps (detect_orfs.py:74).
    """
    t = np.full(_lib.RT_LEN_TABLE, _lib.RT_LEN_UNUSED, dtype=np.int32)
    if read_lengths is not None:
        t[:] = _lib.RT_LEN_FILTERED
        for length in read_lengths:
            if 0 <= int(length) < _lib.RT_LEN_TABLE:
                t[int(length)] = _lib.RT_LEN_UNUSED
    for length, off in (psite_offsets or {}).items():
        if 0 <= int(length) < _lib.RT_LEN_TABLE and t[int(length)] != _lib.RT_LEN_FILTERED:
            t[int(length)] = int(off)
    return t


@dataclass
class ScoreParams:
    phase_score_cutoff: float = CUTOFF
    min_valid_codons: float = MINIMUM_VALID_CODONS
    min_reads_per_codon: float = MINIMUM_READS_PER_CODON
    min_valid_codons_ratio: float = MINIMUM_VALID_CODONS_RATIO
    min_density_over_orf: float = MINIMUM_DENSITY_OVER_ORF

    def as_c(self) -> _lib.ScoreParams:
        return _lib.ScoreParams(float(self.phase_score_cutoff), float(self.min_valid_codons),
                                float(self.min_reads_per_codon), float(self.min_valid_codons_ratio),
                                float(self.min_density_over_orf))


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Engine:
    """Owns one ``rt_ctx``.  Fails loudly without the library or a B200."""

    def __init__(self, device: int = 0):
        import torch

        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.RtError("ribotricer_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.torch = torch
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        torch.cuda.set_device(self.device)
        ctx = C.c_void_p()
        _lib.check(self.lib.rt_create(self.device_index, C.byref(ctx)))
        self.ctx = ctx
        self.contig_names: list[str] = []
        self.contig_len = np.zeros(0, np.int64)
        self.contig_base = np.zeros(0, np.int64)
        self.pad = 0
        self.plane = 0
        self.n_orf = 0

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.rt_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -------------------------------------------------------------- helpers
    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        _lib.check(rc, self.ctx)

    @property
    def launches(self) -> int:
        return int(self.lib.rt_launch_count(self.ctx))

    @property
    def h2d_bytes(self) -> int:
        """Bytes of read data the host-buffer entry points have copied to the device so far."""
        return int(self.lib.rt_h2d_bytes(self.ctx))

    # --------------------------------------------------------------- genome
    def set_genome(self, contig_names, contig_len, pad: int = DEFAULT_PAD):
        self.contig_names = [str(c) for c in contig_names]
        self.contig_len = np.ascontiguousarray(contig_len, dtype=np.int64)
        if len(self.contig_names) != len(self.contig_len):
            raise ValueError("contig_names and contig_len differ in length")
        self.pad = int(pad)
        self._check(self.lib.rt_set_genome(self.ctx, len(self.contig_len), _np_ptr(self.contig_len), self.pad))
        self.plane = int(self.lib.rt_plane_elems(self.ctx))
        self.contig_base = np.zeros(len(self.contig_len), np.int64)
        self._check(self.lib.rt_get_contig_base(self.ctx, _np_ptr(self.contig_base)))
        self.n_orf = 0
        self.layout = "dense"
        self._resident_index = None
        self._contig_lut = {n: i for i, n in enumerate(self.contig_names)}

    def contig_id(self, name: str) -> int:
        if not hasattr(self, "_contig_lut") or len(self._contig_lut) != len(self.contig_names):
            self._contig_lut = {n: i for i, n in enumerate(self.contig_names)}
        return self._contig_lut.get(name, -1)

    def set_length_table(self, psite_offsets=None, read_lengths=None, table: np.ndarray | None = None):
        t = make_len_table(psite_offsets, read_lengths) if table is None else np.ascontiguousarray(table, np.int32)
        self._check(self.lib.rt_set_length_table(self.ctx, _np_ptr(t)))
        self.len_table = t

    def new_coverage(self):
        """Zeroed int32 coverage buffer of the current layout (dense: [2 * plane], plane 0 '+', plane 1 '-')."""
        return self.torch.zeros(self.coverage_elems(), dtype=self.torch.int32, device=self.device)

    def set_layout(self, layout: str):
        """'dense' = genome-wide planes (default; WIG / metagene need it); 'compact' = exon union of the
        index only (``rt_set_layout``): same scores, a 13x smaller buffer for the human index."""
        self._check(self.lib.rt_set_layout(self.ctx, {"dense": 0, "compact": 1}[layout]))
        self.layout = layout

    def ensure_dense(self):
        """Back to the genome-wide planes (a no-op when they are the current layout)."""
        if getattr(self, "layout", "dense") != "dense":
            self.set_layout("dense")

    def coverage_elems(self) -> int:
        return int(self.lib.rt_coverage_elems(self.ctx))

    def clear_coverage(self, cov):
        self._check(self.lib.rt_clear_coverage(self.ctx, C.c_void_p(cov.data_ptr()), self._stream()))

    def track_touched(self, enable: bool = True):
        """Make K1 remember the slots it bumps, so ``clear_touched`` can zero just those."""
        self._check(self.lib.rt_track_touched(self.ctx, int(enable)))

    def clear_touched(self, cov):
        """Sparse clear of a recycled coverage buffer (see ``rt_clear_touched``)."""
        self._check(self.lib.rt_clear_touched(self.ctx, C.c_void_p(cov.data_ptr()), self._stream()))

    # ---------------------------------------------------------------- index
    def set_index(self, exon_ptr, exon_start, exon_end, orf_contig, orf_strand):
        exon_ptr = np.ascontiguousarray(exon_ptr, np.int64)
        exon_start = np.ascontiguousarray(exon_start, np.int32)
        exon_end = np.ascontiguousarray(exon_end, np.int32)
        orf_contig = np.ascontiguousarray(orf_contig, np.int32)
        orf_strand = np.ascontiguousarray(orf_strand, np.uint8)
        n = len(orf_contig)
        if len(exon_ptr) != n + 1 or len(orf_strand) != n or len(exon_start) != len(exon_end) \
                or (n and exon_ptr[-1] != len(exon_start)):
            raise ValueError("inconsistent CSR index arrays")
        self._check(self.lib.rt_set_index(self.ctx, n, _np_ptr(exon_ptr), _np_ptr(exon_start), _np_ptr(exon_end),
                                          _np_ptr(orf_contig), _np_ptr(orf_strand)))
        self.n_orf = n
        self.layout = "dense"
        self._resident_index = None

    def score_bytes(self, lo: int = 0, hi: int | None = None) -> int:
        hi = self.n_orf if hi is None else hi
        return int(self.lib.rt_index_score_bytes(self.ctx, lo, hi))

    def total_nt(self, lo: int = 0, hi: int | None = None) -> int:
        hi = self.n_orf if hi is None else hi
        return int(self.lib.rt_index_total_nt(self.ctx, lo, hi))

    def shard_bounds(self, n_shards: int) -> np.ndarray:
        b = np.zeros(n_shards + 1, np.int64)
        self._check(self.lib.rt_shard_bounds(self.ctx, int(n_shards), _np_ptr(b)))
        return b

    # ------------------------------------------------------------------- K1
    def upload_reads(self, cols: dict) -> dict:
        """Host columns -> device tensors (plumbing only)."""
        t = self.torch
        out = {}
        for name, dt in READ_COLUMNS:
            a = np.ascontiguousarray(cols[name], dtype=dt)
            # torch has no uint16 arithmetic but can hold the bytes; view as int16 for transport
            if dt == np.uint16:
                out[name] = t.from_numpy(a.view(np.int16)).to(self.device)
            else:
                out[name] = t.from_numpy(a).to(self.device)
        return out

    def new_bin_accumulators(self):
        t = self.torch
        return (t.zeros(_lib.RT_N_STATS, dtype=t.int64, device=self.device),
                t.zeros(_lib.RT_LEN_TABLE, dtype=t.int64, device=self.device))

    def bin_reads_device(self, cov, dcols: dict, protocol, stats, len_counts, sorted_hint: bool = False,
                         n: int | None = None, weight: int = 1):
        """Enqueue K1 on device-resident read columns (no host sync).  ``weight=-1`` takes the same
        reads out again (coverage, stats and length counts return to their previous values)."""
        n = int(dcols["ref_id"].numel()) if n is None else int(n)
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        self._check(self.lib.rt_bin_reads(
            self.ctx, p(cov), n, p(dcols["ref_id"]), p(dcols["first"]), p(dcols["last"]), p(dcols["mlen"]),
            p(dcols["flag"]), p(dcols["mapq"]), p(dcols["nh"]), protocol_code(protocol), int(sorted_hint),
            int(weight), p(stats), p(len_counts), self._stream()))

    def bin_reads_host(self, cov, cols: dict, protocol, sorted_hint: bool = False):
        """K1 on HOST read columns (numpy or pinned torch CPU tensors): chunked H2D inside the call.

        Returns ``(stats: dict, read_length_counts: np.ndarray[RT_LEN_TABLE])``.
        """
        ptrs, keep = [], []
        n = None
        for name, dt in READ_COLUMNS:
            a = cols[name]
            if hasattr(a, "data_ptr"):   # torch CPU tensor (possibly pinned)
                if a.is_cuda or not a.is_contiguous() or a.element_size() != np.dtype(dt).itemsize:
                    raise ValueError(f"column {name}: need a contiguous CPU tensor of {np.dtype(dt).itemsize}-byte items")
                ptrs.append(C.c_void_p(a.data_ptr()))
                m = a.numel()
            else:
                a = np.ascontiguousarray(a, dtype=dt)
                ptrs.append(_np_ptr(a))
                m = len(a)
            keep.append(a)
            if n is None:
                n = m
            elif n != m:
                raise ValueError("read columns differ in length")
        stats = np.zeros(_lib.RT_N_STATS, np.int64)
        len_counts = np.zeros(_lib.RT_LEN_TABLE, np.int64)
        self.torch.cuda.current_stream(self.device).synchronize()   # cov may have pending work on torch's stream
        self._check(self.lib.rt_bin_reads_host(self.ctx, C.c_void_p(cov.data_ptr()), int(n), *ptrs,
                                               protocol_code(protocol), int(sorted_hint), _np_ptr(stats),
                                               _np_ptr(len_counts)))
        return dict(zip(_lib.ST_NAMES, stats.tolist())), len_counts

    def pack_reads(self, cols: dict, pinned: bool = False, max_runs: int | None = None) -> dict:
        """Packed read records for ``bin_reads_packed_host`` (``rt_pack_read_meta``): 11 B/read instead of
        18.  ``first/last/mlen`` are reused as they are; ``flag/mapq/nh`` collapse into one ``meta`` byte
        (filter cascade decided on the host) and ``ref_id`` into a run table.  Raises when the reads are
        not grouped by reference (more than ``max_runs`` runs)."""
        t = self.torch
        host = {}
        for name, dt in READ_COLUMNS:
            v = cols[name]
            if hasattr(v, "cpu"):                       # torch tensor (16-bit columns are stored as int16)
                v = v.cpu().numpy()
                if v.dtype.itemsize == np.dtype(dt).itemsize and v.dtype != dt:
                    v = v.view(dt)
            host[name] = np.ascontiguousarray(v, dt)
        n = len(host["ref_id"])
        cap = int(max_runs if max_runs is not None else max(64, 4 * len(self.contig_len) + 8))
        meta = np.empty(n, np.uint8)
        run_start = np.zeros(cap + 1, np.int64)
        run_ref = np.zeros(cap, np.int32)
        n_runs = C.c_int64(0)
        rc = self.lib.rt_pack_read_meta(n, _np_ptr(host["ref_id"]), _np_ptr(host["flag"]), _np_ptr(host["mapq"]),
                                        _np_ptr(host["nh"]), _np_ptr(meta), cap, _np_ptr(run_start), _np_ptr(run_ref),
                                        C.byref(n_runs))
        if rc != 0:
            raise _lib.RtError(self.lib.rt_io_last_error().decode() or f"rt_pack_read_meta failed ({rc})")
        k = int(n_runs.value)
        out = dict(first=host["first"], last=host["last"], mlen=host["mlen"], meta=meta)
        if pinned:
            out = {name: t.from_numpy(np.ascontiguousarray(a)).pin_memory() for name, a in out.items()}
        out["run_start"] = np.ascontiguousarray(run_start[:k + 1])
        out["run_ref"] = np.ascontiguousarray(run_ref[:k])
        out["n"] = n
        return out

    def upload_packed(self, packed: dict) -> dict:
        """Packed host records (``pack_reads``) -> device tensors, run table included (plumbing only)."""
        t = self.torch

        def dev(a):
            if hasattr(a, "data_ptr"):
                return a.to(self.device)
            a = np.ascontiguousarray(a)
            return t.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).to(self.device)

        out = {k: dev(packed[k]) for k in ("first", "last", "mlen", "meta", "run_start", "run_ref")}
        out["n"] = int(packed["n"])
        return out

    def bin_reads_packed_device(self, cov, dpacked: dict, protocol, stats, len_counts, weight: int = 1):
        """Enqueue K1 on device-resident PACKED records (11 B/read; no host sync)."""
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        self._check(self.lib.rt_bin_reads_packed(
            self.ctx, p(cov), int(dpacked["n"]), p(dpacked["first"]), p(dpacked["last"]), p(dpacked["mlen"]),
            p(dpacked["meta"]), 0, int(dpacked["run_ref"].numel()), p(dpacked["run_start"]), p(dpacked["run_ref"]),
            protocol_code(protocol), int(weight), p(stats), p(len_counts), self._stream()))

    def bin_reads_packed_host(self, cov, packed: dict, protocol):
        """K1 on packed HOST records (see ``pack_reads``): chunked H2D of 11 B/read inside the call.
        Returns ``(stats, read_length_counts)`` exactly like ``bin_reads_host``."""
        def ptr(a):
            return C.c_void_p(a.data_ptr()) if hasattr(a, "data_ptr") else _np_ptr(a)

        stats = np.zeros(_lib.RT_N_STATS, np.int64)
        len_counts = np.zeros(_lib.RT_LEN_TABLE, np.int64)
        self.torch.cuda.current_stream(self.device).synchronize()
        self._check(self.lib.rt_bin_reads_packed_host(
            self.ctx, C.c_void_p(cov.data_ptr()), int(packed["n"]), ptr(packed["first"]), ptr(packed["last"]),
            ptr(packed["mlen"]), ptr(packed["meta"]), len(packed["run_ref"]), _np_ptr(packed["run_start"]),
            _np_ptr(packed["run_ref"]), protocol_code(protocol), _np_ptr(stats), _np_ptr(len_counts)))
        return dict(zip(_lib.ST_NAMES, stats.tolist())), len_counts

    def stream_reads(self, cols: dict, pinned: bool = False, n_threads: int = 0) -> dict:
        """A coordinate-sorted library as the 4 B/read record stream of ``rt_stream_pack`` (blocks of 256 delta-coded
        records; the raw filter bits travel with every read and the cascade runs on the device).  Raises ``RtError``
        when the library cannot be coded (not sorted): use the column entry points then."""
        t = self.torch
        host = {}
        for name, dt in READ_COLUMNS:
            v = cols[name]
            if hasattr(v, "cpu"):                       # torch tensor (16-bit columns are stored as int16)
                v = v.cpu().numpy()
                if v.dtype.itemsize == np.dtype(dt).itemsize and v.dtype != dt:
                    v = v.view(dt)
            host[name] = np.ascontiguousarray(v, dt)
        n = len(host["ref_id"])
        ptrs = [_np_ptr(host[name]) for name, _ in READ_COLUMNS]
        n_blocks = C.c_int64(0)
        rc = self.lib.rt_stream_pack(n, *ptrs, int(n_threads), 0, None, None, C.byref(n_blocks))
        if rc != 0:
            raise _lib.RtError(self.lib.rt_io_last_error().decode() or f"rt_stream_pack failed ({rc})")
        nb = int(n_blocks.value)
        if pinned:
            rec = t.empty(max(nb, 1) * _lib.RT_STREAM_BLOCK, dtype=t.int32).pin_memory()
            hdr = t.empty(max(nb, 1) * 4, dtype=t.int32).pin_memory()
            rp, hp = C.c_void_p(rec.data_ptr()), C.c_void_p(hdr.data_ptr())
        else:
            rec = np.empty(max(nb, 1) * _lib.RT_STREAM_BLOCK, np.uint32)
            hdr = np.empty(max(nb, 1) * 4, np.int32)
            rp, hp = _np_ptr(rec), _np_ptr(hdr)
        rc = self.lib.rt_stream_pack(n, *ptrs, int(n_threads), nb, rp, hp, C.byref(n_blocks))
        if rc != 0:
            raise _lib.RtError(self.lib.rt_io_last_error().decode() or f"rt_stream_pack failed ({rc})")
        return dict(records=rec, hdr=hdr, n_blocks=nb, n=n)

    def upload_stream(self, stream: dict) -> dict:
        """Host record stream (``stream_reads``) -> device tensors (plumbing only)."""
        t = self.torch

        def dev(a):
            if hasattr(a, "data_ptr"):
                return a.to(self.device)
            return t.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(self.device)

        return dict(records=dev(stream["records"]), hdr=dev(stream["hdr"]), n_blocks=int(stream["n_blocks"]), n=int(stream["n"]))

    def bin_stream_device(self, cov, dstream: dict, protocol, stats, len_counts, weight: int = 1, fresh: bool = False):
        """Enqueue K1 on a device-resident record stream (4 B/read; no host sync).  ``fresh=True`` (compact layout):
        the call overwrites the whole buffer zone by zone (``rt_bin_stream_fresh``), so ``cov`` need not be cleared."""
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        if fresh:
            if weight != 1:
                raise ValueError("fresh binning adds the library once (weight 1)")
            self._check(self.lib.rt_bin_stream_fresh(
                self.ctx, p(cov), int(dstream["n_blocks"]), p(dstream["records"]), p(dstream["hdr"]),
                protocol_code(protocol), p(stats), p(len_counts), self._stream()))
            return
        self._check(self.lib.rt_bin_stream(
            self.ctx, p(cov), int(dstream["n_blocks"]), p(dstream["records"]), p(dstream["hdr"]),
            protocol_code(protocol), int(weight), p(stats), p(len_counts), self._stream()))

    def bin_stream_host(self, cov, stream: dict, protocol):
        """K1 on a HOST record stream (see ``stream_reads``): chunked H2D of 4 B/read inside the call.
        Returns ``(stats, read_length_counts)`` exactly like ``bin_reads_host``."""
        def ptr(a):
            return C.c_void_p(a.data_ptr()) if hasattr(a, "data_ptr") else _np_ptr(a)

        stats = np.zeros(_lib.RT_N_STATS, np.int64)
        len_counts = np.zeros(_lib.RT_LEN_TABLE, np.int64)
        self.torch.cuda.current_stream(self.device).synchronize()
        self._check(self.lib.rt_bin_stream_host(
            self.ctx, C.c_void_p(cov.data_ptr()), int(stream["n_blocks"]), ptr(stream["records"]), ptr(stream["hdr"]),
            protocol_code(protocol), _np_ptr(stats), _np_ptr(len_counts)))
        return dict(zip(_lib.ST_NAMES, stats.tolist())), len_counts

    # ---------------------------------------------------------------- K2+K3
    def new_score_columns(self, n: int, diagnostics: bool = False, min_codon: bool | None = None) -> dict:
        """Device result columns.  ``min_codon`` (the minimum codon sum, an extra the reference never
        prints) is only produced on request or with ``diagnostics``."""
        t = self.torch
        d = self.device
        cols = dict(score=t.empty(n, dtype=t.float64, device=d), valid=t.empty(n, dtype=t.int32, device=d),
                    count=t.empty(n, dtype=t.int64, device=d), length=t.empty(n, dtype=t.int32, device=d),
                    status=t.empty(n, dtype=t.uint8, device=d))
        if min_codon or (min_codon is None and diagnostics):
            cols["min_codon"] = t.empty(n, dtype=t.int32, device=d)
        if diagnostics:
            cols["frame_K"] = t.empty((n, 3), dtype=t.int32, device=d)
            cols["frame_s"] = t.empty((n, 3), dtype=t.float64, device=d)
        return cols

    def score_device(self, cov, out: dict, lo: int = 0, hi: int | None = None, params: ScoreParams | None = None):
        """Enqueue the fused gather+score kernel; ``out`` are device columns (no host sync)."""
        hi = self.n_orf if hi is None else hi
        prm = (params or ScoreParams()).as_c()
        o = _lib.ScoreOut(*[C.c_void_p(out[k].data_ptr()) if k in out else None
                            for k in ("score", "valid", "count", "length", "min_codon", "status", "frame_K", "frame_s")])
        self._check(self.lib.rt_score(self.ctx, C.c_void_p(cov.data_ptr()), int(lo), int(hi), C.byref(prm),
                                      C.byref(o), self._stream()))

    def new_host_score_columns(self, n: int, diagnostics: bool = False, min_codon: bool = False) -> dict:
        """Page-locked HOST result columns for ``score_host(..., out=...)``: the D2H copies inside
        ``rt_score_host`` then run at full PCIe speed instead of being staged through pageable memory."""
        t = self.torch
        spec = dict(score=(t.float64, ()), valid=(t.int32, ()), count=(t.int64, ()), length=(t.int32, ()),
                    status=(t.uint8, ()))
        if min_codon or diagnostics:
            spec["min_codon"] = (t.int32, ())
        if diagnostics:
            spec["frame_K"] = (t.int32, (3,))
            spec["frame_s"] = (t.float64, (3,))
        return {k: t.empty((n,) + shape, dtype=dt).pin_memory().numpy() for k, (dt, shape) in spec.items()}

    def score_host(self, cov, lo: int = 0, hi: int | None = None, params: ScoreParams | None = None,
                   diagnostics: bool = False, min_codon: bool | None = None, out: dict | None = None) -> dict:
        """Score ORFs [lo, hi) and return HOST numpy columns (D2H inside the C call).  ``min_codon``
        (minimum codon sum, not a reference output) is produced on request or with ``diagnostics``.
        ``out`` (from ``new_host_score_columns``) is filled and returned instead of fresh arrays."""
        hi = self.n_orf if hi is None else hi
        n = hi - lo
        if out is not None:
            for k in ("score", "valid", "count", "length"):
                if k not in out:
                    raise ValueError(f"out lacks the required column {k!r}")
            for k, a in out.items():
                if len(a) != n or not a.flags["C_CONTIGUOUS"]:
                    raise ValueError(f"out[{k!r}] must be a contiguous array of {n} rows")
        else:
            out = dict(score=np.empty(n, np.float64), valid=np.empty(n, np.int32), count=np.empty(n, np.int64),
                       length=np.empty(n, np.int32), status=np.empty(n, np.uint8))
            if min_codon or (min_codon is None and diagnostics):
                out["min_codon"] = np.empty(n, np.int32)
            if diagnostics:
                out["frame_K"] = np.empty((n, 3), np.int32)
                out["frame_s"] = np.empty((n, 3), np.float64)
        prm = (params or ScoreParams()).as_c()
        o = _lib.ScoreOut(*[_np_ptr(out[k]) if k in out else None
                            for k in ("score", "valid", "count", "length", "min_codon", "status", "frame_K", "frame_s")])
        self.torch.cuda.current_stream(self.device).synchronize()
        self._check(self.lib.rt_score_host(self.ctx, C.c_void_p(cov.data_ptr()), int(lo), int(hi), C.byref(prm),
                                           C.byref(o)))
        return out

    # ----------------------------------------------- dense planes -> compact buffer, covered positions
    def compact_from_dense(self, dense_cov, compact_cov):
        """Copy the slots the resident index reads from genome-wide planes into a compact-layout buffer
        (``rt_compact_from_dense``; enqueued, no host sync)."""
        self._check(self.lib.rt_compact_from_dense(self.ctx, C.c_void_p(dense_cov.data_ptr()),
                                                   C.c_void_p(compact_cov.data_ptr()), self._stream()))

    def nonzero_slots(self, cov, lo: int, n: int):
        """Non-zero slots of ``cov[lo:lo+n]`` in slot order -> (slot numbers relative to ``lo``, counts) on the host
        (``rt_wig_count`` / ``rt_wig_fill``: tile counts, an exclusive prefix on the host, ordered compaction)."""
        t = self.torch
        n_tiles = int(self.lib.rt_wig_tiles(int(n)))
        if n_tiles == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.int32)
        base = C.c_void_p(cov.data_ptr() + 4 * int(lo))
        d_counts = t.empty(n_tiles, dtype=t.int32, device=self.device)
        self._check(self.lib.rt_wig_count(self.ctx, base, int(n), C.c_void_p(d_counts.data_ptr()), self._stream()))
        counts = d_counts.cpu().numpy().view(np.uint32).astype(np.int64)
        offsets = np.zeros(n_tiles + 1, np.int64)
        np.cumsum(counts, out=offsets[1:])
        total = int(offsets[-1])
        if total == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.int32)
        d_off = t.from_numpy(offsets[:-1].copy()).to(self.device)
        d_slot = t.empty(total, dtype=t.int64, device=self.device)
        d_val = t.empty(total, dtype=t.int32, device=self.device)
        self._check(self.lib.rt_wig_fill(self.ctx, base, int(n), C.c_void_p(d_off.data_ptr()), C.c_void_p(d_slot.data_ptr()),
                                         C.c_void_p(d_val.data_ptr()), self._stream()))
        return d_slot.cpu().numpy(), d_val.cpu().numpy()

    # ------------------------------------------------------------------- K4
    def gather_profiles(self, cov, orf_ids, lengths):
        """Profiles of the selected ORFs: returns ``(out_ptr, flat int32 profiles)`` on the host."""
        t = self.torch
        orf_ids = np.ascontiguousarray(orf_ids, np.int64)
        lengths = np.ascontiguousarray(lengths, np.int64)
        out_ptr = np.zeros(len(orf_ids) + 1, np.int64)
        np.cumsum(lengths, out=out_ptr[1:])
        total = int(out_ptr[-1])
        if len(orf_ids) == 0:
            return out_ptr, np.zeros(0, np.int32)
        d_ids = t.from_numpy(orf_ids).to(self.device)
        d_ptr = t.from_numpy(out_ptr).to(self.device)
        d_out = t.empty(max(total, 1), dtype=t.int32, device=self.device)
        self._check(self.lib.rt_gather_profiles(self.ctx, C.c_void_p(cov.data_ptr()), len(orf_ids),
                                                C.c_void_p(d_ids.data_ptr()), C.c_void_p(d_ptr.data_ptr()),
                                                C.c_void_p(d_out.data_ptr()), self._stream()))
        return out_ptr, d_out[:total].cpu().numpy()

    # --------------------------------------------------------------- prepare-orfs
    def orf_search(self, codes, tx_base, exon_ptr, exon_start, exon_end, tx_strand, tx_cds, start_mask: int,
                   stop_mask: int, min_orf_length: int, longest: bool, stage_ms: np.ndarray | None = None) -> dict:
        """Candidate ORFs of every transcript (``rt_orf_search`` + ``rt_orf_fetch``): HOST columns ``row_tx``,
        ``row_start`` / ``row_stop`` (the oriented range [start, stop) in the transcript), ``row_type``, ``row_codon``
        and the genomic intervals as CSR ``iv_ptr`` / ``iv_start`` / ``iv_end``, rows by transcript, then start."""
        arr = lambda a, dt: np.ascontiguousarray(a, dt)  # noqa: E731
        codes, tx_base, exon_ptr = arr(codes, np.uint8), arr(tx_base, np.int64), arr(exon_ptr, np.int64)
        exon_start, exon_end = arr(exon_start, np.int32), arr(exon_end, np.int32)
        tx_strand, tx_cds = arr(tx_strand, np.uint8), arr(tx_cds, np.int32)
        q = _lib.OrfQuery(len(tx_base), _np_ptr(exon_ptr), _np_ptr(exon_start), _np_ptr(exon_end), _np_ptr(tx_base),
                          _np_ptr(tx_strand), _np_ptr(tx_cds), _np_ptr(codes), len(codes), int(start_mask),
                          int(stop_mask), int(min_orf_length), int(bool(longest)))
        n_rows, n_iv = C.c_int64(0), C.c_int64(0)
        ms = np.zeros(_lib.RT_ORF_STAGES, np.float32)
        self._check(self.lib.rt_orf_search(self.ctx, C.byref(q), C.byref(n_rows), C.byref(n_iv), _np_ptr(ms)))
        if stage_ms is not None:
            stage_ms[:] = ms
        n, m = int(n_rows.value), int(n_iv.value)
        out = dict(row_tx=np.empty(n, np.int32), row_start=np.empty(n, np.int32), row_stop=np.empty(n, np.int32),
                   row_type=np.empty(n, np.uint8), row_codon=np.empty(n, np.uint8), iv_ptr=np.empty(n + 1, np.int64),
                   iv_start=np.empty(m, np.int32), iv_end=np.empty(m, np.int32))
        self._check(self.lib.rt_orf_fetch(self.ctx, *[_np_ptr(out[k]) for k in (
            "row_tx", "row_start", "row_stop", "row_type", "row_codon", "iv_ptr", "iv_start", "iv_end")]))
        return out
