#!/usr/bin/env python
"""Benchmark of the detect-orfs scoring path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" is one pass of the hot path over one synthetic Ribo-seq library:
K1 bin P-sites -> K2+K3 gather+score every candidate ORF -> clear of the resident
coverage buffer for the next library.  At N=1 the workload is BASELINE.json
configs[1] (human GENCODE-scale: 2.5 M candidate ORFs, 100 M reads).  At N>1 it is
configs[2] (10 M candidate ORFs, 500 M reads, "ORF-sharded at 1/2/4/8 B200"): ONE
index, cut into byte-balanced blocks along the genome (multi_gpu.shard_plan); rank r
holds block r as its resident index, bins the slice of the coordinate-sorted library
that can reach the block and scores it -> strong scaling, no collective on the data
path (north_star item 4).  `--config` overrides the workload at any N.

`value` is ORFs scored per second with all inputs resident in HBM; `e2e` is the
same metric through the host-buffer C-ABI calls (pinned host read columns in,
host result columns out, all copies inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "candidate ORFs scored/sec (P-site binning + gather + phase score + filters)"
UNIT = "ORFs/s"


def workload_text(name: str, n_orf: int, n_reads: int) -> str:
    """The same words in both arms (ours and --impl reference): the driver compares the configs."""
    return (f"{name}: synthetic human GENCODE-scale detect-orfs, ONE index of {n_orf} candidate ORFs and ONE library of "
            f"{n_reads} reads (coordinate-sorted, lengths 26-32), default thresholds (cutoff 0.428571428571, "
            f"min_valid_codons 5, the other filters at their 0 defaults)")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, help="C1..C5; default C2 at N=1, C3 at N>1")
    ap.add_argument("--index-order", default="genome", choices=["genome", "random"],
                    help="row order of the synthetic index (random = the round-1 generator, for A/B runs)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink ORF/read counts (debugging only)")
    ap.add_argument("--contig-scale", type=float, default=1.0, help="shrink contigs (debugging only)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--libraries", type=int, default=64, help="--config C4: libraries in the batch")
    ap.add_argument("--distinct", type=int, default=4, help="--config C4: distinct libraries generated (cycled through)")
    ap.add_argument("--min-reads-per-codon", type=float, default=0.0,
                    help="--min_reads_per_codon of the scoring step (> 0 selects the kernels that also carry per-frame minima)")
    ap.add_argument("--reads-format", default="stream", choices=["stream", "columns"],
                    help="resident library of the device-timed step: the 4 B/read record stream (rt_bin_stream, default) or the "
                         "decoder's 18 B/read columns (rt_bin_reads)")
    ap.add_argument("--k1", default="fresh", choices=["fresh", "red"],
                    help="K1 of the device-timed step on the record stream: rt_bin_stream_fresh (zones: the call overwrites the "
                         "buffer, the step has no clear) or rt_bin_stream into a buffer the step clears (A/B)")
    ap.add_argument("--layout", default="compact", choices=["compact", "dense"],
                    help="coverage layout: exon union of the index (default) or genome-wide planes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result columns of the last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no per-ORF results")
    return args


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, device_index: int, period_s: float = 0.002):
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self.period = period_s
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = device_index
            if visible:
                try:
                    phys = int(visible.split(",")[device_index])
                except ValueError:
                    phys = device_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as exc:   # pragma: no cover - depends on the box
            self.nv = None
            self.err = str(exc)

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------- CPU baseline
def _cpu_worker(args):
    """Score a slice of ORFs exactly like the body of export_orf_coverages (detect_orfs.py:274-299)
    with the SciPy call of statistics.py:101-107 (oracle_py.phasescore_scipy)."""
    orfs, merged = args
    if merged is None:
        merged = _CPU_MERGED        # inherited through fork(): the coverage dict is not pickled once per slice
    from oracle import oracle_py as O

    n = 0
    for chrom, strand, ivs in orfs:
        cov = O.orf_profile(chrom, strand, ivs, merged)
        O.score_profile(cov, scorer=O.phasescore_scipy)
        n += 1
    return n


_CPU_MERGED = None


def cpu_reference_run(config_name: str, seconds: float, cores: int | None = None, steps: int = 1):
    """The reference's CPU path (faithful port: same SciPy call) on a bounded sample of the workload.

    The sample is the same synthetic configuration generated at a small scale (same genome, same
    ORF-length and reads-per-ORF distributions), scored with all host cores by multiprocessing
    over ORF slices -- the reference itself is single-process (SURVEY.md 2.1).
    Returns (ORFs/s per step list, description dict).
    """
    import multiprocessing as mp

    from oracle import oracle_py as O
    from ribotricer_b200 import synth

    cores = cores or os.cpu_count() or 1
    # ~21 ORFs/s/core for the reference (SURVEY.md section 6): at least 2,000 ORFs per step, more when the budget allows
    per_step_target = int(max(2000, min(20000, seconds * cores * 15)))
    n_sample = per_step_target * max(1, steps)
    full = synth.config(config_name)
    scale = n_sample / full.n_orf
    cfg = synth.config(config_name, scale)
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, device="cpu"))
    aln, _, _ = O.split_reads(reads, "forward", None, idx.contig_names)
    merged = O.merge_read_lengths(aln, synth.TRUE_OFFSETS)
    merged = {s: dict(t) for s, t in merged.items()}
    global _CPU_MERGED
    _CPU_MERGED = merged
    orfs = []
    for o in range(idx.n_orf):
        a, b = idx.exon_ptr[o], idx.exon_ptr[o + 1]
        orfs.append((idx.contig_names[idx.orf_contig[o]], "+" if idx.orf_strand[o] == 0 else "-",
                     list(zip(idx.exon_start[a:b].tolist(), idx.exon_end[a:b].tolist()))))
    per_step = max(cores, len(orfs) // max(1, steps))
    # how the reference really runs: one process, one thread (SURVEY.md 2.1), on a small slice of the same sample
    single_n = min(len(orfs), 150)
    t0 = time.perf_counter()
    _cpu_worker((orfs[:single_n], merged))
    single_rate = single_n / (time.perf_counter() - t0)
    rates = []
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for s in range(steps):
            chunk = orfs[s * per_step:(s + 1) * per_step] or orfs[:per_step]
            slices = [(chunk[i::cores * 4], None) for i in range(cores * 4)]
            t0 = time.perf_counter()
            done = sum(pool.map(_cpu_worker, slices))
            dt = time.perf_counter() - t0
            rates.append(done / dt)
    import scipy
    desc = {"kind": "port", "cores": cores,
            "single_process": {"value": single_rate, "unit": UNIT, "cores": 1, "sample": f"{single_n} ORFs of the same sample, one "
                               "process: the reference has no parallelism of its own"},
            "sample": f"{per_step} ORFs/step of synthetic {config_name} generated at scale {scale:.2e} "
                      f"({idx.n_orf} ORFs, {len(reads['ref_id'])} reads, mean {idx.orf_len.mean():.0f} nt); "
                      f"oracle_py.phasescore_scipy = the reference's scipy.signal.coherence call "
                      f"(scipy {scipy.__version__}), multiprocessing over ORF slices"}
    return rates, desc


def cpu_closed_form_run(config_name: str, n_orf: int = 200_000):
    """Second CPU line: the C restatement of the same arithmetic (oracle/rt_oracle.c, OpenMP, all
    cores) on a scaled copy of the workload -- a much tougher CPU baseline than the reference."""
    from oracle import c_oracle as CO
    from ribotricer_b200 import synth

    full = synth.config(config_name)
    scale = min(1.0, n_orf / full.n_orf)
    cfg = synth.config(config_name, scale, contig_scale=max(scale, 0.01))
    idx = synth.make_index(cfg)
    reads = synth.reads_to_numpy(synth.make_reads(cfg, idx, device="cpu"))
    pad = 256
    base, plane = CO.genome_layout(idx.contig_len, pad)
    cov, _, _ = CO.bin_reads(reads, 0, CO.make_len_table(synth.TRUE_OFFSETS), base, idx.contig_len, pad, plane)
    t0 = time.perf_counter()
    CO.score(idx.as_dict(), cov, base, idx.contig_len, pad, plane, [0.428571428571, 5, 0, 0, 0.0],
             diagnostics=False)
    dt = time.perf_counter() - t0
    return {"value": idx.n_orf / dt, "unit": UNIT, "cores": CO.lib().orc_max_threads(), "kind": "port (closed form, C+OpenMP)",
            "sample": f"{idx.n_orf} ORFs of synthetic {config_name} at scale {scale:.2e}, contigs shrunk to fit host RAM"}


# --------------------------------------------------------------------------- --dump-outputs
DUMP_ROWS = 1_000_000   # ORFs written at most: six float64 files of this length stay under 64 MB


def dump_outputs(out_dir: str, cols: dict, rows: np.ndarray, n_total: int, suffix: str = ""):
    """Write the per-ORF result columns (score, valid, count, length, status) of the last timed step as float64
    ``out_dir/<name><suffix>.npy``, with ``orf_index`` = the index row of each value.  ``rows`` are the index rows of
    ``cols``.  An index of more than DUMP_ROWS ORFs is sampled: the same rows (seed 0) for every build and rank count,
    so that two builds can be compared value for value."""
    os.makedirs(out_dir, exist_ok=True)
    if n_total > DUMP_ROWS:
        keep = np.sort(np.random.default_rng(0).choice(n_total, DUMP_ROWS, replace=False))
        pick = np.flatnonzero(np.isin(rows, keep))
    else:
        pick = np.arange(len(rows))
    arrays = {k: cols[k] for k in ("score", "valid", "count", "length", "status")}
    arrays["orf_index"] = rows
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), np.asarray(a)[pick].astype(np.float64))


# --------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ribotricer_b200 import synth

    cores = os.cpu_count() or 1
    total_steps = args.steps + args.warmup
    budget = 150.0   # whole run within a few minutes
    rates, desc = cpu_reference_run(args.config, budget / max(1, total_steps) * 1.0, cores, steps=total_steps)
    timed = rates[args.warmup:] or rates
    value = float(len(timed) / sum(1.0 / r for r in timed))   # harmonic mean = total ORFs / total time
    per_step = int(desc["sample"].split(" ORFs/step")[0])
    ms_per_step = 1e3 * per_step / value
    full = synth.config(args.config)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(args.config, full.n_orf, full.n_reads), "orfs": full.n_orf, "reads": full.n_reads,
                   "sample": "bounded sample of this workload per step, see cpu_baseline.sample"},
        "cpu_baseline": dict(desc, value=value, unit=UNIT),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from ribotricer_b200 import synth
    from ribotricer_b200.engine import READ_BYTES, Engine, ScoreParams

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:     # the ranks of one box share its host cores: the coding pipelines of rt_bin_reads_host split them
        os.environ.setdefault("RT_PACK_PIPES", str(max(2, (os.cpu_count() or 16) // world)))

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    # ---- workload: ONE index and ONE library; this rank's genomic block of the index and its slice of the reads
    from ribotricer_b200 import multi_gpu

    cfg = synth.config(args.config, args.scale, args.contig_scale)
    cfg.genome_order = args.index_order == "genome"
    idx = synth.make_index(cfg)
    plan = multi_gpu.shard_plan(idx.exon_ptr, idx.exon_start, idx.exon_end, idx.orf_contig, world)
    shard = plan[rank]
    eng = Engine(local)
    eng.set_genome(idx.contig_names, idx.contig_len)
    eng.set_length_table(synth.TRUE_OFFSETS, None)
    eng.set_index(**multi_gpu.sub_index(idx.as_dict(), shard.rows))
    dreads = synth.make_reads(cfg, idx, device=dev)
    n_reads_total = int(dreads["ref_id"].numel())
    if world > 1:   # the slices of the coordinate-sorted library that can reach this block (multi_gpu.read_slices, on the device)
        reach = max(synth.TRUE_OFFSETS.values()) + int((dreads["last"].long() - dreads["first"].long()).max().item())
        key = dreads["ref_id"].long() * (1 << 32) + dreads["first"].long()
        keep = torch.zeros(n_reads_total, dtype=torch.bool, device=dev)
        for c, lo, hi in shard.spans:
            a = int(torch.searchsorted(key, torch.tensor(c * (1 << 32) + max(lo - 1 - reach, 0), device=dev), right=False))
            b = int(torch.searchsorted(key, torch.tensor(c * (1 << 32) + hi + max(synth.TRUE_OFFSETS.values()), device=dev), right=True))
            keep[a:b] = True
        dreads = {k: v[keep].contiguous() for k, v in dreads.items()}
        del key, keep
        torch.cuda.empty_cache()
    n_reads = int(dreads["ref_id"].numel())
    # host columns exactly as a BAM decoder produces them (18 B/read: ref_id, first, last, mlen, flag, mapq, nh), page-locked
    hreads = {k: v.cpu().pin_memory() for k, v in dreads.items()}
    use_stream = args.reads_format == "stream" and args.layout == "compact"
    hstream = dstream = None
    use_fresh = use_stream and args.k1 == "fresh"
    if use_stream:       # the library as a record stream (rt_stream_pack): resident copy for `value`, host copy for e2e_stream
        hstream = eng.stream_reads({k: v.numpy() for k, v in hreads.items()}, pinned=True)
        dstream = eng.upload_stream(hstream)
        del dreads
        dreads = None
        torch.cuda.empty_cache()
    n_orf = len(shard.rows)
    n_orf_total = idx.n_orf
    if args.layout == "compact":
        eng.set_layout("compact")   # coverage over the exon union of the index (scoring needs nothing else)
    else:
        eng.track_touched(True)
    cov = eng.new_coverage()
    stats, len_counts = eng.new_bin_accumulators()
    out = eng.new_score_columns(n_orf)
    params = ScoreParams(min_reads_per_codon=args.min_reads_per_codon)
    score_bytes = eng.score_bytes()
    total_nt = eng.total_nt()
    bin_bytes = 23 * n_reads   # BASELINE.md 4.5: 15 B columns + 8 B RMW per read (we move 18 + 8)
    counts = torch.tensor([n_orf, n_reads, score_bytes], dtype=torch.int64, device=dev)
    if world > 1:
        all_counts = [torch.zeros_like(counts) for _ in range(world)]
        dist.all_gather(all_counts, counts)
        per_rank = [c.tolist() for c in all_counts]
    else:
        per_rank = [counts.tolist()]
    torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def step(events=None):
        if events is not None:
            events[0].record()
        if use_stream:
            eng.bin_stream_device(cov, dstream, "forward", stats, len_counts, fresh=use_fresh)
        else:
            eng.bin_reads_device(cov, dreads, "forward", stats, len_counts, sorted_hint=True)
        if events is not None:
            events[1].record()
        eng.score_device(cov, out, 0, n_orf, params)
        if events is not None:
            events[2].record()
        if not use_fresh:
            eng.clear_touched(cov)      # dense: zero exactly the sectors this library touched; compact: memset
        if events is not None:
            events[3].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = eng.launches
    per_step_events = [[ev() for _ in range(4)] for _ in range(args.steps)]
    t_start, t_end = ev(), ev()
    with ClockSampler(local) as clocks:
        barrier()
        t_start.record()
        for k in range(args.steps):
            step(per_step_events[k])
        t_end.record()
        barrier()
    launches = eng.launches - launches0
    total_ms = t_start.elapsed_time(t_end)
    bin_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in per_step_events]))
    score_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in per_step_events]))
    unbin_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in per_step_events]))
    if not use_fresh:
        assert int(cov.abs().max().item()) == 0, "coverage did not return to zero after the sparse clear"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in out.items()}, np.asarray(shard.rows), n_orf_total,
                     f".rank{rank}" if world > 1 else "")

    # ---- e2e: host buffers in, host buffers out, through the host-buffer C-ABI calls
    # From the decoder's host columns nothing is prepared outside the timed region: rt_bin_reads_host delta-codes every
    # chunk into the 4 B/read record stream on host threads while other chunks are on the wire and K1 runs on the stream.
    del dreads, dstream
    torch.cuda.empty_cache()
    e2e_steps = args.steps
    hout = eng.new_host_score_columns(n_orf)      # pinned result columns, like the pinned read columns
    for _ in range(2):
        eng.clear_touched(cov)
        eng.bin_reads_host(cov, hreads, "forward", sorted_hint=True)
        res = eng.score_host(cov, 0, n_orf, params, out=hout)
    barrier()
    e0, e1 = ev(), ev()
    h2d0 = eng.h2d_bytes
    e0.record()
    for _ in range(e2e_steps):
        eng.clear_touched(cov)
        st_host, _ = eng.bin_reads_host(cov, hreads, "forward", sorted_hint=True)
        res = eng.score_host(cov, 0, n_orf, params, out=hout)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    h2d_step = (eng.h2d_bytes - h2d0) // e2e_steps          # counted by the library from the copies it issued
    # second line: the library handed over as the record stream itself (what rt_stream_pack makes of a decoded BAM once,
    # e.g. for a library that is scored against several indexes): no host packing inside the call
    e2e_stream_ms = None
    if hstream is not None:
        for _ in range(2):
            eng.clear_touched(cov)
            eng.bin_stream_host(cov, hstream, "forward")
            eng.score_host(cov, 0, n_orf, params, out=hout)
        barrier()
        e0.record()
        for _ in range(e2e_steps):
            eng.clear_touched(cov)
            st_stream, _ = eng.bin_stream_host(cov, hstream, "forward")
            eng.score_host(cov, 0, n_orf, params, out=hout)
        e1.record()
        barrier()
        e2e_stream_ms = e0.elapsed_time(e1) / e2e_steps
        assert st_stream == st_host, "record stream and columns disagree"

    score_ms_local, bin_ms_local = score_ms, bin_ms       # the roofline is this rank's kernels over this rank's bytes
    stream_blocks = int(hstream["n_blocks"]) if hstream is not None else 0
    times = torch.tensor([total_ms, e2e_ms, score_ms, bin_ms, unbin_ms, e2e_stream_ms or 0.0], dtype=torch.float64, device=dev)
    blocks_all = torch.tensor([stream_blocks, h2d_step], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(blocks_all, op=dist.ReduceOp.SUM)
    total_ms, e2e_ms, score_ms, bin_ms, unbin_ms, e2e_stream_ms = times.tolist()
    stream_bytes = int(blocks_all[0].item()) * (256 * 4 + 16)
    h2d_total = int(blocks_all[1].item())
    ms_per_step = total_ms / args.steps
    value = n_orf_total / (ms_per_step * 1e-3)          # the whole index, in the time of the slowest rank
    e2e_value = n_orf_total / (e2e_ms * 1e-3)

    if rank == 0:
        achieved = score_bytes / (score_ms_local * 1e-3) / 1e9
        # all ranks together, as counted by the library: 4 B/read for the chunks that crossed as a record stream, 18 B/read
        # for those the plain pipeline shipped
        h2d = h2d_total
        d2h = world * 8 * (9 + 65536) + sum(25 * c[0] for c in per_rank)
        # dram__bytes_read.sum + dram__bytes_write.sum of the scoring kernel from the committed ncu capture
        traffic, traffic_src, bin_traffic = None, None, None
        scan_path = os.environ.get("RT_SCORE_PATH") == "scan"
        kernel_names = ("score_orfs_packed_kernel",) if scan_path else ("atom_pass_kernel", "compose_refs_kernel")
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            same = lambda e: e.get("workload") == args.config and e.get("layout", "dense") == args.layout  # noqa: E731
            if all(same(t[k]) for k in kernel_names) and args.scale == 1.0:
                traffic = sum(t[k]["dram_bytes"] for k in kernel_names)
                traffic_src = "; ".join(sorted({t[k]["source"].split(" (")[0] for k in kernel_names})) + \
                    " (ncu --set full, one launch of each kernel inside bench.py's step)"
            k1_name = "bin_stream_kernel" if use_stream else "bin_psites_kernel"
            if same(t.get(k1_name, {})) and args.scale == 1.0:
                bin_traffic = t[k1_name]["dram_bytes"]
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": workload_text(args.config, n_orf_total, n_reads_total),
                "orfs": n_orf_total, "reads": n_reads_total, "index_order": args.index_order,
                "sharding": f"{world} byte-balanced block(s) of the index along the genome; a rank bins the slice of the "
                            f"sorted library that can reach its block; no replication, no collective",
                "per_rank": [{"orfs": c[0], "reads": c[1], "score_bytes": c[2]} for c in per_rank],
                "l2": "inputs larger than L2 (coverage buffer %.1f GB, %s %.2f GB)" % (
                    cov.numel() * 4 / 1e9, "record stream" if use_stream else "read columns",
                    (stream_blocks * (256 * 4 + 16) if use_stream else READ_BYTES * n_reads) / 1e9),
                "coverage_layout": args.layout, "min_reads_per_codon": args.min_reads_per_codon,
                "resident_library": ("record stream, 4 B/read (rt_stream_pack; raw filter bits per read, cascade on the device), "
                                     "%.2f GB" % (stream_bytes / max(1, world) / 1e9)) if use_stream else "decoder columns, 18 B/read",
                "step": ("bin P-sites (rt_bin_stream_fresh: every block zeroes its zone of the compact buffer and adds its reads, "
                         "so the library overwrites the previous one and the step has no clear) -> gather+score") if use_fresh else
                        ("bin P-sites -> gather+score -> clear (resident coverage back to zero: memset of the compact "
                         "buffer, or sparse clear of the touched sectors of the dense planes)"),
            },
            "reads_binned_per_s": n_reads_total / (ms_per_step * 1e-3),
            "kernels_ms": {"bin_psites": bin_ms, "score_orfs": score_ms, "clear": unbin_ms},
            "roofline": {"bound": "hbm", "kernel": " + ".join(kernel_names) + " (+ fallback launch)", "bin_kernel": "bin_stream_kernel" if use_stream else "bin_psites_kernel", "achieved": achieved,
                         "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "algorithmic_bytes": score_bytes, "peak_source": peak_src,
                         "bin_psites": {"achieved": bin_bytes / (bin_ms_local * 1e-3) / 1e9,
                                        "frac": bin_bytes / (bin_ms_local * 1e-3) / 1e9 / hbm_peak,
                                        "algorithmic_bytes": bin_bytes, "traffic": bin_traffic}},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "path": "Engine.clear_touched + bin_reads_host (rt_bin_reads_host on the decoder's 18 B/read host columns; "
                            "delta-coded to the 4 B/read record stream per chunk on host threads inside the call, overlapped with "
                            "the copies and K1) + score_host (rt_score_host, pinned result columns)",
                    "from_record_stream": None if not e2e_stream_ms else {
                        "value": n_orf_total / (e2e_stream_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_stream_ms,
                        "path": "Engine.clear_touched + bin_stream_host (rt_bin_stream_host on a host record stream made once "
                                "by rt_stream_pack) + score_host"}},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "translating": int(res["status"].sum()), "valid_reads": st_host["valid"],
        }
        if world > 1 and args.scale == 1.0:
            # The N > 1 runs split ONE C3 library; the default N = 1 run is C2 (the configuration the metric is quoted on),
            # so value(N) / value(1) of the default lines compares two workloads.  The single-GPU figure of THIS workload,
            # measured separately with `python bench.py --config <this>` and committed under profiles/, travels with the line.
            try:
                one = json.load(open(os.path.join(ROOT, "profiles", f"r2_bench_{args.config}_n1.json")))
                if one.get("n_gpus") == 1 and one["config"]["orfs"] == n_orf_total and one["config"]["reads"] == n_reads_total:
                    line["same_workload_n1"] = {
                        "value": one["value"], "unit": one["unit"], "ms_per_step": one["ms_per_step"],
                        "e2e_ms_per_step": one["e2e"]["ms_per_step"],
                        "e2e_from_record_stream_ms_per_step": (one["e2e"].get("from_record_stream") or {}).get("ms_per_step"),
                        "source": f"profiles/r2_bench_{args.config}_n1.json (python bench.py --config {args.config} on one B200, "
                                  f"an earlier run: not measured in this process)"}
            except Exception:
                pass
        if world == 1 and not args.no_cpu_baseline:
            try:
                rates, desc = cpu_reference_run(args.config, args.cpu_seconds)
                line["cpu_baseline"] = dict(desc, value=float(rates[0]), unit=UNIT)
                line["cpu_closed_form"] = cpu_closed_form_run(args.config)
            except Exception as exc:   # the GPU numbers must still be reported
                line["cpu_baseline"] = {"error": repr(exc)}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- config 4: a batch of libraries
def run_batch(args):
    """BASELINE.json configs[3]: 64 libraries against one shared, resident human index; libraries dealt to the ranks
    round-robin (ribotricer_b200.batch.LibraryPipeline: copy of library k+1, kernels of library k and the result
    copy of library k-1 overlap).  Host records are the page-locked 4 B/read record stream (rt_stream_pack) the BAM decoder's columns
    are coded into once; `--distinct` different libraries are generated and cycled through.  Not a driver bench line: an
    artefact for profiles/ (libraries/s at 1 and N GPUs, seconds-long timed region)."""
    import torch
    import torch.distributed as dist

    from ribotricer_b200 import synth
    from ribotricer_b200.batch import LibraryPipeline
    from ribotricer_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    cfg = synth.config("C4", args.scale, args.contig_scale)
    idx = synth.make_index(synth.config("C2", args.scale, args.contig_scale))      # the index is C2's
    eng = Engine(local)
    eng.set_genome(idx.contig_names, idx.contig_len)
    eng.set_length_table(synth.TRUE_OFFSETS, None)
    eng.set_index(**idx.as_dict())
    eng.set_layout("compact")
    libs = []
    for k in range(args.distinct):
        d = synth.make_reads(cfg, idx, device=dev, seed_offset=1000 * k + rank)
        libs.append(eng.stream_reads({kk: v.cpu() for kk, v in d.items()}, pinned=True))
        del d
        torch.cuda.empty_cache()
    n_lib_total = args.libraries
    mine = list(range(rank, n_lib_total, world))
    results = []
    last_cols = {}

    def on_result(tag, st, rlc, cols, cov):
        results.append((tag, st["valid"], int(cols["status"].sum())))
        last_cols["cols"] = cols      # the pipeline's host buffer: valid after drain() for the last library

    pipe = LibraryPipeline(eng, "forward", on_result)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(min(3, len(mine))):           # warm-up
        pipe.submit(-1, libs[k % len(libs)])
    pipe.drain()
    results.clear()
    launches0 = eng.launches
    with ClockSampler(local) as clocks:
        barrier()
        t0 = time.perf_counter()
        for k in mine:
            pipe.submit(k, libs[k % len(libs)])
        pipe.drain()
        torch.cuda.synchronize()
        dt_local = time.perf_counter() - t0
        barrier()
    if args.dump_outputs and last_cols:
        dump_outputs(args.dump_outputs, last_cols["cols"], np.arange(idx.n_orf), idx.n_orf, f".rank{rank}" if world > 1 else "")
    t = torch.tensor([dt_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    if rank == 0:
        n_reads = int(libs[0]["n"])
        line = {
            "metric": METRIC, "value": n_lib_total * idx.n_orf / dt, "unit": UNIT, "n_gpus": world, "steps": len(mine),
            "warmup": min(3, len(mine)), "ms_per_step": 1e3 * dt / max(1, len(mine)), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C4: batch of {n_lib_total} synthetic Ribo-seq libraries ({n_reads} reads each, "
                                   f"{args.distinct} distinct ones cycled) against ONE resident human index of {idx.n_orf} "
                                   f"candidate ORFs; libraries dealt round-robin to {world} rank(s)",
                       "step": "one library: H2D of its 4 B/read record stream (copy stream) | clear + K1 + phase A + B + "
                               "D2H of the result columns (compute stream), two coverage buffers alternating",
                       "timed_region_s": dt},
            "libraries_per_s": n_lib_total / dt,
            "e2e": {"value": n_lib_total * idx.n_orf / dt, "unit": UNIT, "h2d_bytes_per_step": int(libs[0]["n_blocks"]) * (256 * 4 + 16),
                    "d2h_bytes_per_step": 25 * idx.n_orf + 8 * (9 + 65536),
                    "path": "ribotricer_b200.batch.LibraryPipeline (host records in, host result columns out, every step)"},
            "gpu_launches": eng.launches - launches0, "clocks": clocks.summary(),
            "libraries_done_rank0": len(results), "translating_first": results[0][2] if results else None,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def emit(line: dict):
    """The contract is ONE JSON line on stdout: libraries that write to fd 1 on their own (NCCL prints
    its version banner there) are sent to stderr instead, see main()."""
    (_JSON_OUT or sys.stdout).write(json.dumps(line) + "\n")
    (_JSON_OUT or sys.stdout).flush()


def main():
    global _JSON_OUT
    args = parse_args()
    if args.config is None:
        args.config = "C2" if int(os.environ.get("WORLD_SIZE", "1")) == 1 else "C3"
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")   # the real stdout, for the JSON line only
    os.dup2(2, 1)                           # everything else that writes to fd 1 goes to stderr
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "C4":
        run_batch(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
