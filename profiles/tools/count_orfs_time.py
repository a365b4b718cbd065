"""count-orfs stage times on the workload of count_orfs_codon_time.py: the human-scale synthetic annotation (GRCh38
contig lengths, ~60 k genes) indexed with prepare-orfs, and the detected-ORFs TSV of every index row with Poisson
profiles that its ``write_tsv`` writes.

    python profiles/tools/count_orfs_time.py --out OUT.txt [--genes 60000] [--tx-per-gene 4.2] [--seed 38]

Two selections run --repeats times each through ``count_orfs_gpu``: the translating rows, and every row (--report_all);
all ORF types are features.  Host stages are timed with a host clock (BGZF sniff, index load, TSV load, the device
call, the table write); the stages inside rt_count_orfs with CUDA events (upload, count_emit_kernel, sort,
count_keep_kernel, copy-back) and the host gather with a host clock.  The first run includes CUDA set-up.  In the same
run the plain-Python ``count_orfs`` (one core) reads the same translating selection from the whole index and TSV and
its table is compared byte for byte.  For --report_all, ``count_orfs`` runs on the rows of a fixed sample of gene ids
(with an index of their rows alone); its table must equal those genes' rows of the GPU table, and its rate there is
the CPU arm.  The GPU name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import hashlib
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from count_orfs_codon_time import write_tsv  # noqa: E402  (the workload generator, shared)

STAGES = ("inflate", "index_load", "tsv_load", "orf_counts", "device:host_gather", "device:upload",
          "device:count_emit_kernel", "device:sort", "device:count_keep_kernel", "device:copy_back", "write", "total")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--tx-per-gene", type=float, default=4.2)
    ap.add_argument("--seed", type=int, default=38)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--lam", type=float, default=0.3)
    ap.add_argument("--translating", type=float, default=0.1)
    ap.add_argument("--sample-genes", type=int, default=200)
    args = ap.parse_args()

    import numpy as np
    import torch

    from ribotricer_b200 import synth
    from ribotricer_b200.count_orfs import count_orfs, count_orfs_gpu
    from ribotricer_b200.index import load_native_index
    from ribotricer_b200.prepare_orfs import prepare_orfs

    if not torch.cuda.is_available():
        sys.exit("count_orfs_time.py measures the GPU path: no CUDA device")
    lines = []

    def say(msg=""):
        print(msg, flush=True)
        lines.append(msg)

    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()
    except FileNotFoundError:
        smi = []
    say(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi[0] if smi else 'n/a'} | host cores: {os.cpu_count()}")
    work = tempfile.mkdtemp(prefix="count_orfs_time_")
    t0 = time.perf_counter()
    ann = synth.make_annotation(work, n_genes=args.genes, tx_per_gene=args.tx_per_gene, seed=args.seed,
                                contigs=synth.GRCH38_CONTIGS, edge_cases=False)
    say(f"workload: synth.make_annotation(n_genes={args.genes}, tx_per_gene={args.tx_per_gene}, seed={args.seed}, "
        f"GRCh38 contig lengths) generated in {time.perf_counter() - t0:.1f} s")
    prefix = os.path.join(work, "idx", "human")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    idx = load_native_index(ipath)
    lengths = idx.lengths()
    index_lines = open(ipath).read().splitlines()[1:]
    types = sorted({line.split("\t", 2)[1] for line in index_lines})
    tpath = os.path.join(work, "human_translating_ORFs.tsv")
    rng = np.random.default_rng(args.seed)
    t0 = time.perf_counter()
    n_tr = write_tsv(tpath, index_lines, lengths, rng, args.lam, args.translating)
    say(f"index: {idx.n_orf} rows, {int(lengths.sum()) / 1e6:.0f} Mnt, {os.path.getsize(ipath) / 1e6:.0f} MB; "
        f"detected-ORFs TSV {os.path.getsize(tpath) / 1e9:.2f} GB (all rows, {n_tr} translating, Poisson({args.lam}) "
        f"profiles capped at 9, written in {time.perf_counter() - t0:.0f} s); features: {','.join(types)}")
    outs, infos = {}, {}
    for report_all in (False, True):
        mode = "report_all" if report_all else "translating"
        out = os.path.join(work, "out", f"{mode}_counts.tsv")
        os.makedirs(os.path.dirname(out), exist_ok=True)
        runs = []
        for _ in range(args.repeats):
            st = {}
            t = time.perf_counter()
            info = count_orfs_gpu(ipath, tpath, set(types), out, report_all, stage_ms=st)
            st["total"] = (time.perf_counter() - t) * 1e3
            runs.append(st)
        outs[mode], infos[mode] = out, info
        say("")
        say(f"selection {mode}: {info['rows']} rows, {info['genes']} genes, {info['positions']} positions kept, "
            f"{info['duplicates']} duplicates skipped")
        say(f"table sha256: {hashlib.sha256(open(out, 'rb').read()).hexdigest()}")
        say("stage (ms)                " + "".join(f"run {k + 1:>2}    " for k in range(len(runs))))
        for name in STAGES:
            say(f"{name:<26}" + "".join(f"{r[name]:>9.1f} " for r in runs))
        best = min(runs[1:] or runs, key=lambda r: r["total"])
        named = info["positions"] + info["duplicates"]
        say(f"warm run (best of runs 2..{len(runs)}): end to end {best['total'] / 1e3:.2f} s = "
            f"{named / best['total'] / 1e3:.0f} Mnt/s, {info['rows'] / best['total']:.0f} k rows/s; device call "
            f"{best['orf_counts']:.0f} ms")
    # CPU arm 1: count_orfs on the whole index and TSV, translating rows
    say("")
    want = os.path.join(work, "out", "translating_py.tsv")
    t = time.perf_counter()
    count_orfs(ipath, tpath, set(types), want, False)
    py_s = time.perf_counter() - t
    named = infos["translating"]["positions"] + infos["translating"]["duplicates"]
    same = open(want, "rb").read() == open(outs["translating"], "rb").read()
    say(f"count_orfs (plain Python, one core), translating: {py_s:.1f} s = {named / py_s / 1e6:.2f} Mnt/s, "
        f"{infos['translating']['rows'] / py_s / 1e3:.1f} k rows/s; table {'IDENTICAL' if same else 'DIFFERENT'} "
        f"to count_orfs_gpu byte for byte")
    ok = same
    # CPU arm 2: count_orfs on the rows of a fixed sample of gene ids, report_all
    ids = sorted({line.split("\t")[4] for line in index_lines})
    pick = set(np.random.default_rng(args.seed + 1).choice(ids, min(args.sample_genes, len(ids)), replace=False).tolist())
    keep = [o for o, line in enumerate(index_lines) if line.split("\t")[4] in pick]
    sub = os.path.join(work, "sample")
    os.makedirs(sub, exist_ok=True)
    with open(os.path.join(sub, "index.tsv"), "w") as fh:
        fh.write(open(ipath).readline() + "".join(index_lines[o] + "\n" for o in keep))
    with open(tpath, "rb") as fin, open(os.path.join(sub, "orfs.tsv"), "wb") as fout:
        fout.write(fin.readline())
        for line in fin:
            if line.split(b"\t", 12)[11].decode() in pick:
                fout.write(line)
    sample_out = os.path.join(sub, "counts.tsv")
    t = time.perf_counter()
    count_orfs(os.path.join(sub, "index.tsv"), os.path.join(sub, "orfs.tsv"), set(types), sample_out, True)
    ref_s = time.perf_counter() - t
    sample_nt = int(lengths[keep].sum())
    got = [line for line in open(outs["report_all"]).read().splitlines(keepends=True)[1:] if line.split("\t", 1)[0] in pick]
    same = got == open(sample_out).read().splitlines(keepends=True)[1:]
    ok &= same
    say(f"count_orfs (plain Python, one core), report_all on {len(pick)} sampled gene ids ({len(keep)} rows, "
        f"{sample_nt / 1e6:.1f} Mnt, {len(got)} table rows): {ref_s:.2f} s = {sample_nt / ref_s / 1e6:.2f} Mnt/s, "
        f"{len(keep) / ref_s / 1e3:.1f} k rows/s; those rows {'IDENTICAL' if same else 'DIFFERENT'} to count_orfs_gpu")
    say("the reference tool itself was not run: its time on this workload is not measured")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if not ok:
        sys.exit("cross-check failed")


if __name__ == "__main__":
    main()
