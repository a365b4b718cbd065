"""orfs-seq stage times on a human-scale synthetic annotation (GRCh38 contig lengths, ~60 k genes), generated from a
seed and indexed with prepare-orfs on the GPU.

    python profiles/tools/orfs_seq_time.py --out OUT.txt [--genes 60000] [--tx-per-gene 4.2] [--seed 38]

Host stages are timed with a host clock (index load + ids, FASTA load, contig codes, the device call with its file
write); the device stages inside ``rt_orf_seq_write`` with CUDA events (upload, orf_seq_kernel summed over chunks,
copy-back summed over chunks).  Both modes (nucleotide, protein) run ``--repeats`` times; the first run of each includes
CUDA set-up.  A fixed sample of the rows on chr21 / chr22 is cross-checked against the plain-Python statement of the rules
(``oracle/seq_py.py``), whose rate on that sample is reported as the CPU arm.  The GPU name and power limit are read in
the same run.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--tx-per-gene", type=float, default=4.2)
    ap.add_argument("--seed", type=int, default=38)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sample-rows", type=int, default=20_000)
    args = ap.parse_args()

    import numpy as np
    import torch

    from oracle import seq_py as S
    from ribotricer_b200 import synth
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    if not torch.cuda.is_available():
        sys.exit("orfs_seq_time.py measures the GPU path: no CUDA device")
    lines = []

    def say(msg=""):
        print(msg, flush=True)
        lines.append(msg)

    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()
    except FileNotFoundError:
        smi = []
    say(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi[0] if smi else 'n/a'}")
    work = tempfile.mkdtemp(prefix="seq_time_")
    t0 = time.perf_counter()
    ann = synth.make_annotation(work, n_genes=args.genes, tx_per_gene=args.tx_per_gene, seed=args.seed,
                                contigs=synth.GRCH38_CONTIGS, edge_cases=False)
    say(f"workload: synth.make_annotation(n_genes={args.genes}, tx_per_gene={args.tx_per_gene}, seed={args.seed}, "
        f"GRCh38 contig lengths) generated in {time.perf_counter() - t0:.1f} s; FASTA "
        f"{os.path.getsize(ann['fasta']) / 1e9:.2f} GB")
    prefix = os.path.join(work, "idx", "human")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    say(f"index: prepare_orfs defaults, {os.path.getsize(ipath) / 1e6:.0f} MB")
    results = {}
    for protein in (False, True):
        mode = "protein" if protein else "nt"
        out = os.path.join(work, f"seq_{mode}.tsv")
        runs = []
        for _ in range(args.repeats):
            st = {}
            t = time.perf_counter()
            info = orf_seq(ipath, ann["fasta"], out, translate=protein, stage_ms=st)
            st["total"] = (time.perf_counter() - t) * 1e3
            runs.append(st)
        results[mode] = (info, runs, out)
        say("")
        say(f"mode {mode}: {info['n_orf']} rows, {info['residues']} {info['unit']}, output {info['bytes'] / 1e6:.1f} MB")
        say("stage (ms)                " + "".join(f"run {k + 1:>2}    " for k in range(len(runs))))
        for name in runs[0]:
            say(f"{name:<26}" + "".join(f"{r[name]:>9.1f} " for r in runs))
        best = min(runs[1:] or runs, key=lambda r: r["total"])
        say(f"warm run (best of runs 2..{len(runs)}): end to end {best['total'] / 1e3:.2f} s = "
            f"{info['bytes'] / best['total'] * 1e3 / 1e9:.2f} GB/s written; device call (incl. upload and file "
            f"write) {best['write']:.0f} ms = {info['bytes'] / best['write'] * 1e3 / 1e9:.2f} GB/s; kernels "
            f"{best['device:orf_seq_kernel']:.1f} ms = {info['bytes'] / best['device:orf_seq_kernel'] * 1e3 / 1e9:.1f} "
            f"GB/s of lines")
    # cross-check: a fixed sample of the rows on chr21 / chr22 against the plain-Python statement
    from ribotricer_b200.prepare_orfs import Genome

    rows = S.parse_rows(ipath)
    rng = np.random.default_rng(args.seed)
    chroms = ("chr21", "chr22")
    on = np.flatnonzero([r[1] in chroms for r in rows])
    pick = np.sort(rng.choice(on, min(args.sample_rows, len(on)), replace=False))
    genome = {}
    g = Genome(ann["fasta"])
    letters = np.frombuffer(b"ACGTN", np.uint8)
    for c in chroms:
        genome[c] = letters[g.codes([g.names.index(c)])].tobytes().decode()
    g.close()
    say("")
    ok = True
    for mode, (info, _, out) in results.items():
        got = open(out).read().splitlines(keepends=True)[1:]
        t = time.perf_counter()
        want = S.lines_text([rows[i] for i in pick], genome, mode == "protein")
        ref_s = time.perf_counter() - t
        same = [got[i] for i in pick] == want.splitlines(keepends=True)[1:]
        ok &= same
        say(f"cross-check {mode}: {len(pick)} sampled rows {'identical' if same else 'DIFFERENT'} to the plain-Python "
            f"statement; plain Python (one core) on that sample: {ref_s:.2f} s = {len(pick) / ref_s / 1e3:.1f} k rows/s")
    say("the reference tool itself (pandas iterrows + pyfaidx) was not run: its time on human is not measured")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if not ok:
        sys.exit("cross-check failed")


if __name__ == "__main__":
    main()
