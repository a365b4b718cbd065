"""prepare-orfs stage times on a human-scale synthetic annotation (GRCh38 contig lengths, ~60 k genes, ~250 k
transcripts), generated from a seed.

    python profiles/tools/prepare_orfs_time.py --out OUT.txt [--genes 60000] [--tx-per-gene 4.2] [--seed 38]

Host stages are timed with a host clock (FASTA load, GTF load, transcript table, annotated rows, device call, text);
the device stages inside ``rt_orf_search`` with CUDA events (upload, splice, count, row scan, fill, interval count +
scan, interval fill).  The run is repeated (the first includes CUDA context set-up and module load).  A fixed sample of
genes on chr21 / chr22 is cross-checked against the plain-Python statement of the rules, whose rate on that sample is
reported as the reference-style CPU arm.  The GPU name and power limit are read in the same run.
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
    ap.add_argument("--sample-genes", type=int, default=150)
    args = ap.parse_args()

    import numpy as np
    import torch

    from oracle import prepare_py as P
    from ribotricer_b200 import synth
    from ribotricer_b200.prepare_orfs import Genome, prepare_orfs

    if not torch.cuda.is_available():
        sys.exit("prepare_orfs_time.py measures the GPU path: no CUDA device")
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
    work = tempfile.mkdtemp(prefix="prep_time_")
    t0 = time.perf_counter()
    ann = synth.make_annotation(work, n_genes=args.genes, tx_per_gene=args.tx_per_gene, seed=args.seed,
                                contigs=synth.GRCH38_CONTIGS, edge_cases=False)
    say(f"workload: synth.make_annotation(n_genes={args.genes}, tx_per_gene={args.tx_per_gene}, seed={args.seed}, "
        f"GRCh38 contig lengths) generated in {time.perf_counter() - t0:.1f} s; "
        f"FASTA {os.path.getsize(ann['fasta']) / 1e9:.2f} GB, GTF {os.path.getsize(ann['gtf']) / 1e6:.0f} MB")
    prefix = os.path.join(work, "out", "human")
    runs = []
    for k in range(args.repeats):
        st = {}
        t = time.perf_counter()
        info = prepare_orfs(ann["gtf"], ann["fasta"], prefix, stage_ms=st)
        st["total"] = (time.perf_counter() - t) * 1e3
        runs.append(st)
    path = prefix + "_candidate_orfs.tsv"
    n_rows = info["n_annotated"] + info["n_candidates"]
    # spliced nt the kernels scanned: sum of the kept transcripts' merged exon lengths
    from ribotricer_b200.prepare_orfs import build_transcripts, load_gtf
    g = Genome(ann["fasta"])
    tx = build_transcripts(load_gtf(ann["gtf"]), g)
    nt = int((tx["exon_end"].astype(np.int64) - tx["exon_start"] + 1).sum())
    say(f"transcripts {info['n_tx']} (skipped {info['n_skipped']}), rows {n_rows} ({info['n_annotated']} annotated), "
        f"spliced nt {nt}, index file {os.path.getsize(path) / 1e6:.0f} MB")
    say("")
    names = list(runs[0])
    say("stage (ms)                          " + "".join(f"run {k + 1:>2}    " for k in range(len(runs))))
    for name in names:
        say(f"{name:<36}" + "".join(f"{r[name]:>9.1f} " for r in runs))
    best = min(runs[1:] or runs, key=lambda r: r["total"])
    dev = sum(v for k, v in best.items() if k.startswith("device:") and "upload" not in k)
    say("")
    say(f"warm run (best of runs 2..{len(runs)}): end to end {best['total'] / 1e3:.2f} s = "
        f"{n_rows / best['total'] * 1e3 / 1e6:.2f} M rows/s, {nt / best['total'] * 1e3 / 1e9:.2f} G spliced nt/s")
    say(f"kernels + scans (device events, upload excluded): {dev:.1f} ms = {nt / dev * 1e3 / 1e9:.1f} G spliced nt/s, "
        f"{n_rows / dev * 1e3 / 1e6:.1f} M rows/s")
    # cross-check: genes on chr21 / chr22 against the plain-Python statement of the rules
    rng = np.random.default_rng(args.seed)
    gtf_lines = open(ann["gtf"]).read().splitlines()
    body = [ln for ln in gtf_lines if ln and not ln.startswith("#") and ln.split("\t", 1)[0] in ("chr21", "chr22")]
    genes = sorted({ln.split('gene_id "', 1)[1].split('"', 1)[0] for ln in body})
    pick = set(rng.choice(genes, min(args.sample_genes, len(genes)), replace=False).tolist())
    sub = os.path.join(work, "sample.gtf")
    with open(sub, "w") as fh:
        for ln in body:
            if ln.split('gene_id "', 1)[1].split('"', 1)[0] in pick:
                fh.write(ln + "\n")
    letters = np.frombuffer(b"ACGTN", np.uint8)
    ids = [g.names.index(c) for c in ("chr21", "chr22")]
    genome = {c: letters[g.codes([i])].tobytes().decode() for c, i in zip(("chr21", "chr22"), ids)}
    t = time.perf_counter()
    txs, _ = P.transcripts(P.parse_gtf(sub), genome)
    want = P.annotated_rows(txs, genome, {"ATG"}) + P.candidate_rows(txs, genome, {"ATG"}, {"TAG", "TAA", "TGA"}, 60,
                                                                     False)
    ref_s = time.perf_counter() - t
    tids = {t["transcript_id"] for t in txs}
    got = [ln for ln in open(path).read().splitlines(keepends=True)[1:] if ln.split("\t", 3)[2] in tids]
    ok = got == want
    sample_nt = sum(e - s + 1 for t in txs for s, e in t["exons"])
    say("")
    say(f"cross-check: {len(pick)} genes on chr21/chr22, {len(txs)} transcripts, {len(want)} rows: "
        f"{'identical' if ok else 'DIFFERENT'} to the plain-Python statement")
    say(f"reference-style CPU arm (plain Python, str.find, one core) on that sample: {ref_s:.2f} s = "
        f"{len(want) / ref_s / 1e3:.1f} k rows/s, {sample_nt / ref_s / 1e6:.2f} M spliced nt/s")
    say("the reference tool itself was not run: its time on human is not measured")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if not ok:
        sys.exit("cross-check failed")


if __name__ == "__main__":
    main()
