"""count-orfs-codon stage times on a human-scale synthetic annotation (GRCh38 contig lengths, ~60 k genes), generated
from a seed, indexed with prepare-orfs and written out by orfs-seq on the GPU.

    python profiles/tools/count_orfs_codon_time.py --out OUT.txt [--genes 60000] [--tx-per-gene 4.2] [--seed 38]

A detected-ORFs TSV holding every index row is written in the detect-orfs format with Poisson profiles (one value per
nt, mean --lam, at most 9), ~--translating of the rows marked translating, so no BAM or detect-orfs run is needed.
Two selections run --repeats times each: the translating rows, and every row (--report_all); all ORF types are
features.  Host stages are timed with a host clock (index load, TSV load, sequence check, the device call, the table
write); the stages inside rt_codon_counts with CUDA events (upload, codon_emit_kernel, dedup sort + keep, count sorts,
codon_stats_kernel, copy-back) and the host gather with a host clock.  The first run includes CUDA set-up.  For a fixed
sample of genes, the per-gene rows are cross-checked against the plain-Python statement of the rules
(``oracle/codon_py.py``) run on those genes' rows alone, and its rate on that sample is reported as the CPU arm.  The
GPU name and power limit are read in the same run.
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

TSV_HEADER = ("ORF_ID\tORF_type\tstatus\tphase_score\tread_count\tlength\tvalid_codons\tvalid_codons_ratio\t"
              "read_density\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\t"
              "start_codon\tprofile\n")


def write_tsv(path, index_lines, lengths, rng, lam, translating):
    """Every index row as a detect-orfs line with a Poisson profile of one value per nt."""
    import numpy as np

    status = rng.random(len(index_lines)) < translating
    with open(path, "wb") as fh:
        fh.write(TSV_HEADER.encode())
        for lo in range(0, len(index_lines), 50_000):
            hi = min(len(index_lines), lo + 50_000)
            n = int(lengths[lo:hi].sum())
            vals = np.minimum(rng.poisson(lam, n), 9).astype(np.uint8) + 48
            text = np.empty((n, 3), np.uint8)
            text[:, 0], text[:, 1], text[:, 2] = vals, ord(","), ord(" ")
            flat = text.tobytes()
            at, out = 0, []
            for o in range(lo, hi):
                f = index_lines[o].split("\t")
                L = int(lengths[o])
                tid = f[2]
                ivs = [tuple(map(int, g.split("-"))) for g in f[10].split(",")]
                ivs.sort()
                oid = f"{tid}_{ivs[0][0]}_{ivs[-1][1]}_{L}"
                head = (f"{oid}\t{f[1]}\t{'translating' if status[o] else 'nontranslating'}\t0.5\t{L}\t{L}\t1\t0.1\t"
                        f"1.0\t{tid}\t{f[3]}\t{f[4]}\t{f[5]}\t{f[6]}\t{f[7]}\t{f[8]}\t{f[9][:3]}\t[")
                out.append(head.encode() + flat[3 * at:3 * (at + L) - 2] + b"]\n" if L else head.encode() + b"]\n")
                at += L
            fh.write(b"".join(out))
    return int(status.sum())


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

    from oracle import codon_py as CP
    from ribotricer_b200 import synth
    from ribotricer_b200.count_orfs import count_orfs_codon
    from ribotricer_b200.index import load_native_index
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    if not torch.cuda.is_available():
        sys.exit("count_orfs_codon_time.py measures the GPU path: no CUDA device")
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
    work = tempfile.mkdtemp(prefix="codon_time_")
    t0 = time.perf_counter()
    ann = synth.make_annotation(work, n_genes=args.genes, tx_per_gene=args.tx_per_gene, seed=args.seed,
                                contigs=synth.GRCH38_CONTIGS, edge_cases=False)
    say(f"workload: synth.make_annotation(n_genes={args.genes}, tx_per_gene={args.tx_per_gene}, seed={args.seed}, "
        f"GRCh38 contig lengths) generated in {time.perf_counter() - t0:.1f} s")
    prefix = os.path.join(work, "idx", "human")
    prepare_orfs(ann["gtf"], ann["fasta"], prefix)
    ipath = prefix + "_candidate_orfs.tsv"
    spath = os.path.join(work, "idx", "human_seq.tsv")
    orf_seq(ipath, ann["fasta"], spath)
    idx = load_native_index(ipath)
    lengths = idx.lengths()
    index_lines = open(ipath).read().splitlines()[1:]
    types = sorted({line.split("\t", 2)[1] for line in index_lines})
    tpath = os.path.join(work, "human_translating_ORFs.tsv")
    rng = np.random.default_rng(args.seed)
    t0 = time.perf_counter()
    n_tr = write_tsv(tpath, index_lines, lengths, rng, args.lam, args.translating)
    say(f"index: {idx.n_orf} rows, {int(lengths.sum()) / 1e6:.0f} Mnt, {os.path.getsize(ipath) / 1e6:.0f} MB; orfs-seq "
        f"file {os.path.getsize(spath) / 1e6:.0f} MB; detected-ORFs TSV {os.path.getsize(tpath) / 1e9:.2f} GB "
        f"(all rows, {n_tr} translating, Poisson({args.lam}) profiles capped at 9, written in "
        f"{time.perf_counter() - t0:.0f} s); features: {','.join(types)}")
    outs = {}
    for report_all in (False, True):
        mode = "report_all" if report_all else "translating"
        out = os.path.join(work, "out", mode)
        runs = []
        for _ in range(args.repeats):
            st = {}
            t = time.perf_counter()
            info = count_orfs_codon(ipath, tpath, set(types), spath, out, report_all, stage_ms=st)
            st["total"] = (time.perf_counter() - t) * 1e3
            runs.append(st)
        outs[mode] = out
        say("")
        say(f"selection {mode}: {info['rows']} rows, {info['genes']} genes, {info['codons']} codons kept, "
            f"{info['duplicates']} duplicates skipped, {info['codons_with_n']} codons with N")
        say("tables sha256: " + ", ".join(f"{suffix} {hashlib.sha256(open(out + suffix, 'rb').read()).hexdigest()}"
                                          for suffix in ("_codon_counts_by_gene.tsv", "_codon_counts.tsv")))
        say("stage (ms)                " + "".join(f"run {k + 1:>2}    " for k in range(len(runs))))
        for name in runs[0]:
            say(f"{name:<26}" + "".join(f"{r[name]:>9.1f} " for r in runs))
        best = min(runs[1:] or runs, key=lambda r: r["total"])
        say(f"warm run (best of runs 2..{len(runs)}): end to end {best['total'] / 1e3:.2f} s; device call "
            f"{best['codon_counts']:.0f} ms")
    # cross-check: the per-gene rows of a fixed sample of gene ids against the statement on their rows alone
    say("")
    ids = sorted({line.split("\t")[4] for line in index_lines})
    pick = set(np.random.default_rng(args.seed + 1).choice(ids, min(args.sample_genes, len(ids)), replace=False).tolist())
    keep = [o for o, line in enumerate(index_lines) if line.split("\t")[4] in pick]
    keep_set = set(keep)
    sub = os.path.join(work, "sample")
    os.makedirs(sub, exist_ok=True)
    with open(os.path.join(sub, "index.tsv"), "w") as fh:
        fh.write(open(ipath).readline() + "".join(index_lines[o] + "\n" for o in keep))
    seq_lines = open(spath).read().splitlines()
    with open(os.path.join(sub, "seq.tsv"), "w") as fh:
        fh.write(seq_lines[0] + "\n" + "".join(seq_lines[o + 1] + "\n" for o in keep))
    del seq_lines
    with open(tpath, "rb") as fin, open(os.path.join(sub, "orfs.tsv"), "wb") as fout:
        fout.write(fin.readline())
        for line in fin:
            if line.split(b"\t", 12)[11].decode() in pick:
                fout.write(line)
    ok = True
    for report_all, mode in ((False, "translating"), (True, "report_all")):
        t = time.perf_counter()
        gene_text, _, s = CP.count_orfs_codon_text(os.path.join(sub, "index.tsv"), os.path.join(sub, "orfs.tsv"), types,
                                                   os.path.join(sub, "seq.tsv"), report_all)
        ref_s = time.perf_counter() - t
        got = [line for line in open(outs[mode] + "_codon_counts_by_gene.tsv").read().splitlines(keepends=True)[1:]
               if line.split("\t", 1)[0] in pick]
        same = got == gene_text.splitlines(keepends=True)[1:]
        ok &= same
        say(f"cross-check {mode}: {len(pick)} sampled gene ids ({len(keep_set)} index rows, {s['rows']} TSV rows, "
            f"{len(got)} table rows) {'identical' if same else 'DIFFERENT'} to the plain-Python statement; plain Python "
            f"(one core) on that sample: {ref_s:.2f} s = {s['rows'] / ref_s / 1e3:.2f} k TSV rows/s")
    say("the reference tool itself was not run: its time on this workload is not measured")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if not ok:
        sys.exit("cross-check failed")


if __name__ == "__main__":
    main()
