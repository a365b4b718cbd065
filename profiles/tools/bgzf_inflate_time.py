"""BGZF inflate on the GPU (rt_bgzf_inflate, DESIGN.md section 12) on a human-scale synthetic annotation (GRCh38 contig
lengths, ~60 k genes, 3.14 GB FASTA), generated from a seed; the FASTA and the GTF are bgzipped at zlib's default level
in 0xFF00-byte members, as bgzip writes them.

    python profiles/tools/bgzf_inflate_time.py --out OUT.txt [--genes 60000] [--tx-per-gene 4.2] [--seed 38]

Per file, ``--repeats`` calls of ``Engine.inflate_bgzf``: the stage times rt_bgzf_inflate reports (file read and header
walk by host clock; upload, bgzf_inflate_kernel and copy-back into page-locked buffers by CUDA events; drain into the
text and host decode of refused members by host clock; upload, kernel, copy-back and drain overlap), the inflated GB/s of the kernel and of the whole call (host clock around it), and the members handed to the
host.  The first run includes CUDA set-up.  Every result is compared with the plain file byte for byte.  In the same
run, the host decoder inflates the same members (rt_inflate_raw + rt_crc32 per member, all cores through a thread pool;
ctypes releases the GIL), and prepare-orfs and orfs-seq run end to end from the BGZF inputs and from the plain files,
alternating, with their outputs compared.  The GPU name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import ctypes as C
import os
import struct
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

EOF_MEMBER = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzip(src: str, dst: str, pool) -> None:
    def member(payload: bytes) -> bytes:
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        data = c.compress(payload) + c.flush()
        return (b"\x1f\x8b\x08\x04" + struct.pack("<IBBH", 0, 0, 0xFF, 6) + b"BC" +
                struct.pack("<HH", 2, len(data) + 25) + data +
                struct.pack("<II", zlib.crc32(payload) & 0xFFFFFFFF, len(payload)))

    with open(src, "rb") as fh, open(dst, "wb") as out:
        while True:
            chunk = fh.read(0xFF00 * 4096)
            if not chunk:
                break
            for m in pool.map(member, [chunk[i:i + 0xFF00] for i in range(0, len(chunk), 0xFF00)]):
                out.write(m)
        out.write(EOF_MEMBER)


def members(data: bytes):
    """(payload offset, payload length, ISIZE, CRC-32) of every member."""
    out, off = [], 0
    while off < len(data):
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        bsize = struct.unpack_from("<H", data, off + 16)[0]
        total = bsize + 1
        crc, isize = struct.unpack_from("<II", data, off + total - 8)
        out.append((off + 12 + xlen, total - 12 - xlen - 8, isize, crc))
        off += total
    return out


def host_inflate(lib, data: bytes, blocks, threads: int):
    """All members through rt_inflate_raw + rt_crc32 on `threads` threads; returns (seconds, output)."""
    import numpy as np

    src = np.frombuffer(data, np.uint8)
    out_off = np.concatenate([[0], np.cumsum([b[2] for b in blocks])]).astype(np.int64)
    out = np.empty(int(out_off[-1]), np.uint8)
    sp, dp = src.ctypes.data, out.ctypes.data
    step = 256

    def run(k0):
        bad = 0
        for k in range(k0, min(len(blocks), k0 + step)):
            a, n, isize, crc = blocks[k]
            if isize == 0:
                continue
            if lib.rt_inflate_raw(sp + a, n, dp + int(out_off[k]), isize) != 0 or \
                    lib.rt_crc32(dp + int(out_off[k]), isize) != crc:
                bad += 1
        return bad

    with cf.ThreadPoolExecutor(threads) as pool:
        t = time.perf_counter()
        bad = sum(pool.map(run, range(0, len(blocks), step)))
        dt = time.perf_counter() - t
    return dt, out, bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--tx-per-gene", type=float, default=4.2)
    ap.add_argument("--seed", type=int, default=38)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()

    import numpy as np
    import torch

    from ribotricer_b200 import _lib, synth
    from ribotricer_b200.detect_orfs import get_engine
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    if not torch.cuda.is_available():
        sys.exit("bgzf_inflate_time.py measures the GPU path: no CUDA device")
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
    work = tempfile.mkdtemp(prefix="bgzf_time_")
    t0 = time.perf_counter()
    ann = synth.make_annotation(work, n_genes=args.genes, tx_per_gene=args.tx_per_gene, seed=args.seed,
                                contigs=synth.GRCH38_CONTIGS, edge_cases=False)
    say(f"workload: synth.make_annotation(n_genes={args.genes}, tx_per_gene={args.tx_per_gene}, seed={args.seed}, "
        f"GRCh38 contig lengths) generated in {time.perf_counter() - t0:.1f} s")
    threads = os.cpu_count() or 1
    bz = {}
    with cf.ThreadPoolExecutor(threads) as pool:
        for key in ("fasta", "gtf"):
            t0 = time.perf_counter()
            bz[key] = ann[key] + ".bgz"
            bgzip(ann[key], bz[key], pool)
            say(f"{key}: {os.path.getsize(ann[key]) / 1e9:.3f} GB plain, {os.path.getsize(bz[key]) / 1e9:.3f} GB BGZF "
                f"(zlib level 6, 0xFF00-byte members; written in {time.perf_counter() - t0:.1f} s)")
    eng = get_engine()
    lib = _lib.load()
    names = ("read", "header_walk", "upload", "bgzf_inflate_kernel", "copy_back", "drain", "host_fallback")
    for key in ("fasta", "gtf"):
        plain = np.fromfile(ann[key], np.uint8)
        runs = []
        for _ in range(args.repeats):
            sm, ms = np.zeros(4, np.int64), np.zeros(len(names), np.float32)
            t = time.perf_counter()
            text = eng.inflate_bgzf(bz[key], summary=sm, stage_ms=ms)
            wall = (time.perf_counter() - t) * 1e3
            same = np.array_equal(text.view(), plain)
            del text
            runs.append((dict(zip(names, ms.tolist()), total=wall), sm.copy(), same))
        sm = runs[0][1]
        say("")
        say(f"{key}: {sm[0]} members, {sm[1] / 1e9:.3f} GB compressed -> {sm[2] / 1e9:.3f} GB inflated; members handed to "
            f"the host: {[int(r[1][3]) for r in runs]}; identical to the plain file: {[r[2] for r in runs]}")
        say("stage (ms)                " + "".join(f"run {k + 1:>2}    " for k in range(len(runs))))
        for name in list(names) + ["total"]:
            say(f"{name:<26}" + "".join(f"{r[0][name]:>9.1f} " for r in runs))
        warm = runs[1:] or runs
        best = min(warm, key=lambda r: r[0]["total"])[0]
        gb = sm[2] / 1e9
        say(f"warm (best of runs 2..{len(runs)}): kernel {best['bgzf_inflate_kernel']:.1f} ms = "
            f"{gb / best['bgzf_inflate_kernel'] * 1e3:.1f} GB/s inflated; whole call {best['total']:.0f} ms = "
            f"{gb / best['total'] * 1e3:.2f} GB/s; upload {best['upload']:.0f} ms, copy-back {best['copy_back']:.0f} ms, drain "
            f"{best['drain']:.0f} ms (the three overlap)")
        data = open(bz[key], "rb").read()
        blocks = members(data)
        for _ in range(2):
            dt, out, bad = host_inflate(lib, data, blocks, threads)
        same = np.array_equal(out, plain)
        say(f"host decoder, same members (rt_inflate_raw + rt_crc32, {threads} threads, second of two runs): "
            f"{dt * 1e3:.0f} ms = {gb / dt:.2f} GB/s; refused {bad}; identical: {same}")
        del out, plain
    # the commands end to end, BGZF against plain, alternating
    say("")
    pfx = os.path.join(work, "p", "human")
    seq_out = os.path.join(work, "seq.tsv")
    t_prep = {"plain": [], "bgzf": []}
    for _ in range(2):
        for kind, (g, f) in (("plain", (ann["gtf"], ann["fasta"])), ("bgzf", (bz["gtf"], bz["fasta"]))):
            t = time.perf_counter()
            prepare_orfs(g, f, pfx + "_" + kind)
            t_prep[kind].append(time.perf_counter() - t)
    same = open(pfx + "_plain_candidate_orfs.tsv", "rb").read() == open(pfx + "_bgzf_candidate_orfs.tsv", "rb").read()
    say(f"prepare-orfs end to end (s, two runs each, alternating): plain {t_prep['plain']}, BGZF {t_prep['bgzf']}; "
        f"index identical: {same}")
    ipath = pfx + "_plain_candidate_orfs.tsv"
    with cf.ThreadPoolExecutor(threads) as pool:
        bgzip(ipath, ipath + ".bgz", pool)
    t_seq = {"plain": [], "bgzf": []}
    for _ in range(2):
        for kind, (i, f) in (("plain", (ipath, ann["fasta"])), ("bgzf", (ipath + ".bgz", bz["fasta"]))):
            t = time.perf_counter()
            orf_seq(i, f, seq_out + "." + kind)
            t_seq[kind].append(time.perf_counter() - t)
    same = open(seq_out + ".plain", "rb").read() == open(seq_out + ".bgzf", "rb").read()
    say(f"orfs-seq (nt) end to end (s, two runs each, alternating): plain {t_seq['plain']}, BGZF {t_seq['bgzf']}; "
        f"output identical: {same}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
