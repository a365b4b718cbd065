"""Run the HOST logic of one build of the library under the fake cudart and print a digest of every host-to-device upload:
set_genome, set_index (+ layout), rt_score over several ranges and rt_score_host in parts, for several synthetic indexes;
then rt_codon_counts and rt_count_orfs on random selections, an empty one and one without genes.  `rows` as the first
argument after the library runs only the last two."""
import ctypes as C, sys, os, hashlib
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))))
from ribotricer_b200 import synth

fake = C.CDLL(os.environ.get("FAKE_CUDART", "/tmp/stub/lib/libcudart.so.12"), mode=C.RTLD_GLOBAL)
fake.fake_log_size.restype = C.c_size_t
lib = C.CDLL(sys.argv[1])
vp, i64 = C.c_void_p, C.c_int64
lib.rt_last_error.restype = C.c_char_p; lib.rt_last_error.argtypes = [vp]
lib.rt_create.argtypes = [C.c_int, C.POINTER(vp)]
lib.rt_set_genome.argtypes = [vp, C.c_int, vp, C.c_int]
lib.rt_set_index.argtypes = [vp, i64, vp, vp, vp, vp, vp]
lib.rt_set_layout.argtypes = [vp, C.c_int]
lib.rt_coverage_elems.restype = i64; lib.rt_coverage_elems.argtypes = [vp]
lib.rt_plane_elems.restype = i64; lib.rt_plane_elems.argtypes = [vp]
class Params(C.Structure): _fields_ = [(n, C.c_double) for n in ("a", "b", "c", "d", "e")]
class Out(C.Structure): _fields_ = [(n, vp) for n in ("score", "valid", "count", "length", "min_codon", "status", "frame_K", "frame_s")]
lib.rt_score.argtypes = [vp, vp, i64, i64, C.POINTER(Params), C.POINTER(Out), vp]
lib.rt_score_host.argtypes = [vp, vp, i64, i64, C.POINTER(Params), C.POINTER(Out)]
lib.rt_destroy.argtypes = [vp]
from ribotricer_b200._lib import CodonQuery, CountQuery
lib.rt_codon_counts.argtypes = [vp, C.POINTER(CodonQuery), vp, vp, vp, vp]
lib.rt_count_orfs.argtypes = [vp, C.POINTER(CountQuery), vp, vp, vp, vp]

def digest(tag, unordered=False):
    n = fake.fake_log_size(); buf = (C.c_ulonglong * max(1, n))(); fake.fake_log_copy(buf); fake.fake_log_clear()
    raw = bytes(buf)[:8 * n]
    line = f"{tag}: {n // 2} uploads, {sum(buf[i] for i in range(0, n, 2))} bytes, md5 {hashlib.md5(raw).hexdigest()}"
    if unordered:      # the same (size, FNV-1a) pairs in any order
        pairs = sorted(zip(buf[0:n:2], buf[1:n:2]))
        line += f", unordered md5 {hashlib.md5(np.array(pairs, np.uint64).tobytes()).hexdigest()}"
    print(line)

def check(rc, ctx):
    assert rc == 0, lib.rt_last_error(ctx)

p = lambda a: a.ctypes.data_as(vp)
def rows_query(rng, n_orf, n_sel, n_gene, genome=300_000):
    """A random index of n_orf rows (1-4 ascending intervals) and n_sel selected rows with profiles and letters."""
    n_ex = rng.integers(1, 5, n_orf)
    ptr = np.concatenate([[0], np.cumsum(n_ex)]).astype(np.int64)
    starts, ends = [], []
    for k in n_ex.tolist():
        s = np.sort(rng.choice(genome // 1000, k, replace=False)) * 1000 + 1
        starts.append(s); ends.append(s + rng.integers(2, 600, k))
    starts, ends = np.concatenate(starts).astype(np.int32), np.concatenate(ends).astype(np.int32)
    lengths = np.add.reduceat(ends.astype(np.int64) - starts + 1, ptr[:-1])
    seq = rng.choice(np.frombuffer(b"ACGTN", np.uint8), int(lengths.sum()))
    row = rng.integers(0, n_orf, n_sel).astype(np.int64)
    texts = [("[" + ", ".join(map(str, rng.poisson(1.2, int(lengths[r])).tolist())) + "]").encode() for r in row]
    prof_len = np.array([len(t) for t in texts], np.int64)
    cols = dict(row=row, gene=rng.integers(0, max(n_gene, 1), n_sel).astype(np.int32),
                gseq=rng.integers(0, 2 * max(n_gene, 1), n_sel).astype(np.int32),
                prof_off=np.concatenate([[0], np.cumsum(prof_len)[:-1]]).astype(np.int64), prof_len=prof_len,
                tsv=np.frombuffer(b"".join(texts) or b"\0", np.uint8),
                seq_off=np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64), seq=seq, exon_ptr=ptr,
                exon_start=starts, exon_end=ends, orf_strand=rng.integers(0, 2, n_orf).astype(np.uint8))
    return cols, n_gene


def run_rows():
    ctx = vp(); check(lib.rt_create(0, C.byref(ctx)), None)
    rng = np.random.default_rng(7)
    for tag, n_orf, n_sel, n_gene in (("random", 3000, 2500, 40), ("empty", 3000, 0, 40), ("no genes", 3000, 0, 0)):
        c, n_gene = rows_query(rng, n_orf, n_sel, n_gene)
        ptr = {k: p(v) for k, v in c.items()}
        cq = CodonQuery(n_sel=n_sel, n_orf=n_orf, n_gene=n_gene, n_gseq=2 * n_gene,
                        **{k: ptr[k] for k, _ in CodonQuery._fields_ if k in ptr})
        gene_tab, pooled_tab = np.zeros((64 * n_gene + 1) * 5, np.uint64), np.zeros(64 * 5, np.uint64)
        summary = np.zeros(6, np.int64)
        check(lib.rt_codon_counts(ctx, C.byref(cq), p(gene_tab), p(pooled_tab), p(summary), None), ctx)
        digest(f"rows {tag} ({n_sel} of {n_orf}, {n_gene} genes) rt_codon_counts", unordered=True)
        nq = CountQuery(n_sel=n_sel, n_orf=n_orf, n_gene=n_gene, **{k: ptr[k] for k, _ in CountQuery._fields_ if k in ptr})
        total, length = np.zeros(n_gene + 1, np.uint64), np.zeros(n_gene + 1, np.uint64)
        summary = np.zeros(4, np.int64)
        check(lib.rt_count_orfs(ctx, C.byref(nq), p(total), p(length), p(summary), None), ctx)
        digest(f"rows {tag} ({n_sel} of {n_orf}, {n_gene} genes) rt_count_orfs", unordered=True)
    lib.rt_destroy(ctx)


cases = [("tiny", 1.0, 1.0), ("C1", 0.3, 1.0), ("C5", 0.02, 0.05), ("C2", 0.5, 0.5)]
for name, scale, cscale in cases if sys.argv[2:3] != ["rows"] else []:
    cfg = synth.config(name, scale, cscale); idx = synth.make_index(cfg); d = idx.as_dict()
    ctx = vp(); check(lib.rt_create(0, C.byref(ctx)), None)
    lens = np.ascontiguousarray(idx.contig_len, np.int64)
    check(lib.rt_set_genome(ctx, len(lens), p(lens), 256), ctx)
    cols = [np.ascontiguousarray(d[k], dt) for k, dt in (("exon_ptr", np.int64), ("exon_start", np.int32), ("exon_end", np.int32), ("orf_contig", np.int32), ("orf_strand", np.uint8))]
    check(lib.rt_set_index(ctx, idx.n_orf, *[p(c) for c in cols]), ctx)
    digest(f"{name} set_index ({idx.n_orf} ORFs)")
    for layout in (1, 0):          # compact, dense
        check(lib.rt_set_layout(ctx, layout), ctx)
        digest(f"{name} set_layout {layout}")
        n = idx.n_orf; elems = lib.rt_coverage_elems(ctx)
        cov = np.zeros(elems + 64, np.int32)
        cols_out = dict(score=np.zeros(n), valid=np.zeros(n, np.int32), count=np.zeros(n, np.int64), length=np.zeros(n, np.int32),
                        min_codon=np.zeros(n, np.int32), status=np.zeros(n, np.uint8))
        out = Out(p(cols_out["score"]), p(cols_out["valid"]), p(cols_out["count"]), p(cols_out["length"]), p(cols_out["min_codon"]), p(cols_out["status"]), None, None)
        prm = Params(0.428571428571, 5, 0, 0, 0.0)
        for lo, hi in ((0, n), (n // 3, n - n // 5), (0, min(n, 1000))):
            check(lib.rt_score(ctx, p(cov), lo, hi, C.byref(prm), C.byref(out), None), ctx)
            digest(f"{name} layout {layout} rt_score [{lo}, {hi})")
        for parts in ("1", "3", "4", "16"):
            os.environ["RT_SCORE_HOST_PARTS"] = parts
            check(lib.rt_score_host(ctx, p(cov), 7, n - 3, C.byref(prm), C.byref(out)), ctx)
            digest(f"{name} layout {layout} rt_score_host parts {parts}")
        os.environ.pop("RT_SCORE_HOST_PARTS", None)
    lib.rt_destroy(ctx)
run_rows()
