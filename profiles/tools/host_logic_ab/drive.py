"""Run the HOST logic of one build of the library under the fake cudart and print a digest of every host-to-device upload:
set_genome, set_index (+ layout), rt_score over several ranges and rt_score_host in parts, for several synthetic indexes."""
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

def digest(tag):
    n = fake.fake_log_size(); buf = (C.c_ulonglong * max(1, n))(); fake.fake_log_copy(buf); fake.fake_log_clear()
    raw = bytes(buf)[:8 * n]
    print(f"{tag}: {n // 2} uploads, {sum(buf[i] for i in range(0, n, 2))} bytes, md5 {hashlib.md5(raw).hexdigest()}")

def check(rc, ctx):
    assert rc == 0, lib.rt_last_error(ctx)

p = lambda a: a.ctypes.data_as(vp)
cases = [("tiny", 1.0, 1.0), ("C1", 0.3, 1.0), ("C5", 0.02, 0.05), ("C2", 0.5, 0.5)]
for name, scale, cscale in cases:
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
