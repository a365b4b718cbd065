"""BGZF-compressed inputs of prepare-orfs, orfs-seq and count-orfs-codon (DESIGN.md section 12).

CPU tests drive the host flow (sniffing, the ``*_load_text`` loaders, the commands and the CLI) with
``Engine.inflate_bgzf`` answered by zlib through ``rt_text_alloc``, and the device calls answered by the statement
engines of the commands' own test files.  The GPU tests check ``rt_bgzf_inflate`` (bgzf_inflate_kernel) against
``gzip.decompress`` on DEFLATE streams of every shape, its refusals, and the commands end to end on the real engine.
"""
from __future__ import annotations

import gzip
import os
import struct
import zlib
from collections import Counter

import numpy as np
import pytest

import test_count_orfs_codon as TC
import test_orfs_seq as TS
import test_prepare_orfs as TP
from bam_writer import BGZF_EOF, bgzf_block


# ------------------------------------------------------------------------------------------------ BGZF writers
def write_bgzf(path, data: bytes, block=0xFF00, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, eof=True) -> str:
    with open(path, "wb") as fh:
        for i in range(0, len(data), block):
            fh.write(bgzf_block(data[i:i + block], level, strategy))
        if eof:
            fh.write(BGZF_EOF)
    return str(path)


def member(deflate: bytes, payload: bytes, extra: bytes = b"") -> bytes:
    """One BGZF member around a raw DEFLATE stream; ``extra`` = subfields placed before 'BC'."""
    xlen = len(extra) + 6
    bsize = 12 + xlen + len(deflate) + 8 - 1
    return (b"\x1f\x8b\x08\x04" + struct.pack("<IBBH", 0, 0, 0xFF, xlen) + extra + b"BC" + struct.pack("<HH", 2, bsize)
            + deflate + struct.pack("<II", zlib.crc32(payload) & 0xFFFFFFFF, len(payload)))


def raw_deflate(payload: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_every=0) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    if not flush_every:
        return c.compress(payload) + c.flush()
    out = b""
    for i in range(0, len(payload), flush_every):
        out += c.compress(payload[i:i + flush_every]) + c.flush(zlib.Z_SYNC_FLUSH if i // flush_every % 2 else zlib.Z_FULL_FLUSH)
    return out + c.flush()


# A small DEFLATE encoder (RFC 1951) for streams zlib never writes: distance 32768, a dynamic block with a single
# distance code or none.  Tokens are literal byte values or (length, distance) pairs.
LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXT = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
         6145, 8193, 12289, 16385, 24577]
DEXT = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


class BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v, k):
        self.acc |= v << self.n
        self.n += k
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, k):                       # Huffman codes are sent most significant bit first
        self.bits(int(format(c, f"0{k}b")[::-1], 2) if k else 0, k)

    def done(self) -> bytes:
        if self.n:
            self.out.append(self.acc & 255)
        return bytes(self.out)


def canonical(lens):
    count = Counter(x for x in lens if x)
    code, nxt = 0, {}
    for b in range(1, 16):
        code = (code + count.get(b - 1, 0)) << 1
        nxt[b] = code
    out = {}
    for s, x in enumerate(lens):
        if x:
            out[s] = (nxt[x], x)
            nxt[x] += 1
    return out


def _encode(w, tokens, lit, dist):
    for t in tokens:
        if isinstance(t, int):
            w.code(*lit[t])
            continue
        n, d = t
        s = max(k for k in range(29) if LBASE[k] <= n)
        w.code(*lit[257 + s])
        w.bits(n - LBASE[s], LEXT[s])
        ds = max(k for k in range(30) if DBASE[k] <= d)
        w.code(*dist[ds])
        w.bits(d - DBASE[ds], DEXT[ds])
    w.code(*lit[256])


def fixed_deflate(tokens) -> bytes:
    w = BitWriter()
    w.bits(1, 1)
    w.bits(1, 2)
    _encode(w, tokens, canonical([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8), canonical([5] * 30))
    return w.done()


def dynamic_deflate(tokens, dist_lens) -> bytes:
    lit_lens = [9] * 256 + [5, 5] + [6] * 28          # 286 symbols, a complete code
    w = BitWriter()
    w.bits(1, 1)
    w.bits(2, 2)
    w.bits(len(lit_lens) - 257, 5)
    w.bits(len(dist_lens) - 1, 5)
    w.bits(19 - 4, 4)
    cl = canonical([4] * 16 + [0, 0, 0])
    for s in CL_ORDER:
        w.bits(4 if s < 16 else 0, 3)
    for x in lit_lens + dist_lens:
        w.code(*cl[x])
    _encode(w, tokens, canonical(lit_lens), canonical(dist_lens))
    return w.done()


def expand(tokens) -> bytes:
    out = bytearray()
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        else:
            for _ in range(t[0]):
                out.append(out[-t[1]])
    return bytes(out)


def text_of(seed: int, n: int, crlf=False) -> bytes:
    """Compressible annotation-like text."""
    rng = np.random.default_rng(seed)
    words = [b"chr1", b"exon", b"CDS", b"gene_id", b"ENSG000001", b"transcript_id", b"protein_coding", b"+", b"-"]
    out, eol = bytearray(), b"\r\n" if crlf else b"\n"
    while len(out) < n:
        line = b"\t".join(words[int(k)] for k in rng.integers(0, len(words), 6))
        out += line + b"\t" + str(int(rng.integers(1, 10 ** 8))).encode() + eol
        out += bytes(rng.choice(list(b"ACGT"), 60).tolist()) + eol
    return bytes(out[:n])


# ------------------------------------------------------------------------------------------------ CPU engine
class ZlibEngine(TP.StatementEngine, TS.StatementEngine, TC.StatementEngine):
    """The statement engines of the three commands, and ``inflate_bgzf`` answered by zlib through rt_text_alloc."""

    def __init__(self):
        super().__init__()
        self.inflated = []

    def inflate_bgzf(self, path, summary=None, stage_ms=None):
        data = gzip.decompress(open(path, "rb").read())
        self.inflated.append(str(path))
        return native_text(data, path)


def native_text(data: bytes, path):
    from ribotricer_b200.bgzf import NativeText

    t = NativeText.alloc(len(data), str(path))
    t.view()[:] = np.frombuffer(data, np.uint8)
    return t


@pytest.fixture
def zlib_engine(built, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    eng = ZlibEngine()
    monkeypatch.setattr(D, "_ENGINE", eng)
    return eng


@pytest.fixture
def gpu_engine(engine, monkeypatch):
    from ribotricer_b200 import detect_orfs as D

    monkeypatch.setattr(D, "_ENGINE", engine)
    return engine


@pytest.fixture(scope="module")
def annotation(tmp_path_factory):
    from ribotricer_b200 import synth

    return synth.make_annotation(str(tmp_path_factory.mktemp("annot")), n_genes=40, genome_size=400_000, seed=11)


def _bgz(path, tmp_path, **kw) -> str:
    return write_bgzf(os.path.join(str(tmp_path), os.path.basename(path) + ".bgz"), open(path, "rb").read(), **kw)


def _files_under(d) -> list:
    return [os.path.join(r, f) for r, _, fs in os.walk(d) for f in fs]


def _plain_gzip(path, tmp_path) -> str:
    out = os.path.join(str(tmp_path), os.path.basename(path) + ".gzip")
    with gzip.open(out, "wb") as fh:
        fh.write(open(path, "rb").read())
    return out


# ------------------------------------------------------------------------------------------------ sniffing
def test_sniff_tells_plain_bgzf_and_gzip(tmp_path, built):
    from ribotricer_b200.bgzf import sniff

    plain, short = tmp_path / "a.txt", tmp_path / "b.txt"
    plain.write_bytes(b"plain\n")
    short.write_bytes(b"\x1f\x8b")
    assert sniff(str(plain)) == "plain" and sniff(str(short)) == "gzip"
    assert sniff(_plain_gzip(str(plain), tmp_path)) == "gzip"
    assert sniff(write_bgzf(tmp_path / "c.bgz", b"x" * 100)) == "bgzf"
    other = tmp_path / "d.bgz"
    other.write_bytes(member(raw_deflate(b"abc"), b"abc", extra=b"XY\x03\x00xyz") + BGZF_EOF)
    assert sniff(str(other)) == "bgzf"
    empty = tmp_path / "e.bgz"
    empty.write_bytes(BGZF_EOF)
    assert sniff(str(empty)) == "bgzf"


# ------------------------------------------------------------------------------------------------ *_text loaders
def test_text_loaders_give_what_the_file_loaders_give(tmp_path, annotation, built):
    from ribotricer_b200.count_orfs import CodonInput
    from ribotricer_b200.index import load_native_index
    from ribotricer_b200.prepare_orfs import Genome, load_gtf

    text = lambda p: native_text(open(p, "rb").read(), p)  # noqa: E731
    g_file, g_text = load_gtf(annotation["gtf"]), load_gtf(text(annotation["gtf"]))
    assert g_file.keys() == g_text.keys()
    for k in g_file:
        assert np.array_equal(np.asarray(g_file[k]), np.asarray(g_text[k])), k
    f_file, f_text = Genome(annotation["fasta"]), Genome(text(annotation["fasta"]))
    assert f_file.names == f_text.names and np.array_equal(f_file.lengths, f_text.lengths)
    every = np.arange(len(f_file.names), dtype=np.int32)
    assert np.array_equal(f_file.codes(every), f_text.codes(every))
    idx, tsv, seq = TC.random_case(tmp_path, 3, n_rows=200)
    i_file, i_text = load_native_index(idx), load_native_index(text(idx))
    for k in ("exon_ptr", "exon_start", "exon_end", "orf_chrom_id", "orf_strand_code"):
        assert np.array_equal(getattr(i_file, k), getattr(i_text, k)), k
    assert i_file.chrom_names == i_text.chrom_names and i_file.n_annotated_prefix == i_text.n_annotated_prefix
    assert [np.array_equal(a, b) for a, b in zip(i_file.ids(), i_text.ids())] == [True, True]
    c_file, c_text = CodonInput(i_file, tsv, TC.FEATURES), CodonInput(i_text, text(tsv), TC.FEATURES)
    c_file.load_seq(seq)
    c_text.load_seq(text(seq))
    for k in c_file.sel:
        assert np.array_equal(c_file.sel[k], c_text.sel[k]), k
    assert bytes(c_file.text(0)) == bytes(c_text.text(0)) and bytes(c_file.text(1)) == bytes(c_text.text(1))


def test_text_loaders_give_the_file_loaders_errors(tmp_path, built):
    from ribotricer_b200.count_orfs import CodonInput
    from ribotricer_b200.index import load_native_index
    from ribotricer_b200.prepare_orfs import Genome, load_gtf

    def same_error(load, path):
        with pytest.raises(ValueError) as want:
            load(path)
        with pytest.raises(ValueError) as got:
            load(native_text(open(path, "rb").read(), path))
        assert str(got.value) == str(want.value) and path in str(got.value)

    gtf, fa = tmp_path / "bad.gtf", tmp_path / "dup.fa"
    gtf.write_text("#c\nc\tt\texon\tX\t10\t.\t+\t.\tgene_id \"g\";\n")
    fa.write_text(">a\nACGT\n>a\nGG\n")
    same_error(load_gtf, str(gtf))
    same_error(Genome, str(fa))
    bad_idx = tmp_path / "bad_idx.tsv"
    bad_idx.write_text(TC.INDEX_HEADER + "A\tuORF\tT\tpc\tG\tg\tpc\tc\t+\tATG\t5-x\n")
    same_error(load_native_index, str(bad_idx))
    idx, tsv, seq = TC._known(tmp_path)
    short = open(tsv).read().replace("\tATG\t[", "\t[", 1)
    bad_tsv = tmp_path / "short.tsv"
    bad_tsv.write_text(short)
    same_error(lambda p: CodonInput(load_native_index(idx), p, TC.FEATURES), str(bad_tsv))
    bad_seq = tmp_path / "seq.tsv"
    bad_seq.write_text(open(seq).read()[:-3])
    inp = lambda: CodonInput(load_native_index(idx), tsv, TC.FEATURES)  # noqa: E731
    same_error(lambda p: inp().load_seq(p), str(bad_seq))


# ------------------------------------------------------------------------------------------------ commands, CPU
def _prepare(tmp_path, gtf, fasta, name, capsys):
    from ribotricer_b200.prepare_orfs import prepare_orfs

    prefix = os.path.join(str(tmp_path), name, "idx")
    prepare_orfs(gtf, fasta, prefix, **TP.PARAM_SETS["near_cognate_min30"])
    text = open(prefix + "_candidate_orfs.tsv", "rb").read()
    return text, capsys.readouterr().out.replace(prefix, "PREFIX")


def _check_prepare(tmp_path, annotation, capsys):
    gtf, fa = annotation["gtf"], annotation["fasta"]
    bgtf, bfa = _bgz(gtf, tmp_path), _bgz(fa, tmp_path, level=1, block=10_000)
    want = _prepare(tmp_path, gtf, fa, "plain", capsys)
    assert want[0].count(b"\n") > 50
    for k, (g, f) in enumerate(((bgtf, fa), (gtf, bfa), (bgtf, bfa))):
        assert _prepare(tmp_path, g, f, f"bgzf{k}", capsys) == want


def _seq_run(tmp_path, idx, fa, protein, name):
    from ribotricer_b200.orf_seq import orf_seq

    out = os.path.join(str(tmp_path), name, "seq.tsv")
    orf_seq(idx, fa, out, protein)
    return open(out, "rb").read()


def _check_seq(tmp_path, annotation):
    idx = TS._index_file(tmp_path, annotation, TS.PARAM_SETS["defaults"])
    fa = annotation["fasta"]
    bidx, bfa = _bgz(idx, tmp_path, level=9), _bgz(fa, tmp_path, strategy=zlib.Z_RLE)
    for protein in (False, True):
        want = _seq_run(tmp_path, idx, fa, protein, f"plain{protein}")
        assert want.count(b"\n") > 50
        for k, (i, f) in enumerate(((bidx, fa), (idx, bfa), (bidx, bfa))):
            assert _seq_run(tmp_path, i, f, protein, f"bgzf{protein}{k}") == want


def _codon_run(tmp_path, *args, name):
    gene, codon, summary = TC._run(tmp_path, *args, name=name)
    return gene, codon, {k: v for k, v in summary.items() if k not in ("gene_table", "codon_table")}


def _check_codon(tmp_path):
    idx, tsv, seq = TC.random_case(tmp_path, 5, big=True)
    want = _codon_run(tmp_path, idx, tsv, seq, name="plain")
    assert want[2]["rows"] > 50
    b = [_bgz(p, tmp_path, block=4000) for p in (idx, tsv, seq)]
    for k, args in enumerate(((b[0], tsv, seq), (idx, b[1], seq), (idx, tsv, b[2]), tuple(b))):
        assert _codon_run(tmp_path, *args, name=f"bgzf{k}") == want


def test_prepare_orfs_from_bgzf_writes_the_same_bytes(tmp_path, annotation, zlib_engine, capsys):
    _check_prepare(tmp_path, annotation, capsys)
    assert len(zlib_engine.inflated) == 4


def test_orfs_seq_from_bgzf_writes_the_same_bytes(tmp_path, annotation, zlib_engine):
    _check_seq(tmp_path, annotation)
    assert len(zlib_engine.inflated) == 8


def test_count_orfs_codon_from_bgzf_writes_the_same_bytes(tmp_path, zlib_engine):
    _check_codon(tmp_path)
    assert len(zlib_engine.inflated) == 6


def test_plain_gzip_keeps_todays_message(tmp_path, annotation, zlib_engine):
    from ribotricer_b200.count_orfs import count_orfs_codon
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    gtf, fa = annotation["gtf"], annotation["fasta"]
    out = str(tmp_path / "out")
    for g, f in ((_plain_gzip(gtf, tmp_path), fa), (gtf, _plain_gzip(fa, tmp_path))):
        bad = g if g != gtf else f
        with pytest.raises(ValueError, match=f"^{bad} is gzip-compressed; prepare-orfs reads plain text only$"):
            prepare_orfs(g, f, os.path.join(out, "p"))
    idx = TS._index_file(tmp_path, annotation, TS.PARAM_SETS["defaults"])
    for i, f in ((_plain_gzip(idx, tmp_path), fa), (idx, _plain_gzip(fa, tmp_path))):
        bad = i if i != idx else f
        with pytest.raises(ValueError, match=f"^{bad} is gzip-compressed; orfs-seq reads plain text only$"):
            orf_seq(i, f, os.path.join(out, "s.tsv"))
    cidx, tsv, seq = TC._known(tmp_path)
    for k in range(3):
        args = [cidx, tsv, seq]
        args[k] = _plain_gzip(args[k], tmp_path)
        with pytest.raises(ValueError, match=f"^{args[k]} is gzip-compressed; count-orfs-codon reads plain text only$"):
            count_orfs_codon(args[0], args[1], TC.FEATURES, args[2], os.path.join(out, "c"))
    assert _files_under(out) == [] and zlib_engine.inflated == []
    # a plain gzip input is refused before a BGZF one is inflated
    bfa, bidx = _bgz(fa, tmp_path), _bgz(cidx, tmp_path)
    gz_gtf, gz_seq = _plain_gzip(gtf, tmp_path), _plain_gzip(seq, tmp_path)
    with pytest.raises(ValueError, match="gzip-compressed; prepare-orfs"):
        prepare_orfs(gz_gtf, bfa, os.path.join(out, "p"))
    with pytest.raises(ValueError, match="gzip-compressed; orfs-seq"):
        orf_seq(_bgz(idx, tmp_path), _plain_gzip(fa, tmp_path), os.path.join(out, "s.tsv"))
    with pytest.raises(ValueError, match="gzip-compressed; count-orfs-codon"):
        count_orfs_codon(bidx, tsv, TC.FEATURES, gz_seq, os.path.join(out, "c"))
    assert _files_under(out) == [] and zlib_engine.inflated == []


def test_cli_reads_bgzf_and_keeps_the_compressed_name_message(tmp_path, annotation, zlib_engine):
    from click.testing import CliRunner

    from ribotricer_b200.cli import cli
    from ribotricer_b200.prepare_orfs import prepare_orfs

    gtf, fa = annotation["gtf"], annotation["fasta"]
    want = os.path.join(str(tmp_path), "py", "idx")
    prepare_orfs(gtf, fa, want)
    bgtf = write_bgzf(tmp_path / "a.gtf.gz", open(gtf, "rb").read())
    bfa = write_bgzf(tmp_path / "a.fa.bgz", open(fa, "rb").read())
    prefix = os.path.join(str(tmp_path), "cli", "idx")
    res = CliRunner().invoke(cli, ["prepare-orfs", "--gtf", bgtf, "--fasta", bfa, "--prefix", prefix])
    assert res.exit_code == 0, res.output
    assert open(prefix + "_candidate_orfs.tsv", "rb").read() == open(want + "_candidate_orfs.tsv", "rb").read()
    pgz = _plain_gzip(gtf, tmp_path)
    named = os.path.join(str(tmp_path), "plain.gtf.gz")
    os.replace(pgz, named)
    res = CliRunner().invoke(cli, ["prepare-orfs", "--gtf", named, "--fasta", fa, "--prefix", prefix + "2"])
    assert res.exit_code != 0
    assert str(res.exception) == (f"Error: GTF file {named} is compressed; prepare-orfs reads plain text only "
                                  "(decompress it first)")
    res = CliRunner().invoke(cli, ["prepare-orfs", "--gtf", gtf, "--fasta", _plain_gzip(fa, tmp_path), "--prefix",
                                   prefix + "3"])
    assert res.exit_code != 0 and "is gzip-compressed; prepare-orfs reads plain text only" in str(res.exception)
    # orfs-seq and count-orfs-codon from BGZF through the CLI
    idx = TS._index_file(tmp_path, annotation, TS.PARAM_SETS["defaults"])
    seq_want = _seq_run(tmp_path, idx, fa, True, "seq_py")
    out = os.path.join(str(tmp_path), "cli_seq", "seq.tsv")
    res = CliRunner().invoke(cli, ["orfs-seq", "--ribotricer_index", _bgz(idx, tmp_path), "--fasta", bfa, "--saveto", out,
                                   "--protein"])
    assert res.exit_code == 0, res.output
    assert open(out, "rb").read() == seq_want
    cidx, tsv, seq = TC.random_case(tmp_path, 9)
    c_want = TC._run(tmp_path, cidx, tsv, seq, features={"uORF", "annotated"}, report_all=True)
    cprefix = str(tmp_path / "cli_codon" / "run")
    res = CliRunner().invoke(cli, ["count-orfs-codon", "--ribotricer_index", _bgz(cidx, tmp_path), "--detected_orfs",
                                   _bgz(tsv, tmp_path), "--features", "uORF,annotated", "--ribotricer_index_fasta",
                                   _bgz(seq, tmp_path), "--prefix", cprefix, "--report_all"])
    assert res.exit_code == 0, res.output
    assert open(cprefix + "_codon_counts_by_gene.tsv", "rb").read().decode("latin-1") == c_want[0]
    assert open(cprefix + "_codon_counts.tsv", "rb").read().decode("latin-1") == c_want[1]


# ------------------------------------------------------------------------------------------------ GPU: the decoder
def _far_and_long():
    rng = np.random.default_rng(1)
    lits = [int(x) for x in rng.integers(0, 256, 32768)]
    tokens = lits + [(258, 32768), (258, 1), (3, 32768), (258, 258)]
    return [member(fixed_deflate(tokens), expand(tokens))]


def _dynamic(dist_lens, with_matches):
    text = text_of(5, 3000)
    tokens = [int(b) for b in text]
    if with_matches:                                   # the one distance code is symbol 3: distance 4
        tokens += [(20, 4), 65, (258, 4), (3, 4)]
    return [member(dynamic_deflate(tokens, dist_lens), expand(tokens))]


def _cases():
    big = text_of(1, 0xFF00 * 3 + 1234)
    rng = np.random.default_rng(2)
    noisy = bytes(rng.integers(32, 127, 0xFF00, dtype=np.uint8))       # many literals: several DEFLATE blocks
    small = text_of(4, 20_500 * 40)
    return {
        "stored": [bgzf_block(big[i:i + 0xFF00], 0) for i in range(0, len(big), 0xFF00)],
        "fixed": [bgzf_block(big[i:i + 0xFF00], 6, zlib.Z_FIXED) for i in range(0, len(big), 0xFF00)],
        "level1": [bgzf_block(big[i:i + 0xFF00], 1) for i in range(0, len(big), 0xFF00)],
        "level9": [bgzf_block(big[i:i + 0xFF00], 9) for i in range(0, len(big), 0xFF00)],
        "huffman_only": [bgzf_block(big[i:i + 0xFF00], 6, zlib.Z_HUFFMAN_ONLY) for i in range(0, len(big), 0xFF00)],
        "rle": [bgzf_block(big[i:i + 0xFF00], 6, zlib.Z_RLE) for i in range(0, len(big), 0xFF00)],
        "filtered": [bgzf_block(big[i:i + 0xFF00], 6, zlib.Z_FILTERED) for i in range(0, len(big), 0xFF00)],
        "several_blocks": [bgzf_block(noisy), member(raw_deflate(big[:0xFF00], flush_every=5000), big[:0xFF00])],
        "empty_and_64k": [bgzf_block(b""), bgzf_block(text_of(3, 65536)), bgzf_block(b"")],
        "distance_32768_length_258": _far_and_long(),
        "dynamic_one_distance_code": _dynamic([0, 0, 0, 1], True),
        "dynamic_no_distance_code": _dynamic([0], False),
        "subfield_before_bc": [member(raw_deflate(big[:5000]), big[:5000], extra=b"XY\x03\x00xyz")],
        "many_members": [bgzf_block(small[i:i + 40]) for i in range(0, len(small), 40)],
        "crlf": [bgzf_block(text_of(6, 200_000, crlf=True)[i:i + 0xFF00]) for i in range(0, 200_000, 0xFF00)],
    }


def _inflate(engine, path):
    summary = np.zeros(4, np.int64)
    ms = np.zeros(7, np.float32)
    t = engine.inflate_bgzf(path, summary=summary, stage_ms=ms)
    return bytes(t.view()), summary, ms


@pytest.mark.gpu
@pytest.mark.parametrize("eof", [True, False])
def test_gpu_inflate_matches_gzip(tmp_path, engine, eof):
    for name, members in _cases().items():
        path = tmp_path / f"{name}.bgz"
        data = b"".join(members) + (BGZF_EOF if eof else b"")
        path.write_bytes(data)
        got, summary, ms = _inflate(engine, str(path))
        want = gzip.decompress(data)
        assert got == want, name
        assert summary.tolist() == [len(members) + eof, len(data), len(want), 0], name
        assert (ms >= 0).all()
    assert len(_cases()["many_members"]) > 20_000


RULE4_KINDS = ("header", "truncated", "trailing", "crc", "isize")


def _broken(kind, text=None, block=0xFF00):
    """(file bytes, member number, its byte offset, message) for one rule-4 case made from ``text``."""
    text = text_of(7, 0xFF00 * 3) if text is None else text
    ms = [bgzf_block(text[i:i + block]) for i in range(0, len(text), block)]
    assert len(ms) >= 3
    at, m, rest = len(ms[0]), bytearray(ms[1]), b"".join(ms[2:])
    if kind == "header":
        m[12:14] = b"BD"
        return ms[0] + bytes(m) + rest + BGZF_EOF, 1, at, "not a BGZF member header"
    if kind == "truncated":
        data = b"".join(ms)
        return data[:-10], len(ms) - 1, len(data) - len(ms[-1]), "truncated, the file ends inside it"
    if kind == "trailing":
        data = b"".join(ms) + BGZF_EOF
        return data + b"trailing", len(ms) + 1, len(data), "bytes after the last member are not a BGZF member"
    if kind == "crc":
        m[-8] ^= 1
    elif kind == "isize":
        m[-4:] = struct.pack("<I", struct.unpack("<I", bytes(m[-4:]))[0] + 1)
    elif kind == "payload":
        m[len(m) // 2] ^= 0x5A
    return ms[0] + bytes(m) + rest + BGZF_EOF, 1, at, "does not inflate to its ISIZE of"


@pytest.mark.gpu
def test_gpu_refuses_broken_files_naming_the_member(tmp_path, engine):
    for kind in RULE4_KINDS + ("payload",):
        data, k, at, message = _broken(kind)
        path = tmp_path / f"{kind}.bgz"
        path.write_bytes(data)
        summary = np.zeros(4, np.int64)
        with pytest.raises(ValueError) as err:
            engine.inflate_bgzf(str(path), summary=summary)
        assert str(err.value).startswith(f"{path}: BGZF block {k} at byte {at}: "), (kind, str(err.value))
        assert message in str(err.value), kind
        if kind in ("crc", "isize", "payload"):
            assert summary[3] == 1, kind                  # the device refused it, then the host did


@pytest.mark.gpu
def test_gpu_commands_leave_no_file_on_a_broken_input(tmp_path, annotation, gpu_engine):
    from ribotricer_b200.count_orfs import count_orfs_codon
    from ribotricer_b200.orf_seq import orf_seq
    from ribotricer_b200.prepare_orfs import prepare_orfs

    out = str(tmp_path / "out")
    idx = TS._index_file(tmp_path, annotation, TS.PARAM_SETS["defaults"])
    cidx, tsv, seq = TC.random_case(tmp_path, 5)
    runs = [(annotation["fasta"], lambda f: prepare_orfs(annotation["gtf"], f, os.path.join(out, "p"))),
            (annotation["gtf"], lambda g: prepare_orfs(g, annotation["fasta"], os.path.join(out, "p"))),
            (idx, lambda i: orf_seq(i, annotation["fasta"], os.path.join(out, "s.tsv"))),
            (annotation["fasta"], lambda f: orf_seq(idx, f, os.path.join(out, "s.tsv"))),
            (cidx, lambda i: count_orfs_codon(i, tsv, TC.FEATURES, seq, os.path.join(out, "c"))),
            (tsv, lambda t: count_orfs_codon(cidx, t, TC.FEATURES, seq, os.path.join(out, "c"))),
            (seq, lambda q: count_orfs_codon(cidx, tsv, TC.FEATURES, q, os.path.join(out, "c")))]
    for kind in RULE4_KINDS:
        for r, (src, run) in enumerate(runs):
            data, k, at, message = _broken(kind, open(src, "rb").read(), block=2000)
            bad = os.path.join(str(tmp_path), f"{kind}{r}_{os.path.basename(src)}.bgz")
            open(bad, "wb").write(data)
            with pytest.raises(ValueError) as err:
                run(bad)
            assert str(err.value).startswith(f"{bad}: BGZF block {k} at byte {at}: ") and message in str(err.value), \
                (kind, r, str(err.value))
            assert _files_under(out) == [], (kind, r)


# ------------------------------------------------------------------------------------------------ GPU: end to end
@pytest.mark.gpu
def test_gpu_prepare_orfs_from_bgzf(tmp_path, annotation, gpu_engine, capsys):
    _check_prepare(tmp_path, annotation, capsys)


@pytest.mark.gpu
def test_gpu_orfs_seq_from_bgzf(tmp_path, annotation, gpu_engine):
    _check_seq(tmp_path, annotation)


@pytest.mark.gpu
def test_gpu_count_orfs_codon_from_bgzf(tmp_path, gpu_engine):
    _check_codon(tmp_path)
