"""Host-side logic that needs no GPU: CLI validation, index parsing, sharding arithmetic."""
import os

import numpy as np
import pytest


def test_cli_validation(tmp_path):
    """Flag validation messages of cli.py:236-270 (no GPU work happens on these paths)."""
    from click.testing import CliRunner

    from ribotricer_b200.cli import cli

    f = tmp_path / "x.npz"
    f.write_bytes(b"")
    i = tmp_path / "i.tsv"
    i.write_text("h\n")
    run = CliRunner().invoke
    base = ["detect-orfs", "--bam", str(f), "--ribotricer_index", str(i), "--prefix", str(tmp_path / "p")]
    r = run(cli, ["detect-orfs", "--bam", "nope", "--ribotricer_index", str(i), "--prefix", "p"])
    assert "Error: BAM file not found" in str(r.exception) or "Error: BAM file not found" in r.output
    r = run(cli, base + ["--psite_offsets", "12"])
    assert "psite_offsets only allowed when read_lengths is provided" in str(r.exception) + r.output
    r = run(cli, base + ["--read_lengths", "28,29", "--psite_offsets", "12"])
    assert "psite_offsets must match read_lengths" in str(r.exception) + r.output
    r = run(cli, base + ["--read_lengths", "28", "--psite_offsets", "28"])
    assert "P-site offset must be smaller than read length" in str(r.exception) + r.output
    r = run(cli, base + ["--read_lengths", "a"])
    assert "cannot convert read_lengths into integers" in str(r.exception) + r.output


def test_index_parser_matches_reference_rules(tmp_path):
    """orf.py:121-182: 11 columns, intervals sorted by start, oid re-derived (orf.py:100-103)."""
    import pytest

    from ribotricer_b200.index import ORF, parse_index

    p = tmp_path / "idx.tsv"
    p.write_text("ORF_ID\tORF_type\ttranscript_id\ttranscript_type\tgene_id\tgene_name\tgene_type\tchrom\tstrand\tstart_codon\tcoordinate\n"
                 "IGNORED\tannotated\ttxA\tprotein_coding\tgA\tGA\tprotein_coding\tchrI\t+\tATG\t201-212,101-109\n"
                 "IGNORED\tuORF\ttxB\tprotein_coding\tgB\tGB\tprotein_coding\tchrI\t-\tCTG\t301-318\n")
    idx = parse_index(str(p))
    assert idx.n_orf == 2 and idx.n_annotated_prefix == 1
    assert idx.exon_start.tolist() == [101, 201, 301] and idx.exon_end.tolist() == [109, 212, 318]
    assert idx.oid(0) == "txA_101_212_21" and idx.oid(1) == "txB_301_318_18"
    assert idx.lengths().tolist() == [21, 18]
    orf = ORF.from_string("x\tannotated\ttxA\tpc\tgA\tGA\tpc\tchrI\t+\tATG\t201-212,101-109\n")
    assert orf.oid == "txA_101_212_21" and orf.intervals == [(101, 109), (201, 212)]
    with pytest.raises(SystemExit):
        ORF.from_string("too\tfew\tcolumns")
    cols = idx.device_columns({"chrI": 0})
    assert cols["orf_contig"].tolist() == [0, 0] and cols["orf_strand"].tolist() == [0, 1]
    assert idx.device_columns({})["orf_contig"].tolist() == [-1, -1]


def test_native_index_loader_matches_python_rules(tmp_path, built):
    """csrc/rt_host_io.cpp against the Python statement of orf.py:121-182 on the golden indexes
    (shuffled interval order, unknown chromosomes) and on a synthetic 3,000-row index."""
    import pytest

    from helpers import load_golden
    from ribotricer_b200 import synth
    from ribotricer_b200.index import NativeIndex, parse_index

    paths = []
    for case in load_golden("pipeline_cases.json.gz")["cases"]:
        p = tmp_path / f"{case['name']}.tsv"
        p.write_text("\n".join(case["index"]) + "\n")
        paths.append(str(p))
    p = tmp_path / "synth.tsv"
    synth.make_index(synth.config("tiny")).write_tsv(str(p))
    paths.append(str(p))
    for path in paths:
        py, nat = parse_index(path), NativeIndex(path)
        assert nat.n_orf == py.n_orf and nat.n_annotated_prefix == py.n_annotated_prefix
        for k in ("exon_ptr", "exon_start", "exon_end"):
            assert (getattr(nat, k) == getattr(py, k)).all(), k
        assert nat.contig_table() == py.contig_table()
        lut = {c: i for i, c in enumerate(py.contig_table()[:-1])}      # last chromosome unknown to the "BAM"
        a, b = nat.device_columns(lut), py.device_columns(lut)
        for k in a:
            assert (a[k] == b[k]).all(), k
        for o in list(range(0, py.n_orf, max(1, py.n_orf // 50))) + [py.n_orf - 1]:
            assert nat.fields[o] == py.fields[o] and nat.chrom[o] == py.chrom[o] and nat.strand[o] == py.strand[o]
            assert nat.oid(o) == py.oid(o)
        assert (nat.lengths() == py.lengths()).all()
    bad = tmp_path / "bad.tsv"
    bad.write_text("h\na\tb\tc\n")
    with pytest.raises(SystemExit) as exc:
        NativeIndex(str(bad))
    assert "unexpected number of columns" in str(exc.value)


def test_native_index_loader_chunked_parse(tmp_path, built, monkeypatch):
    """A large index is parsed in chunks by several threads and merged: forced here on small files (RT_INDEX_THREADS).
    Columns, chromosome order (first appearance in the file), the annotated prefix and every field must equal the
    one-thread parse; the FIRST bad row in file order decides the error, as in the reference's row-by-row loop."""
    import pytest

    from ribotricer_b200 import synth
    from ribotricer_b200.index import NativeIndex

    p = tmp_path / "synth.tsv"
    synth.make_index(synth.config("tiny")).write_tsv(str(p))
    lines = p.read_text().split("\n")
    # a chromosome that first appears late, rows with shuffled and negative coordinates, the annotated prefix broken early
    row = lines[5].split("\t")
    lines.insert(900, "\t".join(row[:7] + ["chrLate", "-", "ATG", "300-310,-5-20,100-120"]))
    lines.insert(3, "\t".join(row[:1] + ["novel"] + row[2:]))
    p.write_text("\n".join(lines))
    monkeypatch.setenv("RT_INDEX_THREADS", "1")
    want = NativeIndex(str(p))
    assert want.n_annotated_prefix == 2
    for threads in (2, 3, 7, 16, 64):
        monkeypatch.setenv("RT_INDEX_THREADS", str(threads))
        got = NativeIndex(str(p))
        assert got.n_orf == want.n_orf and got.n_annotated_prefix == want.n_annotated_prefix
        for k in ("exon_ptr", "exon_start", "exon_end"):
            assert (getattr(got, k) == getattr(want, k)).all(), (threads, k)
        assert got.contig_table() == want.contig_table()
        assert list(got.chrom) == list(want.chrom) and list(got.strand) == list(want.strand)
        for o in range(0, want.n_orf, 7):
            assert got.fields[o] == want.fields[o] and got.oid(o) == want.oid(o)
    # errors: the earlier of a bad coordinate (row 1,501) and a short row (row 2,001) wins, whatever the chunking
    body = p.read_text().split("\n")
    body[1501] = body[1501].rsplit("\t", 1)[0] + "\t12-x"
    body[2001] = "a\tb"
    p.write_text("\n".join(body))
    for threads in (1, 5, 16):
        monkeypatch.setenv("RT_INDEX_THREADS", str(threads))
        with pytest.raises((SystemExit, OSError, ValueError)) as exc:
            NativeIndex(str(p))
        assert "bad coordinate in index row 1501" in str(exc.value), threads
    body[1000] = "a\tb"
    p.write_text("\n".join(body))
    for threads in (1, 5, 16):
        monkeypatch.setenv("RT_INDEX_THREADS", str(threads))
        with pytest.raises(SystemExit) as exc:
            NativeIndex(str(p))
        assert "unexpected number of columns" in str(exc.value)


def test_native_tsv_writer_matches_reference_formatting(tmp_path, built):
    """rt_tsv_write rows against the rows the reference wrote (golden TSV text): feeding the
    writer the reference's own numbers must reproduce its text byte for byte (float repr, int/int
    ratio, np.float64 density, list repr of the profile)."""
    import ctypes as C

    from helpers import load_golden
    from ribotricer_b200 import _lib
    from ribotricer_b200.index import NativeIndex

    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    # + rows whose start_codon field is not three characters long (the TSV prints ORF.start_codon, orf.py:108-119)
    for case in load_golden("pipeline_cases.json.gz")["cases"] + load_golden("start_codon_case.json.gz")["cases"]:
        path = tmp_path / f"{case['name']}.tsv"
        path.write_text("\n".join(case["index"]) + "\n")
        idx = NativeIndex(str(path))
        for run in case["tsv"]:
            ref_lines = run["text"].split("\n")
            rows = [r.split("\t") for r in ref_lines[1:] if r]
            # rows are in index order; oids can repeat, so match them sequentially
            sel, o = [], 0
            for r in rows:
                while idx.oid(o) != r[0] or "\t".join(idx.fields[o][1:6]) != "\t".join(r[9:14]):
                    o += 1
                sel.append(o)
                o += 1
            sel = np.array(sel, np.int64)
            n = idx.n_orf
            score, valid = np.zeros(n), np.zeros(n, np.int32)
            count, length, status = np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.uint8)
            profs = []
            for o, r in zip(sel, rows):
                score[o], count[o], length[o], valid[o] = float(r[3]), int(r[4]), int(r[5]), int(r[6])
                status[o] = r[2] == "translating"
                profs.append(np.array(eval(r[17]), np.int32))
            ptr = np.zeros(len(sel) + 1, np.int64)
            np.cumsum([len(x) for x in profs], out=ptr[1:])
            prof = np.concatenate(profs) if profs else np.zeros(0, np.int32)
            out = tmp_path / "out.tsv"
            h = C.c_void_p()
            assert lib.rt_tsv_open(str(out).encode(), 1, C.byref(h)) == 0
            assert lib.rt_tsv_write(h, idx.handle, len(sel), p(sel), 0, p(score), p(valid), p(count), p(length),
                                    p(status), p(ptr), p(prof)) == 0
            assert lib.rt_tsv_close(h) == 0
            assert out.read_text() == run["text"]


@pytest.mark.parametrize("rows", [0, 3000])
def test_tsv_writer_reports_a_refused_write(tmp_path, built, rows):
    """A disk that refuses the text: with no rows the header fails when the file is closed, with megabytes of rows
    the write-behind thread meets the failure; either way the caller gets an error code and a message, and the
    close returns (the writer thread is not left waiting)."""
    import ctypes as C

    from helpers import load_golden
    from ribotricer_b200 import _lib
    from ribotricer_b200.index import NativeIndex

    if not os.path.exists("/dev/full"):
        pytest.skip("no /dev/full")
    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    path = tmp_path / "idx.tsv"
    path.write_text("\n".join(load_golden("pipeline_cases.json.gz")["cases"][0]["index"]) + "\n")
    idx = NativeIndex(str(path))
    n = idx.n_orf
    sel = np.zeros(rows, np.int64)                      # one ORF, many times, with a long profile each
    score, valid = np.full(n, 0.5), np.ones(n, np.int32)
    count, length, status = np.full(n, 7, np.int64), np.full(n, 30, np.int32), np.ones(n, np.uint8)
    ptr = np.arange(rows + 1, dtype=np.int64) * 1000
    prof = np.full(rows * 1000, 12, np.int32)
    assert lib.rt_tsv_open(str(tmp_path / "missing" / "x.tsv").encode(), 1, C.byref(C.c_void_p())) != 0
    assert lib.rt_io_last_error().decode().startswith("cannot open")
    h = C.c_void_p()
    assert lib.rt_tsv_open(b"/dev/full", 1, C.byref(h)) == 0
    for _ in range(3):                                  # a write may or may not see the failure yet: it is asynchronous
        lib.rt_tsv_write(h, idx.handle, rows, p(sel), 0, p(score), p(valid), p(count), p(length), p(status), p(ptr), p(prof))
    rc = lib.rt_tsv_close(h)
    assert rc != 0                                      # the close reports it whatever the writes returned
    assert "write failed" in lib.rt_io_last_error().decode()


def test_repr_double_is_python_repr(built):
    import ctypes as C

    from ribotricer_b200 import _lib

    lib = _lib.load()
    buf = C.create_string_buffer(64)
    rng = np.random.default_rng(2)
    vals = [0.0, 1.0, 0.5, 1e-5, 1e-4, 123456789.0, 1e15, 1e16, 1.5e16, 1e22, 1 / 3, 5e-324, 1.7976931348623157e308,
            0.1 + 0.2, 100.0] + rng.random(3000).tolist() + (10.0 ** rng.uniform(-12, 22, 3000)).tolist()
    for v in vals:
        lib.rt_repr_double(float(v), buf, 64)
        assert buf.value.decode() == repr(float(v)) == str(np.float64(v))


def _expected_span(pos, cigar):
    """get_reference_positions() semantics (bam.py:95-99): positions of M, = and X only."""
    positions, cur = [], pos
    for op, length in cigar:
        if op in "M=X":
            positions.extend(range(cur, cur + length))
            cur += length
        elif op in "DN":
            cur += length
    if not positions:
        return 0, 0, 0
    return positions[0], positions[-1], len(positions)


def test_native_bam_decoder(tmp_path, built):
    """csrc/rt_bam.cpp on BAM files written by tests/bam_writer.py: CIGARs with every operation,
    NH tags of every integer type hidden among other aux fields, unmapped records, records that
    straddle BGZF blocks, multi-threaded and single-threaded."""
    import bam_writer as W
    import pytest
    from ribotricer_b200.bam import load_reads, read_bam_columns_native

    rng = np.random.default_rng(4)
    refs = [("chrI", 230218), ("chrII", 813184), ("chrM", 85779)]
    recs, exp = [], []
    for i in range(30000):
        kind = rng.random()
        if kind < 0.03:                       # unmapped, no CIGAR
            flag, ref_id, pos, cigar = 4, -1, -1, []
        else:
            flag = int(rng.choice([0, 16, 256, 272, 1024, 512, 2048, 0, 16, 0]))
            ref_id = int(rng.integers(0, len(refs)))
            pos = int(rng.integers(0, refs[ref_id][1] - 500))
            cigar = []
            if rng.random() < 0.3:
                cigar.append(("S", int(rng.integers(1, 6))))
            for k in range(int(rng.integers(1, 7))):
                cigar.append((str(rng.choice(list("MMMM=XIDN"))), int(rng.integers(1, 40))))
            if rng.random() < 0.2:
                cigar.append((str(rng.choice(list("SHP"))), int(rng.integers(1, 5))))
        mapq = int(rng.choice([0, 1, 3, 255, 60]))
        aux, nh = b"", 0
        if rng.random() < 0.5:
            aux += W.aux_field("NM", "i", int(rng.integers(0, 5))) + W.aux_field("MD", "Z", "10A5^AC6")
        if rng.random() < 0.3:
            aux += W.aux_field("XS", "A", "+") + W.aux_field("ZB", "Bs", [1, -2, 3]) + W.aux_field("XF", "f", 1.5)
        if rng.random() < 0.8:
            typ = str(rng.choice(list("cCsSiI")))
            nh = int(rng.choice([1, 1, 1, 2, 3, 10, 100, 300 if typ in "sSiI" else 7]))
            aux += W.aux_field("NH", typ, nh)
        if rng.random() < 0.3:
            aux += W.aux_field("HI", "C", 1) + W.aux_field("ZZ", "BI", list(range(int(rng.integers(0, 9)))))
        recs.append(W.record(ref_id, pos, mapq, flag, cigar, name=b"read%d" % i, aux=aux))
        first, last, n = _expected_span(pos, cigar)
        exp.append((ref_id, first, last, n, flag, mapq, min(nh, 255)))
    path = tmp_path / "t.bam"
    W.write_bam(str(path), refs, recs, sorted_header=True, block_payload=4099)   # odd size: records split everywhere
    exp = np.array(exp, np.int64)
    for threads in (1, 4):
        rc = read_bam_columns_native(str(path), threads)
        assert rc.contig_names == [r[0] for r in refs] and rc.contig_len.tolist() == [r[1] for r in refs]
        assert rc.sorted_by_coordinate and len(rc) == len(recs)
        for j, name in enumerate(("ref_id", "first", "last", "mlen", "flag", "mapq", "nh")):
            assert (rc.cols[name].astype(np.int64) == exp[:, j]).all(), name
    W.write_bam(str(path), refs, recs[:100], sorted_header=False)
    rc = load_reads(str(path))
    assert not rc.sorted_by_coordinate and len(rc) == 100
    bad = tmp_path / "bad.bam"
    bad.write_bytes(b"not a bam file at all")
    with pytest.raises(OSError):
        read_bam_columns_native(str(bad))


def test_count_orfs_text_matches_reference(tmp_path, built):
    """ribotricer_b200.count_orfs.count_orfs (same signature as count_orfs.py:28) on the golden TSVs."""
    from helpers import load_golden
    from ribotricer_b200.count_orfs import count_orfs

    pipe = {c["name"]: c for c in load_golden("pipeline_cases.json.gz")["cases"]}
    n = 0
    for c in load_golden("count_orfs_cases.json.gz")["cases"]:
        case = pipe[c["case"]]
        idx = tmp_path / "idx.tsv"
        idx.write_text("\n".join(case["index"]) + "\n")
        tsv = tmp_path / "in.tsv"
        tsv.write_text(case["tsv"][c["tsv"]]["text"])
        out = tmp_path / "counts.tsv"
        count_orfs(str(idx), str(tsv), set(c["features"]), str(out), c["report_all"])
        assert out.read_text() == c["text"], (c["case"], c["tsv"], c["features"], c["report_all"])
        n += 1
    assert n == 72


def _stream_columns(seed=5, n=60_000):
    """Sorted read columns with everything the record stream has to code: spliced reads, reads longer than 255,
    gaps above 32,767 and above 2^30, several references, flag-decided reads with junk positions, an unmapped tail."""
    rng = np.random.default_rng(seed)
    ref = np.sort(rng.choice([0, 1, 2, 5], n, p=[0.5, 0.3, 0.15, 0.05])).astype(np.int32)
    step = rng.choice([0, 0, 1, 3, 40, 900, 40_000, 70_000], n, p=[0.3, 0.2, 0.2, 0.15, 0.1, 0.03, 0.015, 0.005]).astype(np.int64)
    first = np.zeros(n, np.int64)
    for r in np.unique(ref):
        m = ref == r
        first[m] = np.cumsum(step[m])
    big = np.flatnonzero(ref == 5)
    first[big[len(big) // 2:]] += (1 << 30) + 12345          # one jump that no skip record holds
    mlen = rng.choice([0, 1, 26, 28, 29, 30, 32, 150, 255, 256, 300, 5000], n,
                      p=[0.002, 0.008, 0.2, 0.3, 0.2, 0.1, 0.1, 0.04, 0.02, 0.01, 0.01, 0.01]).astype(np.int64)
    extra = np.where(rng.random(n) < 0.15, rng.choice([1, 2, 85, 6_000, 70_000, (1 << 22) - 1], n), 0)
    last = first + mlen - 1 + extra
    flag = np.where(rng.random(n) < 0.5, 16, 0)
    flag = np.where(rng.random(n) < 0.12, flag | rng.choice([4, 256, 512, 1024, 2048, 0x704], n), flag).astype(np.uint16)
    junk = (flag & 0x704) != 0
    first = np.where(junk & (rng.random(n) < 0.5), -1, first)  # unmapped mates and the like: any position at all
    nh = rng.choice([0, 1, 1, 1, 2, 255], n).astype(np.uint8)
    mapq = rng.choice([255, 255, 3, 0], n).astype(np.uint8)
    tail = slice(n - 700, n)
    ref[tail] = -1
    flag[tail] |= 4
    return dict(ref_id=ref, first=first.astype(np.int32), last=last.astype(np.int32), mlen=mlen.astype(np.uint16), flag=flag,
                mapq=mapq, nh=nh)


def _stream_pack(lib, cols, n_threads=3):
    import ctypes as C

    p = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    n = len(cols["ref_id"])
    args = [p(cols[k]) for k in ("ref_id", "first", "last", "mlen", "flag", "mapq", "nh")]
    nb = C.c_int64(0)
    rc = lib.rt_stream_pack(n, *args, n_threads, 0, None, None, C.byref(nb))
    if rc != 0:
        return rc, None, None, 0
    rec = np.zeros(max(1, nb.value) * _lib_block(), np.uint32)
    hdr = np.zeros(max(1, nb.value) * 4, np.int32)
    rc = lib.rt_stream_pack(n, *args, n_threads, nb.value, p(rec), p(hdr), C.byref(nb))
    return rc, rec, hdr, nb.value


def test_stream_pack_round_trip(built):
    """rt_stream_pack (4 B/read delta-coded records) decodes back to the columns it was given: every read the flags do
    not decide keeps ref_id / first / last / mlen, every read keeps the seven raw bits the cascade of bam.py:77-91 +
    common.py:33-69 looks at (checked against oracle_py), blocks are whole, extensions stay inside their block."""
    from helpers import decode_stream
    from oracle import oracle_py as O
    from ribotricer_b200 import _lib

    lib = _lib.load()
    cols = _stream_columns()
    n = len(cols["ref_id"])
    rc, rec, hdr, nb = _stream_pack(lib, cols)
    assert rc == 0 and nb >= (n + _lib_block() - 1) // _lib_block()
    got = decode_stream(rec, hdr, nb)
    assert len(got) == n
    n_checked = 0
    for i, (ref, first, last, mlen, meta) in enumerate(got):
        flag, mapq, nh = int(cols["flag"][i]), int(cols["mapq"][i]), int(cols["nh"][i])
        want_meta = (1 if flag & O.FLAG_UNMAPPED else 0) | (2 if flag & O.FLAG_SECONDARY else 0) | (4 if flag & O.FLAG_QCFAIL else 0) \
            | (8 if flag & O.FLAG_DUPLICATE else 0) | (16 if flag & O.FLAG_REVERSE else 0)
        state = (1 if mapq == 255 else 0) if nh == 0 else (2 if nh == 1 else 3)
        assert meta == want_meta | state << 5, i
        if flag & 0x704:
            continue
        # among the reads the flags let through, the two "unique" states are exactly what is_read_uniq_mapping accepts
        assert (state in (1, 2)) == bool(O.is_read_uniq_mapping(flag, mapq, nh)), i
        n_checked += 1
        assert (ref, first, last, mlen) == (int(cols["ref_id"][i]), int(cols["first"][i]), int(cols["last"][i]), int(cols["mlen"][i])), i
    assert n_checked > n // 2
    # one thread or many: the same stream
    rc1, rec1, hdr1, nb1 = _stream_pack(lib, cols, n_threads=1)
    assert rc1 == 0 and nb1 == nb and (rec1 == rec).all() and (hdr1 == hdr).all()
    # one read that starts before its predecessor (a CIGAR that opens with D or N) costs a block, not the stream ...
    bad = {k: v.copy() for k, v in cols.items()}
    clean = np.flatnonzero((bad["flag"] & 0x704) == 0)
    i, j = clean[100], clean[101]
    bad["first"][j] = bad["first"][i] - 1
    bad["last"][j] = bad["first"][j] + int(bad["mlen"][j]) - 1
    bad["ref_id"][j] = bad["ref_id"][i]
    rcb, recb, hdrb, nbb = _stream_pack(lib, bad)
    assert rcb == 0 and nb <= nbb <= nb + 2
    back = decode_stream(recb, hdrb, nbb)
    assert back[j][:4] == (int(bad["ref_id"][j]), int(bad["first"][j]), int(bad["last"][j]), int(bad["mlen"][j]))
    # ... a library that is not sorted at all is refused (the caller falls back to the columns), so is a span beyond 22 bits
    order = np.random.default_rng(1).permutation(n)
    assert _stream_pack(lib, {k: v[order] for k, v in cols.items()})[0] == _lib_estate()
    wide = {k: v.copy() for k, v in cols.items()}
    wide["last"][clean[7]] = wide["first"][clean[7]] + int(wide["mlen"][clean[7]]) - 1 + (1 << 22)
    assert _stream_pack(lib, wide)[0] == _lib_estate()
    # no reads: no blocks
    rc0, _, _, nb0 = _stream_pack(lib, {k: v[:0] for k, v in cols.items()})
    assert rc0 == 0 and nb0 == 0


def _lib_estate():
    return -4


def _lib_block():
    from ribotricer_b200 import _lib

    return _lib.RT_STREAM_BLOCK


def test_bam_stream_matches_the_decoder_columns(tmp_path, built):
    """rt_bam_stream (the decoder hands over the 4 B/read record stream) == rt_stream_pack on the decoder's columns, and
    the stream decodes back to those columns (a coordinate-sorted golden BAM with spliced reads, reads without CIGAR,
    unmapped reads that carry coordinates)."""
    import base64
    import ctypes as C

    from helpers import decode_stream, load_golden
    from ribotricer_b200 import _lib
    from ribotricer_b200.bam import read_bam_columns_native

    case = load_golden("split_bam_case.json.gz")["case"]
    path = tmp_path / "g.bam"
    path.write_bytes(base64.b64decode(case["bam_b64"]))
    rc = read_bam_columns_native(str(path), 2)
    lib = _lib.load()
    vp = C.c_void_p
    p = lambda a: a.ctypes.data_as(vp)      # noqa: E731
    code, rec, hdr, nb = _stream_pack(lib, rc.cols, n_threads=2)
    handle = vp()
    assert lib.rt_bam_load(str(path).encode(), 2, C.byref(handle)) == 0
    try:
        nb2 = C.c_int64(0)
        code2 = lib.rt_bam_stream(handle, 2, 0, None, None, C.byref(nb2))
        assert code2 == code
        if code != 0:
            assert not rc.sorted_by_coordinate or code == _lib_estate()
            return
        rec2 = np.zeros(max(1, nb2.value) * _lib_block(), np.uint32)
        hdr2 = np.zeros(max(1, nb2.value) * 4, np.int32)
        assert lib.rt_bam_stream(handle, 2, nb2.value, p(rec2), p(hdr2), C.byref(nb2)) == 0
    finally:
        lib.rt_bam_free(handle)
    assert nb2.value == nb and (rec2 == rec).all() and (hdr2 == hdr).all()
    got = decode_stream(rec, hdr, nb)
    assert len(got) == len(rc)
    for i, (ref, first, last, mlen, meta) in enumerate(got):
        if int(rc.cols["flag"][i]) & 0x704:
            continue
        assert (ref, first, last, mlen) == (int(rc.cols["ref_id"][i]), int(rc.cols["first"][i]), int(rc.cols["last"][i]),
                                            int(rc.cols["mlen"][i])), i


def test_stream_pack_ignores_positions_of_flag_decided_reads(built):
    """A read the flags decide (unmapped, secondary, qcfail, duplicate) may carry any position, also as the first read of
    a block or of the library: the library still codes, and the other reads keep their coordinates."""
    from helpers import decode_stream
    from ribotricer_b200 import _lib

    lib = _lib.load()
    n = 4 * _lib_block() + 17
    cols = dict(ref_id=np.zeros(n, np.int32), first=(np.arange(n) * 3).astype(np.int32), last=None,
                mlen=np.full(n, 28, np.uint16), flag=np.zeros(n, np.uint16), mapq=np.full(n, 255, np.uint8),
                nh=np.ones(n, np.uint8))
    for k, i in enumerate((0, _lib_block(), 2 * _lib_block() - 1, 3 * _lib_block(), n - 1)):      # block starts and ends among them
        cols["flag"][i] = 4                                     # e.g. an unmapped mate: same reference, any position
        cols["first"][i] = 2 ** 31 - 1 if k % 2 else -1
    cols["last"] = (cols["first"].astype(np.int64) + 27).clip(-2 ** 31, 2 ** 31 - 1).astype(np.int32)
    rc, rec, hdr, nb = _stream_pack(lib, cols, n_threads=2)
    assert rc == 0
    got = decode_stream(rec, hdr, nb)
    assert len(got) == n
    for i, (ref, first, last, mlen, meta) in enumerate(got):
        if cols["flag"][i] & 4:
            assert meta & 1
        else:
            assert (ref, first, last, mlen) == (0, int(cols["first"][i]), int(cols["last"][i]), 28), i


def test_stream_pack_random_small_libraries(built):
    """Many small random libraries (fixed seed) through rt_stream_pack and back: whatever the mix of references, gaps,
    descents, spliced / long / empty reads and flag-decided reads with junk positions, a stream that is produced decodes
    to the columns, and a refusal is the documented one (a span the extension record cannot hold)."""
    from helpers import decode_stream
    from ribotricer_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(2024)
    coded = refused = 0
    for case in range(300):
        n = int(rng.integers(1, 1200))
        n_ref = int(rng.integers(1, 6))
        ref = np.sort(rng.integers(0, n_ref, n)).astype(np.int32)
        step = rng.choice([0, 1, 5, 300, 33_000, 70_000, 1 << 30], n, p=[0.3, 0.3, 0.2, 0.1, 0.05, 0.04, 0.01]).astype(np.int64)
        first = np.zeros(n, np.int64)
        for r in np.unique(ref):
            m = ref == r
            first[m] = np.minimum(np.cumsum(step[m]), 2 ** 31 - 70_000)
        descents = rng.random(n) < rng.choice([0.0, 0.01, 0.6])          # none, a few, or an unsorted library
        first = np.where(descents, np.maximum(first - rng.integers(1, 50, n), 0), first)
        mlen = rng.choice([0, 1, 28, 30, 255, 256, 4000], n, p=[0.02, 0.03, 0.5, 0.3, 0.05, 0.05, 0.05]).astype(np.int64)
        big = rng.random() < 0.05
        extra = np.where(rng.random(n) < 0.2, rng.choice([1, 900, 60_000, (1 << 22) - 1, (1 << 22) if big else 7], n), 0)
        last = first + mlen - 1 + extra
        flag = np.where(rng.random(n) < 0.5, 16, 0) | np.where(rng.random(n) < 0.15, rng.choice([4, 256, 512, 1024], n), 0)
        junk = (flag & 0x704) != 0
        first = np.where(junk & (rng.random(n) < 0.5), rng.choice([-1, 0, 2 ** 31 - 1], n), first)
        cols = dict(ref_id=ref, first=first.astype(np.int32), last=np.clip(last, -2 ** 31, 2 ** 31 - 1).astype(np.int32),
                    mlen=mlen.astype(np.uint16), flag=flag.astype(np.uint16), mapq=rng.choice([255, 3, 0], n).astype(np.uint8),
                    nh=rng.choice([0, 1, 2], n).astype(np.uint8))
        rc, rec, hdr, nb = _stream_pack(lib, cols, n_threads=int(rng.integers(1, 4)))
        clean = ~junk
        if rc != 0:
            refused += 1
            assert rc == _lib_estate()
            spans = (cols["last"].astype(np.int64) - cols["first"] + 1 - cols["mlen"])[clean]
            assert (spans >= 1 << 22).any() or (spans < 0).any(), case     # (too small for the padding rule)
            continue
        coded += 1
        got = decode_stream(rec, hdr, nb)
        assert len(got) == n, case
        for i in np.flatnonzero(clean):
            assert got[i][:4] == (int(cols["ref_id"][i]), int(cols["first"][i]), int(cols["last"][i]), int(cols["mlen"][i])), (case, i)
    assert coded > 150 and refused > 10


def test_wig_long_block_is_formatted_in_order(tmp_path, built):
    """rt_wig_block formats a long block (a chromosome with hundreds of thousands of covered positions) with several
    threads; the text is the reference's, line for line (detect_orfs.py:338-345)."""
    import ctypes as C

    from ribotricer_b200 import _lib

    lib = _lib.load()
    n = 400_000
    rng = np.random.default_rng(3)
    pos = np.cumsum(rng.integers(1, 50, n)).astype(np.int64)
    cnt = rng.integers(1, 100_000, n).astype(np.int32)
    path = tmp_path / "x_pos.wig"
    h = C.c_void_p()
    assert lib.rt_wig_open(str(path).encode(), C.byref(h)) == 0
    p = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    assert lib.rt_wig_block(h, b"chr1", n, p(pos), p(cnt)) == 0
    assert lib.rt_wig_block(h, b"chr2", 1000, p(pos), p(cnt)) == 0
    lib.rt_wig_close(h)
    want = "variableStep chrom=chr1\n" + "".join(f"{a}\t{b}\n" for a, b in zip(pos.tolist(), cnt.tolist())) + \
        "variableStep chrom=chr2\n" + "".join(f"{a}\t{b}\n" for a, b in zip(pos[:1000].tolist(), cnt[:1000].tolist()))
    assert path.read_text() == want
    # the writers hand their text to a write-behind thread: a disk that refuses it must surface at the latest on close
    if os.path.exists("/dev/full"):
        h = C.c_void_p()
        assert lib.rt_wig_open(b"/dev/full", C.byref(h)) == 0
        rcs = [lib.rt_wig_block(h, b"chr1", n, p(pos), p(cnt)) for _ in range(3)]
        assert lib.rt_wig_close(h) != 0 or any(rcs), "a failed write went unnoticed"


def _deflate_payload(rng, kind, n):
    if kind == 0:
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()                      # incompressible: stored blocks
    if kind == 1:
        return bytes(n)                                                                 # one long run (distance 1)
    if kind == 2:
        return rng.integers(0, 4, n, dtype=np.uint8).tobytes()                          # short codes: literal pairs
    if kind == 3:
        per = int(rng.integers(2, 12))
        return (rng.integers(0, 256, per, dtype=np.uint8).tobytes() * (n // per + 1))[:n]   # overlapping copies
    if kind == 4:
        p = 0.5 ** np.arange(1, 257)
        return bytes(rng.choice(256, n, p=p / p.sum()).astype(np.uint8))              # codes longer than 11 bits
    words = [bytes(rng.integers(97, 123, int(rng.integers(2, 12)), dtype=np.uint8)) for _ in range(200)]
    return b" ".join(words[int(i)] for i in rng.integers(0, 200, n // 5 + 1))[:n]      # text-like: long matches


def test_inflate_and_crc32_match_zlib(built):
    """csrc/rt_inflate.cpp against zlib: every compression level and strategy (stored, fixed and dynamic blocks, sync
    flushes in the middle), sizes around the margins of the fast loop; a wrong announced size, a truncated stream and a
    flipped bit are refused or decoded, never written past the output; rt_crc32 == zlib.crc32 at every length mod 16."""
    import ctypes as C
    import zlib

    from ribotricer_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(11)
    for n in list(range(0, 150)) + [1000, 4096, 65280, 65536, (1 << 20) + 13]:
        d = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert lib.rt_crc32(d, n) == zlib.crc32(d), n
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
    sizes = [0, 1, 2, 5, 100, 287, 288, 289, 320, 1000, 4099, 65280, 65536, 150000]
    n_ok = 0
    for trial in range(600):
        kind, n = int(rng.integers(0, 6)), int(rng.choice(sizes))
        data = _deflate_payload(rng, kind, n)
        co = zlib.compressobj(int(rng.integers(0, 10)), zlib.DEFLATED, -15, int(rng.integers(1, 10)), int(rng.choice(strategies)))
        if n > 1000 and trial % 3 == 0:
            k = n // 3
            comp = (co.compress(data[:k]) + co.flush(zlib.Z_SYNC_FLUSH) + co.compress(data[k:2 * k]) + co.flush(zlib.Z_FULL_FLUSH)
                    + co.compress(data[2 * k:]) + co.flush())
        else:
            comp = co.compress(data) + co.flush()
        out = C.create_string_buffer(n + 64)
        C.memset(out, 0xAB, n + 64)
        assert lib.rt_inflate_raw(comp, len(comp), out, n) == 0, (kind, n)
        assert out.raw[:n] == data and out.raw[n:] == b"\xab" * 64, (kind, n)
        n_ok += 1
        if n:
            assert lib.rt_inflate_raw(comp, len(comp), out, n - 1) != 0            # announced size too small
            assert lib.rt_inflate_raw(comp, len(comp), out, n + 1) != 0            # ... too large
            cut = int(rng.integers(0, len(comp)))
            assert lib.rt_inflate_raw(comp[:cut], cut, out, n) != 0                 # truncated stream
        if len(comp) > 4:
            bad = bytearray(comp)
            bad[int(rng.integers(0, len(bad)))] ^= 1 << int(rng.integers(0, 8))
            C.memset(out, 0xAB, n + 64)
            lib.rt_inflate_raw(bytes(bad), len(bad), out, n)                        # any verdict, but inside the buffer
            assert out.raw[n:] == b"\xab" * 64
    assert n_ok == 600


def test_bam_batches_carry_records_and_header_across_boundaries(tmp_path, built, monkeypatch):
    """rt_bam_load cuts the file into batches that are inflated and decoded by different threads; the walk hands the
    unfinished record (or header) from one batch to the next.  With batches of a few hundred bytes every record and the
    header (300 references) span several batches, a 70 kB record spans hundreds; the columns must not depend on the
    batch size, the thread count or the inflater.  Damaged files are refused with a message."""
    import bam_writer as W
    import pytest
    from ribotricer_b200.bam import read_bam_columns_native

    rng = np.random.default_rng(5)
    refs = [("contig_%04d" % i, 100000 + i) for i in range(300)]
    recs = []
    for i in range(4000):
        ref = int(rng.integers(0, len(refs)))
        cigar = [("M", int(rng.integers(20, 40)))]
        if rng.random() < 0.2:
            cigar += [("N", int(rng.integers(50, 500))), ("M", int(rng.integers(5, 30)))]
        aux = W.aux_field("NH", "C", int(rng.choice([1, 1, 1, 2, 5])))
        if i == 1234:                                                   # one huge record (a long Z tag)
            aux = W.aux_field("XL", "Z", "x" * 70000) + aux
        recs.append(W.record(ref, int(rng.integers(0, 90000)), int(rng.choice([255, 3, 0])), int(rng.choice([0, 16, 256, 4])), cigar,
                             name=b"q%d" % i, aux=aux))
    path = tmp_path / "b.bam"
    W.write_bam(str(path), refs, recs, block_payload=3001)
    monkeypatch.delenv("RT_BAM_BATCH_BYTES", raising=False)
    monkeypatch.delenv("RT_BAM_ZLIB", raising=False)
    want = read_bam_columns_native(str(path), 1)
    assert len(want) == len(recs) and want.contig_names == [r[0] for r in refs]
    for batch, threads, zl in ((1, 3, False), (300, 4, False), (7000, 2, True), (1 << 16, 8, False), (1 << 26, 2, True)):
        monkeypatch.setenv("RT_BAM_BATCH_BYTES", str(batch))
        if zl:
            monkeypatch.setenv("RT_BAM_ZLIB", "1")
        else:
            monkeypatch.delenv("RT_BAM_ZLIB", raising=False)
        got = read_bam_columns_native(str(path), threads)
        assert got.contig_names == want.contig_names and got.contig_len.tolist() == want.contig_len.tolist()
        for name in want.cols:
            assert np.array_equal(got.cols[name], want.cols[name]), (batch, threads, name)
    # the same records from other compressors: stored blocks (samtools -u), level 1 and 9, fixed-Huffman and
    # Huffman-only streams, full-size blocks, a file without the EOF marker
    import zlib
    monkeypatch.delenv("RT_BAM_ZLIB", raising=False)
    other = tmp_path / "o.bam"
    for level, strategy, payload, eof in ((0, zlib.Z_DEFAULT_STRATEGY, 0xFF00, True), (1, zlib.Z_DEFAULT_STRATEGY, 0xFF00, True),
                                          (9, zlib.Z_DEFAULT_STRATEGY, 777, False), (6, zlib.Z_FIXED, 0xFF00, True),
                                          (6, zlib.Z_HUFFMAN_ONLY, 5000, True), (4, zlib.Z_RLE, 0xFF00, False)):
        W.write_bam(str(other), refs, recs, block_payload=payload, level=level, strategy=strategy, eof=eof)
        for batch in (4000, 1 << 20):
            monkeypatch.setenv("RT_BAM_BATCH_BYTES", str(batch))
            got = read_bam_columns_native(str(other), 3)
            for name in want.cols:
                assert np.array_equal(got.cols[name], want.cols[name]), (level, strategy, batch, name)
    monkeypatch.setenv("RT_BAM_BATCH_BYTES", "5000")
    raw = path.read_bytes()
    bad = tmp_path / "bad.bam"
    for what, data in (("block cut short", raw[:len(raw) // 2]),
                       ("record cut short", b"".join(W.bgzf_block(x) for x in [_bam_stream_bytes(W, refs, recs)[:50000]]) + W.BGZF_EOF),
                       ("header cut short", W.bgzf_block(_bam_stream_bytes(W, refs, recs)[:100]) + W.BGZF_EOF),
                       ("flipped payload bit", raw[:40] + bytes([raw[40] ^ 4]) + raw[41:]),
                       ("record size below the fixed fields", W.bgzf_block(_bam_stream_bytes(W, refs[:1], [b"\x08\0\0\0" + bytes(8)])) + W.BGZF_EOF)):
        bad.write_bytes(data)
        for threads in (1, 4):
            with pytest.raises(OSError):
                read_bam_columns_native(str(bad), threads)


def _bam_stream_bytes(W, refs, recs):
    """The uncompressed byte stream bam_writer.write_bam would compress."""
    import struct

    text = b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(("@SQ\tSN:%s\tLN:%d\n" % (n, ln)).encode() for n, ln in refs)
    head = b"BAM\1" + struct.pack("<I", len(text)) + text + struct.pack("<I", len(refs))
    for n, ln in refs:
        nb = n.encode() + b"\0"
        head += struct.pack("<I", len(nb)) + nb + struct.pack("<I", ln)
    return head + b"".join(recs)


def _metagene_sums_numpy(flat, lens, width):
    """The matrix statement of metagene.py:204-252 the native routine replaced (rows padded to `width`)."""
    n = len(lens)
    mat = np.zeros((n, width), np.float64)
    have = np.arange(width)[None, :] < lens[:, None]
    mat[have] = flat
    mean = mat.sum(1) / np.maximum(lens, 1)                      # metagene.py:214
    use = mean > 0
    norm = np.where(have[use], mat[use] / mean[use, None], 0.0)
    stop = np.zeros_like(norm)
    hs = np.zeros_like(have[use])
    l_use = lens[use]
    for k in np.unique(l_use):
        rows = l_use == k
        stop[rows, width - k:] = norm[rows, :k]
        hs[rows, width - k:] = True
    return norm.sum(0), have[use].sum(0), stop.sum(0), hs.sum(0)


def test_metagene_sums_match_the_matrix_statement(built):
    """rt_metagene_sums (rows normalised by their mean, summed start-aligned and stop-aligned by all cores) against the
    numpy matrix form: counts exact, sums to 1e-12 relative (the order of the additions differs); rows without reads,
    empty rows and rows shorter than the matrix; the result must not depend on the number of rows per block."""
    from ribotricer_b200 import _lib
    from ribotricer_b200.metagene import metagene_sums

    lib = _lib.load()
    rng = np.random.default_rng(21)
    for n, width in ((0, 0), (1, 1), (5, 7), (300, 620), (7000, 620), (5000, 33)):
        lens = rng.integers(0, width + 1, n).astype(np.int64) if width else np.zeros(n, np.int64)
        if n:
            lens[rng.random(n) < 0.5] = width                    # most CDS reach the full width
            width = int(lens.max())
        ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        flat = (rng.random(int(ptr[-1])) < 0.2) * rng.integers(1, 50, int(ptr[-1]))
        for i in np.flatnonzero(rng.random(n) < 0.2):            # ORFs without a single read
            flat[ptr[i]:ptr[i + 1]] = 0
        flat = flat.astype(np.int32)
        got = metagene_sums(lib, flat, ptr, width)
        want = _metagene_sums_numpy(flat, lens, width) if n else (np.zeros(0),) * 4
        assert np.array_equal(got[1], want[1]) and np.array_equal(got[3], want[3]), (n, width)
        assert np.allclose(got[0], want[0], rtol=1e-12, atol=0) and np.allclose(got[2], want[2], rtol=1e-12, atol=0), (n, width)
    import pytest
    with pytest.raises(ValueError):
        metagene_sums(lib, np.zeros(10, np.int32), np.array([0, 10], np.int64), 5)      # a row wider than the matrix


def test_metagene_host_logic_against_reference_golden(built, tmp_path, monkeypatch):
    """The host side of the P-site offset inference on the CPU: metagene_coverage (windows of the annotated ORFs, rows
    normalised and summed by rt_metagene_sums, profile assembly, the two profile files) and align_metagenes, against
    what the UNMODIFIED reference returned for the same library (tests/golden/metagene_case).  The device calls of the
    step -- K1 per read length, K4 over the windows, phasescore of a float profile -- are stood in for by the oracle
    (tests/oracle_engine.py; the GPU twin of this test is test_gpu_api.py::test_metagene_and_offset_inference)."""
    from helpers import SCORE_TOL, alignments_to_reads, load_golden
    from oracle_engine import install
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200 import metagene as mg
    from ribotricer_b200.bam import ReadColumns, split_bam

    case = load_golden("metagene_case.json.gz")["case"]
    names = [c[0] for c in case["contigs"]]
    case = dict(case, alignments=sorted(case["alignments"], key=lambda a: a[0]))     # read_length_counts insertion order
    reads = ReadColumns(names, np.array([c[1] for c in case["contigs"]], np.int64), alignments_to_reads(case, names))
    eng = install(monkeypatch)
    idx_path = tmp_path / "mg_index.tsv"
    idx_path.write_text("\n".join(case["index"]) + "\n")
    prefix = str(tmp_path / "mg")
    annotated, _ = D.parse_ribotricer_index(str(idx_path))
    assert len(annotated) == len(case["index"]) - 1
    alignments, rlc = split_bam(reads, "forward", prefix, None, engine=eng)
    assert {str(k): v for k, v in rlc.items()} == case["read_length_counts_in"]
    rlc = dict(sorted(rlc.items()))
    metagenes = mg.metagene_coverage(annotated, alignments, rlc, prefix, meta_min_reads=case["meta_min_reads"])
    assert list(rlc) == case["kept_lengths"]
    for length, ref in case["metagenes"].items():
        m = metagenes[int(length)]
        assert m[0][0] == ref["idx5"] and m[1][0] == ref["idx3"]
        assert np.allclose(m[0][1], ref["prof5"], rtol=0, atol=1e-9) and np.allclose(m[1][1], ref["prof3"], rtol=0, atol=1e-9)
        assert abs(m[2] - ref["ps5"]) <= SCORE_TOL and m[3] == ref["v5"]
        assert abs(m[4] - ref["ps3"]) <= SCORE_TOL and m[5] == ref["v3"]
    got_rows = open(f"{prefix}_metagene_profiles_5p.tsv").read().split("\n")
    want_rows = case["profiles_5p_tsv"].split("\n")
    assert len(got_rows) == len(want_rows) and got_rows[0] == want_rows[0]
    for g, w in zip(got_rows[1:], want_rows[1:]):
        assert g.split("\t")[:2] == w.split("\t")[:2]
    offsets = mg.align_metagenes(metagenes, rlc, prefix, 0.428571428571, True)
    assert {str(k): v for k, v in offsets.items()} == case["psite_offsets"]
    assert open(f"{prefix}_psite_offsets.txt").read() == case["psite_offsets_txt"]
    # the whole default-flag call: protocol, read lengths and offsets inferred on the way
    D.detect_orfs(reads, str(idx_path), prefix, None, None, None, 0.428571428571, 5, 0, 0, 0.0, True,
                  meta_min_reads=case["meta_min_reads"])
    assert open(f"{prefix}_protocol.txt").read().startswith("In total")
    assert open(f"{prefix}_psite_offsets.txt").read() == case["psite_offsets_txt"]
    rows = open(f"{prefix}_translating_ORFs.tsv").read().split("\n")
    assert len(rows) == len(case["index"]) + 1
    assert sum(1 for r in rows[1:] if r.split("\t")[2:3] == ["translating"]) > 0.5 * (len(case["index"]) - 1)


def test_detect_orfs_host_flow_against_reference_golden(built, tmp_path, monkeypatch):
    """detect_orfs() from end to end on the CPU with the device calls stood in for by the oracle (tests/oracle_engine.py):
    what is under test is the HOST flow of the product -- index loader, split_bam bookkeeping and summary file, the metagene
    step, the dense -> compact hand-over, row selection and chunking of write_tsv, the native TSV / WIG writers -- against
    the files the unmodified reference wrote for the same inputs (four parameter sets per case).  GPU twin:
    test_gpu_api.py::test_detect_orfs_end_to_end."""
    from helpers import alignments_to_reads, compare_tsv, load_golden
    from oracle_engine import install
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200.bam import ReadColumns

    eng = install(monkeypatch)
    for case in load_golden("pipeline_cases.json.gz")["cases"]:
        names = [c[0] for c in case["contigs"]]
        reads = ReadColumns(names, np.array([c[1] for c in case["contigs"]], np.int64), alignments_to_reads(case, names))
        idx_path = tmp_path / f"{case['name']}_index.tsv"
        idx_path.write_text("\n".join(case["index"]) + "\n")
        offsets = {int(k): v for k, v in case["psite_offsets"].items()}
        for run in case["tsv"]:
            prm = run["params"]
            prefix = str(tmp_path / "out" / case["name"])
            eng.calls.clear()
            D.detect_orfs(reads, str(idx_path), prefix, "forward", None, dict(offsets), prm["phase_score_cutoff"],
                          prm["min_valid_codons"], prm["min_reads_per_codon"], prm["min_valid_codons_ratio"],
                          prm["min_density_over_orf"], prm["report_all"], meta_min_reads=10 ** 9)
            assert "compact_from_dense" in eng.calls and "score_host" in eng.calls      # scored in the compact layout
            got_text = open(f"{prefix}_translating_ORFs.tsv").read()
            compare_tsv(got_text, run["text"], prm["phase_score_cutoff"], what=case["name"] + ": ")
        for tag, text in case["wig"].items():
            assert open(f"{prefix}_{tag}.wig").read() == text
        summary = open(f"{prefix}_bam_summary.txt").read()
        assert summary.startswith(f"summary:\n\ttotal_reads: {len(reads)}\n\tunique_mapped: {len(reads)}\n")
        # the same call with the rows cut into many small chunks (one being formatted on the helper thread while the next
        # is gathered): the file must not change
        one_chunk = open(f"{prefix}_translating_ORFs.tsv", "rb").read()
        whole = D.write_tsv
        eng.calls.clear()
        with monkeypatch.context() as m:
            m.setattr(D, "write_tsv", lambda *a, **k: whole(*a, **dict(k, chunk_nt=1)))         # one row per chunk
            D.detect_orfs(reads, str(idx_path), prefix + "_chunks", "forward", None, dict(offsets), prm["phase_score_cutoff"],
                          prm["min_valid_codons"], prm["min_reads_per_codon"], prm["min_valid_codons_ratio"],
                          prm["min_density_over_orf"], prm["report_all"], meta_min_reads=10 ** 9)
        assert eng.calls.count("gather_profiles") == max(1, one_chunk.count(b"\n") - 1)
        assert open(f"{prefix}_chunks_translating_ORFs.tsv", "rb").read() == one_chunk
        # and from a BAM file of the same reads (native decoder -> columns -> the same flow)
        import bam_writer as W
        c = reads.cols
        recs = [W.record(int(c["ref_id"][i]), int(c["first"][i]), 255, int(c["flag"][i]), [("M", int(c["mlen"][i]))],
                         name=b"r%d" % i, aux=W.aux_field("NH", "C", 1)) for i in range(len(reads))]
        bam_path = tmp_path / f"{case['name']}.bam"
        W.write_bam(str(bam_path), [(n, int(ln)) for n, ln in zip(names, reads.contig_len)], recs, sorted_header=False)
        D.detect_orfs(str(bam_path), str(idx_path), prefix + "_bam", "forward", None, dict(offsets), prm["phase_score_cutoff"],
                      prm["min_valid_codons"], prm["min_reads_per_codon"], prm["min_valid_codons_ratio"],
                      prm["min_density_over_orf"], prm["report_all"], meta_min_reads=10 ** 9)
        assert open(f"{prefix}_bam_translating_ORFs.tsv", "rb").read() == one_chunk
        assert open(f"{prefix}_bam_bam_summary.txt").read() == summary


def test_cli_detect_orfs_end_to_end_on_the_cpu_twin(built, tmp_path, monkeypatch):
    """`ribotricer detect-orfs` flags -> detect_orfs() arguments -> files (cli.py:132-289), driven through click on a BAM
    file: --stranded yes, --read_lengths / --psite_offsets, the five thresholds and --report_all must give the TSV that the
    Python call with the same values gives (itself held to the reference's golden files above); --stranded reverse must
    change the result."""
    from click.testing import CliRunner

    import bam_writer as W
    from helpers import alignments_to_reads, load_golden
    from oracle_engine import install
    from ribotricer_b200 import detect_orfs as D
    from ribotricer_b200.bam import ReadColumns
    from ribotricer_b200.cli import cli

    install(monkeypatch)
    case = load_golden("pipeline_cases.json.gz")["cases"][0]
    names = [c[0] for c in case["contigs"]]
    cols = alignments_to_reads(case, names)
    reads = ReadColumns(names, np.array([c[1] for c in case["contigs"]], np.int64), cols)
    recs = [W.record(int(cols["ref_id"][i]), int(cols["first"][i]), 255, int(cols["flag"][i]), [("M", int(cols["mlen"][i]))],
                     name=b"r%d" % i, aux=W.aux_field("NH", "C", 1)) for i in range(len(reads))]
    bam = tmp_path / "lib.bam"
    W.write_bam(str(bam), [(n, int(ln)) for n, ln in zip(names, reads.contig_len)], recs, sorted_header=False)
    idx_path = tmp_path / "index.tsv"
    idx_path.write_text("\n".join(case["index"]) + "\n")
    offsets = {int(k): v for k, v in case["psite_offsets"].items()}
    lengths = sorted(offsets)
    base = ["detect-orfs", "--bam", str(bam), "--ribotricer_index", str(idx_path), "--read_lengths", ",".join(map(str, lengths)),
            "--psite_offsets", ",".join(str(offsets[k]) for k in lengths), "--meta-min-reads", str(10 ** 9)]
    for run in case["tsv"]:
        prm = run["params"]
        flags = ["--phase_score_cutoff", repr(prm["phase_score_cutoff"]), "--min_valid_codons", str(prm["min_valid_codons"]),
                 "--min_reads_per_codon", str(int(prm["min_reads_per_codon"])), "--min_valid_codons_ratio",
                 repr(prm["min_valid_codons_ratio"]), "--min_read_density", repr(prm["min_density_over_orf"])]
        if prm["report_all"]:
            flags.append("--report_all")
        r = CliRunner().invoke(cli, base + ["--prefix", str(tmp_path / "cli"), "--stranded", "yes"] + flags)
        assert r.exit_code == 0, (r.output, r.exception)
        D.detect_orfs(reads, str(idx_path), str(tmp_path / "api"), "forward", lengths, dict(offsets), prm["phase_score_cutoff"],
                      prm["min_valid_codons"], int(prm["min_reads_per_codon"]), prm["min_valid_codons_ratio"],
                      prm["min_density_over_orf"], prm["report_all"], meta_min_reads=10 ** 9)
        for suffix in ("_translating_ORFs.tsv", "_bam_summary.txt", "_pos.wig"):
            assert open(str(tmp_path / "cli") + suffix, "rb").read() == open(str(tmp_path / "api") + suffix, "rb").read(), suffix
    r = CliRunner().invoke(cli, base + ["--prefix", str(tmp_path / "rev"), "--stranded", "reverse", "--report_all"])
    assert r.exit_code == 0, (r.output, r.exception)
    assert open(str(tmp_path / "rev") + "_translating_ORFs.tsv", "rb").read() != open(str(tmp_path / "cli") + "_translating_ORFs.tsv", "rb").read()
