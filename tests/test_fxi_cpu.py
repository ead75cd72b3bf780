"""Host logic of the .fxi writer / loader (pyfastx_b200/fxi.py) without a GPU: rows produced by the CPU
oracle are written with the reference's schema; the compiled reference opened such files as its own index and
served the right sequences (tests/golden/make_golden_interop.py recorded those files' digests and its answers),
and an index written by the reference must load back into the same rows."""
import gzip
import os
import sqlite3

import numpy as np

import gen
import goldenlib as G
from oracle import fxo
from pyfastx_b200 import fxi
from pyfastx_b200._cabi import FASTA_ROW, FASTQ_ROW


def as_rows(exp, dtype):
    rows = np.zeros(len(exp), dtype=dtype)
    for f in exp.dtype.names:
        if f in rows.dtype.names:
            rows[f] = exp[f]
    return rows


def test_fasta_fxi_roundtrip_and_reference_reads_it(tmp_path):
    data = gzip.open(os.path.join(G.GOLD, "data", "test.fa.gz")).read()
    path = tmp_path / "t.fa"
    path.write_bytes(data)
    exp, total, _ = fxo.fasta_scan(data)
    rows = as_rows(exp, FASTA_ROW)
    names = fxo.fasta_names(data, exp)
    con = fxi.write_fasta_index(str(path) + ".fxi", rows, names, total)
    con.close()
    # schema: the reference's tables and index names (src/index.c:178-207,366)
    db = sqlite3.connect(str(path) + ".fxi")
    tabs = {r[0] for r in db.execute("SELECT name FROM sqlite_master")}
    assert {"seq", "stat", "comp", "gzindex", "chromidx"} <= tabs
    assert db.execute("SELECT seqnum, seqlen FROM stat").fetchone() == (len(rows), total)
    db.close()
    con, back, back_names, stat = fxi.load_fasta_index(str(path) + ".fxi")
    con.close()
    for f in ("boff", "blen", "slen", "llen", "elen", "norm", "dlen"):
        assert np.array_equal(back[f], rows[f]), f
    assert back_names.tolist() == [n.decode() for n in names] and tuple(stat[:2]) == (len(rows), total)
    # the reference loaded this very file as its index (it did not rebuild it) and served these records
    gold = G.interop("fxi_test_fa")
    assert G.fxi_digest(str(path) + ".fxi") == gold["digest"]
    assert gold["len"] == len(rows) == 211 and gold["size"] == total
    for i, name, n, seq, anti in gold["records"]:
        assert name == names[i].decode() and n == int(rows["slen"][i])
        assert G.digest(fxo.subseq(data, exp[i], 0, int(rows["slen"][i]))) == seq
        assert G.digest(fxo.subseq(data, exp[i], 5, 50, fxo.REVERSE | fxo.COMPLEMENT)) == anti


def test_fastq_fxi_roundtrip_and_reference_reads_it(tmp_path):
    data = gen.random_fastq(5, n_reads=700)
    path = tmp_path / "t.fq"
    path.write_bytes(data)
    exp, size, nlines = fxo.fastq_scan(data)
    rows = as_rows(exp, FASTQ_ROW)
    names = fxo.fastq_names(data, exp)
    con = fxi.write_fastq_index(str(path) + ".fxi", rows, names, nlines, size)
    con.close()
    con, back, back_names, stat = fxi.load_fastq_index(str(path) + ".fxi")
    con.close()
    for f in ("dlen", "rlen", "soff", "qoff"):
        assert np.array_equal(back[f], rows[f]), f
    assert back_names.tolist() == [n.decode("latin-1") for n in names]
    gold = G.interop("fxi_random5_fq")                 # the reference loaded this very file and served these reads
    assert G.fxi_digest(str(path) + ".fxi") == gold["digest"] and gold["len"] == len(rows)
    for i, name, seq, qual in gold["reads"]:
        es, eq = fxo.read_fetch(data, exp[i])
        assert G.digest(es) == seq and G.digest(eq) == qual and name == names[i].decode("latin-1")


def test_reference_written_index_loads_here(tmp_path):
    data = gen.random_fasta(9, n_records=80)
    path = tmp_path / "r.fa"
    path.write_bytes(data)
    G.reference_index("random9.fa", str(path) + ".fxi")    # the index the reference built for r.fa
    con, back, back_names, stat = fxi.load_fasta_index(str(path) + ".fxi")
    con.close()
    exp, total, _ = fxo.fasta_scan(data)
    for f in ("boff", "blen", "slen", "llen", "elen", "norm", "dlen"):
        assert np.array_equal(back[f], exp[f]), f
    assert back_names.tolist() == [n.decode("latin-1") for n in fxo.fasta_names(data, exp)]


def _dump(path, tables):
    """digest of every table's rows, integrity check, index names"""
    out = {t: G.digest(rows) for t, rows in G.fxi_rows(path, tables).items()}
    db = sqlite3.connect(path)
    ok = db.execute("PRAGMA integrity_check").fetchall()
    idx = sorted(r[0] for r in db.execute("SELECT name FROM sqlite_master WHERE type='index'"))
    db.close()
    return out, ok, idx


def test_native_writer_is_select_equal_with_the_reference(tmp_path):
    """the file libfxg writes page by page and the file the reference fills with INSERTs answer every SELECT
    the same (rows of seq / stat / read compared column by column, through digests of the reference's rows),
    and sqlite's integrity_check accepts ours"""
    data = gen.random_fasta(31, n_records=3000, crlf_prob=0.2)
    b = tmp_path / "b.fa"
    b.write_bytes(data)
    exp, total, _ = fxo.fasta_scan(data)
    fxi.write_fasta_index(str(b) + ".fxi", as_rows(exp, FASTA_ROW), fxo.fasta_names(data, exp), total).close()
    gold = G.interop("ref_random31_fa")
    rb, ok, ib = _dump(str(b) + ".fxi", ("seq", "stat", "comp", "gzindex"))
    assert ok == [("ok",)] and rb == gold["tables"] and ib == gold["indexes"] == ["chromidx"]
    fq = gen.random_fastq(32, n_reads=5000)
    b = tmp_path / "b.fq"
    b.write_bytes(fq)
    qexp, size, nlines = fxo.fastq_scan(fq)
    fxi.write_fastq_index(str(b) + ".fxi", as_rows(qexp, FASTQ_ROW), fxo.fastq_names(fq, qexp), nlines, size).close()
    gold = G.interop("ref_random32_fq")
    rb, ok, ib = _dump(str(b) + ".fxi", ("read", "stat", "base", "meta", "gzindex"))
    assert ok == [("ok",)] and rb == gold["tables"] and ib == gold["indexes"] == ["readidx"]


def test_native_writer_edge_cases(tmp_path):
    """0 / 1 / many rows, multi-level b-trees, names long enough to need overflow pages, duplicate names
    (no UNIQUE index, as in the reference), and lookups THROUGH the name index"""
    rng = np.random.default_rng(4)
    for n, kind in ((0, ""), (1, ""), (3, "long"), (2500, "dup"), (200000, "")):
        rows = np.zeros(n, dtype=FASTA_ROW)
        rows["boff"] = np.cumsum(rng.integers(1, 1 << 33, size=n)) if n else 0
        rows["blen"] = rng.integers(0, 1 << 45, size=n)
        rows["slen"] = rng.integers(-5, 300, size=n)
        rows["llen"], rows["elen"], rows["norm"], rows["dlen"] = 61, 1, rng.integers(0, 2, size=n), rng.integers(0, 70000, size=n)
        names = [b"chr%d_%d" % (i * 7919 % max(n, 1), i) for i in range(n)]
        if kind == "long":
            names = [b"A" * 5000, b"B" * 70000, b"C" * 1001]
        if kind == "dup":
            names = [b"n%d" % (i // 2) for i in range(n)]
        p = str(tmp_path / ("e%d%s.fxi" % (n, kind)))
        fxi.write_fasta_index(p, rows, names, 12345).close()
        db = sqlite3.connect(p)
        db.text_factory = bytes
        assert db.execute("PRAGMA integrity_check").fetchall() == [(b"ok",)]
        got = db.execute("SELECT ID,chrom,boff,blen,slen,llen,elen,norm,dlen FROM seq ORDER BY ID").fetchall()
        assert len(got) == n
        for i in (list(range(min(n, 50))) + [n // 2, n - 1] if n else []):
            r = rows[i]
            assert got[i] == (i + 1, names[i], int(r["boff"]), int(r["blen"]), int(r["slen"]), 61, 1, int(r["norm"]), int(r["dlen"]))
        has_idx = db.execute("SELECT count(*) FROM sqlite_master WHERE name='chromidx'").fetchone()[0]
        assert has_idx == (0 if kind == "dup" else 1)
        if has_idx and n:
            for i in (0, n // 3, n - 1):
                assert db.execute("SELECT ID FROM seq INDEXED BY chromidx WHERE chrom=?", (names[i].decode(),)).fetchall() == [(i + 1,)]
            assert db.execute("SELECT count(*) FROM seq INDEXED BY chromidx WHERE chrom>=''").fetchone()[0] == n
        db.close()


def test_packed_names_table():
    names = [b"seq%d" % i for i in range(100000)] + [b"", b"dup", b"dup", "caf\u00e9".encode("utf-8"), b"\xff\xfe"]
    pn = fxi.PackedNames.from_list(names)
    assert len(pn) == len(names) and pn.get(7) == "seq7" and pn.find("seq99999") == 99999 and pn.find("nope") == -1
    assert pn.find("dup") == 100001 and pn.find("") == 100000 and pn.find("caf\u00e9") == 100003
    assert pn.find("\xff\xfe") == 100004            # non-UTF-8 names are shown (and found) as latin-1
    q = ["seq5", "x", "dup", "seq0"]
    assert pn.lookup(q).tolist() == [5, -1, 100001, 0]
    big = pn.lookup(pn)
    assert big[:100001].tolist() == list(range(100001)) and big[100002] == 100001


def test_gz_index_rows_pass_the_reference_import(tmp_path):
    """a .fxi written for a BGZF input carries zran-layout gzindex rows (src/util.c:442-540): the reference opened it
    (pyfastx_load_gzip_index, src/util.c:744-767) and served sequences through it"""
    import struct, zlib
    data = gen.random_fasta(12, n_records=300, crlf_prob=0.0)
    blocks = []
    for o in range(0, len(data), 0xff00):
        chunk = data[o:o + 0xff00]
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        blocks.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25)
                      + comp + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    blocks.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    z = b"".join(blocks)
    path = tmp_path / "b.fa.gz"
    path.write_bytes(z)
    # member table by hand (the C walk needs no GPU either, but keep this test independent of it)
    cmp_off, ucmp_off, p, u = [0], [0], 0, 0
    for b in blocks:
        p += len(b); u += struct.unpack("<I", b[-4:])[0]
        cmp_off.append(p); ucmp_off.append(u)
    gz = fxi.bgzf_gzindex(np.frombuffer(z, np.uint8), np.array(cmp_off), np.array(ucmp_off))
    assert gz["cmp_offset"][0] == 18 and gz["uncmp_offset"][0] == 0 and gz["uncompressed_size"] == len(data)
    exp, total, _ = fxo.fasta_scan(data)
    fxi.write_fasta_index(str(path) + ".fxi", as_rows(exp, FASTA_ROW), fxo.fasta_names(data, exp), total, gz=gz).close()
    db = sqlite3.connect(str(path) + ".fxi")
    blobs = [r[0] for r in db.execute("SELECT content FROM gzindex ORDER BY ID")]
    db.close()
    npts = len(gz["cmp_offset"])
    assert len(blobs) == 8 + 4 * npts and blobs[0] == b"GZIDX" and blobs[1] == b"\x01"
    assert struct.unpack("<Q", blobs[3])[0] == len(z) and struct.unpack("<Q", blobs[4])[0] == len(data)
    assert struct.unpack("<I", blobs[5])[0] >= struct.unpack("<I", blobs[6])[0] >= 32768
    # the reference imported a file with these tables and these gzindex field widths, and served these records
    gold = G.interop("fxi_bgzf_random12")
    assert G.fxi_digest(str(path) + ".fxi", skip=("gzindex",)) == gold["digest"]
    assert [len(b) for b in blobs] == gold["gzindex"]["header"] + gold["gzindex"]["point"] * npts
    assert gold["len"] == len(exp)
    for i, seq in gold["records"]:
        assert G.digest(fxo.subseq(data, exp[i], 0, int(exp["slen"][i]))) == seq
