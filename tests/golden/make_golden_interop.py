#!/usr/bin/env python3
"""Generate tests/golden/golden_interop.json and the reference-written indexes tests/golden/data/*.fxi.gz from the
UNMODIFIED reference (oracle/_ref build): what the reference answers on the seeded inputs of the interoperability
tests (tests/test_oracle_pinned.py, test_fxi_cpu.py, test_gzip_cpu.py, test_api_gpu.py), so that those tests check
against the reference without it.

    bash oracle/build_ref.sh && python tests/golden/make_golden_interop.py

Needs libfxg.so (its .fxi writer runs on the host) but no GPU.  Where the reference opens an index written here, the
generator checks that it loaded that file instead of rebuilding it and stores the file's digest (goldenlib.fxi_digest),
so the tests can require the same file.  Sequences are stored as SHA-256 digests (goldenlib.digest)."""
import ctypes as C
import gzip
import json
import os
import shutil
import sqlite3
import struct
import sys
import tempfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyfastx  # noqa: E402  (the compiled reference)
import gen  # noqa: E402
import goldenlib as G  # noqa: E402
from oracle import fxo  # noqa: E402
from pyfastx_b200 import _cabi, fxi  # noqa: E402
from pyfastx_b200._cabi import FASTA_ROW, FASTQ_ROW  # noqa: E402

D = G.digest
FASTA_TABLES = ("seq", "stat", "comp", "gzindex")
FASTQ_TABLES = ("read", "stat", "base", "meta", "gzindex")


def as_rows(exp, dtype):
    rows = np.zeros(len(exp), dtype=dtype)
    for f in exp.dtype.names:
        if f in rows.dtype.names:
            rows[f] = exp[f]
    return rows


def select(path, sql):
    con = sqlite3.connect(path)
    con.text_factory = bytes
    out = con.execute(sql).fetchall()
    con.close()
    return out


def index_names(path):
    return sorted(r[0].decode() for r in select(path, "SELECT name FROM sqlite_master WHERE type='index'"))


def write_ours_fasta(path, data, gz=None):
    exp, total, _ = fxo.fasta_scan(data)
    fxi.write_fasta_index(path + ".fxi", as_rows(exp, FASTA_ROW), fxo.fasta_names(data, exp), total, gz=gz).close()
    return os.path.getmtime(path + ".fxi")


def loaded_ours(path, mtime):
    assert os.path.getmtime(path + ".fxi") == mtime, "the reference rebuilt the index instead of loading it"


def gz_layout(path, npoints):
    """byte widths of the gzindex header rows and of one checkpoint's rows (the reference reads fixed widths)"""
    blobs = [r[0] for r in select(path, "SELECT content FROM gzindex ORDER BY ID")]
    head, point = [len(b) for b in blobs[:8]], [len(b) for b in blobs[8:12]]
    assert [len(b) for b in blobs[8:8 + 4 * npoints]] == point * npoints
    return {"header": head, "point": point}


def bgzf(data):
    blocks = []
    for o in range(0, len(data), 0xff00):
        chunk = data[o:o + 0xff00]
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        blocks.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25)
                      + comp + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    blocks.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return blocks


def oracle_pinned(tmp, out):
    """test_oracle_pinned: the reference's rows and answers on seeded FASTA / FASTQ"""
    for seed in range(6):
        data = gen.random_fasta(100 + seed, n_records=40, no_trailing_newline=(seed % 2 == 0))
        path = os.path.join(tmp, "p%d.fa" % seed)
        open(path, "wb").write(data)
        fa = pyfastx.Fasta(path)
        exp = [[r[0], r[1].decode("latin-1")] + list(r[2:]) for r in select(path + ".fxi", "SELECT * FROM seq ORDER BY ID")]
        rows, _, _ = fxo.fasta_scan(data)
        rid, s, e = gen.random_queries(rows, 60, seed)
        queries = []
        for i, a, b in zip(rid, s, e):
            r = rows[i]
            if r["norm"] and int(r["slen"]) != len(fxo.subseq(data, r, 0, int(r["slen"])).rstrip(b"\0")):
                continue      # stripped length != slen: reference returns stale bytes (SURVEY Q3)
            sub = fa[exp[i][1]][int(a):int(b)]
            queries.append([int(i), int(a), int(b), D(sub.seq), D(sub.antisense)])
        del fa
        out["fasta_seed%d" % seed] = {"rows": exp, "queries": queries}
    for seed in range(4):
        data = gen.random_fastq(200 + seed, n_reads=150, crlf=(seed % 2 == 1), partial_tail=seed % 3)
        path = os.path.join(tmp, "p%d.fq" % seed)
        open(path, "wb").write(data)
        fq = pyfastx.Fastq(path)
        exp = [[r[0], r[1].decode("latin-1")] + list(r[2:]) for r in select(path + ".fxi", "SELECT * FROM read ORDER BY ID")]
        stat = select(path + ".fxi", "SELECT * FROM stat")[0]
        reads = [[i, D(fq[i].seq), D(fq[i].qual)] for i in range(0, len(exp), 17)]
        del fq
        out["fastq_seed%d" % seed] = {"rows": exp, "stat": [stat[0], stat[1]], "reads": reads}


def fxi_interop(tmp, out):
    """test_fxi_cpu / test_api_gpu: indexes written here that the reference loads, and indexes it writes"""
    data = gzip.open(os.path.join(G.GOLD, "data", "test.fa.gz")).read()
    path = os.path.join(tmp, "t.fa")
    open(path, "wb").write(data)
    mtime = write_ours_fasta(path, data)
    rf = pyfastx.Fasta(path)
    loaded_ours(path, mtime)
    out["fxi_test_fa"] = {"digest": G.fxi_digest(path + ".fxi"), "len": len(rf), "size": rf.size,
                          "records": [[i, rf[i].name, len(rf[i]), D(rf[i].seq), D(rf[i][5:50].antisense)] for i in (0, 17, 210)]}
    del rf
    theirs = os.path.join(tmp, "theirs.fa")
    open(theirs, "wb").write(data)
    rf = pyfastx.Fasta(theirs)
    out["ref_test_fa"] = {"keys": [s.name for s in rf], "seq3_10_200": D(rf[3][10:200].seq)}
    del rf
    save_index(theirs, "test.fa")

    fq_data = gzip.open(os.path.join(G.GOLD, "data", "test.fq.gz")).read()
    for key, data in (("fxi_test_fq", fq_data), ("fxi_random5_fq", gen.random_fastq(5, n_reads=700))):
        path = os.path.join(tmp, key + ".fq")
        open(path, "wb").write(data)
        exp, size, nlines = fxo.fastq_scan(data)
        fxi.write_fastq_index(path + ".fxi", as_rows(exp, FASTQ_ROW), fxo.fastq_names(data, exp), nlines, size).close()
        mtime = os.path.getmtime(path + ".fxi")
        rq = pyfastx.Fastq(path)
        loaded_ours(path, mtime)
        n = len(rq)
        out[key] = {"digest": G.fxi_digest(path + ".fxi"), "len": n,
                    "reads": [[i, rq[i].name, D(rq[i].seq), D(rq[i].qual)] for i in sorted({0, 5, 333 % n, n - 1})]}
        del rq

    # an index the reference writes, loaded here
    path = os.path.join(tmp, "random9.fa")
    open(path, "wb").write(gen.random_fasta(9, n_records=80))
    pyfastx.Fasta(path)
    save_index(path, "random9.fa")

    # the native writer against the reference's own file, table by table
    data = gen.random_fasta(31, n_records=3000, crlf_prob=0.2)
    path = os.path.join(tmp, "a.fa")
    open(path, "wb").write(data)
    pyfastx.Fasta(path)
    out["ref_random31_fa"] = {"tables": {t: D(v) for t, v in G.fxi_rows(path + ".fxi", FASTA_TABLES).items()},
                              "indexes": index_names(path + ".fxi")}
    data = gen.random_fastq(32, n_reads=5000)
    path = os.path.join(tmp, "a.fq")
    open(path, "wb").write(data)
    pyfastx.Fastq(path)
    out["ref_random32_fq"] = {"tables": {t: D(v) for t, v in G.fxi_rows(path + ".fxi", FASTQ_TABLES).items()},
                              "indexes": index_names(path + ".fxi")}


def gz_interop(tmp, out):
    """test_fxi_cpu (BGZF) / test_gzip_cpu (plain gzip): gzindex rows written here that the reference imports"""
    data = gen.random_fasta(12, n_records=300, crlf_prob=0.0)
    blocks = bgzf(data)
    z = b"".join(blocks)
    path = os.path.join(tmp, "b.fa.gz")
    open(path, "wb").write(z)
    cmp_off, ucmp_off, p, u = [0], [0], 0, 0
    for b in blocks:
        p += len(b); u += struct.unpack("<I", b[-4:])[0]
        cmp_off.append(p); ucmp_off.append(u)
    gz = fxi.bgzf_gzindex(np.frombuffer(z, np.uint8), np.array(cmp_off), np.array(ucmp_off))
    mtime = write_ours_fasta(path, data, gz=gz)
    rf = pyfastx.Fasta(path)
    loaded_ours(path, mtime)
    out["fxi_bgzf_random12"] = {"digest": G.fxi_digest(path + ".fxi", skip=("gzindex",)),
                                "gzindex": gz_layout(path + ".fxi", len(gz["cmp_offset"])), "len": len(rf),
                                "records": [[i, D(rf[i].seq)] for i in (0, 150, 299)]}
    del rf

    raw = gen.random_fasta(21, n_records=900, crlf_prob=0.0)
    z = gzip.compress(raw, compresslevel=6)
    a = np.frombuffer(z, dtype=np.uint8)
    h = C.c_void_p()
    L = _cabi.lib()
    _cabi.check(L.fxg_gzip_inflate_host(a.ctypes.data, a.size, 65536, C.byref(h)))
    gzi = _cabi.GzIndex()
    _cabi.check(L.fxg_gzip_index(h, C.byref(gzi)))
    path = os.path.join(tmp, "g.fa.gz")
    open(path, "wb").write(z)
    mtime = write_ours_fasta(path, raw, gz=gzi)
    L.fxg_gzip_free(h)
    rf = pyfastx.Fasta(path)
    loaded_ours(path, mtime)
    out["fxi_gzip_random21"] = {"digest": G.fxi_digest(path + ".fxi", skip=("gzindex",)),
                                "gzindex": gz_layout(path + ".fxi", gzi.npoints), "len": len(rf),
                                "records": [[len(rf) - 1, D(rf[len(rf) - 1].seq)]]}
    del rf


def save_index(path, name):
    dst = os.path.join(HERE, "data", name + ".fxi.gz")
    with open(path + ".fxi", "rb") as f, gzip.GzipFile(dst, "wb", mtime=0) as o:
        o.write(f.read())


def main():
    tmp = tempfile.mkdtemp(prefix="fxginterop")
    out = {}
    try:
        oracle_pinned(tmp, out)
        fxi_interop(tmp, out)
        gz_interop(tmp, out)
    finally:
        shutil.rmtree(tmp)
    dst = os.path.join(HERE, "golden_interop.json")
    with open(dst, "w") as f:                             # one line per case
        f.write('{"reference": %s,\n"cases": {\n' % json.dumps(pyfastx.version(debug=True)))
        f.write(",\n".join("%s: %s" % (json.dumps(k), json.dumps(out[k], separators=(",", ":"))) for k in sorted(out)))
        f.write("\n}}\n")
    print("wrote", dst, os.path.getsize(dst), "bytes;", len(out), "cases")


if __name__ == "__main__":
    main()
