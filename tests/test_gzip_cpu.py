"""Generic (non-BGZF) gzip on the host (csrc/fxg_gzip.cpp): the one sequential zlib pass must reproduce the input
and every checkpoint it collects must be a REAL zran access point -- raw inflate restarted there with
inflatePrime(bits) + inflateSetDictionary(window) yields exactly the bytes that follow.  The rows the .fxi then
carries pass the reference's import (src/util.c:575-609) and the reference serves sequences through our index
(recorded by tests/golden/make_golden_interop.py)."""
import ctypes as C
import gzip
import sqlite3
import struct
import zlib

import numpy as np
import pytest

import gen
import goldenlib as G
from oracle import fxo
from pyfastx_b200 import _cabi, fxi
from pyfastx_b200._cabi import FASTA_ROW


def inflate_host(z, spacing=0):
    L = _cabi.lib()
    a = np.frombuffer(z, dtype=np.uint8)
    h = C.c_void_p()
    _cabi.check(L.fxg_gzip_inflate_host(a.ctypes.data, a.size, spacing, C.byref(h)))
    n = C.c_int64(0)
    p = L.fxg_gzip_data(h, C.byref(n))
    data = bytes((C.c_uint8 * n.value).from_address(p)) if n.value else b""
    gz = _cabi.GzIndex()
    _cabi.check(L.fxg_gzip_index(h, C.byref(gz)))
    k = gz.npoints
    pts = {"cmp": np.frombuffer((C.c_int64 * k).from_address(gz.cmp_offset), dtype=np.int64).copy(),
           "ucmp": np.frombuffer((C.c_int64 * k).from_address(gz.uncmp_offset), dtype=np.int64).copy(),
           "bits": np.frombuffer((C.c_uint8 * k).from_address(gz.bits), dtype=np.uint8).copy(),
           "has": np.frombuffer((C.c_uint8 * k).from_address(gz.has_data), dtype=np.uint8).copy()}
    nw = int(pts["has"].sum())
    pts["win"] = bytes((C.c_uint8 * (nw * gz.window_size)).from_address(gz.windows)) if nw else b""
    return data, gz, pts, h


def resume(z, data, pts, i, wsize=32768):
    """inflate from checkpoint i to the next checkpoint (or the end of the member) with plain zlib"""
    c, u, bits = int(pts["cmp"][i]), int(pts["ucmp"][i]), int(pts["bits"][i])
    d = zlib.decompressobj(-15, zdict=pts["win"][int(pts["has"][:i].sum()) * wsize:][:wsize]) if pts["has"][i] else zlib.decompressobj(-15)
    stream = z[c:]
    if bits:
        # zlib's python binding has no inflatePrime: shift the stream so that the block starts on a byte boundary
        pre = z[c - 1] >> (8 - bits)
        v = int.from_bytes(stream[:1 << 16], "little")
        v = (v << bits) | pre
        stream = v.to_bytes((1 << 16) + 1, "little")
    want = 4096
    out = d.decompress(stream[:1 << 16], want)
    return out, data[u:u + len(out)]


@pytest.mark.parametrize("level,size", [(1, 300000), (6, 5 << 20), (9, 1 << 20)])
def test_one_pass_inflates_and_checkpoints_are_real_access_points(level, size):
    raw = gen.random_fasta(level, n_records=max(20, size // 4000), crlf_prob=0.0)[:size]
    z = gzip.compress(raw, compresslevel=level)
    data, gz, pts, h = inflate_host(z, spacing=65536)
    assert data == raw and gz.uncompressed_size == len(raw) and gz.compressed_size == len(z)
    assert gz.window_size == 32768 and gz.spacing >= gz.window_size
    k = gz.npoints
    assert k >= 1 and pts["ucmp"][0] == 0 and pts["has"][0] == 0 and (np.diff(pts["ucmp"]) >= 65536).all()
    assert len(raw) < 200000 or k >= len(raw) // (65536 * 4)
    for i in range(k):
        got, exp = resume(z, raw, pts, i)
        assert len(got) > 0 and got == exp, "checkpoint %d (bits %d) does not resume the stream" % (i, pts["bits"][i])
    _cabi.lib().fxg_gzip_free(h)


def test_concatenated_members_and_corrupt_streams():
    a, b = gen.random_fasta(1, n_records=50), gen.random_fasta(2, n_records=70)
    z = gzip.compress(a) + gzip.compress(b)
    data, gz, pts, h = inflate_host(z)
    assert data == a + b and pts["ucmp"].tolist()[:2] == [0, len(a)]
    _cabi.lib().fxg_gzip_free(h)
    bad = bytearray(gzip.compress(a))
    bad[len(bad) // 2] ^= 0x55
    with pytest.raises(_cabi.FxgError):
        inflate_host(bytes(bad))
    with pytest.raises(_cabi.FxgError):
        inflate_host(gzip.compress(a)[:-20])


def test_fxi_for_plain_gzip_carries_windows_and_the_reference_opens_it(tmp_path):
    raw = gen.random_fasta(21, n_records=900, crlf_prob=0.0)
    z = gzip.compress(raw, compresslevel=6)
    data, gz, pts, h = inflate_host(z, spacing=65536)
    exp, total, _ = fxo.fasta_scan(raw)
    rows = np.zeros(len(exp), dtype=FASTA_ROW)
    for f in exp.dtype.names:
        if f in rows.dtype.names:
            rows[f] = exp[f]
    path = tmp_path / "g.fa.gz"
    path.write_bytes(z)
    fxi.write_fasta_index(str(path) + ".fxi", rows, fxo.fasta_names(raw, exp), total, gz=gz).close()
    db = sqlite3.connect(str(path) + ".fxi")
    blobs = [r[0] for r in db.execute("SELECT content FROM gzindex ORDER BY ID")]
    assert db.execute("PRAGMA integrity_check").fetchall() == [("ok",)]
    db.close()
    k, nw = gz.npoints, int(pts["has"].sum())
    assert len(blobs) == 8 + 4 * k + nw and blobs[0] == b"GZIDX"
    assert struct.unpack("<I", blobs[7])[0] == k and all(len(b) == 32768 for b in blobs[8 + 4 * k:])
    assert blobs[8 + 4 * k:] == [pts["win"][i * 32768:(i + 1) * 32768] for i in range(nw)]
    # the loader that feeds the GPU inflate-from-checkpoints path reads the same table back
    back = fxi.read_gzindex(str(path) + ".fxi")
    assert back is not None and back["npoints"] == k and back["windows"] == nw
    assert back["compressed_size"] == len(z) and back["uncompressed_size"] == len(raw)
    co, uo, bt, hs, wn = back["keep"]
    assert np.array_equal(co, pts["cmp"]) and np.array_equal(uo, pts["ucmp"]) and np.array_equal(bt, pts["bits"])
    assert np.array_equal(hs, pts["has"]) and wn.tobytes() == pts["win"]
    _cabi.lib().fxg_gzip_free(h)
    assert fxi.read_gzindex(str(tmp_path / "absent.fxi")) is None
    # the reference imported a file with these tables and these gzindex field widths, and served this record
    gold = G.interop("fxi_gzip_random21")
    assert G.fxi_digest(str(path) + ".fxi", skip=("gzindex",)) == gold["digest"]
    assert [len(b) for b in blobs[:8 + 4 * k]] == gold["gzindex"]["header"] + gold["gzindex"]["point"] * k
    assert gold["len"] == len(exp)
    for i, seq in gold["records"]:
        assert G.digest(fxo.subseq(raw, exp[i], 0, int(exp["slen"][i]))) == seq
