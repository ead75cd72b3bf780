"""Load tests/golden/golden.json and golden_interop.json (reference-generated, see tests/golden/make_golden.py and
make_golden_interop.py)."""
import base64
import gzip
import hashlib
import json
import os
import sqlite3

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
_CACHE = {}


def _synth(spec):
    from pyfastx_b200 import synth
    _, kind, n, seed = spec.split(":")
    n, seed = int(n), int(seed)
    if kind == "fasta":
        return synth.synth_fasta(n, seed=seed)
    if kind == "fasta_w60crlf":
        return synth.synth_fasta(n, seed=seed, min_len=1, max_len=700, width=60, crlf=True)
    if kind == "fastq":
        return synth.synth_fastq(n, seed=seed)
    raise ValueError(spec)


def case_data(case):
    if "data_b64" in case:
        return base64.b64decode(case["data_b64"])
    df = case["datafile"]
    if df.startswith("synth:"):
        return _synth(df)
    return gzip.open(os.path.join(GOLD, "data", df), "rb").read()


def cases(kind=None):
    if "all" not in _CACHE:
        with open(os.path.join(GOLD, "golden.json")) as f:
            _CACHE["all"] = json.load(f)["cases"]
    return [c for c in _CACHE["all"] if kind is None or c["kind"] == kind]


def case_ids(kind=None):
    return [c["name"] for c in cases(kind)]


def interop(key):
    """what the reference answered on one input of the interoperability tests (golden_interop.json)"""
    if "interop" not in _CACHE:
        with open(os.path.join(GOLD, "golden_interop.json")) as f:
            _CACHE["interop"] = json.load(f)["cases"]
    return _CACHE["interop"][key]


def reference_index(name, dst):
    """write the reference-written index tests/golden/data/<name>.fxi.gz to `dst`"""
    with gzip.open(os.path.join(GOLD, "data", name + ".fxi.gz"), "rb") as f, open(dst, "wb") as o:
        o.write(f.read())


def digest(x):
    """SHA-256 (first 128 bits) of a sequence (str or bytes) or of the repr of rows: how golden_interop.json stores
    large values"""
    if isinstance(x, str):
        x = x.encode("latin-1")
    elif not isinstance(x, (bytes, bytearray)):
        x = repr(x).encode()
    return hashlib.sha256(x).hexdigest()[:32]


def fxi_rows(path, tables):
    """{table: rows in rowid order} of an index file, text as bytes"""
    db = sqlite3.connect(path)
    db.text_factory = bytes
    out = {t: db.execute("SELECT * FROM %s ORDER BY rowid" % t).fetchall() for t in tables}
    db.close()
    return out


def fxi_digest(path, skip=()):
    """digest of an index file's schema and of every table but `skip`: two files with the same digest answer
    every SELECT the same"""
    db = sqlite3.connect(path)
    db.text_factory = bytes
    schema = db.execute("SELECT type, name, tbl_name, sql FROM sqlite_master ORDER BY type, name").fetchall()
    db.close()
    tables = [n.decode() for t, n, _, _ in schema if t == b"table" and n.decode() not in skip]
    return digest((schema, fxi_rows(path, tables)))
