"""The pyfastx-compatible object API end to end on the GPU: index build -> .fxi (reference schema)
-> getters, mirroring the reference's own tests (tests/test_fasta.py, test_sequence.py,
test_fastq.py, test_read.py) with the golden vectors standing in for pyfaidx."""
import gzip
import os
import sqlite3

import numpy as np
import pytest

import goldenlib as G
import pyfastx_b200 as pyfastx

pytestmark = pytest.mark.gpu


def fxi_rows(path, table):
    con = sqlite3.connect(path)
    rows = [list(r) for r in con.execute("SELECT * FROM %s ORDER BY ID" % table)]
    stat = [list(r) for r in con.execute("SELECT * FROM stat")]
    idx = [r[0] for r in con.execute("SELECT name FROM sqlite_master WHERE type='index'")]
    con.close()
    return rows, stat, idx


def write(tmp_path, name, data):
    p = tmp_path / name
    p.write_bytes(data)
    return str(p)


@pytest.mark.parametrize("case", [c for c in G.cases("fasta") if not any(r[1] in (None, "") for r in c["rows"])],
                         ids=lambda c: c["name"])
def test_fasta_api_golden(tmp_path, case):
    path = write(tmp_path, "x.fa", G.case_data(case))
    fa = pyfastx.Fasta(path, uppercase=case["uppercase"], full_name=case["full_name"])
    rows, stat, idx = fxi_rows(path + ".fxi", "seq")
    assert rows == case["rows"]
    assert stat[0][:2] == case["stat"] and stat[0][2:] == [None, None, None, None]
    assert len(fa) == case["stat"][0] and fa.size == case["stat"][1]
    names = [r[1] for r in case["rows"]]
    if len(set(names)) == len(names):
        assert "chromidx" in idx
    for q in case["queries"][:25]:
        sub = fa[names[q["row"]]][q["s"]:q["e"]]
        assert len(sub) == q["e"] - q["s"]
        assert (sub.seq, sub.antisense, sub.reverse, sub.complement) == (q["seq"], q["antisense"], q["reverse"], q["complement"])
        assert (sub.start, sub.end) == (q["s"] + 1, q["e"])
    for q in case["fetch"]:
        iv = [tuple(x) for x in q["intervals"]]
        arg = iv[0] if len(iv) == 1 else iv
        assert fa.fetch(names[q["row"]], arg, strand=q["strand"]) == q["seq"]
    for g in case["gc"]:
        sq = fa[g["row"]]
        assert sq.composition == g["composition"]
        if g["gc_content"] is not None:
            assert sq.gc_content == g["gc_content"]
        if g["gc_skew"] is not None:
            assert sq.gc_skew == g["gc_skew"]
    # batched form == per-query form
    qs = case["queries"]
    if qs:
        got = fa.fetch_many([names[q["row"]] for q in qs], [q["s"] + 1 for q in qs], [q["e"] for q in qs],
                            ["-" if i % 2 else "+" for i in range(len(qs))])
        uniform = all(r[7] == 1 for r in case["rows"]) and "first_line" not in case["name"] and "norm_rules" not in case["name"]
        for i, q in enumerate(qs):
            # fetch semantics index into the whole stripped record; identical to slicing on
            # records whose lines are uniform, and always identical to fetch() itself
            assert got[i] == fa.fetch(names[q["row"]], (q["s"] + 1, q["e"]), strand="-" if i % 2 else "+")
            if uniform:
                assert got[i] == (q["antisense"] if i % 2 else q["seq"])
    # reload from the .fxi we wrote
    fb = pyfastx.Fasta(path, uppercase=case["uppercase"], full_name=case["full_name"])
    assert len(fb) == len(fa) and fb.keys() == fa.keys()
    for q in qs[:5]:
        assert fb[names[q["row"]]][q["s"]:q["e"]].seq == q["seq"]


def test_fasta_readme_answers(tmp_path):
    """README.rst known answers (SURVEY.md section 8c)"""
    data = gzip.open(os.path.join(G.GOLD, "data", "test.fa.gz")).read()
    fa = pyfastx.Fasta(write(tmp_path, "test.fa", data))
    assert len(fa) == 211 and fa.size == 86262
    assert fa.gc_content == 43.529014587402344 and fa.gc_skew == 0.004287730902433395
    assert fa.composition == {"A": 24534, "C": 18694, "G": 18855, "T": 24179}
    assert fa.fetch("JZ822577.1", (1, 10)) == "CTCTAGAGAT"
    assert fa.fetch("JZ822577.1", [(1, 10), (50, 60)]) == "CTCTAGAGATTTTAGTTTGAC"
    assert fa.fetch("JZ822577.1", (1, 10), strand="-") == "ATCTCTAGAG"
    s = fa[-1]
    assert s.gc_content == 46.26865768432617 and s.composition == {"A": 31, "C": 37, "G": 25, "T": 41}
    assert s[10:30].seq == "CTTCTTCCTGTGGAAAGTAA" and s[-10:].seq == "CCATGTTGGT"
    assert "JZ822577.1" in fa and "nope" not in fa
    assert fa.type == "DNA"
    assert s[0] == s.seq[0] and s[-1] == s.seq[-1]
    left, right = fa.flank("JZ822577.1", 100, 110, flank_length=20)
    whole = fa["JZ822577.1"].seq
    assert left == whole[79:99] and right == whole[110:130]
    assert pyfastx.reverse_complement("ATCGNatcgn") == "ncgatNCGAT"


def test_fasta_errors(tmp_path):
    with pytest.raises(FileExistsError):
        pyfastx.Fasta(str(tmp_path / "missing.fa"))
    with pytest.raises(RuntimeError):
        pyfastx.Fasta(write(tmp_path, "bad.fa", b"@r1\nACGT\n+\nIIII\n"))
    with pytest.raises(TypeError):
        pyfastx.Fasta(write(tmp_path, "k.fa", b">a\nAC\n"), key_func=3)
    fa = pyfastx.Fasta(write(tmp_path, "ok.fa", b">a desc\nACGTACGT\nACGT\n>b\nGGCC\n"))
    with pytest.raises(KeyError):
        fa["zzz"]
    with pytest.raises(IndexError):
        fa[5]
    with pytest.raises(NameError):
        fa.fetch("zzz", (1, 2))
    with pytest.raises(ValueError):
        fa.fetch("a", (5, 2))
    with pytest.raises(ValueError):
        fa.fetch("a", 5)
    with pytest.raises(ValueError):
        fa["a"][::2]
    assert fa["a"][2:6].seq == "GTAC" and fa["a"].description == "a desc" and fa["a"].raw == ">a desc\nACGTACGT\nACGT\n"
    assert [len(s) for s in fa] == [12, 4]
    assert fa.longest.name == "a" and fa.shortest.name == "b" and fa.mean == 8.0 and fa.median == 8.0
    assert fa.nl(50) == (12, 1) and fa.count(5) == 1
    assert list(fa["a"]) == ["ACGTACGT", "ACGT"]
    assert fa["a"].search("GTAC") == 3 and fa["a"].search("GTAC", "-") == 3


def test_key_func_and_memory_index(tmp_path):
    path = write(tmp_path, "k.fa", b">sp|P1|X desc\nACGT\n>sp|P2|Y\nGG\n")
    fa = pyfastx.Fasta(path, key_func=lambda x: x.split("|")[1], memory_index=True)
    assert fa.keys() == ["P1", "P2"] and fa["P2"].seq == "GG"
    assert not os.path.exists(path + ".fxi")


def test_gzip_input(tmp_path):
    raw = gzip.open(os.path.join(G.GOLD, "data", "test_crlf.fa.gz")).read()
    p = tmp_path / "t.fa.gz"
    p.write_bytes(open(os.path.join(G.GOLD, "data", "test_crlf.fa.gz"), "rb").read())
    fa = pyfastx.Fasta(str(p))
    case = [c for c in G.cases("fasta") if c["name"] == "test_fa_crlf"][0]
    rows, _, _ = fxi_rows(str(p) + ".fxi", "seq")
    assert rows == case["rows"] and fa.is_gzip and pyfastx.gzip_check(str(p))
    q = case["queries"][0]
    assert fa[q["row"]][q["s"]:q["e"]].seq == q["seq"]
    assert len(raw) > 0


@pytest.mark.parametrize("case", G.cases("fastq"), ids=G.case_ids("fastq"))
def test_fastq_api_golden(tmp_path, case):
    path = write(tmp_path, "x.fq", G.case_data(case))
    fq = pyfastx.Fastq(path)
    rows, stat, idx = fxi_rows(path + ".fxi", "read")
    assert rows == case["rows"]
    assert stat[0][:2] == case["stat"][:2] and (stat[0][2] == case["stat"][2] or case["stat"][0] == 0)
    assert len(fq) == case["stat"][0] and fq.size == case["stat"][1]
    for q in case["reads"]:
        r = fq[q["id"]]
        assert (r.seq, r.qual, r.antisense) == (q["seq"], q["qual"], q["antisense"])
        assert r.quali == [ord(c) - 33 for c in q["qual"]]
        assert fq[r.name].seq == q["seq"] or len(set(fq.keys())) != len(fq.keys())
    if case["reads"]:
        ids = [q["id"] for q in case["reads"]]
        seq, qual, off = fq.reads_many(ids)
        for i, q in enumerate(case["reads"]):
            assert seq[off[i]:off[i + 1]].tobytes().decode() == q["seq"] and qual[off[i]:off[i + 1]].tobytes().decode() == q["qual"]
    with pytest.raises(IndexError):
        fq[len(fq) + 5]
    with pytest.raises(KeyError):
        fq["definitely-not-a-read"]


def test_fxi_interoperates_with_reference(tmp_path):
    """the reference loads an index written here, and we load one written by the reference: an index written here
    has the digest of the file the reference loaded as its own (tests/golden/make_golden_interop.py), whose records
    it served as recorded there; the reference-written index is stored under tests/golden/data"""
    data = gzip.open(os.path.join(G.GOLD, "data", "test.fa.gz")).read()
    ours = write(tmp_path, "ours.fa", data)
    fa = pyfastx.Fasta(ours)                       # writes ours.fa.fxi on the GPU path
    gold = G.interop("fxi_test_fa")
    assert G.fxi_digest(ours + ".fxi") == gold["digest"]
    assert gold["len"] == len(fa) == 211
    for i, name, n, seq, anti in gold["records"]:
        assert G.digest(fa[i].seq) == seq and fa[i].name == name and len(fa[i]) == n
        assert G.digest(fa[i][5:50].antisense) == anti
    theirs = write(tmp_path, "theirs.fa", data)
    G.reference_index("test.fa", theirs + ".fxi")  # the index the reference built for test.fa
    fb = pyfastx.Fasta(theirs)                     # we load THEIR index
    gold = G.interop("ref_test_fa")
    assert fb.keys() == gold["keys"]
    assert G.digest(fb[3][10:200].seq) == gold["seq3_10_200"]
    fq_data = gzip.open(os.path.join(G.GOLD, "data", "test.fq.gz")).read()
    oq = write(tmp_path, "ours.fq", fq_data)
    fq = pyfastx.Fastq(oq)
    gold = G.interop("fxi_test_fq")
    assert G.fxi_digest(oq + ".fxi") == gold["digest"]
    assert gold["len"] == len(fq) == 800
    for i, name, seq, qual in gold["reads"]:
        assert fq[i].name == name and G.digest(fq[i].seq) == seq and G.digest(fq[i].qual) == qual


def test_compiled_object_layer_keys_and_fastx(tmp_path):
    """the object layer in use is the compiled CPython extension (PyInit_pyfastx); key views and the Fastx iterator"""
    assert pyfastx.COMPILED and pyfastx.Fasta.__module__.endswith("pyfastx")
    data = gzip.open(os.path.join(G.GOLD, "data", "test.fa.gz")).read()
    case = [c for c in G.cases("fasta") if c["name"] == "test_fa"][0]
    path = write(tmp_path, "t.fa", data)
    fa = pyfastx.Fasta(path)
    keys = fa.keys()
    names = [r[1] for r in case["rows"]]
    assert isinstance(keys, pyfastx.FastaKeys) and len(keys) == 211 and list(keys) == names
    assert keys[0] == names[0] and keys[-1] == names[-1] and names[5] in keys and "nope" not in keys
    recs = list(pyfastx.Fastx(path))
    assert [r[0] for r in recs] == names and all(recs[i][1] == fa[i].seq for i in (0, 100, 210))
    with_comment = list(pyfastx.Fastx(path, comment=True))
    assert with_comment[0][2] == fa[0].description[len(names[0]) + 1:]
    fq_case = [c for c in G.cases("fastq") if c["name"] == "test_fq"][0]
    qpath = write(tmp_path, "t.fq", G.case_data(fq_case))
    fq = pyfastx.Fastq(qpath)
    recs = list(pyfastx.Fastx(qpath))
    assert len(recs) == 800 and isinstance(fq.keys(), pyfastx.FastqKeys)
    for q in fq_case["reads"][:10]:
        assert recs[q["id"]][1] == q["seq"] and recs[q["id"]][2] == q["qual"] and recs[q["id"]][0] == fq[q["id"]].name


@pytest.mark.gpu
@pytest.mark.parametrize("service", ["1", "0"])
def test_per_object_getters_service_and_launch_paths(tmp_path, monkeypatch, service):
    """fa[name][s:e].seq / .antisense and fq[i].seq / .qual one query per call -- through the resident service kernel
    (mapped-memory requests, no launch per query) and through the launch + synchronise path: identical to the batched
    API, also after the service kernel has left on its idle period (sleep) and for queries that span several warps"""
    import time
    monkeypatch.setenv("FXG_ONE_SERVICE", service)
    import pyfastx_b200
    from pyfastx_b200 import synth
    p = tmp_path / "s.fa"
    p.write_bytes(synth.synth_fasta(60, seed=11))
    fa = pyfastx_b200.Fasta(str(p))
    rng = np.random.default_rng(5)
    names, qs, qe, minus = [], [], [], []
    for k in range(300):
        i = int(rng.integers(0, len(fa)))
        n = len(fa[i])
        L = int(rng.choice([1, 15, 16, 17, 100, 1000, 2047, 2048, 5000, n]))
        L = min(L, n)
        a = int(rng.integers(0, n - L + 1))
        names.append(fa[i].name); qs.append(a); qe.append(a + L); minus.append(bool(k & 1))
    want = fa.fetch_many(names, np.array(qs) + 1, np.array(qe), ["-" if m else "+" for m in minus])
    for k in range(300):
        sub = fa[names[k]][qs[k]:qe[k]]
        assert (sub.antisense if minus[k] else sub.seq) == want[k], k
        if k == 150:
            time.sleep(0.02)                                  # longer than the service kernel's idle period: it relaunches
    q = tmp_path / "s.fq"
    q.write_bytes(synth.synth_fastq(500, seed=12))
    fq = pyfastx_b200.Fastq(str(q))
    ids = [int(x) for x in rng.integers(0, len(fq), size=100)]
    sq, ql, off = fq.reads_many(ids)
    for k, i in enumerate(ids):
        r = fq[i]
        want_seq = bytes(sq[off[k]:off[k + 1]]).decode()
        assert r.seq == want_seq and r.qual == bytes(ql[off[k]:off[k + 1]]).decode()
        assert r.antisense == pyfastx_b200.reverse_complement(want_seq)


@pytest.mark.gpu
def test_device_buffer_pool_reuse():
    """fxg_file_free keeps one spare buffer per device; the next allocation that fits takes it (same pointer), a much
    larger one does not, fxg_pool_trim returns it"""
    from pyfastx_b200 import _cabi, engine
    eng = engine.get_engine(0)
    L = _cabi.lib()
    L.fxg_pool_trim()
    a = eng.alloc_file(600 << 20)
    pa = a.devptr
    a.free()
    b = eng.alloc_file(400 << 20)                             # fits into the spare (within 2x + 256 MiB)
    assert b.devptr == pa
    b.free()
    c = eng.alloc_file(20 << 20)                              # far smaller than the spare: a fresh allocation
    assert c.devptr != pa
    c.free()
    L.fxg_pool_trim()
    d = eng.alloc_file(100 << 20)
    d.free()
    L.fxg_pool_trim()


@pytest.mark.gpu
def test_plain_gzip_second_open_inflates_on_the_gpu_from_checkpoints(tmp_path):
    """a plain (non-BGZF) .gz: the first open runs the one sequential host pass and stores real zran checkpoints in the
    .fxi; the second open inflates every checkpoint's segment with its own GPU thread (verified against the gzip
    trailer's CRC-32) -- same bytes, same rows, same sequences; checkpoints that do not fit the file fall back"""
    import gzip as _gzip
    import pyfastx_b200
    from pyfastx_b200 import synth
    raw = synth.synth_fasta(520, seed=31)                        # ~5.3 MB: several 1 MiB checkpoints
    p = tmp_path / "plain.fa.gz"
    p.write_bytes(_gzip.compress(raw, compresslevel=6))
    a = pyfastx_b200.Fasta(str(p))
    assert a._st.gzip_path == "host-zlib" and a.is_gzip
    first, last, n, size = a[0].seq, a[len(a) - 1][100:3000].antisense, len(a), a.size
    del a
    b = pyfastx_b200.Fasta(str(p))
    assert b._st.gzip_path == "gpu-checkpoints"
    assert bytes(b._st.dfile.download()) == raw
    assert (len(b), b.size) == (n, size) and b[0].seq == first and b[len(b) - 1][100:3000].antisense == last
    del b
    # another file's checkpoints (same index path): the CRC check rejects the result, the host pass takes over
    raw2 = synth.synth_fasta(520, seed=32)
    z2 = _gzip.compress(raw2, compresslevel=6)
    q = tmp_path / "other.fa.gz"
    q.write_bytes(z2)
    os.replace(str(p) + ".fxi", str(q) + ".fxi")
    c = pyfastx_b200.Fasta(str(q))
    assert c._st.gzip_path == "host-zlib" and bytes(c._st.dfile.download()) == raw2
