#!/usr/bin/env python3
"""bench.py -- index-build GB/s (+ subseq-extract Mbases/s) of the B200-native pyfastx hot path.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU path (oracle/_ref)
    python bench.py ... --dump-outputs DIR     # + what the last timed step computed, as DIR/<name>.npy

One JSON line on rank 0.  Workloads (BASELINE.json configs, synthetic, generated in HBM; every file is far
larger than L2, so no flush is needed between steps):

  headline (C2)   ONE synthetic plain FASTA of N x 1M records (10.16 GB per GPU, weak scaling).  Every rank takes
                  the byte range [i*S/N, (i+1)*S/N) of that file, moved to the next header line FOUND ON THE DATA
                  (fxg_split_point_dev), and a "step" is one sharded index build of the resident range:
                  fxg_scan_begin (mark + prefix) -> fxg_shard_exchange (ncclAllGather of the 128-byte shard
                  infos on the context's stream) -> fxg_scan_finish (rows) -- the C-ABI call fxg_scan_sharded.
  "fastq" (C4)    ONE 41.5 GB FASTQ (126M reads x 150 bp + qual) for every N (STRONG scaling): rank i scans the
                  byte range i of N, cut at line starts found on the data; the global line phase comes from the
                  all-gather, boundary reads are completed on the device from the gathered edge lines.
  "extract" (C3)  10M random (record, start, end, strand) 1 kb queries per GPU on its resident range, plus the
                  mixed-length set L ~ U[50, 5000].
  "bgzf" (C5)     N = 1: the C2 file as BGZF (zlib level 6): member walk + GPU inflate + scan + 1M fetches.
  "e2e"           the call a user makes: pyfastx_b200.Fasta(path) on a tmpfs file -- staging (pread -> pinned ->
                  H2D), scan, names D2H, `.fxi` written by the native bulk writer.
Every arm times --steps K steps: the scans and extractions after --warmup W (at least 3) steps, the e2e and BGZF
builds after one warm-up build (e2e: median, BGZF: best of the K builds).
Parity (rank-local, before anything is reported): ALL rows of C2 and C4 against the CPU oracle (oracle/fxo.c)
on the downloaded range, >= 3M C4 reads and a C2 sample against the compiled reference (oracle/_ref), ALL 10M
C3 outputs byte-compared with the oracle, C5 inflated bytes == input bytes.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                      # the tree may be read-only: no __pycache__ written into it

SEED_FASTA = 20240601
SEED_FASTQ = 20240602
SEED_QUERIES = 123
SEED_DUMP = 7
FQ_FIXED = 5 + 11 + 1 + 150 + 1 + 2 + 150 + 1      # "@read" + " 1:N:0:ACGT" + "\n" + seq "\n" "+\n" qual "\n"
DUMP_ROW_BLOCKS, DUMP_QUERIES, DUMP_LIMIT = 128, 1024, 64 << 20


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step computed (rank 0), for comparing two builds output for output.  Outputs
# too large to keep whole are sampled at indices fixed by SEED_DUMP; 64 MB in all.
# ---------------------------------------------------------------------------------------------
def dump(c, name, a, dtype=np.float64):
    a = np.ascontiguousarray(a, dtype=dtype)
    c.dump_bytes += a.nbytes
    assert c.dump_bytes <= DUMP_LIMIT, "--dump-outputs: more than %d bytes" % DUMP_LIMIT
    np.save(os.path.join(c.dump, name + ".npy"), a)


def dump_sample(n, count):
    """sorted indices of a fixed sample of `count` of n items (all of them when n <= count)"""
    if n <= count:
        return np.arange(n)
    return np.sort(np.random.default_rng(SEED_DUMP).choice(n, size=count, replace=False))


def dump_rows(c, name, d_rows, st, dtype):
    """scan stats and DUMP_ROW_BLOCKS blocks of 1024 consecutive rows from the device: <name>_row (the row numbers),
    <name>_<field> per field"""
    n_rows, blk = int(st["n_rows"]), 1024
    parts = []
    for a in dump_sample(-(-n_rows // blk), DUMP_ROW_BLOCKS) * blk:
        part = np.zeros(min(blk, n_rows - a), dtype=dtype)
        c.check(c.L.fxg_rows_download(c.eng.ctx, d_rows + int(a) * dtype.itemsize, part.size, dtype.itemsize, part.ctypes.data))
        parts.append((np.arange(a, a + part.size), part))
    rows = np.concatenate([p for _, p in parts]) if parts else np.zeros(0, dtype=dtype)
    dump(c, name + "_stats", [st[k] for k in ("n_rows", "n_lines", "total_len", "end_position", "lead_lines", "lead_bytes", "lead_llen")])
    dump(c, name + "_row", np.concatenate([i for i, _ in parts]) if parts else [])
    for f in dtype.names:
        if f != "pad":
            dump(c, name + "_" + f, rows[f])


def dump_extract(c, label, d_off, d_out):
    """a fixed sample of DUMP_QUERIES queries of an extraction: extract_<label>_query (query numbers), _length, _bytes"""
    off = d_off.cpu().numpy()
    sel = dump_sample(off.size - 1, DUMP_QUERIES)
    pos = np.concatenate([np.arange(off[i], off[i + 1]) for i in sel])
    out = d_out[c.torch.from_numpy(pos).to(d_out.device)].cpu().numpy()
    dump(c, "extract_%s_query" % label, sel)
    dump(c, "extract_%s_length" % label, off[sel + 1] - off[sel])
    dump(c, "extract_%s_bytes" % label, out, np.float32)


# ---------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------
def ncu_traffic(kernel, alg_bytes):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full captures (profiles/*_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum next to the algorithmic bytes of the captured launch)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))[kernel]
            ratio = t["dram_bytes"] / t["algorithmic_bytes"]
            return {"traffic": ratio * alg_bytes, "traffic_over_algorithmic": ratio,
                    "traffic_source": "profiles/%s (%s)" % (name, t["capture"])}
        except Exception:
            continue
    return {"traffic": None}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under load (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    clk, cmx, util = float(f[1]), float(f[2]), float(f[8])
                except ValueError:
                    continue
                if util < 50:
                    continue                                    # only samples taken under load
                sm.append(clk); mx.append(cmx)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def pinned_array(n, dtype):
    from pyfastx_b200 import _cabi
    dt = np.dtype(dtype)
    p = C.c_void_p()
    _cabi.check(_cabi.lib().fxg_host_alloc(int(n) * dt.itemsize, C.byref(p)))
    buf = (C.c_uint8 * (int(n) * dt.itemsize)).from_address(p.value)
    a = np.frombuffer(buf, dtype=dt, count=int(n))
    return a, p


def shm_dir():
    return "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else tempfile.gettempdir()


def n_threads(cap=64):
    return max(1, min(cap, os.cpu_count() or 1))


def digits_upto(i):
    """total decimal digits of 1..i"""
    total, lo, d = 0, 1, 1
    while lo <= i:
        hi = lo * 10 - 1
        total += (min(i, hi) - lo + 1) * d
        lo *= 10
        d += 1
    return total


def fq_off(r):
    """byte offset of read r (0-based) of the synthetic FASTQ"""
    return r * FQ_FIXED + digits_upto(r)


def fq_read_at(byte, n_reads):
    """index of the read containing `byte` (n_reads if past the end)"""
    lo, hi = 0, n_reads
    while lo < hi:
        mid = (lo + hi) // 2
        if fq_off(mid + 1) <= byte:
            lo = mid + 1
        else:
            hi = mid
    return lo


# ---------------------------------------------------------------------------------------------
# the reference (oracle/_ref) and the oracle (oracle/fxo.c): checkers and CPU baselines only
# ---------------------------------------------------------------------------------------------
def load_reference():
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(ref_dir) and any(f.startswith("pyfastx") and f.endswith(".so") for f in os.listdir(ref_dir)):
        if ref_dir not in sys.path:
            sys.path.insert(0, ref_dir)
        import pyfastx  # noqa: the unmodified reference, compiled by oracle/build_ref.sh
        return pyfastx
    return None


def reference_index_build(pyfastx_ref, path, data, kind="fasta"):
    """one index build on the reference CPU path; returns seconds"""
    if pyfastx_ref is not None:
        fxi = path + ".fxi"
        if os.path.exists(fxi):
            os.unlink(fxi)
        t0 = time.perf_counter()
        obj = pyfastx_ref.Fasta(path) if kind == "fasta" else pyfastx_ref.Fastq(path)
        dt = time.perf_counter() - t0
        del obj
        return dt
    from oracle import fxo
    t0 = time.perf_counter()
    (fxo.fasta_scan if kind == "fasta" else fxo.fastq_scan)(data)
    return time.perf_counter() - t0


def oracle_fasta_rows(host, rec_off, n_threads_):
    """all rows of a record-aligned FASTA buffer through oracle/fxo.c, chunked over threads (the C call drops the
    GIL).  rec_off = byte offsets of the records (n+1), relative to the buffer."""
    from oracle import fxo
    L = fxo.lib()
    n = rec_off.size - 1
    rows = np.zeros(n, dtype=fxo.FASTA_ROW)
    nchunk = max(1, min(n_threads_ * 4, n // 2000 + 1))
    bounds = [n * k // nchunk for k in range(nchunk + 1)]
    totals = [0] * nchunk

    def work(k):
        a, b = bounds[k], bounds[k + 1]
        if b <= a:
            return
        lo, hi = int(rec_off[a]), int(rec_off[b])
        part = host[lo:hi]
        tot, noh = C.c_int64(0), C.c_int(0)
        got = L.fxo_fasta_scan(part.ctypes.data, part.size, 0, rows[a:b].ctypes.data, b - a, C.byref(tot), C.byref(noh))
        assert got == b - a, "oracle found %d records in a chunk of %d" % (got, b - a)
        rows["boff"][a:b] += lo
        totals[k] = tot.value

    with ThreadPoolExecutor(n_threads_) as ex:
        list(ex.map(work, range(nchunk)))
    return rows, sum(totals)


def oracle_fastq_rows(host, first_read, n_reads, base, n_threads_):
    """all rows of a read-aligned FASTQ buffer (reads first_read.. of the synthetic file, buffer byte 0 = file
    offset `base`) through oracle/fxo.c, chunked over threads"""
    from oracle import fxo
    L = fxo.lib()
    rows = np.zeros(n_reads, dtype=fxo.FASTQ_ROW)
    nchunk = max(1, min(n_threads_ * 4, n_reads // 20000 + 1))
    bounds = [n_reads * k // nchunk for k in range(nchunk + 1)]
    sizes = [0] * nchunk

    def work(k):
        a, b = bounds[k], bounds[k + 1]
        if b <= a:
            return
        lo, hi = fq_off(first_read + a) - base, fq_off(first_read + b) - base
        part = host[lo:hi]
        size, nl = C.c_int64(0), C.c_int64(0)
        got = L.fxo_fastq_scan(part.ctypes.data, part.size, rows[a:b].ctypes.data, b - a, C.byref(size), C.byref(nl))
        assert got == b - a and nl.value == 4 * (b - a)
        rows["soff"][a:b] += lo + base
        rows["qoff"][a:b] += lo + base
        sizes[k] = size.value

    with ThreadPoolExecutor(n_threads_) as ex:
        list(ex.map(work, range(nchunk)))
    return rows, sum(sizes)


def oracle_extract_compare(host, exp_rows, rid, qs, qe, flags, out_host, off_host, n_threads_):
    """every query's bytes from oracle/fxo.c against the GPU output; returns the number of queries compared"""
    from oracle import fxo
    nq = rid.size
    nchunk = max(1, min(n_threads_ * 4, nq // 5000 + 1))
    bounds = [nq * k // nchunk for k in range(nchunk + 1)]
    bad = []

    def work(k):
        a, b = bounds[k], bounds[k + 1]
        if b <= a:
            return
        eo, eoff, _ = fxo.subseq_batch(host, exp_rows, rid[a:b], qs[a:b], qe[a:b], flags[a:b])
        lo, hi = int(off_host[a]), int(off_host[b])
        if hi - lo != eo.size or not np.array_equal(out_host[lo:hi], eo) or \
                not np.array_equal(off_host[a:b + 1] - lo, eoff):
            bad.append(k)

    with ThreadPoolExecutor(n_threads_) as ex:
        list(ex.map(work, range(nchunk)))
    assert not bad, "GPU extraction differs from the oracle in query chunks %s" % bad[:5]
    return nq


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref)
# ---------------------------------------------------------------------------------------------
def _synth_chunk(args):
    path, first, count, seed, off0 = args
    from pyfastx_b200 import synth
    lens = synth.fasta_lengths(first + count, seed)[first:]
    parts = []
    for k in range(count):
        i, L = first + k, int(lens[k])
        b = synth.bases(seed, i, L)
        nfull = L // 80
        parts.append(synth.fasta_header(i, L) + b"\n")
        if nfull:
            body = b[:nfull * 80].reshape(nfull, 80)
            parts.append(np.concatenate([body, np.full((nfull, 1), 10, np.uint8)], axis=1).tobytes())
        if L % 80:
            parts.append(b[nfull * 80:].tobytes() + b"\n")
    data = b"".join(parts)
    fd = os.open(path, os.O_WRONLY)
    try:
        os.pwrite(fd, data, off0)
    finally:
        os.close(fd)
    return len(data)


def write_synth_fasta(path, n_rec, seed):
    """the C2 file written to `path` by all host cores (numpy generator, byte-identical to the HBM generator)"""
    import multiprocessing as mp
    from pyfastx_b200 import synth
    lens = synth.fasta_lengths(n_rec, seed)
    off = np.zeros(n_rec + 1, dtype=np.int64)
    np.cumsum(synth.fasta_record_sizes(lens), out=off[1:])
    with open(path, "wb") as f:
        f.truncate(int(off[-1]))
    per = 2000
    tasks = [(path, a, min(per, n_rec - a), seed, int(off[a])) for a in range(0, n_rec, per)]
    procs = max(1, min(os.cpu_count() or 1, 96, len(tasks)))
    if procs == 1:
        for t in tasks:
            _synth_chunk(t)
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_synth_chunk, tasks, chunksize=1)
    return int(off[-1])


def c2_workload(n_rec, nbytes, n_gpus):
    return ("C2: %.2f GB synthetic plain FASTA per GPU (%d records x U[9000,11000] bp, 80-col, LF), index build"
            % (nbytes / 1e9, n_rec))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    pyfastx_ref = load_reference()
    n_rec = int(args.records)
    budget_s = float(args.ref_budget_s)
    path = os.path.join(shm_dir(), "fxg_bench_ref_%d.fa" % os.getpid())
    t0 = time.perf_counter()
    nbytes = write_synth_fasta(path, n_rec, SEED_FASTA)
    log("reference arm: wrote the full C2 file (%.2f GB, %d records) in %.1f s" % (nbytes / 1e9, n_rec, time.perf_counter() - t0))
    data = None
    if pyfastx_ref is None:
        data = np.fromfile(path, dtype=np.uint8)
    try:
        # probe on a prefix to decide whether K + W builds of the FULL file fit the time budget
        from pyfastx_b200 import synth
        lens = synth.fasta_lengths(n_rec, SEED_FASTA)
        off = np.zeros(n_rec + 1, dtype=np.int64)
        np.cumsum(synth.fasta_record_sizes(lens), out=off[1:])
        probe_rec = min(n_rec, 25000)
        ppath = path + ".probe"
        with open(path, "rb") as src, open(ppath, "wb") as dst:
            dst.write(src.read(int(off[probe_rec])))
        tp = reference_index_build(pyfastx_ref, ppath, None if data is None else data[:int(off[probe_rec])])
        for p in (ppath, ppath + ".fxi"):
            if os.path.exists(p):
                os.unlink(p)
        per_byte = tp / float(off[probe_rec])
        total_runs = args.steps + args.warmup
        use_rec = n_rec
        if per_byte * nbytes * total_runs > budget_s:
            want = budget_s / (per_byte * total_runs)
            use_rec = max(1000, int(np.searchsorted(off, want, side="right")) - 1)
            os.truncate(path, int(off[use_rec]))
            log("reference arm: %d builds of the full file would take %.0f s > %.0f s budget; sample = first %d records"
                % (total_runs, per_byte * nbytes * total_runs, budget_s, use_rec))
        use_bytes = int(off[use_rec])
        if data is not None:
            data = data[:use_bytes]
        for _ in range(args.warmup):
            reference_index_build(pyfastx_ref, path, data)
        times = [reference_index_build(pyfastx_ref, path, data) for _ in range(args.steps)]
    finally:
        for p in (path, path + ".fxi"):
            if os.path.exists(p):
                os.unlink(p)
    total = sum(times)
    gbs = use_bytes * args.steps / total / 1e9
    full = use_rec == n_rec
    line = {
        "impl": "reference", "metric": "index_build_GBps", "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": c2_workload(n_rec, nbytes, 1),
                   "sample": "the full file" if full else "first %d records (%.2f GB) of it, so that %d builds fit %.0f s"
                             % (use_rec, use_bytes / 1e9, total_runs, budget_s),
                   "api": "pyfastx.Fasta(path) incl. sqlite .fxi write" if pyfastx_ref else "oracle/fxo.c fasta_scan",
                   "file_in": "tmpfs, warm page cache"},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": 1,
                         "kind": "reference" if pyfastx_ref else "port",
                         "sample": "%d records / %.3f GB per step; the reference index build is single-threaded" % (use_rec, use_bytes / 1e9),
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
class Ctx:
    pass


def setup(args):
    import torch
    import torch.distributed as dist
    from pyfastx_b200 import _cabi, engine, shard
    c = Ctx()
    c.torch, c.dist = torch, dist
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    torch.cuda.set_device(c.local)
    if c.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", c.local))
    c.L = _cabi.lib()
    c.eng = engine.Engine(c.local)
    c.stream = torch.cuda.Stream()
    c.eng.set_stream(c.stream.cuda_stream)
    c.comm = shard.Comm(c.eng)                      # fxg_comm over NCCL (None handle when world == 1)
    c.peak, c.peak_src = measured_peaks()
    c.check = _cabi.check
    _cabi.check(c.L.fxg_profile_enable(c.eng.ctx, 1))
    c.dump = args.dump_outputs if c.rank == 0 else None
    c.dump_bytes = 0
    if c.dump:
        os.makedirs(c.dump, exist_ok=True)
    return c


def barrier(c):
    if c.world > 1:
        c.dist.barrier()
    c.torch.cuda.synchronize()


def allmax(c, v):
    t = c.torch.tensor([float(v)], dtype=c.torch.float64, device="cuda")
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return float(t.item())


def allsum(c, v):
    t = c.torch.tensor([int(v)], dtype=c.torch.int64, device="cuda")
    if c.world > 1:
        c.dist.all_reduce(t)
    return int(t.item())


def prof_ms(c, slot):
    ms = C.c_float()
    c.check(c.L.fxg_profile_last_ms(c.eng.ctx, slot, C.byref(ms)))
    return ms.value


def timed_scan(c, dfile, mode, base_offset, steps, warmup):
    """K sharded index builds of the resident range; -> dict of timings + last (d_rows, stats, infos)"""
    eng = c.eng
    for _ in range(warmup):
        d_rows, st, infos = eng.scan_sharded_dev(c.comm.handle, dfile, mode, base_offset)
    barrier(c)
    launches0 = c.L.fxg_ctx_launch_count(eng.ctx)
    ev0, ev1 = c.torch.cuda.Event(enable_timing=True), c.torch.cuda.Event(enable_timing=True)
    k_ms = {0: [], 1: [], 4: [], 5: []}
    ev0.record(c.stream)
    for _ in range(steps):
        d_rows, st, infos = eng.scan_sharded_dev(c.comm.handle, dfile, mode, base_offset)
        for slot in k_ms:
            k_ms[slot].append(prof_ms(c, slot))
    ev1.record(c.stream)
    barrier(c)
    launches = c.L.fxg_ctx_launch_count(eng.ctx) - launches0
    elapsed = allmax(c, ev0.elapsed_time(ev1))
    return {"elapsed_ms": elapsed, "launches": int(launches), "mark_ms": float(np.mean(k_ms[0])),
            "prefix_ms": float(np.mean(k_ms[4])), "rows_ms": float(np.mean(k_ms[5])),
            "finalize_ms": float(np.mean(k_ms[1])), "d_rows": d_rows, "st": st, "infos": infos}


def scan_roofline(c, t, file_bytes, n_rows, row_bytes, kernel):
    """SURVEY 8(d): (file bytes + row_bytes x rows) over the summed duration of ALL scan kernels"""
    all_ms = t["mark_ms"] + t["prefix_ms"] + t["rows_ms"] + t["finalize_ms"]
    alg = file_bytes + n_rows * row_bytes
    ach = alg / (all_ms * 1e-3) / 1e9
    mark_ach = file_bytes / (t["mark_ms"] * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "all scan kernels (mark + prefix + rows + finalize)", "achieved": ach, "peak": c.peak,
            "unit": "GB/s", "frac": ach / c.peak, "frac_of_nominal_8TBs": ach / 8000.0, "peak_source": c.peak_src,
            "algorithmic_bytes_per_launch": alg, "kernel_ms": all_ms,
            "mark_kernel": {"name": kernel, "ms": t["mark_ms"], "achieved": mark_ach, "frac": mark_ach / c.peak,
                            "algorithmic_bytes": file_bytes},
            "prefix_kernels_ms": t["prefix_ms"], "rows_kernels_ms": t["rows_ms"], "finalize_kernel_ms": t["finalize_ms"]}


# ---- C2 FASTA ------------------------------------------------------------------------------------------------------
def make_fasta_shard(c, per_rank):
    """this rank's byte range of ONE N x per_rank-record FASTA, cut at header lines found on the data"""
    from pyfastx_b200 import synth
    eng, L = c.eng, c.L
    n_all = per_rank * c.world
    lengths_all = synth.fasta_lengths(n_all, SEED_FASTA)
    off_all = np.zeros(n_all + 1, dtype=np.int64)
    np.cumsum(synth.fasta_record_sizes(lengths_all), out=off_all[1:])
    S = int(off_all[-1])
    p0, p1 = S * c.rank // c.world, S * (c.rank + 1) // c.world
    ra = max(0, int(np.searchsorted(off_all, p0, side="right")) - 1)            # record containing byte p0
    rb = min(n_all, int(np.searchsorted(off_all, p1, side="right")) + 1)        # one record past the one containing p1
    base = int(off_all[ra])
    with c.torch.cuda.stream(c.stream):
        tmp = eng.alloc_file(int(off_all[rb]) - base)
        d_len = eng.upload_rows(np.ascontiguousarray(lengths_all[ra:rb]))
        d_off = eng.upload_rows(np.ascontiguousarray(off_all[ra:rb + 1] - base))
        c.check(L.fxg_synth_fasta_dev(eng.ctx, SEED_FASTA, d_len.devptr, d_off.devptr, rb - ra, ra, 80, tmp.devptr))
        q0 = base + eng.split_point(tmp, p0 - base, want_header=True) if c.rank > 0 else 0
        q1 = base + eng.split_point(tmp, p1 - base, want_header=True) if c.rank < c.world - 1 else S
        if q0 == base and q1 == int(off_all[rb]):
            dfile = tmp
        else:
            dfile = eng.slice_file(tmp, q0 - base, q1 - base)
            eng.sync()
            tmp.free()
    r0, r1 = int(np.searchsorted(off_all, q0)), int(np.searchsorted(off_all, q1))
    assert off_all[r0] == q0 and off_all[r1] == q1, "split points are not header starts"
    info = {"S": S, "nominal": (p0, p1), "range": (q0, q1), "records": (r0, r1),
            "lengths": np.ascontiguousarray(lengths_all[r0:r1]), "rec_off": np.ascontiguousarray(off_all[r0:r1 + 1] - q0)}
    return dfile, info


def run_fasta(c, args, result):
    eng, L = c.eng, c.L
    per_rank = int(args.records)
    dfile, info = make_fasta_shard(c, per_rank)
    q0, q1 = info["range"]
    shard_bytes = q1 - q0
    log("rank %d: FASTA range [%d, %d) of %d (nominal [%d, %d)), %.3f GB, records %d..%d"
        % (c.rank, q0, q1, info["S"], info["nominal"][0], info["nominal"][1], shard_bytes / 1e9, *info["records"]))
    clocks = ClockSampler(c.local)
    clocks.start()
    t = timed_scan(c, dfile, 0, q0, args.steps, args.warmup)
    from pyfastx_b200 import engine
    if c.dump:
        dump_rows(c, "fasta_rows", t["d_rows"], t["st"], engine.FASTA_ROW)
    if args.dump_outputs:
        barrier(c)                                      # rank 0 dumped alone; the scans below are collective
    # keep the GPU busy for >= 1 s in total so that nvidia-smi sees the load (clock / throttle record).  Every scan is a
    # collective exchange, so every rank runs the same number of them, from the step time all ranks agree on.
    for _ in range(int(1200.0 * args.steps / t["elapsed_ms"]) + 1):
        eng.scan_sharded_dev(c.comm.handle, dfile, 0, q0)
    barrier(c)
    clk = clocks.stop()
    total_bytes = allsum(c, shard_bytes)
    st, infos = t["st"], t["infos"]
    n_rows = st["n_rows"]
    rows = np.zeros(n_rows, dtype=engine.FASTA_ROW)
    c.check(L.fxg_rows_download(eng.ctx, t["d_rows"], n_rows, 48, rows.ctypes.data))
    assert n_rows == info["records"][1] - info["records"][0], "row count differs from the generator's"
    assert np.array_equal(rows["slen"], info["lengths"]), "scan rows disagree with the generator's record lengths"
    assert int(infos["n_rows"].sum()) == per_rank * c.world and int(infos["bytes"].sum()) == info["S"]
    value = total_bytes * args.steps / (t["elapsed_ms"] * 1e-3) / 1e9
    result.update({
        "metric": "index_build_GBps", "value": value, "unit": "GB/s", "n_gpus": c.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t["elapsed_ms"] / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": c2_workload(per_rank, shard_bytes, c.world),
                   "file": "ONE %.2f GB file of %d records; rank i scans byte range i of %d, moved to the next header line "
                           "found on the data (fxg_split_point_dev)" % (info["S"] / 1e9, per_rank * c.world, c.world),
                   "step": "fxg_scan_sharded = fxg_scan_begin (mark + prefix) -> fxg_shard_exchange (ncclAllGather, "
                           "128 B per rank, in stream) -> fxg_scan_finish (rows); one host sync per step",
                   "parallelism": ("byte-range shards, 1 process/GPU, %d NCCL ranks" % c.world) if c.world > 1 else "1 GPU",
                   "l2": "inputs (10 GB per GPU) larger than L2 (126 MB); no flush needed",
                   "rows_per_gpu": int(n_rows)},
        "gpu_launches": t["launches"],
        "clocks": clk,
        "roofline": {**scan_roofline(c, t, shard_bytes, n_rows, 48, "mark_kernel<FASTA>"),
                     **ncu_traffic("scan_all_fasta", shard_bytes + 48 * n_rows)},
    })
    return dfile, info, rows, st


# ---- C3 extraction ---------------------------------------------------------------------------------------------------
def run_extract(c, args, dfile, info, rows, result, host_file):
    from pyfastx_b200 import _cabi, synth
    eng, L, torch = c.eng, c.L, c.torch
    n_rows = len(rows)
    q0 = info["range"][0]
    local_rows = rows.copy()
    local_rows["boff"] -= q0                                    # the resident range starts at device offset 0
    drows = eng.upload_rows(local_rows)
    nq = int(args.queries)
    out = {}
    for label, mixed in (("fixed_1kb", False), ("mixed_50_5000", True)):
        rid, qs, qe, minus = synth.random_queries(rows["slen"], nq, seed=SEED_QUERIES + c.rank + (1000 if mixed else 0),
                                                  window=1000, mixed=mixed)
        flags = np.where(minus, _cabi.X_REVERSE | _cabi.X_COMPLEMENT, 0).astype(np.int32)
        bases = int((qe - qs).sum())
        bpl = (rows["llen"] - rows["elen"])[rid]
        read_bytes = (qe - qs) + rows["elen"][rid].astype(np.int64) * (qe // bpl - qs // bpl)
        alg = int(read_bytes.sum()) + bases
        with torch.cuda.stream(c.stream):
            d_rid, d_s, d_e = (torch.from_numpy(x).cuda() for x in (rid, qs, qe))
            d_fl = torch.from_numpy(flags).cuda()
            d_ooff = torch.empty(nq + 1, dtype=torch.int64, device="cuda")
            d_out = torch.empty(bases + 64, dtype=torch.uint8, device="cuda")

            def step():
                c.check(L.fxg_extract_plan_dev(eng.ctx, d_s.data_ptr(), d_e.data_ptr(), nq, d_ooff.data_ptr(), None))
                c.check(L.fxg_extract_dev(eng.ctx, dfile.handle, drows.devptr, n_rows, d_rid.data_ptr(), d_s.data_ptr(),
                                          d_e.data_ptr(), d_fl.data_ptr(), nq, d_ooff.data_ptr(), d_out.data_ptr(), None))

            for _ in range(args.warmup):
                step()
            barrier(c)
            x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = L.fxg_ctx_launch_count(eng.ctx)
            gms = []
            x0.record(c.stream)
            for _ in range(args.steps):
                step()
                gms.append(prof_ms(c, 2))
            x1.record(c.stream)
            barrier(c)
            launches = L.fxg_ctx_launch_count(eng.ctx) - l0
            if c.dump:
                dump_extract(c, label, d_ooff, d_out)
        x_ms = allmax(c, x0.elapsed_time(x1))
        tot_bases = allsum(c, bases)
        g_ms = float(np.mean(gms))
        ach = alg / (g_ms * 1e-3) / 1e9
        rec = {"metric": "subseq_extract_Mbases_per_s", "value": tot_bases * args.steps / (x_ms * 1e-3) / 1e6,
               "unit": "Mbases/s", "ms_per_step": x_ms / args.steps, "queries_per_gpu": nq,
               "gpu_launches": int(launches),
               "roofline": {"bound": "hbm", "kernel": "extract_bulk_kernel", "achieved": ach, "peak": c.peak,
                            "unit": "GB/s", "frac": ach / c.peak, "frac_of_nominal_8TBs": ach / 8000.0,
                            "algorithmic_bytes_per_launch": alg, "kernel_ms": g_ms,
                            **ncu_traffic("extract_kernel_mixed" if mixed else "extract_kernel", alg)}}
        if mixed:
            out["mixed_length"] = rec
            del d_rid, d_s, d_e, d_fl, d_ooff, d_out
            continue
        out.update(rec)
        out["config"] = {"workload": "C3: %d random (record, start, end, strand) queries per GPU on its resident range, 1 kb "
                                     "windows, strand '-' (reverse-complement) with p=0.5; mixed_length = L ~ U[50, 5000]" % nq}
        # ---- e2e: host queries -> packed bytes on the host, through the C-ABI ----
        out_host, hp2 = pinned_array(bases + 64, np.uint8)
        q_pinned = []
        for arr in (rid, qs, qe):
            a, p = pinned_array(nq, np.int64); a[:] = arr; q_pinned.append((a, p))
        fl_p, hp3 = pinned_array(nq, np.int32); fl_p[:] = flags
        off_host, hp4 = pinned_array(nq + 1, np.int64)

        def e2e_extract():
            c.check(L.fxg_extract_host(eng.ctx, dfile.handle, drows.devptr, n_rows, q_pinned[0][0].ctypes.data,
                                       q_pinned[1][0].ctypes.data, q_pinned[2][0].ctypes.data, fl_p.ctypes.data, nq,
                                       off_host.ctypes.data, out_host.ctypes.data, out_host.size, None))

        e2e_extract()
        barrier(c)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_extract()
        torch.cuda.synchronize()
        e2e_x = allmax(c, time.perf_counter() - t0)
        out["e2e"] = {"value": tot_bases * args.steps / e2e_x / 1e6, "unit": "Mbases/s",
                      "h2d_bytes_per_step": nq * 28, "d2h_bytes_per_step": bases + (nq + 1) * 8, "steps": args.steps,
                      "api": "fxg_extract_host (pinned host queries -> packed bytes on host)"}
        # ---- parity: ALL queries, byte for byte, against oracle/fxo.c on the downloaded range ----
        if host_file is not None and not args.no_parity:
            t0 = time.perf_counter()
            n_cmp = oracle_extract_compare(host_file, local_rows, rid, qs, qe, flags, out_host, off_host, n_threads())
            out["parity"] = {"queries_compared_with_oracle": int(n_cmp), "of": nq, "bytes": bases,
                             "seconds": time.perf_counter() - t0}
        c.x_keep = (rid, qs, qe, minus, flags, out_host, off_host)      # out_host / off_host stay alive (pinned: hp2, hp4)
        for p in (hp3,) + tuple(p for _, p in q_pinned):
            L.fxg_host_free(p)
        c.x_pinned = (hp2, hp4)
        del d_rid, d_s, d_e, d_fl, d_ooff, d_out
    result["extract"] = out
    return drows, local_rows


# ---- e2e through the object API + CPU baselines (N = 1) ---------------------------------------------------------------
def run_e2e_and_cpu(c, args, info, rows, st, host_file, result):
    import pyfastx_b200
    from pyfastx_b200 import fxi
    n_rows = len(rows)
    shard_bytes = host_file.size
    path = os.path.join(shm_dir(), "fxg_bench_%d.fa" % os.getpid())
    t0 = time.perf_counter()
    host_file.tofile(path)
    log("wrote %s (%.2f GB) in %.1f s" % (path, shard_bytes / 1e9, time.perf_counter() - t0))
    pyfastx_ref = load_reference()
    try:
        # ---- the drop-in call: Fasta(path) = stage + scan + names + .fxi write ----
        times, parts = [], None
        for k in range(args.steps + 1):                       # first build is the warm-up
            if os.path.exists(path + ".fxi"):
                os.unlink(path + ".fxi")
            t0 = time.perf_counter()
            fa = pyfastx_b200.Fasta(path)
            dt = time.perf_counter() - t0
            if k:
                times.append(dt)
            if k == args.steps:
                assert len(fa) == n_rows and fa.size == int(st["total_len"])
                assert np.array_equal(fa._rows["boff"], rows["boff"] - info["range"][0])
                # the reference's per-object idiom through this package (a GPU round trip per query)
                sel = np.arange(0, min(20000, c.x_keep[0].size))
                rid, qs, qe, minus = (x[sel] for x in c.x_keep[:4])
                names = ["seq%d" % (info["records"][0] + int(i) + 1) for i in rid]
                qs_l, qe_l = [int(v) for v in qs], [int(v) for v in qe]
                for j in range(min(200, sel.size)):                  # untimed: the lazily built name table, the service kernel's
                    _ = fa[names[j]][qs_l[j]:qe_l[j]].seq              # first launch (module load) -- one-time costs of an open file
                t1 = time.perf_counter()
                got = []
                for j in range(sel.size):
                    sub = fa[names[j]][qs_l[j]:qe_l[j]]
                    got.append(sub.antisense if minus[j] else sub.seq)
                per_obj = time.perf_counter() - t1
                out_host, off_host = c.x_keep[5], c.x_keep[6]
                for j in range(sel.size):
                    want = out_host[off_host[j]:off_host[j + 1]].tobytes()
                    if got[j].encode() != want:
                        g = got[j].encode()
                        k = next((x for x in range(min(len(g), len(want))) if g[x] != want[x]), -1)
                        raise AssertionError("per-object getter differs from the batch: query %d (%s, %d:%d, minus=%s) lengths %d/%d, "
                                             "first difference at %d: %r vs %r" % (j, names[j], qs[j], qe[j], minus[j], len(g), len(want), k,
                                                                                 g[max(0, k - 8):k + 24], want[max(0, k - 8):k + 24]))
                result["extract"]["per_object_idiom"] = {
                    "api": "fa[name][s:e].seq / .antisense through pyfastx_b200 (one query per call: resident service kernel fed through "
                           "mapped host memory, no launch / stream sync per query; FXG_ONE_SERVICE=0 = launch + sync per query)",
                    "queries_per_s": sel.size / per_obj, "Mbases_per_s": float((qe - qs).sum()) / per_obj / 1e6,
                    "queries": int(sel.size)}
                t1 = time.perf_counter()
                many = fa.fetch_many(names, qs + 1, qe, ["-" if m else "+" for m in minus])
                result["extract"]["batched_api"] = {"api": "Fasta.fetch_many (names resolved by the native hash table)",
                                                    "queries_per_s": sel.size / (time.perf_counter() - t1)}
                assert [m.encode() for m in many] == [out_host[off_host[j]:off_host[j + 1]].tobytes() for j in range(sel.size)]
            fxi_bytes = os.path.getsize(path + ".fxi")
            del fa
        best = float(np.median(times))                          # median of the measured builds (the first one is the warm-up)
        result["e2e"] = {"value": shard_bytes / best / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(shard_bytes),
                         "d2h_bytes_per_step": int(n_rows * 48 + int(rows["nlen"].sum())), "steps": args.steps,
                         "seconds_per_build": best,
                         "api": "pyfastx_b200.Fasta(path): tmpfs file -> pinned chunks -> HBM -> scan -> rows + names on host "
                                "-> .fxi written (native bulk writer, %d B)" % fxi_bytes}
        # ---- .fxi writer on its own ----
        fa_names = fxi.PackedNames.from_list([b"seq%d" % (info["records"][0] + i + 1) for i in range(n_rows)])
        wp = os.path.join(shm_dir(), "fxg_bench_w_%d.fxi" % os.getpid())
        t0 = time.perf_counter()
        con = fxi.write_fasta_index_packed(wp, rows, fa_names.blob, fa_names.off, int(st["total_len"]))
        tw = time.perf_counter() - t0
        con.close()
        result["fxi_write"] = {"seconds": tw, "rows": int(n_rows), "rows_per_s": n_rows / tw, "file_bytes": os.path.getsize(wp),
                               "api": "fxg_fxi_write_fasta: SQLite pages written directly, UNIQUE name index by parallel sample sort"}
        os.unlink(wp)
        if args.no_cpu_baseline:
            return
        # ---- CPU baseline: the compiled reference on a bounded sample of the same file ----
        n_rec = min(n_rows, int(args.ref_sample_records))
        nb = int(info["rec_off"][n_rec])
        spath = os.path.join(shm_dir(), "fxg_bench_cpu_%d.fa" % os.getpid())
        host_file[:nb].tofile(spath)
        try:
            best = min(reference_index_build(pyfastx_ref, spath, host_file[:nb]) for _ in range(3))
            result["cpu_baseline"] = {
                "value": nb / best / 1e9, "unit": "GB/s", "cores": 1, "kind": "reference" if pyfastx_ref else "port",
                "sample": "first %d records (%.3f GB) of the same file, tmpfs, best of 3; pyfastx.Fasta(path) incl. .fxi write; "
                          "the reference index build is single-threaded" % (n_rec, nb / 1e9),
                "host_cores_available": os.cpu_count()}
            if pyfastx_ref is not None:
                rid, qs, qe, minus, flags, out_host, off_host = c.x_keep
                sel = np.nonzero(rid < n_rec)[0][:100000]
                names = ["seq%d" % (info["records"][0] + i + 1) for i in range(n_rec)]
                fa = pyfastx_ref.Fasta(spath)
                t0 = time.perf_counter()
                got = []
                for i in sel:
                    sub = fa[names[rid[i]]][int(qs[i]):int(qe[i])]
                    got.append(sub.antisense if minus[i] else sub.seq)
                cpu_x = time.perf_counter() - t0
                for k, i in enumerate(sel):
                    assert out_host[off_host[i]:off_host[i + 1]].tobytes().decode() == got[k], "extract mismatch q=%d" % i
                del fa
                bsel = int((qe[sel] - qs[sel]).sum())
                result["extract"]["cpu_baseline"] = {
                    "value": bsel / cpu_x / 1e6, "unit": "Mbases/s", "cores": 1, "kind": "reference",
                    "sample": "%d of the same queries via fa[name][s:e].seq/.antisense" % sel.size,
                    "queries_per_s": sel.size / cpu_x, "parity_checked_queries_vs_reference": int(sel.size)}
                # all host cores: the documented multiprocessing pattern, one Fasta per worker (docs/advance.rst:4-40)
                result["extract"]["cpu_baseline_all_cores"] = all_cores_extract(spath, names, rid, qs, qe, minus, n_rec)
        finally:
            for p in (spath, spath + ".fxi"):
                if os.path.exists(p):
                    os.unlink(p)
    finally:
        for p in (path, path + ".fxi"):
            if os.path.exists(p):
                os.unlink(p)


def run_e2e_sharded(c, args, dfile, info, rows, st, host_file, result):
    """N > 1: the drop-in multi-GPU build of ONE file on tmpfs through the public API shard.build_index_sharded -- every rank
    stages ITS byte range of the file (pread -> pinned ring -> its own PCIe link), split-phase scan with the mailbox
    exchange, rows + names gathered to rank 0, which writes the `.fxi`.  Timed from a barrier to a barrier, max over ranks."""
    from pyfastx_b200 import shard
    q0, q1 = info["range"]
    S = info["S"]
    port = os.environ.get("MASTER_PORT", "0")
    path = os.path.join(shm_dir(), "fxg_bench_shared_%s.fa" % port)
    if host_file is None:
        host_file, hp = pinned_array(q1 - q0, np.uint8)
        c.check(c.L.fxg_file_download(c.eng.ctx, dfile.handle, 0, host_file.ctypes.data, q1 - q0))
    else:
        hp = None
    if c.rank == 0:
        with open(path, "wb") as fh:
            fh.truncate(S)
    barrier(c)
    t0 = time.perf_counter()
    fd = os.open(path, os.O_WRONLY)
    try:
        mv, off, step = memoryview(host_file), 0, 256 << 20
        while off < q1 - q0:
            off += os.pwrite(fd, mv[off:off + step], q0 + off)
    finally:
        os.close(fd)
    barrier(c)
    if c.rank == 0:
        log("wrote %s (%.2f GB, %d ranks in parallel) in %.1f s" % (path, S / 1e9, c.world, time.perf_counter() - t0))
    try:
        times = []
        res = None
        for k in range(args.steps + 1):                       # first build is the warm-up
            if c.rank == 0 and os.path.exists(path + ".fxi"):
                os.unlink(path + ".fxi")
            barrier(c)
            t0 = time.perf_counter()
            res = shard.build_index_sharded(path, "fasta", engine=c.eng, comm=c.comm, index_file=path + ".fxi")
            barrier(c)
            dt = allmax(c, time.perf_counter() - t0)
            if k:
                times.append(dt)
        assert np.array_equal(res["rows"]["boff"], rows["boff"]) and np.array_equal(res["rows"]["slen"], rows["slen"])
        names_bytes = 0
        if c.rank == 0:
            assert len(res["all_rows"]) == args.records * c.world or len(res["all_rows"]) == int(args.records) * c.world
            names_bytes = int(sum(int(p[1][-1]) for p in res["name_parts"]))
            fxi_bytes = os.path.getsize(path + ".fxi")
        best = float(np.median(times))                          # median of the measured builds (the first one is the warm-up)
        if c.rank == 0:
            result["e2e"] = {"value": S / best / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(S),
                             "d2h_bytes_per_step": int(int(args.records) * c.world * 48 + names_bytes), "steps": args.steps,
                             "seconds_per_build": best,
                             "api": "pyfastx_b200.shard.build_index_sharded(path, 'fasta') on %d ranks: ONE tmpfs file of %.2f GB -> every rank "
                                    "stages its byte range (pread -> pinned ring -> HBM) -> sharded scan -> rows + names gathered to rank 0 "
                                    "-> .fxi written (native bulk writer, %d B)" % (c.world, S / 1e9, fxi_bytes)}
    finally:
        barrier(c)
        if c.rank == 0:
            for p in (path, path + ".fxi"):
                if os.path.exists(p):
                    os.unlink(p)
        if hp is not None:
            c.L.fxg_host_free(hp)


def _ref_worker(args):
    spath, names, rid, qs, qe, minus = args
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    import pyfastx
    fa = pyfastx.Fasta(spath)
    t0 = time.perf_counter()
    n = 0
    for i in range(rid.size):
        sub = fa[names[rid[i]]][int(qs[i]):int(qe[i])]
        n += len(sub.antisense if minus[i] else sub.seq)
    return n, time.perf_counter() - t0


def all_cores_extract(spath, names, rid, qs, qe, minus, n_rec):
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    sel = np.nonzero(rid < n_rec)[0]
    per = 20000
    sel = sel[:cores * per]
    chunks = np.array_split(sel, cores)
    tasks = [(spath, names, rid[ch], qs[ch], qe[ch], minus[ch]) for ch in chunks if ch.size]
    t0 = time.perf_counter()
    # spawn, not fork: this process holds a CUDA context and pinned memory, which a forked child must not touch
    with mp.get_context("spawn").Pool(len(tasks)) as pool:
        res = pool.map(_ref_worker, tasks, chunksize=1)
    wall = time.perf_counter() - t0
    bases = sum(r[0] for r in res)
    work = max(r[1] for r in res)
    return {"value": bases / work / 1e6, "unit": "Mbases/s", "cores": len(tasks), "kind": "reference",
            "sample": "%d queries split over %d workers, one pyfastx.Fasta per worker, index pre-built; slowest worker's "
                      "loop time (pool start-up excluded: %.2f s wall)" % (sel.size, len(tasks), wall)}


# ---- C4 FASTQ, strong scaling ----------------------------------------------------------------------------------------
def run_fastq(c, args, result):
    from pyfastx_b200 import engine
    eng, L, torch = c.eng, c.L, c.torch
    R = int(args.fastq_reads)
    S = fq_off(R)
    p0, p1 = S * c.rank // c.world, S * (c.rank + 1) // c.world
    ra = fq_read_at(p0, R)
    rb = min(R, fq_read_at(p1, R) + 1)
    base = fq_off(ra)
    with torch.cuda.stream(c.stream):
        tmp = eng.alloc_file(fq_off(rb) - base)
        c.check(L.fxg_synth_fastq_dev(eng.ctx, SEED_FASTQ, rb - ra, ra, 150, None, tmp.devptr))
        q0 = base + eng.split_point(tmp, p0 - base, want_header=False) if c.rank > 0 else 0
        q1 = base + eng.split_point(tmp, p1 - base, want_header=False) if c.rank < c.world - 1 else S
        if q0 == base and q1 == fq_off(rb):
            dfile = tmp
        else:
            dfile = eng.slice_file(tmp, q0 - base, q1 - base)
            eng.sync()
            tmp.free()
    shard_bytes = q1 - q0
    log("rank %d: FASTQ range [%d, %d) of %d (nominal [%d, %d)), %.3f GB" % (c.rank, q0, q1, S, p0, p1, shard_bytes / 1e9))
    t = timed_scan(c, dfile, 1, q0, args.steps, args.warmup)
    if c.dump:
        dump_rows(c, "fastq_rows", t["d_rows"], t["st"], engine.FASTQ_ROW)
    st, infos = t["st"], t["infos"]
    n_rows = st["n_rows"]
    total_reads = allsum(c, n_rows)
    assert total_reads == R and int(infos["n_lines"].sum()) == 4 * R and int(infos["bytes"].sum()) == S
    value = S * args.steps / (t["elapsed_ms"] * 1e-3) / 1e9
    rec = {"metric": "fastq_index_build_GBps", "value": value, "unit": "GB/s", "n_gpus": c.world, "scaling": "strong",
           "ms_per_step": t["elapsed_ms"] / args.steps, "reads": R, "file_gb": S / 1e9,
           "config": {"workload": "C4: ONE %.2f GB synthetic FASTQ (%d reads x 150 bp + qual); rank i scans byte range i of %d, "
                                  "cut at line starts found on the data; line phase from the ncclAllGather, boundary reads "
                                  "completed on the device" % (S / 1e9, R, c.world),
                      "range_of_rank0": [int(q0), int(q1)], "rows_rank0": int(n_rows), "first_line_rank0": int(st["lead_lines"])},
           "gpu_launches": t["launches"],
           "roofline": {**scan_roofline(c, t, shard_bytes, n_rows, 32, "mark_kernel<FASTQ>"),
                        **ncu_traffic("scan_all_fastq", shard_bytes + 32 * n_rows)}}
    # ---- parity: ALL rows of this rank against oracle/fxo.c on the downloaded range ----
    if not args.no_parity:
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 1 << 62
        rows = np.zeros(n_rows, dtype=engine.FASTQ_ROW)
        c.check(L.fxg_rows_download(eng.ctx, t["d_rows"], n_rows, 32, rows.ctypes.data))
        # reads owned by this rank: name line at or after q0
        first_read = fq_read_at(q0, R) + (0 if fq_off(fq_read_at(q0, R)) == q0 else 1)
        if avail > shard_bytes * 1.3 + (12 << 30):
            t0 = time.perf_counter()
            # download the bytes of the owned reads (they may end in the next rank's range: take them from the generator
            # range this rank produced) -- the owned reads all START in [q0, q1)
            lo, hi = fq_off(first_read), fq_off(first_read + n_rows)
            host = np.empty(min(hi, q1) - lo, dtype=np.uint8)
            c.check(L.fxg_file_download(eng.ctx, dfile.handle, lo - q0, host.ctypes.data, host.size))
            n_full = n_rows if hi <= q1 else n_rows - 1            # the last owned read may continue in the next range
            exp, size = oracle_fastq_rows(host, first_read, n_full, lo, n_threads())
            for fld in ("soff", "qoff", "rlen", "dlen", "nlen"):
                assert np.array_equal(exp[fld], rows[fld][:n_full]), "GPU FASTQ rows differ from the oracle in " + fld
            if n_full < n_rows:                                     # the stitched boundary read: analytic layout
                r = first_read + n_full
                d = len(str(r + 1))
                assert (int(rows["soff"][-1]), int(rows["qoff"][-1]), int(rows["rlen"][-1]), int(rows["dlen"][-1]), int(rows["nlen"][-1])) == \
                    (fq_off(r) + 5 + d + 12, fq_off(r) + 5 + d + 12 + 153, 150, 5 + d + 11, 4 + d)
            rec["parity"] = {"rows_compared_with_oracle": int(n_full), "of": int(n_rows), "stitched_boundary_rows_checked": int(n_rows - n_full),
                             "seconds": time.perf_counter() - t0}
            # the compiled reference on the first 3M reads of the file (rank 0)
            pyfastx_ref = load_reference()
            if c.rank == 0 and pyfastx_ref is not None and args.ref_fastq_reads > 0:
                k = int(min(args.ref_fastq_reads, n_full))
                fpath = os.path.join(shm_dir(), "fxg_bench_%d.fq" % os.getpid())
                host[:fq_off(k) - lo].tofile(fpath)
                try:
                    t0 = time.perf_counter()
                    fq = pyfastx_ref.Fastq(fpath)
                    dt = time.perf_counter() - t0
                    assert len(fq) == k
                    import sqlite3
                    con = sqlite3.connect(fpath + ".fxi")
                    got = np.array(con.execute("SELECT dlen,rlen,soff,qoff,length(name) FROM read ORDER BY ID").fetchall(), dtype=np.int64)
                    con.close()
                    for j, fld in enumerate(("dlen", "rlen", "soff", "qoff", "nlen")):
                        assert np.array_equal(got[:, j], rows[fld][:k].astype(np.int64)), "GPU FASTQ rows differ from the reference in " + fld
                    rec["parity"]["rows_compared_with_reference"] = k
                    rec["cpu_baseline"] = {"value": (fq_off(k) - lo) / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "reference",
                                           "sample": "pyfastx.Fastq(path) on the first %d reads (%.2f GB), tmpfs, incl. .fxi write" % (k, (fq_off(k) - lo) / 1e9)}
                    del fq
                finally:
                    for p in (fpath, fpath + ".fxi"):
                        if os.path.exists(p):
                            os.unlink(p)
            del host
            # the step after the scan: names gathered on the GPU + the native .fxi writer on all rows of the file
            if c.world == 1 and not args.skip_e2e:
                from pyfastx_b200 import fxi
                t0 = time.perf_counter()
                blob, noff = eng.gather_ranges(dfile, rows["soff"] - rows["dlen"] - q0, rows["nlen"].astype(np.int64))
                t1 = time.perf_counter()
                wp = os.path.join(shm_dir(), "fxg_bench_%d.fq.fxi" % os.getpid())
                con = fxi.write_fastq_index_packed(wp, rows, blob, noff, 4 * R, int(st["total_len"]))
                t2 = time.perf_counter()
                nchk = con.execute("SELECT COUNT(1) FROM read").fetchone()[0]
                probe = con.execute("SELECT ID FROM read WHERE name=?", ("read%d" % (R // 2 + 1),)).fetchall()
                con.close()
                assert nchk == n_rows and probe == [(R // 2 + 1,)]
                rec["fxi_write"] = {"rows": int(n_rows), "names_gather_seconds": t1 - t0, "write_seconds": t2 - t1,
                                    "rows_per_s": n_rows / (t2 - t1), "file_bytes": os.path.getsize(wp),
                                    "api": "fxg_fxi_write_fastq (read table + UNIQUE readidx, SQLite pages written directly)"}
                os.unlink(wp)
                del blob, noff
        else:
            rec["parity"] = {"skipped": "host memory: %.0f GB available" % (avail / 1e9)}
    result["fastq"] = rec
    dfile.free()


# ---- C5 BGZF ------------------------------------------------------------------------------------------------------------
BGZF_BLOCK = 0xff00
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_compress(host, level, workers):
    """the C2 bytes as BGZF, by all host threads (fxg_bgzf_compress_host: zlib deflate per 0xff00-byte block)"""
    from pyfastx_b200 import _cabi
    L = _cabi.lib()
    out, n = C.c_void_p(), C.c_int64(0)
    _cabi.check(L.fxg_bgzf_compress_host(host.ctypes.data, host.size, level, C.byref(out), C.byref(n)))
    z = np.frombuffer((C.c_uint8 * n.value).from_address(out.value), dtype=np.uint8).copy()
    L.fxg_free_host(out)
    return z


def run_bgzf(c, args, dfile_plain, rows_plain, drows, host_file, result):
    from pyfastx_b200 import _cabi, synth
    eng, L = c.eng, c.L
    total = host_file.size
    t0 = time.perf_counter()
    z = bgzf_compress(host_file, args.bgzf_level, n_threads(128))
    t_comp = time.perf_counter() - t0
    zpin, zp = pinned_array(z.size, np.uint8)
    zpin[:] = z
    del z
    best, f = None, None
    for k in range(args.steps + 1):                         # first build is the warm-up
        if f is not None:
            f.free()
        t0 = time.perf_counter()
        nm, tot = C.c_int64(0), C.c_int64(0)
        c.check(L.fxg_bgzf_members_host(zp.value, zpin.size, None, None, 0, C.byref(nm), C.byref(tot)))
        t_walk = time.perf_counter() - t0
        t1 = time.perf_counter()
        f = eng.stage_bgzf(zpin)
        eng.sync()
        t_inf = time.perf_counter() - t1
        inflate_ms = prof_ms(c, 2)
        t2 = time.perf_counter()
        rows, st = eng.fasta_scan(f)
        t_scan = time.perf_counter() - t2
        recd = {"walk_s": t_walk, "stage_plus_inflate_s": t_inf, "inflate_kernel_ms": inflate_ms, "scan_s": t_scan,
                "total_s": time.perf_counter() - t0}
        if k and (best is None or recd["total_s"] < best["total_s"]):
            best = recd
    assert tot.value == total and f.size == total
    # parity: inflated bytes == the input bytes; rows == the plain-file rows; fetches == the plain-file fetches
    back = f.download()
    assert np.array_equal(back, host_file), "inflated bytes differ from the input"
    del back
    for fld in ("boff", "blen", "slen", "llen", "dlen", "nlen", "elen", "norm"):
        assert np.array_equal(rows[fld], rows_plain[fld]), fld
    nq = int(args.bgzf_queries)
    rid, s, e, minus = synth.random_queries(rows_plain["slen"], nq, seed=124)
    flags = np.where(minus, _cabi.X_REVERSE | _cabi.X_COMPLEMENT, 0).astype(np.int32)
    t0 = time.perf_counter()
    a, oa, _ = eng.extract(f, drows, rid, s, e, flags)
    t_fetch = time.perf_counter() - t0
    n_cmp = 0
    if not args.no_parity:
        n_cmp = oracle_extract_compare(host_file, rows_plain, rid, s, e, flags, a, oa, n_threads())
    result["bgzf"] = {
        "metric": "bgzf_index_build_GBps_uncompressed", "value": total / best["total_s"] / 1e9, "unit": "GB/s", "n_gpus": 1,
        "config": {"workload": "C5: %.2f GB FASTA (C2 content) as BGZF level %d, %d members, %.2f GB compressed: member walk "
                               "(host) + H2D + GPU inflate + index scan, from pinned host memory" % (
                                   total / 1e9, args.bgzf_level, nm.value, zpin.size / 1e9)},
        "members": nm.value, "compressed_gb": zpin.size / 1e9, "uncompressed_gb": total / 1e9,
        "inflate_kernel_ms": best["inflate_kernel_ms"], "inflate_GBps_output": total / (best["inflate_kernel_ms"] * 1e-3) / 1e9,
        "timing_s": best, "steps": args.steps, "host_compress_s": t_comp,
        "fetch": {"queries": nq, "seconds_host_to_host": t_fetch, "Mbases_per_s": float((e - s).sum()) / t_fetch / 1e6},
        "parity": {"inflated_bytes_equal_input": int(total), "rows_equal_plain_scan": int(len(rows)),
                   "fetches_compared_with_oracle": int(n_cmp)}}
    f.free()
    L.fxg_host_free(zp)


def run_b200(args):
    c = setup(args)
    result = {}
    dfile, info, rows, st = run_fasta(c, args, result)
    shard_bytes = info["range"][1] - info["range"][0]
    host_file = hp1 = None
    single = c.world == 1
    if not args.no_parity or single:
        host_file, hp1 = pinned_array(shard_bytes, np.uint8)
        c.check(c.L.fxg_file_download(c.eng.ctx, dfile.handle, 0, host_file.ctypes.data, shard_bytes))
    # ---- parity: ALL rows x all columns + stat against oracle/fxo.c ----
    if not args.no_parity:
        t0 = time.perf_counter()
        exp_rows, exp_total = oracle_fasta_rows(host_file, info["rec_off"], n_threads())
        exp_rows["boff"] += info["range"][0]
        for fld in ("boff", "blen", "slen", "llen", "dlen", "nlen", "elen", "norm"):
            assert np.array_equal(exp_rows[fld], rows[fld]), "GPU rows differ from the oracle in " + fld
        assert exp_total == st["total_len"]
        result["parity"] = {"rows_compared_with_oracle": int(len(rows)), "columns": 8, "stat_total_len": int(exp_total),
                            "seconds": time.perf_counter() - t0}
        result["parity_checked_rows"] = int(len(rows))
    drows, local_rows = run_extract(c, args, dfile, info, rows, result, host_file)
    if single and not args.skip_e2e:
        run_e2e_and_cpu(c, args, info, rows, st, host_file, result)
    elif not args.skip_e2e:
        run_e2e_sharded(c, args, dfile, info, rows, st, host_file, result)
    else:
        result["e2e"] = None
    if single and not args.skip_bgzf:
        try:
            run_bgzf(c, args, dfile, local_rows, drows, host_file, result)
        except AssertionError:
            raise
        except Exception as ex:                                   # resources (host memory, time): report, keep the line
            result["bgzf"] = {"error": repr(ex)}
    drows.free()
    dfile.free()
    if hp1 is not None:
        host_file = None
        c.L.fxg_host_free(hp1)
    if getattr(c, "x_pinned", None) is not None:
        c.x_keep = None
        for p in c.x_pinned:
            c.L.fxg_host_free(p)
    if not args.skip_fastq:
        run_fastq(c, args, result)
    p2p = bool(c.world > 1 and c.comm.handle and c.L.fxg_comm_uses_p2p(c.comm.handle))
    result["comm"] = {"nranks": c.world,
                      "collective": ("none (single rank: device copy)" if c.world == 1 else
                                     "fxg_shard_exchange over peer-memory mailboxes: one kernel per rank stores its 128-byte block into every "
                                     "rank's HBM over NVLink/NVSwitch (CUDA IPC mappings) and waits for the peers' flags; NCCL only at set-up"
                                     if p2p else "ncclAllGather via fxg_shard_exchange (libfxg.so, dlopen libnccl.so.2)"),
                      "p2p_mailboxes": p2p}
    if c.rank == 0:
        print(json.dumps(result), flush=True)
    if c.world > 1:
        c.dist.barrier()
        c.comm.close()
        c.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--records", type=float, default=1e6, help="FASTA records per GPU (C2: 1M records = 10.15 GB)")
    ap.add_argument("--queries", type=float, default=10e6, help="C3 queries per GPU")
    ap.add_argument("--fastq-reads", type=float, default=126e6, help="C4: reads of the ONE FASTQ file (126M = 41.5 GB)")
    ap.add_argument("--bgzf-queries", type=float, default=1e6)
    ap.add_argument("--bgzf-level", type=int, default=6)
    ap.add_argument("--ref-sample-records", type=float, default=50000,
                    help="bounded CPU sample for cpu_baseline: 50k records = 0.51 GB")
    ap.add_argument("--ref-fastq-reads", type=float, default=3e6, help="C4 reads checked against the compiled reference")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="reference arm: time budget for K + W builds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--skip-fastq", action="store_true")
    ap.add_argument("--skip-bgzf", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (fixed samples of large outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs: the b200 arm only")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
