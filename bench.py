#!/usr/bin/env python
"""bench.py -- the similarity-search hot path on synthetic corpora (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is ONE single-query top-100 scan of the whole corpus (configs[1]: 10M x 256-byte rows
per GPU, k = 100).  With N > 1 the corpus is row-sharded (10M rows on every GPU, N x 10M in
total: weak scaling), every rank scans its shard, and the k records per shard are exchanged and
merged by ONE kernel over NVLink peer memory (post, signal, wait, merge; an NCCL all-gather +
merge kernel is the fallback).  The 2.56 GB per GPU exceed the 126 MB L2, so no L2 flush is
needed between steps.

value    = corpus GB/s scanned by the whole job with the query already in HBM (queries/s beside it)
e2e      = the same through the host-buffer API: pinned host query -> H2D -> search -> D2H result
batched  = configs[2]: a batch of 1024 queries through the tensor-core path, with its own roofline
           against the int8 ceiling measured in the same run (pbx_int8_peak)
northstar= (N >= 2) configs[3]: 1B x 256 bytes in total, row-sharded over the N GPUs, single + batched
c1_sqlite= (N = 1) configs[0]: 100k x 256 in SQLite, top-50: verbatim SQL + UDF on one host thread, the
           bare loop, and the GPU path through the Engine mirror including hydration
--impl reference = the CPU restatement of the reference's scan (oracle/, the reference itself
           needs a Rust toolchain this image does not have) on all host cores.
--dump-outputs DIR = after the timed steps, write what the last step of each timed path returned as DIR/<name>.npy
           (single_*: the headline step, e2e_*: the host-buffer step, batched_*: the last batch; see result_arrays).
           The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 42
NQ = 64          # distinct queries cycled through (SURVEY.md 8d, C2)
PLANT_IDS = (3_000_000_003, 3_000_000_005)      # two identical planted rows (one on the first, one on the last shard)
NORTHSTAR_ROWS = 1_000_000_000
SWEEP_ROWS = 100_000_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows-per-gpu", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batched", action="store_true", help="skip the 1024-query tensor-core measurement")
    ap.add_argument("--no-northstar", action="store_true", help="skip the 1B-row section of a multi-GPU run")
    ap.add_argument("--northstar-rows", type=int, default=NORTHSTAR_ROWS)
    ap.add_argument("--no-c1", action="store_true", help="skip the configs[0] SQLite comparison of a 1-GPU run")
    ap.add_argument("--sweep", action="store_true", help="run the configs[4] d x k sweep at N = 1 too (always on for N >= 2)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the configs[4] sweep of a multi-GPU run")
    ap.add_argument("--sweep-rows", type=int, default=SWEEP_ROWS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step of each path as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU arm (oracle): bounded sample of the same workload
# ---------------------------------------------------------------------------------------------
def cpu_scan(rows: int, dim: int, k: int, queries: np.ndarray, threads: int, steps: int, warmup: int):
    """Times oracle.topk (the restatement of src/engine.rs:572-588 + :375-383 as a bare loop) over the
    first `rows` rows of the synthetic corpus.  Returns (seconds per step, checksum of ids)."""
    from oracle import oracle
    from pixelbox_b200 import synth
    corpus = np.empty((rows, dim), np.uint8)
    for r0 in range(0, rows, 1 << 20):                  # C generator of the oracle library, chunked
        r1 = min(rows, r0 + (1 << 20))
        corpus[r0:r1] = oracle.synth_rows(SEED, r0, r1 - r0, dim)
    assert np.array_equal(corpus[:8], synth.synth_rows(SEED, 0, 8, dim))
    ids = np.arange(1, rows + 1, dtype=np.int64)
    for i in range(warmup):
        oracle.topk(corpus, ids, queries[i % len(queries)], k, 1e3, threads=threads)
    t0 = time.perf_counter()
    chk = 0
    for i in range(steps):
        o_ids, _, _, _ = oracle.topk(corpus, ids, queries[i % len(queries)], k, 1e3, threads=threads)
        chk ^= int(o_ids.sum())
    return (time.perf_counter() - t0) / steps, chk


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle
    from pixelbox_b200 import synth
    threads = oracle.max_threads()
    dim, k = args.dim, args.k
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    # ~0.77 us per row per thread at d=256.  The sample is sized so that the WHOLE run (warm-up + steps, as asked for)
    # stays near 60 s of wall clock: a step is a bounded sample of the workload, never a clamped step count.
    per_row_s = 0.77e-6 * dim / 256.0 / threads
    rows = args.cpu_rows or int(min(args.rows_per_gpu, max(50_000, 60.0 / ((steps + warmup) * per_row_s))))
    queries = synth.synth_queries(7, NQ, dim, args.rows_per_gpu * args.gpus, SEED)
    sec, _ = cpu_scan(rows, dim, k, queries, threads, steps, warmup)
    gbs = rows * dim / sec / 1e9
    sample = (f"first {rows} of {args.rows_per_gpu * args.gpus} rows x {dim} B, {steps} single-query top-{k} scans, "
              f"oracle/pbx_oracle.c (C restatement of src/engine.rs:572-588 + :375-383; upstream is 1 thread, "
              f"this arm splits rows over {threads} pthreads)")
    cfg = workload_config(args)
    cfg["cpu_sample_rows"] = rows
    cfg["value_is"] = "rate over the CPU sample (rows of the sample x dim / time per scan of the sample), not a full-corpus scan"
    line = {
        "impl": "reference", "metric": "corpus_GB_per_s_scanned", "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "queries_per_sec_on_sample": 1.0 / sec,
        "queries_per_sec_full_corpus_extrapolated": gbs * 1e9 / (args.rows_per_gpu * args.gpus * dim),
        "config": cfg,
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


TRAFFIC_CSV = "r2_scan_kernel_ncu_full_summary.csv"      # ncu --set full of the scan kernel, this round's build


def ncu_traffic(rows: int, dim: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the scan kernel per launch, from the committed ncu --set full
    capture of this workload (profiles/); None for any other workload (ncu cannot run inside a timed bench)."""
    if rows != 10_000_000 or dim != 256:
        return None
    for name in (TRAFFIC_CSV, "r1i_scan_kernel_ncu_full_summary.csv"):
        path = os.path.join(ROOT, "profiles", name)
        try:
            import csv
            with open(path) as f:
                r = list(csv.reader(f))
            hdr, units, first = r[0], r[1], r[2]
            rd = float(first[hdr.index("dram__bytes_read.sum")]) * (1e9 if units[hdr.index("dram__bytes_read.sum")].startswith("G") else 1e6)
            wr = float(first[hdr.index("dram__bytes_write.sum")]) * (1e9 if units[hdr.index("dram__bytes_write.sum")].startswith("G") else 1e6)
            return rd + wr, name
        except Exception:
            continue
    return None


def workload_config(args):
    return {"workload": f"{args.rows_per_gpu // 1_000_000}M x {args.dim}-byte corpus per GPU, single query top-{args.k} "
                        f"(BASELINE configs[1]); row-sharded x{args.gpus}",
            "rows_per_gpu": args.rows_per_gpu, "rows_total": args.rows_per_gpu * args.gpus, "dim": args.dim, "k": args.k,
            "max_dist": 1e3, "distinct_queries": NQ, "parallelism": f"row-shard x{args.gpus}",
            "planted_rows": "2 identical rows (ids 3000000003 / 3000000005) beyond the synthetic ones, on the first and the last shard",
            "l2": "corpus shard (2.56 GB) >> 126 MB L2, no flush between steps"}


# ---------------------------------------------------------------------------------------------
# parity of what was timed, at full size: returned rows + a random stripe of every shard + the planted tie
# ---------------------------------------------------------------------------------------------
def planted_row(dim: int) -> np.ndarray:
    return np.random.default_rng(99).integers(0, 256, size=dim, dtype=np.uint8)


def rows_of(ids, dim: int, rows_total: int):
    """Regenerates the corpus rows of the given image ids on the host (synthetic: id = row + 1; planted: fixed bytes)."""
    from pixelbox_b200 import synth
    out = np.empty((len(ids), dim), np.uint8)
    pr = planted_row(dim)
    for j, i in enumerate(ids):
        out[j] = pr if int(i) in PLANT_IDS else synth.synth_rows(SEED, int(i) - 1, 1, dim)[0]
    return out


def completeness_check(ids, dist, query, k, dim, world, rows_per_shard, stripe_rows=200_000, seed=5):
    """(1) the returned rows, re-ranked by the oracle, come back in the same order with the same distance bits;
    (2) in a random stripe of EVERY shard (regenerated on the host) no row beats the k-th hit without being in the
    answer -- so nothing better was missed on any shard; returns (ok, detail)."""
    from oracle import oracle
    ids = np.asarray(ids, np.int64)
    dist = np.asarray(dist, np.float32)
    back = rows_of(ids, dim, world * rows_per_shard)
    o = oracle.topk(back, ids, query, k, 1e3)
    ok = list(o[0]) == list(ids) and np.array_equal(o[1].view(np.uint32), dist.view(np.uint32))
    if not ok:
        return False, "returned rows re-rank differently"
    full = len(ids) == k
    kth = (float(dist[-1]), int(ids[-1])) if full else (float("inf"), np.iinfo(np.int64).max)
    have = set(int(i) for i in ids)
    rng = np.random.default_rng(seed)
    checked = 0
    for s in range(world):
        n_s = min(stripe_rows, rows_per_shard)
        off = int(rng.integers(0, rows_per_shard - n_s + 1))
        first = s * rows_per_shard + off
        stripe = np.empty((n_s, dim), np.uint8)
        for r0 in range(0, n_s, 1 << 20):
            r1 = min(n_s, r0 + (1 << 20))
            stripe[r0:r1] = oracle.synth_rows(SEED, first + r0, r1 - r0, dim)
        s_ids = np.arange(first + 1, first + n_s + 1, dtype=np.int64)
        t_ids, t_dist, _, _ = oracle.topk(stripe, s_ids, query, k, 1e3, threads=oracle.max_threads())
        for i, dd in zip(t_ids, t_dist):
            if (float(dd), int(i)) < kth and int(i) not in have:
                return False, f"row {int(i)} of shard {s} (dist {float(dd)}) beats the k-th hit and is missing"
        checked += n_s
    return True, f"returned rows + {checked} stripe rows over {world} shard(s)"


def planted_check(res_ids, res_dist):
    """The query is the planted row: both copies must lead the list, equal distance bits, lower image_id first."""
    ok = (len(res_ids) >= 2 and int(res_ids[0]) == PLANT_IDS[0] and int(res_ids[1]) == PLANT_IDS[1]
          and np.float32(res_dist[0]).view(np.uint32) == np.float32(res_dist[1]).view(np.uint32))
    return bool(ok)


def result_arrays(name, ids, dist, dot, norm2, counts):
    """--dump-outputs: [nq][k] results as a caller receives them and the [nq] counts.  Entries past a query's count are 0;
    image ids and the int32 terms are stored as float64, which holds them exactly."""
    counts = np.asarray(counts, np.int64).reshape(-1)
    valid = np.arange(np.shape(ids)[-1])[None, :] < counts[:, None]
    out = {f"{name}_count": counts.astype(np.float64)}
    for field, v, t in (("image_id", ids, np.float64), ("dist", dist, np.float32), ("dot", dot, np.float64), ("norm2", norm2, np.float64)):
        out[f"{name}_{field}"] = np.where(valid, np.asarray(v).reshape(len(counts), -1), 0).astype(t)
    return out


def hit_arrays(name, hits, counts):
    """result_arrays of pbx_hit records (bytes or HIT_DTYPE) as the device-resident API returns them."""
    from pixelbox_b200 import _native as nat
    h = np.ascontiguousarray(hits).view(nat.HIT_DTYPE).reshape(len(counts), -1)
    return result_arrays(name, h["image_id"], h["dist"], h["dot"], h["norm2"], counts)


# ---------------------------------------------------------------------------------------------
# configs[0]: 100k x 256 in SQLite, top-50 (the only configuration the reference itself runs end to end)
# ---------------------------------------------------------------------------------------------
def c1_sqlite(device: int):
    """b_sql_ms: the reference's verbatim similarity SQL (src/engine.rs:375-382, LIMIT 50) with the oracle as the
    cosine_distance UDF, one thread; b_loop_ms: the bare scan loop, one thread; gpu_e2e_ms: Engine mirror
    (query_by_image_hash_from_image: pbx_search + hydration of the rows from SQLite).  Identical top-50."""
    import sqlite3
    from oracle import oracle
    from tests import sqlite_oracle
    from pixelbox_b200 import synth
    from pixelbox_b200.engine import Engine, IndexedImage
    n, dim, k = 100_000, 256, 50
    rows = oracle.synth_rows(1, 0, n, dim)
    ids = np.arange(1, n + 1, dtype=np.int64)
    fd, path = tempfile.mkstemp(suffix=".sqlite")
    os.close(fd)
    os.unlink(path)
    try:
        conn = sqlite_oracle.make_db(path, ids, rows)
        conn.close()
        conn = sqlite3.connect(path)
        sqlite_oracle.register(conn)
        q = rows[12344].tobytes()                                   # right-click "find similar" on image 12345
        sqlite_oracle.query(conn, q, 1e3, k)
        t0 = time.perf_counter()
        want = sqlite_oracle.query(conn, q, 1e3, k)
        b_sql = time.perf_counter() - t0
        conn.close()
        oracle.topk(rows, ids, rows[12344], k, 1e3, threads=1)
        t0 = time.perf_counter()
        o = oracle.topk(rows, ids, rows[12344], k, 1e3, threads=1)
        b_loop = time.perf_counter() - t0
        eng = Engine.open(path, device=device)
        img = IndexedImage(visual_hash=q)
        stderr, sys.stderr = sys.stderr, open(os.devnull, "w")      # the mirror prints the reference's timing line
        try:
            eng.query_by_image_hash_from_image(img)
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                eng.query_by_image_hash_from_image(img)
                ts.append(time.perf_counter() - t0)
            # LIMIT 100 upstream: the first 50 of the mirror's list are the top-50
            got = [(r.id, r.distance_from_query) for r in eng.get_query_results()][:k]
            # search alone (no hydration), through the same corpus
            t0 = time.perf_counter()
            for _ in range(20):
                eng.corpus.search(np.frombuffer(q, np.uint8), k, 1e3)
            gpu_search = (time.perf_counter() - t0) / 20
        finally:
            sys.stderr.close()
            sys.stderr = stderr
            eng.close()
        same = [i for i, _ in got] == [i for i, _ in want] and [float(np.float32(d)) for _, d in got] == [float(np.float32(d)) for _, d in want]
        same = same and list(o[0]) == [i for i, _ in want]
        return {"workload": "100k x 256-byte semantic_hashes table in SQLite, one query (row 12345's hash), top-50 (BASELINE configs[0])",
                "b_sql_ms": b_sql * 1e3, "b_sql": "verbatim SQL of src/engine.rs:375-382 with LIMIT 50, UDF = oracle, Python sqlite3 "
                                                  f"(SQLite {sqlite3.sqlite_version}), 1 thread",
                "b_loop_ms": b_loop * 1e3, "b_loop": "oracle.topk bare loop, 1 thread",
                "gpu_e2e_ms": float(np.median(ts)) * 1e3, "gpu_e2e": "Engine.query_by_image_hash_from_image: pbx_search (LIMIT 100) + hydration of "
                                                                     "100 rows from SQLite",
                "gpu_search_ms": gpu_search * 1e3, "speedup_e2e_vs_b_sql": b_sql / float(np.median(ts)), "parity_check": "ok" if same else "MISMATCH"}
    finally:
        for suffix in ("", "-wal", "-shm"):
            try:
                os.unlink(path + suffix)
            except OSError:
                pass


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes
    import torch
    import torch.distributed as dist
    from pixelbox_b200 import _native as nat
    from pixelbox_b200 import synth
    from pixelbox_b200.corpus import Corpus
    from pixelbox_b200.shard import ShardedCorpus

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if rank == 0:
            sys.stderr.write(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run\n")
        if world == 1 and args.gpus > 1:
            return 2
    L = nat.lib()                                 # fails loudly if the CUDA library is missing
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: pixelbox_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dim, k = args.dim, args.k
    stream = torch.cuda.Stream()
    peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def make_corpus(rows, dim=args.dim):
        """Row-sharded synthetic corpus of `rows` rows per GPU + the two planted identical rows."""
        if world > 1:
            sc = ShardedCorpus(dim, capacity_hint=rows + 1024, device=local_rank, use_peer_exchange=os.environ.get("PBX_NO_PEER_EXCHANGE") is None)
            sc.fill_synthetic(rows, SEED)
            corpus = sc.local
        else:
            sc = None
            corpus = Corpus(dim, capacity_hint=rows + 1024, device=local_rank)
            corpus.fill_synthetic(rows, SEED, 0)
        pr = planted_row(dim).reshape(1, dim)
        if rank == 0:
            corpus.append(np.array([PLANT_IDS[1]], np.int64), pr)
        if rank == world - 1:
            corpus.append(np.array([PLANT_IDS[0]], np.int64), pr)
        return sc, corpus

    def searcher(sc, corpus, dq, d_hits, d_cnt):
        def step_device(q, nq=1):
            """Returns (hits, counts): on one GPU the whole buffers, in which query q has slot q; sharded, this call's."""
            if sc is None:
                corpus.search_device(dq.data_ptr() + q * dim, nq, k, 1e3, d_hits.data_ptr() + q * k * 24, d_cnt.data_ptr() + 4 * q, stream.cuda_stream)
                return d_hits, d_cnt
            return sc.search_device(dq[q:q + nq].reshape(-1), nq, k, 1e3)
        return step_device

    def time_batch(step, nqb, reps):
        with torch.cuda.stream(stream):
            for _ in range(2):
                step()
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record(stream)
            out = None
            for _ in range(reps):
                out = step()
            b1.record(stream)
            barrier()
        return allmax([b0.elapsed_time(b1) / reps])[0], out

    # =========================================================================================
    # configs[1]: 10M x 256 per GPU, single query (the headline)
    # =========================================================================================
    rows = args.rows_per_gpu
    total_rows = rows * world
    queries = synth.synth_queries(7, NQ, dim, total_rows, SEED)
    queries[NQ - 1] = planted_row(dim)                       # the last query IS the planted row
    sc, corpus = make_corpus(rows)
    dq = torch.from_numpy(queries).cuda()
    d_hits = torch.zeros(NQ * k * 24, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(NQ, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    step_device = searcher(sc, corpus, dq, d_hits, d_cnt)

    def step_e2e(i):
        q = queries[i % NQ]
        if sc is None:
            return corpus.search(q, k, 1e3)[0]
        return sc.search(q, k, 1e3)[0]

    launches_per_step = 3 + (1 if world > 1 else 0)   # prep+seed, scan, finalize (+ exchange/merge); the exact pass is device-launched on demand
    warm = max(args.warmup, 3)
    with torch.cuda.stream(stream):
        for i in range(warm):
            step_device(i % NQ)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(args.steps):
            out = step_device(i % NQ)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        dump = {}
        if args.dump_outputs and rank == 0:
            slot = (args.steps - 1) % NQ if sc is None else 0
            dump.update(hit_arrays("single", out[0][slot * k * 24:(slot + 1) * k * 24].cpu().numpy(), out[1][slot:slot + 1].cpu().numpy()))
        # ---- e2e: host buffers through the public API --------------------------------------------
        for i in range(3):
            step_e2e(i)
        barrier()
        t0 = time.perf_counter()
        last = None
        for i in range(args.steps):
            last = step_e2e(i)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        barrier()
        if args.dump_outputs and rank == 0:
            dump.update(result_arrays("e2e", last.ids, last.dist, last.dot, last.norm2, [len(last.ids)]))
        clocks = sampler.stop() if rank == 0 else None
    ms, e2e_ms = allmax([ms, e2e_s * 1e3])

    # ---- dominant kernel: per-launch duration of the scan, CUDA events on its own stream ---------
    scan_ms = []
    corpus.set_profiling(True)
    for i in range(min(args.steps, 50)):
        corpus.search(queries[i % NQ], k, 1e3)
        scan_ms.append(corpus.stats().last_scan_ms)
    corpus.set_profiling(False)
    scan_ms = float(np.mean(scan_ms))
    st = corpus.stats()

    # ---- parity of what was timed: completeness at full size + the planted cross-shard tie --------
    last_q = (args.steps - 1) % NQ
    tie = step_e2e(NQ - 1)
    check = "skipped"
    if rank == 0:
        okc, detail = completeness_check(last.ids, last.dist, queries[last_q], k, dim, world, rows)
        okt = planted_check(tie.ids, tie.dist)
        check = f"ok ({detail}; planted tie across shards ordered by image_id)" if okc and okt else f"MISMATCH ({detail}; planted tie ok={okt})"

    # =========================================================================================
    # configs[2]: a batch of 1024 queries through the tensor-core path
    # =========================================================================================
    batched = None
    nqb = 1024
    bq = synth.synth_queries(43, nqb, dim, total_rows, SEED)
    if dim % 32 == 0 and dim <= 1024 and not args.no_batched:
        d_bq = torch.from_numpy(bq).cuda()
        d_bh = torch.zeros(nqb * k * 24, dtype=torch.uint8, device="cuda")
        d_bc = torch.zeros(nqb, dtype=torch.int32, device="cuda")

        def batch_step():
            if sc is None:
                corpus.search_device(d_bq.data_ptr(), nqb, k, 1e3, d_bh.data_ptr(), d_bc.data_ptr(), stream.cuda_stream)
                return d_bh, d_bc
            return sc.search_device(d_bq, nqb, k, 1e3)          # every shard contracts its rows against all queries, then the exchange

        bms, (out_b, out_bc) = time_batch(batch_step, nqb, 10)
        bh = out_b.cpu().numpy().view(nat.HIT_DTYPE).reshape(nqb, k)
        if args.dump_outputs and rank == 0:
            dump.update(hit_arrays("batched", bh, out_bc.cpu().numpy()))
        tops = 2.0 * total_rows * nqb * dim / (bms * 1e-3) / 1e12
        peak_tops = ctypes.c_double(0.0)
        nat.check(L.pbx_int8_peak(local_rank, ctypes.byref(peak_tops)))
        bcheck = "skipped"
        if rank == 0:
            okb, det = True, ""
            for qi in (0, 511, 1023):
                o1, det = completeness_check(bh[qi]["image_id"], bh[qi]["dist"], bq[qi], k, dim, world, rows, stripe_rows=100_000, seed=qi)
                okb &= o1
            bcheck = f"ok (3 queries: {det})" if okb else f"MISMATCH ({det})"
        batched = {"workload": f"{rows // 1_000_000}M x {dim}-byte corpus per GPU x{world}, batch of {nqb} queries top-{k} (BASELINE configs[2])",
                   "ms_per_batch": bms, "queries_per_sec": nqb / (bms * 1e-3), "int8_tops": tops,
                   "roofline": {"bound": "tensor", "kernel": "batch_mma_kernel<2,false> (tcgen05.mma.cta_group::2.kind::i8, TMA, TMEM, fused top-k)",
                                "achieved": tops, "peak": peak_tops.value * world, "unit": "TOP/s (dense int8)", "frac": tops / (peak_tops.value * world),
                                "peak_source": "measured in this run: pbx_int8_peak (the kernel's MMA shape, operands resident in shared memory, "
                                               "accumulators never read; burst)",
                                "frac_of_nominal": tops / (4500.0 * world), "peak_nominal": 4500.0 * world,
                                "algorithmic_ops_per_batch": 2.0 * total_rows * nqb * dim, "whole_batch": "prep + seed pass + main pass + finalize",
                                "tensor_pipe_pct": "profiles/ (ncu sm__pipe_tensor_cycles_active of the main pass)"},
                   "parity_check": bcheck}

    # =========================================================================================
    # configs[3] (N >= 2): 1B x 256 bytes in total, row-sharded over the N GPUs
    # =========================================================================================
    northstar = None
    if world > 1 and not args.no_northstar:
        d_bq = d_bh = d_bc = None
        sc.close()
        del sc, corpus
        torch.cuda.empty_cache()
        barrier()
        ns_rows = args.northstar_rows // world
        ns_total = ns_rows * world
        sc, corpus = make_corpus(ns_rows)
        nsq = synth.synth_queries(11, 8, dim, ns_total, SEED)
        nsq[7] = planted_row(dim)
        d_nq = torch.from_numpy(nsq).cuda()
        ns_steps = 20

        def ns_step(i):
            return sc.search_device(d_nq[i % 8], 1, k, 1e3)

        with torch.cuda.stream(stream):
            for i in range(3):
                ns_step(i)
            barrier()
            n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0.record(stream)
            for i in range(ns_steps):
                ns_step(i)
            n1.record(stream)
            barrier()
        ns_ms = allmax([n0.elapsed_time(n1) / ns_steps])[0]
        for i in range(3):                                   # the host-buffer path's own first-call set-up stays outside
            sc.search(nsq[i % 8], k, 1e3)
        barrier()
        t0 = time.perf_counter()
        for i in range(16):
            res_ns = sc.search(nsq[i % 8], k, 1e3)[0]
        ns_e2e = allmax([(time.perf_counter() - t0) / 16 * 1e3])[0]
        res_q0 = sc.search(nsq[0], k, 1e3)[0]
        ns_check = "skipped"
        if rank == 0:
            okc, detail = completeness_check(res_q0.ids, res_q0.dist, nsq[0], k, dim, world, ns_rows)
            okt = planted_check(res_ns.ids, res_ns.dist)                    # the last of the 8 queries is the planted row
            ns_check = f"ok ({detail}; planted tie across shards ordered by image_id)" if okc and okt else f"MISMATCH ({detail}; planted tie ok={okt})"
        ns_batched = None
        if not args.no_batched:
            nbq = synth.synth_queries(47, nqb, dim, ns_total, SEED)
            d_nbq = torch.from_numpy(nbq).cuda()
            nb_ms, out_nb = time_batch(lambda: sc.search_device(d_nbq, nqb, k, 1e3)[0], nqb, 3)
            nbh = out_nb.cpu().numpy().view(nat.HIT_DTYPE).reshape(nqb, k)
            nb_check = "skipped"
            if rank == 0:
                okb, det = completeness_check(nbh[5]["image_id"], nbh[5]["dist"], nbq[5], k, dim, world, ns_rows, stripe_rows=100_000, seed=3)
                nb_check = f"ok (1 query: {det})" if okb else f"MISMATCH ({det})"
            nb_tops = 2.0 * ns_total * nqb * dim / (nb_ms * 1e-3) / 1e12
            ns_batched = {"ms_per_batch": nb_ms, "queries_per_sec": nqb / (nb_ms * 1e-3), "int8_tops": nb_tops,
                          "frac_of_nominal_int8_peak": nb_tops / (4500.0 * world), "parity_check": nb_check}
        ns_gbs = ns_total * dim / (ns_ms * 1e-3) / 1e9
        northstar = {"workload": f"{ns_total} x {dim}-byte corpus row-sharded over {world} B200 ({ns_rows} rows = {ns_rows * dim / 1e9:.1f} GB per GPU), "
                                 f"single query top-{k} and a batch of {nqb} (BASELINE configs[3])",
                     "queries_per_sec": 1e3 / ns_ms, "ms_per_query": ns_ms, "aggregate_GB_per_s": ns_gbs,
                     "frac_of_measured_hbm_peak": ns_gbs / (peak * world), "frac_of_nominal_8TBps": ns_gbs / (8000.0 * world),
                     "e2e_ms_per_query": ns_e2e, "e2e_queries_per_sec": 1e3 / ns_e2e, "steps": ns_steps,
                     "target": ">= 200 queries/s on 8 GPUs at >= 80 % of aggregate HBM bandwidth, results identical to the reference",
                     "parity_check": ns_check, "batched": ns_batched}
        sc.close()

    # =========================================================================================
    # configs[4]: 100M rows in total x d in {64, 256, 1024} x k in {10, 100, 1000}, row-sharded over the N GPUs
    # =========================================================================================
    sweep = None
    if (world > 1 or args.sweep) and not args.no_sweep:
        d_bq = d_bh = d_bc = None
        if world > 1 and northstar is None:
            sc.close()
        if world == 1:
            corpus.close()
        torch.cuda.empty_cache()
        barrier()
        sw_rows = args.sweep_rows // world
        sw_total = sw_rows * world
        cells = []
        for sd in (64, 256, 1024):
            s_sc, s_corpus = make_corpus(sw_rows, sd)
            sq = synth.synth_queries(13, 8, sd, sw_total, SEED)
            sbq = synth.synth_queries(17, nqb, sd, sw_total, SEED)
            d_sq, d_sbq = torch.from_numpy(sq).cuda(), torch.from_numpy(sbq).cuda()
            for sk in (10, 100, 1000):
                d_sh = torch.zeros(nqb * sk * 24, dtype=torch.uint8, device="cuda")
                d_scn = torch.zeros(nqb, dtype=torch.int32, device="cuda")

                def sw_step(q, nq, src):
                    if s_sc is None:
                        s_corpus.search_device(src.data_ptr() + q * sd, nq, sk, 1e3, d_sh.data_ptr(), d_scn.data_ptr(), stream.cuda_stream)
                        return d_sh, d_scn
                    return s_sc.search_device(src[q:q + nq].reshape(-1), nq, sk, 1e3)

                it = [0]

                def one():
                    it[0] += 1
                    return sw_step(it[0] % 8, 1, d_sq)

                s_ms, _ = time_batch(one, 1, 20)
                with torch.cuda.stream(stream):
                    h1, c1 = sw_step(0, 1, d_sq)
                    torch.cuda.synchronize()
                r1 = h1.cpu().numpy()[:sk * 24].view(nat.HIT_DTYPE)[:int(c1.cpu()[0])]
                b_ms, (hb, cb) = time_batch(lambda: sw_step(0, nqb, d_sbq), nqb, 2)
                rb = hb.cpu().numpy()[:nqb * sk * 24].view(nat.HIT_DTYPE).reshape(nqb, sk)[3][:int(cb.cpu()[3])]
                cell_check = "skipped"
                if rank == 0:
                    ok1, det1 = completeness_check(r1["image_id"], r1["dist"], sq[0], sk, sd, world, sw_rows, stripe_rows=50_000, seed=sk)
                    ok2, det2 = completeness_check(rb["image_id"], rb["dist"], sbq[3], sk, sd, world, sw_rows, stripe_rows=50_000, seed=sk + 1)
                    cell_check = "ok" if ok1 and ok2 else f"MISMATCH (single: {det1}; batched: {det2})"
                gbs = sw_total * sd / (s_ms * 1e-3) / 1e9
                cells.append({"dim": sd, "k": sk, "ms_per_query": s_ms, "queries_per_sec": 1e3 / s_ms, "aggregate_GB_per_s": gbs,
                              "frac_of_measured_hbm_peak": gbs / (peak * world), "batch1024_ms": b_ms,
                              "batch1024_queries_per_sec": nqb / (b_ms * 1e-3),
                              "batch1024_int8_tops": 2.0 * sw_total * nqb * sd / (b_ms * 1e-3) / 1e12, "parity_check": cell_check})
                d_sh = d_scn = None
            if s_sc is not None:
                s_sc.close()
            else:
                s_corpus.close()
            d_sq = d_sbq = None
            torch.cuda.empty_cache()
            barrier()
        sweep = {"workload": f"{sw_total} rows row-sharded over {world} B200 ({sw_rows} per GPU), d x k grid, single query (20 steps, 8 distinct "
                             f"queries) and a batch of {nqb} (BASELINE configs[4])",
                 "parity_check": "per cell: one single query and one query of the batch: returned rows re-ranked by the oracle + a 50k-row "
                                 "stripe of every shard",
                 "cells": cells}

    if rank == 0:
        ms_step = ms / args.steps
        bytes_step = total_rows * dim
        value = bytes_step / (ms_step * 1e-3) / 1e9
        e2e_step = e2e_ms / args.steps
        achieved = rows * dim / (scan_ms * 1e-3) / 1e9
        traffic = ncu_traffic(rows, dim)
        line = {
            "metric": "corpus_GB_per_s_scanned", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8 x s16 -> int32 (IDP.2A), f32 replay on candidates", "data": "synthetic",
            "queries_per_sec": 1e3 / ms_step,
            "config": workload_config(args),
            "e2e": {"value": bytes_step / (e2e_step * 1e-3) / 1e9, "unit": "GB/s", "queries_per_sec": 1e3 / e2e_step,
                    "ms_per_query": e2e_step, "h2d_bytes_per_step": dim, "d2h_bytes_per_step": k * 24 + 4,
                    "api": "pbx_search (C ABI, host buffers)" if world == 1 else "ShardedCorpus.search (host buffers; exchange as in 'exchange')"},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "hbm", "kernel": "scan_kernel<16,1,false,3>" if dim == 256 else "scan_kernel", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic[0] if traffic else None,
                         "traffic_source": (f"profiles/{traffic[1]} (committed ncu --set full capture of this kernel on this workload, bytes per "
                                            "launch; ncu cannot run inside the timed bench)") if traffic else None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": rows * dim, "launch_ms": scan_ms,
                         "share_of_step": scan_ms / ms_step},
            "clocks": clocks,
            "exact_passes": int(st.exact_passes), "scan_grid": int(st.scan_grid), "parity_check": check,
            "exchange": None if world == 1 else ("one kernel over NVLink peer memory (post + signal + wait + merge)"
                                                 if os.environ.get("PBX_NO_PEER_EXCHANGE") is None else "NCCL all-gather + merge kernel"),
        }
        if batched is not None:
            line["batched"] = batched
        if northstar is not None:
            line["northstar"] = northstar
        if sweep is not None:
            line["sweep"] = sweep
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        if world == 1:
            # free the 10M-row corpus before the small-table comparison and the CPU baseline
            corpus.close()
            if not args.no_c1:
                try:
                    line["c1_sqlite"] = c1_sqlite(local_rank)
                except Exception as e:                      # never lose the headline line to the side measurement
                    line["c1_sqlite"] = {"error": repr(e)}
            if not args.no_cpu_baseline:
                from oracle import oracle
                cpu_rows = args.cpu_rows or min(rows, 2_000_000 * 256 // dim)
                cpu_steps = 8
                sec, _ = cpu_scan(cpu_rows, dim, k, queries, 1, cpu_steps, 1)
                line["cpu_baseline"] = {
                    "value": cpu_rows * dim / sec / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
                    "queries_per_sec_full_corpus_extrapolated": 1.0 / (sec * rows / cpu_rows),
                    "host_cores_available": oracle.max_threads(),
                    "sample": f"first {cpu_rows} of {rows} rows x {dim} B, {cpu_steps} single-query top-{k} scans, 1 thread "
                              f"(the reference scans inside one SQLite statement on one thread), oracle/pbx_oracle.c"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
