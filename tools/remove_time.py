"""Cost of pbx_corpus_remove on a 10M x 256 synthetic shard, and search times before / after a 1 % removal.
    python tools/remove_time.py [--rows 10000000] [--dim 256]

For m in {1, 1k, 100k, 1M} random ids: the host-clock time of the synchronous call (median of 3, the shard refilled
before each), then one more call under torch.profiler split by kernel: mark (remove_mark_kernel), rank
(remove_count / remove_scan / remove_place), move (remove_move_kernel), block metadata (block_meta_kernel); the rest of
the call (host sort of the request, its upload, launches, the one mid-call synchronisation) is reported as `host_other`.
Prints the card name and power limit first; one JSON line per measurement.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pixelbox_b200 import synth  # noqa: E402
from pixelbox_b200.corpus import Corpus  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # noqa: BLE001
        out = f"unavailable ({e})"
    return out


def stage(name):
    for key, part in (("remove_mark_kernel", "mark"), ("remove_count_kernel", "rank"), ("remove_scan_kernel", "rank"),
                      ("remove_place_kernel", "rank"), ("remove_move_kernel", "move"), ("block_meta_kernel", "block_meta")):
        if key in name:
            return part
    return None


def timed_remove(c, ids):
    t0 = time.perf_counter()
    removed = c.remove(ids)
    return (time.perf_counter() - t0) * 1e3, removed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=256)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    n, d, seed = args.rows, args.dim, 42
    print(json.dumps({"card": card(), "rows": n, "dim": d}), flush=True)
    rng = np.random.default_rng(1)
    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed)
        c.remove([-1])                           # warm-up: first launches load the module
        for m in (1, 1000, 100_000, 1_000_000):
            ids = rng.choice(np.arange(1, n + 1), m, replace=False).astype(np.int64)
            calls = []
            for _ in range(3):
                c.fill_synthetic(n, seed)
                ms, removed = timed_remove(c, ids)
                assert removed == m
                calls.append(ms)
            c.fill_synthetic(n, seed)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                ms_prof, _ = timed_remove(c, ids)
            parts = {"mark": 0.0, "rank": 0.0, "move": 0.0, "block_meta": 0.0}
            for ev in prof.key_averages():
                s = stage(ev.key)
                if s:
                    us = getattr(ev, "self_device_time_total", None)
                    parts[s] += (us if us is not None else ev.self_cuda_time_total) / 1e3
            device_ms = sum(parts.values())
            print(json.dumps({"m": m, "call_ms_median": round(float(np.median(calls)), 3), "calls_ms": [round(x, 3) for x in calls],
                              "profiled_call_ms": round(ms_prof, 3), **{k + "_ms": round(v, 4) for k, v in parts.items()},
                              "device_kernels_ms": round(device_ms, 4),
                              "host_other_ms": round(float(np.median(calls)) - device_ms, 3)}), flush=True)

        # search before / after removing 1 % of the rows
        c.fill_synthetic(n, seed)
        queries = synth.synth_queries(3, 1024, d, n, seed)

        def search_times():
            c.search(queries[0], 100)
            c.search(queries, 100)
            single = []
            for q in queries[:64]:
                t0 = time.perf_counter()
                c.search(q, 100)
                single.append((time.perf_counter() - t0) * 1e3)
            batch = []
            for _ in range(5):
                t0 = time.perf_counter()
                c.search(queries, 100)
                batch.append((time.perf_counter() - t0) * 1e3)
            return round(float(np.median(single)), 4), round(float(np.median(batch)), 3)

        s0, b0 = search_times()
        gone = rng.choice(np.arange(1, n + 1), n // 100, replace=False).astype(np.int64)
        ms, removed = timed_remove(c, gone)
        s1, b1 = search_times()
        print(json.dumps({"search": "k=100", "single_query_ms_median_before": s0, "single_query_ms_median_after": s1,
                          "batch1024_ms_median_before": b0, "batch1024_ms_median_after": b1,
                          "removed": removed, "remove_call_ms": round(ms, 3)}), flush=True)


if __name__ == "__main__":
    main()
