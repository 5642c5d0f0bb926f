"""Cost of filtered searches (pbx_search_device_filtered) on a 10M x 256 synthetic shard (ids = row + 1).
    python tools/filter_time.py [--rows 10000000] [--dim 256] [--singles 400] [--batches 6] [--out FILE]

Workloads: device-resident single queries (k = 100, enqueued back to back on one stream, timed with CUDA events over
blocks of 50 after a warm-up) and batches of 1024 queries (the tensor-core path, CUDA events per batch).  Filters:
none, include 50 %, include 1 %, include 1000 ids, exclude 1 id -- the device form, ids sorted on the device.  Each
filtered block runs right after an unfiltered block of the same workload in the same process (alternated), so the two
see the same clocks and neighbours.  Per configuration: median ms per query / per batch, the exact passes per query
(pbx_stats), and the mark pass on its own (mark_ids_kernel's device time under torch.profiler, in a separate run of 20
calls so that the timed blocks are not traced).  Prints the card name and power limit first; one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pixelbox_b200 import _native as nat, synth  # noqa: E402
from pixelbox_b200.corpus import Corpus  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # noqa: BLE001
        out = f"unavailable ({e})"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--singles", type=int, default=400, help="timed single queries per configuration (after warm-up)")
    ap.add_argument("--batches", type=int, default=6, help="timed 1024-query batches per configuration")
    ap.add_argument("--out", help="also write the JSON document here")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    n, d, k, seed = args.rows, args.dim, 100, 42
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(7)
    all_ids = np.arange(1, n + 1, dtype=np.int64)
    filters = {
        "include_50pct": (nat.PBX_FILTER_INCLUDE, all_ids[rng.random(n) < 0.5]),
        "include_1pct": (nat.PBX_FILTER_INCLUDE, all_ids[rng.random(n) < 0.01]),
        "include_1000": (nat.PBX_FILTER_INCLUDE, np.sort(rng.choice(all_ids, 1000, replace=False))),
        "exclude_1": (nat.PBX_FILTER_EXCLUDE, all_ids[[n // 2]]),
    }
    d_filters = {name: (mode, torch.from_numpy(ids).to(dev)) for name, (mode, ids) in filters.items()}
    doc = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "rows": n, "dim": d, "k": k, "configs": {}}
    print(json.dumps({"card": doc["card"], "rows": n, "dim": d}), flush=True)

    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed)
        queries = synth.synth_queries(5, 1024, d, n, seed)
        d_q = torch.from_numpy(queries).to(dev)
        hits = torch.empty(1024 * k * nat.HIT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        cnt = torch.empty(1024, dtype=torch.int32, device=dev)
        stream = torch.cuda.current_stream().cuda_stream

        def run(name, nq, q0):
            qp = d_q[q0:q0 + nq].data_ptr()
            if name is None:
                c.search_device(qp, nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), stream)
            else:
                mode, f = d_filters[name]
                c.search_device_filtered(qp, nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), f.data_ptr(), f.numel(), mode, stream)

        def block(name, nq, reps, q_off):
            """ms per call over `reps` calls enqueued back to back (CUDA events), and exact passes per query."""
            xp0 = c.stats().exact_passes
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(reps):
                run(name, nq, (q_off + i) % (1024 - nq + 1) if nq == 1 else 0)
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / reps, (c.stats().exact_passes - xp0) / (reps * nq)

        for name in [None] + list(filters):                      # warm-up of every path and filter
            run(name, 1, 0)
            run(name, 1024, 0)
        torch.cuda.synchronize()
        base = {"single_ms": [], "batch_ms": []}
        for name in filters:
            res = {"single_ms": [], "batch_ms": [], "unfiltered_single_ms": [], "unfiltered_batch_ms": [], "exact_per_query": [0.0, 0.0]}
            for b in range(args.singles // 50):                  # alternate: unfiltered block, filtered block
                u, _ = block(None, 1, 50, 50 * b)
                f, xp = block(name, 1, 50, 50 * b)
                res["unfiltered_single_ms"].append(u)
                res["single_ms"].append(f)
                res["exact_per_query"][0] += xp / (args.singles // 50)
            for b in range(args.batches):
                u, _ = block(None, 1024, 1, 0)
                f, xp = block(name, 1024, 1, 0)
                res["unfiltered_batch_ms"].append(u)
                res["batch_ms"].append(f)
                res["exact_per_query"][1] += xp / args.batches
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(20):
                    run(name, 1, i)
                torch.cuda.synchronize()
            mark_us = [(getattr(ev, "self_device_time_total", None) or ev.self_cuda_time_total) / ev.count
                       for ev in prof.key_averages() if "mark_ids_kernel" in ev.key and ev.count]
            mode, ids = filters[name]
            out = {
                "mode": "include" if mode == nat.PBX_FILTER_INCLUDE else "exclude", "n_ids": int(ids.size),
                "single_ms_median": round(float(np.median(res["single_ms"])), 4),
                "unfiltered_single_ms_median": round(float(np.median(res["unfiltered_single_ms"])), 4),
                "batch1024_ms_median": round(float(np.median(res["batch_ms"])), 3),
                "unfiltered_batch1024_ms_median": round(float(np.median(res["unfiltered_batch_ms"])), 3),
                "mark_pass_ms_mean": round(float(mark_us[0]) / 1e3, 4) if mark_us else None,
                "exact_passes_per_query_single": round(res["exact_per_query"][0], 4),
                "exact_passes_per_query_batched": round(res["exact_per_query"][1], 4),
            }
            base["single_ms"] += res["unfiltered_single_ms"]
            base["batch_ms"] += res["unfiltered_batch_ms"]
            doc["configs"][name] = out
            print(json.dumps({name: out}), flush=True)
        doc["configs"]["unfiltered"] = {"single_ms_median": round(float(np.median(base["single_ms"])), 4),
                                        "batch1024_ms_median": round(float(np.median(base["batch_ms"])), 3)}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc), flush=True)


if __name__ == "__main__":
    main()
