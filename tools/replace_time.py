"""Cost of pbx_corpus_replace on a 10M x 256 synthetic shard, against remove + append of the same ids and a full load.
    python tools/replace_time.py [--rows 10000000] [--dim 256] [--out profiles/replace_time_10Mx256.json]

For m in {1, 1k, 100k, all rows} random ids (in random order) with random new hashes:
  - replace: the host-clock time of the synchronous call (median of 3), then one more call under torch.profiler split by
    kernel: mark (replace_mark_kernel), write (replace_write_kernel), row_meta (replace_row_meta_kernel), block_meta
    (replace_block_meta_kernel), and the copies (the request upload, the count read back).  `host_other` is the median
    call minus the device time: the host sort of the request, its padded copy, launches and synchronisations.
  - remove + append of the same rows (the shard refilled before each pair): host-clock time of each call (median of 3;
    1 for all rows), and the device time of one pair under torch.profiler.
  - for all rows, also pbx_corpus_load of the updated table (host-clock time, and its device time).
Prints the card name and power limit first; one JSON line per measurement; --out also writes them all as one JSON file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pixelbox_b200.corpus import Corpus  # noqa: E402

STAGES = (("replace_mark_kernel", "mark"), ("replace_write_kernel", "write"), ("replace_row_meta_kernel", "row_meta"),
          ("replace_block_meta_kernel", "block_meta"), ("Memcpy", "copies"))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # noqa: BLE001
        out = f"unavailable ({e})"
    return out


def timed(fn, *args):
    t0 = time.perf_counter()
    r = fn(*args)
    return (time.perf_counter() - t0) * 1e3, r


def profiled(fn, *args):
    """(host-clock ms, {stage: device ms}, total device ms) of one call under torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ms, _ = timed(fn, *args)
    parts = {name: 0.0 for _, name in STAGES}
    total = 0.0
    for ev in prof.key_averages():
        us = getattr(ev, "self_device_time_total", None)
        us = (us if us is not None else ev.self_cuda_time_total) / 1e3
        total += us
        for key, name in STAGES:
            if key in ev.key:
                parts[name] += us
    return ms, parts, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    n, d, seed = args.rows, args.dim, 42
    records = [{"card": card(), "rows": n, "dim": d}]
    print(json.dumps(records[0]), flush=True)

    def emit(rec):
        records.append(rec)
        print(json.dumps(rec), flush=True)

    rng = np.random.default_rng(1)
    with Corpus(d, capacity_hint=n + 4096) as c:
        c.fill_synthetic(n, seed)
        c.replace([-1], np.zeros((1, d), np.uint8))          # warm-up: first launches load the module
        c.remove([-1])
        for m in (1, 1000, 100_000, n):
            ids = (rng.permutation(n)[:m] + 1).astype(np.int64)      # fill_synthetic: image_id = row + 1
            hashes = rng.integers(0, 256, size=(m, d), dtype=np.uint8)
            reps = 3 if m < n else 1
            c.fill_synthetic(n, seed)
            calls = []
            for _ in range(3):
                ms, replaced = timed(c.replace, ids, hashes)
                assert replaced == m
                calls.append(ms)
            ms_prof, parts, dev = profiled(c.replace, ids, hashes)
            call = float(np.median(calls))
            emit({"op": "replace", "m": m, "call_ms_median": round(call, 3), "calls_ms": [round(x, 3) for x in calls],
                  "profiled_call_ms": round(ms_prof, 3), **{k + "_ms": round(v, 4) for k, v in parts.items()},
                  "device_ms": round(dev, 4), "host_other_ms": round(call - dev, 3)})
            rem, app = [], []
            for _ in range(reps):
                c.fill_synthetic(n, seed)
                ms_r, removed = timed(c.remove, ids)
                assert removed == m
                ms_a, _ = timed(c.append, ids, hashes)
                c.flush()
                rem.append(ms_r)
                app.append(ms_a)
            c.fill_synthetic(n, seed)
            _, _, dev_r = profiled(c.remove, ids)
            _, _, dev_a = profiled(lambda: (c.append(ids, hashes), c.flush()))
            r_ms, a_ms = float(np.median(rem)), float(np.median(app))
            emit({"op": "remove+append", "m": m, "remove_ms_median": round(r_ms, 3), "append_ms_median": round(a_ms, 3),
                  "total_ms": round(r_ms + a_ms, 3), "device_ms": round(dev_r + dev_a, 4),
                  "host_other_ms": round(r_ms + a_ms - dev_r - dev_a, 3)})
            if m == n:
                ms_l, _ = timed(c.load, ids, hashes)
                _, _, dev_l = profiled(c.load, ids, hashes)
                emit({"op": "load", "m": m, "call_ms": round(ms_l, 3), "device_ms": round(dev_l, 4), "host_other_ms": round(ms_l - dev_l, 3)})
            del hashes
    if args.out:
        with open(args.out, "w") as f:
            json.dump(records, f, indent=1)


if __name__ == "__main__":
    main()
