"""Cost of range searches (pbx_search_range) on a 10M x 256 synthetic shard (ids = row + 1), beside the ways to get the
same answer before them.
    python tools/range_time.py [--rows 10000000] [--dim 256] [--reps 10] [--out FILE]

One perturbed corpus row is the query.  Its answer sizes of about 100, 10k and 1M rows are set by radii read from its
whole ordered answer (the radius just above the target-th row's dist), plus the default max_dist = 1e3.  Per radius, in
one process and alternated call by call:
  - the range search with host buffers (capacity = the answer), and the same with capacity = 0 (count only);
  - paging to the same answer with pbx_search_page at k = 2048 (every page a full search, chained by the last row);
  - a top-k search (k = 100, pbx_search) as the floor.
Host clock around each call (every call ends with a device synchronisation); medians.  torch.profiler passes of their
own then give the mean device time of each kernel of a range search and of a count per radius, and of the top-k search,
and the streaming rate of each scan kernel (rows x dim bytes over its time).  The card name and power limit are read
first; one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys
import time

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
    ap.add_argument("--reps", type=int, default=10, help="timed calls per configuration (paging: whole chains)")
    ap.add_argument("--out", help="also write the JSON document here")
    args = ap.parse_args()
    import torch
    n, d, seed = args.rows, args.dim, 42
    torch.cuda.set_device(0)
    doc = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "rows": n, "dim": d, "configs": {}}
    print(json.dumps({"card": doc["card"], "rows": n, "dim": d}), flush=True)
    L = nat.lib()
    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed)
        q = np.ascontiguousarray(synth.synth_queries(3, 2, d, n, seed)[:1])
        everything = c.search_range(q, 1e7)[0]
        assert everything.total == n
        radii = {}
        for target in (100, 10_000, 1_000_000):
            radii[f"about_{target}"] = float(np.nextafter(everything.dist[target - 1], np.float32(np.inf)))
        radii["default_1e3"] = 1e3
        del everything
        hits = np.empty(n, nat.HIT_DTYPE)
        off, tot = np.zeros(2, np.uint64), np.zeros(1, np.uint64)
        page = np.empty(2048, nat.HIT_DTYPE)
        pcnt = np.zeros(1, np.uint32)
        nofilt = np.zeros(0, np.int64)

        def range_call(md, cap):
            nat.check(L.pbx_search_range(c.handle, nat.ptr(q), 1, md, None, None, 0, nat.PBX_FILTER_EXCLUDE,
                                         nat.ptr(hits) if cap else None, cap, nat.ptr(off), nat.ptr(tot)))
            return int(tot[0])

        def paging(md):
            cur, rows_seen, pages = None, 0, 0
            while True:
                nat.check(L.pbx_search_page(c.handle, nat.ptr(q), 1, 2048, md, nat.ptr(cur) if cur is not None else None,
                                            nat.ptr(nofilt), 0, nat.PBX_FILTER_EXCLUDE, nat.ptr(page), nat.ptr(pcnt)))
                m = int(pcnt[0])
                rows_seen += m
                pages += 1
                if m < 2048:
                    return rows_seen, pages
                cur = page[m - 1:m].copy()

        def timed(fn, *a):
            t0 = time.perf_counter()
            r = fn(*a)
            return (time.perf_counter() - t0) * 1e3, r

        for name, md in radii.items():
            total = range_call(md, n)                  # warm-up (grows the scratch to this answer) and the answer's size
            range_call(md, 0)
            c.search(q, 100, md)
            res = {"range_ms": [], "count_ms": [], "topk100_ms": []}
            for _ in range(args.reps):
                for key, fn, a in (("range_ms", range_call, (md, n)), ("count_ms", range_call, (md, 0)),
                                   ("topk100_ms", c.search, (q, 100, md))):
                    ms, r = timed(fn, *a)
                    res[key].append(ms)
                    if key != "topk100_ms":
                        assert r == total
            page_ms, (rows_paged, pages) = timed(paging, md)
            assert rows_paged == total
            page_runs = [page_ms] + [timed(paging, md)[0] for _ in range(1 if total > 2_000_000 else 2)]
            out = {"max_dist": md, "total": total, **{k2.replace("_ms", "_ms_median"): round(float(np.median(v)), 4) for k2, v in res.items()},
                   "paging_k2048_ms_median": round(float(np.median(page_runs)), 3), "pages": pages}
            doc["configs"][name] = out
            print(json.dumps({name: out}), flush=True)

        # device time per kernel: profiled passes apart from the timed ones, one per radius and mode, and one of the top-k
        from torch.profiler import ProfilerActivity, profile

        def kernels(fn, *a):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    fn(*a)
            out = {}
            for ev in prof.key_averages():
                if ev.device_type is not None and "CUDA" in str(ev.device_type) and ev.count:
                    t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                    out[ev.key[:90]] = {"calls": ev.count, "mean_us": round(t / ev.count, 2)}
            return out

        kern = {}
        for name, md in radii.items():
            kern[f"{name} range"] = kernels(range_call, md, n)
            kern[f"{name} count"] = kernels(range_call, md, 0)
        kern["topk100"] = kernels(c.search, q, 100, 1e3)
        rates = {}
        for name, ks in kern.items():
            for key, v in ks.items():
                if ("range_scan_kernel" in key or key.startswith("void pbx::scan_kernel<")) and v["mean_us"] > 0:
                    rates[name] = {"kernel_us": v["mean_us"], "tb_per_s": round(n * d / (v["mean_us"] * 1e-6) / 1e12, 3)}
        doc["kernels"] = kern
        doc["scan"] = rates
        print(json.dumps({"scan": rates}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc), flush=True)


if __name__ == "__main__":
    main()
