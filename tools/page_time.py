"""Cost of paged searches (pbx_search_device_page) on a 10M x 256 synthetic shard (ids = row + 1).
    python tools/page_time.py [--rows 10000000] [--dim 256] [--singles 400] [--batches 6] [--out FILE]

Workloads (k = 100, device form): single queries enqueued back to back on one stream, timed with CUDA events over blocks
of 50 after a warm-up, and batches of 1024 queries (the tensor-core path, CUDA events per batch).  The cursor of every
query is its own row at depth D of the deep order (taken from pages of 1000 beforehand): D = 0 (the cursor -inf, so the
paged path with nothing before the cursor), 100, 1000, 10000 for single queries, 0, 1000, 10000 for batches, and one
filtered point (include 50 %, depth 1000).  Each paged block runs right after an unpaged block of the same workload in
the same process (alternated), so the two see the same clocks and neighbours.  Per configuration: median ms per query /
per batch and exact passes per query (pbx_stats).  Prints the card name and power limit first; one JSON document.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pixelbox_b200 import _native as nat, synth  # noqa: E402
from pixelbox_b200.corpus import Corpus  # noqa: E402
from tools.filter_time import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--singles", type=int, default=400, help="timed single queries per configuration (after warm-up)")
    ap.add_argument("--batches", type=int, default=6, help="timed 1024-query batches per configuration")
    ap.add_argument("--out", help="also write the JSON document here")
    args = ap.parse_args()
    import torch
    n, d, k, seed, nq = args.rows, args.dim, 100, 42, 1024
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(7)
    doc = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "rows": n, "dim": d, "k": k, "configs": {}}
    print(json.dumps({"card": doc["card"], "rows": n, "dim": d}), flush=True)
    fset = np.arange(1, n + 1, dtype=np.int64)[rng.random(n) < 0.5]

    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed)
        queries = synth.synth_queries(5, nq, d, n, seed)

        def cursors(depth, within=None):
            """[nq] records: each query's row at `depth` of its deep order ({-inf, INT64_MIN} for depth 0)."""
            cur = nat.page_cursors([None] * nq, nq)
            if depth == 0:
                return cur
            done = 0
            while done < depth:
                step = min(1000, depth - done)
                res = c.search(queries, step, 1e3, after=cur, within=within)
                for i, r in enumerate(res):
                    assert len(r.ids) == step, "the corpus ran out of rows before the depth"
                    cur[i]["dist"], cur[i]["image_id"] = r.dist[-1], r.ids[-1]
                done += step
            return cur

        d_q = torch.from_numpy(queries).to(dev)
        d_f = torch.from_numpy(fset).to(dev)
        hits = torch.empty(nq * k * nat.HIT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        cnt = torch.empty(nq, dtype=torch.int32, device=dev)
        stream = torch.cuda.current_stream().cuda_stream
        rec = nat.HIT_DTYPE.itemsize

        def run(d_after, filtered, q_at_once, q0):
            qp = d_q[q0:q0 + q_at_once].data_ptr()
            if d_after is None:
                c.search_device(qp, q_at_once, k, 1e3, hits.data_ptr(), cnt.data_ptr(), stream)
            else:
                c.search_device_page(qp, q_at_once, k, 1e3, hits.data_ptr(), cnt.data_ptr(), d_after.data_ptr() + q0 * rec,
                                     d_f.data_ptr() if filtered else 0, d_f.numel() if filtered else 0,
                                     nat.PBX_FILTER_INCLUDE if filtered else nat.PBX_FILTER_EXCLUDE, stream)

        def block(d_after, filtered, q_at_once, reps, q_off):
            xp0 = c.stats().exact_passes
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(reps):
                run(d_after, filtered, q_at_once, (q_off + i) % nq if q_at_once == 1 else 0)
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / reps, (c.stats().exact_passes - xp0) / (reps * q_at_once)

        configs = [("single_depth0", 0, False, 1), ("single_depth100", 100, False, 1), ("single_depth1000", 1000, False, 1),
                   ("single_depth10000", 10000, False, 1), ("batch_depth0", 0, False, nq), ("batch_depth1000", 1000, False, nq),
                   ("batch_depth10000", 10000, False, nq), ("single_within50pct_depth1000", 1000, True, 1),
                   ("batch_within50pct_depth1000", 1000, True, nq)]
        run(None, False, 1, 0)
        run(None, False, nq, 0)
        for name, depth, filtered, q_at_once in configs:
            d_after = torch.from_numpy(cursors(depth, fset if filtered else None).view(np.uint8).copy()).to(dev)
            run(d_after, filtered, 1, 0)
            run(d_after, filtered, nq, 0)
            torch.cuda.synchronize()
            paged, unpaged, xps = [], [], []
            if q_at_once == 1:
                for b in range(args.singles // 50):
                    u, _ = block(None, False, 1, 50, 50 * b)
                    p, xp = block(d_after, filtered, 1, 50, 50 * b)
                    unpaged.append(u); paged.append(p); xps.append(xp)
            else:
                for b in range(args.batches):
                    u, _ = block(None, False, nq, 1, 0)
                    p, xp = block(d_after, filtered, nq, 1, 0)
                    unpaged.append(u); paged.append(p); xps.append(xp)
            out = {"depth": depth, "queries_per_call": q_at_once, "filter": "include 50 %" if filtered else None,
                   "paged_ms_median": round(float(np.median(paged)), 4), "unpaged_ms_median": round(float(np.median(unpaged)), 4),
                   "ratio": round(float(np.median(paged) / np.median(unpaged)), 3),
                   "exact_passes_per_query": round(float(np.mean(xps)), 4)}
            doc["configs"][name] = out
            print(json.dumps({name: out}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc), flush=True)


if __name__ == "__main__":
    main()
