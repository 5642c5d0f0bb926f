"""Cost of searches on a view (pbx_corpus_view_create) beside the per-call filter, on a 10M x 256 synthetic shard (ids =
row + 1).
    python tools/view_time.py [--rows 10000000] [--dim 256] [--singles 400] [--batches 6] [--reps 10] [--out FILE]

Sets: 1000 ids, 1 % and 50 % of the rows.  Per set, in one process:
  - device-resident single queries (k = 100, enqueued back to back on one stream, CUDA events over blocks of 50) and
    1024-query batches (CUDA events per batch) on the view, with the per-call filter of the same ids on the parent (the
    device form, ids sorted on the device) and unfiltered on the parent; the three alternate block by block, so they see
    the same clocks and neighbours;
  - the build time of the view (host clock around pbx_corpus_view_create, which synchronises);
  - what the view adds to a 1-row append (append + flush), a 1000-row remove and a 1000-row replace on the parent: the
    median host time of each call with the view minus the same without it (both measured in this run, the view's
    absence first).  The appended row's id is in the set, so it joins the view; the removed ids are half in the set; the
    replaced ids are in the set.  Removed rows are appended back, untimed.
Prints the card name and power limit first; one JSON document.
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
    ap.add_argument("--singles", type=int, default=400, help="timed single queries per configuration (after warm-up)")
    ap.add_argument("--batches", type=int, default=6, help="timed 1024-query batches per configuration")
    ap.add_argument("--reps", type=int, default=10, help="timed repetitions of each mutation, with and without the view")
    ap.add_argument("--out", help="also write the JSON document here")
    args = ap.parse_args()
    import torch
    n, d, k, seed = args.rows, args.dim, 100, 42
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(7)
    all_ids = np.arange(1, n + 1, dtype=np.int64)
    sets = {
        "1000": np.sort(rng.choice(all_ids, 1000, replace=False)),
        "1pct": all_ids[rng.random(n) < 0.01],
        "50pct": all_ids[rng.random(n) < 0.5],
    }
    doc = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "rows": n, "dim": d, "k": k, "configs": {}}
    print(json.dumps({"card": doc["card"], "rows": n, "dim": d}), flush=True)

    with Corpus(d, capacity_hint=n + 4096) as c:
        c.fill_synthetic(n, seed)
        queries = synth.synth_queries(5, 1024, d, n, seed)
        d_q = torch.from_numpy(queries).to(dev)
        hits = torch.empty(1024 * k * nat.HIT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        cnt = torch.empty(1024, dtype=torch.int32, device=dev)
        stream = torch.cuda.current_stream().cuda_stream

        def mutations(fset):
            """Median host ms of a 1-row append + flush, a 1000-row remove and a 1000-row replace."""
            out = {"append1_ms": [], "remove1000_ms": [], "replace1000_ms": []}
            for r in range(args.reps):
                row = rng.integers(0, 256, size=(1, d), dtype=np.uint8)
                a_id = np.array([fset[r % len(fset)]], np.int64)        # an id of the set: the row joins the view
                t0 = time.perf_counter()
                c.append(a_id, row)
                c.flush()
                out["append1_ms"].append((time.perf_counter() - t0) * 1e3)
                c.remove(a_id)                                          # untimed: back to one row per id
                ids_rm = np.concatenate([rng.choice(fset, 500, replace=len(fset) < 500), rng.choice(all_ids, 500)])
                ids_rm = np.unique(ids_rm)
                t0 = time.perf_counter()
                c.remove(ids_rm)
                out["remove1000_ms"].append((time.perf_counter() - t0) * 1e3)
                c.append(ids_rm, synth_rows(ids_rm))                    # untimed: the table is whole again
                ids_rp = np.unique(rng.choice(fset, 1000, replace=len(fset) < 1000))
                t0 = time.perf_counter()
                c.replace(ids_rp, rng.integers(0, 256, size=(len(ids_rp), d), dtype=np.uint8))
                out["replace1000_ms"].append((time.perf_counter() - t0) * 1e3)
            return {key: round(float(np.median(v)), 4) for key, v in out.items()}

        def synth_rows(ids):
            """The synthetic rows of these ids (id = row + 1): what a re-append must restore."""
            return np.concatenate([synth.synth_rows(seed, int(i) - 1, 1, d) for i in ids])

        for name, fset in sets.items():
            d_f = torch.from_numpy(fset).to(dev)
            base_mut = mutations(fset)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            v = c.view(fset)
            build_ms = (time.perf_counter() - t0) * 1e3

            def run(kind, nq, q0):
                qp = d_q[q0:q0 + nq].data_ptr()
                if kind == "view":
                    v.search_device(qp, nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), stream)
                elif kind == "filter":
                    c.search_device_filtered(qp, nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), d_f.data_ptr(), d_f.numel(),
                                             nat.PBX_FILTER_INCLUDE, stream)
                else:
                    c.search_device(qp, nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), stream)

            def block(kind, nq, reps, q_off):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(reps):
                    run(kind, nq, (q_off + i) % (1024 - nq + 1) if nq == 1 else 0)
                e1.record()
                e1.synchronize()
                return e0.elapsed_time(e1) / reps

            kinds = ("view", "filter", "none")
            for kind in kinds:                                          # warm-up of every path
                run(kind, 1, 0)
                run(kind, 1024, 0)
            torch.cuda.synchronize()
            res = {f"{kind}_{w}": [] for kind in kinds for w in ("single", "batch")}
            for b in range(args.singles // 50):
                for kind in kinds:
                    res[f"{kind}_single"].append(block(kind, 1, 50, 50 * b))
            for b in range(args.batches):
                for kind in kinds:
                    res[f"{kind}_batch"].append(block(kind, 1024, 1, 0))
            batched0 = v.stats().batched_queries
            run("view", 1024, 0)
            torch.cuda.synchronize()
            view_mut = mutations(fset)
            out = {
                "n_ids": int(fset.size), "view_rows": len(v), "build_ms": round(build_ms, 3),
                "view_batch_uses_tensor_core_path": v.stats().batched_queries > batched0,
                **{f"{key}_ms_median": round(float(np.median(val)), 4) for key, val in res.items()},
                "mutation_ms_without_view": base_mut, "mutation_ms_with_view": view_mut,
                "view_adds_ms": {key: round(view_mut[key] - base_mut[key], 4) for key in base_mut},
            }
            v.close()
            doc["configs"][name] = out
            print(json.dumps({name: out}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc), flush=True)


if __name__ == "__main__":
    main()
