"""Range searches (ShardedCorpus.search_range / count_within) of the row-sharded path with every rank ON THE SAME GPU
(so it runs on a 1-GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tools/range_exchange_check.py

One process per rank over gloo, every rank a GPU shard on cuda:0 (as tools/page_exchange_check.py).  Each shard runs the
range search of its rows; the totals and the shards' first rows are all-gathered and merged on the device.  Every answer
must be the range oracle's over the whole table: ids, order, dist bit for bit, dot, norm2 and the total -- unfiltered,
filtered, from a cursor, cut at a limit, and across a tie of identical rows that spans both shards.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pixelbox_b200.shard import ShardedCorpus  # noqa: E402
from tests import range_oracle  # noqa: E402


def main():
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    ok = True
    rng = np.random.default_rng(97)
    n, d = 40_000, 64
    cent = rng.integers(0, 256, size=(40, d))
    rows = np.clip(cent[rng.integers(0, 40, n)] + rng.integers(-3, 4, size=(n, d)), 0, 255).astype(np.uint8)
    rows[100:400] = rows[100]                    # a tie in shard 0 ...
    rows[n - 300:] = rows[100]                   # ... continued in the last shard
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 3
    queries = np.stack([rows[100], rows[20_000], rng.integers(0, 256, d, dtype=np.uint8)])
    fset = ids[rng.random(n) < 0.4]
    allowed = np.isin(ids, fset)
    sc = ShardedCorpus(d, device=0, use_peer_exchange=False)
    sc.load_table(ids, rows)
    for q in queries:
        dist_all = range_oracle.page_oracle.order(rows, ids, q, 1e7)[1]
        for md in (0.0, float(np.sort(dist_all)[2500]), 1e3, 1e7):
            full = range_oracle.answer(rows, ids, q, md, dists=dist_all)
            cur = (full[1][len(full[1]) // 2], int(full[0][len(full[0]) // 2])) if len(full[0]) else None
            cases = (("all", {}, full, None),
                     ("limit 250", {"limit": 250}, tuple(a[:250] for a in full), len(full[0])),
                     ("within 40 %", {"within": fset}, range_oracle.answer(rows, ids, q, md, allowed=allowed, dists=dist_all), None),
                     ("after", {"after": [cur]}, range_oracle.answer(rows, ids, q, md, cur, dists=dist_all), None))
            for name, kw, w, total in cases:
                r = sc.search_range(q, md, **kw)[0]
                good = (list(r.ids) == list(w[0]) and np.array_equal(r.dist.view(np.uint32), w[1].view(np.uint32))
                        and sorted(zip(r.ids.tolist(), r.dot.tolist(), r.norm2.tolist())) == sorted(zip(w[0].tolist(), w[2].tolist(), w[3].tolist()))
                        and r.total == (len(w[0]) if total is None else total))
                cnt_kw = {k: v for k, v in kw.items() if k != "limit"}
                good &= int(sc.count_within(q, md, **cnt_kw)[0]) == (len(w[0]) if total is None else total)
                if not good and rank == 0:
                    print(f"MISMATCH {name} max_dist={md} rows={len(r.ids)}/{len(w[0])} total={r.total}")
                ok &= good
    sc.close()
    flag = torch.tensor([1 if ok else 0])
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("range_exchange_check", "OK" if int(flag.item()) == 1 else "FAILED", f"world={world} (all ranks on cuda:0)")
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
