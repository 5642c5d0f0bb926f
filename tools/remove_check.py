"""ShardedCorpus.remove with every rank ON THE SAME GPU (so it runs on a 1-GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tools/remove_check.py

One process per rank over gloo, every rank a GPU shard on cuda:0 (as tools/exchange_check.py).  All ranks remove the
same ids, spread over both shards and including a tie that straddles them; every rank must receive the global count,
and rank 0 compares the merged results with the oracle over the surviving rows.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle  # noqa: E402
from pixelbox_b200.shard import ShardedCorpus  # noqa: E402


def main():
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    rng = np.random.default_rng(61)
    n, d = 40_000, 256
    cent = rng.integers(0, 256, size=(40, d))
    rows = np.clip(cent[rng.integers(0, 40, n)] + rng.integers(-3, 4, size=(n, d)), 0, 255).astype(np.uint8)
    rows[100:400] = rows[100]                    # a plateau in shard 0 ...
    rows[n - 300:] = rows[100]                   # ... continued in the last shard
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 7
    gone = rng.random(n) < 0.1
    gone[200:300] = True
    gone[n - 150:] = True
    queries = np.concatenate([rows[[100, 25_000]], rows[np.flatnonzero(gone)[:2]], rng.integers(0, 256, size=(36, d), dtype=np.uint8)])
    ok = True
    sc = ShardedCorpus(d, device=0)
    sc.load_table(ids, rows)
    removed = sc.remove(ids[gone])
    if removed != int(gone.sum()) or sc.total_rows() != n - removed:
        print(f"rank {rank}: removed {removed}, expected {int(gone.sum())}")
        ok = False
    s_ids, s_rows = ids[~gone], rows[~gone]
    for k, md, qs in ((100, 1e3, queries), (10, 1e3, queries[:4]), (500, 1e7, queries[:2])):
        res = sc.search(qs, k, md)
        if rank == 0:
            for qi, q in enumerate(qs):
                o_ids, o_dist, o_dot, o_n2 = oracle.topk(s_rows, s_ids, q, k, md, threads=4)
                good = (list(res[qi].ids) == list(o_ids) and np.array_equal(res[qi].dist.view(np.uint32), o_dist.view(np.uint32))
                        and np.array_equal(res[qi].dot, o_dot) and np.array_equal(res[qi].norm2, o_n2))
                if not good:
                    print(f"MISMATCH k={k} md={md} q={qi}")
                ok &= good
    sc.close()
    flag = torch.tensor([1 if ok else 0])
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("remove_check", "OK" if int(flag.item()) == 1 else "FAILED", f"world={world} (all ranks on cuda:0)")
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
