"""ShardedCorpus.replace with every rank ON THE SAME GPU (so it runs on a 1-GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tools/replace_exchange_check.py

One process per rank over gloo, every rank a GPU shard on cuda:0 (as tools/remove_check.py).  All ranks pass the same
(ids, hashes): ids on both shards, one id held by a row of each shard, and an id listed twice (its last hash wins).  Every
rank must receive the global count, and rank 0 compares the merged results with the oracle over the updated table.
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
    rng = np.random.default_rng(67)
    n, d = 40_000, 256
    cent = rng.integers(0, 256, size=(40, d))
    rows = np.clip(cent[rng.integers(0, 40, n)] + rng.integers(-3, 4, size=(n, d)), 0, 255).astype(np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 7
    ids[n - 1] = ids[3]                          # one id in shard 0 and in the last shard
    pick = np.concatenate([[3], rng.choice(np.arange(4, n - 1), 4000, replace=False)])
    req_ids = np.concatenate([ids[pick], ids[pick[1:2]]])
    req_rows = np.clip(cent[rng.integers(0, 40, len(req_ids))] + rng.integers(-3, 4, size=(len(req_ids), d)), 0, 255).astype(np.uint8)
    new = rows.copy()
    for i, r in zip(req_ids.tolist(), req_rows):  # UPDATE per (id, hash), in order
        new[ids == i] = r
    expect = int(np.isin(ids, req_ids).sum())
    queries = np.concatenate([req_rows[[0, 1, -1]], rows[pick[:2]], rng.integers(0, 256, size=(35, d), dtype=np.uint8)])
    ok = True
    sc = ShardedCorpus(d, device=0)
    sc.load_table(ids, rows)
    replaced = sc.replace(req_ids, req_rows)
    if replaced != expect or sc.total_rows() != n:
        print(f"rank {rank}: replaced {replaced}, expected {expect}")
        ok = False
    for k, md, qs in ((100, 1e3, queries), (10, 1e3, queries[:5]), (500, 1e7, queries[:2])):
        res = sc.search(qs, k, md)
        if rank == 0:
            for qi, q in enumerate(qs):
                o_ids, o_dist, o_dot, o_n2 = oracle.topk(new, ids, q, k, md, threads=4)
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
        print("replace_exchange_check", "OK" if int(flag.item()) == 1 else "FAILED", f"world={world} (all ranks on cuda:0)")
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
