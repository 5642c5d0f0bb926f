"""Filtered searches (within= / excluding=) of the row-sharded path with every rank ON THE SAME GPU (so it runs on a
1-GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tools/filter_exchange_check.py

One process per rank over gloo, every rank a GPU shard on cuda:0 (as tools/exchange_check.py).  Every rank passes the
same global ids; each shard marks its own rows, searches them exactly, and the unchanged merge (the peer-memory kernel
pbx_exchange_search_hits_filtered, or the all-gather + merge kernel fallback over pbx_search_device_filtered) must give
the oracle's top-k over the allowed rows of the whole table.  Sets: one spanning every shard, one inside a single shard,
a plateau of identical rows half inside the set, and an exclusion.
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
    ok = True
    rng = np.random.default_rng(83)
    n, d = 60_000, 256
    cent = rng.integers(0, 256, size=(50, d))
    rows = np.clip(cent[rng.integers(0, 50, n)] + rng.integers(-3, 4, size=(n, d)), 0, 255).astype(np.uint8)
    rows[200:500] = rows[200]                    # a plateau in shard 0 ...
    rows[n - 400:] = rows[200]                   # ... continued in the last shard
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 5
    queries = np.concatenate([rows[[200, 31_000]], rng.integers(0, 256, size=(30, d), dtype=np.uint8)])
    spread = ids[rng.random(n) < 0.02]
    sets = [
        ("within 2 %", "within", np.concatenate([spread, ids[300:350], ids[n - 100:], [3, 7]])),   # + ids that match nothing
        ("within one shard", "within", ids[1000:1040][::-1].copy()),                                # unsorted on purpose
        ("excluding", "excluding", np.concatenate([ids[rng.random(n) < 0.3], ids[200:450]])),
    ]
    for peer in (True, False):
        sc = ShardedCorpus(d, device=0, use_peer_exchange=peer)
        sc.load_table(ids, rows)
        used_peer = sc._exchange is not None
        if peer and not used_peer and rank == 0:
            print("note: CUDA IPC mapping unavailable, the peer path was not exercised")
        for name, kw, fset in sets:
            allowed = np.isin(ids, fset) if kw == "within" else ~np.isin(ids, fset)
            a_ids, a_rows = ids[allowed], rows[allowed]
            for k, md, qs in ((100, 1e3, queries), (10, 1e3, queries[:3]), (500, 1e7, queries[:2]), (100, 1e3, queries[:1])):
                res = sc.search(qs, k, md, **{kw: fset})
                if rank == 0:
                    for qi, q in enumerate(qs):
                        o_ids, o_dist, o_dot, o_n2 = oracle.topk(a_rows, a_ids, q, k, md, threads=4)
                        good = (list(res[qi].ids) == list(o_ids) and np.array_equal(res[qi].dist.view(np.uint32), o_dist.view(np.uint32))
                                and np.array_equal(res[qi].dot, o_dot) and np.array_equal(res[qi].norm2, o_n2))
                        if not good:
                            print(f"MISMATCH peer={used_peer} set={name} k={k} md={md} q={qi}")
                        ok &= good
        if rank == 0:
            print(f"filtered exchange path {'peer-memory kernel' if used_peer else 'all-gather + merge kernel'}: {'ok' if ok else 'FAILED'}")
        sc.close()
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("filter_exchange_check", "OK" if ok else "FAILED", f"world={world} (all ranks on cuda:0)")
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
