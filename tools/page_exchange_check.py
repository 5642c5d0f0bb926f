"""Paged searches (after=) of the row-sharded path with every rank ON THE SAME GPU (so it runs on a 1-GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tools/page_exchange_check.py

One process per rank over gloo, every rank a GPU shard on cuda:0 (as tools/filter_exchange_check.py).  Every rank passes the
same cursors; each shard returns its next k rows after the same global cursor, and the unchanged merge (the peer-memory
kernel pbx_exchange_search_hits_page, or the all-gather + merge kernel fallback over pbx_search_device_page) must give the
keyset SQL's page of the whole table.  Pages are iterated past PBX_MAX_K rows, unfiltered and with a filter, from the
first page, from -inf and from cursors inside a tie of identical rows that spans two shards.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pixelbox_b200.shard import ShardedCorpus  # noqa: E402
from tests import page_oracle  # noqa: E402

INT64_MIN = int(np.iinfo(np.int64).min)


def main():
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    ok = True
    rng = np.random.default_rng(89)
    n, d = 40_000, 128
    cent = rng.integers(0, 256, size=(40, d))
    rows = np.clip(cent[rng.integers(0, 40, n)] + rng.integers(-3, 4, size=(n, d)), 0, 255).astype(np.uint8)
    rows[100:400] = rows[100]                    # a tie in shard 0 ...
    rows[n - 300:] = rows[100]                   # ... continued in the last shard
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 3
    queries = np.concatenate([rows[[100, 20_000]], rng.integers(0, 256, size=(2, d), dtype=np.uint8)])
    fset = ids[rng.random(n) < 0.4]
    tie_d = page_oracle.order(rows, ids, queries[0], 1e3)[1][100]
    for peer in (True, False):
        sc = ShardedCorpus(d, device=0, use_peer_exchange=peer)
        sc.load_table(ids, rows)
        used_peer = sc._exchange is not None
        if peer and not used_peer and rank == 0:
            print("note: CUDA IPC mapping unavailable, the peer path was not exercised")
        for name, kw, allowed in (("all rows", {}, None), ("within 40 %", {"within": fset}, np.isin(ids, fset))):
            for k, starts in ((700, [None, (np.float32(-np.inf), INT64_MIN), (tie_d, int(ids[250])), None]),
                              (100, [(tie_d, INT64_MIN)] * 2)):
                qs = queries[:len(starts)]
                curs = list(starts)
                for _ in range(4):
                    res = sc.search(qs, k, 1e3, after=curs, **kw)
                    for qi, q in enumerate(qs):
                        w = page_oracle.page(rows, ids, q, k, 1e3, curs[qi], allowed)
                        good = (list(res[qi].ids) == list(w[0]) and np.array_equal(res[qi].dist.view(np.uint32), w[1].view(np.uint32))
                                and np.array_equal(res[qi].dot, w[2]) and np.array_equal(res[qi].norm2, w[3]))
                        if not good and rank == 0:
                            print(f"MISMATCH peer={used_peer} {name} k={k} q={qi} cursor={curs[qi]}")
                        ok &= good
                        if len(res[qi].ids):
                            curs[qi] = (res[qi].dist[-1], int(res[qi].ids[-1]))
        if rank == 0:
            print(f"paged exchange path {'peer-memory kernel' if used_peer else 'all-gather + merge kernel'}: {'ok' if ok else 'FAILED'}")
        sc.close()
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("page_exchange_check", "OK" if ok else "FAILED", f"world={world} (all ranks on cuda:0)")
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
