"""Views (ShardedCorpus.view) on the row-sharded path with every rank ON THE SAME GPU (so it runs on a 1-GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tools/view_exchange_check.py

One process per rank over gloo, every rank a GPU shard on cuda:0 (as tools/filter_exchange_check.py).  Every rank makes a
view of its own shard with the same global ids and searches it through the exchange calls; each answer must equal the
filtered search of the whole table (pbx_exchange_search_hits_filtered) bit for bit, and the oracle's top-k over the
allowed rows.  The views then follow a removal, a replacement, a view_add and a view_drop of the parent."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle  # noqa: E402
from pixelbox_b200.shard import ShardedCorpus  # noqa: E402


def same(a, b):
    return (list(a.ids) == list(b.ids) and np.array_equal(a.dist.view(np.uint32), b.dist.view(np.uint32))
            and np.array_equal(a.dot, b.dot) and np.array_equal(a.norm2, b.norm2))


def main():
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    ok = True
    rng = np.random.default_rng(97)
    n, d = 60_000, 256
    cent = rng.integers(0, 256, size=(50, d))
    rows = np.clip(cent[rng.integers(0, 50, n)] + rng.integers(-3, 4, size=(n, d)), 0, 255).astype(np.uint8)
    rows[200:500] = rows[200]                    # a plateau in shard 0 ...
    rows[n - 400:] = rows[200]                   # ... continued in the last shard
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 5
    queries = np.concatenate([rows[[200, 31_000]], rng.integers(0, 256, size=(30, d), dtype=np.uint8)])
    fset = np.concatenate([ids[rng.random(n) < 0.05], ids[300:350], ids[n - 100:], [3, 7]])    # + ids that match nothing
    for peer in (True, False):
        sc = ShardedCorpus(d, device=0, use_peer_exchange=peer)
        sc.load_table(ids, rows)
        used_peer = sc._exchange is not None
        view = sc.view(fset)
        table_rows, table_ids, cur_set = rows.copy(), ids.copy(), np.unique(fset)
        for step in ("built", "remove", "replace", "add", "drop"):
            if step == "remove":
                gone = np.concatenate([fset[:40], ids[:100]])
                sc.remove(gone)
                keep = ~np.isin(table_ids, gone)
                table_rows, table_ids = table_rows[keep], table_ids[keep]
            elif step == "replace":
                pick = np.unique(np.concatenate([cur_set[50:90], table_ids[1000:1040]]))
                pick = pick[np.isin(pick, table_ids)]
                new = rng.integers(0, 256, size=(len(pick), d), dtype=np.uint8)
                sc.replace(pick, new)
                at = {int(i): j for j, i in enumerate(pick.tolist())}
                for r, i in enumerate(table_ids.tolist()):
                    if i in at:
                        table_rows[r] = new[at[i]]
            elif step == "add":
                extra = table_ids[5000:5600]
                view.view_add(extra)
                cur_set = np.union1d(cur_set, extra)
            elif step == "drop":
                view.view_drop(cur_set[::3])
                cur_set = np.setdiff1d(cur_set, cur_set[::3])
            allowed = np.isin(table_ids, cur_set)
            for k, md, qs in ((100, 1e3, queries), (10, 1e3, queries[:3]), (500, 1e7, queries[:2]), (100, 1e3, queries[:1])):
                got = view.search(qs, k, md)
                want = sc.search(qs, k, md, within=cur_set)
                if rank == 0:
                    for qi, q in enumerate(qs):
                        o = oracle.topk(table_rows[allowed], table_ids[allowed], q, k, md, threads=4)
                        good = same(got[qi], want[qi]) and list(got[qi].ids) == list(o[0]) and np.array_equal(
                            got[qi].dist.view(np.uint32), o[1].view(np.uint32))
                        if not good:
                            print(f"MISMATCH peer={used_peer} step={step} k={k} md={md} q={qi}")
                        ok &= good
        if rank == 0:
            print(f"view exchange path {'peer-memory kernel' if used_peer else 'all-gather + merge kernel'}: {'ok' if ok else 'FAILED'}")
        view.close()
        sc.close()
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("view_exchange_check", "OK" if ok else "FAILED", f"world={world} (all ranks on cuda:0)")
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
