"""ShardedCorpus: the `semantic_hashes` table row-sharded over the GPUs of one box.

One process per GPU (torch.distributed); every rank owns one Corpus shard, answers each query
over its rows and contributes its k best records; ONE all-gather of those records is the only
exchange step of the path, followed by a merge under the reference's order (dist asc, image_id
asc) on every rank (SURVEY.md section 8e).  On GPUs the exchange and the merge are one kernel
over NVLink peer memory (pbx_exchange_*: CUDA IPC mailboxes, release/acquire flags); NCCL
all_gather_into_tensor + pbx_merge_hits_device is the fallback, gloo + pbx_merge_hits the CPU test path.

torch is plumbing here (process group, device buffers, streams); the search, the records and
both merge implementations are the C-ABI library's.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _native as nat
from .corpus import Corpus, RangeResult, SearchResult, merge_hits

HIT_BYTES = nat.HIT_DTYPE.itemsize


def shard_rows(n_rows: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block partition of a table of n_rows rows: [first, first + count) of `rank`."""
    base, rem = divmod(n_rows, world)
    first = rank * base + min(rank, rem)
    return first, base + (1 if rank < rem else 0)


class ShardedCorpus:
    """`local` is this rank's shard.  Tests on CPU (gloo) inject an object with the same
    `search_hits(queries, k, max_dist) -> (hits[nq][k], counts[nq])` method; on GPUs it is a Corpus."""

    def __init__(self, dim: int, local=None, capacity_hint: int = 0, device: Optional[int] = None, group=None,
                 use_peer_exchange: bool = True):
        if not dist.is_initialized():
            raise RuntimeError("ShardedCorpus needs an initialised torch.distributed process group")
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        if self.world > 64:
            raise nat.PbxError(-1, "at most 64 shards")
        self.backend = dist.get_backend(group)
        self.dim = int(dim)
        # GPU shards: always with NCCL; with gloo when a device is named (two ranks sharing one GPU in the 1-GPU test:
        # NCCL refuses two ranks per device, the exchange over CUDA IPC mailboxes does not care)
        self.on_gpu = self.backend == "nccl" or (local is None and device is not None)
        if local is None and self.on_gpu:
            if device is None:
                device = torch.cuda.current_device()
            local = Corpus(dim, capacity_hint=capacity_hint, device=device)
        if local is None:
            raise nat.PbxError(-1, "ShardedCorpus on CPU (gloo) needs an injected `local` shard object")
        self.local = local
        self.device = device if device is not None else 0
        self._bufs = {}
        self._exchange = None
        if self.on_gpu and self.world > 1 and use_peer_exchange:
            self._connect_exchange()

    # -- exchange over NVLink peer memory ----------------------------------------------------------------
    MAX_RECORDS = 131072            # nq * k per call the mailboxes are sized for
    MAX_QUERIES = 1024

    def _connect_exchange(self) -> None:
        """Creates this rank's mailbox, all-gathers the CUDA IPC handles once (NCCL) and maps the peers' mailboxes.
        If peer mapping is not possible the NCCL all-gather + merge kernel path stays in use (same results)."""
        import ctypes
        L = nat.lib()
        h = ctypes.c_void_p(0)
        nat.check(L.pbx_exchange_create(self.device, self.rank, self.world, self.MAX_RECORDS, self.MAX_QUERIES, ctypes.byref(h)))
        mine = np.zeros(64, np.uint8)
        nat.check(L.pbx_exchange_handle(h, nat.ptr(mine)))
        handles = np.ascontiguousarray(self._all_gather_bytes(mine).reshape(-1))
        rc = L.pbx_exchange_connect(h, nat.ptr(handles))
        ok = torch.tensor([1 if rc == 0 else 0], dtype=torch.int32, device=self._comm_dev())
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)        # all ranks or none
        if int(ok.item()) == 1:
            self._exchange = h
        else:
            L.pbx_exchange_destroy(h)
        dist.barrier(group=self.group)

    def _comm_dev(self):
        """Device of the tensors handed to torch.distributed: the GPU with NCCL, the host with gloo."""
        return torch.device("cuda", self.device) if self.backend == "nccl" else torch.device("cpu")

    def _all_gather_bytes(self, mine: np.ndarray) -> np.ndarray:
        """[world][len(mine)] uint8: every rank's small host buffer (IPC handles)."""
        t_mine = torch.from_numpy(np.ascontiguousarray(mine)).to(self._comm_dev())
        t_all = torch.empty(self.world * t_mine.numel(), dtype=torch.uint8, device=self._comm_dev())
        if self.backend == "nccl":
            dist.all_gather_into_tensor(t_all, t_mine, group=self.group)
        else:
            parts = [torch.empty_like(t_mine) for _ in range(self.world)]
            dist.all_gather(parts, t_mine, group=self.group)
            t_all = torch.cat(parts)
        return t_all.cpu().numpy().reshape(self.world, -1)

    # -- contents ----------------------------------------------------------------------------------
    def load_table(self, image_ids, hashes) -> None:
        """Every rank passes the same table (rows ordered by image_id, as `SELECT image_id, hash FROM
        semantic_hashes ORDER BY image_id` yields them) and keeps its contiguous block."""
        first, count = shard_rows(len(image_ids), self.rank, self.world)
        self.local.load(np.asarray(image_ids)[first:first + count], np.asarray(hashes)[first:first + count])

    def fill_synthetic(self, rows_per_shard: int, seed: int) -> None:
        """Shard r holds global rows [r*rows_per_shard, (r+1)*rows_per_shard) of the synthetic corpus."""
        self.local.fill_synthetic(rows_per_shard, seed, self.rank * rows_per_shard)

    def remove(self, image_ids) -> int:
        """Every rank passes the same ids (they are global: any shard may hold them) and removes them from its shard;
        returns the number of rows removed over all ranks, on every rank."""
        mine = np.array([self.local.remove(image_ids)], np.int64)
        return int(self._all_gather_bytes(mine.view(np.uint8)).view(np.int64).sum())

    def replace(self, image_ids, hashes) -> int:
        """Every rank passes the same (ids, hashes) and replaces the hashes of the rows its shard holds; returns the number
        of rows written over all ranks, on every rank."""
        mine = np.array([self.local.replace(image_ids, hashes)], np.int64)
        return int(self._all_gather_bytes(mine.view(np.uint8)).view(np.int64).sum())

    def view(self, image_ids) -> "ShardedCorpus":
        """A ShardedCorpus over a view of every rank's shard (Corpus.view; every rank passes the same global ids).  It shares
        this corpus' process group and exchange, so its searches are the same collective calls with the same results as
        search(..., within=image_ids) here, at the cost of the view's rows.  close() it before this corpus."""
        if not isinstance(self.local, Corpus):
            raise nat.PbxError(-1, "a view needs GPU shards")
        v = ShardedCorpus.__new__(ShardedCorpus)
        v.__dict__.update(self.__dict__)
        v.local = self.local.view(image_ids)
        v._bufs = {}
        v._view_of = self
        return v

    def view_add(self, image_ids) -> int:
        """Corpus.view_add on every rank's view; returns the rows added over all ranks, on every rank."""
        mine = np.array([self.local.view_add(image_ids)], np.int64)
        return int(self._all_gather_bytes(mine.view(np.uint8)).view(np.int64).sum())

    def view_drop(self, image_ids) -> int:
        """Corpus.view_drop on every rank's view; returns the rows dropped over all ranks, on every rank."""
        mine = np.array([self.local.view_drop(image_ids)], np.int64)
        return int(self._all_gather_bytes(mine.view(np.uint8)).view(np.int64).sum())

    def total_rows(self) -> int:
        t = torch.tensor([len(self.local)], dtype=torch.int64, device=self._comm_dev())
        dist.all_reduce(t, group=self.group)
        return int(t.item())

    def _dev(self):
        return torch.device("cuda", self.device) if self.on_gpu else torch.device("cpu")

    # -- search ------------------------------------------------------------------------------------
    def _buffers(self, nq: int, k: int):
        key = (nq, k)
        if key not in self._bufs:
            dev = self._dev()
            self._bufs[key] = dict(
                q=torch.empty(nq * self.dim, dtype=torch.uint8, device=dev),
                hq=torch.empty(nq * self.dim, dtype=torch.uint8).pin_memory() if self.on_gpu else None,
                local=torch.empty(nq * k * HIT_BYTES, dtype=torch.uint8, device=dev),
                cnt=torch.empty(nq, dtype=torch.int32, device=dev),
                gathered=torch.empty(self.world * nq * k * HIT_BYTES, dtype=torch.uint8, device=dev),
                out=torch.empty(nq * k * HIT_BYTES, dtype=torch.uint8, device=dev),
                out_cnt=torch.empty(nq, dtype=torch.int32, device=dev),
                h_out=torch.empty(nq * k * HIT_BYTES, dtype=torch.uint8).pin_memory() if self.on_gpu else None,
                h_cnt=torch.empty(nq, dtype=torch.int32).pin_memory() if self.on_gpu else None,
            )
        return self._bufs[key]

    def search_device(self, d_queries: torch.Tensor, nq: int, k: int, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None,
                      excluding=None, after=None):
        """Device-resident sharded search on the current torch stream, no host synchronisation:
        local search -> exchange of the [nq][k] records + merge (one kernel over peer memory, or NCCL
        all-gather + merge kernel).  Returns (hits, counts) device tensors (uint8 view of pbx_hit
        records, int32).  within / excluding: global image ids as in Corpus.search (every rank passes the same
        ones); each shard searches its allowed rows exactly, so the merge gives the filtered result of the table.
        after: cursors as in Corpus.search (every rank passes the same ones); each shard returns its next k rows after
        the same global cursor, so the merge gives the table's next page."""
        assert self.on_gpu
        b = self._buffers(nq, k)
        stream = torch.cuda.current_stream().cuda_stream
        if after is not None:
            fids, mode = nat.page_filter_args(within, excluding)
            d_fids = torch.from_numpy(np.unique(fids)).to(self._dev())
            d_after = torch.from_numpy(nat.page_cursors(after, nq).view(np.uint8)).to(self._dev())
            self.local.search_device_page(d_queries.data_ptr(), nq, k, max_dist, b["local"].data_ptr(), b["cnt"].data_ptr(),
                                          d_after.data_ptr(), d_fids.data_ptr() if d_fids.numel() else 0, d_fids.numel(), mode, stream)
        elif within is not None or excluding is not None:
            fids, mode = nat.filter_args(within, excluding)
            d_fids = torch.from_numpy(np.unique(fids)).to(self._dev())          # the device form wants them sorted
            self.local.search_device_filtered(d_queries.data_ptr(), nq, k, max_dist, b["local"].data_ptr(), b["cnt"].data_ptr(),
                                              d_fids.data_ptr(), d_fids.numel(), mode, stream)
        else:
            self.local.search_device(d_queries.data_ptr(), nq, k, max_dist, b["local"].data_ptr(), b["cnt"].data_ptr(), stream)
        if self.world == 1:
            return b["local"], b["cnt"]
        if self._exchange is not None and nq * k <= self.MAX_RECORDS and nq <= self.MAX_QUERIES:
            # one kernel: post to every peer's mailbox over NVLink, signal, wait, merge
            nat.check(nat.lib().pbx_exchange_allgather_merge(self._exchange, b["local"].data_ptr(), nq, k, b["out"].data_ptr(),
                                                             b["out_cnt"].data_ptr(), stream if stream else 1))
            return b["out"], b["out_cnt"]
        if self.backend == "nccl":
            dist.all_gather_into_tensor(b["gathered"], b["local"], group=self.group)
        else:                                   # gloo has no device all-gather: stage the records through the host
            torch.cuda.current_stream().synchronize()
            parts = [torch.empty(b["local"].numel(), dtype=torch.uint8) for _ in range(self.world)]
            dist.all_gather(parts, b["local"].cpu(), group=self.group)
            b["gathered"].copy_(torch.cat(parts))
        nat.check(nat.lib().pbx_merge_hits_device(self.device, b["gathered"].data_ptr(), None, self.world, nq, k,
                                                  b["out"].data_ptr(), b["out_cnt"].data_ptr(), stream if stream else 1))
        return b["out"], b["out_cnt"]

    def search(self, queries, k: int = nat.DEFAULT_K, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None,
               excluding=None, after=None) -> List[SearchResult]:
        """Host buffers in, host buffers out, on every rank (all ranks pass the same queries, and the same
        within / excluding image ids and after cursors: see Corpus.search)."""
        filtered = within is not None or excluding is not None
        if filtered:
            fids, mode = nat.filter_args(within, excluding)
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.uint8))
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise nat.PbxError(-2, f"search: expected [nq][{self.dim}] bytes, got {tuple(q.shape)}")
        nq = q.shape[0]
        if self.on_gpu and self._exchange is not None and nq * k <= self.MAX_RECORDS and nq <= self.MAX_QUERIES:
            # the whole step inside the library: H2D, local search, exchange + merge kernel, D2H, one synchronisation
            hits = np.empty((nq, k), nat.HIT_DTYPE)
            cnt = np.empty(nq, np.uint32)
            if after is not None:
                fids, mode = nat.page_filter_args(within, excluding)
                cur = nat.page_cursors(after, nq)
                nat.check(nat.lib().pbx_exchange_search_hits_page(self._exchange, self.local.handle, nat.ptr(q), nq, int(k), float(max_dist),
                                                                  nat.ptr(cur), nat.ptr(fids), fids.size, mode, nat.ptr(hits),
                                                                  nat.ptr(cnt)))
            elif filtered:
                nat.check(nat.lib().pbx_exchange_search_hits_filtered(self._exchange, self.local.handle, nat.ptr(q), nq, int(k),
                                                                      float(max_dist), nat.ptr(hits), nat.ptr(cnt), nat.ptr(fids),
                                                                      fids.size, mode))
            else:
                nat.check(nat.lib().pbx_exchange_search_hits(self._exchange, self.local.handle, nat.ptr(q), nq, int(k), float(max_dist),
                                                             nat.ptr(hits), nat.ptr(cnt)))
        elif self.on_gpu:
            b = self._buffers(nq, k)
            b["hq"].copy_(torch.from_numpy(q.reshape(-1)))
            b["q"].copy_(b["hq"], non_blocking=True)
            d_hits, d_cnt = self.search_device(b["q"], nq, k, max_dist, within=within, excluding=excluding, after=after)
            b["h_out"].copy_(d_hits, non_blocking=True)
            b["h_cnt"].copy_(d_cnt, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            hits = b["h_out"].numpy().view(nat.HIT_DTYPE).reshape(nq, k)
            cnt = b["h_cnt"].numpy().astype(np.uint32)
            if (cnt == 0xFFFFFFFF).any():
                raise nat.PbxError(-8, "peer exchange timed out: a rank did not post its records")
        elif filtered or after is not None:
            raise nat.PbxError(-1, "filtered or paged search needs GPU shards")
        else:
            l_hits, l_cnt = self.local.search_hits(q, k, max_dist)
            mine = torch.from_numpy(np.ascontiguousarray(l_hits).view(np.uint8).reshape(-1).copy())
            mine_cnt = torch.from_numpy(l_cnt.astype(np.int32))
            g_hits = [torch.empty_like(mine) for _ in range(self.world)]
            g_cnt = [torch.empty_like(mine_cnt) for _ in range(self.world)]
            dist.all_gather(g_hits, mine, group=self.group)
            dist.all_gather(g_cnt, mine_cnt, group=self.group)
            gathered = np.stack([t.numpy().view(nat.HIT_DTYPE).reshape(nq, k) for t in g_hits])
            counts = np.stack([t.numpy().astype(np.uint32) for t in g_cnt])
            hits, cnt = merge_hits(gathered, counts, k)
        return [SearchResult(hits[i]["image_id"][:cnt[i]].copy(), hits[i]["dist"][:cnt[i]].copy(),
                             hits[i]["dot"][:cnt[i]].copy(), hits[i]["norm2"][:cnt[i]].copy()) for i in range(nq)]

    def _all_gather_i64(self, values) -> np.ndarray:
        """[world][len(values)] int64 of every rank's values."""
        mine = np.ascontiguousarray(np.asarray(values, dtype=np.int64).reshape(-1))
        return self._all_gather_bytes(mine.view(np.uint8)).view(np.int64).reshape(self.world, -1)

    def count_within(self, queries, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None, excluding=None, after=None) -> np.ndarray:
        """Corpus.count_within over the table (every rank passes the same arguments): the shards' counts, summed."""
        if not isinstance(self.local, Corpus):
            raise nat.PbxError(-1, "a range search needs GPU shards")
        mine = self.local.count_within(queries, max_dist, within=within, excluding=excluding, after=after)
        return self._all_gather_i64(mine.astype(np.int64)).sum(axis=0).astype(np.uint64)

    def search_range(self, queries, max_dist: float = nat.DEFAULT_MAX_DIST, *, limit: Optional[int] = None, within=None,
                     excluding=None, after=None) -> List[RangeResult]:
        """Corpus.search_range over the table (every rank passes the same arguments), on every rank: each shard's range
        search, an all-gather of the totals and of the shards' first rows (each padded to the same length with dist =
        +inf), then the merge kernel on this rank's device.  The first `limit` rows of the table lie among the first
        `limit` rows of each shard, so the merge is exact."""
        if not isinstance(self.local, Corpus):
            raise nat.PbxError(-1, "a range search needs GPU shards")
        local = self.local.search_range(queries, max_dist, limit=limit, within=within, excluding=excluding, after=after)
        nq = len(local)
        g = self._all_gather_i64([r.total for r in local] + [len(r.ids) for r in local])
        totals, lens = g[:, :nq].sum(axis=0), g[:, nq:]
        out = []
        for i, r in enumerate(local):
            k = int(lens[:, i].sum()) if limit is None else min(int(limit), int(lens[:, i].sum()))
            if k == 0:
                e = np.zeros(0, nat.HIT_DTYPE)
                out.append(RangeResult(e["image_id"], e["dist"], e["dot"], e["norm2"], int(totals[i])))
                continue
            mine = np.zeros(k, nat.HIT_DTYPE)
            mine["image_id"], mine["dist"] = np.iinfo(np.int64).max, np.inf      # padding: no row has dist = +inf
            m = min(len(r.ids), k)
            mine["image_id"][:m], mine["dist"][:m], mine["dot"][:m], mine["norm2"][:m] = r.ids[:m], r.dist[:m], r.dot[:m], r.norm2[:m]
            gathered = torch.from_numpy(self._all_gather_bytes(mine.view(np.uint8)).reshape(-1)).to(self._dev())
            merged = torch.empty(k * HIT_BYTES, dtype=torch.uint8, device=self._dev())
            cnt = torch.empty(1, dtype=torch.int32, device=self._dev())
            stream = torch.cuda.current_stream().cuda_stream
            nat.check(nat.lib().pbx_merge_hits_device(self.device, gathered.data_ptr(), None, self.world, 1, k, merged.data_ptr(),
                                                      cnt.data_ptr(), stream if stream else 1))
            hits = merged.cpu().numpy().view(nat.HIT_DTYPE)[:int(cnt.cpu().item())]
            out.append(RangeResult(hits["image_id"].copy(), hits["dist"].copy(), hits["dot"].copy(), hits["norm2"].copy(),
                                   int(totals[i])))
        return out

    def close(self) -> None:
        if getattr(self, "_view_of", None) is not None:     # a view: the exchange belongs to the corpus it views
            self.local.close()
            return
        if self._exchange is not None:
            torch.cuda.synchronize()
            dist.barrier(group=self.group)                 # nobody may still be writing into a mailbox that goes away
            nat.lib().pbx_exchange_destroy(self._exchange)
            self._exchange = None
        if isinstance(self.local, Corpus):
            self.local.close()
