"""Row-sharded table across the GPUs of one NVSwitch box: one process per GPU.

SURVEY.md 8(e): rows are independent, so the table is partitioned by
``shard = mix64(id) mod G`` (balanced under upsert/delete churn); every rank receives the
full query batch, scans its shard, and only the k candidates per query are exchanged:
ONE ``all_gather`` of a result block per rank (ids | distance bits | counts, 292 B per
query at k=12), then the on-device merge (``orx_merge_topk_strided``, reading the gathered
buffer in place) with the same ordering contract
(distance ASC, NaN last, id ASC).  Distances are the canonical binary64 values, so shard
results are comparable bit for bit and the merged answer equals the single-GPU answer.

The local index and the merge are injectable so that the partition / exchange logic is
covered by world_size-2 ``gloo`` tests on CPU (tests/test_sharded_gloo.py).
"""
from __future__ import annotations

import os
from typing import Callable, Optional

import numpy as np
import torch
import torch.distributed as dist

from .engine import Index, _device_result, ids_to_array

_GOLD = np.uint64(0x9E3779B97F4A7C15)
_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)


def shard_of(ids: np.ndarray, world: int) -> np.ndarray:
    """``mix64(hi * GOLD ^ lo) mod world`` for ``uint64 [n, 2]`` ids -> int64 [n]."""
    ids = np.asarray(ids, dtype=np.uint64).reshape(-1, 2)
    with np.errstate(over="ignore"):
        z = ids[:, 0] * _GOLD ^ ids[:, 1]
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
        z = z ^ (z >> np.uint64(31))
    return (z % np.uint64(world)).astype(np.int64)


def pack_results(ids: torch.Tensor, dist_: torch.Tensor, counts: torch.Tensor) -> torch.Tensor:
    """[nq,k,2] int64 + [nq,k] float64 + [nq] int32 -> one int64 [nq, 3k+1] block (bit copies)."""
    nq, k = dist_.shape
    out = torch.empty((nq, 3 * k + 1), dtype=torch.int64, device=ids.device)
    out[:, :2 * k] = ids.reshape(nq, 2 * k)
    out[:, 2 * k:3 * k] = dist_.view(torch.int64)
    out[:, 3 * k] = counts.to(torch.int64)
    return out


def unpack_results(block: torch.Tensor, k: int):
    """inverse of :func:`pack_results` for a ``[..., nq, 3k+1]`` block."""
    ids = block[..., :2 * k].contiguous().reshape(*block.shape[:-1], k, 2)
    dist_ = block[..., 2 * k:3 * k].contiguous().view(torch.float64)
    counts = block[..., 3 * k].to(torch.int32).contiguous()
    return ids, dist_, counts


class ShardedIndex:
    """The table of one rank + the exchange step.  All ranks must call every method
    collectively with the same arguments (upsert/delete take the FULL batch and keep only
    the rows this rank owns, so no data-path collective is needed on the write side)."""

    def __init__(self, dtype: str = "fp32", capacity_per_rank: int = 0, device: Optional[int] = None,
                 group=None, local_index=None, merge_fn: Optional[Callable] = None):
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.local = local_index if local_index is not None else Index(dtype, capacity_per_rank, device)
        self._merge = merge_fn if merge_fn is not None else self.local.merge_topk
        self.gather_launches = 0
        self._plans = {}
        self._outs = {}
        # Exchange: "p2p" = the library's fused publish + merge over NVLink peer memory (default on
        # GPUs); "nccl" = all_gather + orx_merge_topk_strided (baseline, ORX_SHARD_EXCHANGE=nccl).
        self.exchange = "none" if self.world == 1 else "nccl"
        want = os.environ.get("ORX_SHARD_EXCHANGE", "p2p")
        if (self.world > 1 and want == "p2p" and isinstance(self.local, Index)
                and dist.get_backend(self.group) == "nccl"):
            self._connect_p2p()

    def _connect_p2p(self) -> None:
        dev = torch.device(f"cuda:{self.local.device}")
        handle = self.local.shard_export(self.world, self.rank)
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=dev)
        everyone = torch.empty(self.world * len(handle), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(everyone, mine, group=self.group)
        blob = everyone.cpu().numpy().tobytes()
        n = len(handle)
        ok = torch.ones(1, dtype=torch.int32, device=dev)
        try:
            self.local.shard_connect([blob[i * n:(i + 1) * n] for i in range(self.world)])
        except Exception as e:        # no peer access between these GPUs: every rank falls back together
            ok.zero_()
            self._p2p_error = str(e)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
        if int(ok.item()) == 1:
            self.exchange = "p2p"

    def _plan(self, nq: int, k: int, device):
        """Reusable device buffers for one (nq, k): my result block (the scan's output arrays are
        views of it), the gathered blocks of all ranks, and the merged result."""
        key = (nq, k, str(device))
        p = self._plans.get(key)
        if p is None:
            words = nq * k * 3 + (nq + 1) // 2                       # ids 2nk | dist nk | counts ceil(nq/2)
            block = torch.zeros(words, dtype=torch.int64, device=device)
            p = {
                "words": words, "block": block,
                "ids": block[:2 * nq * k].view(nq, k, 2),
                "dist": block[2 * nq * k:3 * nq * k].view(torch.float64).view(nq, k),
                "cnt": block[3 * nq * k:].view(torch.int32)[:nq],
                "gathered": torch.zeros(self.world * words, dtype=torch.int64, device=device),
                "out_ids": torch.zeros((nq, k, 2), dtype=torch.int64, device=device),
                "out_dist": torch.zeros((nq, k), dtype=torch.float64, device=device),
                "out_cnt": torch.zeros((nq,), dtype=torch.int32, device=device),
            }
            self._plans[key] = p
        return p

    def __len__(self) -> int:
        return len(self.local)

    def global_size(self) -> int:
        n = torch.tensor([len(self.local)], dtype=torch.int64)
        if self.world > 1:
            backend = dist.get_backend(self.group)
            if backend == "nccl":
                n = n.cuda()
            dist.all_reduce(n, group=self.group)
        return int(n.item())

    # ------------------------------------------------------------------ writes
    def _mine(self, ida: np.ndarray) -> np.ndarray:
        return np.nonzero(shard_of(ida, self.world) == self.rank)[0]

    def upsert(self, ids, vecs) -> int:
        ida = ids_to_array(ids)
        sel = self._mine(ida)
        if sel.size:
            v = vecs[torch.as_tensor(sel, device=vecs.device)] if isinstance(vecs, torch.Tensor) \
                else np.asarray(vecs, np.float32)[sel]
            self.local.upsert(ida[sel], v)
        return int(sel.size)

    def upsert_local(self, ids, vecs) -> None:
        """Rows the caller already knows belong to this rank (bulk load of a pre-partitioned table)."""
        self.local.upsert(ids, vecs)

    def delete(self, ids) -> int:
        ida = ids_to_array(ids)
        sel = self._mine(ida)
        return self.local.delete(ida[sel]) if sel.size else 0

    def load_pgcopy(self, chunks) -> tuple[int, int]:
        """Cold start of a row-sharded table: every rank feeds the SAME `COPY ... (FORMAT binary)` stream;
        the loader keeps the rows this rank owns (the C side applies `shard_of`).  No collective.
        -> (rows loaded on this rank, rows with a NULL embedding in the whole stream)."""
        return self.local.load_pgcopy(chunks, self.world, self.rank)

    # ------------------------------------------------------------------- reads
    def search(self, queries, k: int = 12):
        """Global top-k on every rank.  ``queries`` is identical on all ranks (CUDA tensor for the
        NCCL path; NumPy for the CPU/gloo test path).  On the CUDA path the returned tensors are
        reusable per-(nq, k) buffers: they are overwritten by the next search of the same shape."""
        if self.exchange == "p2p":
            if isinstance(queries, torch.Tensor) and queries.is_cuda:
                q = queries if queries.dim() == 2 else queries.unsqueeze(0)
                key = (q.shape[0], k)
                out = self._outs.get(key)
                if out is None:
                    out = self._outs[key] = _device_result(q.shape[0], k, q.device)
                return self.local.search_sharded(q, k, out)
            return self.local.search_sharded(queries, k)
        if self.world > 1 and isinstance(queries, torch.Tensor) and queries.is_cuda and hasattr(self.local, "search_into"):
            q = queries if queries.dim() == 2 else queries.unsqueeze(0)
            nq = q.shape[0]
            p = self._plan(nq, k, q.device)
            self.local.search_into(q, k, p["ids"], p["dist"], p["cnt"])
            dist.all_gather_into_tensor(p["gathered"], p["block"], group=self.group)
            self.gather_launches += 1
            self.local.merge_blocks(p["gathered"], self.world, nq, k, p["words"] * 8, p["out_ids"], p["out_dist"],
                                    p["out_cnt"])
            return p["out_ids"], p["out_dist"], p["out_cnt"]
        if self.world == 1 and isinstance(queries, torch.Tensor) and queries.is_cuda and isinstance(self.local, Index):
            q = queries if queries.dim() == 2 else queries.unsqueeze(0)
            key = (q.shape[0], k)
            out = self._outs.get(key)
            if out is None:
                out = self._outs[key] = _device_result(q.shape[0], k, q.device)
            return self.local.search(q, k, out=out)
        ids, dist_, cnt = self.local.search(queries, k)
        if self.world == 1:
            return ids, dist_, cnt
        return self._gather_merge(ids, dist_, cnt, k)

    # -- throughput mode: two searches in flight (device tensors only)
    def search_submit(self, queries, k: int = 12):
        """Launch a (collective) search of a float32 CUDA tensor and return `(ticket, out)`; `search_wait(ticket)`
        completes it and `out` = (ids, dist, counts) CUDA tensors is valid afterwards.  At most two tickets may be
        outstanding, waited for in submission order (on every rank alike).  The output tensors alternate between two
        cached sets per (nq, k): a result is overwritten by the submit after next."""
        q = queries if queries.dim() == 2 else queries.unsqueeze(0)
        self._submits = getattr(self, "_submits", 0)
        key = (q.shape[0], k, self._submits & 1)
        self._submits += 1
        out = self._outs.get(key)
        if out is None:
            out = self._outs[key] = _device_result(q.shape[0], k, q.device)
        if self.world > 1 and self.exchange != "p2p":
            raise RuntimeError("search_submit needs the peer-memory exchange (or a single rank)")
        return self.local.search_submit(q, k, out, sharded=self.world > 1), out

    def search_wait(self, ticket: int) -> None:
        self.local.search_wait(ticket)

    def search_filtered(self, queries, k: int, allow_ids):
        """COLLECTIVE filtered search (`WHERE langchain_id IN (...)`, see Index.search_filtered): every rank
        resolves the predicate against its own shard -- it is handed only the ids it owns -- and the k
        candidates per rank are exchanged and merged like `search`.  Host (NumPy) queries and results."""
        ida = ids_to_array(allow_ids)
        if self.world > 1:
            ida = ida[self._mine(ida)]
        ids, dist_, cnt = self.local.search_filtered(queries, k, ida)
        if self.world == 1:
            return ids, dist_, cnt
        return self._gather_merge(ids, dist_, cnt, k)

    def _gather_merge(self, ids, dist_, cnt, k: int):
        """One all_gather of the packed per-rank results + the merge; NumPy in -> NumPy out."""
        as_numpy = not isinstance(ids, torch.Tensor)
        if as_numpy:
            ids = torch.from_numpy(np.ascontiguousarray(ids).view(np.int64))
            dist_ = torch.from_numpy(np.ascontiguousarray(dist_))
            cnt = torch.from_numpy(np.ascontiguousarray(cnt))
        block = pack_results(ids, dist_, cnt)
        if not block.is_cuda and dist.get_backend(self.group) == "nccl":
            block = block.cuda(getattr(self.local, "device", None))      # NCCL moves device buffers only
        nq = block.shape[0]
        gathered = torch.empty((self.world * nq, block.shape[1]), dtype=torch.int64, device=block.device)
        dist.all_gather_into_tensor(gathered, block, group=self.group)   # rank-major concatenation
        gathered = gathered.view(self.world, nq, block.shape[1])
        self.gather_launches += 1
        g_ids, g_dist, g_cnt = unpack_results(gathered, k)
        if as_numpy:
            return self._merge(g_ids.cpu().numpy().view(np.uint64), g_dist.cpu().numpy(), g_cnt.cpu().numpy(), k)
        return self._merge(g_ids, g_dist, g_cnt, k)


__all__ = ["ShardedIndex", "shard_of", "pack_results", "unpack_results"]
