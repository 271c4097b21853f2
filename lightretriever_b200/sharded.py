"""Row-sharded flat inner-product search across the GPUs of one box (one process per GPU).

The reference shards the corpus with Faiss ``GpuMultipleClonerOptions.shard = True`` and merges per-shard results on
the host (retriever/faiss_index.py:60-70), and additionally walks the corpus in chunks merged by a Python heap
(retriever/hybrid_search.py:301-344, 182-205).  Here every rank keeps one contiguous shard resident in HBM, runs the
fused scoring/top-k kernel on it, and only the per-shard top-k candidate keys ([Q, k] u64 = 8 bytes per candidate,
ids already global) cross NVLink: one ``all_gather_into_tensor`` (NCCL) followed by the on-device merge kernel.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.distributed as dist

from .filters import DocDeletions


def shard_range(n_total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous row shard [lo, hi) of rank `rank`; sizes differ by at most one row."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad rank/world {rank}/{world}")
    return (n_total * rank) // world, (n_total * (rank + 1)) // world


def exchange_candidates(local_keys: torch.Tensor, group=None) -> torch.Tensor:
    """all-gather of the per-shard candidate keys: [Q, k] int64 -> [world, Q, k] (same on every rank)."""
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    local_keys = local_keys.contiguous()
    if world == 1:
        return local_keys.unsqueeze(0)
    out = torch.empty((world,) + tuple(local_keys.shape), dtype=local_keys.dtype, device=local_keys.device)
    if local_keys.device.type == "cuda":
        dist.all_gather_into_tensor(out, local_keys, group=group)
    else:  # gloo (CPU tests of the host logic)
        parts = [torch.empty_like(local_keys) for _ in range(world)]
        dist.all_gather(parts, local_keys, group=group)
        out = torch.stack(parts, dim=0)
    return out


class ShardedFlatIPIndex(DocDeletions):
    """One shard per rank; ``search_device`` returns the exact global top-k on every rank.  Same search surface as
    ``FlatIPIndex`` (``search_device / search_keys / search / reset``), so the searchers use either.  ``delete`` /
    ``restore`` take global ids (passage ids when ``_passage_ids`` is set): every rank applies the same call to its
    replicated bitmap of all ``n_total`` documents, with no collective, and passes it to its shard's search."""

    def __init__(self, dim: int, n_total: int, device: Optional[torch.device] = None, group=None, id_base: int = 0):
        from .search import FlatIPIndex  # requires the CUDA library

        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.n_total = int(n_total)
        self.dim = dim
        self.id_offset = int(id_base)  # id of global row 0 (a chunk of a larger corpus starts at its first row)
        self.lo, self.hi = shard_range(self.n_total, self.rank, self.world)
        if self.id_offset + self.n_total >= (1 << 32) - 2:
            raise ValueError("global ids must stay below 2^32")
        self.local = FlatIPIndex(dim, device=device, id_offset=self.id_offset + self.lo)
        self.local.reserve(self.hi - self.lo)
        self._passage_ids = None
        self.device = self.local.device
        self._live = None

    def _live_rows(self) -> int:
        return self.n_total

    @property
    def ntotal(self) -> int:
        return self.n_total

    def add_local(self, emb) -> None:
        """Append rows of this rank's shard (global row ids lo .. hi-1, in order)."""
        if self.local.ntotal + emb.shape[0] > self.hi - self.lo:
            raise ValueError("more rows than this rank's shard holds")
        if emb.shape[0]:
            self.local.add(emb)

    def search_keys(self, query, k: int, d_used: Optional[int] = None, **filters) -> torch.Tensor:
        """``filters``: ``live`` (replaces the index's own bitmap) / ``allow`` / ``q_filter`` over global ids."""
        from .search import flatip_topk_sharded

        if self.local.ntotal != self.hi - self.lo:
            raise RuntimeError(f"shard incomplete: {self.local.ntotal} of {self.hi - self.lo} rows")
        if filters.get("live") is None:
            filters["live"] = self._live
        if self.world == 1:
            return self.local.search_keys(query, k, d_used=d_used, **filters)
        if self.hi == self.lo:  # more ranks than rows: this rank contributes empty lists to both exchanges
            keys = torch.zeros((query.shape[0], k), dtype=torch.int64, device=self.local.device)
            self._merge_across(keys)
        else:
            # shared warm start: every rank scores 1/world of the prefix; the k-th best of the union seeds all of them
            keys = flatip_topk_sharded(self.local._query(query), self.local.corpus, k, self.world, self._merge_across,
                                       d_used=d_used, id_offset=self.local.id_offset, **filters)[2]
        return self._merge_across(keys)

    def _merge_across(self, keys: torch.Tensor) -> torch.Tensor:
        """all-gather of per-rank sorted keys [Q, k] + on-device merge -> the global sorted keys [Q, k] on every rank."""
        from .search import topk_merge

        gathered = exchange_candidates(keys, self.group)  # [world, Q, k]
        return topk_merge(gathered, keys.shape[1], return_keys=True)[2]

    def search_device(self, query, k: int, d_used: Optional[int] = None, return_keys: bool = False, **filters):
        from .search import decode_keys

        keys = self.search_keys(query, k, d_used=d_used, **filters)
        s, i = decode_keys(keys)
        return (s, i, keys) if return_keys else (s, i)

    def search(self, query_embeddings, k: int, **kwargs):
        """FaissIndex.search arrays (faiss_index.py:27-40) of the global result, identical on every rank."""
        import numpy as np

        s, i = self.search_device(query_embeddings, k)
        s, i = s.cpu().numpy(), i.cpu().numpy()
        if self._passage_ids is not None:
            valid = i >= 0
            i = np.where(valid, self._passage_ids[np.where(valid, i - self.id_offset, 0)], -1)
        return s, i

    def reset(self) -> None:
        self.local.reset()
        self._live = None


class ShardedImpactIndex(DocDeletions):
    """Document-sharded sparse impact index: the sparse twin of ``ShardedFlatIPIndex`` (SURVEY §8e: "same for CSR postings
    — shard by doc, per-shard inverted index").  Rank r indexes documents ``[lo, hi)`` as its own token-major inverted index
    (local doc ids, ``id_offset = lo``); a search runs ``lr_sparse_score_topk`` on the shard and only the per-shard top-k
    keys ``[Q, k]`` u64 (integer score << 32 | ~global id) cross NVLink, then ``lr_topk_merge`` with integer scores.  The
    reference has no multi-GPU sparse path (Anserini is one JVM, retriever/anserini_search.py:143-216); the exchange is the
    one the dense path uses.  ``delete`` / ``restore`` take global ids; as for ``ShardedFlatIPIndex`` every rank keeps the
    same bitmap of all documents and applies the same calls, with no collective."""

    def __init__(self, vocab_size: int, n_total: int, device: Optional[torch.device] = None, group=None):
        from .sparse_search import ImpactIndex  # requires the CUDA library

        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.n_total = int(n_total)
        self.lo, self.hi = shard_range(self.n_total, self.rank, self.world)
        if self.n_total >= (1 << 32) - 2:
            raise ValueError("global ids must stay below 2^32")
        self.local = ImpactIndex(vocab_size, device=device, id_offset=self.lo)
        self.device = self.local.device
        self.id_offset = 0
        self._live = None

    def _live_rows(self) -> int:
        return self.n_total

    def add_local_csr(self, indptr, tok, imp) -> None:
        """Append documents of this rank's shard (global ids lo .. hi-1, in order) as doc-major CSR."""
        self.local.add_csr(indptr, tok, imp)
        if self.local.N > self.hi - self.lo:
            raise ValueError("more documents than this rank's shard holds")

    def search_device(self, q_indptr, q_tok, q_cnt, k: int, **filters):
        """``filters``: ``live`` (replaces the index's own bitmap) / ``allow`` / ``q_filter`` over global ids."""
        from . import _C
        from .search import topk_merge

        if self.local.N != self.hi - self.lo:
            raise RuntimeError(f"shard incomplete: {self.local.N} of {self.hi - self.lo} documents")
        if filters.get("live") is None:
            filters["live"] = self._live
        if self.world == 1:
            return self.local.search_device(q_indptr, q_tok, q_cnt, k, **filters)
        _, _, keys = self.local.search_device(q_indptr, q_tok, q_cnt, k, return_keys=True, **filters)
        gathered = exchange_candidates(keys, self.group)  # [world, Q, k]
        return topk_merge(gathered, k, score_kind=_C.LR_SCORE_U32)
