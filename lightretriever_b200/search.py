"""Exact flat inner-product search (K2) — host side, seam S2.

Mirrors
  * ``FaissIndex`` (reference retriever/faiss_index.py:20-73): ``build / search / to_gpu / reset / save``;
    ``search(q, k) -> (scores float32 [Q,k] descending, ids int64 [Q,k])``;
  * ``FlatIPFaissSearch`` / ``DenseRetrievalFaissSearch`` (retriever/faiss_search.py:46-293, 477-510):
    ``index(corpus_emb, corpus_ids)``, ``retrieve_with_emb(query_emb, query_ids, top_k)``, ``_clear()``, ``search``.
The corpus lives in HBM as bf16 rows; scoring + top-k is one fused tcgen05 kernel plus a merge
(csrc/umma_gemm.cuh, csrc/topk_merge.cu).  Results are device arrays first: a search yields sorted candidate keys
``[Q, k]`` (u64 = order-preserving score << 32 | ~id); chunk loops and shards combine them with ``lr_topk_merge`` and the
reference's nested dicts are built once, at the end, by ``arrays_to_dict``.  With ``use_multiple_gpu=True`` under an
initialised ``torch.distributed`` group every rank keeps one row shard (``sharded.ShardedFlatIPIndex``, the counterpart
of Faiss ``shard=True``, faiss_index.py:60-70).  Differences from Faiss that are part of the contract:
  * equal scores are ordered by ascending id (Faiss: unspecified);
  * when fewer than k documents exist the tail is (score -inf, id -1) and is dropped from result dicts
    (the reference lets numpy wrap id -1 to the last passage, SURVEY §8c trap 8).
"""
from __future__ import annotations

import csv
import logging
import struct
import os
import time
from typing import Optional, Sequence

import numpy as np
import torch

from . import _C
from ._util import Workspace, require_cuda, stream_ptr
from .filters import DocDeletions, filter_args

logger = logging.getLogger(__name__)

_WS = Workspace()


def _flatip_operands(query, corpus, d_used, q_scale, c_scale):
    q = require_cuda(query, "query")
    c = require_cuda(corpus, "corpus")
    if q.dtype != torch.bfloat16 or c.dtype != torch.bfloat16:
        raise ValueError("flatip_topk takes bfloat16 query and corpus (convert once at index / encode time)")
    if q.ndim != 2 or c.ndim != 2:
        raise ValueError("query and corpus must be 2-D")
    if q.stride(1) != 1:
        q = q.contiguous()
    if c.stride(1) != 1:
        c = c.contiguous()
    d = int(d_used) if d_used else min(q.shape[1], c.shape[1])
    if d_used is None and q.shape[1] != c.shape[1]:
        raise ValueError(f"dimension mismatch: query {q.shape[1]} vs corpus {c.shape[1]}")
    dev = q.device
    if c.device != dev:
        raise ValueError("query and corpus must be on the same device")
    for name, s, n in (("q_scale", q_scale, q.shape[0]), ("c_scale", c_scale, c.shape[0])):
        if s is not None and (s.dtype != torch.float32 or s.numel() != n or not s.is_contiguous() or s.device != dev):
            raise ValueError(f"{name} must be a contiguous float32 tensor with {n} elements on {dev}")
    return q, c, d, dev


def flatip_topk(query: torch.Tensor, corpus: torch.Tensor, k: int, d_used: Optional[int] = None,
                q_scale: Optional[torch.Tensor] = None, c_scale: Optional[torch.Tensor] = None,
                id_offset: int = 0, return_keys: bool = False, workspace: Optional[Workspace] = None,
                live: Optional[torch.Tensor] = None, allow: Optional[torch.Tensor] = None,
                q_filter: Optional[torch.Tensor] = None):
    """scores, ids (and optionally sorted u64 keys) of the k largest ``query @ corpus.T`` per query.

    query [Q, >=d_used] bf16, corpus [N, >=d_used] bf16, both on the same B200; rows may be strided views
    (e.g. an MRL prefix ``x[:, :m]`` of full-width vectors) as long as the inner stride is 1.
    ``live`` / ``allow`` / ``q_filter``: document bitmaps (``filters.py``); the result is the exact top-k of the allowed
    documents, with a (-inf, -1) tail when fewer than k are allowed.  All None = the unfiltered kernel path.
    """
    q, c, d, dev = _flatip_operands(query, corpus, d_used, q_scale, c_scale)
    Q, N = q.shape[0], c.shape[0]
    flt = filter_args(live, allow, q_filter, Q, dev)
    lib = _C.load()
    ws = (workspace or _WS).get(lib.lr_flatip_workspace_bytes_for(Q, N, k, d), dev)
    scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
    ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
    keys = torch.empty((Q, k), dtype=torch.int64, device=dev) if return_keys else None
    args = (q.data_ptr(), q.stride(0), c.data_ptr(), c.stride(0), Q, N, d,
            None if q_scale is None else q_scale.data_ptr(), None if c_scale is None else c_scale.data_ptr(),
            int(id_offset), int(k), scores.data_ptr(), ids.data_ptr(), None if keys is None else keys.data_ptr())
    with torch.cuda.device(dev):
        if flt is None:
            _C.check(lib.lr_flatip_topk(*args, ws.data_ptr(), ws.numel(), stream_ptr(dev)))
        else:
            _C.check(lib.lr_flatip_topk_filtered(*args, *flt, ws.data_ptr(), ws.numel(), stream_ptr(dev)))
    return (scores, ids, keys) if return_keys else (scores, ids)


def flatip_topk_sharded(query: torch.Tensor, corpus: torch.Tensor, k: int, n_shards: int, exchange,
                        d_used: Optional[int] = None, q_scale: Optional[torch.Tensor] = None,
                        c_scale: Optional[torch.Tensor] = None, id_offset: int = 0,
                        workspace: Optional[Workspace] = None, live: Optional[torch.Tensor] = None,
                        allow: Optional[torch.Tensor] = None, q_filter: Optional[torch.Tensor] = None):
    """One shard's part of a row-sharded search (Faiss ``shard=True``, faiss_index.py:60-70) with a SHARED warm start:
    ``lr_flatip_topk_begin`` scores this shard's 1/n_shards of the warm-start prefix, ``exchange(prefix_keys [Q,k])``
    returns the merged top-k keys of every shard's prefix (all-gather + ``lr_topk_merge``), and ``lr_flatip_topk_finish``
    runs the remaining passes with the k-th best score of the whole prefix as the starting threshold.  Returns
    (scores, ids, keys) of this shard; a row may hold fewer than k entries — only documents that can still reach the
    global top-k are kept.  ``live`` / ``allow`` / ``q_filter`` as in ``flatip_topk``: bitmaps over GLOBAL ids, the same
    (replicated) tensors on every shard."""
    q, c, d, dev = _flatip_operands(query, corpus, d_used, q_scale, c_scale)
    Q, N = q.shape[0], c.shape[0]
    flt = filter_args(live, allow, q_filter, Q, dev)
    lib = _C.load()
    ws = (workspace or _WS).get(lib.lr_flatip_workspace_bytes_sharded(Q, N, k, d, int(n_shards)), dev)
    scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
    ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
    keys = torch.empty((Q, k), dtype=torch.int64, device=dev)
    prefix_keys = torch.empty((Q, k), dtype=torch.int64, device=dev)
    qs = None if q_scale is None else q_scale.data_ptr()
    cs = None if c_scale is None else c_scale.data_ptr()
    tail = (ws.data_ptr(), ws.numel(), stream_ptr(dev))
    with torch.cuda.device(dev):
        if flt is None:
            _C.check(lib.lr_flatip_topk_begin(q.data_ptr(), q.stride(0), c.data_ptr(), c.stride(0), Q, N, d, qs, cs,
                                              int(k), int(n_shards), prefix_keys.data_ptr(), *tail))
        else:
            _C.check(lib.lr_flatip_topk_begin_filtered(q.data_ptr(), q.stride(0), c.data_ptr(), c.stride(0), Q, N, d, qs,
                                                       cs, int(id_offset), int(k), int(n_shards), prefix_keys.data_ptr(),
                                                       *flt, *tail))
        seed = exchange(prefix_keys)
        if seed is not None:
            if seed.shape != (Q, k) or seed.dtype != torch.int64 or not seed.is_contiguous() or seed.device != dev:
                raise ValueError("exchange() must return contiguous int64 [Q, k] keys on the search device")
        args = (q.data_ptr(), q.stride(0), c.data_ptr(), c.stride(0), Q, N, d, qs, cs, int(id_offset), int(k),
                int(n_shards), None if seed is None else seed.data_ptr(), scores.data_ptr(), ids.data_ptr(),
                keys.data_ptr())
        if flt is None:
            _C.check(lib.lr_flatip_topk_finish(*args, *tail))
        else:
            _C.check(lib.lr_flatip_topk_finish_filtered(*args, *flt, *tail))
    return scores, ids, keys


def flatip_scores(query: torch.Tensor, corpus: torch.Tensor, d_used: Optional[int] = None) -> torch.Tensor:
    """Full [Q, N] f32 score matrix through the same TMA + tcgen05 main loop (parity/debug; small shapes)."""
    q = require_cuda(query, "query")
    c = require_cuda(corpus, "corpus")
    if q.dtype != torch.bfloat16 or c.dtype != torch.bfloat16:
        raise ValueError("flatip_scores takes bfloat16 inputs")
    d = int(d_used) if d_used else q.shape[1]
    out = torch.empty((q.shape[0], c.shape[0]), dtype=torch.float32, device=q.device)
    lib = _C.load()
    with torch.cuda.device(q.device):
        _C.check(lib.lr_flatip_scores(q.data_ptr(), q.stride(0), c.data_ptr(), c.stride(0), q.shape[0], c.shape[0], d,
                                      out.data_ptr(), stream_ptr(q.device)))
    return out


def topk_merge(keys: torch.Tensor, k: int, counts: Optional[torch.Tensor] = None, score_kind: int = _C.LR_SCORE_F32,
               id_offset: int = 0, return_keys: bool = False):
    """Exact top-k of L candidate lists per query.  keys: int64/uint64-bit [L, Q, cap] (0 = empty slot), contiguous or a
    view whose lists are spaced by a whole number of query rows: strides (q_stride * cap, cap, 1) with q_stride >= Q, e.g.
    ``gathered[:, s]`` of a ``[L, S, Q, cap]`` exchange that carries S systems at once."""
    keys = require_cuda(keys, "keys")
    if keys.ndim != 3 or keys.dtype != torch.int64:
        raise ValueError("keys must be an int64 [L, Q, cap] tensor of candidate keys")
    L, Q, cap = keys.shape
    q_stride = Q
    if not keys.is_contiguous():
        s0, s1, s2 = keys.stride()
        if s2 != 1 or s1 != cap or s0 % cap or s0 // cap < Q or counts is not None:
            raise ValueError("keys must be a contiguous int64 [L, Q, cap] tensor of candidate keys, or a view with "
                             "strides (q_stride * cap, cap, 1), q_stride >= Q (without counts)")
        q_stride = s0 // cap
    dev = keys.device
    if counts is not None:
        counts = counts.to(torch.int32).contiguous()
        if counts.shape != (L, Q) or counts.device != dev:
            raise ValueError("counts must be [L, Q] on the keys' device")
    scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
    ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
    okeys = torch.empty((Q, k), dtype=torch.int64, device=dev) if return_keys else None
    lib = _C.load()
    with torch.cuda.device(dev):
        _C.check(lib.lr_topk_merge(keys.data_ptr(), None if counts is None else counts.data_ptr(), L, Q, q_stride, cap, int(k),
                                   score_kind, int(id_offset), scores.data_ptr(), ids.data_ptr(),
                                   None if okeys is None else okeys.data_ptr(), stream_ptr(dev)))
    return (scores, ids, okeys) if return_keys else (scores, ids)


def encode_keys(scores: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    scores = require_cuda(scores, "scores").to(torch.float32).contiguous()
    ids = require_cuda(ids, "ids").to(torch.int64).contiguous()
    keys = torch.empty(scores.shape, dtype=torch.int64, device=scores.device)
    lib = _C.load()
    with torch.cuda.device(scores.device):
        _C.check(lib.lr_encode_keys(scores.data_ptr(), ids.data_ptr(), scores.numel(), keys.data_ptr(),
                                    stream_ptr(scores.device)))
    return keys


def decode_keys(keys: torch.Tensor, score_kind: int = _C.LR_SCORE_F32):
    """Sorted candidate keys [Q, k] -> (scores f32 [Q, k], ids i64 [Q, k]); empty slots become (-inf, -1)."""
    return topk_merge(keys.unsqueeze(0).contiguous(), keys.shape[1], score_kind=score_kind)


def merge_keys(key_lists: Sequence[torch.Tensor], k: int, score_kind: int = _C.LR_SCORE_F32) -> torch.Tensor:
    """Exact top-k (as sorted keys [Q, k]) of the union of several per-query key lists [Q, k_i] with global ids: the
    device form of the reference's heap merge (hybrid_search.py:182-205).  Lists may have different widths."""
    width = max(t.shape[1] for t in key_lists)
    stack = torch.zeros((len(key_lists), key_lists[0].shape[0], width), dtype=torch.int64, device=key_lists[0].device)
    for l, t in enumerate(key_lists):
        stack[l, :, :t.shape[1]] = t
    return topk_merge(stack, k, score_kind=score_kind, return_keys=True)[2]


def drop_identical(keys: torch.Tensor, self_pos: torch.Tensor) -> torch.Tensor:
    """`ignore_identical_ids` (hybrid_search.py:193): the candidate whose id equals the query's own corpus position
    (self_pos [Q] i64, -1 = the query is not a corpus document) becomes an empty slot."""
    ids = 0xFFFFFFFF - (keys & 0xFFFFFFFF)
    return torch.where((ids == self_pos.to(keys.device)[:, None]) & (keys != 0), torch.zeros_like(keys), keys)


_FAISS_FLAT_IP = 0x49467849  # fourcc("IxFI")
_FAISS_HEADER = struct.Struct("<Iiqqq?iQ")  # fourcc, d, ntotal, dummy, dummy, is_trained, metric_type, n_floats


class FlatIPIndex(DocDeletions):
    """HBM-resident flat inner-product index with the ``FaissIndex`` surface (faiss_index.py:20-73).  ``delete(ids)`` /
    ``restore(ids)`` (``DocDeletions``) hide documents from every later search without touching their rows."""

    def __init__(self, dim: Optional[int] = None, passage_ids: Optional[Sequence[int]] = None,
                 device: Optional[torch.device] = None, id_offset: int = 0):
        self.dim = dim
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._buf: Optional[torch.Tensor] = None  # [capacity, dim] bf16; rows [0, _n) are filled
        self._n = 0
        self._passage_ids = None if passage_ids is None else np.asarray(passage_ids, dtype=np.int64)
        self.id_offset = int(id_offset)
        self._live = None

    def _live_rows(self) -> int:
        return self._n

    def reserve(self, n_rows: int) -> None:
        """Size the resident buffer up front so that ``add`` copies every chunk straight into place: no concatenation
        and no second copy of the shard (a 72 GB corpus must not peak at 144 GB)."""
        if self.dim is None:
            raise ValueError("reserve() needs the dimension")
        if self._buf is not None and self._buf.shape[0] >= n_rows:
            return
        new = torch.empty((int(n_rows), self.dim), dtype=torch.bfloat16, device=self.device)
        if self._n:
            new[:self._n] = self._buf[:self._n]
        self._buf = new

    # faiss.IndexFlatIP.add
    def add(self, emb) -> None:
        t = emb if isinstance(emb, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(emb))
        if t.ndim != 2:
            raise ValueError("embeddings must be [n, d]")
        if self.dim is None:
            self.dim = t.shape[1]
        if t.shape[1] != self.dim:
            raise ValueError(f"dimension mismatch: index {self.dim}, got {t.shape[1]}")
        need = self._n + t.shape[0]
        if self._buf is None or self._buf.shape[0] < need:  # not reserved: grow geometrically (amortised copies)
            self.reserve(max(need, 2 * self._n))
        self._buf[self._n:need].copy_(t, non_blocking=True)  # dtype conversion (-> bf16) happens in the copy
        old, self._n = self._n, need
        self._extend_live(old)

    @property
    def ntotal(self) -> int:
        return self._n

    @property
    def corpus(self) -> torch.Tensor:
        if self._n == 0:
            raise RuntimeError("index is empty")
        return self._buf[:self._n]

    @classmethod
    def build(cls, passage_ids: Sequence[int], passage_embeddings, index: Optional["FlatIPIndex"] = None,
              buffer_size: int = 50000) -> "FlatIPIndex":
        if index is None:
            index = cls(passage_embeddings.shape[1])
        if index.dim is None:
            index.dim = passage_embeddings.shape[1]
        n_rows = passage_embeddings.shape[0]
        if passage_ids is not None and len(passage_ids) != n_rows:
            raise ValueError(f"{len(passage_ids)} passage ids for {n_rows} embeddings")
        index.reserve(index.ntotal + n_rows)
        for start in range(0, n_rows, buffer_size):
            index.add(passage_embeddings[start:start + buffer_size])
        # passage_ids None: results are row positions (+ id_offset), the form chunk loops and shards exchange
        index._passage_ids = None if passage_ids is None else np.asarray(passage_ids, dtype=np.int64)
        return index

    def _query(self, query_embeddings) -> torch.Tensor:
        q = query_embeddings
        if not isinstance(q, torch.Tensor):
            q = torch.from_numpy(np.ascontiguousarray(q))
        return q.to(device=self.device, dtype=torch.bfloat16, non_blocking=True)

    def search_device(self, query_embeddings, k: int, d_used: Optional[int] = None, live: Optional[torch.Tensor] = None,
                      **kw):
        """``flatip_topk`` over the resident rows.  ``live`` replaces the index's own deletions bitmap for this call;
        ``allow`` / ``q_filter`` (keywords) restrict queries to subsets."""
        return flatip_topk(self._query(query_embeddings), self.corpus, k, d_used=d_used, id_offset=self.id_offset,
                           live=self._live if live is None else live, **kw)

    def search_keys(self, query_embeddings, k: int, d_used: Optional[int] = None, **kw) -> torch.Tensor:
        """Sorted candidate keys [Q, k] with ids offset by ``id_offset`` (what shards and chunk loops exchange)."""
        return self.search_device(query_embeddings, k, d_used=d_used, return_keys=True, **kw)[2]

    def search(self, query_embeddings, k: int, **kwargs) -> tuple[np.ndarray, np.ndarray]:
        num_queries = query_embeddings.shape[0]
        start_time = time.time()
        scores, ids = self.search_device(query_embeddings, k)
        scores_arr = scores.cpu().numpy()
        ids_arr = ids.cpu().numpy()
        if self._passage_ids is not None:
            valid = ids_arr >= 0
            mapped = self._passage_ids[np.where(valid, ids_arr - self.id_offset, 0).reshape(-1)].reshape(num_queries, -1)
            ids_arr = np.where(valid, mapped, -1)
        total_time = time.time() - start_time
        logger.info("Num of queries: %d\tSearch time (s): %.3f\tQPS: %.3f", num_queries, total_time,
                    num_queries / max(total_time, 1e-9))
        return scores_arr, ids_arr

    def to_gpu(self, group=None):
        """faiss_index.py:60-70.  The rows are already in HBM; under an initialised process group with more than one rank
        the index becomes this rank's shard of a ``ShardedFlatIPIndex`` (the counterpart of Faiss ``shard=True``): every
        rank must hold the same rows when calling this, and each keeps ``[lo, hi)``."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return self
        from .sharded import ShardedFlatIPIndex

        sh = ShardedFlatIPIndex(self.dim, self.ntotal, device=self.device, group=group, id_base=self.id_offset)
        sh.add_local(self.corpus[sh.lo:sh.hi])
        sh._passage_ids = self._passage_ids
        self.reset()
        return sh

    def reset(self) -> None:
        self._buf = None
        self._n = 0
        self._live = None

    # ---- persistent format: the file faiss.write_index writes for an IndexFlatIP (faiss_index.py:42-43,
    #      faiss_search.py:113-123, 477-488): fourcc "IxFI", d, ntotal, two dummies, is_trained, metric_type (0 = inner
    #      product), then the row-major fp32 vectors as a length-prefixed array.  Restated from Faiss's index_write.cpp
    #      (Faiss itself is not installed here: the round trip below is self-consistent, not pinned against Faiss).
    def save(self, fname: str, rows_per_write: int = 1 << 16) -> None:
        if self.n_live != self.ntotal:
            # the Faiss file has no tombstones: writing the rows would resurrect the deleted documents on reload
            raise ValueError(f"the index holds {self.ntotal - self.n_live} deleted documents, which the Faiss IndexFlatIP "
                             "file cannot record; restore them or rebuild the index without them before saving")
        n, d = self.ntotal, int(self.dim)
        with open(fname, "wb") as f:
            f.write(_FAISS_HEADER.pack(_FAISS_FLAT_IP, d, n, 1 << 20, 1 << 20, True, 0, n * d))
            for lo in range(0, n, rows_per_write):
                f.write(self._buf[lo:min(lo + rows_per_write, n)].float().cpu().numpy().tobytes())

    @classmethod
    def load(cls, fname: str, passage_ids: Optional[Sequence[int]] = None, device: Optional[torch.device] = None,
             rows: Optional[tuple[int, int]] = None, id_offset: int = 0, rows_per_read: int = 1 << 16) -> "FlatIPIndex":
        """Read a Faiss ``IndexFlatIP`` file straight into HBM (fp32 on disk -> bf16 rows), optionally only the row range
        ``rows = (lo, hi)`` — a rank's shard of a reference-built index."""
        with open(fname, "rb") as f:
            hdr = f.read(_FAISS_HEADER.size)
        if len(hdr) < _FAISS_HEADER.size:
            raise ValueError(f"{fname}: too short for a Faiss index")
        fourcc, d, n, _, _, _, metric, n_floats = _FAISS_HEADER.unpack(hdr)
        if fourcc != _FAISS_FLAT_IP or metric != 0:
            raise ValueError(f"{fname}: not a Faiss IndexFlatIP file (fourcc {fourcc:#x}, metric {metric}); only the exact "
                             "inner-product index is on the hot path")
        if d <= 0 or n < 0 or n_floats != n * d:
            raise ValueError(f"{fname}: inconsistent header (d={d}, ntotal={n}, floats={n_floats})")
        lo, hi = (0, n) if rows is None else rows
        if not 0 <= lo <= hi <= n:
            raise ValueError(f"row range {rows} outside [0, {n}]")
        data = np.memmap(fname, dtype=np.float32, mode="r", offset=_FAISS_HEADER.size, shape=(n, d))
        idx = cls(d, passage_ids, device=device, id_offset=id_offset)
        idx.reserve(hi - lo)
        for a in range(lo, hi, rows_per_read):
            idx.add(np.ascontiguousarray(data[a:min(a + rows_per_read, hi)]))
        return idx


def save_dict_to_tsv(_dict: dict, output_path: str, keys=()):
    with open(output_path, "w") as f:
        writer = csv.writer(f, delimiter="\t", quoting=csv.QUOTE_MINIMAL)
        if keys:
            writer.writerow(keys)
        for key, value in _dict.items():
            writer.writerow([key, value])


def load_tsv_to_dict(input_path: str, header: bool = True) -> dict:
    mappings = {}
    with open(input_path, encoding="utf-8") as f:
        reader = csv.reader(f, delimiter="\t", quoting=csv.QUOTE_MINIMAL)
        if header:
            next(reader)
        for row in reader:
            mappings[row[0]] = int(row[1])
    return mappings


def sorted_corpus(corpus: dict) -> tuple[list, list]:
    """Longest document first, the order every reference searcher walks a dict corpus in (faiss_search.py:209-212)."""
    ids = sorted(corpus, key=lambda c: len(corpus[c].get("text", "")) if isinstance(corpus[c], dict) else len(corpus[c]),
                 reverse=True)
    return ids, [corpus[c] for c in ids]


def rows_to_dict(scores: torch.Tensor, ids: torch.Tensor, query_ids: Sequence, names, keep_empty: bool = True) -> dict:
    """(scores [Q, k], ids [Q, k] with -1 padding) -> ``dict[qid -> dict[name(id) -> float]]``, built in one pass over
    host copies.  ``names`` maps a document position to its corpus id (a sequence, or a callable)."""
    s, i = scores.cpu().numpy(), ids.cpu().numpy()
    look = names if callable(names) else names.__getitem__
    out = {}
    for r, qid in enumerate(query_ids):
        row = {look(doc): sc for doc, sc in zip(i[r].tolist(), s[r].tolist()) if doc >= 0}
        if row or keep_empty:
            out[qid] = row
    return out


class FlatIPSearch:
    """``FlatIPFaissSearch`` surface (faiss_search.py:46-293, 477-510) over ``FlatIPIndex`` / ``ShardedFlatIPIndex``."""

    def __init__(self, model=None, batch_size: int = 128, corpus_chunk_size: Optional[int] = None,
                 use_single_gpu: bool = False, use_multiple_gpu: bool = False, **kwargs):
        self.model = model
        self.batch_size = batch_size
        self.corpus_chunk_size = batch_size * 800 if corpus_chunk_size is None else corpus_chunk_size
        self.show_progress_bar = kwargs.get("show_progress_bar", True)
        self.convert_to_tensor = kwargs.get("convert_to_tensor", True)
        self.mapping_tsv_keys = ["beir-docid", "faiss-docid"]
        self.faiss_index = None
        # The corpus always lives in HBM, so `use_single_gpu` changes nothing; `use_multiple_gpu` shards it over the ranks
        # of `group` (one process per GPU) when torch.distributed is initialised, as Faiss shard=True does over the
        # visible devices of one process (faiss_search.py:480-504).
        self.use_single_gpu = use_single_gpu
        self.use_multiple_gpu = use_multiple_gpu
        self.group = kwargs.get("group", None)
        self.dim_size = None
        self.mapping: dict = {}
        self.rev_mapping: dict = {}
        self.device = kwargs.get("device", None)

    @classmethod
    def name(cls):
        return "flat_ip_b200_search"

    def get_index_name(self):
        return "flat_faiss_index"

    def encode(self, sentences, batch_size: int, **kwargs):
        return self.model.encode(sentences=sentences, batch_size=batch_size, **kwargs)

    def encode_queries(self, queries, batch_size: int, **kwargs):
        return self.model.encode_queries(queries=queries, batch_size=batch_size, **kwargs)

    def encode_corpus(self, corpus, batch_size: int, **kwargs):
        return self.model.encode_corpus(corpus=corpus, batch_size=batch_size, **kwargs)

    def _world(self) -> int:
        import torch.distributed as dist

        if self.use_multiple_gpu and dist.is_available() and dist.is_initialized():
            return dist.get_world_size(self.group)
        return 1

    def _create_mapping_ids(self, corpus_ids):
        if not all(isinstance(doc_id, int) for doc_id in corpus_ids):
            self.mapping = {cid: idx for idx, cid in enumerate(corpus_ids)}
            self.rev_mapping = dict(enumerate(corpus_ids))

    def _clear(self):
        if self.faiss_index is not None:
            self.faiss_index.reset()
        self.faiss_index = None
        self.dim_size = None
        self.mapping = {}
        self.rev_mapping = {}

    def _build_index(self, corpus_emb, passage_ids, id_base: int = 0):
        """Resident index over `corpus_emb` whose result ids start at `id_base`; a row shard per rank when sharded."""
        if self._world() > 1:
            from .sharded import ShardedFlatIPIndex

            sh = ShardedFlatIPIndex(corpus_emb.shape[1], corpus_emb.shape[0], device=self.device, group=self.group,
                                    id_base=id_base)
            sh.add_local(corpus_emb[sh.lo:sh.hi])
            sh._passage_ids = None if passage_ids is None else np.asarray(passage_ids, dtype=np.int64)
            return sh
        return FlatIPIndex.build(passage_ids, corpus_emb, FlatIPIndex(corpus_emb.shape[1], device=self.device,
                                                                     id_offset=id_base))

    def index(self, corpus_emb, corpus_ids: Sequence[str]):
        self._create_mapping_ids(corpus_ids)
        self.dim_size = corpus_emb.shape[1]
        passage_ids = list(range(len(corpus_ids))) if self.mapping else [int(c) for c in corpus_ids]
        self.faiss_index = self._build_index(corpus_emb, passage_ids)

    def retrieve_arrays(self, query_emb, top_k: int, **kwargs):
        """Device arrays (scores f32 [Q,k], doc positions i64 [Q,k], -1 padded): results stay on device and become the
        reference's nested dicts only when a caller asks for them (`arrays_to_dict`)."""
        if self.faiss_index is None:
            raise RuntimeError("index() must be called before retrieve_arrays()")
        return self.faiss_index.search_device(query_emb, top_k, **kwargs)

    def _doc_name(self, pos: int):
        pid = self.faiss_index._passage_ids
        doc = int(pid[pos - self.faiss_index.id_offset]) if pid is not None else pos
        return self.rev_mapping[doc] if self.rev_mapping else str(doc)

    def arrays_to_dict(self, scores, ids, query_ids: Sequence[str]) -> dict:
        return rows_to_dict(scores, ids, query_ids, self._doc_name)

    def retrieve_with_emb(self, query_emb, query_ids: Sequence[str], top_k: int, **kwargs) -> dict:
        """faiss_search.py:143-173: ``dict[qid -> dict[pid -> score]]`` (the (-inf, -1) padding of a corpus with fewer
        than k documents is dropped)."""
        if self.faiss_index is None:
            raise RuntimeError("index() must be called before retrieve_with_emb()")
        return self.arrays_to_dict(*self.retrieve_arrays(query_emb, top_k, **kwargs), query_ids)

    def save(self, output_dir: str, prefix: str = "my-index", ext: str = "flat"):
        """The reference's two files (faiss_search.py:113-123): `<prefix>.<ext>.tsv` id map + `<prefix>.<ext>.faiss`."""
        if not isinstance(self.faiss_index, FlatIPIndex):
            raise NotImplementedError("save() writes one Faiss file: gather the shards or save per rank with FlatIPIndex.save")
        save_dict_to_tsv(self.mapping, os.path.join(output_dir, f"{prefix}.{ext}.tsv"), keys=self.mapping_tsv_keys)
        self.faiss_index.save(os.path.join(output_dir, f"{prefix}.{ext}.faiss"))

    def load(self, input_dir: str, prefix: str = "my-index", ext: str = "flat"):
        """faiss_search.py:99-111, 478-488: reads an index saved by this class or by the reference's FlatIPFaissSearch."""
        self.mapping = load_tsv_to_dict(os.path.join(input_dir, f"{prefix}.{ext}.tsv"), header=True)
        self.rev_mapping = {v: k for k, v in self.mapping.items()}
        passage_ids = sorted(self.rev_mapping)
        path = os.path.join(input_dir, f"{prefix}.{ext}.faiss")
        idx = FlatIPIndex.load(path, passage_ids or None, device=self.device)
        self.faiss_index = idx.to_gpu(self.group) if self._world() > 1 else idx
        self.dim_size = idx.dim

    def search_arrays(self, corpus_chunks, query_embeddings, top_k: int, self_pos: Optional[torch.Tensor] = None):
        """Exact top-k over a corpus that arrives in chunks: every chunk is indexed with its global row offset, searched,
        and folded into a running device top-k with ``lr_topk_merge``; nothing crosses to the host.  `corpus_chunks`
        yields ``(first_row, embeddings [n, d])``.  Returns (scores, ids) with ids = global rows."""
        run = None
        for first_row, emb in corpus_chunks:
            idx = self._build_index(emb, None, id_base=first_row)
            keys = idx.search_keys(query_embeddings, top_k)
            idx.reset()
            if self_pos is not None:
                keys = drop_identical(keys, self_pos)
            run = keys if run is None else merge_keys([run, keys], top_k)
        if run is None:
            raise ValueError("empty corpus")
        return decode_keys(run)

    def search(self, corpus, queries, top_k: int = 1000, score_function: str = None, return_sorted: bool = False,
               ignore_identical_ids: bool = False, **kwargs) -> dict:
        """Chunked encode -> index -> retrieve -> merge of DenseRetrievalFaissSearch.search (faiss_search.py:176-293).
        The per-chunk results are merged on device; the result dicts are built once at the end."""
        if not isinstance(queries, dict) or not isinstance(corpus, dict):
            raise NotImplementedError("FlatIPSearch.search takes dict corpora / queries")
        query_ids = list(queries.keys())
        query_embeddings = self.model.encode_queries([queries[qid] for qid in queries], batch_size=self.batch_size,
                                                     show_progress_bar=self.show_progress_bar,
                                                     convert_to_tensor=self.convert_to_tensor)
        corpus_ids, corpus_list = sorted_corpus(corpus)

        def chunks():
            for start in range(0, len(corpus_list), self.corpus_chunk_size):
                sub = self.model.encode_corpus(corpus_list[start:start + self.corpus_chunk_size],
                                               batch_size=self.batch_size, show_progress_bar=self.show_progress_bar,
                                               convert_to_tensor=self.convert_to_tensor)
                if isinstance(sub, dict):
                    if "dense_reps" not in sub:
                        raise ValueError(f"HybridModel: Return Multi-vector with keys {sub.keys()}, but not `dense_reps`")
                    sub = sub["dense_reps"]
                yield start, sub

        scores, ids = self.search_arrays(chunks(), query_embeddings, top_k,
                                         identical_positions(query_ids, corpus_ids) if ignore_identical_ids else None)
        return rows_to_dict(scores, ids, query_ids, corpus_ids)


def identical_positions(query_ids: Sequence, corpus_ids: Sequence) -> torch.Tensor:
    """Corpus position of the document that carries the same id as each query (-1 = none), for `ignore_identical_ids`."""
    pos = {cid: i for i, cid in enumerate(corpus_ids)}
    return torch.tensor([pos.get(qid, -1) for qid in query_ids], dtype=torch.int64)
