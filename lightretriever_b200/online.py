"""Online serving step (BASELINE configs[4]: batch 1 / 32, p50 / p99 latency) as ONE CUDA-graph replay.

The reference answers an online query with a Python call chain — EmbeddingBag forward (finetune/modeling_hybrid.py:474),
``F.normalize`` (:489-490), ``FaissIndex.search`` (retriever/faiss_index.py:27-40) and, over shards, a host merge
(:65-68).  Here the same chain is five to eight kernels and at most one NCCL all-gather; at ~1.5 ms per request the
host's launch path is a visible part of the latency, so the whole step is captured once per (batch, max_tokens) shape
and replayed: the request's ids / offsets are copied into static device buffers, unused id slots hold ``padding_idx``
(skipped by the encoder exactly like torch's ``padding_idx``) and unused bags are empty.

``OnlineHybridSearcher`` serves the reference's default hybrid result (``emb_tok``, retriever/hybrid_search.py:123-180)
the same way: dense ``emb`` and sparse token-count ``tok`` retrieval and their fusion in one replay.

Inserts need no recapture either: with ``insert_capacity`` > 0 a searcher owns a fixed-size, append-only delta segment
(zeroed bf16 rows for K2; for the hybrid also a document-major sparse segment, ``ImpactDelta``) whose documents get the
global ids ``[insert_id_base, insert_id_base + insert_capacity)``.  Every replay searches the main shard and the delta
with the same bitmaps and merges the two lists per system before anything else, so the result is the exact top-k of
main + inserted documents.  ``insert`` writes the next slots and sets their live bits last (unfilled slots are dead);
slots are never reused, and an update is ``delete(old)`` + ``insert(new)``.  ``export_inserts`` returns the filled
delta for the next offline rebuild.

Deletions and per-request filters need no recapture: every searcher owns a static ``live`` bitmap (global ids
``[0, id_offset + N)``) and, when given ``filters`` [F, ld_words], a static ``[batch]`` row choice per query.
``delete(ids)`` / ``restore(ids)`` and in-place edits of ``filters`` are kernels enqueued on the stream the replays run
on, so the next request sees them; ``search(..., filter_rows=...)`` picks each query's filter row (-1 = unrestricted).

A graph that captured NCCL collectives (world > 1) must not outlive the communicator: tearing the process group down
under such a graph can hang.  Release the searchers (or end the process without tearing it down) first.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
import torch.distributed as dist

from . import _C
from ._util import Workspace
from .encode import B200EmbeddingBag
from .filters import doc_bitmap, doc_bitmap_update
from .hybrid import fuse_topk_device
from .search import flatip_topk, topk_merge
from .sharded import exchange_candidates
from .sparse_search import MAX_TOP_K, QUERY_MAX_BAG, ImpactDelta, ImpactIndex, query_token_counts


def _insert_layout(world: int, id_offset: int, n_rows: int, insert_capacity, insert_id_base) -> tuple[int, int]:
    """(capacity, id of the first delta slot) of a searcher's delta segment.  With one GPU the delta continues the
    shard's ids by default, so a rebuilt index numbers the same documents the same way; with several each rank needs
    its own range above every main id (e.g. ``n_total + rank * insert_capacity``)."""
    cap = int(insert_capacity)
    if cap < 0:
        raise ValueError(f"insert_capacity ({cap}) must be >= 0")
    if cap == 0:
        return 0, 0
    if insert_id_base is None:
        if world > 1:
            raise ValueError("insert_id_base is required when the searcher is sharded over several GPUs: give each "
                             "rank its own id range above every main id, e.g. n_total + rank * insert_capacity")
        insert_id_base = id_offset + n_rows
    base = int(insert_id_base)
    if base < id_offset + n_rows and base + cap > id_offset:
        raise ValueError(f"the delta's ids [{base}, {base + cap}) overlap the shard's [{id_offset}, {id_offset + n_rows})")
    if base < 0 or base + cap > (1 << 32) - 2:
        raise ValueError(f"the delta's ids [{base}, {base + cap}) must lie in [0, 2^32 - 2)")
    return cap, base


class _CapturedStep:
    """Static request buffers + one captured ``_step``: the part every online searcher shares."""

    def __init__(self, bag: B200EmbeddingBag, corpus: torch.Tensor, k: int, batch: int, max_tokens: int,
                 id_offset: int, shrink_dim: Optional[int], group, live: Optional[torch.Tensor] = None,
                 filters: Optional[torch.Tensor] = None, insert_capacity: int = 0, insert_id_base: Optional[int] = None):
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.insert_capacity, self.insert_id_base = _insert_layout(self.world, int(id_offset), corpus.shape[0],
                                                                   insert_capacity, insert_id_base)
        n_ids = int(id_offset) + corpus.shape[0]
        if self.insert_capacity:
            n_ids = max(n_ids, self.insert_id_base + self.insert_capacity)
            if filters is not None and (filters.ndim != 2 or filters.shape[1] < (n_ids + 31) // 32):
                raise ValueError(f"filters must cover the inserted documents' ids: [F, >= {(n_ids + 31) // 32}] words")
        if bag.padding_idx is None:
            raise ValueError(f"{type(self).__name__} pads requests with padding_idx: the bag needs one")
        if corpus.dtype != torch.bfloat16 or not corpus.is_cuda:
            raise ValueError("corpus must be a bfloat16 CUDA tensor (the resident shard)")
        self.bag, self.corpus, self.k, self.batch, self.max_tokens = bag, corpus, int(k), int(batch), int(max_tokens)
        self.id_offset, self.shrink_dim, self.group = int(id_offset), shrink_dim, group
        self._ids = self._static_ids(bag.padding_idx)
        self._offs = self._static_offsets()
        self._graph = None
        self._out = None
        dev, n_main = corpus.device, self.id_offset + corpus.shape[0]
        if live is None:
            self._live = doc_bitmap(n_main, device=dev)
        else:
            if live.dtype != torch.int32 or live.ndim != 1 or live.device != dev or live.numel() < (n_main + 31) // 32:
                raise ValueError(f"live must be a 1-D int32 bitmap of >= {(n_main + 31) // 32} words on {dev}")
            self._live = live.clone()  # the searcher's own static copy: its deletions do not touch the caller's bitmap
        self._n_inserted = 0
        if self.insert_capacity:
            # the bitmap grows to the delta's ids, whose slots start dead: K2 scores the delta's zero rows too
            width = max((n_ids + 31) // 32, self._live.numel(), 0 if filters is None else filters.shape[1])
            self._live = torch.cat([self._live, self._live.new_zeros(width - self._live.numel())])
            base = self.insert_id_base
            doc_bitmap_update(self._live, torch.arange(base, base + self.insert_capacity, device=dev), False)
            self._delta = torch.zeros((self.insert_capacity, corpus.shape[1]), dtype=torch.bfloat16, device=dev)
            self._ws_delta = Workspace()
        if filters is not None:
            if (filters.dtype != torch.int32 or filters.ndim != 2 or not filters.is_contiguous() or filters.device != dev
                    or filters.shape[1] != self._live.numel()):
                raise ValueError(f"filters must be a contiguous int32 [F, {self._live.numel()}] table on {dev}")
        self._filters = filters  # kept by reference: in-place edits reach the next replay
        self._qf = torch.full((self.batch,), -1, dtype=torch.int32, device=dev) if filters is not None else None

    def _filter_kw(self) -> dict:
        return dict(live=self._live, allow=self._filters, q_filter=self._qf)

    def delete(self, ids) -> None:
        """Hide documents (global ids) from every later request; enqueued on the current stream, no recapture."""
        doc_bitmap_update(self._live, ids, False)

    def restore(self, ids) -> None:
        """Bring deleted documents back.  An inserted document's id is only valid once its slot is filled."""
        if self.insert_capacity:
            g = torch.as_tensor(ids, dtype=torch.int64).reshape(-1).cpu()
            lo = self.insert_id_base + self._n_inserted
            if ((g >= lo) & (g < self.insert_id_base + self.insert_capacity)).any():
                raise ValueError(f"restore: ids in [{lo}, {self.insert_id_base + self.insert_capacity}) belong to delta "
                                 "slots that hold no document yet")
        doc_bitmap_update(self._live, ids, True)

    def _insert_rows(self, rows: torch.Tensor) -> int:
        """Validate a batch of dense rows against the delta (shape, free slots); returns its size.  Writes nothing."""
        if not self.insert_capacity:
            raise ValueError("insert needs a searcher constructed with insert_capacity > 0")
        if rows.ndim != 2 or rows.shape[1] != self._delta.shape[1]:
            raise ValueError(f"rows must be [n, {self._delta.shape[1]}]")
        n = rows.shape[0]
        if self._n_inserted + n > self.insert_capacity:
            raise ValueError(f"the delta segment is full: {self._n_inserted} + {n} documents (capacity "
                             f"{self.insert_capacity})")
        return n

    def _commit_rows(self, rows: torch.Tensor) -> torch.Tensor:
        """Write validated rows into the next delta slots, then set their live bits; returns their global ids."""
        n, a = rows.shape[0], self._n_inserted
        self._delta[a:a + n].copy_(rows.to(self._delta.device, torch.bfloat16))
        ids = torch.arange(self.insert_id_base + a, self.insert_id_base + a + n, dtype=torch.int64)
        self._n_inserted = a + n
        doc_bitmap_update(self._live, ids, True)
        return ids

    def _dense_lists(self, qv: torch.Tensor, workspace: Optional[Workspace] = None) -> torch.Tensor:
        """Candidate keys [2, Q, k] of the main shard and of the delta, each searched by K2 (merged by the caller)."""
        main = flatip_topk(qv, self._dense_corpus(), self.k, id_offset=self.id_offset, return_keys=True,
                           workspace=workspace, **self._filter_kw())[2]
        delta = self._delta if self.shrink_dim is None else self._delta[:, :self.shrink_dim]
        new = flatip_topk(qv, delta, self.k, id_offset=self.insert_id_base, return_keys=True, workspace=self._ws_delta,
                          **self._filter_kw())[2]
        return torch.stack((main, new))

    def _stage_filters(self, filter_rows, n: int) -> None:
        if filter_rows is None:
            if self._qf is not None:
                self._qf.fill_(-1)
            return
        if self._filters is None:
            raise ValueError("filter_rows needs a searcher constructed with filters")
        fr = torch.as_tensor(filter_rows, dtype=torch.int32).reshape(-1)
        if fr.numel() != n:
            raise ValueError(f"{fr.numel()} filter rows for {n} queries")
        self._qf.fill_(-1)
        self._qf[:n].copy_(fr, non_blocking=True)

    def _static_ids(self, pad: int) -> torch.Tensor:
        return torch.full((self.max_tokens,), pad, dtype=torch.int64, device=self.corpus.device)

    def _static_offsets(self) -> torch.Tensor:
        return torch.full((self.batch,), self.max_tokens, dtype=torch.int64, device=self.corpus.device)

    def _encode(self) -> torch.Tensor:
        return self.bag.encode(self._ids, self._offs, shrink_dim=self.shrink_dim, normalize=True, check_ids=False)

    def _dense_corpus(self) -> torch.Tensor:
        return self.corpus if self.shrink_dim is None else self.corpus[:, :self.shrink_dim]

    def _step(self):
        raise NotImplementedError

    def _capture(self, workspaces: Sequence[Workspace] = ()):
        if self.insert_capacity:
            workspaces = tuple(workspaces) + (self._ws_delta,)
        side = torch.cuda.Stream(device=self.corpus.device)
        side.wait_stream(torch.cuda.current_stream(self.corpus.device))
        with torch.cuda.stream(side):  # warm-up: workspace allocation, attribute calls, NCCL channels
            for _ in range(3):
                self._step()
        torch.cuda.current_stream(self.corpus.device).wait_stream(side)
        torch.cuda.synchronize(self.corpus.device)
        for ws in workspaces:  # the warm-up's buffers (keyed by the side stream) are not the graph's
            ws.clear()
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._out = self._step()

    def _check_request(self, ids: torch.Tensor, offsets: torch.Tensor, what: str = "request"):
        n_ids, n_bags = ids.numel(), offsets.numel()
        if n_bags > self.batch or n_ids > self.max_tokens:
            raise ValueError(f"{what} ({n_bags} bags, {n_ids} ids) exceeds the captured shape "
                             f"({self.batch}, {self.max_tokens})")

    @staticmethod
    def _stage(buf_ids: torch.Tensor, buf_offs: torch.Tensor, pad: int, ids: torch.Tensor, offsets: torch.Tensor):
        n_ids, n_bags = ids.numel(), offsets.numel()
        buf_ids.fill_(pad)
        buf_ids[:n_ids].copy_(ids, non_blocking=True)
        buf_offs.fill_(n_ids)  # unused bags are empty; the last real bag ends where the padding ids start
        buf_offs[:n_bags].copy_(offsets, non_blocking=True)

    def _run(self):
        if self._graph is not None:
            self._graph.replay()
            return self._out
        return self._step()


class OnlineSearcher(_CapturedStep):
    """``live``: initial deletions bitmap (copied; default all live), ``filters``: optional static [F, ld_words] table
    of per-request filters (see the module docstring).  ``insert_capacity`` > 0 adds a delta segment of that many rows
    for ``insert`` (ids from ``insert_id_base``, see the module docstring)."""

    def __init__(self, bag: B200EmbeddingBag, corpus: torch.Tensor, k: int, batch: int, max_tokens: int,
                 id_offset: int = 0, shrink_dim: Optional[int] = None, group=None, use_graph: bool = True,
                 live: Optional[torch.Tensor] = None, filters: Optional[torch.Tensor] = None, insert_capacity: int = 0,
                 insert_id_base: Optional[int] = None):
        super().__init__(bag, corpus, k, batch, max_tokens, id_offset, shrink_dim, group, live, filters,
                         insert_capacity, insert_id_base)
        if use_graph:
            self._capture()

    def insert(self, rows: torch.Tensor) -> torch.Tensor:
        """Append documents (dense rows [n, d]) to the delta segment; returns their global ids.  Enqueued on the current
        stream like ``delete``: the next request sees them, without recapture.  A batch that does not fit raises
        ValueError and changes nothing."""
        self._insert_rows(rows)
        return self._commit_rows(rows)

    def export_inserts(self) -> tuple[torch.Tensor, torch.Tensor]:
        """(rows bf16 [n, d], global ids i64 [n]) of the inserted documents: what an offline rebuild folds into the
        main shard."""
        if not self.insert_capacity:
            raise ValueError("export_inserts needs a searcher constructed with insert_capacity > 0")
        n = self._n_inserted
        return self._delta[:n].clone(), torch.arange(self.insert_id_base, self.insert_id_base + n, dtype=torch.int64)

    def _step(self):
        qv = self._encode()
        corpus = self._dense_corpus()
        if self.insert_capacity:
            lists = self._dense_lists(qv)
            if self.world == 1:
                return topk_merge(lists, self.k)
            return topk_merge(exchange_candidates(topk_merge(lists, self.k, return_keys=True)[2], self.group), self.k)
        if self.world == 1:
            return flatip_topk(qv, corpus, self.k, id_offset=self.id_offset, **self._filter_kw())
        _, _, keys = flatip_topk(qv, corpus, self.k, id_offset=self.id_offset, return_keys=True, **self._filter_kw())
        return topk_merge(exchange_candidates(keys, self.group), self.k)

    def search(self, input_ids: torch.Tensor, offsets: torch.Tensor, filter_rows=None):
        """(scores [n_bags, k] f32, ids [n_bags, k] i64) for a request of up to ``batch`` bags / ``max_tokens`` ids.
        ``filter_rows`` [n_bags]: each query's row of ``filters`` (-1 = unrestricted; None = all unrestricted).
        The returned tensors are views of the searcher's static outputs: consume them before the next call."""
        self._check_request(input_ids, offsets)
        n_bags = offsets.numel()
        self._stage_filters(filter_rows, n_bags)
        self._stage(self._ids, self._offs, self.bag.padding_idx, input_ids, offsets)
        s, i = self._run()
        return s[:n_bags], i[:n_bags]


class OnlineHybridSearcher(_CapturedStep):
    """Dense + sparse + fusion as one CUDA-graph replay per request.

    Per step: K1 encode -> K2 ``flatip_topk`` (dense ``emb``); ``query_token_counts`` -> K4
    ``ImpactIndex.search_device`` (sparse ``tok``: the query's token counts, or a count of 1 per distinct token with
    ``token_kind="bow"``); when world > 1 ONE all-gather carries both systems' keys ([2, Q, k] per rank) and each half is
    merged in place; then ``lr_fuse_topk`` (``method`` "linear" with ``weights``, or "rrf") on every rank, so every rank
    holds the same result.  ``corpus`` and ``sparse_index`` are this rank's shards of the same documents (same
    ``id_offset``, same count).  Both halves read the same ``live`` bitmap (default: a copy of the sparse index's, or all
    live) and ``filters`` table, so the fused list never holds a deleted or filtered-out id."""

    def __init__(self, bag: B200EmbeddingBag, corpus: torch.Tensor, sparse_index: ImpactIndex, k: int, batch: int,
                 max_tokens: int, id_offset: int = 0, shrink_dim: Optional[int] = None, method: str = "linear",
                 weights: Sequence[float] = (0.7, 0.3), token_kind: str = "sum", group=None, use_graph: bool = True,
                 live: Optional[torch.Tensor] = None, filters: Optional[torch.Tensor] = None, insert_capacity: int = 0,
                 insert_postings_capacity: Optional[int] = None, insert_id_base: Optional[int] = None):
        if insert_postings_capacity is not None and int(insert_postings_capacity) < 0:
            raise ValueError(f"insert_postings_capacity ({insert_postings_capacity}) must be >= 0")
        if not 1 <= int(k) <= MAX_TOP_K:
            raise ValueError(f"k={k} must be in [1, {MAX_TOP_K}] (the sparse kernel's limit)")
        if sparse_index.id_offset != int(id_offset) or sparse_index.N != corpus.shape[0]:
            raise ValueError(f"the sparse index (id_offset {sparse_index.id_offset}, {sparse_index.N} documents) and the "
                             f"dense shard (id_offset {id_offset}, {corpus.shape[0]} rows) must number the same documents")
        if sparse_index.device != corpus.device:
            raise ValueError("the sparse index and the dense shard must be on the same device")
        if method not in ("linear", "rrf"):
            raise NotImplementedError(f"score_fuse_method {method} is not supported.")
        if token_kind not in ("sum", "bow"):
            raise ValueError(f"token_kind must be 'sum' or 'bow', got {token_kind!r}")
        if live is None:
            live = sparse_index.live_words
        super().__init__(bag, corpus, k, batch, max_tokens, id_offset, shrink_dim, group, live, filters,
                         insert_capacity, insert_id_base)
        self.sparse_index, self.method, self.weights, self.token_kind = sparse_index, method, tuple(weights), token_kind
        self._sparse_delta = None
        if self.insert_capacity:
            # default: room for the main shard's mean document length
            n_post = (-(-int(sparse_index.build()[0][-1]) * self.insert_capacity // max(sparse_index.N, 1))
                      if insert_postings_capacity is None else int(insert_postings_capacity))
            self._sparse_delta = ImpactDelta(sparse_index.V, self.insert_capacity, n_post, corpus.device,
                                             self.insert_id_base)
            self._ws_sparse_delta = Workspace()
        # the sparse query's ids have their own buffer: padding_idx is a real token to the sparse index, -1 is not
        self._tok = self._static_ids(-1)
        self._tok_offs = self._static_offsets()
        self._max_bag = min(self.max_tokens, QUERY_MAX_BAG)
        # owned scratch: a graph must not point into a module-wide buffer that another call can regrow
        self._ws_dense, self._ws_counts, self._ws_sparse = Workspace(), Workspace(), Workspace()
        sparse_index.build()
        if use_graph:
            ws = (self._ws_dense, self._ws_counts, self._ws_sparse)
            self._capture(ws + ((self._ws_sparse_delta,) if self.insert_capacity else ()))

    def insert(self, rows: torch.Tensor, indptr, tok, imp) -> torch.Tensor:
        """Append documents to both delta segments: dense rows [n, d] and their sparse vectors as doc-major CSR (as
        ``ImpactIndex.add_csr``); returns their global ids.  The whole batch is validated first: one that does not fit
        either capacity raises ValueError and changes nothing.  Enqueued on the current stream, no recapture."""
        n = self._insert_rows(rows)
        prepared = self._sparse_delta.prepare_csr(indptr, tok, imp)
        if prepared[0].numel() != n:
            raise ValueError(f"{n} dense rows but {prepared[0].numel()} sparse documents")
        self._sparse_delta.commit(prepared)
        return self._commit_rows(rows)

    def export_inserts(self):
        """(rows bf16 [n, d], (indptr i64 [n+1], tok i32, imp i16), global ids i64 [n]) of the inserted documents: what
        an offline rebuild folds into the main shard and its inverted index."""
        if not self.insert_capacity:
            raise ValueError("export_inserts needs a searcher constructed with insert_capacity > 0")
        n = self._n_inserted
        return (self._delta[:n].clone(), self._sparse_delta.export_csr(),
                torch.arange(self.insert_id_base, self.insert_id_base + n, dtype=torch.int64))

    def _step(self):
        Q, k, V = self.batch, self.k, self.sparse_index.V
        qv = self._encode()
        q_csr = query_token_counts(self._tok, self._tok_offs, V, kind=self.token_kind, max_bag=self._max_bag,
                                   check=False, workspace=self._ws_counts)
        if self.insert_capacity:  # main + delta merged per system before the exchange, whose payload stays [2, Q, k]
            dl = self._dense_lists(qv, self._ws_dense)
            sl = torch.stack((
                self.sparse_index.search_device(*q_csr, k, return_keys=True, workspace=self._ws_sparse,
                                                **self._filter_kw())[2],
                self._sparse_delta.search_device(*q_csr, k, return_keys=True, workspace=self._ws_sparse_delta,
                                                 **self._filter_kw())[2]))
            if self.world == 1:
                ds, di = topk_merge(dl, k)
                ss, si = topk_merge(sl, k, score_kind=_C.LR_SCORE_U32)
            else:
                dk = topk_merge(dl, k, return_keys=True)[2]
                sk = topk_merge(sl, k, score_kind=_C.LR_SCORE_U32, return_keys=True)[2]
                gathered = exchange_candidates(torch.stack((dk, sk)), self.group)
                ds, di = topk_merge(gathered[:, 0], k)
                ss, si = topk_merge(gathered[:, 1], k, score_kind=_C.LR_SCORE_U32)
            fused = fuse_topk_device(ds, di, ss, si, method=self.method, weights=self.weights)
            return (ds, di), (ss, si), fused
        if self.world == 1:
            ds, di = flatip_topk(qv, self._dense_corpus(), k, id_offset=self.id_offset, workspace=self._ws_dense,
                                 **self._filter_kw())
            ss, si = self.sparse_index.search_device(*q_csr, k, workspace=self._ws_sparse, **self._filter_kw())
        else:
            dk = flatip_topk(qv, self._dense_corpus(), k, id_offset=self.id_offset, return_keys=True,
                             workspace=self._ws_dense, **self._filter_kw())[2]
            sk = self.sparse_index.search_device(*q_csr, k, return_keys=True, workspace=self._ws_sparse,
                                                 **self._filter_kw())[2]
            gathered = exchange_candidates(torch.stack((dk, sk)), self.group)  # [world, 2, Q, k]: one exchange for both
            ds, di = topk_merge(gathered[:, 0], k)                                 # lists spaced by 2Q query rows
            ss, si = topk_merge(gathered[:, 1], k, score_kind=_C.LR_SCORE_U32)    # sparse half: offset Q*k
        fused = fuse_topk_device(ds, di, ss, si, method=self.method, weights=self.weights)
        return (ds, di), (ss, si), fused

    def search(self, input_ids: torch.Tensor, offsets: torch.Tensor, token_ids: Optional[torch.Tensor] = None,
               token_offsets: Optional[torch.Tensor] = None, filter_rows=None):
        """One request of up to ``batch`` queries: ``input_ids`` / ``offsets`` are the EmbeddingBag's flattened ids,
        ``token_ids`` / ``token_offsets`` the sparse query's (the reference tokenises ``" " + text`` for it); both
        ``None`` reuses the bag ids.  Returns ``dense`` (scores f32, ids i64) [n, k], ``sparse`` (scores f32, ids i64)
        [n, k] with a (-inf, -1) tail, and ``fused`` (ids i64 [n, 2k], scores f64 [n, 2k], counts i32 [n]) as
        ``fuse_topk_device`` returns it.  ``filter_rows`` as in ``OnlineSearcher.search``.  All are views of the searcher's static outputs: consume them before the next
        call."""
        if (token_ids is None) != (token_offsets is None):
            raise ValueError("token_ids and token_offsets go together")
        if token_ids is None:
            token_ids, token_offsets = input_ids, offsets
        n = offsets.numel()
        if token_offsets.numel() != n:
            raise ValueError(f"{n} dense queries but {token_offsets.numel()} sparse ones")
        self._check_request(input_ids, offsets)
        self._check_request(token_ids, token_offsets, "sparse request")
        if self.max_tokens > QUERY_MAX_BAG and token_ids.numel() > QUERY_MAX_BAG:
            ends = torch.cat([token_offsets.reshape(-1)[1:].cpu(), torch.tensor([token_ids.numel()])])
            if int((ends - token_offsets.reshape(-1).cpu()).max()) > QUERY_MAX_BAG:
                raise ValueError(f"a sparse query longer than {QUERY_MAX_BAG} ids")
        self._stage_filters(filter_rows, n)
        self._stage(self._ids, self._offs, self.bag.padding_idx, input_ids, offsets)
        self._stage(self._tok, self._tok_offs, -1, token_ids, token_offsets)
        (ds, di), (ss, si), (fi, fs, fc) = self._run()
        return (ds[:n], di[:n]), (ss[:n], si[:n]), (fi[:n], fs[:n], fc[:n])
