"""Online serving step (BASELINE configs[4]: batch 1 / 32, p50 / p99 latency) as ONE CUDA-graph replay.

The reference answers an online query with a Python call chain — EmbeddingBag forward (finetune/modeling_hybrid.py:474),
``F.normalize`` (:489-490), ``FaissIndex.search`` (retriever/faiss_index.py:27-40) and, over shards, a host merge
(:65-68).  Here the same chain is five to eight kernels and at most one NCCL all-gather; at ~1.5 ms per request the
host's launch path is a visible part of the latency, so the whole step is captured once per (batch, max_tokens) shape
and replayed: the request's ids / offsets are copied into static device buffers, unused id slots hold ``padding_idx``
(skipped by the encoder exactly like torch's ``padding_idx``) and unused bags are empty.

``OnlineHybridSearcher`` serves the reference's default hybrid result (``emb_tok``, retriever/hybrid_search.py:123-180)
the same way: dense ``emb`` and sparse token-count ``tok`` retrieval and their fusion in one replay.

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
from .sparse_search import MAX_TOP_K, QUERY_MAX_BAG, ImpactIndex, query_token_counts


class _CapturedStep:
    """Static request buffers + one captured ``_step``: the part every online searcher shares."""

    def __init__(self, bag: B200EmbeddingBag, corpus: torch.Tensor, k: int, batch: int, max_tokens: int,
                 id_offset: int, shrink_dim: Optional[int], group, live: Optional[torch.Tensor] = None,
                 filters: Optional[torch.Tensor] = None):
        if bag.padding_idx is None:
            raise ValueError(f"{type(self).__name__} pads requests with padding_idx: the bag needs one")
        if corpus.dtype != torch.bfloat16 or not corpus.is_cuda:
            raise ValueError("corpus must be a bfloat16 CUDA tensor (the resident shard)")
        self.bag, self.corpus, self.k, self.batch, self.max_tokens = bag, corpus, int(k), int(batch), int(max_tokens)
        self.id_offset, self.shrink_dim, self.group = int(id_offset), shrink_dim, group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self._ids = self._static_ids(bag.padding_idx)
        self._offs = self._static_offsets()
        self._graph = None
        self._out = None
        dev, n_ids = corpus.device, self.id_offset + corpus.shape[0]
        if live is None:
            self._live = doc_bitmap(n_ids, device=dev)
        else:
            if live.dtype != torch.int32 or live.ndim != 1 or live.device != dev or live.numel() < (n_ids + 31) // 32:
                raise ValueError(f"live must be a 1-D int32 bitmap of >= {(n_ids + 31) // 32} words on {dev}")
            self._live = live.clone()  # the searcher's own static copy: its deletions do not touch the caller's bitmap
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
        doc_bitmap_update(self._live, ids, True)

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
    of per-request filters (see the module docstring)."""

    def __init__(self, bag: B200EmbeddingBag, corpus: torch.Tensor, k: int, batch: int, max_tokens: int,
                 id_offset: int = 0, shrink_dim: Optional[int] = None, group=None, use_graph: bool = True,
                 live: Optional[torch.Tensor] = None, filters: Optional[torch.Tensor] = None):
        super().__init__(bag, corpus, k, batch, max_tokens, id_offset, shrink_dim, group, live, filters)
        if use_graph:
            self._capture()

    def _step(self):
        qv = self._encode()
        corpus = self._dense_corpus()
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
                 live: Optional[torch.Tensor] = None, filters: Optional[torch.Tensor] = None):
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
        super().__init__(bag, corpus, k, batch, max_tokens, id_offset, shrink_dim, group, live, filters)
        self.sparse_index, self.method, self.weights, self.token_kind = sparse_index, method, tuple(weights), token_kind
        # the sparse query's ids have their own buffer: padding_idx is a real token to the sparse index, -1 is not
        self._tok = self._static_ids(-1)
        self._tok_offs = self._static_offsets()
        self._max_bag = min(self.max_tokens, QUERY_MAX_BAG)
        # owned scratch: a graph must not point into a module-wide buffer that another call can regrow
        self._ws_dense, self._ws_counts, self._ws_sparse = Workspace(), Workspace(), Workspace()
        sparse_index.build()
        if use_graph:
            self._capture((self._ws_dense, self._ws_counts, self._ws_sparse))

    def _step(self):
        Q, k, V = self.batch, self.k, self.sparse_index.V
        qv = self._encode()
        q_csr = query_token_counts(self._tok, self._tok_offs, V, kind=self.token_kind, max_bag=self._max_bag,
                                   check=False, workspace=self._ws_counts)
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
