"""Sparse impact search (K4) — host side, seam S4.

Mirrors ``AnseriniSearch`` (reference retriever/anserini_search.py:31-216): ``index(corpus_emb, corpus_ids)`` takes the
``list[dict[str(token_id) -> int impact]]`` produced by ``convert_sparse_reps_to_json`` (JsonVectorCollection) and may
be called repeatedly (chunks are appended, anserini_search.py:89-111); ``retrieve_with_emb(query_emb, query_ids,
top_k)`` takes the pseudo-query strings ``"id id id ..."`` emitted by ``EncodeCollator`` (inference/
exact_search_base.py:393-435; a repeated id = a count) or ``{token_id: count}`` dicts; ``_clear()`` drops the index.
Instead of JSONL on disk + a JVM, documents become a token-major inverted index in HBM and scoring is
``lr_sparse_score_topk`` (csrc/sparse_score.cu).  Scores are the exact integer dot products Lucene's impact search
computes (scripts/asymmetric_sparse_infer.ipynb:207-228); only matching documents are returned.
"""
from __future__ import annotations

from collections import Counter
from typing import Optional, Sequence

import numpy as np
import torch

from . import _C
from ._util import Workspace, require_cuda, stream_ptr
from .filters import DocDeletions, filter_args

_WS = Workspace()
MAX_TOP_K = 1024  # lr_sparse_score_topk's list capacity
QUERY_MAX_BAG = 8192  # LR_QUERY_MAX_BAG: in-range ids one bag of lr_query_token_counts may hold


def json_to_csr(corpus_emb: Sequence[dict]) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """list[dict[str|int -> int]] -> doc-major CSR. The reference's empty-document marker {"-1": 1} has no postings."""
    indptr = np.zeros(len(corpus_emb) + 1, dtype=np.int64)
    toks, imps = [], []
    for i, d in enumerate(corpus_emb):
        n = 0
        for k, v in d.items():
            t = int(k)
            if t < 0 or int(v) <= 0:
                continue
            toks.append(t)
            imps.append(int(v))
            n += 1
        indptr[i + 1] = indptr[i] + n
    return indptr, np.asarray(toks, dtype=np.int32), np.asarray(imps, dtype=np.int64)


def parse_queries(query_emb: Sequence, vocab_size: Optional[int] = None) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Pseudo-query strings / dicts -> CSR of (token, count). A token repeated in the string counts that many times,
    which is what Lucene's boolean query of repeated terms scores (exact_search_base.py:413-424)."""
    indptr = np.zeros(len(query_emb) + 1, dtype=np.int32)
    toks, cnts = [], []
    for i, qe in enumerate(query_emb):
        if isinstance(qe, str):
            c = Counter(int(t) for t in qe.split())
        elif isinstance(qe, dict):
            c = {int(k): int(v) for k, v in qe.items()}
        else:
            c = Counter(int(t) for t in qe)
        n = 0
        for t, v in c.items():
            if t < 0 or v <= 0 or (vocab_size is not None and t >= vocab_size):
                continue  # a token the corpus never produced matches nothing
            toks.append(t)
            cnts.append(v)
            n += 1
        indptr[i + 1] = indptr[i] + n
    return indptr, np.asarray(toks, dtype=np.int32), np.asarray(cnts, dtype=np.int32)


def query_token_counts(ids: torch.Tensor, offsets: torch.Tensor, vocab_size: int, kind: str = "sum",
                       max_bag: Optional[int] = None, out=None, check: bool = True,
                       workspace: Optional[Workspace] = None):
    """Device form of ``parse_queries`` for token ids: flattened ids + bag offsets (the layout ``B200EmbeddingBag.encode``
    takes) -> the query CSR ``(q_indptr [n_bags+1], q_tok [n_ids], q_cnt [n_ids])`` int32 that ``ImpactIndex.search_device``
    takes, by ``lr_query_token_counts``.  ``kind="sum"`` counts repeats (``Counter(ids)``), ``"bow"`` counts each distinct
    token once (exact_search_base.py:398-424).  Tokens of a bag ascend; ids outside ``[0, vocab_size)`` are dropped, so
    -1 works as padding.  Only the first ``q_indptr[-1]`` rows of ``q_tok`` / ``q_cnt`` hold terms (the rest are 0).

    ``max_bag`` bounds the in-range ids of any bag (default ``min(n_ids, QUERY_MAX_BAG)``, from shapes alone).  A bag
    beyond it, or malformed offsets, leave that bag empty and raise ValueError when ``check`` (a device synchronisation);
    ``check=False`` keeps the call free of host synchronisation, for CUDA-graph capture.  ``out`` = preallocated
    ``(q_indptr, q_tok, q_cnt)`` int32 tensors of those shapes."""
    if kind not in ("sum", "bow"):
        raise ValueError(f"kind must be 'sum' or 'bow', got {kind!r}")
    ids = require_cuda(ids, "ids")
    dev = ids.device
    ids = ids.to(torch.int64).contiguous()
    offs = require_cuda(offsets, "offsets").to(dev, torch.int64).contiguous()
    if ids.ndim != 1 or offs.ndim != 1 or offs.numel() < 1:
        raise ValueError("ids and offsets must be 1-D, with at least one bag")
    n_ids, n_bags = ids.numel(), offs.numel()
    max_bag = min(n_ids, QUERY_MAX_BAG) if max_bag is None else int(max_bag)
    if out is None:
        out = (torch.empty(n_bags + 1, dtype=torch.int32, device=dev),
               torch.empty(max(n_ids, 1), dtype=torch.int32, device=dev),
               torch.empty(max(n_ids, 1), dtype=torch.int32, device=dev))
    q_indptr, q_tok, q_cnt = out
    for t, n in ((q_indptr, n_bags + 1), (q_tok, n_ids), (q_cnt, n_ids)):
        if t.dtype != torch.int32 or not t.is_contiguous() or t.device != dev or t.numel() < max(n, 1) or t.ndim != 1:
            raise ValueError(f"out tensors must be contiguous 1-D int32 on {dev}: [n_bags + 1], [n_ids], [n_ids]")
    lib = _C.load()
    ws = (workspace or _WS).get(lib.lr_query_token_counts_scratch_bytes(n_ids, n_bags), dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _C.check(lib.lr_query_token_counts(ids.data_ptr(), offs.data_ptr(), n_ids, n_bags, int(vocab_size), max_bag,
                                           int(kind == "bow"), q_indptr.data_ptr(), q_tok.data_ptr(), q_cnt.data_ptr(),
                                           err.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr(dev)))
    if check and int(err.item()) != 0:
        raise ValueError(f"query_token_counts: a bag holds more than max_bag={max_bag} in-range ids, or the offsets are "
                         "not ascending within [0, n_ids]")
    return q_indptr, q_tok, q_cnt


class ImpactIndex(DocDeletions):
    """Token-major inverted index resident in HBM: post_indptr [V+1] i64, post_doc i32 (ascending per token),
    post_imp u16, plus per-token block pointers (see include/lr_b200.h).  ``delete(ids)`` / ``restore(ids)`` take ids
    ``id_offset + row`` and hide documents from every later search without touching the postings."""

    def __init__(self, vocab_size: int, device: Optional[torch.device] = None, id_offset: int = 0):
        self.V = int(vocab_size)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.id_offset = int(id_offset)
        self._doc_chunks: list[tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = []
        self.N = 0
        self._built = None
        self._live = None

    def _live_rows(self) -> int:
        return self.N

    def add_csr(self, indptr, tok, imp) -> None:
        """Append documents given as doc-major CSR (numpy or torch, host or device).  Staged as (lengths i32, tokens i32,
        impacts i16 = the uint16 bit pattern): 6 bytes per posting, the size of the final index."""
        ip = torch.as_tensor(indptr).to(torch.int64)
        tk = torch.as_tensor(tok).to(self.device)
        im = torch.as_tensor(imp).to(self.device)
        if tk.numel() and (int(tk.min()) < 0 or int(tk.max()) >= self.V):
            raise ValueError("token id out of range [0, vocab_size)")
        if im.dtype != torch.int16:  # int16 = uint16 bit pattern from sparsify_quantize, already in range
            if im.numel() and (int(im.min()) < 0 or int(im.max()) > 65535):
                raise ValueError("impacts must fit uint16")
            im = im.to(torch.int32).to(torch.int16)  # two's-complement wrap keeps the low 16 bits
        n_docs = ip.numel() - 1
        lens = (ip[1:] - ip[:-1]).to(self.device, torch.int32)
        if int(lens.sum()) != tk.numel() or tk.numel() != im.numel():
            raise ValueError("indptr, tok and imp disagree on the number of postings")
        self._doc_chunks.append((lens, tk.to(torch.int32).contiguous(), im.contiguous()))
        self.N += n_docs
        self._built = None
        self._extend_live(self.N - n_docs)

    def add_dense_rows(self, tok: torch.Tensor, imp: torch.Tensor) -> None:
        """Append documents given as fixed-width rows ``tok [n, w]`` / ``imp [n, w]`` (device tensors); a token repeated
        inside a row keeps its first impact (a sparse vector has one weight per token)."""
        tk = require_cuda(tok, "tok").to(torch.int32)
        n, w = tk.shape
        order = torch.sort(tk, dim=1, stable=True)
        st = order.values
        si = torch.gather(require_cuda(imp, "imp").to(torch.int32), 1, order.indices)
        keep = torch.ones_like(st, dtype=torch.bool)
        keep[:, 1:] = st[:, 1:] != st[:, :-1]
        lens = keep.sum(dim=1)
        indptr = torch.zeros(n + 1, dtype=torch.int64, device=tk.device)
        indptr[1:] = torch.cumsum(lens, 0)
        self.add_csr(indptr, st[keep], si[keep])

    def build(self):
        if self._built is not None:
            return self._built
        if self.N == 0:
            raise RuntimeError("index is empty")
        dev = self.device
        # index time (not the query path): counting sort by token, one staged chunk at a time, so that the peak is the
        # final index + the staged chunks (6 B per posting each) + one piece of scratch — 8.8M x 256 postings build on
        # one GPU.  Chunks are visited in document order and sorted stably, so doc ids ascend inside a posting list.
        counts = torch.zeros(self.V, dtype=torch.int64, device=dev)
        for _, tk, _ in self._doc_chunks:
            counts += torch.bincount(tk, minlength=self.V)
        post_indptr = torch.zeros(self.V + 1, dtype=torch.int64, device=dev)
        post_indptr[1:] = torch.cumsum(counts, 0)
        nnz = int(post_indptr[-1])
        post_doc = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        post_imp = torch.empty(max(nnz, 1), dtype=torch.int16, device=dev)  # uint16 bit pattern
        if nnz == 0:
            post_doc.zero_()
            post_imp.zero_()
        cursor = post_indptr[:-1].clone()
        doc0 = 0
        piece = 1 << 25  # postings sorted per step
        for lens, tk, im in self._doc_chunks:
            n_docs = lens.numel()
            ends = torch.cumsum(lens.to(torch.int64), 0)
            for a in range(0, tk.numel(), piece):
                e = min(a + piece, tk.numel())
                t = tk[a:e]
                # document of posting j = number of documents that end at or before j
                doc = (torch.searchsorted(ends, torch.arange(a, e, device=dev), right=True) + doc0).to(torch.int32)
                st = torch.sort(t, stable=True)
                c = torch.bincount(t, minlength=self.V)
                run_start = torch.cumsum(c, 0) - c
                tl = st.values.long()
                pos = cursor[tl] + (torch.arange(e - a, device=dev) - run_start[tl])
                post_doc[pos] = doc[st.indices]
                post_imp[pos] = im[a:e][st.indices]
                cursor += c
                del doc, st, c, run_start, tl, pos
            doc0 += n_docs
        # the staged rows stay (6 B per posting): a later add_csr() + build() re-sorts everything, as repeated
        # AnseriniSearch.index() calls append to one collection (anserini_search.py:89-111)
        lib = _C.load()
        bd = lib.lr_sparse_block_docs()
        nblk = (self.N + bd - 1) // bd
        blockptr = torch.empty(self.V * (nblk + 1), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _C.check(lib.lr_sparse_build_blockptr(post_indptr.data_ptr(), post_doc.data_ptr(), self.V, self.N,
                                                  blockptr.data_ptr(), stream_ptr(dev)))
        self._built = (post_indptr, post_doc, post_imp, blockptr)
        return self._built

    def search_device(self, q_indptr, q_tok, q_cnt, k: int, return_keys: bool = False,
                      workspace: Optional[Workspace] = None, live: Optional[torch.Tensor] = None,
                      allow: Optional[torch.Tensor] = None, q_filter: Optional[torch.Tensor] = None):
        """(scores f32 [Q, k], ids i64 [Q, k]) of the query CSR; ``workspace`` as in ``flatip_topk`` (default: a
        module-wide buffer per device, stream and thread).  ``live`` (replaces the index's own deletions bitmap for this
        call), ``allow`` and ``q_filter``: document bitmaps as in ``flatip_topk``."""
        post_indptr, post_doc, post_imp, blockptr = self.build()
        dev = self.device
        qi = torch.as_tensor(q_indptr).to(dev, torch.int32).contiguous()
        qt = torch.as_tensor(q_tok).to(dev, torch.int32).contiguous()
        qc = torch.as_tensor(q_cnt).to(dev, torch.int32).contiguous()
        if qt.numel() == 0:
            qt = torch.zeros(1, dtype=torch.int32, device=dev)
            qc = torch.zeros(1, dtype=torch.int32, device=dev)
        Q = qi.numel() - 1
        flt = filter_args(self._live if live is None else live, allow, q_filter, Q, dev)
        lib = _C.load()
        ws = (workspace or _WS).get(lib.lr_sparse_score_workspace_bytes(Q, self.N, k), dev)
        scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
        ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
        keys = torch.empty((Q, k), dtype=torch.int64, device=dev) if return_keys else None
        args = (qi.data_ptr(), qt.data_ptr(), qc.data_ptr(), Q, post_indptr.data_ptr(), post_doc.data_ptr(),
                post_imp.data_ptr(), blockptr.data_ptr(), self.V, self.N, self.id_offset, int(k), scores.data_ptr(),
                ids.data_ptr(), None if keys is None else keys.data_ptr())
        with torch.cuda.device(dev):
            if flt is None:
                _C.check(lib.lr_sparse_score_topk(*args, ws.data_ptr(), ws.numel(), stream_ptr(dev)))
            else:
                _C.check(lib.lr_sparse_score_topk_filtered(*args, *flt, ws.data_ptr(), ws.numel(), stream_ptr(dev)))
        return (scores, ids, keys) if return_keys else (scores, ids)


class ImpactSearch:
    """``AnseriniSearch`` surface (anserini_search.py:31-216) over ``ImpactIndex`` (impact search only)."""

    def __init__(self, model=None, batch_size: int = 128, corpus_chunk_size: Optional[int] = None,
                 vocab_size: Optional[int] = None, **kwargs):
        self.model = model
        self.batch_size = batch_size
        self.corpus_chunk_size = batch_size * 800 if corpus_chunk_size is None else corpus_chunk_size
        self.show_progress_bar = kwargs.get("show_progress_bar", True)
        self.convert_to_tensor = kwargs.get("convert_to_tensor", True)
        if not kwargs.get("anserini_impact_search", True):
            raise NotImplementedError("BM25 scoring is not on the hot path; only impact (dot-product) search is built")
        self.vocab_size = vocab_size
        self.device = kwargs.get("device", None)
        self._index: Optional[ImpactIndex] = None
        self._corpus_ids: list = []
        self._pending: list = []
        self.n_dumped = 0

    @classmethod
    def name(cls):
        return "impact_b200_search"

    def _clear(self):
        self._index = None
        self._corpus_ids = []
        self._pending = []
        self.n_dumped = 0

    def encode(self, sentences, batch_size: int, **kwargs):
        return self.model.encode(sentences=sentences, batch_size=batch_size, **kwargs)

    def encode_queries(self, queries, batch_size: int, **kwargs):
        return self.model.encode_queries(queries=queries, batch_size=batch_size, **kwargs)

    def encode_corpus(self, corpus, batch_size: int, **kwargs):
        return self.model.encode_corpus(corpus=corpus, batch_size=batch_size, **kwargs)

    def index(self, corpus_emb, corpus_ids: Sequence[str]):
        """corpus_emb: list[dict[str,int]] (JsonVectorCollection) or a CSR triple (indptr, tok, imp)."""
        if isinstance(corpus_emb, tuple) and len(corpus_emb) == 3:
            csr = corpus_emb
        else:
            if len(corpus_emb) and isinstance(corpus_emb[0], str):
                corpus_emb = [dict(Counter(s.split())) for s in corpus_emb]  # JsonCollection pseudo-text
            csr = json_to_csr(corpus_emb)
        self._pending.append(csr)
        self._corpus_ids.extend(corpus_ids)
        self.n_dumped += len(corpus_ids)
        self._index = None

    # ---- on-disk compatibility with the reference's dump (anserini_search.py:89-111): JsonVectorCollection lines
    #      {"id": ..., "content": "", "vector": {token: int}} in corpusNNNNN.jsonl files of 2000 documents
    def dump_jsonl(self, folder: str, chunk_docs: int = 2000) -> None:
        """Write the pending corpus in the reference's JSONL layout (what IndexCollection would ingest)."""
        import json
        import os

        os.makedirs(folder, exist_ok=True)
        n = 0
        f = None
        for (indptr, tok, imp), ids in self._pending_with_ids():
            ip = torch.as_tensor(indptr).tolist()
            tk = torch.as_tensor(tok).tolist()
            im = torch.as_tensor(imp).cpu()
            im = ((im.to(torch.int32) & 0xFFFF) if im.dtype == torch.int16 else im).tolist()
            for j, cid in enumerate(ids):
                if n % chunk_docs == 0:
                    if f:
                        f.close()
                    f = open(os.path.join(folder, f"corpus{n // chunk_docs:05d}.jsonl"), "w")
                vec = {str(tk[i]): int(im[i]) for i in range(ip[j], ip[j + 1])} or {"-1": 1}
                f.write(json.dumps({"id": cid, "content": "", "vector": vec}) + "\n")
                n += 1
        if f:
            f.close()

    def index_from_jsonl(self, folder: str) -> int:
        """Ingest a corpus dumped by the reference's AnseriniSearch.index (encoded_corpus/corpusNNNNN.jsonl)."""
        import glob
        import json
        import os

        n = 0
        for path in sorted(glob.glob(os.path.join(folder, "corpus*.jsonl"))):
            ids, vecs = [], []
            with open(path) as f:
                for line in f:
                    if not line.strip():
                        continue
                    rec = json.loads(line)
                    ids.append(rec["id"])
                    vecs.append(rec.get("vector") or {})
            if ids:
                self.index(vecs, ids)
                n += len(ids)
        return n

    def _pending_with_ids(self):
        pos = 0
        for csr in self._pending:
            n_docs = len(csr[0]) - 1
            yield csr, self._corpus_ids[pos:pos + n_docs]
            pos += n_docs

    def retrieve_arrays(self, query_emb: Sequence, top_k: int):
        """Device arrays (scores f32 [Q,k], doc positions i64 [Q,k], -1 padded) — no dict materialisation."""
        idx = self._ensure_index()
        if int(top_k) > MAX_TOP_K:
            # the reference hands `-hits top_k` to Anserini unchanged (anserini_search.py:178-202); silently returning
            # fewer sparse hits would change the min-max normalisation of a hybrid fusion
            raise ValueError(f"top_k={top_k} exceeds the sparse kernel's limit of {MAX_TOP_K} results per query")
        qi, qt, qc = parse_queries(query_emb, idx.V)
        return idx.search_device(qi, qt, qc, int(top_k))

    def _ensure_index(self) -> ImpactIndex:
        if self._index is None:
            if not self._pending:
                raise RuntimeError("index() must be called before retrieve_with_emb()")
            V = self.vocab_size
            if V is None:
                V = 1 + max((int(torch.as_tensor(c[1]).max()) if len(c[1]) else 0) for c in self._pending)
            idx = ImpactIndex(V, device=self.device)
            for c in self._pending:
                idx.add_csr(*c)
            self._index = idx
        return self._index

    def retrieve_with_emb(self, query_emb: Sequence, query_ids: Sequence[str], top_k: int) -> dict:
        """anserini_search.py:143-216: ``dict[qid -> dict[pid -> score]]``; Lucene writes no TREC line for a query without
        hits (:208-214), so such queries are absent."""
        from .search import rows_to_dict

        scores, ids = self.retrieve_arrays(query_emb, top_k)
        return rows_to_dict(scores, ids, query_ids, self._corpus_ids, keep_empty=False)

    def search(self, corpus, queries, top_k: int = 1000, score_function: str = None, return_sorted: bool = False,
               ignore_identical_ids: bool = False, **kwargs) -> dict:
        """AnseriniSearch.search (anserini_search.py:218-309): encode the queries, encode + index the corpus in chunks
        (longest document first), retrieve once, clear.  Like the reference, `ignore_identical_ids` is accepted and unused."""
        from .search import sorted_corpus

        if not isinstance(queries, dict) or not isinstance(corpus, dict):
            raise NotImplementedError("ImpactSearch.search takes dict corpora / queries")
        query_ids = list(queries.keys())
        query_embeddings = self.model.encode_queries([queries[qid] for qid in queries], batch_size=self.batch_size,
                                                     show_progress_bar=self.show_progress_bar,
                                                     convert_to_tensor=self.convert_to_tensor)
        if isinstance(query_embeddings, dict):
            for key in ("token_id_reps", "sparse_reps"):
                if query_embeddings.get(key) is not None:
                    query_embeddings = query_embeddings[key]
                    break
            else:
                raise ValueError(f"HybridModel: query embeddings with keys {query_embeddings.keys()} hold no sparse vector")
        corpus_ids, corpus_list = sorted_corpus(corpus)
        for start in range(0, len(corpus_list), self.corpus_chunk_size):
            sub = self.model.encode_corpus(corpus_list[start:start + self.corpus_chunk_size], batch_size=self.batch_size,
                                           show_progress_bar=self.show_progress_bar,
                                           convert_to_tensor=self.convert_to_tensor)
            if isinstance(sub, dict):
                if "sparse_reps" not in sub:
                    raise ValueError(f"HybridModel: Return Multi-vector with keys {sub.keys()}, but not `sparse_reps`")
                sub = sub["sparse_reps"]
            self.index(sub, corpus_ids[start:start + self.corpus_chunk_size])
        results = self.retrieve_with_emb(query_embeddings, query_ids, top_k=top_k)
        self._clear()
        return results
