"""oracle.py — CPU restatement of the reference's serving-side retrieval path.

TEST INFRASTRUCTURE ONLY.  Nothing under lightretriever_b200/ may import this module; only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs do, and only as the checker or as the
timed CPU baseline — never as the product path.

The reference (caskcsg/lightretriever, /root/reference) is pure Python on top of torch, Faiss, Anserini (JVM) and a
Rust wheel.  Each function cites the reference lines it follows.  Pin status (oracle/gen_golden.py produced
tests/golden/*.npz by importing the reference itself in the build container):

  embbag_encode         PINNED   = torch.nn.EmbeddingBag (the reference's own dependency) + slice + F.normalize
  lasttoken_head        PINNED   vs lightretriever.finetune.dense_pooling.pooling (imported)
  sparse_attention_mask PINNED   vs lightretriever.finetune.sparse_pooling.get_sparse_attention_mask (imported)
  max_linear_map        PINNED   vs lightretriever.utils.max_linear_map.max_linear_mapping (imported)
  top_k_sampling        PINNED   vs lightretriever.finetune.sparse_pooling.top_k_sampling (imported)
  top_p_sampling        PINNED   vs lightretriever.finetune.sparse_pooling.top_p_sampling (imported; gen_golden_r2.py)
  quantize_reps         PINNED   vs SparseConverterMixin.convert_sparse_reps_to_json_pt (imported with the missing Rust
                                 wheel stubbed); the Rust converter itself is absent -> its rounding is PARITY UNPINNED
  fuse_linear/fuse_rrf  PINNED   vs lightretriever.retriever.score_fuse_utils (imported)
  add_to_heap           PINNED   vs HybridSearch._add_to_heap (imported)
  flatten_token_ids     PINNED   vs tokenize_nonctx_qry_emb_bag when the module imports, else restated (see gen_golden)
  flatip_topk           PARITY UNPINNED: faiss (>=1.7.4, no lock file) is not installed and the reference holds no golden
                                 vectors for it; restated from its call sites (retriever/faiss_index.py:27-40) and anchored
                                 on the score definition torch.matmul(q, p.T) (finetune/modeling_encoder.py:414-427); the
                                 score line of scripts/asymmetric_dense_infer.ipynb:231 is exec'd by gen_golden_r2.py
  impact_topk           io.anserini:anserini:0.25.0 (JVM) is absent, so Lucene's tie order stays PARITY UNPINNED; the SCORE
                                 definition is PINNED: impact_scores equals the notebook's own compute_similarity cell
                                 (scripts/asymmetric_sparse_infer.ipynb:207-228), exec'd by gen_golden_r2.py
"""
from __future__ import annotations

import heapq
from collections import Counter
from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------- K1
def flatten_token_ids(token_id_lists: Sequence[Sequence[int]]):
    """finetune/nonctx_emb_utils.py:217-218: offsets = cumsum([0] + lens[:-1]); input_ids = concat."""
    offsets = np.cumsum([0] + [len(t) for t in token_id_lists[:-1]]).astype(np.int64)
    input_ids = np.concatenate([np.asarray(t, dtype=np.int64) for t in token_id_lists]).astype(np.int64)
    return input_ids, offsets


def emb_bag_table_inputs(prompt_token_ids: Sequence[int], eos_token_id: int, start: int, end: int) -> np.ndarray:
    """finetune/nonctx_emb_utils.py:270-296: rows ``prompt (with bos) + [v] + [eos]`` for v in [start, end) — plain loops."""
    rows = []
    for v in range(start, end):
        rows.append(list(prompt_token_ids) + [v, eos_token_id])
    return np.asarray(rows, dtype=np.int64).reshape(end - start, len(prompt_token_ids) + 2)


def embbag_encode(ids, offsets, table, padding_idx: Optional[int] = None, shrink_dim: Optional[int] = None,
                  normalize: bool = False) -> torch.Tensor:
    """finetune/modeling_hybrid.py:474 (emb_bag.forward) + :487-488 (shrink) + :489-490 (F.normalize), fp32.

    The bag is what the reference builds: EmbeddingBag.from_pretrained(table, padding_idx=pad) -> mode='mean'
    (finetune/nonctx_emb_utils.py:310-312)."""
    table = torch.as_tensor(table).float()
    bag = torch.nn.EmbeddingBag.from_pretrained(table, padding_idx=padding_idx)
    reps = bag.forward(input=torch.as_tensor(ids).long(), offsets=torch.as_tensor(offsets).long())
    if shrink_dim:
        reps = reps[..., :shrink_dim]
    if normalize:
        reps = F.normalize(reps, p=2, dim=-1)
    return reps


def lasttoken_head(last_hidden, attention_mask, shrink_dim: Optional[int] = None, normalize: bool = False):
    """finetune/dense_pooling.py:48-55 ('lasttoken') + modeling_hybrid.py:266-278 (shrink, normalize)."""
    last_hidden = torch.as_tensor(last_hidden).float()
    attention_mask = torch.as_tensor(attention_mask)
    left_padding = bool(attention_mask[:, -1].sum() == attention_mask.shape[0])
    if left_padding:
        reps = last_hidden[:, -1]
    else:
        idx = attention_mask.sum(dim=1) - 1
        reps = last_hidden[torch.arange(last_hidden.shape[0]), idx]
    if shrink_dim:
        reps = reps[..., :shrink_dim]
    if normalize:
        reps = F.normalize(reps, p=2, dim=-1)
    return reps


# ----------------------------------------------------------------------------------------------- K2
def sort_desc_id_asc(scores: np.ndarray, ids: np.ndarray, k: int):
    """(score desc, id asc) ordering of one candidate row, truncated to k."""
    order = np.lexsort((ids, -scores.astype(np.float64)))[:k]
    return scores[order], ids[order]


def flatip_scores(q, corpus) -> torch.Tensor:
    """The score definition of the dense path: scripts/asymmetric_dense_infer.ipynb:231
    (`scores = query_embeddings @ corpus_embedding.T`), finetune/modeling_encoder.py:414-427; fp32."""
    return torch.as_tensor(q).float() @ torch.as_tensor(corpus).float().T


def flatip_topk(q, corpus, k: int, id_offset: int = 0, chunk: int = 65536):
    """retriever/faiss_index.py:27-40: IndexFlatIP.search(q, k) -> (scores f32 [Q,k] descending, ids i64 [Q,k]).

    fp32 inner products (the reference keeps Faiss in fp32, faiss_index.py:67).  Equal scores are ordered by ascending
    id (Faiss leaves it unspecified); fewer than k documents -> (-inf, -1) tail (Faiss's convention)."""
    q = torch.as_tensor(q).float()
    corpus = torch.as_tensor(corpus).float()
    Q, N = q.shape[0], corpus.shape[0]
    best_s = np.full((Q, 0), -np.inf, dtype=np.float32)
    best_i = np.full((Q, 0), -1, dtype=np.int64)
    for lo in range(0, N, chunk):
        s = flatip_scores(q, corpus[lo:lo + chunk]).numpy()
        i = np.broadcast_to(np.arange(lo, lo + s.shape[1], dtype=np.int64), s.shape)
        cs = np.concatenate([best_s, s], axis=1)
        ci = np.concatenate([best_i, i], axis=1)
        ns, ni = np.empty((Q, min(k, cs.shape[1])), np.float32), np.empty((Q, min(k, cs.shape[1])), np.int64)
        for r in range(Q):
            ns[r], ni[r] = sort_desc_id_asc(cs[r], ci[r], k)
        best_s, best_i = ns, ni
    if best_s.shape[1] < k:
        pad = k - best_s.shape[1]
        best_s = np.concatenate([best_s, np.full((Q, pad), -np.inf, np.float32)], axis=1)
        best_i = np.concatenate([best_i, np.full((Q, pad), -1, np.int64)], axis=1)
    return best_s, np.where(best_i >= 0, best_i + id_offset, -1)


def flatip_topk_fast(q, corpus, k: int, chunk: int = 262144):
    """Same result up to tie order, vectorised (torch.topk per chunk + merge) — the CPU baseline that gets timed."""
    q = torch.as_tensor(q).float()
    corpus = torch.as_tensor(corpus)
    best_s = best_i = None
    for lo in range(0, corpus.shape[0], chunk):
        s = q @ corpus[lo:lo + chunk].float().T
        kk = min(k, s.shape[1])
        ts, ti = torch.topk(s, kk, dim=1, sorted=True)
        ti = ti + lo
        if best_s is None:
            best_s, best_i = ts, ti
        else:
            cs, ci = torch.cat([best_s, ts], 1), torch.cat([best_i, ti], 1)
            ms, mi = torch.topk(cs, min(k, cs.shape[1]), dim=1, sorted=True)
            best_s, best_i = ms, torch.gather(ci, 1, mi)
    return best_s, best_i


def add_to_heap(sub_results: dict, result_heaps: dict, top_k: int, ignore_identical_ids: bool = False) -> dict:
    """retriever/hybrid_search.py:182-205."""
    for qid, pid_to_score in sub_results.items():
        for pid, score in pid_to_score.items():
            if ignore_identical_ids and (qid == pid):
                continue
            if qid not in result_heaps:
                result_heaps[qid] = []
            if len(result_heaps[qid]) < top_k:
                heapq.heappush(result_heaps[qid], (score, pid))
            else:
                heapq.heappushpop(result_heaps[qid], (score, pid))
    return result_heaps


def merge_topk(score_lists: Sequence[np.ndarray], id_lists: Sequence[np.ndarray], k: int):
    """Exact top-k of the union of per-chunk / per-shard top-k lists (the array form of add_to_heap)."""
    cs = np.concatenate(score_lists, axis=1)
    ci = np.concatenate(id_lists, axis=1)
    Q = cs.shape[0]
    out_s = np.full((Q, k), -np.inf, np.float32)
    out_i = np.full((Q, k), -1, np.int64)
    for r in range(Q):
        valid = ci[r] >= 0
        s, i = sort_desc_id_asc(cs[r][valid], ci[r][valid], k)
        out_s[r, :len(s)], out_i[r, :len(i)] = s, i
    return out_s, out_i


# key encoding used on the wire between shards (documented in include/lr_b200.h)
def f32_to_key(x: np.ndarray) -> np.ndarray:
    u = (np.asarray(x, np.float32) + np.float32(0.0)).view(np.uint32)
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def key_to_f32(k: np.ndarray) -> np.ndarray:
    k = np.asarray(k, np.uint32)
    u = np.where(k & np.uint32(0x80000000), k & np.uint32(0x7FFFFFFF), ~k).astype(np.uint32)
    return u.view(np.float32)


def encode_keys(scores: np.ndarray, ids: np.ndarray) -> np.ndarray:
    hi = f32_to_key(scores).astype(np.uint64) << np.uint64(32)
    lo = (np.uint64(0xFFFFFFFF) - np.asarray(ids, np.int64).astype(np.uint64)) & np.uint64(0xFFFFFFFF)
    return np.where(np.asarray(ids) >= 0, hi | lo, np.uint64(0)).astype(np.uint64)


def decode_keys(keys: np.ndarray):
    keys = np.asarray(keys, np.uint64)
    scores = key_to_f32((keys >> np.uint64(32)).astype(np.uint32))
    ids = (np.uint64(0xFFFFFFFF) - (keys & np.uint64(0xFFFFFFFF))).astype(np.int64)
    return np.where(keys != 0, scores, -np.inf).astype(np.float32), np.where(keys != 0, ids, -1)


# ----------------------------------------------------------------------------------------------- K3
def get_prompt_mask(input_ids: torch.Tensor, sep_token_id: int):
    """finetune/sparse_pooling.py:43-59."""
    if sep_token_id not in input_ids:
        return torch.zeros_like(input_ids, dtype=torch.bool)
    positions = torch.argmax((input_ids == sep_token_id).int(), dim=-1)
    if torch.all(positions == input_ids.shape[-1] - 1):
        return torch.zeros_like(input_ids, dtype=torch.bool)
    col = torch.arange(input_ids.shape[-1]).unsqueeze(0)
    return col <= positions.unsqueeze(1)


def sparse_attention_mask(input_ids, attention_mask, sep_token_id: int, remove_prompt: bool = False):
    """finetune/sparse_pooling.py:23-41: drop position 0, the last valid position, pads (and the prompt)."""
    input_ids, attention_mask = torch.as_tensor(input_ids), torch.as_tensor(attention_mask)
    mask = attention_mask.bool()
    if remove_prompt:
        mask = mask.masked_fill(get_prompt_mask(input_ids, sep_token_id), False)
    bs = torch.arange(attention_mask.shape[0])
    last = attention_mask.sum(dim=1) - 1
    mask[bs, [0] * attention_mask.shape[0]] = False
    mask[bs, last] = False
    return mask


def max_linear_map(hidden, weight_dv, bias=None, mask=None, fill: Optional[float] = None) -> torch.Tensor:
    """utils/max_linear_map.py:10-90: out[b,v] = max_t (h[b,t] @ W + bias) with masked positions (and the initial
    value) at finfo(dtype).min.  fp32 math; `fill` defaults to finfo(bfloat16).min, the value the reference uses under
    bf16 autocast (max_linear_map.py:27,58)."""
    h = torch.as_tensor(hidden).float()
    W = torch.as_tensor(weight_dv).float()
    fill = torch.finfo(torch.bfloat16).min if fill is None else fill
    out = torch.full((h.shape[0], W.shape[1]), fill, dtype=torch.float32)
    for t in range(h.shape[1]):
        logits = h[:, t] @ W
        if bias is not None:
            logits = logits + torch.as_tensor(bias).float()
        if mask is not None:
            logits = logits.masked_fill(~torch.as_tensor(mask)[:, t:t + 1].bool(), fill)
        out = torch.where(logits > out, logits, out)
    return out


def top_k_sampling(scores: torch.Tensor, top_k: int, filter_value: float = 0.0, min_tokens_to_keep: int = 1):
    """finetune/sparse_pooling.py:89-106 (all ties at the threshold survive)."""
    if top_k <= 0:
        return scores
    top_k = min(max(top_k, min_tokens_to_keep), scores.size(-1))
    remove = scores < torch.topk(scores, top_k)[0][..., -1, None]
    return scores.masked_fill(remove, filter_value)


def top_p_sampling(scores: torch.Tensor, top_p: float, filter_value: float = 0.0, min_tokens_to_keep: int = 1):
    """finetune/sparse_pooling.py:64-87: ascending sort, softmax, cumsum; remove while cumulative <= 1 - top_p, never the
    last min_tokens_to_keep of the sorted order.  Returns (filtered scores, cumulative probability of every entry in
    the original indexing) — the second value lets a test state which entries sit on the bound."""
    if top_p <= 0 or top_p >= 1:
        return scores, None
    sorted_logits, sorted_indices = torch.sort(scores, descending=False, stable=True)
    cum = sorted_logits.softmax(dim=-1).cumsum(dim=-1)
    remove_sorted = cum <= (1 - top_p)
    remove_sorted[..., -min_tokens_to_keep:] = False
    remove = remove_sorted.scatter(1, sorted_indices, remove_sorted)
    cum_orig = torch.empty_like(cum).scatter(1, sorted_indices, cum)
    return scores.masked_fill(remove, filter_value), cum_orig


def get_sparse_emb(logits, relu: bool = True, log1p: bool = True, top_k: int = 0, min_tokens_to_keep: int = 8,
                   top_p: float = 1.0):
    """finetune/modeling_hybrid.py:183-201: relu, log1p, top-p (its default 1.0 is a no-op, sparse_pooling.py:73-74), top-k."""
    x = torch.as_tensor(logits).float().clone()
    if relu:
        x = torch.relu(x)
    if log1p:
        x = torch.log1p(x)
    x = top_p_sampling(x, top_p, min_tokens_to_keep=min_tokens_to_keep)[0]
    return top_k_sampling(x, top_k, min_tokens_to_keep=min_tokens_to_keep)


def quantize_reps(reps, quantization_factor: float = 100.0) -> list[dict[str, int]]:
    """finetune/sparse_converter_mixin.py:103-160 (the in-repo torch twin of the Rust converter):
    clamp(min=0) -> round(x*q) -> int, keep non-zeros, empty document -> {"-1": 1}."""
    x = torch.as_tensor(reps).float()
    if x.ndim == 1:
        x = x.unsqueeze(0)
    q = torch.round(torch.clamp(x, min=0.0) * quantization_factor).to(torch.int)
    out = []
    for b in range(q.shape[0]):
        nz = torch.nonzero(q[b]).flatten().tolist()
        d = {str(v): int(q[b, v]) for v in nz}
        out.append(d if d else {"-1": 1})
    return out


# ----------------------------------------------------------------------------------------------- K4
def query_counts(token_ids: Sequence[int], kind: str = "sum") -> dict[int, int]:
    """inference/exact_search_base.py:398-424: 'sum' -> Counter(ids); 'bow' -> {id: 1 for id in set(ids)}."""
    return dict(Counter(token_ids)) if kind == "sum" else {t: 1 for t in set(token_ids)}


def impact_scores(queries: Sequence[dict], docs: Sequence[dict]) -> np.ndarray:
    """scripts/asymmetric_sparse_infer.ipynb:207-228 (compute_similarity), int64: sum_t count_q(t) * impact_d(t)."""
    out = np.zeros((len(queries), len(docs)), dtype=np.int64)
    inv: dict[int, list] = {}
    for j, d in enumerate(docs):
        for t, w in d.items():
            t = int(t)
            if t >= 0:
                inv.setdefault(t, []).append((j, int(w)))
    for i, q in enumerate(queries):
        for t, c in q.items():
            for j, w in inv.get(int(t), ()):
                out[i, j] += int(c) * w
    return out


def impact_topk(queries: Sequence[dict], docs: Sequence[dict], k: int, id_offset: int = 0):
    """retriever/anserini_search.py:143-216 with -impact -hits k: matching documents only (score > 0), best first;
    ties by ascending document index; missing tail (-inf, -1)."""
    S = impact_scores(queries, docs)
    Q = S.shape[0]
    out_s = np.full((Q, k), -np.inf, np.float32)
    out_i = np.full((Q, k), -1, np.int64)
    for r in range(Q):
        hit = np.nonzero(S[r] > 0)[0]
        order = hit[np.lexsort((hit, -S[r][hit]))][:k]
        out_s[r, :len(order)] = S[r][order].astype(np.float32)
        out_i[r, :len(order)] = order + id_offset
    return out_s, out_i


# ----------------------------------------------------------------------------------------------- fusion
def fuse_linear(results_list: Sequence[dict], weights=(0.7, 0.3), eps: float = 1e-8) -> dict:
    """retriever/score_fuse_utils.py:48-90."""
    fused: dict = {}
    for system_results, weight in zip(results_list, weights):
        for qid, passages in system_results.items():
            qid = str(qid)
            fused.setdefault(qid, {})
            pids = list(passages.keys())
            scores = np.array([float(passages[p]) for p in pids])
            normed = (scores - scores.min()) / (scores.max() - scores.min() + eps)
            for p, s in zip(pids, normed * weight):
                fused[qid][str(p)] = fused[qid].get(str(p), 0.0) + float(s)
    return fused


def fuse_rrf(results_list: Sequence[dict], k: int = 60) -> dict:
    """retriever/score_fuse_utils.py:3-46."""
    fused: dict = {}
    for system_results in results_list:
        for qid, passages in system_results.items():
            qid = str(qid)
            fused.setdefault(qid, {})
            pids = list(passages.keys())
            scores = np.array([float(passages[p]) for p in pids])
            order = np.argsort(-scores)
            for rank, p in enumerate(np.array(pids)[order], start=1):
                fused[qid][str(p)] = fused[qid].get(str(p), 0.0) + float(1 / (k + rank))
    return fused


# ----------------------------------------------------------------------------------------------- comparator
def check_topk_parity(got_scores, got_ids, ref_scores_full: np.ndarray, k: int, rtol: float = 1e-2,
                      id_offset: int = 0, atol: float = 1e-5) -> None:
    """The north star's parity rule for the dense path, against the FULL fp32 reference score matrix [Q, N]:

      * every returned score is within `rtol` relative (+atol) of the fp32 reference score of the returned id;
      * ids match the fp32 top-k exactly, except documents whose reference score lies within
        tol = rtol * |s_k| (+atol) of the k-th reference score (the bf16-vs-fp32 tie band): every returned id must have
        ref score >= s_k - tol and every reference id with score > s_k + tol must be returned;
      * returned scores are sorted descending; ids are unique.
    """
    got_scores = np.asarray(got_scores, np.float32)
    got_ids = np.asarray(got_ids, np.int64)
    Q, N = ref_scores_full.shape
    kk = min(k, N)
    for r in range(Q):
        ids = got_ids[r]
        valid = ids >= 0
        assert valid[:kk].all() and not valid[kk:].any(), f"row {r}: padding misplaced"
        loc = ids[:kk] - id_offset
        assert len(np.unique(loc)) == kk, f"row {r}: duplicate ids"
        assert (np.diff(got_scores[r, :kk]) <= 0).all(), f"row {r}: scores not sorted descending"
        ref_row = ref_scores_full[r]
        ref_at = ref_row[loc]
        np.testing.assert_allclose(got_scores[r, :kk], ref_at, rtol=rtol, atol=atol,
                                   err_msg=f"row {r}: score mismatch")
        order = np.lexsort((np.arange(N), -ref_row.astype(np.float64)))
        s_k = ref_row[order[kk - 1]]
        tol = rtol * abs(float(s_k)) + atol
        assert (ref_at >= s_k - tol).all(), f"row {r}: returned a document below the tie band"
        must = order[:kk][ref_row[order[:kk]] > s_k + tol]
        missing = np.setdiff1d(must, loc)
        assert missing.size == 0, f"row {r}: missing documents above the tie band: {missing[:5]}"
        if kk < k:
            assert np.isneginf(got_scores[r, kk:]).all(), f"row {r}: padding scores must be -inf"


def check_sparse_impacts(got_json: Sequence[dict], reps: np.ndarray, eps: np.ndarray, top_k: int,
                         min_tokens_to_keep: int = 8, quantization_factor: float = 100.0):
    """The parity rule of the fused sparse head (max-linear -> relu/log1p -> top-k -> quantise) against high-precision
    reference reps [B, V], given a per-entry bound `eps` [B, V] of the kernel's rep error:

      * every emitted impact equals round_half_even(q * ref); a difference of 1 is allowed only where q * ref lies within
        q * eps of a half-integer (the rounding is undecided there);
      * a token may be in one set and not the other only inside the top-k tie band (|ref - ref_kth| <= eps + eps_kth)
        or where q * ref lies within q * eps of 0.5 (the `impact >= 1` cut).

    Returns (violations, band): a list of (document, token, got, expected) that break the rule, and the number of tokens
    that were accepted only because they fell inside a band (a test reports it, so that a vacuous pass shows up)."""
    reps = np.asarray(reps, np.float64)
    eps = np.asarray(eps, np.float64)
    B, V = reps.shape
    q = float(quantization_factor)
    keff = min(max(top_k, min_tokens_to_keep), V) if top_k > 0 else 0
    violations, band = [], 0
    for b in range(B):
        x, e = reps[b], eps[b]
        pos = np.maximum(x, 0.0)
        if keff:
            j = np.argpartition(-pos, keff - 1)[keff - 1]
            kth, e_kth = pos[j], e[j]
            kept = pos >= kth
        else:
            kth, e_kth, kept = -np.inf, 0.0, np.ones(V, bool)
        exp_imp = np.rint(pos * q)                         # numpy rounds half to even
        want = {int(t) for t in np.nonzero(kept & (exp_imp >= 1))[0]}
        got = {int(t): int(v) for t, v in got_json[b].items() if int(t) >= 0}
        for t in set(got) | want:
            half = abs(pos[t] * q - (np.floor(pos[t] * q) + 0.5)) <= q * e[t]
            if (t in got) != (t in want):
                tie = abs(pos[t] - kth) <= e[t] + e_kth
                cut = abs(pos[t] * q - 0.5) <= q * e[t]
                if not (tie or cut):
                    violations.append((b, t, got.get(t), int(exp_imp[t]) if t in want else None))
                    continue
                band += 1
            if t in got:
                d = abs(got[t] - int(exp_imp[t]))
                if d > (1 if half else 0):
                    violations.append((b, t, got[t], int(exp_imp[t])))
                elif d:
                    band += 1
        if not want and not got and got_json[b] != {"-1": 1}:
            violations.append((b, -1, got_json[b], {"-1": 1}))
    return violations, band
