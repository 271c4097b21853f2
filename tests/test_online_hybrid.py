"""Online hybrid search: query token counts on the device (lr_query_token_counts) and OnlineHybridSearcher, which runs
K1 -> K2 (dense ``emb``), token counts -> K4 (sparse ``tok``), one exchange for both systems, and lr_fuse_topk as one
CUDA-graph replay.  Every result is checked against the host parse (``parse_queries`` / ``oracle.query_counts``), the
composition of the existing public calls, and the oracle: dense by the tie rule against a float64 reference, sparse
exactly, fusion bit for bit."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import lightretriever_b200 as lr
from lightretriever_b200 import _C
from lightretriever_b200.sparse_search import QUERY_MAX_BAG, json_to_csr, parse_queries
from oracle import oracle

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BN = 256                                  # corpus tile (documents) of K2
N_C5, D_C5, K_C5, V_C5 = 1_100_000, 3584, 100, 128256


# ------------------------------------------------------------------------------------------------ C ABI (no GPU)
def test_query_token_counts_rejects_bad_arguments():
    lib = _C.load()
    assert QUERY_MAX_BAG == 8192
    buf = (ctypes.c_int64 * 4)()
    p = ctypes.addressof(buf)
    ok = dict(ids=p, offsets=p, n_ids=4, n_bags=1, V=10, max_bag=4, bow=0, q_indptr=p, q_tok=p, q_cnt=p, err_flag=None,
              scratch=p, scratch_bytes=1 << 20, stream=None)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.lr_query_token_counts(*a.values())

    for bad in (dict(ids=None), dict(offsets=None), dict(q_indptr=None), dict(q_tok=None), dict(q_cnt=None),
                dict(scratch=None), dict(n_bags=0), dict(n_bags=-1), dict(max_bag=QUERY_MAX_BAG + 1), dict(max_bag=-1),
                dict(V=0), dict(bow=2)):
        rc = call(**bad)
        assert rc == _C.LR_EINVAL, bad
        with pytest.raises(ValueError):
            _C.check(rc)
    assert "max_bag" in (call(max_bag=QUERY_MAX_BAG + 1), _C.last_error())[1]
    rc = call(scratch_bytes=16)
    assert rc == _C.LR_EWORKSPACE and "scratch" in _C.last_error()


def test_query_token_counts_scratch_sizing_needs_no_gpu():
    lib = _C.load()
    assert lib.lr_query_token_counts_scratch_bytes(0, 0) == 0
    a = lib.lr_query_token_counts_scratch_bytes(1000, 32)
    assert a >= 1000 * 8 + 32 * 4 and a % 256 == 0
    assert lib.lr_query_token_counts_scratch_bytes(0, 1) > 0
    assert lib.lr_query_token_counts_scratch_bytes(330_000, 10_000) > lib.lr_query_token_counts_scratch_bytes(1000, 32)


# ------------------------------------------------------------------------------------------------ token counts (GPU)
def _bags(lens, V, gen):
    """Ragged bags of ids in [-1, V] (so ids == -1 and == V occur); a list per bag + flat ids / offsets."""
    bags = [torch.randint(-1, V + 1, (int(n),), generator=gen).tolist() for n in lens]
    return bags


def _flat(bags):
    ids = torch.tensor([t for b in bags for t in b], dtype=torch.int64)
    offs = torch.tensor(np.cumsum([0] + [len(b) for b in bags[:-1]]), dtype=torch.int64)
    return ids.cuda(), offs.cuda()


def _csr_rows(qi, qt, qc):
    qi, qt, qc = qi.cpu().tolist(), qt.cpu().tolist(), qc.cpu().tolist()
    return [(qt[qi[r]:qi[r + 1]], qc[qi[r]:qi[r + 1]]) for r in range(len(qi) - 1)]


def _check_counts(bags, V, kind, got):
    qi, qt, qc = got
    rows = _csr_rows(qi, qt, qc)
    assert len(rows) == len(bags)
    hi, ht, hc = parse_queries([[t for t in b if 0 <= t < V] for b in bags], V)
    host = _csr_rows(torch.from_numpy(hi), torch.from_numpy(ht), torch.from_numpy(hc))
    for r, (b, (toks, cnts), (htoks, hcnts)) in enumerate(zip(bags, rows, host)):
        exp = oracle.query_counts([t for t in b if 0 <= t < V], kind)
        assert dict(zip(toks, cnts)) == exp, r
        assert toks == sorted(exp) and all(c >= 1 for c in cnts), r                  # ascending, no zero entries
        if kind == "sum":
            assert dict(zip(htoks, hcnts)) == exp, r                                  # the host parse agrees
    n = int(qi[-1])
    assert (qt[n:] == 0).all() and (qc[n:] == 0).all()                                # deterministic tail


@gpu
@pytest.mark.parametrize("kind", ["sum", "bow"])
@pytest.mark.parametrize("Q", [1, 32, 10_000])
def test_query_token_counts_match_host_parse(Q, kind):
    """Ragged bags (0..40 ids) with empty first / last bags, bags of out-of-range ids only, ids equal to V and -1."""
    V = 300 if Q > 1 else 5000
    gen = torch.Generator().manual_seed(Q)
    lens = torch.randint(0, 41, (Q,), generator=gen)
    if Q > 1:
        lens[0] = lens[-1] = 0
    bags = _bags(lens, V, gen)
    if Q >= 32:
        bags[3] = [-1, V, V + 7, -5, V]            # nothing in range
        bags[4] = [7] * 5 + [V] + [7]
    ids, offs = _flat(bags)
    _check_counts(bags, V, kind, lr.query_token_counts(ids, offs, V, kind=kind))


@gpu
@pytest.mark.parametrize("kind", ["sum", "bow"])
def test_query_token_counts_at_max_bag(kind):
    """One bag of max_bag copies of one token, one of max_bag distinct tokens (reversed), between short bags."""
    V, M = 20_000, QUERY_MAX_BAG
    bags = [[3, 3, 9], [17] * M, list(range(M + 100, 100, -1))[:M], [], [V - 1, -1, V - 1]]
    ids, offs = _flat(bags)
    _check_counts(bags, V, kind, lr.query_token_counts(ids, offs, V, kind=kind, max_bag=M))
    # a bag beyond the bound is flagged and left empty
    with pytest.raises(ValueError, match="max_bag"):
        lr.query_token_counts(ids, offs, V, kind=kind, max_bag=M - 1)
    qi, _, _ = lr.query_token_counts(ids, offs, V, kind=kind, max_bag=M - 1, check=False)
    qi = qi.cpu().tolist()
    assert qi[2] - qi[1] == 0 and qi[3] - qi[2] == 0 and qi[1] == 2


@gpu
def test_query_token_counts_under_graph_capture():
    """Captured once, replayed over new ids written into the same buffers: every replay equals the eager call."""
    V, B, T = 1000, 16, 256
    ids = torch.full((T,), -1, dtype=torch.int64, device="cuda")
    offs = torch.zeros(B, dtype=torch.int64, device="cuda")
    out = tuple(torch.empty(n, dtype=torch.int32, device="cuda") for n in (B + 1, T, T))
    ws = lr._util.Workspace()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        lr.query_token_counts(ids, offs, V, out=out, check=False, workspace=ws)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        lr.query_token_counts(ids, offs, V, out=out, check=False, workspace=ws)
    gen = torch.Generator().manual_seed(9)
    for rep in range(3):
        lens = torch.randint(0, 17, (B,), generator=gen)
        bags = _bags(lens, V, gen)
        fi, fo = _flat(bags)
        ids.fill_(-1)
        ids[:fi.numel()].copy_(fi)
        offs.copy_(fo)
        g.replay()
        got = tuple(t.clone() for t in out)
        exp = lr.query_token_counts(ids, offs, V)
        assert all(torch.equal(a, b) for a, b in zip(got, exp)), rep
        _check_counts(bags, V, "sum", got)


# ------------------------------------------------------------------------------------------------ merge of a strided view
@gpu
def test_topk_merge_takes_the_two_system_view():
    """[L, 2, Q, cap] keys: each half merged in place (q_stride = 2Q) equals the merge of a contiguous copy."""
    gen = torch.Generator(device="cuda").manual_seed(4)
    L, Q, cap, k = 3, 5, 40, 25
    s = torch.randn(L, 2, Q, cap, device="cuda", generator=gen).abs()
    s[:, 1] = torch.randint(1, 50, (L, Q, cap), device="cuda", generator=gen).float()   # integer sparse scores
    i = torch.randperm(L * 2 * Q * cap, device="cuda", generator=gen).view(L, 2, Q, cap) % 997
    keys = torch.empty_like(i)
    for l in range(L):
        keys[l, 0] = lr.merge_keys([lr.encode_keys(s[l, 0], i[l, 0])], cap)     # sorted float-score keys (dense)
        keys[l, 1] = _u32_keys(s[l, 1], i[l, 1])                                 # sorted integer-score keys (sparse)
    for h, kind in ((0, _C.LR_SCORE_F32), (1, _C.LR_SCORE_U32)):
        view = keys[:, h]
        assert not view.is_contiguous()
        a = lr.topk_merge(view, k, score_kind=kind, return_keys=True)
        b = lr.topk_merge(view.contiguous(), k, score_kind=kind, return_keys=True)
        assert all(torch.equal(x, y) for x, y in zip(a, b)), h
    with pytest.raises(ValueError):
        lr.topk_merge(keys[:, :, 0], k)                    # lists not spaced by whole query rows


def _u32_keys(scores, ids):
    """Sorted integer-score keys (score << 32 | ~id), the form K4 exchanges."""
    key = (scores.long() << 32) | (0xFFFFFFFF - ids)
    return torch.sort(key, dim=1, descending=True).values


# ------------------------------------------------------------------------------------------------ searcher helpers
def _np(t):
    return t.detach().cpu().numpy()


def _scores64(q, c, chunk=1 << 17):
    q64 = q.double()
    out = torch.empty((q.shape[0], c.shape[0]), dtype=torch.float64, device=q.device)
    for lo in range(0, c.shape[0], chunk):
        out[:, lo:lo + chunk] = q64 @ c[lo:lo + chunk].double().T
    return out


def _check_parity(s, i, ref, k, rtol=1e-2, id_offset=0):
    """oracle.check_topk_parity over the columns that decide it (the reference top-k and the returned ids)."""
    kk = min(k, ref.shape[1])
    top = torch.topk(ref, kk, dim=1).indices.cpu().numpy()
    s, i = _np(s), _np(i)
    for r in range(ref.shape[0]):
        got = i[r] - id_offset
        cols = np.union1d(top[r], got[i[r] >= 0])
        row = ref[r, torch.from_numpy(cols).to(ref.device)].cpu().numpy()[None]
        loc = np.where(i[r] >= 0, np.searchsorted(cols, got), -1)
        try:
            oracle.check_topk_parity(s[r:r + 1], loc[None], row, k, rtol=rtol)
        except AssertionError as e:
            raise AssertionError(f"query {r}: {e}") from None


def _check_fused(dense, sparse, fused, method, weights):
    """lr_fuse_topk output == oracle fusion of the returned per-system lists, bit for bit.  A system without a hit for
    a query is absent from that query's results (as Anserini writes no line); rrf ranks are the list positions."""
    (ds, di), (ss, si) = (tuple(map(_np, dense)), tuple(map(_np, sparse)))
    fi, fs, fc = map(_np, fused)
    for q in range(di.shape[0]):
        systems = []
        for s_, i_ in ((ds[q], di[q]), (ss[q], si[q])):
            keep = i_ >= 0
            if method == "linear":
                systems.append({"q": {str(a): float(b) for a, b in zip(i_[keep], s_[keep])}} if keep.any() else {})
            else:  # rank = position in the returned list (ties by ascending id); numpy's argsort leaves ties unordered
                systems.append({"q": {str(a): -float(r) for r, a in enumerate(i_[keep])}} if keep.any() else {})
        ref = (oracle.fuse_linear(systems, weights=list(weights)) if method == "linear"
               else oracle.fuse_rrf(systems)).get("q", {})
        n = int(fc[q])
        assert n == len(ref), q
        got = {str(a): b for a, b in zip(fi[q, :n], fs[q, :n])}
        assert got.keys() == ref.keys(), q
        for pid, v in ref.items():
            assert got[pid] == v, (q, pid, got[pid], v)
        assert (fi[q, n:] == -1).all()


def _compose(srv, ids, offs, tids, toffs, kind, method, weights):
    """The same request through the existing public calls: bag.encode -> flatip_topk; host parse_queries ->
    ImpactIndex.search_device; fuse_topk_device."""
    qv = srv.bag.encode(ids, offs, shrink_dim=srv.shrink_dim, normalize=True)
    dense = lr.flatip_topk(qv, srv.corpus, srv.k, id_offset=srv.id_offset)
    bags = _split(tids, toffs)
    V = srv.sparse_index.V
    qs = [[t for t in b if 0 <= t < V] for b in bags]
    qs = qs if kind == "sum" else [sorted(set(b)) for b in qs]
    sparse = srv.sparse_index.search_device(*parse_queries(qs, V), srv.k)
    fused = lr.fuse_topk_device(*dense, *sparse, method=method, weights=weights)
    return qv, dense, sparse, fused, bags


def _split(ids, offs):
    ids, offs = ids.cpu().tolist(), offs.cpu().tolist()
    return [ids[a:b] for a, b in zip(offs, offs[1:] + [len(ids)])]


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def _serve_and_check(srv, reqs, kind, method, weights, sparse_ref):
    """Each request through the captured graph, then: replay == eager _step (same staged buffers), == the composition of
    public calls; dense by the tie rule, sparse exactly against ``sparse_ref(bags)``, fusion against the oracle."""
    for ids, offs, tids, toffs in reqs:
        n = offs.numel()
        got = srv.search(ids, offs, tids, toffs)
        got = tuple(tuple(t.clone() for t in part) for part in got)
        eager = srv._step()
        for g_part, e_part in zip(got, eager):
            assert _same(g_part, (t[:n] for t in e_part)), "graph replay differs from the eager step"
        qv, dense, sparse, fused, bags = _compose(srv, ids, offs, ids if tids is None else tids,
                                                  offs if toffs is None else toffs, kind, method, weights)
        assert _same(got[0], dense) and _same(got[1], sparse) and _same(got[2], fused)
        _check_parity(*got[0], _scores64(qv, srv.corpus), srv.k, id_offset=srv.id_offset)
        es, ei = sparse_ref([[t for t in b if 0 <= t < srv.sparse_index.V] for b in bags])
        assert (_np(got[1][1]) == ei).all() and (_np(got[1][0]) == es).all()
        _check_fused(got[0], got[1], got[2], method, weights)


# ------------------------------------------------------------------------------------------------ searcher, small shape
N_S, D_S, V_S, K_S, B_S = 50_000, 256, 5000, 100, 8


@pytest.fixture(scope="module")
def small():
    gen = torch.Generator(device="cuda").manual_seed(21)
    table = (torch.randn(V_S, D_S, device="cuda", generator=gen) * 0.02).bfloat16()
    corpus = F.normalize(torch.randn(N_S, D_S, device="cuda", generator=gen), dim=-1).bfloat16()
    rng = np.random.default_rng(22)
    steps = rng.integers(1, 300, (N_S, 16)).cumsum(1)                 # distinct tokens per document (< 16 * 300 < V)
    tok = (rng.integers(0, V_S, (N_S, 1)) + steps) % V_S
    imp = rng.integers(1, 400, (N_S, 16))
    docs = [dict(zip(t.tolist(), m.tolist())) for t, m in zip(tok, imp)]
    index = lr.ImpactIndex(V_S, id_offset=7)
    index.add_csr(*json_to_csr(docs))
    data = {"table": table, "corpus": corpus, "docs": docs, "index": index}
    yield data
    data.clear()
    torch.cuda.empty_cache()


def _requests(V, gen, shared, sizes=(8, 1, 5)):
    """Requests of ``sizes`` queries; a request of 6 or more holds an empty bag and a query whose sparse ids are all out of
    range (separate ids) or whose bag ids are all padding_idx (shared ids)."""
    reqs = []
    for n in sizes:
        special = n >= 6
        lens = torch.randint(1, 33, (n,), generator=gen)
        if special:
            lens[2] = 0
        ids = torch.randint(0, V - 1, (int(lens.sum()),), generator=gen)
        offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
        tids = toffs = None
        if not shared:
            tl = torch.randint(1, 20, (n,), generator=gen)
            tids = torch.randint(0, V, (int(tl.sum()),), generator=gen)
            toffs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), tl[:-1]]), 0)
            if special:
                tids[toffs[5]:toffs[5] + tl[5]] = V + 3                          # no valid sparse token
            tids, toffs = tids.cuda(), toffs.cuda()
        elif special:
            ids[offs[5]:offs[5] + lens[5]] = V - 1                               # the bag's padding_idx ... only
        reqs.append((ids.cuda(), offs.cuda(), tids, toffs))
    return reqs


@gpu
@pytest.mark.parametrize("method,kind,shared", [("linear", "sum", True), ("rrf", "bow", False),
                                                ("linear", "bow", False), ("rrf", "sum", True)])
def test_online_hybrid_small_shape(small, method, kind, shared):
    """50k x 256, V = 5000, k = 100, batch 8; requests of 8, 1, 5 queries through one captured graph."""
    bag = lr.B200EmbeddingBag.from_pretrained(small["table"], padding_idx=V_S - 1)
    index = small["index"]
    weights = (0.6, 0.4)
    srv = lr.OnlineHybridSearcher(bag, small["corpus"], index, K_S, batch=B_S, max_tokens=B_S * 32, id_offset=7,
                                  method=method, weights=weights, token_kind=kind)
    docs = small["docs"]

    def sparse_ref(qs):
        return oracle.impact_topk([oracle.query_counts(q, kind) for q in qs], docs, K_S, id_offset=7)

    gen = torch.Generator().manual_seed(sum(map(ord, method + kind)) + shared)
    _serve_and_check(srv, _requests(V_S, gen, shared), kind, method, weights, sparse_ref)


@gpu
def test_online_hybrid_rejects_mismatched_systems(small):
    bag = lr.B200EmbeddingBag.from_pretrained(small["table"], padding_idx=V_S - 1)
    index = small["index"]
    with pytest.raises(ValueError, match="1024"):
        lr.OnlineHybridSearcher(bag, small["corpus"], index, 1025, 1, 8, id_offset=7, use_graph=False)
    with pytest.raises(ValueError, match="same documents"):
        lr.OnlineHybridSearcher(bag, small["corpus"], index, 10, 1, 8, id_offset=0, use_graph=False)
    with pytest.raises(ValueError, match="same documents"):
        lr.OnlineHybridSearcher(bag, small["corpus"][:-1], index, 10, 1, 8, id_offset=7, use_graph=False)
    srv = lr.OnlineHybridSearcher(bag, small["corpus"], index, 10, 2, 8, id_offset=7, use_graph=False)
    ids = torch.arange(4, device="cuda")
    with pytest.raises(ValueError):
        srv.search(ids, torch.tensor([0, 2], device="cuda"), ids, torch.tensor([0], device="cuda"))
    with pytest.raises(ValueError):
        srv.search(torch.arange(9, device="cuda"), torch.tensor([0], device="cuda"))


# ------------------------------------------------------------------------------------------------ searcher, C5 shape
def _flatip_plan(Q, N, k, d):
    lib = _C.load()
    out, rows, flags = (ctypes.c_int64 * 16)(), (ctypes.c_int64 * 64)(), (ctypes.c_int64 * 2)()
    assert lib.lr_flatip_plan(Q, N, k, out) == 0
    n = lib.lr_flatip_plan_passes_sharded(Q, N, k, d, 1, rows, 16, flags)
    names = ["cl", "pair", "m_tiles", "n_tiles", "cap", "prefix_tiles", "prefix_splits", "prefix_units", "main_begin",
             "main_splits", "main_units", "grid", "band", "ws", "rounds", "n_clusters"]
    return dict(zip(names, list(out))), [tuple(rows[4 * i:4 * i + 4]) for i in range(n)]


def _assert_small_batch_warm_start(Q, N, k, d):
    """One tile per CTA in the prefix (148 splits), lists raised to BN + 64, then the main pass over the rest."""
    p, passes = _flatip_plan(Q, N, k, d)
    assert (p["cl"], p["pair"]) == (1, 0), p
    assert p["cap"] >= BN + 64, p
    assert len(passes) == 2 and passes[0][:3] == (0, 148, 148), passes
    assert passes[1][0] == 148 and passes[1][1] == -(-N // BN) and passes[1][2] >= 100, passes


def test_c5_shapes_select_their_plans():
    _assert_small_batch_warm_start(32, N_C5, K_C5, D_C5)
    assert _flatip_plan(1, N_C5, K_C5, D_C5)[1][0][:2] == (0, -(-N_C5 // BN))   # batch 1: single phase


@gpu
def test_online_hybrid_c5_shape():
    """1.1M x 3584 bf16 corpus, V = 128256 table, 1.1M x 64 Zipf sparse index, k = 100, batch 32 and batch 1.  Sparse
    results are checked against a float64 CSR product on the device (exact for integer scores)."""
    test_c5_shapes_select_their_plans()
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(77)
    table = (torch.randn(V_C5, D_C5, device=dev, generator=gen) * 0.02).bfloat16()
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V_C5 - 1)
    corpus = torch.empty((N_C5, D_C5), dtype=torch.bfloat16, device=dev)
    for lo in range(0, N_C5, 1 << 17):
        corpus[lo:lo + (1 << 17)] = F.normalize(torch.randn(min(1 << 17, N_C5 - lo), D_C5, device=dev, generator=gen),
                                                dim=-1).bfloat16()
    w = 1.0 / torch.arange(1, V_C5 + 1, dtype=torch.float64, device=dev)
    cdf = torch.cumsum(w / w.sum(), 0)
    perm = torch.randperm(V_C5, generator=gen, device=dev)
    tok = perm[torch.searchsorted(cdf, torch.rand(N_C5 * 64, generator=gen, device=dev, dtype=torch.float64))
               .clamp_max(V_C5 - 1)].to(torch.int32).view(N_C5, 64)
    imp = torch.randint(1, 401, (N_C5, 64), generator=gen, device=dev, dtype=torch.int32)
    index = lr.ImpactIndex(V_C5, id_offset=3)
    for lo in range(0, N_C5, 1 << 18):
        index.add_dense_rows(tok[lo:lo + (1 << 18)], imp[lo:lo + (1 << 18)])
    # reference documents: float64 CSR [N, V], a token repeated in a row keeps its first impact (add_dense_rows' rule)
    key = torch.arange(N_C5, device=dev, dtype=torch.int64)[:, None] * V_C5 + tok.long()
    uk, inv = torch.unique(key.view(-1), return_inverse=True)
    first = torch.full((uk.numel(),), N_C5 * 64, dtype=torch.int64, device=dev)
    first.scatter_reduce_(0, inv, torch.arange(N_C5 * 64, device=dev), "amin")
    crow = torch.zeros(N_C5 + 1, dtype=torch.int64, device=dev)
    crow[1:] = torch.cumsum(torch.bincount(uk // V_C5, minlength=N_C5), 0)
    D = torch.sparse_csr_tensor(crow, uk % V_C5, imp.view(-1)[first].double(), size=(N_C5, V_C5))
    del tok, imp, key, uk, inv, first

    def sparse_ref(qs):
        cnt = torch.zeros((V_C5, len(qs)), dtype=torch.float64, device=dev)
        for r, q in enumerate(qs):
            for t, c in oracle.query_counts(q, "sum").items():
                cnt[t, r] = c
        S = (D @ cnt).T                                                          # [Q, N] exact integers
        s, order = torch.sort(S, dim=1, descending=True, stable=True)           # ties: ascending id
        s, order = s[:, :K_C5], order[:, :K_C5]
        hit = s > 0
        return (_np(torch.where(hit, s, -torch.inf).float()), _np(torch.where(hit, order + 3, -1)))

    gen_h = torch.Generator().manual_seed(78)
    for batch, sizes in ((32, (32, 1, 17)), (1, (1,))):
        srv = lr.OnlineHybridSearcher(bag, corpus, index, K_C5, batch=batch, max_tokens=batch * 32, id_offset=3)
        _serve_and_check(srv, _requests(V_C5, gen_h, True, sizes), "sum", "linear", (0.7, 0.3), sparse_ref)
        del srv
    del table, bag, corpus, index, D
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ two GPUs
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one box")
def test_online_hybrid_over_nccl():
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "nccl_hybrid_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and f"nccl hybrid worker OK world={world}" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
