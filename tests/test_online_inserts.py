"""Live document inserts in the online searchers: the forward-segment kernel (lr_sparse_fwd_score_topk) against K4 over an
inverted index of the same documents, bit for bit; ImpactDelta; and OnlineSearcher / OnlineHybridSearcher with a delta
segment against a searcher freshly built over main + export_inserts() with the same deletions and filters, bit for bit,
through one captured graph that is never recaptured."""
import ctypes
import os
import socket
import subprocess
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

import lightretriever_b200 as lr
from lightretriever_b200 import _C
from lightretriever_b200.filters import doc_bitmap
from lightretriever_b200.sparse_search import ImpactDelta

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V_BIG = 128256


# ------------------------------------------------------------------------------------------------ C ABI (no GPU)
def test_sparse_fwd_rejects_bad_arguments():
    lib = _C.load()
    buf = (ctypes.c_int64 * 64)()
    p = ctypes.addressof(buf)
    ok = dict(q_indptr=p, q_tok=p, q_cnt=p, Q=1, doc_ptr=p, n_docs=p, doc_tok=p, doc_imp=p, cap_docs=10, V=10,
              id_offset=0, k=5, out_scores=p, out_ids=p, out_keys=None, live=None, allow=None, ld_words=0, n_filters=0,
              q_filter=None, workspace=p, ws_bytes=1 << 30, stream=None)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.lr_sparse_fwd_score_topk(*a.values())

    cases = [(dict(q_indptr=None), "null"), (dict(q_tok=None), "null"), (dict(q_cnt=None), "null"),
             (dict(doc_ptr=None), "null"), (dict(n_docs=None), "null"), (dict(doc_tok=None), "null"),
             (dict(doc_imp=None), "null"), (dict(k=0), "k"), (dict(k=1025), "k"), (dict(cap_docs=-1), "cap_docs"),
             (dict(live=p, ld_words=0), "ld_words"), (dict(live=p, id_offset=100, ld_words=3), "ld_words"),
             (dict(out_scores=None, out_ids=None), "output"), (dict(Q=0), "Q")]
    for bad, word in cases:
        rc = call(**bad)
        assert rc == _C.LR_EINVAL, bad
        assert word in _C.last_error(), (bad, _C.last_error())
        with pytest.raises(ValueError):
            _C.check(rc)
    rc = call(ws_bytes=16)
    assert rc == _C.LR_EWORKSPACE and "workspace" in _C.last_error()


def test_sparse_fwd_workspace_sizing_needs_no_gpu():
    lib = _C.load()
    f = lib.lr_sparse_fwd_workspace_bytes
    assert f(0, 10, 5) == 0 and f(1, -1, 5) == 0 and f(1, 10, 0) == 0 and f(1, 10, 1025) == 0
    sizes = [f(1, 0, 1), f(32, 16384, 100), f(10_000, 3000, 1024)]
    assert all(s > 0 and s % 256 == 0 for s in sizes)
    assert f(1000, 16384, 100) > f(32, 16384, 100)        # grows with Q
    assert f(32, 16384, 100) > f(32, 1000, 100)           # ... with the capacity
    assert f(32, 16384, 1000) > f(32, 16384, 100)         # ... and with k
    assert f(10_000, 16384, 1024) < (1 << 28)             # query chunks bound it


def _stub_bag():
    return types.SimpleNamespace(padding_idx=0)


def test_insert_arguments_are_checked_without_a_gpu():
    corpus = torch.zeros((100, 16), dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="insert_capacity"):
        lr.OnlineSearcher(_stub_bag(), corpus, 10, 1, 8, insert_capacity=-1)
    with pytest.raises(ValueError, match="filters must cover"):      # 100 + 64 ids need 6 words
        lr.OnlineSearcher(_stub_bag(), corpus, 10, 1, 8, insert_capacity=64, filters=torch.zeros((2, 4), dtype=torch.int32))
    with pytest.raises(ValueError, match="overlap"):
        lr.OnlineSearcher(_stub_bag(), corpus, 10, 1, 8, insert_capacity=64, insert_id_base=50)
    with pytest.raises(ValueError, match="2\\^32"):
        lr.OnlineSearcher(_stub_bag(), corpus, 10, 1, 8, insert_capacity=64, insert_id_base=(1 << 32) - 10)
    index = lr.ImpactIndex(50, device="cpu")
    index.add_csr(np.arange(101), np.zeros(100, dtype=np.int32), np.ones(100, dtype=np.int64))
    with pytest.raises(ValueError, match="insert_postings_capacity"):
        lr.OnlineHybridSearcher(_stub_bag(), corpus, index, 10, 1, 8, insert_capacity=8, insert_postings_capacity=-1)
    with pytest.raises(ValueError, match="insert_capacity"):
        lr.OnlineHybridSearcher(_stub_bag(), corpus, index, 10, 1, 8, insert_capacity=-5)
    with pytest.raises(ValueError, match="cap_docs"):
        ImpactDelta(50, -1, 10, device="cpu")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import lightretriever_b200 as lr_
        corpus = torch.zeros((100, 16), dtype=torch.bfloat16)
        try:
            lr_.OnlineSearcher(_stub_bag(), corpus, 10, 1, 8, id_offset=100 * rank, insert_capacity=64)
        except ValueError as e:
            assert "insert_id_base" in str(e)
            open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_insert_id_base_is_required_when_sharded(tmp_path):
    world = 2
    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


# ------------------------------------------------------------------------------------------------ kernel parity (GPU)
CAP, ID0 = 3000, 1000


def _tokens(kind, n, gen):
    if kind == "uniform":
        return torch.randint(0, V_BIG, (n,), generator=gen)
    w = 1.0 / torch.arange(1, V_BIG + 1, dtype=torch.float64)
    return torch.multinomial(w, n, replacement=True, generator=gen)   # Zipf(1.0): rank r has weight 1 / r


def _documents(kind, seed):
    """CAP documents as CSR (int64 indptr, int32 tok, int64 imp): ragged lengths 0..80 of distinct tokens, plus zero impacts, empty documents, exact duplicates (ties) and impacts whose sums exceed 2^16."""
    gen = torch.Generator().manual_seed(seed)
    lens = torch.randint(0, 81, (CAP,), generator=gen)
    tok = _tokens(kind, int(lens.sum()), gen).to(torch.int32)
    imp = torch.randint(1, 401, (tok.numel(),), generator=gen)
    indptr = torch.zeros(CAP + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(lens, 0)
    docs = []
    for d in range(CAP):  # one posting per (document, token): K4's row kernel takes a document once per posting run
        first = dict(zip(reversed(tok[indptr[d]:indptr[d + 1]].tolist()), reversed(imp[indptr[d]:indptr[d + 1]].tolist())))
        docs.append((list(first), list(first.values())))
    hot = _tokens(kind, 8, gen).tolist()
    docs[0] = (hot[:3], [65535, 65535, 9])                               # sums > 2^16
    docs[1] = ([], [])
    docs[2] = (hot[:4], [0, 0, 0, 0])                                    # zero impacts only: score 0
    docs[3] = (hot[:4], [0, 7, 0, 1])
    for d in (5, 17, CAP // 2, CAP - 1):
        docs[d] = docs[4]                                                # exact ties across the fill levels
    docs[6] = (hot, [65535] * 8)
    lens = torch.tensor([len(t) for t, _ in docs])
    indptr = torch.zeros(CAP + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(lens, 0)
    tok = torch.tensor([t for d in docs for t in d[0]], dtype=torch.int32)
    imp = torch.tensor([m for d in docs for m in d[1]], dtype=torch.int64)
    return indptr, tok, imp, hot


def _queries(kind, Q, hot, seed):
    """Bags of 1..40 ids (repeats give counts > 1), a few over the hot tokens, as lr_query_token_counts' CSR."""
    gen = torch.Generator().manual_seed(seed)
    lens = torch.randint(1, 41, (Q,), generator=gen)
    ids = _tokens(kind, int(lens.sum()), gen)
    offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
    for q in range(min(Q, 4)):
        ids[offs[q]:offs[q] + 3] = torch.tensor(hot[q:q + 1] * 2 + hot[1:2])
    return lr.query_token_counts(ids.cuda(), offs.cuda(), V_BIG)


@pytest.fixture(scope="module")
def corpora():
    data = {}
    for kind in ("zipf", "uniform"):
        indptr, tok, imp, hot = _documents(kind, 5 if kind == "zipf" else 6)
        delta = ImpactDelta(V_BIG, CAP, tok.numel(), id_offset=ID0)
        ids = [delta.append_csr(indptr[:1001], tok[:int(indptr[1000])], imp[:int(indptr[1000])])]
        ids.append(delta.append_csr(indptr[1000:] - indptr[1000], tok[int(indptr[1000]):], imp[int(indptr[1000]):]))
        assert torch.equal(torch.cat(ids), torch.arange(ID0, ID0 + CAP))
        data[kind] = dict(csr=(indptr, tok, imp), hot=hot, delta=delta, k4={})
    yield data
    data.clear()
    torch.cuda.empty_cache()


def _k4(data, n):
    """K4 index over the first n documents (None when n == 0: K4 needs a document)."""
    if n not in data["k4"]:
        indptr, tok, imp = data["csr"]
        idx = None
        if n:
            idx = lr.ImpactIndex(V_BIG, id_offset=ID0)
            idx.add_csr(indptr[:n + 1], tok[:int(indptr[n])], imp[:int(indptr[n])])
            idx.build()
        data["k4"][n] = idx
    return data["k4"][n]


def _fwd_vs_k4(data, q_csr, k, n, **flt):
    delta = data["delta"]
    delta.n_docs.fill_(n)                                  # the documents past n stay in the buffers: must not be read
    got = delta.search_device(*q_csr, k, return_keys=True, **flt)
    idx = _k4(data, n)
    if idx is None:
        assert (got[1] == -1).all() and torch.isinf(got[0]).all() and (got[2] == 0).all()
        return
    exp = idx.search_device(*q_csr, k, return_keys=True, **flt)
    for name, a, b in zip(("scores", "ids", "keys"), got, exp):
        assert torch.equal(a, b), (name, n, k)
    delta.n_docs.fill_(delta.N)


@gpu
@pytest.mark.parametrize("kind", ["zipf", "uniform"])
@pytest.mark.parametrize("Q", [1, 32, 10_000])
@pytest.mark.parametrize("k", [1, 100, 1000, 1024])
def test_fwd_kernel_matches_k4(corpora, kind, Q, k):
    """Scores, ids and keys bit-identical to K4 over an inverted index of the same documents, for n_docs 0, 1, partial,
    cap; V = 128256."""
    data = corpora[kind]
    q_csr = _queries(kind, Q, data["hot"], Q + k)
    for n in (0, 1, 1234, CAP):
        _fwd_vs_k4(data, q_csr, k, n)


@gpu
@pytest.mark.parametrize("Q", [32, 10_000])
def test_fwd_kernel_filters_match_k4(corpora, Q):
    """Deletions (live), allow rows chosen by q_filter, q_filter -1 (unrestricted) and out of range (nothing)."""
    data = corpora["zipf"]
    q_csr = _queries("zipf", Q, data["hot"], 7 + Q)
    gen = torch.Generator(device="cuda").manual_seed(Q)
    words = (ID0 + CAP + 31) // 32
    ids = torch.arange(ID0, ID0 + CAP, device="cuda")
    live = doc_bitmap(ID0 + CAP, ids[torch.rand(CAP, device="cuda", generator=gen) < 0.8], device="cuda")
    allow = torch.stack([doc_bitmap(ID0 + CAP, ids[torch.rand(CAP, device="cuda", generator=gen) < p], device="cuda")
                         for p in (0.5, 0.05)])
    assert allow.shape == (2, words)
    qf = torch.randint(-1, 2, (Q,), device="cuda", generator=gen, dtype=torch.int32)
    qf[0], qf[-1] = 7, -3                                                    # out of range: allows nothing
    for n in (1234, CAP):
        _fwd_vs_k4(data, q_csr, 100, n, live=live)
        _fwd_vs_k4(data, q_csr, 100, n, allow=allow, q_filter=qf)
        _fwd_vs_k4(data, q_csr, 100, n, live=live, allow=allow, q_filter=qf)
        got = data["delta"].search_device(*q_csr, 100, live=live, allow=allow, q_filter=qf)
        assert (got[1][0] == -1).all() and (got[1][-1] == -1).all()


@gpu
def test_fwd_kernel_counts_repeated_tokens():
    """A token repeated in a document counts every time (40 x 65535 per query count here), against exact integers."""
    delta = ImpactDelta(V_BIG, 8, 1000, id_offset=ID0)
    docs = [([5] * 40 + [9], [65535] * 40 + [1]), ([5, 9, 9], [3, 2, 2]), ([9] * 3, [1, 1, 1]), ([], [])]
    delta.append_csr(np.cumsum([0] + [len(t) for t, _ in docs]), [t for d in docs for t in d[0]],
                     [m for d in docs for m in d[1]])
    ids = torch.tensor([5, 5, 9, 7], device="cuda")
    q_csr = lr.query_token_counts(ids, torch.tensor([0], device="cuda"), V_BIG)   # counts {5: 2, 7: 1, 9: 1}
    s, i = delta.search_device(*q_csr, 5)
    exp = [(2 * 40 * 65535 + 1, 0), (2 * 3 + 4, 1), (3, 2)]
    assert i[0].tolist() == [ID0 + d for _, d in exp] + [-1, -1]
    assert s[0, :3].tolist() == [float(v) for v, _ in exp]


@gpu
def test_impact_delta_append_rules(corpora):
    delta = ImpactDelta(V_BIG, 4, 10, id_offset=5)
    with pytest.raises(ValueError, match="out of range"):
        delta.append_csr([0, 1], [V_BIG], [1])
    with pytest.raises(ValueError, match="uint16"):
        delta.append_csr([0, 1], [3], [70000])
    with pytest.raises(ValueError, match="disagree"):
        delta.append_csr([0, 2], [3], [1])
    with pytest.raises(ValueError, match="full"):
        delta.append_csr([0, 11], list(range(11)), [1] * 11)
    assert delta.N == 0 and int(delta.n_docs) == 0
    assert delta.append_csr([0, 2, 2], [3, 3], [1, 2]).tolist() == [5, 6]
    with pytest.raises(ValueError, match="full"):
        delta.append_csr([0, 0, 0, 0], [], [])
    assert int(delta.n_docs) == 2
    ip, tk, im = delta.export_csr()
    assert ip.tolist() == [0, 2, 2] and tk.tolist() == [3, 3] and im.tolist() == [1, 2]


# ------------------------------------------------------------------------------------------------ searchers (GPU)
def _same(a, b):
    if isinstance(a, torch.Tensor):
        return torch.equal(a, b)
    return all(_same(x, y) for x, y in zip(a, b))


def _clone(r):
    return r.clone() if isinstance(r, torch.Tensor) else tuple(_clone(x) for x in r)


def _make_data(N, d, V, L, seed, dev="cuda"):
    gen = torch.Generator(device=dev).manual_seed(seed)
    table = (torch.randn(V, d, device=dev, generator=gen) * 0.02).bfloat16()
    corpus = torch.empty((N, d), dtype=torch.bfloat16, device=dev)
    for lo in range(0, N, 1 << 17):
        corpus[lo:lo + (1 << 17)] = F.normalize(torch.randn(min(1 << 17, N - lo), d, device=dev, generator=gen),
                                                dim=-1).bfloat16()
    tok = torch.randint(0, V, (N, L), device=dev, generator=gen, dtype=torch.int32)
    imp = torch.randint(1, 401, (N, L), device=dev, generator=gen, dtype=torch.int32)
    return table, corpus, tok, imp


def _rows_csr(tok, imp):
    n, L = tok.shape
    return torch.arange(0, n * L + 1, L, dtype=torch.int64), tok.reshape(-1), imp.reshape(-1)


def _requests(V, pad, batch, gen, sizes):
    reqs = []
    for n in sizes:
        lens = torch.randint(1, 33, (n,), generator=gen)
        ids = torch.randint(0, V, (int(lens.sum()),), generator=gen)
        ids[ids == pad] = 0
        offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
        reqs.append((ids.cuda(), offs.cuda()))
    return reqs


def _insert_batches(srv, bag, corpus, tok, imp, reqs, hybrid, gen):
    """Three batches: documents built to outrank the main shard (the query vectors themselves; the queries' tokens with
    impacts of 60000), exact duplicates of main rows (ties), and random documents.  Returns the ids per batch."""
    ids_, offs_ = reqs[0]
    qv = bag.encode(ids_, offs_, normalize=True)
    L = tok.shape[1]
    bags = torch.tensor_split(ids_.cpu(), offs_.cpu()[1:])
    q_tok = torch.stack([b.repeat(L)[:L] for b in bags]).to(torch.int32).cuda()
    n_rand = 700
    batches = [(qv, q_tok, torch.full_like(q_tok, 60000)),
               (corpus[:50].clone(), tok[:50], imp[:50]),
               (F.normalize(torch.randn(n_rand, corpus.shape[1], device="cuda", generator=gen), dim=-1).bfloat16(),
                tok[torch.randint(0, tok.shape[0], (n_rand,), device="cuda", generator=gen)],
                torch.randint(1, 401, (n_rand, L), device="cuda", generator=gen, dtype=torch.int32))]
    return [srv.insert(rows, *_rows_csr(t, m)) if hybrid else srv.insert(rows) for rows, t, m in batches]


def _rebuilt(kw, srv, bag, corpus, tok, imp, hybrid, id_offset, V, filters):
    """A searcher freshly built over main + export_inserts(), without a delta segment."""
    if hybrid:
        rows, (ip, tk, im), ids = srv.export_inserts()
    else:
        rows, ids = srv.export_inserts()
    assert ids[0] == id_offset + corpus.shape[0]
    full = torch.cat([corpus, rows])
    words = (id_offset + full.shape[0] + 31) // 32
    kw = dict(kw, filters=filters[:, :words].contiguous())
    if hybrid:
        index = lr.ImpactIndex(V, id_offset=id_offset)
        index.add_csr(*_rows_csr(tok, imp))
        index.add_csr(ip, tk, im)
        return lr.OnlineHybridSearcher(bag, full, index, id_offset=id_offset, **kw)
    return lr.OnlineSearcher(bag, full, id_offset=id_offset, **kw)


def _equivalence(N, d, V, L, k, batch, sizes, hybrid, seed, id_offset=3):
    table, corpus, tok, imp = _make_data(N, d, V, L, seed)
    pad = V - 1
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=pad)
    cap = 16384
    n_ids = id_offset + N + cap
    gen = torch.Generator(device="cuda").manual_seed(seed + 1)
    keep = torch.nonzero(torch.rand(n_ids, device="cuda", generator=gen) < 0.6).flatten()
    filters = doc_bitmap(n_ids, keep, device="cuda").unsqueeze(0)
    kw = dict(k=k, batch=batch, max_tokens=batch * 32)
    if hybrid:
        index = lr.ImpactIndex(V, id_offset=id_offset)
        index.add_csr(*_rows_csr(tok, imp))
        srv = lr.OnlineHybridSearcher(bag, corpus, index, id_offset=id_offset, insert_capacity=cap, filters=filters,
                                      **kw)
    else:
        srv = lr.OnlineSearcher(bag, corpus, id_offset=id_offset, insert_capacity=cap, filters=filters, **kw)
    graph = srv._graph
    reqs = _requests(V, pad, batch, torch.Generator().manual_seed(seed + 2), sizes)
    before = _clone(srv.search(*reqs[0]))
    ins = _insert_batches(srv, bag, corpus, tok, imp, reqs, hybrid, gen)
    dead = torch.cat([torch.arange(id_offset, id_offset + N, 997), ins[1][::7], ins[2][::7]])
    srv.delete(dead)
    ref = _rebuilt(kw, srv, bag, corpus, tok, imp, hybrid, id_offset, V, filters)
    ref.delete(dead)
    assert srv._graph is graph                                        # never recaptured
    for i, (ids, offs) in enumerate(reqs):
        n = offs.numel()
        for rows in (None, [0 if j % 2 else -1 for j in range(n)]):
            got = _clone(srv.search(ids, offs, filter_rows=rows))
            exp = _clone(ref.search(ids, offs, filter_rows=rows))
            assert _same(got, exp), (i, rows)
            if i == 0 and rows is None:                               # the first batch outranks the main shard
                assert not _same(got, before)
                top = [got[0][1][:, 0], got[1][1][:, 0]] if hybrid else [got[1][:, 0]]
                assert all((t >= id_offset + N).all() for t in top), top
    del srv, ref


@gpu
@pytest.mark.parametrize("hybrid", [False, True])
def test_inserts_equal_a_rebuilt_searcher_small(hybrid):
    """20k x 256, V = 5000, 16 tokens per document, k = 100, batch 8, insert_capacity 16384."""
    _equivalence(20_000, 256, 5000, 16, 100, 8, (8, 1, 5), hybrid, seed=31)


@gpu
@pytest.mark.parametrize("hybrid", [False, True])
def test_inserts_equal_a_rebuilt_searcher_c5(hybrid):
    """1.1M x 3584 bf16, V = 128256, 64 tokens per document, k = 100, batch 32 and batch 1."""
    for batch, sizes in ((32, (32, 7)), (1, (1,))):
        _equivalence(1_100_000, 3584, V_BIG, 64, 100, batch, sizes, hybrid, seed=41 + batch)
    torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("hybrid", [False, True])
def test_insert_atomicity_and_restore_guard(hybrid):
    N, d, V, L = 5000, 128, 3000, 8
    table, corpus, tok, imp = _make_data(N, d, V, L, 51)
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)
    cap = 64
    kw = dict(k=20, batch=4, max_tokens=128, insert_capacity=cap)
    if hybrid:
        index = lr.ImpactIndex(V)
        index.add_csr(*_rows_csr(tok, imp))
        srv = lr.OnlineHybridSearcher(bag, corpus, index, insert_postings_capacity=cap * L, **kw)
    else:
        srv = lr.OnlineSearcher(bag, corpus, **kw)
    req = _requests(V, V - 1, 4, torch.Generator().manual_seed(5), (4,))[0]

    def insert(rows, t, m):
        return srv.insert(rows, *_rows_csr(t, m)) if hybrid else srv.insert(rows)

    r0 = _clone(srv.search(*req))
    assert insert(corpus[:0], tok[:0], imp[:0]).numel() == 0                 # 0 documents: nothing changes
    assert _same(_clone(srv.search(*req)), r0)
    ids = insert(corpus[:40] * 2, tok[:40], imp[:40] * 50)
    assert ids.tolist() == list(range(N, N + 40))
    r1 = _clone(srv.search(*req))
    assert not _same(r1, r0)
    with pytest.raises(ValueError, match="full"):                              # 40 + 30 > 64: nothing is written
        insert(corpus[:30], tok[:30], imp[:30])
    if hybrid:
        with pytest.raises(ValueError, match="full"):                          # postings overflow alone
            srv.insert(corpus[:2], torch.tensor([0, 1, cap * L]), torch.zeros(cap * L, dtype=torch.int32),
                       torch.ones(cap * L, dtype=torch.int32))
        with pytest.raises(ValueError, match="sparse documents"):
            srv.insert(corpus[:2], *_rows_csr(tok[:3], imp[:3]))
    assert _same(_clone(srv.search(*req)), r1)
    assert srv.export_inserts()[0].shape[0] == 40
    with pytest.raises(ValueError, match="no document"):
        srv.restore([N + 40])                                                  # an unfilled slot
    srv.delete(ids[:10])
    srv.restore(ids[:10])                                                      # filled slots: fine
    assert _same(_clone(srv.search(*req)), r1)


@gpu
@pytest.mark.parametrize("hybrid", [False, True])
def test_zero_capacity_is_the_existing_step(hybrid):
    """insert_capacity=0: the eager step launches as many library kernels as a searcher built without the new
    arguments and gives identical outputs."""
    N, d, V, L = 5000, 128, 3000, 8
    table, corpus, tok, imp = _make_data(N, d, V, L, 61)
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)
    lib = _C.load()
    outs, launches = [], []
    for extra in ({}, dict(insert_capacity=0)):
        if hybrid:
            index = lr.ImpactIndex(V)
            index.add_csr(*_rows_csr(tok, imp))
            srv = lr.OnlineHybridSearcher(bag, corpus, index, 20, 4, 128, use_graph=False, **extra)
        else:
            srv = lr.OnlineSearcher(bag, corpus, 20, 4, 128, use_graph=False, **extra)
        req = _requests(V, V - 1, 4, torch.Generator().manual_seed(6), (4,))[0]
        srv.search(*req)
        torch.cuda.synchronize()
        a = lib.lr_kernel_launches()
        outs.append(_clone(srv.search(*req)))
        torch.cuda.synchronize()
        launches.append(lib.lr_kernel_launches() - a)
    assert launches[0] == launches[1] and _same(outs[0], outs[1])


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one box")
def test_inserts_over_nccl():
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "nccl_insert_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and f"nccl insert worker OK world={world}" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
