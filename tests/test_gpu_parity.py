"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the reference-generated golden
fixtures.  Bars: bit-exact for ids / integer impacts / integer scores; dense scores within 1e-2 relative of the fp32
oracle on the same bf16-rounded inputs, ids exact outside the tie band (BASELINE.md §4)."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import lightretriever_b200 as lr
from oracle import oracle

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().float().cpu().numpy() if t.dtype in (torch.bfloat16, torch.float32) else t.detach().cpu().numpy()


# ------------------------------------------------------------------------------------------------ K1
def test_embbag_golden_fp32_is_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "embbag.npz"))
    pad = int(g["pad"])
    bag = lr.B200EmbeddingBag.from_pretrained(torch.from_numpy(g["table"]).cuda(), padding_idx=pad)
    ids, off = torch.from_numpy(g["ids"]).cuda(), torch.from_numpy(g["offsets"]).cuda()
    np.testing.assert_allclose(_np(bag.forward(ids, off)), g["out_full"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(_np(bag.encode(ids, off, shrink_dim=16, normalize=True)), g["out_m16_norm"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(_np(bag.encode(ids, off, normalize=True)), g["out_full_norm"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("V,d,m,norm", [(128256, 2048, None, True), (1000, 4096, 128, True), (777, 3584, 1024, False)])
def test_embbag_bf16_table_vs_oracle(V, d, m, norm):
    gen = torch.Generator().manual_seed(0)
    table = (torch.randn(V, d, generator=gen) * 0.02).bfloat16()
    lens = torch.randint(0, 33, (500,), generator=gen)
    lens[-1] = 5  # last bag runs to the end of ids
    ids = torch.randint(0, V, (int(lens.sum()),), generator=gen)
    pad = V - 3
    ids[::13] = pad
    ids[5:9] = ids[4]  # duplicate ids inside a bag
    offsets = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
    ref = oracle.embbag_encode(ids, offsets, table.float(), pad, m, norm).numpy()
    bag = lr.B200EmbeddingBag.from_pretrained(table.cuda(), padding_idx=pad)
    got32 = _np(bag.encode(ids.cuda(), offsets.cuda(), shrink_dim=m, normalize=norm, out_dtype=torch.float32))
    np.testing.assert_allclose(got32, ref, rtol=1e-5, atol=1e-7)
    got16 = _np(bag.encode(ids.cuda(), offsets.cuda(), shrink_dim=m, normalize=norm))
    np.testing.assert_allclose(got16, ref, rtol=1e-2, atol=1e-5)  # bf16 output rounding
    assert not got32[lens.numpy() == 0].any()  # empty bags -> zero vectors


def test_embbag_errors():
    bag = lr.B200EmbeddingBag.from_pretrained(torch.randn(50, 64).cuda())
    with pytest.raises(IndexError):
        bag.forward(torch.tensor([1, 50]).cuda(), torch.tensor([0]).cuda())
    with pytest.raises(ValueError):
        bag.encode(torch.tensor([1]).cuda(), torch.tensor([0]).cuda(), shrink_dim=12)  # not a multiple of 8
    out = bag.forward(torch.tensor([[1, 2], [3, 3]]).cuda())  # 2-D input = fixed-length bags
    assert out.shape == (2, 64)


def test_lasttoken_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "lasttoken.npz"))
    h = torch.from_numpy(g["hidden"]).cuda()
    for am, out in (("am_right", "out_right"), ("am_left", "out_left")):
        got = lr.lasttoken_head(h, torch.from_numpy(g[am]).cuda())
        np.testing.assert_array_equal(_np(got), g[out])
    ref = oracle.lasttoken_head(g["hidden"], g["am_right"], 8, True).numpy()
    got = lr.lasttoken_head(h.bfloat16(), torch.from_numpy(g["am_right"]).cuda(), 8, True, out_dtype=torch.float32)
    np.testing.assert_allclose(_np(got), oracle.lasttoken_head(h.bfloat16().float().cpu(), g["am_right"], 8, True).numpy(),
                               rtol=1e-5, atol=1e-6)
    assert ref.shape == (4, 8)


# ------------------------------------------------------------------------------------------------ K2
@pytest.mark.parametrize("Q,N,d", [(128, 256, 64), (300, 1000, 4096), (129, 257, 72), (1, 5, 8), (200, 5000, 3584)])
def test_gemm_mainloop_scores(Q, N, d):
    gen = torch.Generator().manual_seed(Q + N)
    q = torch.randn(Q, d, generator=gen).bfloat16().cuda()
    c = torch.randn(N, d, generator=gen).bfloat16().cuda()
    got = lr.flatip_scores(q, c)
    ref = q.float() @ c.float().T
    torch.testing.assert_close(got, ref, rtol=1e-3, atol=1e-3 * d ** 0.5)


@pytest.mark.parametrize("Q,N,d,k", [(64, 5000, 128, 10), (300, 20000, 256, 100), (130, 3000, 2048, 1000),
                                     (5, 100000, 64, 100), (1000, 100000, 2048, 100), (33, 70000, 3584, 1)])
def test_flatip_topk_vs_oracle(Q, N, d, k):
    gen = torch.Generator().manual_seed(k)
    q = F.normalize(torch.randn(Q, d, generator=gen), dim=-1).bfloat16()
    c = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16()
    s, i = lr.flatip_topk(q.cuda(), c.cuda(), k)
    ref = (q.float() @ c.float().T).numpy()  # fp32 math on the bf16-rounded values (SURVEY §8c trap 1)
    oracle.check_topk_parity(_np(s), _np(i), ref, k, rtol=1e-2)


def test_flatip_topk_config1_shape_ids_match_oracle():
    """BASELINE configs[0]: Llama-3.2-1B-shaped bag (V=128256, d=2048), 1k queries <=32 tokens, 100k docs, top-100."""
    gen = torch.Generator().manual_seed(0)
    V, d, Q, N, k = 128256, 2048, 1000, 100_000, 100
    table = (torch.randn(V, d, generator=gen) * 0.02).bfloat16()
    lens = torch.randint(1, 33, (Q,), generator=gen)
    ids = torch.randint(0, V, (int(lens.sum()),), generator=gen)
    offsets = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
    corpus = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16()
    bag = lr.B200EmbeddingBag.from_pretrained(table.cuda(), padding_idx=128002)
    qv = bag.encode(ids.cuda(), offsets.cuda(), normalize=True)
    ref_q = oracle.embbag_encode(ids, offsets, table.float(), 128002, None, True)
    np.testing.assert_allclose(_np(qv), ref_q.numpy(), rtol=1e-2, atol=1e-4)
    s, i = lr.flatip_topk(qv, corpus.cuda(), k)
    ref = (qv.float().cpu() @ corpus.float().T).numpy()
    oracle.check_topk_parity(_np(s), _np(i), ref, k, rtol=1e-2)
    es, ei = oracle.flatip_topk_fast(qv.float().cpu(), corpus.float(), k)
    assert (ei.numpy() == _np(i)).mean() > 0.999  # identical outside fp32 summation-order ties


def test_flatip_topk_edges_exact():
    gen = torch.Generator().manual_seed(2)
    q = torch.randn(7, 64, generator=gen).bfloat16()
    q[2] = 0  # zero query: every score ties at 0 -> ids 0..k-1
    c = torch.randn(50, 64, generator=gen).bfloat16()
    c[10:20] = c[5]  # exact duplicates: ties resolved by ascending id
    for k in (1, 10, 50, 100):  # k > N -> (-inf, -1) tail
        s, i = lr.flatip_topk(q.cuda(), c.cuda(), k, id_offset=1000)
        es, ei = oracle.flatip_topk(q.float(), c.float(), k, id_offset=1000)
        np.testing.assert_array_equal(_np(i), ei)
        np.testing.assert_allclose(_np(s), es, rtol=1e-3, atol=1e-4)
    with pytest.raises(ValueError):
        lr.flatip_topk(q.cuda(), c.cuda(), 0)
    with pytest.raises(ValueError):
        lr.flatip_topk(q.cuda(), c.cuda(), 4096)
    with pytest.raises(ValueError):
        lr.flatip_topk(q.cuda().float(), c.cuda(), 4)


def test_flatip_mrl_prefix_and_scales():
    """MRL (configs[2]): truncate-then-normalise == full-width rows scored on the prefix with reciprocal prefix norms."""
    gen = torch.Generator().manual_seed(3)
    qf = torch.randn(40, 1024, generator=gen).bfloat16()
    cf = torch.randn(3000, 1024, generator=gen).bfloat16()
    for m in (128, 256, 512):
        s, i = lr.flatip_topk(qf.cuda()[:, :m], cf.cuda()[:, :m], 20)  # strided views of full-width rows
        es, ei = oracle.flatip_topk(qf[:, :m].float(), cf[:, :m].float(), 20)
        np.testing.assert_array_equal(_np(i), ei)
        qs = 1.0 / qf[:, :m].float().norm(dim=1)
        cs = 1.0 / cf[:, :m].float().norm(dim=1)
        s2, i2 = lr.flatip_topk(qf.cuda(), cf.cuda(), 20, d_used=m, q_scale=qs.cuda(), c_scale=cs.cuda())
        ref = (F.normalize(qf[:, :m].float(), dim=-1) @ F.normalize(cf[:, :m].float(), dim=-1).T).numpy()
        oracle.check_topk_parity(_np(s2), _np(i2), ref, 20, rtol=1e-3)


def test_flatip_mrl_scales_large_batch_team_schedule():
    """MRL prefix scoring on the large-batch path (cta_group::2 pairs, team schedule with a multi-tile window, folded
    threshold filter with exact re-check): ids and scores against the fp32 oracle."""
    gen = torch.Generator().manual_seed(11)
    Q, N, d, m, k = 2100, 40000, 256, 128, 50
    qf = torch.randn(Q, d, generator=gen).bfloat16()
    cf = (torch.randn(N, d, generator=gen) * (0.5 + torch.rand(N, 1, generator=gen))).bfloat16()
    qs = 1.0 / qf[:, :m].float().norm(dim=1)
    cs = 1.0 / cf[:, :m].float().norm(dim=1)
    s, i = lr.flatip_topk(qf.cuda(), cf.cuda(), k, d_used=m, q_scale=qs.cuda(), c_scale=cs.cuda())
    ref = (F.normalize(qf[:, :m].float(), dim=-1) @ F.normalize(cf[:, :m].float(), dim=-1).T).numpy()
    oracle.check_topk_parity(_np(s), _np(i), ref, k, rtol=1e-3)
    # compact storage [N, m] without scales takes the same schedule
    qn = F.normalize(qf[:, :m].float(), dim=-1).bfloat16()
    cn = F.normalize(cf[:, :m].float(), dim=-1).bfloat16()
    s2, i2 = lr.flatip_topk(qn.cuda(), cn.cuda(), k)
    oracle.check_topk_parity(_np(s2), _np(i2), (qn.float() @ cn.float().T).numpy(), k, rtol=1e-3)


def test_flatip_adversarial_order_stays_exact():
    """Scores ascending with the document id: every document beats the running threshold, so the candidate lists
    overflow and are compacted over and over — the result must still be exact."""
    d, N, k = 64, 30000, 100
    base = torch.zeros(N, d)
    base[:, 0] = torch.linspace(0.1, 1.0, N)
    q = torch.zeros(3, d)
    q[:, 0] = torch.tensor([1.0, 0.5, -1.0])  # last query: descending order instead
    s, i = lr.flatip_topk(q.bfloat16().cuda(), base.bfloat16().cuda(), k)
    es, ei = oracle.flatip_topk(q.bfloat16().float(), base.bfloat16().float(), k)
    np.testing.assert_array_equal(_np(i), ei)


@pytest.mark.parametrize("prefix_docs,cluster", [(512, 2), (2048, 1), (300, 2)])
def test_flatip_two_phase_warm_start_is_exact(monkeypatch, prefix_docs, cluster):
    """Phase A (corpus prefix seeds the thresholds, its top-k joins the merge) + phase B must equal the one-pass result,
    including ties that straddle the prefix boundary and results that live entirely inside the prefix."""
    monkeypatch.setenv("LR_FLATIP_PREFIX_DOCS", str(prefix_docs))
    monkeypatch.setenv("LR_FLATIP_CLUSTER", str(cluster))
    lr._C.reload_env()  # the knobs are cached after the first call
    gen = torch.Generator().manual_seed(prefix_docs)
    Q, N, d, k = 300, 30000, 128, 100
    q = F.normalize(torch.randn(Q, d, generator=gen), dim=-1).bfloat16()
    c = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16()
    c[prefix_docs - 3:prefix_docs + 3] = c[7]          # exact ties across the phase boundary
    c[:50] = q[:50]                                    # best documents of the first queries sit in the prefix
    s, i = lr.flatip_topk(q.cuda(), c.cuda(), k, id_offset=5)
    es, ei = oracle.flatip_topk(q.float(), c.float(), k, id_offset=5)
    ref = (q.float() @ c.float().T).numpy()
    oracle.check_topk_parity(_np(s), _np(i), ref, k, rtol=1e-2, id_offset=5)
    assert (ei == _np(i)).mean() > 0.999
    # adversarial order (scores ascending with the id) under the two-phase plan
    base = torch.zeros(20000, 64)
    base[:, 0] = torch.linspace(0.1, 1.0, 20000)
    qq = torch.zeros(2, 64)
    qq[:, 0] = torch.tensor([1.0, -1.0])
    s2, i2 = lr.flatip_topk(qq.bfloat16().cuda(), base.bfloat16().cuda(), 50)
    _, ei2 = oracle.flatip_topk(qq.bfloat16().float(), base.bfloat16().float(), 50)
    np.testing.assert_array_equal(_np(i2), ei2)
    monkeypatch.undo()
    lr._C.reload_env()


def test_searcher_surface_matches_reference_protocol():
    gen = torch.Generator().manual_seed(4)
    corpus = F.normalize(torch.randn(600, 128, generator=gen), dim=-1)
    queries = F.normalize(torch.randn(5, 128, generator=gen), dim=-1)
    cids = [f"doc-{j}" for j in range(600)]
    qids = [f"q-{j}" for j in range(5)]
    search = lr.FlatIPSearch(model=None)
    search.index(corpus, cids)                                   # faiss_search.py:490-504
    res = search.retrieve_with_emb(queries.numpy(), qids, 10)    # faiss_search.py:143-173
    es, ei = oracle.flatip_topk(queries.bfloat16().float(), corpus.bfloat16().float(), 10)
    for r, qid in enumerate(qids):
        assert list(res[qid].keys()) == [cids[j] for j in ei[r]]
        np.testing.assert_allclose(list(res[qid].values()), es[r], rtol=1e-2, atol=1e-4)
    # chunked search + merge == one-shot search (hybrid_search.py:301-344); the merge runs on device (lr_topk_merge)
    s_c, i_c = search.search_arrays(((lo, corpus[lo:lo + 250]) for lo in range(0, 600, 250)), queries, 10)
    np.testing.assert_array_equal(_np(i_c), ei)
    # ... and equals the reference's host heap merge of the per-chunk dicts (played by the oracle)
    heaps = {}
    for lo in range(0, 600, 250):
        search._clear()
        search.index(corpus[lo:lo + 250], cids[lo:lo + 250])
        oracle.add_to_heap(search.retrieve_with_emb(queries, qids, 10), heaps, 10, False)
    for r, qid in enumerate(qids):
        assert sorted(p for _, p in heaps[qid]) == sorted(res[qid].keys())
    search._clear()
    with pytest.raises(RuntimeError):
        search.retrieve_with_emb(queries, qids, 10)
    # FaissIndex-style arrays, fewer docs than k
    idx = lr.FlatIPIndex.build(list(range(7)), corpus[:7])
    sc, ids = idx.search(queries.numpy(), 10)
    assert sc.dtype == np.float32 and ids.dtype == np.int64 and (ids[:, 7:] == -1).all() and np.isneginf(sc[:, 7:]).all()


def test_merge_kernel_exact():
    rng = np.random.default_rng(0)
    L, Q, cap, k = 8, 33, 100, 100
    scores = rng.standard_normal((L, Q, cap)).astype(np.float32)
    scores[:, :, ::7] = 0.25
    ids = np.stack([rng.permutation(100000)[:L * cap].reshape(L, cap) for _ in range(Q)], 1).astype(np.int64)
    keys = lr.encode_keys(torch.from_numpy(scores).cuda(), torch.from_numpy(ids).cuda())
    np.testing.assert_array_equal(_np(keys).view(np.uint64), oracle.encode_keys(scores, ids))
    s, i, ok = lr.topk_merge(keys, k, return_keys=True)
    es, ei = oracle.merge_topk(list(scores), list(ids), k)
    np.testing.assert_array_equal(_np(i), ei)
    np.testing.assert_array_equal(_np(s), es)
    np.testing.assert_array_equal(_np(ok).view(np.uint64), oracle.encode_keys(es, ei))
    counts = rng.integers(0, cap + 1, (L, Q)).astype(np.int32)
    counts[:, 0] = 0  # a query without any candidate
    s, i = lr.topk_merge(keys, 37, counts=torch.from_numpy(counts).cuda())
    m = np.arange(cap)[None, None] < counts[:, :, None]
    es, ei = oracle.merge_topk(list(np.where(m, scores, -np.inf)), list(np.where(m, ids, -1)), 37)
    np.testing.assert_array_equal(_np(i), ei)
    assert (ei[0] == -1).all()


@pytest.mark.parametrize("L,Q,cap,k", [(6, 3, 5000, 4096), (300, 2, 64, 50), (600, 1, 40, 7), (3, 200, 3000, 2048)])
def test_merge_kernel_shapes_around_the_staging_limits(L, Q, cap, k):
    """Public lr_topk_merge at the edges of the shared-memory staging: k = 4096 with the large staging area, more lists
    than the offset table holds (> 512: streaming passes), long lists with a full grid (48 KB staging, streaming)."""
    rng = np.random.default_rng(L * 7 + k)
    scores = rng.standard_normal((L, Q, cap)).astype(np.float32)
    ids = np.stack([rng.permutation(L * cap + 17)[:L * cap].reshape(L, cap) for _ in range(Q)], 1).astype(np.int64)
    keys = lr.encode_keys(torch.from_numpy(scores).cuda(), torch.from_numpy(ids).cuda())
    s, i = lr.topk_merge(keys, k)
    es, ei = oracle.merge_topk(list(scores), list(ids), k)
    np.testing.assert_array_equal(_np(i), ei)
    np.testing.assert_array_equal(_np(s), es)


# ------------------------------------------------------------------------------------------------ K3
def test_sparse_head_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "sparse_head.npz"))
    h, W, b = (torch.from_numpy(g[n]).cuda() for n in ("h", "W", "bias"))
    mask = torch.from_numpy(g["mask"]).cuda()
    got = _np(lr.max_linear_mapping(h, W, b, mask))  # weight [d, V] as in the reference signature
    fin = g["out_f32"] > -1e30
    # inputs are rounded to bf16 by the kernel: compare with the oracle on the rounded values, and with the
    # reference's own fp32 output inside the bf16 band of max_linear_map.py:192-196
    ref = oracle.max_linear_map(h.bfloat16().float().cpu(), W.bfloat16().float().cpu(), b.cpu(), g["mask"]).numpy()
    np.testing.assert_allclose(got[fin], ref[fin], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(got[fin], g["out_f32"][fin], rtol=5e-2, atol=5e-2)
    assert (got[~fin] < -1e30).all()  # no valid token -> finfo(bf16).min
    got_rl = _np(lr.max_linear_mapping(h, W, b, mask, relu=True, log1p=True))
    np.testing.assert_allclose(got_rl, np.log1p(np.maximum(ref, 0)), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("packed", [True, False])
@pytest.mark.parametrize("B,S,d,V", [(3, 64, 128, 1000), (5, 100, 256, 3001), (2, 512, 512, 5000), (9, 33, 64, 129)])
def test_sparse_head_vs_oracle(B, S, d, V, packed):
    gen = torch.Generator().manual_seed(S)
    h = torch.randn(B, S, d, generator=gen).bfloat16()
    W = (torch.randn(V, d, generator=gen) * 0.05).bfloat16()
    bias = torch.randn(V, generator=gen) * 0.1
    lens = torch.randint(3, S + 1, (B,), generator=gen)
    am = (torch.arange(S)[None] < lens[:, None]).long()
    am[1] = 0
    am[1, :2] = 1  # nothing valid once first/last are dropped
    mask = oracle.sparse_attention_mask(torch.zeros(B, S, dtype=torch.long), am, sep_token_id=-1)
    ref = oracle.max_linear_map(h.float(), W.float().T, bias, mask)
    got = lr.max_linear_mapping(h.cuda(), W.cuda(), bias.cuda(), mask.cuda(), weight_is_vd=True, packed=packed).cpu()
    fin = ref > -1e30
    torch.testing.assert_close(got[fin], ref[fin], rtol=1e-4, atol=1e-4)
    assert bool((got[~fin] < -1e30).all())
    # integer stage is bit-exact given the same fp32 reps
    reps = oracle.get_sparse_emb(ref, True, True, top_k=0)
    for top_k in (0, 16, 64):
        exp = oracle.quantize_reps(oracle.top_k_sampling(reps, top_k, min_tokens_to_keep=8), 100)
        ip, tk, im = lr.sparsify_quantize(reps.cuda(), top_k=top_k, min_tokens_to_keep=8)
        assert lr.csr_to_json(ip, tk, im) == exp
    # fused path: exact impacts and token sets, except where the max-linear error bound (the rtol/atol above) leaves the
    # rounding, the top-k cut or the `impact >= 1` cut undecided
    ip, tk, im = lr.sparse_head(h.cuda(), W.cuda(), bias.cuda(), mask.cuda(), True, True, 64, 8, 100.0)
    eps = (1e-4 * ref.abs() + 1e-4).masked_fill(~fin, 1e-4).numpy()   # a document without tokens: reps are all 0
    bad, band = oracle.check_sparse_impacts(lr.csr_to_json(ip, tk, im), reps.numpy(), eps, 64, 8, 100.0)
    assert not bad, (len(bad), bad[:5], band)


@pytest.mark.parametrize("tiles_per_split", [None, 1, 3, 1000])
def test_sparse_head_packed_ragged_documents(monkeypatch, tiles_per_split):
    """Packed tokens (lr_pack_tokens + lr_sparse_head_max_packed): ragged lengths from 0 to S, empty documents at the
    start, in the middle and at the end, masked tokens inside a document, and splits cut at whole 256-token tiles — with
    one tile per split a 700-token document crosses two cuts and covers a whole split, others end exactly on a cut.
    Bit-identical to the padded kernel (same products, same max), and both match the oracle."""
    B, S, d, V = 37, 700, 128, 2500
    gen = torch.Generator().manual_seed(11)
    h = torch.randn(B, S, d, generator=gen).bfloat16()
    W = (torch.randn(V, d, generator=gen) * 0.05).bfloat16()
    bias = torch.randn(V, generator=gen) * 0.1
    lens = torch.randint(0, 301, (B,), generator=gen)
    lens[[0, 1, 7, 8, 20, B - 1]] = 0
    lens[5] = S
    lens[2] = 256 - int(lens[:2].sum())          # documents 0..2 end exactly on the first tile boundary
    lens[3] = 256
    mask = torch.arange(S)[None] < lens[:, None]
    holes = torch.rand(B, S, generator=gen) > 0.1  # holes inside the documents (not in the two that pin the boundary)
    holes[2:4] = True
    mask &= holes
    if tiles_per_split is not None:
        monkeypatch.setenv("LR_SPARSE_HEAD_TILES_PER_SPLIT", str(tiles_per_split))
    lr._C.reload_env()  # the knobs are cached after the first call
    hp, cu, T = lr.pack_tokens(h.cuda(), mask.cuda())
    assert T == int(mask.sum()) and cu.cpu().tolist() == [0] + torch.cumsum(mask.sum(1), 0).tolist()
    assert torch.equal(hp.cpu(), h[mask])
    got = lr.max_linear_mapping(h.cuda(), W.cuda(), bias.cuda(), mask.cuda(), weight_is_vd=True, valid_tokens=T).cpu()
    pad = lr.max_linear_mapping(h.cuda(), W.cuda(), bias.cuda(), mask.cuda(), weight_is_vd=True, packed=False).cpu()
    assert torch.equal(got, pad)
    ref = oracle.max_linear_map(h.float(), W.float().T, bias, mask)
    fin = ref > -1e30
    torch.testing.assert_close(got[fin], ref[fin], rtol=1e-4, atol=1e-4)
    assert bool((got[~fin] < -1e30).all()) and int((~fin).any(1).sum()) >= 6
    act = lr.max_linear_mapping(h.cuda(), W.cuda(), bias.cuda(), mask.cuda(), relu=True, log1p=True, weight_is_vd=True).cpu()
    torch.testing.assert_close(act, torch.log1p(torch.relu(ref)), rtol=1e-4, atol=1e-5)
    # nothing valid at all
    none = lr.max_linear_mapping(h.cuda(), W.cuda(), None, torch.zeros(B, S, dtype=torch.bool).cuda(), relu=True, log1p=True,
                                 weight_is_vd=True)
    assert float(none.abs().max()) == 0.0
    monkeypatch.undo()
    lr._C.reload_env()


@pytest.mark.parametrize("window", [1, 3])
def test_sparse_head_team_schedule_matches_round_robin(monkeypatch, window):
    """The team schedule (fixed cluster teams per vocabulary band + progress window) only reorders units: results are
    bit-identical to the round-robin schedule and match the oracle."""
    B, S, d, V = 6, 128, 256, 9000
    gen = torch.Generator().manual_seed(window)
    h = torch.randn(B, S, d, generator=gen).bfloat16()
    W = (torch.randn(V, d, generator=gen) * 0.05).bfloat16()
    lens = torch.randint(3, S + 1, (B,), generator=gen)
    mask = (torch.arange(S)[None] < lens[:, None])
    monkeypatch.setenv("LR_SPARSE_HEAD_DOCS_PER_UNIT", "1")
    monkeypatch.setenv("LR_SPARSE_HEAD_SCHED", "0")
    lr._C.reload_env()  # the knobs are cached after the first call
    rr = lr.max_linear_mapping(h.cuda(), W.cuda(), None, mask.cuda(), relu=True, log1p=True, weight_is_vd=True)
    monkeypatch.setenv("LR_SPARSE_HEAD_SCHED", "1")
    monkeypatch.setenv("LR_SPARSE_HEAD_TEAM_BAND", "8")   # 36 row groups -> 4 full bands of 9 teams + a 4-group band
    monkeypatch.setenv("LR_SPARSE_HEAD_TEAM_WINDOW", str(window))
    for mode in ("2", "3"):                                  # multicast cluster, cta_group::2 pair
        monkeypatch.setenv("LR_SPARSE_HEAD_CLUSTER", mode)
        lr._C.reload_env()
        got = lr.max_linear_mapping(h.cuda(), W.cuda(), None, mask.cuda(), relu=True, log1p=True, weight_is_vd=True)
        assert torch.equal(got, rr)
    ref = torch.log1p(torch.relu(oracle.max_linear_map(h.float(), W.float().T, None, mask)))
    torch.testing.assert_close(rr.cpu(), ref, rtol=1e-4, atol=1e-4)
    monkeypatch.undo()
    lr._C.reload_env()


def test_top_p_sampling_golden(golden_dir):
    """lr_top_p_filter vs the imported reference's outputs (tests/golden/top_p.npz).  The reference's float32 cumsum has
    no defined rounding, so an entry may differ only when its cumulative probability lies within 2e-6 of the bound
    1 - top_p (the oracle returns that probability); the entries kept by the min_keep rule must agree exactly."""
    g = np.load(os.path.join(golden_dir, "top_p.npz"))
    reps = torch.from_numpy(g["reps"])
    for name in (k for k in g.files if k != "reps"):
        tp, mk = float(name.split("_")[0][1:]), int(name.split("_k")[1])
        got = _np(lr.top_p_sampling(reps.cuda(), tp, min_tokens_to_keep=mk))
        ref = g[name]
        if tp <= 0 or tp >= 1:
            np.testing.assert_array_equal(got, ref)
            continue
        _, cum = oracle.top_p_sampling(reps.clone(), tp, min_tokens_to_keep=mk)
        diff = got != ref
        near = np.abs(cum.numpy() - (1.0 - tp)) <= 2e-6
        assert not (diff & ~near).any(), (name, int(diff.sum()), int((diff & ~near).sum()))
        assert diff.sum() <= 2 * reps.shape[0], (name, int(diff.sum()))
        assert ((got == 0) | (got == g["reps"])).all()
        # the rows where the min_keep cap binds keep exactly the min_keep largest entries
        for r in range(reps.shape[0]):
            if (ref[r] != 0).sum() == mk and (g["reps"][r] != 0).sum() > mk:
                np.testing.assert_array_equal(got[r], ref[r])
    x = reps.cuda().clone()
    assert lr.top_p_sampling(x, 0.3, min_tokens_to_keep=8, inplace=True).data_ptr() == x.data_ptr()


def test_score_definitions_match_the_reference_notebook_cells_on_device(golden_dir):
    """K4 and K2 against the reference's own notebook cells (exec'd by oracle/gen_golden_r2.py): integer impact scores
    bit-exact, dense scores within 1e-2 relative (bf16 inputs vs the notebook's fp32)."""
    g = np.load(os.path.join(golden_dir, "notebook_cells.npz"))
    queries = [{int(k): v for k, v in q.items()} for q in json.loads(str(g["sparse_queries"]))]
    docs = json.loads(str(g["sparse_docs"]))
    s = lr.ImpactSearch(vocab_size=400)
    s.index(docs, [str(j) for j in range(len(docs))])
    res = s.retrieve_with_emb(queries, [f"q{i}" for i in range(len(queries))], top_k=len(docs))
    ref = g["sparse_scores"]
    for qi in range(len(queries)):
        exp = {str(j): float(ref[qi, j]) for j in range(len(docs)) if ref[qi, j] > 0}
        assert res.get(f"q{qi}", {}) == exp
    q, c = torch.from_numpy(g["dense_q"]).cuda(), torch.from_numpy(g["dense_c"]).cuda()
    got = _np(lr.flatip_scores(q.bfloat16(), c.bfloat16()))
    np.testing.assert_allclose(got, g["dense_scores"], rtol=1e-2, atol=1e-2 * np.abs(g["dense_scores"]).max())


def test_quantiser_golden_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "quantize.npz"))
    got = lr.convert_sparse_reps_to_json(torch.from_numpy(g["reps"]).cuda(), quantization_factor=100)
    assert got == json.loads(str(g["json"]))


def test_topk_sampling_golden_ties(golden_dir):
    g = np.load(os.path.join(golden_dir, "sparse_head.npz"))
    tied = torch.from_numpy(g["tied"]).cuda()
    for top_k, mk, name in ((3, 1, "tied_top3"), (2, 8, "tied_top2_min8"), (0, 8, "tied_top0")):
        ip, tk, im = lr.sparsify_quantize(tied, top_k=top_k, min_tokens_to_keep=mk)
        assert lr.csr_to_json(ip, tk, im) == oracle.quantize_reps(g[name], 100)


# ------------------------------------------------------------------------------------------------ K4
def _rand_docs(rng, n, V, nnz, max_imp=400):
    docs = []
    for _ in range(n):
        toks = rng.choice(V, size=int(rng.integers(0, nnz + 1)), replace=False)
        docs.append({str(int(t)): int(rng.integers(1, max_imp + 1)) for t in toks})
    return docs


@pytest.mark.parametrize("N,V,nnz,Q,k", [(3000, 500, 40, 20, 10), (40000, 2000, 64, 16, 100), (20000, 300, 30, 8, 1000),
                                         (70000, 50, 8, 300, 5)])
def test_sparse_score_bit_exact(N, V, nnz, Q, k):
    rng = np.random.default_rng(N)
    docs = _rand_docs(rng, N, V, nnz)
    queries = [" ".join(str(int(t)) for t in rng.integers(0, V + 5, size=int(rng.integers(1, 33)))) for _ in range(Q)]
    queries[0] = ""  # a query without terms returns nothing
    searcher = lr.ImpactSearch(vocab_size=V)
    half = N // 2
    searcher.index(docs[:half], [f"d{j}" for j in range(half)])  # chunked indexing, anserini_search.py:89-111
    searcher.index(docs[half:], [f"d{j}" for j in range(half, N)])
    res = searcher.retrieve_with_emb(queries, [f"q{j}" for j in range(Q)], k)
    qd = [oracle.query_counts([int(t) for t in s.split()]) for s in queries]
    es, ei = oracle.impact_topk(qd, [{int(a): b for a, b in d.items()} for d in docs], k)
    assert "q0" not in res
    for r in range(Q):
        exp = {f"d{j}": float(s) for s, j in zip(es[r], ei[r]) if j >= 0}
        assert res.get(f"q{r}", {}) == exp, f"query {r}"
    # array form: sorted (score desc, id asc), integer scores, (-inf, -1) tail
    from lightretriever_b200.sparse_search import parse_queries
    s, i = searcher._ensure_index().search_device(*parse_queries(queries, V), k)
    np.testing.assert_array_equal(_np(i), ei)
    np.testing.assert_array_equal(_np(s), es)
    searcher._clear()
    with pytest.raises(RuntimeError):
        searcher.retrieve_with_emb(queries, ["q"] * Q, k)


def test_sparse_score_long_queries_and_dense_blocks():
    """Queries with more than 32 distinct terms (several term chunks per step), a head term present in most documents
    (touched-list overflow -> block scan) and k close to the list capacity; counts <= 0 contribute nothing."""
    rng = np.random.default_rng(77)
    N, V, k = 30000, 400, 300
    docs = _rand_docs(rng, N, V, 24)
    for j in range(0, N, 3):
        docs[j]["7"] = int(rng.integers(1, 50))  # head term
    searcher = lr.ImpactSearch(vocab_size=V)
    searcher.index(docs, [f"d{j}" for j in range(N)])
    queries = [" ".join(str(int(t)) for t in rng.integers(0, V, size=n)) for n in (33, 64, 100, 257, 1, 31, 32)]
    queries.append("7 7 7 8")
    from lightretriever_b200.sparse_search import parse_queries
    qd = [oracle.query_counts([int(t) for t in s.split()]) for s in queries]
    es, ei = oracle.impact_topk(qd, [{int(a): b for a, b in d.items()} for d in docs], k)
    s, i = searcher._ensure_index().search_device(*parse_queries(queries, V), k)
    np.testing.assert_array_equal(_np(i), ei)
    np.testing.assert_array_equal(_np(s), es)
    # a zero / negative count removes the term
    qi, qt, qc = parse_queries(["7 8 9", "7 9"], V)
    qc = np.asarray(qc).copy()
    qt_l = list(np.asarray(qt)[: int(np.asarray(qi)[1])])
    qc[qt_l.index(8)] = 0
    s2, i2 = searcher._ensure_index().search_device(qi, qt, qc, 20)
    np.testing.assert_array_equal(_np(i2)[0], _np(i2)[1])
    np.testing.assert_array_equal(_np(s2)[0], _np(s2)[1])


def test_sparse_score_wide_scores_take_the_int32_pass():
    """Scores above 65535 do not fit the 16-bit accumulators of the first pass: the overflow flag must route the launch
    through the int32 pass, bit-exact; a second search on the same index (small scores) stays on the 16-bit pass."""
    rng = np.random.default_rng(5)
    N, V, k = 20000, 120, 50
    docs = _rand_docs(rng, N, V, 20, max_imp=65535)
    searcher = lr.ImpactSearch(vocab_size=V)
    searcher.index(docs, [f"d{j}" for j in range(N)])
    from lightretriever_b200.sparse_search import parse_queries
    for queries in (["3 3 3 4 5 6 7", "8 9 10 11 12 13 14 15 16 17 18 19 20 21 22", "30"] * 5, ["40", "41 42"]):
        qd = [oracle.query_counts([int(t) for t in s.split()]) for s in queries]
        es, ei = oracle.impact_topk(qd, [{int(a): b for a, b in d.items()} for d in docs], k)
        s, i = searcher._ensure_index().search_device(*parse_queries(queries, V), k)
        np.testing.assert_array_equal(_np(i), ei)
        np.testing.assert_array_equal(_np(s), es)


def test_sparse_score_document_shards_merge_to_the_global_topk():
    """Multi-GPU sparse path (SURVEY §8e) on one device: per-shard inverted indexes with id offsets -> per-shard top-k keys
    -> lr_topk_merge with integer scores == the unsharded search == the oracle.  (The exchange itself is covered by the
    world-2 gloo test; ShardedImpactIndex with world == 1 must equal the plain index.)"""
    from lightretriever_b200 import _C as C
    from lightretriever_b200.sharded import shard_range
    from lightretriever_b200.sparse_search import parse_queries
    rng = np.random.default_rng(21)
    N, V, k, world = 9001, 300, 64, 3
    docs = _rand_docs(rng, N, V, 12)
    ip = np.zeros(N + 1, np.int64)
    tok, imp = [], []
    for j, d in enumerate(docs):
        tok += [int(t) for t in d]
        imp += list(d.values())
        ip[j + 1] = len(tok)
    tok, imp = np.asarray(tok, np.int32), np.asarray(imp, np.int32)
    queries = [" ".join(str(int(t)) for t in rng.integers(0, V, size=int(rng.integers(1, 20)))) for _ in range(33)]
    qi, qt, qc = parse_queries(queries, V)
    keys = []
    for r in range(world):
        lo, hi = shard_range(N, r, world)
        shard = lr.ImpactIndex(V, id_offset=lo)
        shard.add_csr(ip[lo:hi + 1] - ip[lo], tok[ip[lo]:ip[hi]], imp[ip[lo]:ip[hi]])
        keys.append(shard.search_device(qi, qt, qc, k, return_keys=True)[2])
    s, i = lr.topk_merge(torch.stack(keys, 0).contiguous(), k, score_kind=C.LR_SCORE_U32)
    es, ei = oracle.impact_topk([oracle.query_counts([int(t) for t in q.split()]) for q in queries],
                                [{int(a): b for a, b in d.items()} for d in docs], k)
    np.testing.assert_array_equal(_np(i), ei)
    np.testing.assert_array_equal(_np(s), es)
    whole = lr.ShardedImpactIndex(V, N)  # world == 1 here
    whole.add_local_csr(ip, tok, imp)
    s1, i1 = whole.search_device(qi, qt, qc, k)
    np.testing.assert_array_equal(_np(i1), ei)
    np.testing.assert_array_equal(_np(s1), es)


def test_sparse_head_to_sparse_search_roundtrip():
    """K3 output (CSR) feeds K4 directly, and through the reference's JSON form, with identical results."""
    gen = torch.Generator().manual_seed(9)
    B, S, d, V = 40, 32, 64, 300
    h = torch.randn(B, S, d, generator=gen).bfloat16().cuda()
    W = (torch.randn(V, d, generator=gen) * 0.2).bfloat16().cuda()
    mask = torch.ones(B, S, dtype=torch.bool).cuda()
    ip, tk, im = lr.sparse_head(h, W, None, mask, True, True, 16, 8, 100.0)
    docs_json = lr.csr_to_json(ip, tk, im)
    cids = [f"d{j}" for j in range(B)]
    a, b = lr.ImpactSearch(vocab_size=V), lr.ImpactSearch(vocab_size=V)
    a.index((ip, tk, im), cids)
    b.index(docs_json, cids)
    queries = ["1 2 3 4 5 5", "7 8 299", "10"]
    ra = a.retrieve_with_emb(queries, ["a", "b", "c"], 10)
    rb = b.retrieve_with_emb(queries, ["a", "b", "c"], 10)
    assert ra == rb
    es, ei = oracle.impact_topk([oracle.query_counts([int(t) for t in q.split()]) for q in queries],
                                [{int(t): v for t, v in dj.items() if int(t) >= 0} for dj in docs_json], 10)
    for r, qid in enumerate(["a", "b", "c"]):
        assert ra.get(qid, {}) == {f"d{j}": float(s) for s, j in zip(es[r], ei[r]) if j >= 0}


# ------------------------------------------------------------------------------------------------ fusion + hybrid orchestration
@pytest.mark.parametrize("k0,k1,method", [(10, 10, "linear"), (100, 37, "linear"), (1000, 1000, "linear"), (64, 100, "rrf"),
                                          (2048, 2048, "linear"), (2048, 2047, "linear"), (1, 4095, "linear")])
def test_device_fusion_bit_exact_vs_reference_semantics(k0, k1, method):
    rng = np.random.default_rng(k0 + k1)
    Q = 9
    s0 = -np.sort(-rng.standard_normal((Q, k0)).astype(np.float32), axis=1)
    s1 = -np.sort(-rng.integers(1, 5000, (Q, k1)).astype(np.float32), axis=1)
    h = min(k0, k1) // 2  # documents returned by both systems
    uni = np.stack([rng.permutation(3 * (k0 + k1)) for _ in range(Q)]).astype(np.int64)
    i0 = uni[:, :k0].copy()
    i1 = np.concatenate([i0[:, :h], uni[:, k0:k0 + k1 - h]], axis=1)
    i1 = np.stack([rng.permutation(row) for row in i1])  # ids are unique inside a system, shared across systems
    i1[0, -3:] = -1  # padding (fewer than k hits)
    s1[0, -3:] = -np.inf
    ids, fused, counts = lr.fuse_topk_device(torch.from_numpy(s0).cuda(), torch.from_numpy(i0).cuda(),
                                             torch.from_numpy(s1).cuda(), torch.from_numpy(i1).cuda(), method=method)
    ids, fused, counts = _np(ids), fused.cpu().numpy(), _np(counts)
    for q in range(Q):
        d0 = {str(i): float(s) for s, i in zip(s0[q], i0[q]) if i >= 0}
        d1 = {str(i): float(s) for s, i in zip(s1[q], i1[q]) if i >= 0}
        ref = (oracle.fuse_linear([{"q": d0}, {"q": d1}], weights=[0.7, 0.3]) if method == "linear"
               else oracle.fuse_rrf([{"q": d0}, {"q": d1}]))["q"]
        n = counts[q]
        assert n == len(ref)
        got = {str(i): f for i, f in zip(ids[q, :n], fused[q, :n])}
        assert got.keys() == ref.keys()
        for pid, v in ref.items():
            assert got[pid] == v, (pid, got[pid], v)  # float64, same operation order -> bit-exact
        assert (np.diff(fused[q, :n]) <= 0).all() and (ids[q, n:] == -1).all()


def test_hybrid_search_end_to_end_with_fake_model():
    """HybridSearch.search (hybrid_search.py:234-403): chunked dense index/retrieve + heap merge, sparse index per
    chunk + one retrieve, linear fusion — against the same flow played by the oracle."""
    gen = torch.Generator().manual_seed(21)
    n_docs, n_q, d, V, k = 300, 6, 64, 97, 20
    doc_vec = F.normalize(torch.randn(n_docs, d, generator=gen), dim=-1)
    q_vec = F.normalize(torch.randn(n_q, d, generator=gen), dim=-1)
    rng = np.random.default_rng(5)
    doc_sparse = [{str(int(t)): int(rng.integers(1, 300)) for t in rng.choice(V, 12, replace=False)} for _ in range(n_docs)]
    q_tok = [" ".join(str(int(t)) for t in rng.integers(0, V, size=6)) for _ in range(n_q)]
    corpus = {f"d{j}": {"text": "x" * (1 + j % 7), "j": j} for j in range(n_docs)}
    queries = {f"q{j}": f"query {j}" for j in range(n_q)}

    class FakeModel:
        def encode_queries(self, queries, **kw):
            return {"emb_reps": q_vec, "token_id_reps": q_tok}

        def encode_corpus(self, corpus, **kw):
            idx = [c["j"] for c in corpus]
            return {"dense_reps": doc_vec[idx], "sparse_reps": [doc_sparse[j] for j in idx]}

    hs = lr.HybridSearch(FakeModel(), batch_size=16, corpus_chunk_size=128, return_all_results=True, vocab_size=V)
    res = hs.search(corpus, queries, top_k=k)
    # oracle flow
    qb, cb = q_vec.bfloat16().float(), doc_vec.bfloat16().float()
    es, ei = oracle.flatip_topk(qb, cb, k)
    emb = {f"q{r}": {f"d{j}": float(s) for s, j in zip(es[r], ei[r])} for r in range(n_q)}
    ts, ti = oracle.impact_topk([oracle.query_counts([int(t) for t in s.split()]) for s in q_tok],
                                [{int(a): b for a, b in dd.items()} for dd in doc_sparse], k)
    tok = {f"q{r}": {f"d{j}": float(s) for s, j in zip(ts[r], ti[r]) if j >= 0} for r in range(n_q)}
    for r in range(n_q):
        qid = f"q{r}"
        assert res["emb"][qid].keys() == emb[qid].keys()
        assert res["tok"].get(qid, {}) == tok.get(qid, {})
    fused = oracle.fuse_linear([res["emb"], res["tok"]], weights=[0.7, 0.3])
    for qid in fused:
        assert res["emb_tok"][qid].keys() == fused[qid].keys()
        for pid, v in fused[qid].items():
            assert abs(res["emb_tok"][qid][pid] - v) < 1e-12


def test_array_first_retrieval_and_jsonl_roundtrip(tmp_path):
    """Rows f2 / f3: results stay on device as arrays (dicts only on request), and a corpus dumped in the reference's
    Anserini JSONL layout (anserini_search.py:89-111) is ingested back with identical search results."""
    gen = torch.Generator().manual_seed(33)
    n_docs, n_q, d, V, k = 500, 7, 64, 211, 16
    doc_vec = F.normalize(torch.randn(n_docs, d, generator=gen), dim=-1)
    q_vec = F.normalize(torch.randn(n_q, d, generator=gen), dim=-1)
    rng = np.random.default_rng(9)
    docs = [{str(int(t)): int(rng.integers(1, 300)) for t in rng.choice(V, 9, replace=False)} for _ in range(n_docs)]
    docs[17] = {"-1": 1}  # the reference's empty-document marker
    q_tok = [" ".join(str(int(t)) for t in rng.integers(0, V, size=5)) for _ in range(n_q)]
    cids = [f"d{j}" for j in range(n_docs)]
    qids = [f"q{j}" for j in range(n_q)]
    hs = lr.HybridSearch(model=None, vocab_size=V)
    hs.index({"dense_reps": doc_vec, "sparse_reps": docs}, cids)
    fid, fsc, cnt = hs.retrieve_arrays({"emb_reps": q_vec, "token_id_reps": q_tok}, k)
    dict_res = hs.retrieve_with_emb({"emb_reps": q_vec, "token_id_reps": q_tok}, qids, k)
    for r, qid in enumerate(qids):
        n = int(cnt[r])
        got = {f"d{int(i)}": float(s) for i, s in zip(fid[r, :n].tolist(), fsc[r, :n].tolist())}
        ref = dict_res["emb_tok"][qid]
        assert got.keys() == ref.keys()
        for pid, v in ref.items():
            assert abs(got[pid] - v) < 1e-12
    s_arr, i_arr = hs.dense_search.retrieve_arrays(q_vec, k)
    assert hs.dense_search.arrays_to_dict(s_arr, i_arr, qids) == dict_res["emb"]
    # JSONL round trip of the sparse corpus
    hs.sparse_search.dump_jsonl(str(tmp_path / "encoded_corpus"), chunk_docs=128)
    assert len(list((tmp_path / "encoded_corpus").glob("corpus*.jsonl"))) == 4
    other = lr.ImpactSearch(vocab_size=V)
    assert other.index_from_jsonl(str(tmp_path / "encoded_corpus")) == n_docs
    assert other.retrieve_with_emb(q_tok, qids, k) == dict_res["tok"]


# ------------------------------------------------------------------------------------------------ full-size properties
def test_full_width_properties_at_scale():
    """Size-independent properties at a BASELINE-like width (d=4096) and a corpus larger than L2:
    planted documents are found, results are sorted, ids unique, scores equal an fp32 recomputation of the returned
    rows, and a sample of queries matches torch's fp32 matmul+topk on the device."""
    torch.manual_seed(11)
    Q, N, d, k = 512, 300_000, 4096, 100
    c = F.normalize(torch.randn(N, d, device="cuda"), dim=-1).bfloat16()
    q = F.normalize(torch.randn(Q, d, device="cuda"), dim=-1).bfloat16()
    planted = torch.randint(0, N, (Q,), device="cuda")
    c[planted] = q  # each query's own vector sits in the corpus: it must be rank 1 with score ~1
    s, i = lr.flatip_topk(q, c, k)
    assert bool((i[:, 0] == planted).all()) or bool(((s[:, 0] - 1).abs() < 1e-2).all())
    assert bool((s[:, :-1] >= s[:, 1:]).all())
    assert all(len(set(row)) == k for row in i[:16].tolist())
    rec = torch.einsum("qd,qkd->qk", q.float(), c[i].float())
    torch.testing.assert_close(s, rec, rtol=1e-2, atol=1e-4)
    ref = q[:32].float() @ c.float().T
    oracle.check_topk_parity(_np(s[:32]), _np(i[:32]), ref.cpu().numpy(), k, rtol=1e-2)


def test_short_rows_at_scale_refresh_passes_and_two_epilogue_sets():
    """BASELINE configs[2] regime at a size where every large-batch mechanism is on (plan checked below): 32768-document
    prefix, threshold-refresh passes, cta_group::2 pairs on the team schedule, two epilogue warp sets with their own
    candidate lists.  Properties (planted documents, order, unique ids, fp32 recomputation of the returned scores) for
    every query; full parity against an fp32 matmul of the same bf16 values for a sample of queries."""
    torch.manual_seed(13)
    Q, N, d, m, k = 2304, 1_200_000, 256, 128, 100
    c = torch.randn(N, d, device="cuda").bfloat16()
    q = torch.randn(Q, d, device="cuda").bfloat16()
    planted = torch.randperm(N, device="cuda")[:Q]
    c[planted, :m] = q[:, :m]
    cs = (1.0 / c[:, :m].float().norm(dim=1)).contiguous()
    qs = (1.0 / q[:, :m].float().norm(dim=1)).contiguous()
    for scaled in (True, False):
        if scaled:  # full-width rows scored on the first m columns with reciprocal prefix norms
            s, i = lr.flatip_topk(q, c, k, d_used=m, q_scale=qs, c_scale=cs)
            qn, cn = q[:, :m].float() * qs[:, None], None
        else:       # compact storage [N, m], already normalised
            qq = F.normalize(q[:, :m].float(), dim=-1).bfloat16()
            cc = F.normalize(c[:, :m].float(), dim=-1).bfloat16()
            s, i = lr.flatip_topk(qq, cc, k)
            qn = qq.float()
        assert bool((i[:, 0] == planted).all())
        assert bool((s[:, :-1] >= s[:, 1:]).all())
        assert all(len(set(row)) == k for row in i[:16].tolist())
        rows = (c[i][:, :, :m].float() * cs[i][:, :, None]) if scaled else cc[i].float()
        rec = torch.einsum("qd,qkd->qk", qn, rows)
        torch.testing.assert_close(s, rec, rtol=1e-3, atol=1e-5)
        full = (c[:, :m].float() * cs[:, None]) if scaled else cc.float()
        ref = qn[:24] @ full.T
        oracle.check_topk_parity(_np(s[:24]), _np(i[:24]), ref.cpu().numpy(), k, rtol=1e-3)
        del full, ref, rows, rec
    from lightretriever_b200 import _C as C
    import ctypes
    out = (ctypes.c_int64 * 16)()
    C.load().lr_flatip_plan(Q, N, k, out)
    assert out[1] == 1 and out[5] == 128  # pairs + the 32768-document prefix: the regime this test is about


def _plan_of(Q, N, k, d):
    import ctypes
    from lightretriever_b200 import _C as C
    out, rows, flags = (ctypes.c_int64 * 16)(), (ctypes.c_int64 * 64)(), (ctypes.c_int64 * 2)()
    C.load().lr_flatip_plan(Q, N, k, out)
    n = C.load().lr_flatip_plan_passes(Q, N, k, d, rows, 16, flags)
    return list(out), [tuple(rows[4 * i:4 * i + 4]) for i in range(n)]


@pytest.mark.parametrize("k", [100, 1000])
def test_headline_regime_pairs_team_schedule_prefix_full_width(k):
    """The regime that carries the headline number (bench.py: 10k queries x 8.8M x 4096): cta_group::2 pairs on the team
    schedule, one-tile progress window, warm-start prefix, full-width rows (64 k-blocks per tile) — at the smallest size
    that selects exactly that plan (asserted).  Two corpora: random, and rows SORTED by similarity to query 0 (every later
    document beats that query's running threshold: the worst case for warm-start pruning and list cuts).  Properties on
    every row (planted document first, order, unique ids, fp32 recomputation of the returned scores) and full parity
    against an fp32 matmul of the same bf16 values on 48 sampled rows incl. the adversarial one."""
    torch.manual_seed(17)
    Q, N, d = 2304, 1_100_000, 4096
    plan, passes = _plan_of(Q, N, k, d)
    assert plan[0] == 2 and plan[1] == 1, plan            # cluster of two, cta_group::2 pair
    assert len(passes) == 2 and passes[0][0] == 0 and passes[-1][3] == 1, passes   # prefix, then main on the team schedule
    assert passes[0][1] == (128 if k == 100 else 268), passes
    c = torch.empty((N, d), dtype=torch.bfloat16, device="cuda")
    for lo in range(0, N, 1 << 17):
        c[lo:lo + (1 << 17)] = F.normalize(torch.randn(min(1 << 17, N - lo), d, device="cuda"), dim=-1).bfloat16()
    q = F.normalize(torch.randn(Q, d, device="cuda"), dim=-1).bfloat16()
    planted = torch.randperm(N, device="cuda")[:Q]
    c[planted] = q
    sample = torch.cat([torch.tensor([0, 1, 127, 128, 255, 256, Q - 1], device="cuda"),
                        torch.randperm(Q, device="cuda")[:41]]).unique()

    def check(corpus, planted_at):
        s, i = lr.flatip_topk(q, corpus, k)
        assert bool((i[:, 0] == planted_at).all())
        assert bool((s[:, :-1] >= s[:, 1:]).all())
        assert bool((i.sort(dim=1).values.diff(dim=1) > 0).all())          # unique ids in every row
        for lo in range(0, Q, 256):                                        # returned scores == fp32 recomputation
            rec = torch.einsum("qd,qkd->qk", q[lo:lo + 256].float(), corpus[i[lo:lo + 256]].float())
            torch.testing.assert_close(s[lo:lo + 256], rec, rtol=1e-2, atol=1e-4)
        ref = torch.cat([q[sample].float() @ corpus[lo:lo + (1 << 18)].float().T for lo in range(0, N, 1 << 18)], dim=1)
        oracle.check_topk_parity(_np(s[sample]), _np(i[sample]), ref.cpu().numpy(), k, rtol=1e-2)

    check(c, planted)
    # adversarial order for query 0: ascending similarity (its planted twin ends up last)
    sim = torch.cat([c[lo:lo + (1 << 18)].float() @ q[0].float() for lo in range(0, N, 1 << 18)])
    order = torch.argsort(sim)
    inv = torch.empty_like(order)
    inv[order] = torch.arange(N, device="cuda")
    c2 = c[order]
    del c
    check(c2, inv[planted])


@pytest.mark.parametrize("shards,prefix_docs,d", [(4, 4096, 128), (3, 2048, 256), (2, 0, 128)])
def test_sharded_search_with_shared_warm_start_is_exact(monkeypatch, shards, prefix_docs, d):
    """lr_flatip_topk_begin / _finish: every shard scores 1/shards of the warm-start prefix, the merged prefix top-k of all
    shards seeds each shard's thresholds, and a shard keeps only documents that can still reach the GLOBAL top-k.  The
    shards are played one after the other on one device (own workspaces); the merged result must equal the unsharded
    oracle — with ties across shard boundaries, a shard that holds every winner of some queries and a shard that holds
    none (its rows come back empty).  prefix_docs 0 = single-phase plan (the seed alone is the warm start)."""
    monkeypatch.setenv("LR_FLATIP_PREFIX_DOCS", str(prefix_docs))
    lr._C.reload_env()
    from lightretriever_b200._util import Workspace
    from lightretriever_b200.search import flatip_topk_sharded, merge_keys, decode_keys
    gen = torch.Generator().manual_seed(shards * 100 + d)
    Q, N, k = 300, 61_003, 50
    q = F.normalize(torch.randn(Q, d, generator=gen), dim=-1).bfloat16()
    c = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16()
    bounds = [N * r // shards for r in range(shards + 1)]
    c[bounds[1] - 3:bounds[1] + 3] = c[9]                       # exact ties across a shard boundary
    c[bounds[1] + 100:bounds[1] + 100 + 2 * k] = q[0]           # query 0: 2k identical winners, all in shard 1
    qd, cd = q.cuda(), c.cuda()
    ws = [Workspace() for _ in range(shards)]
    pk, calls = [], []
    for r in range(shards):
        calls.append([])

        def exch(prefix_keys, r=r):
            calls[r].append(prefix_keys.clone())
            return None
        # first round: collect the prefix keys; finish(seed=None) must be a plain search of the shard
        s_r, i_r, k_r = flatip_topk_sharded(qd, cd[bounds[r]:bounds[r + 1]], k, shards, exch, id_offset=bounds[r], workspace=ws[r])
        es, ei = oracle.flatip_topk(q.float(), c[bounds[r]:bounds[r + 1]].float(), k, id_offset=bounds[r])
        assert (ei == _np(i_r)).mean() > 0.999
        pk.append(calls[r][0])
    seed = merge_keys(pk, k)
    if prefix_docs == 0:
        assert all(bool((x == 0).all()) for x in pk)            # no warm-start pass in this plan: nothing to exchange
        # play a seed from outside: the k-th best of the first 4000 documents of the whole corpus
        seed = lr.flatip_topk(qd, cd[:4000], k, return_keys=True)[2]
    ref = (q.float() @ c.float().T).numpy()
    es, ei = oracle.flatip_topk(q.float(), c.float(), k)

    def round_with(seed_keys):
        finals, n_kept = [], []
        for r in range(shards):
            s_r, i_r, k_r = flatip_topk_sharded(qd, cd[bounds[r]:bounds[r + 1]], k, shards, lambda _: seed_keys,
                                                id_offset=bounds[r], workspace=ws[r])
            finals.append(k_r)
            n_kept.append((i_r >= 0).sum(dim=1))
            assert bool(((i_r == -1) == torch.isneginf(s_r)).all())
        merged = merge_keys(finals, k)
        gs, gi = decode_keys(merged)
        oracle.check_topk_parity(_np(gs), _np(gi), ref, k, rtol=1e-2)
        assert (ei == _np(gi)).mean() > 0.999
        return merged, torch.stack(n_kept)

    merged, _ = round_with(seed)
    # The tightest valid seed is the global result itself: every shard then keeps only the global winners (and ties with
    # the k-th score), rows of shards without a winner come back empty, and the merge still equals the oracle.
    merged2, kept = round_with(merged)
    assert torch.equal(merged2, merged)
    assert int(kept.sum()) < Q * k + Q * 8 and bool((kept.sum(dim=0) >= k).all())
    assert int(kept[1, 0]) == k and int(kept[:, 0].sum()) == k      # query 0: every winner lives in shard 1
    monkeypatch.undo()
    lr._C.reload_env()


def test_faiss_flat_file_roundtrip_and_sharded_load(tmp_path):
    """Row f3: FlatIPSearch.save writes the reference's two files (<prefix>.flat.tsv + <prefix>.flat.faiss, an IndexFlatIP
    in Faiss's on-disk layout); load reads them straight into HBM — whole, or a row range (a rank's shard)."""
    gen = torch.Generator().manual_seed(8)
    corpus = F.normalize(torch.randn(700, 64, generator=gen), dim=-1).bfloat16().float()  # bf16-exact: fp32 file is lossless
    queries = F.normalize(torch.randn(4, 64, generator=gen), dim=-1)
    cids = [f"doc-{j}" for j in range(700)]
    qids = [f"q{j}" for j in range(4)]
    a = lr.FlatIPSearch(model=None)
    a.index(corpus, cids)
    want = a.retrieve_with_emb(queries, qids, 15)
    a.save(str(tmp_path), prefix="idx")
    assert (tmp_path / "idx.flat.faiss").stat().st_size == 45 + 700 * 64 * 4
    b = lr.FlatIPSearch(model=None)
    b.load(str(tmp_path), prefix="idx")
    assert b.retrieve_with_emb(queries, qids, 15) == want
    shard = lr.FlatIPIndex.load(str(tmp_path / "idx.flat.faiss"), rows=(300, 700), id_offset=300)
    s, i = shard.search_device(queries, 15)
    es, ei = oracle.flatip_topk(queries.bfloat16().float(), corpus[300:], 15, id_offset=300)
    np.testing.assert_array_equal(_np(i), ei)


def test_fusion_dict_adapters_match_reference_golden(golden_dir):
    """fuse_scores_linear / fuse_scores_rrf (dict in, dict out) are adapters over lr_fuse_topk: against the outputs of the
    reference's own functions (tests/golden/fusion.json, float64)."""
    g = json.load(open(os.path.join(golden_dir, "fusion.json")))
    lin = lr.fuse_scores_linear([g["dense"], g["sparse"]], weights=[0.7, 0.3])
    rrf = lr.fuse_scores_rrf([g["dense"], g["sparse"]])
    assert lin.keys() == g["linear"].keys() and rrf.keys() == g["rrf"].keys()
    for q in g["linear"]:
        assert lin[q].keys() == g["linear"][q].keys() and rrf[q].keys() == g["rrf"][q].keys()
        for p, v in g["linear"][q].items():
            assert abs(lin[q][p] - v) < 1e-12
        for p, v in g["rrf"][q].items():
            assert abs(rrf[q][p] - v) < 1e-12


def test_hybrid_search_chunk_loop_runs_without_host_heaps(monkeypatch):
    """HybridSearch.search over a 3-chunk corpus with two dense query kinds, ignore_identical_ids and rrf: per-chunk results
    are merged by lr_topk_merge and fused by lr_fuse_topk — no heapq call — and equal the reference flow played by the
    oracle (per-chunk top-k dicts -> _add_to_heap -> fuse)."""
    import heapq

    def boom(*a, **kw):
        raise AssertionError("host heap merge on the search path")

    gen = torch.Generator().manual_seed(31)
    n_docs, n_q, d, V, k = 330, 5, 64, 83, 12
    doc_vec = F.normalize(torch.randn(n_docs, d, generator=gen), dim=-1)
    q_den = F.normalize(torch.randn(n_q, d, generator=gen), dim=-1)
    q_emb = F.normalize(torch.randn(n_q, d, generator=gen), dim=-1)
    rng = np.random.default_rng(6)
    doc_sparse = [{str(int(t)): int(rng.integers(1, 300)) for t in rng.choice(V, 10, replace=False)} for _ in range(n_docs)]
    q_tok = [" ".join(str(int(t)) for t in rng.integers(0, V, size=5)) for _ in range(n_q)]
    corpus = {f"d{j}": {"text": "x" * (1 + (j * 7) % 11), "j": j} for j in range(n_docs)}
    queries = {(f"d{j * 3}" if j < 3 else f"q{j}"): f"query {j}" for j in range(n_q)}   # three queries ARE corpus documents
    doc_vec[0], doc_vec[3], doc_vec[6] = q_emb[0], q_emb[1], q_emb[2]                   # ... and would retrieve themselves

    class FakeModel:
        def encode_queries(self, queries, **kw):
            return {"dense_reps": q_den, "emb_reps": q_emb, "token_id_reps": q_tok}

        def encode_corpus(self, corpus, **kw):
            idx = [c["j"] for c in corpus]
            return {"dense_reps": doc_vec[idx], "sparse_reps": [doc_sparse[j] for j in idx]}

    hs = lr.HybridSearch(FakeModel(), batch_size=16, corpus_chunk_size=128, return_all_results=True, vocab_size=V,
                         score_fuse_method="rrf")
    with monkeypatch.context() as m:
        m.setattr(heapq, "heappush", boom)
        m.setattr(heapq, "heappushpop", boom)
        res = hs.search(corpus, queries, top_k=k, ignore_identical_ids=True)
    # reference flow on the oracle
    cids = sorted(corpus, key=lambda c_: len(corpus[c_]["text"]), reverse=True)
    order = [corpus[c_]["j"] for c_ in cids]
    qids = list(queries)
    cb = doc_vec.bfloat16().float()[order]
    for name, qv in (("den", q_den), ("emb", q_emb)):
        heaps = {qid: [] for qid in qids}
        for lo in range(0, n_docs, 128):
            es, ei = oracle.flatip_topk(qv.bfloat16().float(), cb[lo:lo + 128], k, id_offset=lo)
            sub = {qid: {cids[j]: float(s_) for s_, j in zip(es[r], ei[r])} for r, qid in enumerate(qids)}
            oracle.add_to_heap(sub, heaps, k, True)
        want = {qid: {pid: sc for sc, pid in heaps[qid]} for qid in qids}
        assert res[name].keys() == want.keys()
        for qid in qids:
            assert res[name][qid].keys() == want[qid].keys(), (name, qid)
            assert qid not in res[name][qid]
            np.testing.assert_allclose([res[name][qid][p] for p in want[qid]], list(want[qid].values()), rtol=1e-2, atol=1e-4)
    ts, ti = oracle.impact_topk([oracle.query_counts([int(t) for t in s_.split()]) for s_ in q_tok],
                                [{int(a): b for a, b in doc_sparse[j].items()} for j in order], k)
    tok = {qid: {cids[j]: float(s_) for s_, j in zip(ts[r], ti[r]) if j >= 0} for r, qid in enumerate(qids)}
    assert res["tok"] == {q_: v for q_, v in tok.items() if v}
    fused = oracle.fuse_rrf([res["emb"], res["tok"]])
    assert res["emb_tok"].keys() == fused.keys()
    for qid in fused:
        assert res["emb_tok"][qid].keys() == fused[qid].keys()
        for pid, v in fused[qid].items():
            assert abs(res["emb_tok"][qid][pid] - v) < 1e-12
    # the sparse searcher's own search() (anserini_search.py:218-309)
    sp = lr.ImpactSearch(FakeModel(), batch_size=16, corpus_chunk_size=100, vocab_size=V)
    assert sp.search(corpus, queries, top_k=k) == res["tok"]
    with pytest.raises(ValueError):
        sp.index(doc_sparse[:4], ["a", "b", "c", "d"])
        sp.retrieve_with_emb(q_tok, qids, 2000)   # beyond the sparse kernel's limit: an error, not a silent clamp


def test_online_searcher_graph_replay_matches_eager():
    """The captured online step (encode -> flat-IP top-k -> merge) must return what the eager calls return, for requests
    of different sizes replayed through the same graph (padding ids, empty unused bags)."""
    gen = torch.Generator().manual_seed(5)
    V, d, N, k = 3000, 256, 50_000, 20
    table = (torch.randn(V, d, generator=gen) * 0.02).bfloat16().cuda()
    corpus = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16().cuda()
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)
    srv = lr.OnlineSearcher(bag, corpus, k, batch=8, max_tokens=8 * 32, id_offset=77)
    for n_bags in (1, 5, 8):
        lens = torch.randint(1, 33, (n_bags,), generator=gen)
        ids = torch.randint(0, V - 1, (int(lens.sum()),), generator=gen).cuda()
        offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).cuda()
        s, i = srv.search(ids, offs)
        qv = bag.encode(ids, offs, normalize=True)
        es, ei = lr.flatip_topk(qv, corpus, k, id_offset=77)
        np.testing.assert_array_equal(_np(i), _np(ei))
        np.testing.assert_array_equal(_np(s), _np(es))
        ref = (qv.float().cpu() @ corpus.float().cpu().T).numpy()
        oracle.check_topk_parity(_np(s), _np(i), ref, k, rtol=1e-2, id_offset=77)
    with pytest.raises(ValueError):
        srv.search(torch.zeros(9 * 32, dtype=torch.long).cuda(), torch.zeros(9, dtype=torch.long).cuda())


@pytest.mark.parametrize("kernel", ["1", "3"])
def test_sparse_score_each_kernel_forced_is_exact(kernel):
    """The regime switch picks the row kernel (dense batches) or the flat kernel (sparse batches) per call; here each one is
    FORCED (LR_SPARSE_KERNEL=1 flat / 3 rows) over the same index: head term present in half of the documents (long runs:
    the batched full-row path), short runs, repeated query terms, a query of more than 32 terms (chunked steps), and
    weights that overflow the 16-bit accumulators (32-bit pass).  Subprocess: the knob is set in its environment."""
    import subprocess
    import sys
    code = r'''
import numpy as np, sys
sys.path.insert(0, %r)
import lightretriever_b200 as lr
from oracle import oracle
from lightretriever_b200.sparse_search import parse_queries
rng = np.random.default_rng(3)
N, V, k = 90000, 3000, 100
docs = []
for j in range(N):
    toks = rng.choice(V, size=int(rng.integers(0, 25)), replace=False)
    docs.append({str(int(t)): int(rng.integers(1, 400)) for t in toks})
for j in range(0, N, 2):
    docs[j]["5"] = int(rng.integers(1, 50))            # head term: runs of thousands of postings per step
queries = [" ".join(str(int(t)) for t in rng.integers(0, V, size=int(rng.integers(1, 33)))) for _ in range(40)]
queries += ["5 6 7", "5 5 9 9 9", " ".join(str(t) for t in range(40))]   # head term, repeated terms, > 32 terms
s = lr.ImpactSearch(vocab_size=V)
s.index(docs, [str(j) for j in range(N)])
dd = [{int(a): b for a, b in d.items()} for d in docs]
qd = [oracle.query_counts([int(t) for t in q.split()]) for q in queries]
es, ei = oracle.impact_topk(qd, dd, k)
gs, gi = s._ensure_index().search_device(*parse_queries(queries, V), k)
assert (gi.cpu().numpy() == ei).all() and (gs.cpu().numpy() == es).all()
wide = [{5: 3000, 6: 1, 7: 40000}, {int(t): int(rng.integers(1, 5000)) for t in rng.integers(0, V, size=20)}]
es, ei = oracle.impact_topk(wide, dd, k)
gs, gi = s._ensure_index().search_device(*parse_queries(wide, V), k)
assert (gi.cpu().numpy() == ei).all() and (gs.cpu().numpy() == es).all()
print("forced kernel exact")
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, LR_SPARSE_KERNEL=kernel)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "forced kernel exact" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
