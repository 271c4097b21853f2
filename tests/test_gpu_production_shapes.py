"""GPU parity at the production shapes whose plans the small-shape suite never selects: the small-batch warm start of K2
(one tile per CTA, then the main pass), single-CTA long lists (k = 1000), the unstaged list compaction (k = 2048), the
sharded begin/finish at the online shape, OnlineSearcher at the C5 shape (d = 3584, 1.1M documents), the packed K3
kernel and the fused sparse head at V = 128256, and K4 over 1.1M Zipf documents in default regime dispatch.

References are computed on the device in float64 from the same bf16 / integer inputs (exact for the integer scores of
K4).  Every shape is pinned to the plan it is meant to exercise by test_production_shapes_select_their_plans, which runs
without a GPU, and again inside each GPU test."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import lightretriever_b200 as lr
from lightretriever_b200 import _C
from oracle import oracle

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BN = 256                                  # corpus tile (documents) of K2
LIST_STAGE_ENTRIES = 768                  # umma_gemm.cuh: per-warp list staging of the default layout
STAGE_BIGLIST_CL1, STAGE_PAIR = 2304, 2816   # staging of the single-CTA BIGLIST layout and of a pair
N_C5, D_C5, K_C5 = 1_100_000, 3584, 100
PREFIX_END = 148 * BN                     # first document of the main pass in the small-batch warm-start plan
V_HEAD, D_HEAD, S_HEAD = 128256, 2048, 512
N_K4, V_K4, NNZ_K4 = 1_100_000, 128256, 64


# ------------------------------------------------------------------------------------------------ plans (host only)
def _flatip_plan(Q, N, k, d, shards=1):
    lib = _C.load()
    out, rows, flags = (ctypes.c_int64 * 16)(), (ctypes.c_int64 * 64)(), (ctypes.c_int64 * 2)()
    assert lib.lr_flatip_plan(Q, N, k, out) == 0
    n = lib.lr_flatip_plan_passes_sharded(Q, N, k, d, shards, rows, 16, flags)
    names = ["cl", "pair", "m_tiles", "n_tiles", "cap", "prefix_tiles", "prefix_splits", "prefix_units", "main_begin",
             "main_splits", "main_units", "grid", "band", "ws", "rounds", "n_clusters"]
    return dict(zip(names, list(out))), [tuple(rows[4 * i:4 * i + 4]) for i in range(n)]


def _assert_small_batch_warm_start(Q, N, k, d, shards=1):
    """One tile per CTA in the prefix (148 splits), lists raised to BN + 64, then the main pass over the rest."""
    p, passes = _flatip_plan(Q, N, k, d, shards)
    assert (p["cl"], p["pair"]) == (1, 0), p
    assert p["cap"] >= BN + 64, p
    assert len(passes) == 2 and passes[0][:3] == (0, 148, 148), passes
    assert passes[1][0] == 148 and passes[1][1] == -(-N // BN) and passes[1][2] >= 100, passes
    return p, passes


def _assert_single_cta_biglist(Q, N, k, warm):
    """cl = 1, no pair, lists longer than the default staging: launch_pass picks the BIGLIST layout (short units)."""
    p, passes = _flatip_plan(Q, N, k, D_C5)
    assert (p["cl"], p["pair"]) == (1, 0) and p["cap"] > LIST_STAGE_ENTRIES, p
    assert (passes[0][:3] == (0, 148, 148)) == warm and len(passes) == (2 if warm else 1), passes
    b, e, s, _ = passes[-1]
    assert -(-(e - b) // s) < 1000, passes                 # tiles per unit: BIGLIST on the single-CTA kernel
    return p, passes


def _assert_unstaged_k2048(Q, N, pair):
    p, passes = _flatip_plan(Q, N, 2048, D_C5)
    assert p["cap"] == 4096 and p["cap"] > (STAGE_PAIR if pair else STAGE_BIGLIST_CL1), p
    assert (p["cl"], p["pair"]) == ((2, 1) if pair else (1, 0)), p
    assert len(passes) == 2, passes                        # a prefix, then lists that overflow over and over
    return p, passes


def _k4_plan(Q, k):
    out = (ctypes.c_int64 * 16)()
    assert _C.load().lr_sparse_score_plan(Q, N_K4, k, out) == 0
    return dict(zip(["bd", "nblk", "cap", "flat", "rows", "S_flat", "S_rows", "S"], list(out)[:8]))


def _head_layout(B, seed):
    """Document lengths U{16..512} with holes, one empty document and one of exactly 512 tokens (host generator, so
    the plan test sees the same token count as the GPU test)."""
    gen = torch.Generator().manual_seed(seed)
    lens = torch.randint(16, S_HEAD + 1, (B,), generator=gen)
    lens[1] = 0
    lens[B // 2] = S_HEAD
    mask = torch.arange(S_HEAD)[None] < lens[:, None]
    holes = torch.rand(B, S_HEAD, generator=gen) > 0.1
    holes[B // 2] = True                                   # the full document stays full
    return mask & holes


def _head_plan(T):
    out = (ctypes.c_int64 * 4)()
    assert _C.load().lr_sparse_head_packed_plan(T, V_HEAD, out) == 0
    return dict(zip(["tiles", "splits", "off_edge", "ws"], list(out)))


def _assert_head_plan(mask):
    """Several splits of whole 256-token tiles, and a document that crosses the last cut (finished by the fix-up)."""
    T = int(mask.sum())
    hp = _head_plan(T)
    assert hp["tiles"] == -(-T // 256) and 2 <= hp["splits"] <= 64, (T, hp)
    cu = [0] + mask.sum(1).cumsum(0).tolist()
    last_cut = ((hp["splits"] - 1) * hp["tiles"]) // hp["splits"] * 256
    assert any(cu[b] < last_cut < cu[b + 1] for b in range(mask.shape[0])), "no document crosses the last cut"
    return hp


HEAD_CASES = [(16, 1), (64, 2)]                            # (B, seed)


def test_production_shapes_select_their_plans():
    """Every shape of the GPU tests below selects the plan it is meant to exercise (no GPU needed).  A planner change
    that moves a shape off its variant fails here instead of silently testing something else."""
    for Q in (4, 32, 128):
        _assert_small_batch_warm_start(Q, N_C5, K_C5, D_C5)
    assert _flatip_plan(1, N_C5, K_C5, D_C5)[1][0][:2] == (0, -(-N_C5 // BN))   # batch-1 searcher: single phase
    for Q in (1, 8, 128):
        _assert_single_cta_biglist(Q, N_C5, 1000, warm=Q >= 4)
        _assert_single_cta_biglist(Q, 200_000, 1000, warm=False)
    _assert_unstaged_k2048(32, N_C5, pair=False)
    _assert_unstaged_k2048(300, N_C5, pair=True)
    _assert_small_batch_warm_start(32, SHARD_DOCS, 100, 128, shards=4)         # each shard scores its own prefix
    for B, seed in HEAD_CASES:
        _assert_head_plan(_head_layout(B, seed))
    assert _k4_plan(2000, 100)["S_flat"] == 11 and _k4_plan(2000, 100)["S_rows"] == 33 and _k4_plan(2000, 100)["S"] == 33
    for Q, k in ((32, 100), (32, 1024)):
        assert (_k4_plan(Q, k)["S_flat"], _k4_plan(Q, k)["S_rows"]) == (64, 64)
    for k in (1000, 1024):
        p = _k4_plan(2000, k)
        assert p["S_flat"] < p["S"] == p["S_rows"] == 33, p
    for Q, k in ((32, 100), (32, 1024), (2000, 100), (2000, 1000)):
        p = _k4_plan(Q, k)
        assert p["flat"] == 1 and p["rows"] == 1, p      # default: the regime is chosen per batch on the device


# ------------------------------------------------------------------------------------------------ K2 helpers
def _np(t):
    return t.detach().cpu().numpy()


def _scores64(q, c, chunk=1 << 17):
    """float64 q @ c.T on the device, from the same bf16 values the kernel reads."""
    q64 = q.double()
    out = torch.empty((q.shape[0], c.shape[0]), dtype=torch.float64, device=q.device)
    for lo in range(0, c.shape[0], chunk):
        out[:, lo:lo + chunk] = q64 @ c[lo:lo + chunk].double().T
    return out


def _check_parity(s, i, ref, k, rtol=1e-2, id_offset=0):
    """oracle.check_topk_parity over the columns that decide it: per row the reference top-k and the returned ids
    (kept in ascending id order, so the tie order of the check is unchanged).  Whatever lies outside both can neither be
    missing above the tie band nor be returned."""
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


def _check_dense(s, i, ref, k, id_offset=0):
    _check_parity(s, i, ref, k, rtol=1e-2, id_offset=id_offset)   # the project's rule (BASELINE.md §4)
    _check_parity(s, i, ref, k, rtol=1e-4, id_offset=id_offset)   # ids exact outside a 100x narrower band


@pytest.fixture(scope="module")
def c5():
    """1.1M x 3584 unit rows (bf16) and 300 unit queries, with planted structure:
    query 1's best 120 documents all lie inside the warm-start prefix (first 148 tiles);
    rows PREFIX_END-3 .. PREFIX_END+2 are exact copies of query 2, straddling the prefix/main boundary (exact ties);
    the adversarial corpus holds the same rows sorted by ascending similarity to query 0."""
    torch.manual_seed(101)
    dev = "cuda"
    q = F.normalize(torch.randn(300, D_C5, device=dev), dim=-1).bfloat16()
    c = torch.empty((N_C5, D_C5), dtype=torch.bfloat16, device=dev)
    for lo in range(0, N_C5, 1 << 17):
        c[lo:lo + (1 << 17)] = F.normalize(torch.randn(min(1 << 17, N_C5 - lo), D_C5, device=dev), dim=-1).bfloat16()
    near = torch.arange(1000, 1000 + 120 * 200, 200, device=dev)          # spread over the prefix tiles
    c[near] = F.normalize(q[1].float() + 0.5 * torch.randn(120, D_C5, device=dev) / D_C5 ** 0.5, dim=-1).bfloat16()
    dups = torch.arange(PREFIX_END - 3, PREFIX_END + 3, device=dev)
    c[dups] = q[2]
    sim = torch.cat([c[lo:lo + (1 << 18)].float() @ q[0].float() for lo in range(0, N_C5, 1 << 18)])
    order = torch.argsort(sim)
    inv = torch.empty_like(order)
    inv[order] = torch.arange(N_C5, device=dev)
    data = {"q": q, "c": c, "c_adv": c[order], "inv": inv, "near": near, "dups": dups}
    del sim, order
    yield data
    data.clear()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ K2: small-batch warm start
@gpu
@pytest.mark.parametrize("Q", [4, 32, 128])
def test_flatip_small_batch_warm_start_at_c5_shape(c5, Q):
    """Prefix of one tile per CTA (148 splits, lists of BN + 64) seeds the thresholds and its top-k joins the merge of
    the 144-split main pass.  Random corpus and the adversarial order (every later document beats query 0's running
    threshold); exact ties across the prefix/main boundary come back in ascending id order; a query whose whole
    top-k lies inside the prefix."""
    _assert_small_batch_warm_start(Q, N_C5, K_C5, D_C5)
    q, k = c5["q"][:Q], K_C5
    for name in ("c", "c_adv"):
        corpus = c5[name]
        s, i = lr.flatip_topk(q, corpus, k)
        ref = _scores64(q, corpus)
        _check_dense(s, i, ref, k)
        dups = c5["dups"] if name == "c" else c5["inv"][c5["dups"]].sort().values
        assert i[2, :6].tolist() == dups.tolist()
        near = c5["near"] if name == "c" else c5["inv"][c5["near"]]
        if name == "c":
            assert bool((i[1] < PREFIX_END).all())
        assert set(i[1].tolist()) <= set(near.tolist())
        del ref


# ------------------------------------------------------------------------------------------------ K2: single-CTA long lists
@gpu
@pytest.mark.parametrize("Q", [1, 8, 128])
def test_flatip_single_cta_biglist_k1000(c5, Q):
    """k = 1000 with Q <= 128: the single-CTA kernel with the BIGLIST layout, with the warm-start prefix (N = 1.1M,
    Q >= 4) and single phase (N = 200k)."""
    q, k = c5["q"][:Q], 1000
    for N in (N_C5, 200_000):
        _assert_single_cta_biglist(Q, N, k, warm=(N == N_C5 and Q >= 4))
        corpus = c5["c"][:N]
        s, i = lr.flatip_topk(q, corpus, k)
        ref = _scores64(q, corpus)
        _check_dense(s, i, ref, k)
        if Q > 2:
            assert i[2, :6].tolist() == c5["dups"].tolist()
        del ref


# ------------------------------------------------------------------------------------------------ K2: k = 2048, unstaged compaction
@gpu
@pytest.mark.parametrize("Q", [32, 300])
def test_flatip_k2048_unstaged_compaction(c5, Q):
    """k = 2048: lists of 4096 exceed every variant's staging, so warp_compact_topk runs its radix passes and compaction
    straight from global memory.  1.1M documents overflow each list hundreds of times; in the adversarial order every
    document beats query 0's threshold, so its list is compacted after every 2048 documents."""
    _assert_unstaged_k2048(Q, N_C5, pair=Q > 128)
    q, k = c5["q"][:Q], 2048
    for name in ("c_adv", "c"):
        s, i = lr.flatip_topk(q, c5[name], k)
        ref = _scores64(q, c5[name])
        _check_dense(s, i, ref, k)
        del ref


# ------------------------------------------------------------------------------------------------ K2: sharded at the online shape
SHARD_DOCS = 310_000


@gpu
def test_flatip_sharded_begin_finish_online_shape():
    """lr_flatip_topk_begin / _finish with Q = 32 and 4 shards of 310k documents: each shard's plan is the small-batch
    warm start (its own 148-tile prefix, not 1/shards of a global one); the merged prefix top-k of all shards seeds every
    shard, and the merge of the shards must equal the unsharded reference — with ties across a shard boundary and a
    query whose 2k identical winners all live in one shard."""
    from lightretriever_b200._util import Workspace
    from lightretriever_b200.search import decode_keys, flatip_topk_sharded, merge_keys
    shards, Q, d, k = 4, 32, 128, 100
    N = shards * SHARD_DOCS
    _assert_small_batch_warm_start(Q, SHARD_DOCS, k, d, shards=shards)
    torch.manual_seed(7)
    q = F.normalize(torch.randn(Q, d, device="cuda"), dim=-1).bfloat16()
    c = F.normalize(torch.randn(N, d, device="cuda"), dim=-1).bfloat16()
    bounds = [SHARD_DOCS * r for r in range(shards + 1)]
    c[bounds[1] - 3:bounds[1] + 3] = c[9]
    c[bounds[2] + 50_000:bounds[2] + 50_000 + 2 * k] = q[0]     # query 0: every winner in shard 2, past its prefix
    c[bounds[3] - 1] = q[1]                                     # query 1: the best document is a shard's last row
    ref = _scores64(q, c)
    ws = [Workspace() for _ in range(shards)]
    prefix = []
    for r in range(shards):
        seen = []
        flatip_topk_sharded(q, c[bounds[r]:bounds[r + 1]], k, shards, lambda pk: seen.append(pk.clone()),
                            id_offset=bounds[r], workspace=ws[r])
        assert bool((seen[0][:, k - 1] != 0).all())            # a full prefix top-k on every shard
        prefix.append(seen[0])
    seed = merge_keys(prefix, k)

    def round_with(seed_keys):
        finals = []
        for r in range(shards):
            s_r, i_r, k_r = flatip_topk_sharded(q, c[bounds[r]:bounds[r + 1]], k, shards, lambda _: seed_keys,
                                                id_offset=bounds[r], workspace=ws[r])
            assert bool(((i_r == -1) == torch.isneginf(s_r)).all())
            finals.append(k_r)
        merged = merge_keys(finals, k)
        gs, gi = decode_keys(merged)
        _check_dense(gs, gi, ref, k)
        assert gi[0].tolist() == list(range(bounds[2] + 50_000, bounds[2] + 50_000 + k))
        assert int(gi[1, 0]) == bounds[3] - 1
        return merged

    merged = round_with(seed)
    assert torch.equal(round_with(merged), merged)             # the tightest valid seed changes nothing


# ------------------------------------------------------------------------------------------------ OnlineSearcher at C5
@gpu
def test_online_searcher_c5_shape_graph_replay(c5):
    """C5: bag table V = 128256 x 3584, 1.1M x 3584 corpus, k = 100; a searcher captured for batch 32 (the warm-start
    plan) serving requests of 1, 17 and 32 bags, and one captured for batch 1 (single phase).  Graph replay equals the
    eager encode + flatip_topk bit for bit, and both match the float64 reference."""
    _assert_small_batch_warm_start(32, N_C5, K_C5, D_C5)
    assert len(_flatip_plan(1, N_C5, K_C5, D_C5)[1]) == 1
    V, k = 128256, K_C5
    gen = torch.Generator(device="cuda").manual_seed(55)
    table = (torch.randn(V, D_C5, device="cuda", generator=gen) * 0.02).bfloat16()
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)
    corpus = c5["c"]
    hgen = torch.Generator().manual_seed(56)
    for batch, sizes in ((32, (1, 17, 32)), (1, (1,))):
        srv = lr.OnlineSearcher(bag, corpus, k, batch=batch, max_tokens=batch * 32, id_offset=11)
        for n_bags in sizes:
            lens = torch.randint(1, 33, (n_bags,), generator=hgen)
            ids = torch.randint(0, V - 1, (int(lens.sum()),), generator=hgen).cuda()
            offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).cuda()
            s, i = (t.clone() for t in srv.search(ids, offs))
            qv = bag.encode(ids, offs, normalize=True)
            es, ei = lr.flatip_topk(qv, corpus, k, id_offset=11)
            assert torch.equal(i, ei) and torch.equal(s, es), (batch, n_bags)
            _check_dense(s, i, _scores64(qv, corpus), k, id_offset=11)
        del srv
    del table, bag
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ K3 at V = 128256
def _head_inputs(B, seed):
    mask = _head_layout(B, seed)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.randn(B, S_HEAD, D_HEAD, device="cuda", generator=gen).bfloat16()
    W = (torch.randn(V_HEAD, D_HEAD, device="cuda", generator=gen) * 0.05).bfloat16()
    bias = torch.randn(V_HEAD, device="cuda", generator=gen) * 0.1
    return h, W, bias, mask.cuda()


def _max_linear64(h, W, bias, mask, chunk=8192):
    """float64 per document: max over valid tokens of h . W^T + b (-inf when no token is valid), chunked over V."""
    B, S, d = h.shape
    h64 = h.reshape(B * S, d).double()
    out = torch.empty((B, W.shape[0]), dtype=torch.float64, device=h.device)
    for lo in range(0, W.shape[0], chunk):
        logits = (h64 @ W[lo:lo + chunk].double().T + bias[lo:lo + chunk].double()).view(B, S, -1)
        out[:, lo:lo + chunk] = logits.masked_fill(~mask[:, :, None], -torch.inf).amax(dim=1)
        del logits
    return out


@gpu
@pytest.mark.parametrize("B,seed", HEAD_CASES)
def test_sparse_head_production_vocab(B, seed):
    """max_linear_mapping (packed default path) at V = 128256, d = 2048: ragged documents of 16..512 tokens with holes,
    an empty one and a full one; documents cross the splits' cuts, the last one included.  Against a float64 reference;
    the padded kernel is bit-identical.  Then the fused sparse head (relu, log1p, top-64, quantise) under the exact
    impact rule of oracle.check_sparse_impacts."""
    _assert_head_plan(_head_layout(B, seed))
    h, W, bias, mask = _head_inputs(B, seed)
    got = lr.max_linear_mapping(h, W, bias, mask, weight_is_vd=True)
    ref = _max_linear64(h, W, bias, mask)
    fin = torch.isfinite(ref)
    assert int((~fin.all(1)).sum()) == 1 and bool(fin[B // 2].all())
    torch.testing.assert_close(got[fin], ref[fin].float(), rtol=1e-4, atol=1e-4)
    assert bool((got[~fin] < -1e30).all())
    pad = lr.max_linear_mapping(h, W, bias, mask, weight_is_vd=True, packed=False)
    assert torch.equal(got, pad)
    del pad
    ip, tk, im = lr.sparse_head(h, W, bias, mask, True, True, 64, 8, 100.0)
    reps = torch.log1p(torch.relu(ref.masked_fill(~fin, 0.0)))
    eps = (1e-4 * ref.abs() + 1e-4).masked_fill(~fin, 1e-4)
    bad, band = oracle.check_sparse_impacts(lr.csr_to_json(ip, tk, im), reps.cpu().numpy(), eps.cpu().numpy(), 64, 8, 100.0)
    print(f"B={B}: {int(tk.numel())} impacts, {band} accepted inside a band")
    assert not bad, (len(bad), bad[:5], band)
    assert int(tk.numel()) >= 64 * (B - 1)


# ------------------------------------------------------------------------------------------------ K4 at 1.1M documents
_K4_SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
import torch
import lightretriever_b200 as lr
N, V, NNZ = %(N)d, %(V)d, %(nnz)d
dev = "cuda"
# Zipf(1.0) as in bench.py: p(rank r) ~ 1/r, inverse CDF over the harmonic numbers, ranks through a fixed permutation
w = 1.0 / torch.arange(1, V + 1, dtype=torch.float64, device=dev)
cdf = torch.cumsum(w / w.sum(), 0)
perm = torch.randperm(V, generator=torch.Generator(device=dev).manual_seed(5), device=dev)

def zipf(n, gen):
    u = torch.rand(n, generator=gen, device=dev, dtype=torch.float64)
    return perm[torch.searchsorted(cdf, u).clamp_max(V - 1)].to(torch.int32)

gen = torch.Generator(device=dev).manual_seed(2024)
tok = zipf(N * NNZ, gen).view(N, NNZ)
imp = torch.randint(1, 401, (N, NNZ), generator=gen, device=dev, dtype=torch.int32)
index = lr.ImpactIndex(V)
for lo in range(0, N, 1 << 18):
    index.add_dense_rows(tok[lo:lo + (1 << 18)], imp[lo:lo + (1 << 18)])
# reference: documents as a float64 CSR matrix [N, V] (a token repeated in a row keeps its first impact), exact for
# integer scores < 2^53; scores of a query chunk = D @ counts
key = torch.arange(N, device=dev, dtype=torch.int64)[:, None] * V + tok.long()
uk, inv = torch.unique(key.view(-1), return_inverse=True)
first = torch.full((uk.numel(),), N * NNZ, dtype=torch.int64, device=dev)
first.scatter_reduce_(0, inv, torch.arange(N * NNZ, device=dev), "amin")
row, col = uk // V, uk %% V
crow = torch.zeros(N + 1, dtype=torch.int64, device=dev)
crow[1:] = torch.cumsum(torch.bincount(row, minlength=N), 0)
D = torch.sparse_csr_tensor(crow, col, imp.view(-1)[first].double(), size=(N, V))
del tok, imp, key, uk, inv, first, row, col

def batch(Q, kind, gen, head=0):
    lens = torch.randint(1, 33, (Q,), generator=gen, device=dev)
    n = int(lens.sum())
    t = zipf(n, gen) if kind == "zipf" else torch.randint(0, V, (n,), generator=gen, device=dev, dtype=torch.int32)
    qid = torch.repeat_interleave(torch.arange(Q, device=dev), lens)
    uq, cnt = torch.unique(qid.long() * V + t.long(), return_counts=True)
    qt, qc, qo = (uq %% V).to(torch.int32), cnt.to(torch.int32), uq // V
    if head:  # the most frequent token with a large count: scores of most documents pass 65535
        hq = torch.arange(Q, device=dev)
        keep = qt != perm[0]
        qo = torch.cat([qo[keep], hq]); qt = torch.cat([qt[keep], perm[:1].repeat(Q)]); qc = torch.cat([qc[keep], torch.full((Q,), head, dtype=torch.int32, device=dev)])
        o = torch.argsort(qo * V + qt.long())
        qo, qt, qc = qo[o], qt[o], qc[o]
    qi = torch.zeros(Q + 1, dtype=torch.int32, device=dev)
    qi[1:] = torch.cumsum(torch.bincount(qo, minlength=Q), 0)
    return qi, qt.contiguous(), qc.contiguous(), qo

def reference(qi, qt, qc, qo, Q, kmax, chunk=256):
    """Top-kmax per query: documents with score > 0, score descending, ties by ascending id (exact int64 keys)."""
    out = []
    for lo in range(0, Q, chunk):
        hi = min(Q, lo + chunk)
        sel = (qo >= lo) & (qo < hi)
        dense = torch.zeros((V, hi - lo), dtype=torch.float64, device=dev)
        dense[qt[sel].long(), qo[sel] - lo] = qc[sel].double()
        sc = (D @ dense).T.round().to(torch.int64)              # [chunk, N]
        assert int(sc.max()) < (1 << 31)
        keys = torch.where(sc > 0, (sc << 32) | (0xFFFFFFFF - torch.arange(N, device=dev)), torch.zeros_like(sc))
        out.append(torch.topk(keys, kmax, dim=1).values)
        del dense, sc, keys
    keys = torch.cat(out)
    return torch.where(keys > 0, keys >> 32, 0), torch.where(keys > 0, 0xFFFFFFFF - (keys & 0xFFFFFFFF), -1)

gen = torch.Generator(device=dev).manual_seed(77)
cases = [("zipf32", 32, "zipf", 0, (100, 1024)), ("zipf2000", 2000, "zipf", 0, (100,)), ("uniform2000", 2000, "uniform", 0, (100,)),
         ("zipf2000", 2000, "zipf", 0, (1000,)), ("uniform2000", 2000, "uniform", 0, (1000,)),
         ("wide64", 64, "zipf", 200, (1024,))]
for name, Q, kind, head, ks in cases:
    qi, qt, qc, qo = batch(Q, kind, gen, head)
    es, ei = reference(qi, qt, qc, qo, Q, max(ks))
    if head:
        assert int(es.max()) > 65535
    for k in ks:
        s, i = index.search_device(qi, qt, qc, k)
        print(f"case {name} k={k}", file=sys.stderr, flush=True)
        torch.cuda.synchronize()
        hit = ei[:, :k] >= 0
        assert torch.equal(i, ei[:, :k]), name
        assert torch.equal(torch.isfinite(s), hit) and torch.equal(s[hit].to(torch.int64), es[:, :k][hit]), name
print("k4 production exact")
'''


@gpu
def test_sparse_score_zipf_1p1m_default_dispatch():
    """K4 over 1.1M documents x 64 Zipf(1.0) postings (V = 128256, impacts 1..400) in the default regime dispatch,
    bit-exact (ids and scores) against a float64 CSR product with ties by ascending id: Zipf batches of 32 and 2000
    queries (dense regime, row kernel), uniform batches of 2000 right after a Zipf batch on the same plan (sparse
    regime, flat kernel: 11 of 33 lists per query at k = 100, the rest must stay empty), a batch whose head-term counts
    push scores past 65535 (32-bit pass), k = 100 / 1000 / 1024.  LR_SPARSE_DEBUG=1 reports the regime and overflow flag
    of each call (on stderr of a subprocess)."""
    for Q, k in ((2000, 100), (2000, 1000)):
        p = _k4_plan(Q, k)
        assert p["S_flat"] < p["S_rows"] == p["S"] == 33, p
    assert _k4_plan(32, 1024)["S"] == 64
    code = _K4_SCRIPT % {"root": ROOT, "N": N_K4, "V": V_K4, "nnz": NNZ_K4}
    env = dict(os.environ, LR_SPARSE_DEBUG="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "k4 production exact" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    line = re.compile(r"S flat (\d+) rows (\d+), 16-bit overflow (\d+), batch postings (\d+) over (\d+) terms, dense from (\d+)")
    calls, pending = [], None
    for ln in r.stderr.splitlines():
        m = line.search(ln)
        if m:
            pending = [int(x) for x in m.groups()]
        elif ln.startswith("case ") and pending is not None:
            name, k = ln.split()[1], int(ln.split("k=")[1])
            s_flat, s_rows, ovf, postings, terms, thresh = pending
            calls.append((name, k, s_flat, s_rows, ovf > 0, postings >= thresh * terms))
            pending = None
    print("\n".join(map(str, calls)))
    assert [c[:2] for c in calls] == [("zipf32", 100), ("zipf32", 1024), ("zipf2000", 100), ("uniform2000", 100),
                                      ("zipf2000", 1000), ("uniform2000", 1000), ("wide64", 1024)], calls
    for name, k, s_flat, s_rows, overflow, dense in calls:
        assert dense == (not name.startswith("uniform")), (name, k)
        assert overflow == (name == "wide64"), (name, k)
        if name.endswith("2000"):
            assert s_flat < s_rows == 33, (name, k, s_flat)
