"""Document filters and deletions inside the exact top-k: the filtered entry points of K2 (lr_flatip_topk_filtered,
_begin/_finish_filtered) and K4 (lr_sparse_score_topk_filtered), lr_doc_bitmap_update, the bitmap helpers, the index
deletions and the online searchers' static bitmaps.

The reference for a filtered search is the float64 score matrix with every disallowed (query, document) pair set to -inf,
cut to its top-k and stripped of the -inf tail: K2 is held to oracle.check_topk_parity (the bf16 tie rule) over that
matrix, K4 must be bit-exact.  Every GPU shape is pinned to the plan it exercises by test_filter_shapes_select_their_plans,
which needs no GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import lightretriever_b200 as lr
from lightretriever_b200 import _C
from lightretriever_b200.filters import doc_bitmap, doc_bitmap_update
from oracle import oracle

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIST_STAGE_ENTRIES, STAGE_BIGLIST_CL1 = 768, 2304          # umma_gemm.cuh list staging (default / single-CTA BIGLIST)
NEW_SYMBOLS = ["lr_flatip_topk_filtered", "lr_flatip_topk_begin_filtered", "lr_flatip_topk_finish_filtered",
               "lr_sparse_score_topk_filtered", "lr_doc_bitmap_update"]

# name: (Q, N, k, d, shards, scales)
K2_CASES = {
    "single_cta": (8, 20001, 100, 256, 1, False),
    "cl2": (200, 30000, 100, 1024, 1, False),
    "pair": (1800, 60000, 100, 1024, 1, False),
    "biglist_k1000": (200, 30000, 1000, 1024, 1, False),
    "unstaged_k2048": (32, 30000, 2048, 256, 1, False),
    "wide_scaled": (300, 30000, 100, 128, 1, True),
    "small_batch_warm": (32, 400_000, 100, 256, 1, False),
    "prefix_refresh": (1024, 1_100_000, 100, 128, 1, False),
    "sharded4": (32, 4 * 310_000, 100, 128, 4, False),
}
K4_N, K4_V = 60_000, 5000


# ------------------------------------------------------------------------------------------------ plans (host only)
def _plan(Q, N, k, d, shards=1):
    lib = _C.load()
    out, rows, flags = (ctypes.c_int64 * 16)(), (ctypes.c_int64 * 64)(), (ctypes.c_int64 * 2)()
    assert lib.lr_flatip_plan(Q, N, k, out) == 0
    n = lib.lr_flatip_plan_passes_sharded(Q, N, k, d, shards, rows, 16, flags)
    names = ["cl", "pair", "m_tiles", "n_tiles", "cap"]
    p = dict(zip(names, list(out)[:5]))
    p["wide"] = flags[0]
    return p, [tuple(rows[4 * i:4 * i + 4]) for i in range(n)]


def _assert_plan(name):
    Q, N, k, d, shards, _ = K2_CASES[name]
    p, passes = _plan(Q, N // shards, k, d, shards)
    if name == "single_cta":
        assert (p["cl"], p["pair"], p["wide"], len(passes)) == (1, 0, 0, 1), (p, passes)
    elif name == "cl2":
        assert (p["cl"], p["pair"], p["wide"], len(passes)) == (2, 0, 0, 1), (p, passes)
    elif name == "pair":
        assert (p["cl"], p["pair"], p["wide"], p["cap"]) == (2, 1, 0, 256) and passes[-1][3] == 1, (p, passes)
    elif name == "biglist_k1000":
        assert (p["cl"], p["pair"]) == (2, 1) and p["cap"] > LIST_STAGE_ENTRIES, p
    elif name == "unstaged_k2048":
        assert (p["cl"], p["pair"]) == (1, 0) and p["cap"] > STAGE_BIGLIST_CL1, p
    elif name == "wide_scaled":
        assert (p["cl"], p["wide"]) == (2, 1), p
    elif name in ("small_batch_warm", "sharded4"):
        assert (p["cl"], p["pair"]) == (1, 0) and len(passes) == 2 and passes[0][:3] == (0, 148, 148), (p, passes)
    elif name == "prefix_refresh":
        assert passes[0][:2] == (0, 128) and len(passes) >= 3 and p["wide"] == 1, (p, passes)  # prefix + refreshes
    return p, passes


def _k4_plan(Q, k):
    out = (ctypes.c_int64 * 16)()
    assert _C.load().lr_sparse_score_plan(Q, K4_N, k, out) == 0
    return dict(zip(["bd", "nblk", "cap", "flat", "rows", "S_flat", "S_rows", "S", "w_flat16", "w_flat32", "w_rows16"],
                    list(out)[:11]))


def test_filter_shapes_select_their_plans():
    """Each GPU shape below runs the variant it is named after (no GPU needed): a planner change fails here."""
    for name in K2_CASES:
        _assert_plan(name)
    p = _k4_plan(2000, 100)
    assert p["S_rows"] > 1 and 2000 > 148 * p["w_rows16"], p    # chained units: more queries than row-kernel workers
    assert p["flat"] == 1 and p["rows"] == 1, p


# ------------------------------------------------------------------------------------------------ C ABI (no GPU)
def test_filtered_symbols_are_declared_and_bound():
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "lr_b200.h")).read(), flags=re.S)
    for name in NEW_SYMBOLS:
        assert re.search(rf"\b{name}\s*\(", text), name
        assert name in _C.PROTOTYPES, name
        assert hasattr(_C.load(), name), name


FAKE = 1 << 20      # a 256-byte aligned address: argument checks never dereference it


def _flatip_filtered(live=FAKE, allow=None, ld=1000, nf=0, qf=None, ws=None, ws_bytes=0, N=20000, off=0, k=10, Q=8):
    lib = _C.load()
    return lib.lr_flatip_topk_filtered(FAKE, 256, FAKE, 256, Q, N, 256, None, None, off, k, FAKE, FAKE, None, live, allow,
                                       ld, nf, qf, ws, ws_bytes, None)


def _sparse_filtered(live=FAKE, allow=None, ld=1000, nf=0, qf=None, ws=None, ws_bytes=0, N=20000, off=0, k=10, Q=8):
    lib = _C.load()
    return lib.lr_sparse_score_topk_filtered(FAKE, FAKE, FAKE, Q, FAKE, FAKE, FAKE, FAKE, 100, N, off, k, FAKE, FAKE, None,
                                             live, allow, ld, nf, qf, ws, ws_bytes, None)


def test_filter_argument_errors_map_to_value_error():
    lib = _C.load()
    for call in (_flatip_filtered, _sparse_filtered):
        for bad, msg in ((dict(ld=624), "ld_words"),                       # 20000 ids need 625 words
                         (dict(off=31, ld=625), "ld_words"),               # 20031 ids need 626
                         (dict(live=None, allow=FAKE, nf=0), "n_filters"),
                         (dict(live=FAKE, qf=FAKE), "q_filter")):
            rc = call(**bad)
            assert rc == _C.LR_EINVAL, (call.__name__, bad)
            with pytest.raises(ValueError, match=msg):
                _C.check(rc)
        assert call(off=31, ld=626) == _C.LR_EWORKSPACE                     # the filter is accepted: on to the workspace
    rc = lib.lr_flatip_topk_begin_filtered(FAKE, 256, FAKE, 256, 8, 20000, 256, None, None, 0, 10, 2, FAKE, FAKE, None, 10,
                                           0, None, None, 0, None)
    assert rc == _C.LR_EINVAL and "ld_words" in _C.last_error()
    rc = lib.lr_flatip_topk_finish_filtered(FAKE, 256, FAKE, 256, 8, 20000, 256, None, None, 0, 10, 2, None, FAKE, FAKE,
                                            None, None, FAKE, 625, 0, None, None, 0, None)
    assert rc == _C.LR_EINVAL and "n_filters" in _C.last_error()
    assert lib.lr_doc_bitmap_update(None, 4, FAKE, 1, 0, None) == _C.LR_EINVAL
    assert lib.lr_doc_bitmap_update(FAKE, 0, FAKE, 1, 0, None) == _C.LR_EINVAL
    assert lib.lr_doc_bitmap_update(FAKE, 4, None, 1, 0, None) == _C.LR_EINVAL
    assert lib.lr_doc_bitmap_update(FAKE, 4, FAKE, 1, 2, None) == _C.LR_EINVAL
    assert lib.lr_doc_bitmap_update(FAKE, 4, None, 0, 1, None) == _C.LR_OK   # nothing to do: no launch


def _needed(rc):
    assert rc == _C.LR_EWORKSPACE
    return int(re.search(r"(\d+) needed", _C.last_error()).group(1))


@pytest.mark.parametrize("name", list(K2_CASES))
def test_filtered_calls_need_no_extra_workspace(name):
    """The filtered entry points ask for exactly the workspace the unfiltered ones are sized with."""
    lib = _C.load()
    Q, N, k, d, shards, _ = K2_CASES[name]
    n = N // shards
    ld = (n + 31) // 32
    want = lib.lr_flatip_workspace_bytes_for(Q, n, k, d) if shards == 1 else \
        lib.lr_flatip_workspace_bytes_sharded(Q, n, k, d, shards)
    if shards == 1:
        got = _needed(lib.lr_flatip_topk_filtered(FAKE, d, FAKE, d, Q, n, d, None, None, 0, k, FAKE, FAKE, None, FAKE, FAKE,
                                                  ld, 2, FAKE, FAKE, 256, None))
    else:
        got = _needed(lib.lr_flatip_topk_begin_filtered(FAKE, d, FAKE, d, Q, n, d, None, None, 0, k, shards, FAKE, FAKE,
                                                        FAKE, ld, 2, FAKE, FAKE, 256, None))
    assert got == want
    if k <= 1024:
        sw = lib.lr_sparse_score_workspace_bytes(Q, n, k)
        assert _needed(_sparse_filtered(N=n, k=k, Q=Q, ld=ld, allow=FAKE, nf=3, qf=FAKE, ws=FAKE, ws_bytes=256)) == sw


# ------------------------------------------------------------------------------------------------ bitmaps and oracle (no GPU)
def test_doc_bitmap_bit_order_matches_little_endian_packbits():
    rng = np.random.default_rng(3)
    for n in (1, 31, 32, 33, 1000, 4099):
        ids = rng.choice(n, size=max(1, n // 3), replace=False)
        bits = np.zeros(-(-n // 32) * 32, dtype=bool)
        bits[ids] = True
        want = np.packbits(bits, bitorder="little").view("<u4").view(np.int32)
        got = doc_bitmap(n, ids, device="cpu").numpy()
        np.testing.assert_array_equal(got, want)
        allset = np.zeros_like(bits)
        allset[:n] = True
        np.testing.assert_array_equal(doc_bitmap(n, device="cpu").numpy(),
                                      np.packbits(allset, bitorder="little").view("<u4").view(np.int32))
    with pytest.raises(ValueError):
        doc_bitmap(10, [10], device="cpu")


def _bits(words: np.ndarray, n_ids: int) -> np.ndarray:
    return np.unpackbits(words.astype("<u4").view(np.uint8), bitorder="little")[:n_ids].astype(bool)


def _filtered_topk(ref: np.ndarray, allowed: np.ndarray, k: int):
    """The filtered oracle: disallowed scores -> -inf, top-k by (score desc, id asc), the -inf tail dropped."""
    m = np.where(allowed, ref, -np.inf)
    out_s = np.full((ref.shape[0], k), -np.inf)
    out_i = np.full((ref.shape[0], k), -1, dtype=np.int64)
    for r in range(ref.shape[0]):
        order = np.lexsort((np.arange(ref.shape[1]), -m[r]))[:k]
        order = order[np.isfinite(m[r, order])]
        out_s[r, :len(order)], out_i[r, :len(order)] = m[r, order], order
    return out_s, out_i


def test_filtered_oracle_matches_brute_force():
    rng = np.random.default_rng(5)
    Q, N, k = 7, 300, 20
    ref = rng.integers(0, 40, size=(Q, N)).astype(np.float64)        # many ties
    live = doc_bitmap(N, rng.choice(N, 200, replace=False), device="cpu").numpy()
    allow = np.stack([doc_bitmap(N, rng.choice(N, c, replace=False), device="cpu").numpy() for c in (150, 10)])
    q_filter = np.array([-1, 0, 1, 2, -3, 0, 1])
    allowed = np.zeros((Q, N), dtype=bool)
    for r, f in enumerate(q_filter):
        row = _bits(live, N)
        if f != -1:
            row = row & (_bits(allow[f], N) if 0 <= f < len(allow) else False)
        allowed[r] = row
    s, i = _filtered_topk(ref, allowed, k)
    for r in range(Q):
        cand = sorted(((-ref[r, j], j) for j in range(N) if allowed[r, j]))[:k]
        assert [j for _, j in cand] == [j for j in i[r] if j >= 0]
        assert [-v for v, _ in cand] == [v for v in s[r] if np.isfinite(v)]
        assert (i[r, len(cand):] == -1).all() and np.isneginf(s[r, len(cand):]).all()
    assert (i[3] == -1).all() and (i[4] == -1).all()                  # out-of-range rows allow nothing


# ------------------------------------------------------------------------------------------------ K2 on the GPU
def _scores64(q, c, chunk=1 << 17):
    q64 = q.double()
    out = torch.empty((q.shape[0], c.shape[0]), dtype=torch.float64, device=q.device)
    for lo in range(0, c.shape[0], chunk):
        out[:, lo:lo + chunk] = q64 @ c[lo:lo + chunk].double().T
    return out


def _unpack(words, n_ids):
    w = words.to(torch.int64) & 0xFFFFFFFF
    b = (w.unsqueeze(1) >> torch.arange(32, device=w.device)) & 1
    return b.reshape(-1)[:n_ids].bool()


def _allowed_rows(f, Q, N, off):
    """[Q, N] bool of what each query may return (live AND its allow row; out-of-range rows allow nothing)."""
    dev = f["live"].device if f.get("live") is not None else f["allow"].device
    out = torch.ones((Q, N), dtype=torch.bool, device=dev)
    if f.get("live") is not None:
        out &= _unpack(f["live"], off + N)[off:][None]
    if f.get("allow") is not None:
        qf = f["q_filter"].tolist()
        for r in range(Q):
            if qf[r] == -1:
                continue
            out[r] &= _unpack(f["allow"][qf[r]], off + N)[off:] if 0 <= qf[r] < f["allow"].shape[0] else False
    return out


def _filters(Q, N, k, off, gen, dev):
    n_ids = off + N
    pick = lambda n: (torch.randperm(N, generator=gen)[:n] + off).tolist()
    keep = max(1, min(N // 1000, k // 2))
    allow = torch.stack([doc_bitmap(n_ids, pick(int(0.3 * N)), dev), doc_bitmap(n_ids, pick(int(0.05 * N)), dev),
                         doc_bitmap(n_ids, pick(max(1, k // 3)), dev)]).contiguous()
    qf = torch.tensor([[-1, 0, 1, 2, 3, -7][r % 6] for r in range(Q)], dtype=torch.int32, device=dev)
    return {
        "none": {"live": doc_bitmap(n_ids, device=dev)},
        "live50": {"live": doc_bitmap(n_ids, pick(N // 2), dev)},
        "live_tiny": {"live": doc_bitmap(n_ids, pick(keep), dev)},            # fewer than k survive: (-inf, -1) tail
        "all_deleted": {"live": torch.zeros((n_ids + 31) // 32, dtype=torch.int32, device=dev)},
        "allow_rows": {"allow": allow, "q_filter": qf},                       # -1, valid rows, out-of-range rows
    }


def _check_masked(s, i, ref, allowed, k, id_offset=0, rtol=1e-2):
    """oracle.check_topk_parity against the masked reference, over the columns that decide it (the _check_parity pattern
    of test_gpu_production_shapes): per row the allowed reference top-k and the returned ids."""
    masked = ref.masked_fill(~allowed, -torch.inf)
    vals, idx = torch.topk(masked, min(k, ref.shape[1]), dim=1)
    vals, idx = vals.cpu().numpy(), idx.cpu().numpy()
    s, i = s.cpu().numpy(), i.cpu().numpy()
    for r in range(ref.shape[0]):
        got = i[r][i[r] >= 0] - id_offset
        cols = np.union1d(idx[r][np.isfinite(vals[r])], got)
        if cols.size == 0:
            assert (i[r] == -1).all() and np.isneginf(s[r]).all(), f"query {r}: results where nothing is allowed"
            continue
        row = masked[r, torch.from_numpy(cols).to(ref.device)].cpu().numpy()[None]
        assert np.isfinite(row).all(), f"query {r}: returned a document it may not return"
        loc = np.where(i[r] >= 0, np.searchsorted(cols, i[r] - id_offset), -1)
        try:
            oracle.check_topk_parity(s[r:r + 1], loc[None], row, k, rtol=rtol)
        except AssertionError as e:
            raise AssertionError(f"query {r}: {e}") from None


def _k2_inputs(name, seed):
    Q, N, k, d, shards, scaled = K2_CASES[name]
    gen = torch.Generator(device="cuda").manual_seed(seed)
    q = F.normalize(torch.randn(Q, d, device="cuda", generator=gen), dim=-1).bfloat16()
    c = F.normalize(torch.randn(N, d, device="cuda", generator=gen), dim=-1).bfloat16()
    qs = cs = None
    if scaled:
        qs = torch.rand(Q, device="cuda", generator=gen) + 0.5
        cs = torch.rand(N, device="cuda", generator=gen) + 0.5
    return q, c, qs, cs


def _ref(q, c, qs, cs):
    ref = _scores64(q, c)
    if qs is not None:
        ref *= qs.double()[:, None] * cs.double()[None]
    return ref


def _sharded(q, c, k, shards, f, off=0):
    """4 shards on one device: begin on every shard, merge of the prefix keys, finish, merge of the shard keys."""
    from lightretriever_b200._util import Workspace
    from lightretriever_b200.search import decode_keys, flatip_topk_sharded, merge_keys
    n = c.shape[0] // shards
    ws = [Workspace() for _ in range(shards)]
    prefix = []
    for r in range(shards):
        flatip_topk_sharded(q, c[r * n:(r + 1) * n], k, shards, lambda pk: prefix.append(pk.clone()),
                            id_offset=off + r * n, workspace=ws[r], **f)
    seed = merge_keys(prefix, k)
    finals = [flatip_topk_sharded(q, c[r * n:(r + 1) * n], k, shards, lambda _: seed, id_offset=off + r * n,
                                  workspace=ws[r], **f)[2] for r in range(shards)]
    return decode_keys(merge_keys(finals, k))


@gpu
@pytest.mark.parametrize("name", list(K2_CASES))
def test_flatip_filtered_plans(name):
    """Every K2 plan under five filters: an all-live bitmap (bit-identical to the unfiltered call), a random half
    deleted, all but fewer than k deleted, all deleted, and per-query allow rows mixing -1, valid and out-of-range rows."""
    _assert_plan(name)
    Q, N, k, d, shards, _ = K2_CASES[name]
    q, c, qs, cs = _k2_inputs(name, 11)
    gen = torch.Generator().manual_seed(12)
    ref = _ref(q, c, qs, cs)
    run = (lambda f: _sharded(q, c, k, shards, f)) if shards > 1 else \
        (lambda f: lr.flatip_topk(q, c, k, q_scale=qs, c_scale=cs, **f))
    base = run({})
    for fname, f in _filters(Q, N, k, 0, gen, "cuda").items():
        s, i = run(f)
        if fname == "none":
            assert torch.equal(s, base[0]) and torch.equal(i, base[1]), name
        if fname == "all_deleted":
            assert bool((i == -1).all()) and bool(torch.isneginf(s).all())
        allowed = _allowed_rows(f, Q, N, 0)
        _check_masked(s, i, ref, allowed, k)
        if fname == "live_tiny":
            assert bool((i[:, -1] == -1).all())                               # the (-inf, -1) tail appears
        del allowed
    del ref


@gpu
def test_flatip_filter_is_applied_before_thresholds():
    """Corpus sorted by similarity to query 0 (descending: the whole warm-start prefix holds its best documents; and
    ascending), with the prefix and the best 10k documents deleted.  A filter applied after the threshold would let the
    deleted documents set it and return too few or wrong ids."""
    name = "small_batch_warm"
    _assert_plan(name)
    Q, N, k, d, _, _ = K2_CASES[name]
    q, c, _, _ = _k2_inputs(name, 21)
    prefix_docs = 148 * 256
    for desc in (True, False):
        order = torch.argsort(c.float() @ q[0].float(), descending=desc)
        cs = c[order].contiguous()
        best = torch.argsort(cs.float() @ q[0].float(), descending=True)[:10_000]
        dead = torch.unique(torch.cat([torch.arange(prefix_docs, device="cuda"), best]))
        live = doc_bitmap(N, device="cuda")
        doc_bitmap_update(live, dead, False)
        s, i = lr.flatip_topk(q, cs, k, live=live)
        assert not bool(torch.isin(i, dead).any())
        allowed = torch.ones((Q, N), dtype=torch.bool, device="cuda")
        allowed[:, dead] = False
        _check_masked(s, i, _scores64(q, cs), allowed, k)


@gpu
@pytest.mark.parametrize("off", [0, 31, 1_000_003])
def test_flatip_filter_bit_offsets_and_duplicates(off):
    """id_offset 0 / 31 / 1000003 (the chunk's bits straddle two words: funnel shift), N = 20001 (not a multiple of 32
    or 256), and exact duplicates of query 3 in rows 30..33 (across a 32-document chunk boundary) with row 31 deleted."""
    name = "single_cta"
    _assert_plan(name)
    Q, N, k, d, _, _ = K2_CASES[name]
    q, c, _, _ = _k2_inputs(name, 31)
    c[30:34] = q[3]
    gen = torch.Generator().manual_seed(32)
    ref = _scores64(q, c)
    live = doc_bitmap(off + N, (torch.randperm(N, generator=gen)[:N // 2] + off).tolist() + [off + r for r in (30, 32, 33)],
                      "cuda")
    doc_bitmap_update(live, [off + 31], False)
    s, i = lr.flatip_topk(q, c, k, id_offset=off, live=live)
    assert i[3, :3].tolist() == [off + 30, off + 32, off + 33]
    _check_masked(s, i, ref, _allowed_rows({"live": live}, Q, N, off), k, id_offset=off)
    f = _filters(Q, N, k, off, gen, "cuda")["allow_rows"]
    s, i = lr.flatip_topk(q, c, k, id_offset=off, **f)
    _check_masked(s, i, ref, _allowed_rows(f, Q, N, off), k, id_offset=off)


# ------------------------------------------------------------------------------------------------ K4 on the GPU
@pytest.fixture(scope="module")
def k4():
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(40)
    nnz = 48
    # skewed tokens (a head of frequent tokens: long posting runs) and impacts 1..400
    tok = (K4_V * torch.rand(K4_N, nnz, generator=gen, device=dev) ** 3).long().clamp_max(K4_V - 1)
    imp = torch.randint(1, 401, (K4_N, nnz), generator=gen, device=dev, dtype=torch.int32)
    index = lr.ImpactIndex(K4_V)
    index.add_dense_rows(tok, imp)
    key = torch.arange(K4_N, device=dev)[:, None] * K4_V + tok
    uk, inv = torch.unique(key.view(-1), return_inverse=True)
    first = torch.full((uk.numel(),), K4_N * nnz, dtype=torch.int64, device=dev)
    first.scatter_reduce_(0, inv, torch.arange(K4_N * nnz, device=dev), "amin")
    row, col = uk // K4_V, uk % K4_V
    crow = torch.zeros(K4_N + 1, dtype=torch.int64, device=dev)
    crow[1:] = torch.cumsum(torch.bincount(row, minlength=K4_N), 0)
    D = torch.sparse_csr_tensor(crow, col, imp.view(-1)[first].double(), size=(K4_N, K4_V))
    head = int(torch.bincount(tok.view(-1), minlength=K4_V).argmax())
    yield {"index": index, "D": D, "head": head}


def _k4_batch(Q, kind, gen, head=None, long_query=True):
    dev = "cuda"
    lens = torch.randint(1, 33, (Q,), generator=gen, device=dev)
    if long_query:
        lens[1] = 45                                                    # a query of more than 32 terms
    n = int(lens.sum())
    if kind == "zipf":
        t = (K4_V * torch.rand(n, generator=gen, device=dev) ** 3).long().clamp_max(K4_V - 1)
    else:
        t = torch.randint(0, K4_V, (n,), generator=gen, device=dev)
    qid = torch.repeat_interleave(torch.arange(Q, device=dev), lens)
    uq, cnt = torch.unique(qid * K4_V + t, return_counts=True)
    qt, qc, qo = (uq % K4_V).to(torch.int32), cnt.to(torch.int32), uq // K4_V
    if head is not None:                                               # scores past 65535: the 32-bit pass runs
        hit = qt == head
        qc[hit] = 300
    qi = torch.zeros(Q + 1, dtype=torch.int32, device=dev)
    qi[1:] = torch.cumsum(torch.bincount(qo, minlength=Q), 0)
    return qi, qt.contiguous(), qc.contiguous(), qo


def _k4_expected(D, qt, qc, qo, Q, allowed, k):
    dense = torch.zeros((K4_V, Q), dtype=torch.float64, device="cuda")
    dense[qt.long(), qo] = qc.double()
    sc = (D @ dense).T.round().to(torch.int64)
    ids = torch.arange(K4_N, device="cuda")
    keys = torch.where((sc > 0) & allowed, (sc << 32) | (0xFFFFFFFF - ids), torch.zeros_like(sc))
    top = torch.topk(keys, k, dim=1).values
    return torch.where(top > 0, top >> 32, 0), torch.where(top > 0, 0xFFFFFFFF - (top & 0xFFFFFFFF), -1), int(sc.max())


@gpu
@pytest.mark.parametrize("kernel", ["1", "3", "0"])
def test_sparse_filtered_bit_exact(k4, kernel, monkeypatch):
    """K4 with each forced kernel (1 = flat, 3 = rows) and the default regime dispatch, Zipf and uniform query tokens,
    2000 queries (more than the row kernel's workers: chained units), a query of 45 terms, a batch whose head-term
    counts push scores past 65535, under deletions and per-query allow rows: bit-exact against the masked float64 CSR
    product, ties by ascending id."""
    monkeypatch.setenv("LR_SPARSE_KERNEL", kernel)
    _C.reload_env()
    try:
        gen = torch.Generator(device="cuda").manual_seed(41 + int(kernel))
        hgen = torch.Generator().manual_seed(42)
        index, k, off = k4["index"], 100, 0
        flts = _filters(2000, K4_N, k, off, hgen, "cuda")
        for Q, kind, head in ((2000, "zipf", None), (2000, "uniform", None), (64, "zipf", k4["head"])):
            qi, qt, qc, qo = _k4_batch(Q, kind, gen, head)
            for fname in ("none", "live50", "live_tiny", "allow_rows"):
                f = dict(flts[fname])
                if "q_filter" in f:
                    f["q_filter"] = f["q_filter"][:Q].contiguous()
                allowed = _allowed_rows(f, Q, K4_N, off)
                es, ei, smax = _k4_expected(k4["D"], qt, qc, qo, Q, allowed, k)
                if head is not None:
                    assert smax > 65535
                s, i = index.search_device(qi, qt, qc, k, **f)
                hit = ei >= 0
                assert torch.equal(i, ei), (kernel, kind, fname)
                assert torch.equal(torch.isfinite(s), hit) and torch.equal(s[hit].to(torch.int64), es[hit]), (kernel, fname)
    finally:
        monkeypatch.undo()
        _C.reload_env()


# ------------------------------------------------------------------------------------------------ indexes (GPU)
@gpu
def test_index_delete_restore():
    """FlatIPIndex / ImpactIndex delete and restore in the result id space; n_live; add extends the live rows; save
    refuses an index with deletions."""
    torch.manual_seed(50)
    d, N = 128, 5000
    emb = F.normalize(torch.randn(N, d), dim=-1)
    idx = lr.FlatIPIndex.build([1000 + 7 * j for j in range(N)], emb, lr.FlatIPIndex(d))
    q = emb[:4].cuda()
    s0, i0 = idx.search(q, 5)
    assert (i0[:, 0] == 1000 + 7 * np.arange(4)).all()
    idx.delete(i0[:, 0])
    assert idx.n_live == N - 4
    s1, i1 = idx.search(q, 5)
    assert not np.isin(i1, i0[:, 0]).any() and (i1[:, :4] == i0[:, 1:]).all()
    with pytest.raises(ValueError):
        idx.delete([3])                                                   # not a passage id of this index
    with pytest.raises(ValueError):
        idx.save("/nonexistent/never-written.faiss")
    idx.restore(i0[:, 0])
    assert idx.n_live == N
    s2, i2 = idx.search(q, 5)
    assert (i2 == i0).all() and (s2 == s0).all()
    sp = lr.ImpactIndex(100, id_offset=10)
    sp.add_csr(np.array([0, 1, 2, 3]), np.array([5, 5, 5]), np.array([3, 2, 1]))
    qi, qt, qc = np.array([0, 1]), np.array([5]), np.array([1])
    sp.delete([10])
    sp.add_csr(np.array([0, 1]), np.array([5]), np.array([9]))
    assert sp.n_live == 3
    s, i = sp.search_device(qi, qt, qc, 4)
    assert i.tolist() == [[13, 11, 12, -1]]


# ------------------------------------------------------------------------------------------------ online (GPU)
def _request(n, V, gen):
    lens = torch.randint(1, 17, (n,), generator=gen)
    ids = torch.randint(0, V - 1, (int(lens.sum()),), generator=gen).cuda()
    offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).cuda()
    return ids, offs


@gpu
def test_online_searchers_delete_restore_and_filter_rows_without_recapture():
    """OnlineSearcher and OnlineHybridSearcher captured at batch 32: deleting every query's top-1 changes the next replay
    to the eager filtered result bit for bit, restore brings the original back, per-request filter rows change results
    between two replays of the same graph, and the graph is never recaptured."""
    torch.manual_seed(60)
    V, d, N, k, B = 5000, 256, 50_000, 10, 32
    gen = torch.Generator().manual_seed(61)
    table = (torch.randn(V, d, generator=gen) * 0.02).bfloat16().cuda()
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)
    corpus = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16().cuda()
    filters = torch.stack([doc_bitmap(N, torch.randperm(N, generator=gen)[:N // 10], "cuda"),
                           doc_bitmap(N, torch.randperm(N, generator=gen)[:N // 100], "cuda")]).contiguous()
    sp = lr.ImpactIndex(V)
    sp.add_dense_rows(torch.randint(0, V, (N, 24), generator=gen).cuda(), torch.randint(1, 100, (N, 24), generator=gen).cuda())
    ids, offs = _request(B, V, gen)
    qv = bag.encode(ids, offs, normalize=True)
    rows = torch.tensor([r % 3 - 1 for r in range(B)], dtype=torch.int32)

    srv = lr.OnlineSearcher(bag, corpus, k, batch=B, max_tokens=B * 16, filters=filters)
    g0 = srv._graph
    s0, i0 = (t.clone() for t in srv.search(ids, offs))
    top1 = torch.unique(i0[:, 0])
    srv.delete(top1)
    s1, i1 = (t.clone() for t in srv.search(ids, offs))
    live = doc_bitmap(N, device="cuda")
    doc_bitmap_update(live, top1, False)
    es, ei = lr.flatip_topk(qv, corpus, k, live=live)
    assert not bool(torch.isin(i1, top1).any()) and torch.equal(i1, ei) and torch.equal(s1, es)
    srv.restore(top1)
    s2, i2 = (t.clone() for t in srv.search(ids, offs))
    assert torch.equal(i2, i0) and torch.equal(s2, s0)
    s3, i3 = (t.clone() for t in srv.search(ids, offs, filter_rows=rows))
    es, ei = lr.flatip_topk(qv, corpus, k, live=doc_bitmap(N, device="cuda"), allow=filters, q_filter=rows.cuda())
    assert not torch.equal(i3, i0) and torch.equal(i3, ei) and torch.equal(s3, es)
    assert srv._graph is g0
    del srv

    hyb = lr.OnlineHybridSearcher(bag, corpus, sp, k, batch=B, max_tokens=B * 16, filters=filters)
    g0 = hyb._graph
    (ds0, di0), (ss0, si0), (fi0, fs0, _) = [tuple(t.clone() for t in r) for r in hyb.search(ids, offs)]
    dead = torch.unique(torch.cat([di0[:, 0], si0[:, 0][si0[:, 0] >= 0]]))
    hyb.delete(dead)
    (ds1, di1), (ss1, si1), (fi1, fs1, _) = [tuple(t.clone() for t in r) for r in hyb.search(ids, offs)]
    live = doc_bitmap(N, device="cuda")
    doc_bitmap_update(live, dead, False)
    es, ei = lr.flatip_topk(qv, corpus, k, live=live)
    q_csr = lr.query_token_counts(ids, offs, V)
    ess, esi = sp.search_device(*q_csr, k, live=live)
    efi, efs, _ = lr.fuse_topk_device(es, ei, ess, esi, method="linear", weights=(0.7, 0.3))
    assert torch.equal(di1, ei) and torch.equal(ds1, es) and torch.equal(si1, esi) and torch.equal(ss1, ess)
    assert torch.equal(fi1, efi) and torch.equal(fs1, efs)
    assert not bool(torch.isin(fi1, dead).any())
    hyb.restore(dead)
    (ds2, di2), (ss2, si2), (fi2, fs2, _) = [tuple(t.clone() for t in r) for r in hyb.search(ids, offs)]
    assert torch.equal(di2, di0) and torch.equal(si2, si0) and torch.equal(fi2, fi0) and torch.equal(fs2, fs0)
    (_, di3), (_, si3), _ = [tuple(t.clone() for t in r) for r in hyb.search(ids, offs, filter_rows=rows)]
    assert not torch.equal(di3, di0)
    allowed = _allowed_rows({"live": doc_bitmap(N, device="cuda"), "allow": filters, "q_filter": rows.cuda()}, B, N, 0)
    assert bool(allowed.gather(1, di3.clamp(min=0))[di3 >= 0].all()) and bool(allowed.gather(1, si3.clamp(min=0))[si3 >= 0].all())
    assert hyb._graph is g0
