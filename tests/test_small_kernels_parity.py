"""Float64 parity of the small kernels every request and every indexed document passes through: the query encoder (K1),
the last-token head (K1b), the top-p filter, the sparsifier and the score fusion, at the shapes production runs and at
the limits of the C ABI.

Each reference is a plain float64 (or integer) restatement computed from the same bf16 / f32 inputs the kernel reads;
the large ones are built on the device in torch.  Bars:
  * K1 f32 output: |got - ref| <= 2e-6 |ref| + len * 2^-24 * max|ref row| (fp32 accumulation of len rows in token
    order, then one divide and the normalisation).  K1b f32 output: bit-equal to the gathered row without normalize,
    within 1e-6 relative of float64 F.normalize with it.
  * bf16 output: the float64 reference rounded to bf16, or its neighbour only where the reference lies within the f32
    error bar of a bf16 rounding midpoint (every bf16 value between round(ref - err) and round(ref + err)).
  * top-p: an entry may differ only where its float64 cumulative probability lies within 1e-6 of the bound; kept values
    are bit-identical to the input.
  * sparsifier and fusion: bit-exact.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import lightretriever_b200 as lr
from lightretriever_b200 import _C
from oracle import oracle

gpu = pytest.mark.gpu

U32 = 2.0 ** -24  # unit roundoff of float32


# ------------------------------------------------------------------------------------------------ shared checks
def _round_bf16(x64: torch.Tensor) -> torch.Tensor:
    """float64 -> nearest bf16 (ties to even) in one rounding, returned as float32 (exact).  torch's own conversion goes
    through float32 first, which can round twice."""
    bits = x64.contiguous().view(torch.int64)
    lsb = (bits >> 45) & 1
    bits = (bits + ((1 << 44) - 1) + lsb) & ~((1 << 45) - 1)
    return bits.view(torch.float64).float()


def _check_out(got: torch.Tensor, ref: torch.Tensor, err: torch.Tensor, what: str):
    """got (f32 or bf16) against the float64 reference with absolute error bar err (per element) of the f32 result."""
    g = got.double()
    if got.dtype == torch.float32:
        bad = (g - ref).abs() > err
    else:
        lo, hi = _round_bf16(ref - err).double(), _round_bf16(ref + err).double()
        bad = (g < lo) | (g > hi)
    bad |= torch.isnan(g)
    if bad.any():
        r, c = (int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} entries off, first at [{r}, {c}]: got {float(g[r, c])!r}, "
                             f"ref {float(ref[r, c])!r}, bar {float(err[r, c])!r}")


# ------------------------------------------------------------------------------------------------ K1
BAG_LENS = (0, 1, 31, 32, 33, 64, 1023, 1024, 1025, 4096)  # the warp kernel's 32-token stage, the 1024-id cache


def _bags(V: int, pad: int, seed: int):
    """Bags of BAG_LENS tokens plus padding-only bags (short and uncached), a bag of one repeated id, short random bags,
    and a last bag of 1025 tokens that runs to the end of ids.  Every 7th id of a bag is the padding id; the 4096-token
    bag holds a run of duplicates."""
    gen = torch.Generator().manual_seed(seed)
    lens = list(BAG_LENS) + [40, 1500, 9] + torch.randint(0, 41, (20,), generator=gen).tolist() + [1025]
    lens_t = torch.tensor(lens)
    offsets = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens_t[:-1]]), 0)
    ids = torch.randint(0, V, (int(lens_t.sum()),), generator=gen)
    for o, n in zip(offsets.tolist(), lens):
        ids[o + 3:o + n:7] = pad
    o = offsets.tolist()
    ids[o[10]:o[10] + 40] = pad                    # padding-only, warp and cached block paths
    ids[o[11]:o[11] + 1500] = pad                  # padding-only, uncached block path
    ids[o[12]:o[12] + 9] = ids[o[12]]              # one id, nine times
    big = o[BAG_LENS.index(4096)]
    ids[big + 100:big + 300] = ids[big + 99]       # duplicates inside the longest bag
    return ids, offsets, lens_t


def _embbag_mean64(table, ids, offsets, pad, out_dim):
    """float64 sum of the first out_dim columns over the non-padding ids of each bag / their count (0 for a bag without
    one); ids outside [0, V) are left out (their rows are expected to be NaN)."""
    dev = table.device
    ids, offsets = ids.to(dev), offsets.to(dev)
    V = table.shape[0]
    valid = (ids != pad) & (ids >= 0) & (ids < V)
    seg = torch.searchsorted(offsets, torch.arange(ids.numel(), device=dev), right=True) - 1
    rows = table[ids.clamp(0, V - 1), :out_dim].double() * valid[:, None]
    sums = torch.zeros((offsets.numel(), out_dim), dtype=torch.float64, device=dev).index_add_(0, seg, rows)
    cnt = torch.zeros(offsets.numel(), dtype=torch.float64, device=dev).index_add_(0, seg, valid.double())
    return sums / cnt.clamp(min=1)[:, None]


def _embbag_ref(mean64, out_dim, normalize, lens):
    ref = mean64[:, :out_dim]
    if normalize:
        ref = F.normalize(ref, p=2, dim=-1, eps=1e-12)
    err = 2e-6 * ref.abs() + (lens.to(ref.device).double() * U32 * ref.abs().amax(dim=1))[:, None]
    return ref, err


def _check_embbag(bag, ids, offsets, lens, mean64, widths, label):
    for out_dim in widths:
        for normalize in (False, True):
            ref, err = _embbag_ref(mean64, out_dim, normalize, lens)
            for out_dtype in (torch.float32, torch.bfloat16):
                got = bag.encode(ids, offsets, shrink_dim=out_dim, normalize=normalize, out_dtype=out_dtype)
                _check_out(got, ref, err, f"{label} out_dim={out_dim} normalize={normalize} out={out_dtype}")


# the bench tables: c5b32 (V = 152064, d = 3584) and c2 (V = 128256, d = 4096)
BENCH_TABLES = {"c5b32": (152064, 3584), "c2": (128256, 4096)}


@pytest.fixture(scope="module")
def bench_tables():
    out = {}
    for name, (V, d) in BENCH_TABLES.items():
        g = torch.Generator(device="cuda").manual_seed(V)
        out[name, torch.bfloat16] = (torch.randn(V, d, generator=g, device="cuda") * 0.02).bfloat16()
        out[name, torch.float32] = torch.randn(16384, d, generator=g, device="cuda") * 0.02  # f32: a smaller vocabulary
    yield out
    out.clear()
    torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("table_dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("cfg", list(BENCH_TABLES))
def test_embbag_bench_tables_vs_float64(bench_tables, cfg, table_dtype):
    """Every bag length across the warp kernel's stage and the block kernel's id cache, at widths that bracket the
    warp / block switch (256 bf16 / 128 f32 columns) up to the full d, normalised and not, into f32 and bf16."""
    table = bench_tables[cfg, table_dtype]
    V, d = table.shape
    pad = V - 3
    ids, offsets, lens = _bags(V, pad, seed=d)
    mean64 = _embbag_mean64(table, ids, offsets, pad, d)
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=pad)
    _check_embbag(bag, ids.cuda(), offsets.cuda(), lens, mean64, (8, 128, 136, 256, 264, d), f"{cfg} {table_dtype}")


@gpu
@pytest.mark.parametrize("table_dtype", [torch.bfloat16, torch.float32])
def test_embbag_widest_out_dim(table_dtype):
    """out_dim up to the 12288 the ABI accepts: the block kernel's row buffer is then more dynamic shared memory than a
    launch gets without opting in."""
    V, d, pad = 64, 12288, 5
    g = torch.Generator(device="cuda").manual_seed(12288)
    table = (torch.randn(V, d, generator=g, device="cuda") * 0.02).to(table_dtype)
    ids, offsets, lens = _bags(V, pad, seed=7)
    mean64 = _embbag_mean64(table, ids, offsets, pad, d)
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=pad)
    _check_embbag(bag, ids.cuda(), offsets.cuda(), lens, mean64, (10232, 10240, 12288), f"d=12288 {table_dtype}")


@gpu
@pytest.mark.parametrize("out_dim", [128, 3584])
def test_embbag_bad_ids_poison_only_their_rows(bench_tables, out_dim):
    """One out-of-range id in a 2000-token bag (uncached on the block kernel) and one negative id in a 20-token bag:
    check_ids=True raises IndexError; check_ids=False leaves those two rows all NaN and every other row meets the bar."""
    table = bench_tables["c5b32", torch.bfloat16]
    V, d = table.shape
    pad = V - 3
    gen = torch.Generator().manual_seed(11)
    lens = torch.tensor([5, 2000, 33, 20, 1025, 0, 7])
    offsets = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
    ids = torch.randint(0, V, (int(lens.sum()),), generator=gen)
    ids[::5] = pad
    ids[int(offsets[1]) + 1234] = V + 7
    ids[int(offsets[3]) + 11] = -3
    bad = torch.tensor([False, True, False, True, False, False, False])
    ids_d, off_d = ids.cuda(), offsets.cuda()
    with pytest.raises(IndexError):
        lr.B200EmbeddingBag.from_pretrained(table, padding_idx=pad).encode(ids_d, off_d, shrink_dim=out_dim)
    mean64 = _embbag_mean64(table, ids, offsets, pad, out_dim)
    for normalize in (False, True):
        ref, err = _embbag_ref(mean64, out_dim, normalize, lens)
        for out_dtype in (torch.float32, torch.bfloat16):
            bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=pad)
            got = bag.encode(ids_d, off_d, shrink_dim=out_dim, normalize=normalize, out_dtype=out_dtype, check_ids=False)
            assert torch.isnan(got[bad.cuda()]).all()
            _check_out(got[~bad.cuda()], ref[~bad.cuda()], err[~bad.cuda()], f"bad ids {out_dim} {normalize} {out_dtype}")


# ------------------------------------------------------------------------------------------------ K1b
def _masks(B: int, S: int, seed: int):
    """name -> int64 [B, S] attention mask: right padding with ragged lengths; left padding (every last column valid,
    so row S - 1 is taken for all rows); a mixed batch that is not left-padded, with holes and one all-zero row (index
    -1 wraps to S - 1, as torch indexing does)."""
    gen = torch.Generator().manual_seed(seed)
    n = torch.randint(1, S + 1, (B,), generator=gen)
    n[0], n[-1] = 1, S
    pos = torch.arange(S)[None, :]
    right = (pos < n[:, None]).long()
    left = (pos >= S - n[:, None]).long()
    mixed = right.clone()
    mixed[1::3] = left[1::3]
    mixed[2::5] = (torch.rand(B, S, generator=gen) < 0.5).long()[2::5]
    mixed[0, -1] = 0
    mixed[B // 2] = 0
    return {"right": right, "left": left, "mixed": mixed}


@gpu
@pytest.mark.parametrize("hidden_dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("B,S,d,widths", [(257, 512, 3584, (8, 1024, 3584)), (257, 512, 4096, (8, 1024, 4096)),
                                          (5, 16, 12288, (12288,))])
def test_lasttoken_head_vs_float64(B, S, d, widths, hidden_dtype):
    g = torch.Generator(device="cuda").manual_seed(d)
    h = torch.randn(B, S, d, generator=g, device="cuda").to(hidden_dtype)
    for name, mask in _masks(B, S, seed=d).items():
        rows = oracle.lasttoken_head(h, mask).double()  # the gathered rows (torch index semantics)
        assert name != "mixed" or bool(mask[:, -1].sum() != B)
        for mdtype in (torch.int64, torch.int32, torch.bool):
            m = mask.to(mdtype).cuda()
            for out_dim in widths:
                for normalize in (False, True):
                    ref = rows[:, :out_dim]
                    if normalize:
                        ref = F.normalize(ref, p=2, dim=-1, eps=1e-12)
                    err = 1e-6 * ref.abs() if normalize else torch.zeros_like(ref)
                    for out_dtype in (torch.float32, torch.bfloat16):
                        got = lr.lasttoken_head(h, m, out_dim, normalize, out_dtype=out_dtype)
                        _check_out(got, ref, err, f"{name} mask={mdtype} out_dim={out_dim} norm={normalize} {out_dtype}")


# ------------------------------------------------------------------------------------------------ top-p
def _top_p_ref64(x: torch.Tensor, top_p: float, min_keep: int):
    """The reference rule step by step in float64: stable ascending sort, softmax, cumulative sum, remove where
    cum <= 1 - float32(top_p), then unremove remove[..., -min_keep:] with Python slice semantics (min_keep = 0 selects
    every column, so nothing is removed; min_keep > V likewise).  Returns (expected f32 output, float64 cumulative
    probability of every entry in the original indexing)."""
    srt, idx = torch.sort(x.double(), dim=-1, stable=True)
    cum = torch.softmax(srt, dim=-1).cumsum(dim=-1)
    remove = cum <= 1.0 - float(np.float32(top_p))
    remove[..., -min_keep:] = False
    remove = torch.zeros_like(remove).scatter(-1, idx, remove)
    return torch.where(remove, torch.zeros_like(x), x), torch.empty_like(cum).scatter(-1, idx, cum)


def _k3_rows(V: int = 128256, n: int = 64, seed: int = 0) -> torch.Tensor:
    """Rows shaped like K3 output, log1p(relu(N(mu, sigma))) with >= 90 % exact zeros (some of them -0.0), followed by
    an all-zero row, a peaked row (the min_keep cap binds), and two rows whose bounds fall inside tie groups of equal
    non-zero values."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    mu = torch.linspace(-3.0, -2.0, n, device="cuda")[:, None]
    sigma = torch.linspace(1.0, 1.5, n, device="cuda")[:, None]
    x = torch.log1p(torch.relu(torch.randn(n, V, generator=g, device="cuda") * sigma + mu))
    assert ((x == 0).float().mean(dim=1) >= 0.9).all()
    flip = (x[:16] == 0) & (torch.rand(16, V, generator=g, device="cuda") < 0.5)
    x[:16] = torch.where(flip, torch.full_like(x[:16], -0.0), x[:16])
    extra = torch.zeros(4, V, device="cuda")
    perm = lambda: torch.randperm(V, generator=g, device="cuda")  # noqa: E731
    extra[1, perm()[:20]] = torch.linspace(12.0, 14.0, 20, device="cuda")
    extra[2, perm()[:8000]] = 1.0
    extra[3, perm()[:64000]] = 0.7
    extra[1:, ::3] = torch.where(extra[1:, ::3] == 0, torch.full_like(extra[1:, ::3], -0.0), extra[1:, ::3])
    return torch.cat([x, extra])


@pytest.fixture(scope="module")
def k3_rows():
    return _k3_rows()


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int32)


@gpu
@pytest.mark.parametrize("top_p", [0.01, 0.1, 0.5, 0.9, 0.99])
def test_top_p_filter_vs_float64_at_v128256(k3_rows, top_p):
    V = k3_rows.shape[1]
    bound = 1.0 - float(np.float32(top_p))
    singles = torch.tensor([[0.0], [0.5], [-0.0]], device="cuda")  # V = 1
    for min_keep in (0, 1, 8, 40, V + 5):
        for x in (k3_rows, singles):
            exp, cum = _top_p_ref64(x, top_p, min_keep)
            got = lr.top_p_sampling(x, top_p, min_tokens_to_keep=min_keep)
            assert got.data_ptr() != x.data_ptr()
            diff = _bits(got) != _bits(exp)
            band = (cum - bound).abs() <= 1e-6
            assert not (diff & ~band).any(), (min_keep, x.shape, int((diff & ~band).sum()),
                                              (diff & ~band).nonzero()[:5].tolist())
            assert ((_bits(got) == _bits(x)) | (got == 0)).all()
            per_row = (diff & band).sum(dim=1)
            print(f"top_p={top_p} min_keep={min_keep} V={x.shape[1]}: {int(per_row.sum())} entries accepted in the band")
            assert int(per_row.max()) < 2


def test_top_p_float64_reference_matches_oracle_restatement(golden_dir):
    """The float64 rule above against oracle.top_p_sampling, the restatement pinned to the imported reference by
    tests/golden/top_p.npz: identical outside the band of the oracle's float32 cumulative sum.  min_keep = 0 comes from
    the oracle's restatement of the reference line remove[..., -min_tokens_to_keep:] = False, whose slice -0: selects
    every column: nothing is removed; the same holds for min_keep > V."""
    g = np.load(f"{golden_dir}/top_p.npz")
    reps = torch.from_numpy(g["reps"])
    V = reps.shape[1]
    cases = [(float(k.split("_")[0][1:]), int(k.split("_k")[1])) for k in g.files if k != "reps"]
    cases += [(0.3, 0), (0.01, 0), (0.9, 0), (0.3, V + 5)]
    for tp, mk in cases:
        if not 0 < tp < 1:
            continue
        exp, cum = _top_p_ref64(reps, tp, mk)
        ref, _ = oracle.top_p_sampling(reps.clone(), tp, min_tokens_to_keep=mk)
        diff = _bits(exp) != _bits(ref)
        band = (cum - (1.0 - float(np.float32(tp)))).abs() <= 2e-6
        assert not (diff & ~band).any(), (tp, mk)
        if mk == 0 or mk > V:
            assert torch.equal(_bits(exp), _bits(reps)) and torch.equal(_bits(ref), _bits(reps))
    assert int((oracle.top_p_sampling(reps.clone(), 0.3, min_tokens_to_keep=1)[0] == 0).sum()) > int((reps == 0).sum())


def test_top_p_rejects_negative_min_keep():
    """A negative min_tokens_to_keep would make the reference's slice keep all but the first few sorted entries; it is
    refused by the Python call and by the C entry point (before any device work)."""
    with pytest.raises(ValueError):
        lr.top_p_sampling(torch.zeros(2, 8), 0.5, min_tokens_to_keep=-1)
    buf = (ctypes.c_float * 8)()
    assert _C.load().lr_top_p_filter(ctypes.addressof(buf), 1, 8, 0.5, -1, None) == _C.LR_EINVAL
    assert "min_keep" in _C.last_error()


# ------------------------------------------------------------------------------------------------ sparsifier
def _with_kth_ties(x: torch.Tensor) -> torch.Tensor:
    """Rows 20..27: 30 entries at 3.0 and 100 at 2.5, so the 64-th largest value is shared by 100 entries."""
    x = x.clone()
    g = torch.Generator(device="cuda").manual_seed(5)
    for r in range(20, 28):
        p = torch.randperm(x.shape[1], generator=g, device="cuda")
        x[r, p[:30]] = 3.0
        x[r, p[30:130]] = 2.5
    return x


@gpu
@pytest.mark.parametrize("top_k", [0, 64, 128256])
@pytest.mark.parametrize("after_top_p", [False, True])
def test_sparsify_quantize_bit_exact_at_v128256(k3_rows, top_k, after_top_p):
    x = _with_kth_ties(k3_rows)
    if after_top_p:
        x = lr.top_p_sampling(x, 0.5, min_tokens_to_keep=8)
    exp = oracle.quantize_reps(oracle.top_k_sampling(x, top_k, min_tokens_to_keep=8).cpu(), 100.0)
    indptr, tok, imp = lr.sparsify_quantize(x, top_k=top_k, min_tokens_to_keep=8, quantization_factor=100.0)
    assert lr.csr_to_json(indptr, tok, imp) == exp


@gpu
def test_sparsify_quantize_retries_when_cap_is_too_small(k3_rows):
    x = _with_kth_ties(k3_rows)
    for top_k in (0, 64):
        full = lr.sparsify_quantize(x, top_k=top_k, min_tokens_to_keep=8)
        nnz = int(full[0][-1])
        assert nnz > 1000
        for cap in (1, nnz // 3, nnz - 1):
            small = lr.sparsify_quantize(x, top_k=top_k, min_tokens_to_keep=8, cap=cap)
            for a, b in zip(small, full):
                assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ fusion
def _fusion_inputs(Q: int, k0: int, k1: int, f64: bool, seed: int):
    """Per-system (scores, ids) [Q, k] sorted by score descending, -1 / -inf padded.  Query 0: system 0 all padding;
    1: system 1 all padding; 2: both; 3: all scores equal within each system; 4: every document of the shorter list
    also in the longer one; 5: no document shared; the rest random, with padding tails and tied scores."""
    rng = np.random.default_rng(seed)
    sdt = np.float64 if f64 else np.float32
    s = [np.empty((Q, k), sdt) for k in (k0, k1)]
    i = [np.empty((Q, k), np.int64) for k in (k0, k1)]
    for q in range(Q):
        uni = rng.permutation(4 * (k0 + k1))
        ids0 = uni[:k0]
        if q == 4:
            shared = min(k0, k1)
            ids1 = np.concatenate([ids0[:shared], uni[k0:k0 + k1 - shared]])
        elif q == 5:
            ids1 = uni[k0:k0 + k1]
        else:
            h = int(rng.integers(0, min(k0, k1) + 1))
            ids1 = np.concatenate([ids0[:h], uni[k0:k0 + k1 - h]])
        for sys_, ids in enumerate((ids0, rng.permutation(ids1))):
            k = ids.size
            if q == 3:
                sc = np.full(k, 0.25 + sys_)
            elif f64:
                sc = rng.standard_normal(k) * 10.0 ** rng.integers(-3, 4)
            else:
                sc = rng.integers(0, 50, k) / 8.0 if q % 2 else rng.standard_normal(k)
            sc = -np.sort(-sc.astype(sdt))
            ids = ids.copy()
            if (q == 0 and sys_ == 0) or (q == 1 and sys_ == 1) or q == 2:
                n_valid = 0
            elif q > 5 and rng.random() < 0.5:
                n_valid = int(rng.integers(1, k + 1))
            else:
                n_valid = k
            ids[n_valid:] = -1
            sc[n_valid:] = -np.inf
            s[sys_][q], i[sys_][q] = sc, ids
    return s[0], i[0], s[1], i[1]


@gpu
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("method", ["linear", "rrf"])
@pytest.mark.parametrize("k0,k1", [(2048, 2048), (2048, 2047), (1, 4095), (1, 2)])
def test_fusion_abi_widths_and_degenerate_queries(k0, k1, method, f64):
    """k0 + k1 up to the 4096 maximum (every shared-memory slot of every thread), sums that are not a power of two, and
    queries where one or both systems return only padding, ties within a system, all shared or none.  Bit-exact against
    oracle.fuse_linear / fuse_rrf over the returned lists; a system without a hit is absent from the query's results;
    rrf ranks are list positions.  Rows are sorted by (fused score desc, id asc)."""
    Q = 33
    s0, i0, s1, i1 = _fusion_inputs(Q, k0, k1, f64, seed=k0 * 7 + k1)
    ids, fused, counts = lr.fuse_topk_device(torch.from_numpy(s0).cuda(), torch.from_numpy(i0).cuda(),
                                             torch.from_numpy(s1).cuda(), torch.from_numpy(i1).cuda(), method=method)
    ids, fused, counts = ids.cpu().numpy(), fused.cpu().numpy(), counts.cpu().numpy()
    for q in range(Q):
        systems = []
        for sc, si in ((s0[q], i0[q]), (s1[q], i1[q])):
            keep = si >= 0
            if not keep.any():
                systems.append({})
            elif method == "linear":
                systems.append({"q": {str(a): float(b) for a, b in zip(si[keep], sc[keep])}})
            else:
                systems.append({"q": {str(a): -float(r) for r, a in enumerate(si[keep])}})
        ref = (oracle.fuse_linear(systems, weights=[0.7, 0.3]) if method == "linear"
               else oracle.fuse_rrf(systems)).get("q", {})
        order = sorted(ref.items(), key=lambda kv: (-kv[1], int(kv[0])))
        n = int(counts[q])
        assert n == len(ref), q
        assert ids[q, :n].tolist() == [int(p) for p, _ in order], q
        assert fused[q, :n].tolist() == [v for _, v in order], q
        assert (ids[q, n:] == -1).all() and np.isneginf(fused[q, n:]).all(), q
    assert counts[2] == 0
