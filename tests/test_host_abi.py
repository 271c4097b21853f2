"""CPU-side checks: the C-ABI library loads and exports exactly what include/lr_b200.h declares, the host logic matches
the reference-pinned oracle, and the product path refuses to run without the GPU (no CPU fallback)."""
import json
import os
import re

import numpy as np
import pytest
import torch

import lightretriever_b200 as lr
from lightretriever_b200 import _C
from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "lr_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _C.load()
    declared = _declared_functions()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/lr_b200.h but not exported"
    assert sorted(_C.PROTOTYPES) == declared, "ctypes prototypes out of sync with the header"
    assert lib.lr_version() == 100


def test_workspace_sizing_needs_no_gpu():
    lib = _C.load()
    ws = lib.lr_flatip_workspace_bytes(10000, 8_800_000, 100)
    assert 0 < ws < (16 << 30)
    assert lib.lr_flatip_workspace_bytes(10000, 8_800_000, 1000) > ws
    assert lib.lr_sparse_score_workspace_bytes(32, 8_800_000, 100) > 0
    assert lib.lr_sparse_block_docs() == 4096
    assert lib.lr_flatip_workspace_bytes(0, 10, 10) == 0


def _plan(Q, N, k):
    import ctypes
    out = (ctypes.c_int64 * 16)()
    assert _C.load().lr_flatip_plan(Q, N, k, out) == 0
    names = ["cl", "pair", "m_tiles", "n_tiles", "cap", "prefix_tiles", "prefix_splits", "prefix_units", "main_begin",
             "main_splits", "main_units", "grid", "band", "ws", "rounds", "n_clusters"]
    return dict(zip(names, list(out)))


def test_flatip_plan_invariants():
    """Host planner (csrc/flatip_topk.cu:make_plan): the two passes partition the corpus tiles, lists are long enough,
    the grid is whole clusters, and the documented regimes pick the documented variants."""
    lib = _C.load()
    for Q, N, k in [(10000, 8_800_000, 100), (10000, 1_100_000, 100), (10000, 8_800_000, 1000), (1, 1_100_000, 100),
                    (32, 1_100_000, 100), (128, 300, 10), (129, 5000, 2048), (1000, 100_000, 100), (7, 50, 100)]:
        p = _plan(Q, N, k)
        assert p["m_tiles"] == -(-Q // 128) and p["n_tiles"] == -(-N // 256)
        assert p["cap"] >= k + 64 and p["cap"] % 64 == 0
        assert p["main_begin"] == p["prefix_tiles"] < p["n_tiles"]              # prefix + main cover [0, n_tiles)
        assert 1 <= p["main_splits"] <= p["n_tiles"] - p["main_begin"]
        groups = -(-p["m_tiles"] // p["cl"])
        assert p["main_units"] == groups * p["main_splits"]
        assert p["prefix_units"] == (groups * p["prefix_splits"] if p["prefix_tiles"] else 0)
        assert p["grid"] % p["cl"] == 0 and 1 <= p["grid"] <= 148
        assert p["pair"] in (0, 1) and (not p["pair"] or p["cl"] == 2)
        assert 0 < p["ws"] == lib.lr_flatip_workspace_bytes_for(Q, N, k, 4096) <= lib.lr_flatip_workspace_bytes(Q, N, k)
        assert lib.lr_flatip_workspace_bytes_for(Q, N, k, 128) <= lib.lr_flatip_workspace_bytes(Q, N, k)
    head = _plan(10000, 8_800_000, 100)
    assert (head["cl"], head["pair"], head["prefix_tiles"], head["cap"]) == (2, 1, 128, 256)   # cta_group::2 pair on the team schedule, 32768-doc prefix
    big_k = _plan(10000, 8_800_000, 1000)
    assert (big_k["cl"], big_k["pair"], big_k["cap"]) == (2, 1, 2048) and big_k["prefix_tiles"] == 1000  # pair + 256k-doc prefix
    online = _plan(32, 1_100_000, 100)
    assert (online["cl"], online["prefix_tiles"], online["prefix_splits"]) == (1, 148, 148)     # one tile per CTA
    assert _plan(1, 1_100_000, 100)["prefix_tiles"] == 0                                          # single query: single phase
    # balanced: the main pass wastes < 3% of its rounds at the headline shape
    assert head["main_units"] / (head["rounds"] * head["n_clusters"]) > 0.97


def test_sparse_score_plan_invariants():
    """Host planner of K4 (csrc/sparse_score.cu:ss_plan): both kernels are planned (regime dispatch), every launch fits the
    227 KB of shared memory, a unit of the row kernel keeps >= 4 steps unless the corpus is smaller, the merge sees at
    most 64 lists per query, and the workspace the planner reports is the one the entry point asks for."""
    import ctypes
    lib = _C.load()
    names = ["bd", "nblk", "cap", "flat", "rows", "S_flat", "S_rows", "S", "w_flat16", "w_flat32", "w_rows16", "w_rows32",
             "smem_flat16", "smem_rows16", "ws", "step_docs"]
    for Q, N, k in [(10000, 1_100_000, 100), (10000, 8_800_000, 100), (32, 1_100_000, 100), (1, 8_800_000, 1000),
                    (20, 3000, 10), (10000, 1_100_000, 1000), (7, 50, 1024)]:
        out = (ctypes.c_int64 * 16)()
        assert lib.lr_sparse_score_plan(Q, N, k, out) == 0
        p = dict(zip(names, list(out)))
        assert p["bd"] == lib.lr_sparse_block_docs() and p["nblk"] == -(-N // p["bd"])
        assert p["cap"] >= k + 128 and p["cap"] % 32 == 0
        assert p["flat"] == 1 and p["rows"] == 1                                   # default: both, chosen on the device
        assert 1 <= p["S_flat"] <= min(64, p["nblk"]) and 1 <= p["S_rows"] <= min(64, p["nblk"])
        assert p["S"] == max(p["S_flat"], p["S_rows"])
        assert all(1 <= p[w] <= 20 for w in ("w_flat16", "w_flat32")) and all(1 <= p[w] <= 11 for w in ("w_rows16", "w_rows32"))
        assert 0 < p["smem_flat16"] <= 227 * 1024 and 0 < p["smem_rows16"] <= 227 * 1024
        assert p["step_docs"] % p["bd"] == 0 and p["step_docs"] >= p["bd"]
        steps = -(-N // p["step_docs"])
        assert p["S_rows"] >= min(64, p["nblk"], steps // 4)                       # slices small enough to stay in L2
        assert p["ws"] == lib.lr_sparse_score_workspace_bytes(Q, N, k) and p["ws"] % 256 == 0
        assert p["ws"] >= p["S"] * Q * p["cap"] * 8
    big = (ctypes.c_int64 * 16)()
    lib.lr_sparse_score_plan(10000, 1_100_000, 100, big)
    assert dict(zip(names, list(big)))["S_rows"] == 33 and dict(zip(names, list(big)))["w_rows16"] == 11


def test_sparse_head_packed_plan_invariants():
    """Host planner of the packed K3 kernel (csrc/sparse_head.cu:packed_plan): balanced runs of whole 256-token tiles, about
    two tiles per split and at most 64 splits, every split non-empty, workspace = counters + split table + edge rows."""
    import ctypes
    lib = _C.load()
    V = 128256
    for T in (1, 255, 256, 257, 5000, 17_000, 67_500, 1_000_000):
        out = (ctypes.c_int64 * 4)()
        assert lib.lr_sparse_head_packed_plan(T, V, out) == 0
        tiles, splits, off_edge, ws = list(out)
        assert tiles == -(-T // 256) and 1 <= splits <= min(64, tiles)
        assert splits == -(-tiles // max(2, -(-tiles // 64)))                       # ~2 tiles per split, more when T is large
        sizes = [((s + 1) * tiles) // splits - (s * tiles) // splits for s in range(splits)]
        assert min(sizes) >= 1 and max(sizes) - min(sizes) <= 1 and sum(sizes) == tiles
        assert ws == lib.lr_sparse_head_packed_workspace_bytes(T, V) == off_edge + splits * 2 * V * 4
        assert off_edge % 256 == 0 and off_edge >= 64 * 1024 + splits * 4
    assert lib.lr_sparse_head_packed_workspace_bytes(0, V) == 0


def test_argument_errors_map_to_value_error():
    lib = _C.load()
    rc = lib.lr_flatip_topk(None, 0, None, 0, 1, 1, 8, None, None, 0, 1, None, None, None, None, 0, None)
    assert rc == _C.LR_EINVAL
    with pytest.raises(ValueError):
        _C.check(rc)
    assert "null" in _C.last_error()
    rc = lib.lr_topk_merge(None, None, 1, 1, 1, 1, 1, 0, 0, None, None, None, None)
    assert rc == _C.LR_EINVAL


def test_no_cpu_fallback():
    bag = lr.B200EmbeddingBag.from_pretrained(torch.randn(10, 8), padding_idx=0)
    with pytest.raises(RuntimeError, match="no CPU path"):
        bag.forward(torch.tensor([1, 2]), torch.tensor([0]))
    with pytest.raises(RuntimeError, match="no CPU path"):
        lr.flatip_topk(torch.randn(2, 8).bfloat16(), torch.randn(4, 8).bfloat16(), 2)
    with pytest.raises(RuntimeError, match="no CPU path"):
        lr.max_linear_mapping(torch.randn(1, 4, 8), torch.randn(8, 16))
    # nothing in the product package imports the oracle
    pkg = os.path.join(ROOT, "lightretriever_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, fn)).read()
                assert "import oracle" not in src and "from oracle" not in src, f"{fn} reaches into oracle/"


def test_flatten_and_query_parsing_match_oracle(golden_dir):
    g = np.load(os.path.join(golden_dir, "flatten.npz"))
    lists = [[(ord(c) % 50) for c in str(q)][:12] for q in g["queries"]]
    enc = lr.flatten_token_ids(lists)
    np.testing.assert_array_equal(enc["input_ids"].numpy(), g["input_ids"])
    np.testing.assert_array_equal(enc["offsets"].numpy(), g["offsets"])

    class FakeTok:
        def __call__(self, queries, max_length, truncation, add_special_tokens, return_attention_mask):
            return {"input_ids": [[(ord(c) % 50) for c in q][:max_length] for q in queries]}

    enc2 = lr.tokenize_nonctx_qry_emb_bag([str(q) for q in g["queries"]], FakeTok(), max_len=12)
    np.testing.assert_array_equal(enc2["input_ids"].numpy(), g["input_ids"])
    from lightretriever_b200.sparse_search import json_to_csr, parse_queries
    qi, qt, qc = parse_queries(["5 7 5 5 900", {"3": 2}, ""], vocab_size=100)
    assert qi.tolist() == [0, 2, 3, 3] and dict(zip(qt[:2].tolist(), qc[:2].tolist())) == oracle.query_counts([5, 7, 5, 5])
    ip, tk, im = json_to_csr([{"4": 10, "2": 3}, {"-1": 1}, {"9": 65535}])
    assert ip.tolist() == [0, 2, 2, 3] and tk.tolist() == [4, 2, 9] and im.tolist() == [10, 3, 65535]


def test_sparse_mask_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "sparse_head.npz"))
    ids, am = torch.from_numpy(g["input_ids"]), torch.from_numpy(g["am"])
    np.testing.assert_array_equal(lr.get_sparse_attention_mask(ids, am, 7, False).numpy(), g["mask"])
    np.testing.assert_array_equal(lr.get_sparse_attention_mask(ids, am, 7, True).numpy(), g["mask_rp"])


def test_fusion_dict_packing_for_the_device_kernel(golden_dir):
    """The dict-shaped fusion functions are adapters over lr_fuse_topk: this is their host half (dicts -> sorted arrays
    over a joint id numbering); the arithmetic is checked against the same golden on the GPU (test_gpu_parity)."""
    from lightretriever_b200.hybrid import _pack_systems
    g = json.load(open(os.path.join(golden_dir, "fusion.json")))
    qn, pn, ((s0, i0), (s1, i1)) = _pack_systems([g["dense"], g["sparse"]], "cpu")
    assert sorted(qn) == sorted(set(g["dense"]) | set(g["sparse"]))
    for res, s, i in ((g["dense"], s0, i0), (g["sparse"], s1, i1)):
        assert s.dtype == torch.float64 and i.dtype == torch.int64
        for r, q in enumerate(qn):
            row = res.get(q, {})
            n = len(row)
            assert (i[r, n:] == -1).all() and (i[r, :n] >= 0).all()
            assert {pn[j]: float(v) for j, v in zip(i[r, :n].tolist(), s[r, :n].tolist())} == {k: float(v) for k, v in row.items()}
            assert bool((s[r, :max(n - 1, 0)] >= s[r, 1:n]).all())  # rank = position (rrf)
    with pytest.raises(NotImplementedError):
        _pack_systems([{}, {}, {}], "cpu")


def test_faiss_flat_file_layout(tmp_path):
    """The on-disk IndexFlatIP layout FlatIPIndex.save/load speak (faiss_index.py:42-43, faiss_search.py:478-488): fourcc
    "IxFI", d, ntotal, two dummies, is_trained, metric 0, float count, fp32 rows.  Header checked byte for byte against a
    file assembled by hand here (Faiss itself is absent: format restated from index_write.cpp, parity unpinned)."""
    import struct
    from lightretriever_b200.search import _FAISS_FLAT_IP, _FAISS_HEADER
    assert _FAISS_HEADER.size == 45 and struct.pack("<I", _FAISS_FLAT_IP) == b"IxFI"
    rows = np.arange(12, dtype=np.float32).reshape(3, 4)
    blob = (b"IxFI" + struct.pack("<i", 4) + struct.pack("<q", 3) + struct.pack("<qq", 1 << 20, 1 << 20) + b"\x01" +
            struct.pack("<i", 0) + struct.pack("<Q", 12) + rows.tobytes())
    assert _FAISS_HEADER.unpack(blob[:45]) == (_FAISS_FLAT_IP, 4, 3, 1 << 20, 1 << 20, True, 0, 12)
    path = tmp_path / "x.flat.faiss"
    path.write_bytes(blob)
    got = np.memmap(path, dtype=np.float32, mode="r", offset=45, shape=(3, 4))
    np.testing.assert_array_equal(np.asarray(got), rows)
    bad = tmp_path / "bad.faiss"
    bad.write_bytes(b"IxF2" + blob[4:])
    with pytest.raises((ValueError, RuntimeError)):
        lr.FlatIPIndex.load(str(bad))


def test_shard_ranges_partition_the_corpus():
    for n, w in [(8_800_000, 8), (10, 3), (7, 8), (1, 1)]:
        r = [lr.shard_range(n, i, w) for i in range(w)]
        assert r[0][0] == 0 and r[-1][1] == n
        assert all(r[i][1] == r[i + 1][0] for i in range(w - 1))
        sizes = [b - a for a, b in r]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        lr.shard_range(10, 3, 3)


def test_flatip_passes_partition_the_corpus():
    """Warm-start prefix, threshold-refresh passes and main pass must cover every corpus tile exactly once, in order, for
    full-width and short rows alike; short rows with large batches refresh the thresholds and run two epilogue sets."""
    import ctypes
    lib = _C.load()

    def passes(Q, N, k, d):
        rows, flags = (ctypes.c_int64 * 64)(), (ctypes.c_int64 * 2)()
        n = lib.lr_flatip_plan_passes(Q, N, k, d, rows, 16, flags)
        assert 1 <= n <= 16
        return [tuple(rows[4 * i:4 * i + 4]) for i in range(n)], tuple(flags)

    for Q in (1, 32, 300, 2304, 10000):
        for N in (50, 70_000, 1_100_000, 8_800_000):
            for k in (10, 100, 1000):
                for d in (64, 128, 512, 768, 1024, 3584, 4096):
                    ps, (wide, lmul) = passes(Q, N, k, d)
                    n_tiles = -(-N // 256)
                    assert ps[0][0] == 0 and ps[-1][1] == n_tiles
                    for (b0, e0, s0, _), (b1, _e1, _s1, _t1) in zip(ps, ps[1:]):
                        assert b0 < e0 == b1
                    for b, e, s, team in ps:
                        assert 1 <= s <= e - b and team in (0, 1)
                    assert lmul == (2 if wide else 1)
                    assert not wide or (d <= 768 and Q > 128 and k <= 352)
    ps, (wide, lmul) = passes(10000, 1_100_000, 100, 128)   # BASELINE configs[2] on a shard
    assert [p[:2] for p in ps] == [(0, 128), (128, 512), (512, 2048), (2048, 4297)] and ps[-1][3] == 1 and (wide, lmul) == (1, 2)
    ps, (wide, _) = passes(10000, 8_800_000, 100, 128)
    assert [p[:2] for p in ps] == [(0, 128), (128, 512), (512, 2048), (2048, 8192), (8192, 34375)] and wide == 1
    ps, (wide, _) = passes(10000, 8_800_000, 100, 4096)      # headline: prefix + one main pass on the team schedule
    assert [p[:2] for p in ps] == [(0, 128), (128, 34375)] and ps[1][3] == 1 and wide == 0
    assert passes(32, 1_100_000, 100, 3584)[0][0][:3] == (0, 148, 148)   # online: one tile per cluster
