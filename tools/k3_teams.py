"""K3 (sparse head) same-box A/B: team schedule (pairs / multicast, window, band) vs the round-robin schedule."""
import json, os, sys, statistics
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import lightretriever_b200 as lr

dev = "cuda"
V, d, S = 128256, 4096, 512
W = (torch.randn(V, d, device=dev) * 0.02).bfloat16()
KNOBS = ("LR_SPARSE_HEAD_DOCS_PER_UNIT", "LR_SPARSE_HEAD_CLUSTER", "LR_SPARSE_HEAD_SCHED", "LR_SPARSE_HEAD_TEAM_BAND",
         "LR_SPARSE_HEAD_TEAM_WINDOW")


def run(B, h, mask, env, ref=None, iters=10):
    for k in KNOBS:
        os.environ.pop(k, None)
    os.environ.update(env)
    lr._C.reload_env()
    f = lambda: lr.max_linear_mapping(h, W, None, mask, relu=True, log1p=True, weight_is_vd=True)
    for _ in range(4):
        out = f()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        f()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / iters
    same = None if ref is None else bool(torch.equal(out, ref))
    return ms, same, out


CFGS = {"rr": {"LR_SPARSE_HEAD_SCHED": "0"},
        "pair_d1": {"LR_SPARSE_HEAD_CLUSTER": "3", "LR_SPARSE_HEAD_DOCS_PER_UNIT": "1"},
        "pair_d2": {"LR_SPARSE_HEAD_CLUSTER": "3", "LR_SPARSE_HEAD_DOCS_PER_UNIT": "2"},
        "mc_d1": {"LR_SPARSE_HEAD_CLUSTER": "2", "LR_SPARSE_HEAD_DOCS_PER_UNIT": "1"},
        "mc_d2": {"LR_SPARSE_HEAD_CLUSTER": "2", "LR_SPARSE_HEAD_DOCS_PER_UNIT": "2"},
        "mc_d4": {"LR_SPARSE_HEAD_CLUSTER": "2", "LR_SPARSE_HEAD_DOCS_PER_UNIT": "4"},
        "mc_band12": {"LR_SPARSE_HEAD_CLUSTER": "2", "LR_SPARSE_HEAD_TEAM_BAND": "12"},
        "pair_band12": {"LR_SPARSE_HEAD_CLUSTER": "3", "LR_SPARSE_HEAD_TEAM_BAND": "12"},
        "default": {}}
for B in (16, 64, 256):
    h = torch.randn(B, S, d, device=dev).bfloat16()
    lens = torch.randint(16, S + 1, (B,), device=dev)
    mask = (torch.arange(S, device=dev)[None] < lens[:, None])
    _, _, ref = run(B, h, mask, CFGS["rr"], iters=2)
    res = {k: [] for k in CFGS}
    ok = True
    for rep in range(4):   # interleaved rounds: box clock / power state drifts between configurations
        for name, env in CFGS.items():
            ms, same, _ = run(B, h, mask, env, ref, iters=max(3, int(300 / (B * 0.5))))
            res[name].append(round(ms, 3))
            ok = ok and same
    for name in CFGS:
        ms = statistics.median(res[name])
        print(json.dumps({"B": B, "cfg": name, "ms_median": ms, "ms_all": res[name], "tflops": round(2.0 * B * S * d * V / ms / 1e9, 1)}), flush=True)
    print(json.dumps({"B": B, "all_bit_identical_to_round_robin": ok}), flush=True)
