"""Cost of document filters inside the exact top-k: each workload timed unfiltered and filtered in the same process,
alternating, with CUDA events around the search call (scoring + merge).

    python tools/bench_filters.py [--reps R] [--only NAME ...]

Workloads (bench.py shapes, random unit vectors; MRL widths read a prefix of full-width rows with reciprocal prefix norms):
    c2_del10      10k queries x 8.8M x 4096, k = 100, 10 % of the documents deleted
    c5b32_del10   32 queries x 1.1M x 3584, k = 100, 10 % deleted
    c5b32_allow1  the same with a per-query allow row admitting 1 % of the documents (8 rows, query q uses row q % 8)
    c3m128_del10  10k queries x 8.8M, MRL prefix of 128 of 4096 columns, k = 100, 10 % deleted (short rows: epilogue-bound)
One JSON line per workload: median ms unfiltered / filtered and their ratio, with the card's name and power limit.  The
numbers are measurements, not a pass/fail bar: a selective filter on short rows is expected to be slower (cold
thresholds: far fewer allowed documents reach each list cut)."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lightretriever_b200 as lr  # noqa: E402
from lightretriever_b200.filters import doc_bitmap  # noqa: E402

WORKLOADS = {  # name: (Q, N, d stored, d used, k, filter)
    "c2_del10": (10_000, 8_800_000, 4096, 4096, 100, "del10"),
    "c5b32_del10": (32, 1_100_000, 3584, 3584, 100, "del10"),
    "c5b32_allow1": (32, 1_100_000, 3584, 3584, 100, "allow1"),
    "c3m128_del10": (10_000, 8_800_000, 4096, 128, 100, "del10"),
}


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        return [x.strip() for x in out.split(",")]
    except Exception as e:  # the numbers stay usable without it
        return [torch.cuda.get_device_name(0), f"unknown ({e})"]


def _corpus(N, d, gen):
    c = torch.empty((N, d), dtype=torch.bfloat16, device="cuda")
    for lo in range(0, N, 1 << 18):
        c[lo:lo + (1 << 18)] = F.normalize(torch.randn(min(1 << 18, N - lo), d, device="cuda", generator=gen), dim=-1)
    return c


def _time(fn, reps):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in ev)[reps // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", nargs="*", default=None)
    args = ap.parse_args()
    name_card, power = _card()
    gen = torch.Generator(device="cuda").manual_seed(0)
    cache = {}
    for name, (Q, N, d, m, k, kind) in WORKLOADS.items():
        if args.only and name not in args.only:
            continue
        if (N, d) not in cache:
            cache.clear()
            torch.cuda.empty_cache()
            cache[(N, d)] = _corpus(N, d, gen)
        c = cache[(N, d)]
        q = F.normalize(torch.randn(Q, m, device="cuda", generator=gen), dim=-1).bfloat16()
        kw = {}
        if m < d:  # MRL: prefix of the stored rows, scored as cosine of the prefixes
            kw = dict(c_scale=(1.0 / c[:, :m].float().norm(dim=1).clamp_min(1e-12)).contiguous(), d_used=m)
        perm = torch.randperm(N, device="cuda", generator=gen)
        if kind == "del10":
            filt = dict(live=doc_bitmap(N, perm[: N - N // 10], "cuda"))
        else:
            allow = torch.stack([doc_bitmap(N, torch.randperm(N, device="cuda", generator=gen)[: N // 100], "cuda")
                                 for _ in range(8)]).contiguous()
            filt = dict(allow=allow, q_filter=(torch.arange(Q, device="cuda") % 8).to(torch.int32))
        plain = lambda: lr.flatip_topk(q, c, k, **kw)
        filtered = lambda: lr.flatip_topk(q, c, k, **kw, **filt)
        plain(), filtered()  # warm-up: module load, workspace, plan cache
        torch.cuda.synchronize()
        t_plain, t_filt = [], []
        for _ in range(2):  # alternate the two arms
            t_plain.append(_time(plain, args.reps))
            t_filt.append(_time(filtered, args.reps))
        a, b = min(t_plain), min(t_filt)
        print(json.dumps({"workload": name, "Q": Q, "N": N, "d_used": m, "k": k, "filter": kind,
                          "ms_unfiltered": round(a, 3), "ms_filtered": round(b, 3), "ratio": round(b / a, 4),
                          "runs_unfiltered": [round(x, 3) for x in t_plain], "runs_filtered": [round(x, 3) for x in t_filt],
                          "gpu": name_card, "power_limit": power}), flush=True)
        del q, kw, filt


if __name__ == "__main__":
    main()
