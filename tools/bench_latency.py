"""Online-serving latency (BASELINE configs[4]): Qwen2.5-7B-shaped (d=3584, V=152064) EmbeddingBag encode + exact top-100
for batch 1 / 32, corpus row-sharded over the GPUs of the box (8.8M docs over 8 GPUs = 1.1M rows per GPU).
Per iteration: K1 encode -> K2 (warm-start + main pass + merge) -> [NCCL all-gather of keys + merge when world > 1].
Latency = CUDA events around one iteration on the current stream, max over ranks; p50 / p99 over --iters iterations.

--hybrid 1 adds a Zipf(1.0) sparse shard (--docs-per-gpu documents x 64 postings, V = the bag's vocabulary) and times
OnlineSearcher (dense only) and OnlineHybridSearcher (dense + token-count sparse + linear fusion) in the same process,
alternating one request of each, both as CUDA-graph replays.  Every result line carries the card's name and power limit,
read in the same run.

    python tools/bench_latency.py [--docs-per-gpu 1100000] [--hybrid 1]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/bench_latency.py
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import lightretriever_b200 as lr  # noqa: E402
from lightretriever_b200.sharded import exchange_candidates  # noqa: E402


def gpu_info(local: int) -> dict:
    """Name and power limit of this rank's card (read-only nvidia-smi query)."""
    try:
        r = subprocess.run(["nvidia-smi", f"--id={local}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, limit = (x.strip() for x in r.stdout.strip().split(","))
        return {"gpu": name, "power_limit": limit}
    except Exception as e:  # the timing stays valid; say that the card could not be read
        return {"gpu": torch.cuda.get_device_name(local), "power_limit": f"unread ({e})"}


def zipf_shard(n: int, V: int, nnz: int, dev, seed: int, id_offset: int):
    """n documents x nnz Zipf(1.0) tokens over a random permutation of the vocabulary, impacts U{1..400}."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    w = 1.0 / torch.arange(1, V + 1, dtype=torch.float64, device=dev)
    cdf = torch.cumsum(w / w.sum(), 0)
    perm = torch.randperm(V, generator=gen, device=dev)
    index = lr.ImpactIndex(V, device=dev, id_offset=id_offset)
    for c0 in range(0, n, 1 << 18):
        m = min(1 << 18, n - c0)
        u = torch.rand(m * nnz, generator=gen, device=dev, dtype=torch.float64)
        tok = perm[torch.searchsorted(cdf, u).clamp_max(V - 1)].to(torch.int32).view(m, nnz)
        imp = torch.randint(1, 401, (m, nnz), generator=gen, device=dev, dtype=torch.int32)
        index.add_dense_rows(tok, imp)
    index.build()
    return index


def percentiles(ts: list, dev, world: int) -> tuple:
    t = torch.tensor(ts, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t = t.sort().values
    return float(t[len(t) // 2]), float(t[int(len(t) * 0.99)]), float(t[0])


def timed(fn) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def run_hybrid(a, bag, corpus, rank, world, dev, info):
    """Dense-only and hybrid searchers over the same shard, one request of each in turn."""
    n = a.docs_per_gpu
    lo = rank * n
    index = zipf_shard(n, a.vocab, 64, dev, seed=1000 + rank, id_offset=lo)
    for B in a.batches:
        gq = torch.Generator().manual_seed(B)
        lens = torch.randint(1, 33, (B,), generator=gq)
        ids = torch.randint(0, a.vocab - 1, (int(lens.sum()),), generator=gq).to(dev)
        offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).to(dev)
        dense = lr.OnlineSearcher(bag, corpus, a.topk, batch=B, max_tokens=32 * B, id_offset=lo)
        hybrid = lr.OnlineHybridSearcher(bag, corpus, index, a.topk, batch=B, max_tokens=32 * B, id_offset=lo)
        arms = {"dense": lambda: dense.search(ids, offs), "hybrid": lambda: hybrid.search(ids, offs)}
        for _ in range(10):
            for fn in arms.values():
                fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ts = {name: [] for name in arms}
        for _ in range(a.iters):
            for name, fn in arms.items():
                ts[name].append(timed(fn))
        res = {name: percentiles(t, dev, world) for name, t in ts.items()}
        if rank == 0:
            line = {"config": "C5 online hybrid", "n_gpus": world, "docs_total": n * world, "docs_per_gpu": n,
                    "dim": a.dim, "vocab": a.vocab, "sparse_postings_per_doc": 64, "batch": B, "k": a.topk,
                    "mode": "cuda_graph", "iters": a.iters, **info}
            for name, (p50, p99, mn) in res.items():
                line[name] = {"p50_ms": p50, "p99_ms": p99, "min_ms": mn}
            line["hybrid_minus_dense_p50_ms"] = res["hybrid"][0] - res["dense"][0]
            print(json.dumps(line), flush=True)
        del dense, hybrid


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs-per-gpu", type=int, default=1_100_000)
    ap.add_argument("--dim", type=int, default=3584)
    ap.add_argument("--vocab", type=int, default=152064)
    ap.add_argument("--topk", type=int, default=100)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 32])
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step as one CUDA graph; 0: eager launches")
    ap.add_argument("--hybrid", type=int, default=0, help="1: time OnlineSearcher and OnlineHybridSearcher side by side")
    a = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    g = torch.Generator(device=dev).manual_seed(rank)
    table = (torch.randn(a.vocab, a.dim, device=dev, generator=torch.Generator(device=dev).manual_seed(0)) * 0.02).bfloat16()
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=a.vocab - 1)
    n = a.docs_per_gpu
    corpus = torch.empty((n, a.dim), dtype=torch.bfloat16, device=dev)
    for c0 in range(0, n, 131072):
        m = min(131072, n - c0)
        corpus[c0:c0 + m] = torch.nn.functional.normalize(torch.randn(m, a.dim, device=dev, generator=g), dim=-1).bfloat16()
    lo = rank * n
    if a.hybrid:
        run_hybrid(a, bag, corpus, rank, world, dev, gpu_info(local))
        finish(world)
        return
    for B in a.batches:
        gq = torch.Generator().manual_seed(B)
        lens = torch.randint(1, 33, (B,), generator=gq)
        ids = torch.randint(0, a.vocab - 1, (int(lens.sum()),), generator=gq).to(dev)
        offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).to(dev)

        def step():
            qv = bag.encode(ids, offs, normalize=True, check_ids=False)
            if world == 1:
                return lr.flatip_topk(qv, corpus, a.topk, id_offset=lo)
            _, _, keys = lr.flatip_topk(qv, corpus, a.topk, id_offset=lo, return_keys=True)
            return lr.topk_merge(exchange_candidates(keys), a.topk)

        mode = "eager"
        if a.graph:  # one CUDA-graph replay per request (lightretriever_b200.online.OnlineSearcher)
            srv = lr.OnlineSearcher(bag, corpus, a.topk, batch=B, max_tokens=32 * B, id_offset=lo)
            eager_step, step = step, (lambda: srv.search(ids, offs))
            mode = "cuda_graph"
        for _ in range(10):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ts = []
        for _ in range(a.iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        t = torch.tensor(ts, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.sort().values
        if rank == 0:
            floor_ms = n * a.dim * 2 / (6547.8e9) * 1e3
            print(json.dumps({"config": "C5 online", "n_gpus": world, "docs_total": n * world, "docs_per_gpu": n, "dim": a.dim,
                              "batch": B, "k": a.topk, "mode": mode, "p50_ms": float(t[len(t) // 2]), "p99_ms": float(t[int(len(t) * 0.99)]),
                              "min_ms": float(t[0]), "hbm_floor_ms": floor_ms,
                              "frac_of_hbm_roofline_p50": floor_ms / float(t[len(t) // 2]), "qps_p50": B / float(t[len(t) // 2]) * 1e3}),
                  flush=True)
    finish(world)


def finish(world: int) -> None:
    if world > 1:
        # the searchers' CUDA graphs captured NCCL collectives: tearing the communicator down under them can hang
        # (bench.py records it at 8 GPUs), so the process ends without the teardown
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
