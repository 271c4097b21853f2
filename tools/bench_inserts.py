"""Cost of the delta segment in the online searcher (c5b32 per-GPU shape: 1.1M x 3584 bf16 rows, batch 32, k = 100).

For insert_capacity 0, 16384 and 65536 it reports the per-request replay latency (p50 / p99 over CUDA events) with the
delta empty and full, and the insert throughput (documents / s, host clock around work that ends in a device
synchronise) for batches of 1, 32 and 1024 documents.  Prints one JSON line per measurement, with the GPU name and its
power limit.  Single GPU; run one process per GPU (torch.distributed.run) for the sharded shape, which is not
implemented here.

    python tools/bench_inserts.py [--rows 1100000] [--requests 300]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lightretriever_b200 as lr  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = torch.cuda.get_device_name(0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_100_000)
    ap.add_argument("--dim", type=int, default=3584)
    ap.add_argument("--vocab", type=int, default=152064)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--requests", type=int, default=300)
    ap.add_argument("--capacities", default="0,16384,65536")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = gpu_info()
    gen = torch.Generator(device=dev).manual_seed(0)
    table = (torch.randn(args.vocab, args.dim, device=dev, generator=gen) * 0.02).bfloat16()
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=args.vocab - 1)
    corpus = torch.empty((args.rows, args.dim), dtype=torch.bfloat16, device=dev)
    for lo in range(0, args.rows, 1 << 17):
        n = min(1 << 17, args.rows - lo)
        corpus[lo:lo + n] = F.normalize(torch.randn(n, args.dim, device=dev, generator=gen), dim=-1).bfloat16()
    hgen = torch.Generator().manual_seed(1)
    lens = torch.randint(1, 33, (args.batch,), generator=hgen)
    ids = torch.randint(0, args.vocab - 1, (int(lens.sum()),), generator=hgen).to(dev)
    offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).to(dev)

    def latency(srv):
        for _ in range(20):
            srv.search(ids, offs)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.requests)]
        for a, b in ev:
            a.record()
            srv.search(ids, offs)
            b.record()
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ev)
        return ms[len(ms) // 2], ms[min(len(ms) - 1, int(len(ms) * 0.99))]

    for cap in (int(c) for c in args.capacities.split(",")):
        srv = lr.OnlineSearcher(bag, corpus, args.k, batch=args.batch, max_tokens=32 * args.batch, insert_capacity=cap)
        p50, p99 = latency(srv)
        print(json.dumps({"insert_capacity": cap, "delta": "empty", "p50_ms": p50, "p99_ms": p99, "gpu": info}),
              flush=True)
        if cap:
            rate = {}
            for nb in (1, 32, 1024):
                rows = F.normalize(torch.randn(nb, args.dim, device=dev, generator=gen), dim=-1).bfloat16()
                reps = max(1, min(64, (cap // 4) // (nb * 3)))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(reps):
                    srv.insert(rows)
                torch.cuda.synchronize()
                rate[nb] = reps * nb / (time.perf_counter() - t0)
            print(json.dumps({"insert_capacity": cap, "insert_docs_per_s": rate, "gpu": info}), flush=True)
            rest = cap - srv._n_inserted
            for lo in range(0, rest, 8192):
                n = min(8192, rest - lo)
                srv.insert(F.normalize(torch.randn(n, args.dim, device=dev, generator=gen), dim=-1).bfloat16())
            p50, p99 = latency(srv)
            print(json.dumps({"insert_capacity": cap, "delta": "full", "p50_ms": p50, "p99_ms": p99, "gpu": info}),
                  flush=True)
        del srv
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
