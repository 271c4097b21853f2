"""Same-box A/B of K2 schedule variants at the headline shape: the corpus is generated once, then each configuration
(a set of LR_FLATIP_* environment knobs, re-read by the library before each configuration) is timed for a few steps with CUDA events,
with SM clocks sampled during the run.  Usage: python tools/ab_bench.py [--docs N] [--queries Q] [--steps K] cfg1 cfg2 ...
where cfg = "NAME:VAR=VAL,VAR=VAL" (e.g. "pair:LR_FLATIP_CLUSTER=3")."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import lightretriever_b200 as lr  # noqa: E402


class Clocks:
    def __init__(self):
        self.rows, self.proc = [], None

    def start(self):
        self.rows = []
        self.proc = subprocess.Popen(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader,nounits",
                                      "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        threading.Thread(target=lambda: [self.rows.append(l) for l in self.proc.stdout], daemon=True).start()

    def stop(self):
        self.proc.terminate()
        sm = [float(r.split(",")[0]) for r in self.rows if "," in r]
        pw = [float(r.split(",")[1]) for r in self.rows if "," in r]
        return (statistics.median(sm) if sm else None, max(pw) if pw else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=8_800_000)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--dim", type=int, default=4096)
    ap.add_argument("--topk", type=int, default=100)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--zeros", action="store_true", help="all-zero corpus (power sensitivity experiment)")
    ap.add_argument("cfgs", nargs="+")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    N, Q, d, k = a.docs, a.queries, a.dim, a.topk
    corpus = torch.empty((N, d), dtype=torch.bfloat16, device=dev)
    if a.zeros:
        corpus.zero_()
    else:
        for c0 in range(0, N, 131072):
            g = torch.Generator(device=dev).manual_seed(1000 + c0 // 131072)
            n = min(131072, N - c0)
            corpus[c0:c0 + n] = torch.nn.functional.normalize(torch.randn(131072, d, generator=g, device=dev), dim=-1)[:n].bfloat16()
    q = torch.nn.functional.normalize(torch.randn(Q, d, device=dev), dim=-1).bfloat16()
    lib = lr._C.load()
    flops = 2.0 * Q * N * d
    clocks = Clocks()
    known = set()
    for rep in range(a.repeat):
        for cfg in a.cfgs:
            name, _, kv = cfg.partition(":")
            for v in known:
                os.environ.pop(v, None)
            for pair in filter(None, kv.split(",")):
                var, val = pair.split("=")
                os.environ[var] = val
                known.add(var)
            lr._C.reload_env()
            for _ in range(2):
                lr.flatip_topk(q, corpus, k)
            torch.cuda.synchronize()
            clocks.start()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
            ev[0].record()
            for s in range(a.steps):
                lr.flatip_topk(q, corpus, k)
                ev[s + 1].record()
            torch.cuda.synchronize()
            mhz, pw = clocks.stop()
            ms = ev[0].elapsed_time(ev[-1]) / a.steps
            tf = flops / ms / 1e9
            util = tf * 1e12 / (148 * 8192 * (mhz or 1) * 1e6) if mhz else None
            print(json.dumps({"cfg": name, "rep": rep, "ms": round(ms, 2), "tflops": round(tf, 1), "sm_mhz": mhz,
                              "power_w_max": pw, "tensor_util_at_clock": round(util, 3) if util else None}), flush=True)
            time.sleep(1.0)


if __name__ == "__main__":
    main()
