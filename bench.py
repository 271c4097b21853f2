#!/usr/bin/env python
"""bench.py — benchmarks of the serving-side retrieval hot path (BASELINE.json metric and configs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Default workload `c2` = BASELINE.json configs[1] at the metric's k=100: Llama-3.1-8B-shaped EmbeddingBag table
(V=128256, d=4096, bf16, random init), batches of 10 000 synthetic queries (1..32 tokens), exact inner-product top-100
over an 8.8M x 4096 bf16 synthetic corpus (72.1 GB), row-sharded over the N GPUs (strong scaling: the corpus is fixed).
One step = one query batch: K1 EmbeddingBag encode (+L2 norm) -> K2 fused tcgen05 scoring/top-k -> merge; with N > 1
every rank scores 1/N of the warm-start prefix, the per-rank prefix top-k are exchanged (NCCL all-gather + merge) so that
all ranks start the main pass from the k-th best score of the whole prefix, then the per-shard top-k keys are
all-gathered and merged on device.

Other workloads (same JSON schema, `--config`):
    c1        configs[0]  Llama-3.2-1B-shaped (V=128256, d=2048): 1k queries, top-100 over 100k docs (the CPU-runnable case)
    c2k1000   configs[1]  at the reference's eval default k=1000
    c3m128 | c3m256 | c3m512 | c3m1024   configs[2]  MRL widths over full-width stored rows (truncation fused into K1 and K2)
    c4        configs[3]  sparse impact scoring (K4): 10k query token-count vectors vs 8.8M docs x 256 postings, Zipf(1.0) tokens
    c4uniform             the same with uniform tokens (closed-form bytes)
    c4head    configs[3]  document sparse head (K3): log1p(relu(max_t h_t.W)) + top-256 sparsify + quantise, 512-token docs
    c5b1 | c5b32  configs[4]  Qwen2.5-7B-shaped (d=3584, V=152064) online serving, batch 1 / 32, one CUDA-graph replay per request

Prints ONE JSON line (rank 0).  `value` = units/s with the step's inputs resident in HBM; `e2e` = the same through the
public API with HOST buffers (pinned inputs in, results out, copies inside the timed region).  `parity` checks sampled
rows of the result of the LAST TIMED STEP (the global, cross-GPU merged result when N > 1) against an fp32 / integer
recomputation; a violation makes the run fail.  `--impl reference` times the reference's CPU path (torch EmbeddingBag fp32
+ matmul + topk — faiss is not installed; scipy CSR product for the sparse path) on the host cores, on a bounded sample of
the same workload whose shape is stated in `config.sample`.

`--dump-outputs DIR` writes what the last timed step returned (the merged result when N > 1), one row per query or
document, as DIR/<name>.npy: ids and token ids as float64, scores and impacts as float32, and rows.npy with the row
numbers written.  A result above 64 MB is cut to a fixed, seeded sample of rows.  Every input is generated from fixed
seeds, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAX_TOK = 32
CHUNK_ROWS = 131072
DUMP_BYTES = 64 << 20

# name -> workload description (BASELINE.json configs)
DENSE = {
    #            V       d     docs       Q      k     m     pad id  requests per step (latency configs)
    "c1":      (128256, 2048, 100_000,   1_000,  100,  None, 128002, 0),
    "c2":      (128256, 4096, 8_800_000, 10_000, 100,  None, 128002, 0),
    "c2k1000": (128256, 4096, 8_800_000, 10_000, 1000, None, 128002, 0),
    "c3m128":  (128256, 4096, 8_800_000, 10_000, 100,  128,  128002, 0),
    "c3m256":  (128256, 4096, 8_800_000, 10_000, 100,  256,  128002, 0),
    "c3m512":  (128256, 4096, 8_800_000, 10_000, 100,  512,  128002, 0),
    "c3m1024": (128256, 4096, 8_800_000, 10_000, 100,  1024, 128002, 0),
    # the same widths over a corpus STORED compact [N, m] (what encoding with dense_shrink_dim = m gives): no column scales
    "c3m128c": (128256, 4096, 8_800_000, 10_000, 100,  128,  128002, 0),
    "c3m256c": (128256, 4096, 8_800_000, 10_000, 100,  256,  128002, 0),
    "c5b1":    (152064, 3584, 8_800_000, 1,      100,  None, 152063, 100),
    "c5b32":   (152064, 3584, 8_800_000, 32,     100,  None, 152063, 100),
}
SPARSE = {"c4": "zipf", "c4uniform": "uniform"}
ALL_CONFIGS = list(DENSE) + list(SPARSE) + ["c4head"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default 5 (c1: 100 — its step lasts about a millisecond)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=ALL_CONFIGS)
    # development overrides (the judged run uses the defaults of the config)
    ap.add_argument("--docs", type=int, default=None)
    ap.add_argument("--queries", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--topk", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--parity-rows", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 100 if a.config == "c1" and a.impl == "b200" else 5
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm keeps no results)")
    return a


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def load_traffic(name, world):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this exact config."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        e = t.get(f"{name}@{world}")
        return (e["dram_bytes_per_launch"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


def make_queries(n_queries: int, seed: int, vocab: int, pad_id: int):
    import torch
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(1, MAX_TOK + 1, (n_queries,), generator=g)
    ids = torch.randint(0, vocab, (int(lens.sum()),), generator=g)
    ids[ids == pad_id] = 0
    offsets = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
    return ids, offsets


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.3] or [r for _, r in self.rows]
        for r in rows:
            parts = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                power.append(float(parts[2]))
                for nme, val in zip(names, parts[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# =================================================================================================== dense workloads
class DenseWorkload:
    """K1 EmbeddingBag encode -> K2 exact inner-product top-k (-> cross-GPU exchange + merge)."""

    unit = "queries/s"
    higher_is_better = True
    dtype = "bf16"
    scaling = "strong"

    def __init__(self, name, args):
        V, d, N, Q, k, m, pad, rps = DENSE[name]
        self.name = name
        self.V, self.pad = V, pad
        self.d = args.dim or d
        self.N = args.docs or N
        self.Q = args.queries or Q
        self.k = args.topk or k
        self.m = m
        self.compact = name.endswith("c") and m is not None   # corpus rows hold only the (re-normalised) MRL prefix
        self.requests_per_step = rps           # > 0: online-serving config, a step = that many requests
        self.n_batches = 4
        self.units_per_step = self.Q * (rps or 1)
        self.parity_rows = args.parity_rows
        width = (f"compact MRL rows m={m}, table " if self.compact else f"MRL prefix m={m} of ") if m else ""
        self.metric = f"QPS (EmbBag encode + exact top-{self.k}, {self.N / 1e6:.3g}M x {width}{self.d} bf16)"
        if name == "c2" and (self.d, self.N, self.Q, self.k) == (4096, 8_800_000, 10_000, 100):
            self.metric = "QPS (EmbBag encode + exact top-100, 8.8M x 4096 bf16)"  # BASELINE.json's wording

    # -------------------------------------------------------------------------------- description
    def config(self, world):
        c = {"workload": (f"{self.name}: EmbeddingBag(V={self.V},d={self.d},bf16) encode + exact IP top-{self.k}, "
                          f"{self.Q}-query batches vs {self.N}-doc bf16 corpus" + (f", MRL width {self.m}" if self.m else "")
                          + (" (corpus stored compact [N, m], unit rows)" if self.compact else "")),
             "queries_per_step": self.units_per_step, "docs": self.N, "dim": self.d, "k": self.k,
             "max_query_tokens": MAX_TOK, "sharding": f"corpus row-sharded over {world} GPU(s)",
             "l2": "inputs larger than L2 (corpus shard streams from HBM every step)"}
        if self.m:
            c["mrl_width"] = self.m
        if self.requests_per_step:
            c["requests_per_step"] = self.requests_per_step
            c["batch"] = self.Q
        if self.N * self.d * 2 // world < (256 << 20):
            c["l2"] = "L2 flushed between steps (a 256 MB buffer is rewritten)"
        return c

    # -------------------------------------------------------------------------------- state
    def setup(self, dev, rank, world):
        import torch
        import lightretriever_b200 as lr
        from lightretriever_b200.sharded import shard_range
        self.lr, self.torch, self.dev, self.rank, self.world = lr, torch, dev, rank, world
        gt = torch.Generator(device=dev).manual_seed(0)
        table = (torch.randn(self.V, self.d, generator=gt, device=dev) * 0.02).bfloat16()
        self.bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=self.pad)
        self.lo, self.hi = shard_range(self.N, rank, world)
        n_local = self.hi - self.lo
        self.corpus = torch.empty((n_local, self.m if self.compact else self.d), dtype=torch.bfloat16, device=dev)
        self.c_scale = torch.empty(n_local, dtype=torch.float32, device=dev) if (self.m and not self.compact) else None
        for c0 in range((self.lo // CHUNK_ROWS) * CHUNK_ROWS, self.hi, CHUNK_ROWS):
            gc = torch.Generator(device=dev).manual_seed(1000 + c0 // CHUNK_ROWS)  # chunk-seeded: every N sees the same corpus
            blk = torch.nn.functional.normalize(torch.randn(CHUNK_ROWS, self.d, generator=gc, device=dev), dim=-1).bfloat16()
            a, b = max(c0, self.lo), min(c0 + CHUNK_ROWS, self.hi)
            if self.compact:  # truncate, then normalise (modeling_hybrid.py:487-490), store the prefix only
                self.corpus[a - self.lo:b - self.lo] = torch.nn.functional.normalize(blk[a - c0:b - c0, :self.m].float(), dim=-1).bfloat16()
                del blk
                continue
            self.corpus[a - self.lo:b - self.lo] = blk[a - c0:b - c0]
            if self.m:  # reciprocal prefix norms of the stored bf16 values (modeling_hybrid.py:487-490: truncate, then normalise)
                self.c_scale[a - self.lo:b - self.lo] = 1.0 / blk[a - c0:b - c0, :self.m].float().norm(dim=1).clamp_min(1e-12)
            del blk
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if self.corpus.numel() * 2 < (256 << 20) else None
        self.host_batches = []
        for i in range(self.n_batches):
            ids, offs = make_queries(self.Q, 100 + i, self.V, self.pad)
            self.host_batches.append((ids.pin_memory(), offs.pin_memory()))
        self.dev_batches = [(a.to(dev), b.to(dev)) for a, b in self.host_batches]
        self.out_s_host = torch.empty((self.Q, self.k), dtype=torch.float32).pin_memory()
        self.out_i_host = torch.empty((self.Q, self.k), dtype=torch.int64).pin_memory()
        self.online = None
        if self.requests_per_step:
            self.online = lr.OnlineSearcher(self.bag, self.corpus, self.k, batch=self.Q, max_tokens=MAX_TOK * self.Q,
                                            id_offset=self.lo)
        self.req_events = []

    def _merge_across(self, keys):
        from lightretriever_b200.sharded import exchange_candidates
        return self.lr.topk_merge(exchange_candidates(keys), self.k, return_keys=True)[2]

    def encode(self, ids, offs):
        return self.bag.encode(ids, offs, shrink_dim=self.m, normalize=True, check_ids=False)          # K1

    def search(self, qv):
        lr = self.lr
        d_used = None if self.compact else self.m
        if self.world == 1:
            return lr.flatip_topk(qv, self.corpus, self.k, d_used=d_used, c_scale=self.c_scale, id_offset=self.lo)
        keys = lr.flatip_topk_sharded(qv, self.corpus, self.k, self.world, self._merge_across, d_used=d_used,
                                      c_scale=self.c_scale, id_offset=self.lo)[2]                      # K2 on the shard
        from lightretriever_b200.sharded import exchange_candidates
        return lr.topk_merge(exchange_candidates(keys), self.k)                                        # all-gather + merge

    def step(self, ids, offs, record=False):
        torch = self.torch
        if self.flush is not None:
            self.flush.zero_()
        if not self.online:
            return self.search(self.encode(ids, offs))
        res = None
        for _ in range(self.requests_per_step):  # online serving: one CUDA-graph replay per request
            if record:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            res = self.online.search(ids, offs)
            if record:
                e1.record()
                self.req_events.append((e0, e1))
        return res

    def step_e2e(self, i):
        ids, offs = self.host_batches[i % self.n_batches]
        if not self.online:
            s_, i_ = self.step(ids.to(self.dev, non_blocking=True), offs.to(self.dev, non_blocking=True))
            self.out_s_host.copy_(s_, non_blocking=True)
            self.out_i_host.copy_(i_, non_blocking=True)
            return
        if self.flush is not None:
            self.flush.zero_()
        for _ in range(self.requests_per_step):  # every request: host ids in, host results out
            s_, i_ = self.online.search(ids.to(self.dev, non_blocking=True), offs.to(self.dev, non_blocking=True))
            self.out_s_host.copy_(s_, non_blocking=True)
            self.out_i_host.copy_(i_, non_blocking=True)

    def io_bytes(self):
        h2d = int(statistics.mean(a.numel() * 8 + b.numel() * 8 for a, b in self.host_batches)) * (self.requests_per_step or 1)
        d2h = self.Q * self.k * (4 + 8) * (self.requests_per_step or 1)
        return h2d, d2h

    # -------------------------------------------------------------------------------- roofline of the dominant kernel
    def roofline(self, kern_ms, step_ms, lib, peaks):
        rows = (ctypes.c_int64 * 64)()
        n = lib.lr_flatip_last_plan_passes(rows, 16)
        main = [int(x) for x in rows[4 * (n - 1):4 * n]] if n > 0 else [0, 0, 0, 0]
        n_local = self.hi - self.lo
        docs_main = min(main[1] * 256, n_local) - main[0] * 256   # documents of the pass the profile events bracket
        m = self.m or self.d
        name = "umma_gemm_kernel<EPI_TOPK> main pass (tcgen05 bf16 GEMM + fused top-k epilogue)"
        passes = [{"tiles": [int(rows[4 * i]), int(rows[4 * i + 1])], "splits": int(rows[4 * i + 2]),
                   "team_schedule": int(rows[4 * i + 3])} for i in range(n)]
        traffic, tsrc = load_traffic(self.name, self.world)
        if self.Q >= 209:   # SURVEY §8d: tensor-bound above the ridge point
            flops = 2.0 * self.Q * docs_main * m
            ach = flops / (kern_ms * 1e-3) / 1e12
            peak = peaks["bf16_tflops_sustained"]
            r = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                 "peak_source": f"{peaks['source']} MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)",
                 "flop_per_launch": flops, "algorithmic": f"2*Q*docs*m = 2*{self.Q}*{docs_main}*{m} (the bracketed main pass only)"}
        else:
            nbytes = float(docs_main) * m * 2
            ach = nbytes / (kern_ms * 1e-3) / 1e9
            peak = peaks["hbm_gbs"]
            r = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                 "peak_source": f"{peaks['source']} MEASURED_PEAKS.json hbm_gbs (copy bandwidth)",
                 "bytes_per_launch": nbytes, "algorithmic": f"docs*m*2 B = {docs_main}*{m}*2 (the bracketed main pass only)"}
        r.update({"kernel_ms": kern_ms, "traffic": traffic, "traffic_source": tsrc,
                  "kernel_share_of_step": kern_ms * (self.requests_per_step or 1) / step_ms, "passes": passes})
        # the same bound applied to the WHOLE step (K1 + every scoring pass + merges + exchange): a lower bound of every
        # kernel's own fraction, with nothing left out of the denominator
        per_req_ms = step_ms / (self.requests_per_step or 1)
        whole = (2.0 * self.Q * n_local * m / 1e12) if r["bound"] == "tensor" else (float(n_local) * m * 2 / 1e9)
        r["whole_step"] = {"work": whole * (1e12 if r["bound"] == "tensor" else 1e9), "ms": per_req_ms,
                           "achieved": whole / (per_req_ms * 1e-3), "frac": whole / (per_req_ms * 1e-3) / r["peak"]}
        return r

    # -------------------------------------------------------------------------------- the timed result
    def outputs(self, res):
        """What a caller receives, one row per query: top-k scores and document ids (-1 where fewer than k hits)."""
        s, i = res
        return {"scores": s.float().cpu(), "ids": i.double().cpu()}

    def parity(self, res, batch_index, dist):
        """Sampled rows of `res` — the (global) result of the last timed step — against an fp32 recomputation: fp32 scores of
        the same bf16 values over the whole (sharded) corpus, exact top-k with ties by ascending id, and the north star's
        tie-band rule (oracle.check_topk_parity semantics).  With N > 1 every rank scores its shard in fp32, the per-rank
        fp32 top-k are all-gathered and merged, and the fp32 scores of the returned ids are summed over their owners."""
        torch = self.torch
        s_got, i_got = res
        Q, k, dev = s_got.shape[0], self.k, self.dev
        ids, offs = self.dev_batches[batch_index]
        qv = self.encode(ids, offs)
        g = torch.Generator().manual_seed(7)
        rows = torch.unique(torch.cat([torch.tensor([0, Q - 1]), torch.randint(0, Q, (self.parity_rows,), generator=g)]))
        rows = rows[:max(1, self.parity_rows)].to(dev)
        m = self.m or self.d
        qs = qv[rows, :m].float()  # with an MRL width K1 has already truncated, then normalised (modeling_hybrid.py:487-490)
        kk = min(k, self.N)
        # (1) fp32 reference top-kk of the local shard, ties by ascending id (stable sort over id-ordered chunks)
        best_s = torch.full((rows.numel(), 0), 0.0, device=dev)
        best_i = torch.zeros((rows.numel(), 0), dtype=torch.int64, device=dev)
        n_local = self.hi - self.lo
        for c0 in range(0, n_local, 1 << 18):
            blk = self.corpus[c0:c0 + (1 << 18), :m].float()
            sc = qs @ blk.T
            if self.c_scale is not None:
                sc = sc * self.c_scale[c0:c0 + (1 << 18)][None, :]
            idx = torch.arange(c0, c0 + sc.shape[1], device=dev)[None, :].expand_as(sc) + self.lo
            cs, ci = torch.cat([best_s, sc], 1), torch.cat([best_i, idx], 1)
            order = torch.sort(cs, dim=1, descending=True, stable=True).indices[:, :kk]   # earlier = lower id wins ties
            best_s, best_i = torch.gather(cs, 1, order), torch.gather(ci, 1, order)
        # (2) fp32 score of every returned id, computed by the rank that owns it
        gi = i_got[rows]
        mine = (gi >= self.lo) & (gi < self.hi)
        loc = torch.where(mine, gi - self.lo, torch.zeros_like(gi))
        ref_at = torch.zeros(gi.shape, dtype=torch.float32, device=dev)
        for r0 in range(0, rows.numel(), 8):
            vec = self.corpus[loc[r0:r0 + 8].reshape(-1), :m].float().view(-1, gi.shape[1], m)
            dot = torch.einsum("rd,rkd->rk", qs[r0:r0 + 8], vec)
            if self.c_scale is not None:
                dot = dot * self.c_scale[loc[r0:r0 + 8]]
            ref_at[r0:r0 + 8] = torch.where(mine[r0:r0 + 8], dot, torch.zeros_like(dot))
        if self.world > 1:
            parts_s = [torch.empty_like(best_s) for _ in range(self.world)]
            parts_i = [torch.empty_like(best_i) for _ in range(self.world)]
            dist.all_gather(parts_s, best_s.contiguous())
            dist.all_gather(parts_i, best_i.contiguous())
            cs, ci = torch.cat(parts_s, 1), torch.cat(parts_i, 1)   # rank order = ascending id order
            order = torch.sort(cs, dim=1, descending=True, stable=True).indices[:, :kk]
            best_s, best_i = torch.gather(cs, 1, order), torch.gather(ci, 1, order)
            dist.all_reduce(ref_at)
        gs = s_got[rows]
        s_k = best_s[:, kk - 1:kk]
        rtol, atol = 1e-2, 1e-5
        tol = rtol * s_k.abs() + atol
        valid = gi[:, :kk] >= 0
        v = {
            "padding_misplaced": int((~valid).sum()) + int((gi[:, kk:] >= 0).sum()),
            "not_sorted": int((gs[:, 1:kk] > gs[:, :kk - 1]).sum()),
            "duplicate_ids": int((gi[:, :kk].sort(dim=1).values.diff(dim=1) == 0).sum()),
            "score_off": int(((gs[:, :kk] - ref_at[:, :kk]).abs() > rtol * ref_at[:, :kk].abs() + atol).sum()),
            "below_tie_band": int((ref_at[:, :kk] < s_k - tol).sum()),
        }
        must = best_s > s_k + tol                                              # fp32 winners outside the tie band ...
        present = (best_i[:, :, None] == gi[:, None, :kk]).any(dim=2)           # ... must all be returned
        v["missing_above_tie_band"] = int((must & ~present).sum())
        rel = ((gs[:, :kk] - ref_at[:, :kk]).abs() / ref_at[:, :kk].abs().clamp_min(1e-6)).max()
        return {"checked": "rows of the last TIMED step's result" + (" (cross-GPU merged)" if self.world > 1 else ""),
                "rows": int(rows.numel()), "k": kk, "rule": "ids exact outside the tie band 1e-2*|s_k|; scores within 1e-2 relative of fp32",
                "ids_identical_to_fp32_topk": float((best_i == gi[:, :kk]).float().mean()),
                "max_rel_score_err": float(rel), "violations": v, "ok": not any(v.values())}

    # -------------------------------------------------------------------------------- CPU reference (bounded sample)
    def cpu_sample(self, seconds, steps=1, warmup=0):
        """The reference's CPU path: fp32 EmbeddingBag + normalize (+ MRL truncation), fp32 matmul + topk
        (torch; faiss absent).  Full size when it fits the time budget (c1), else a row sub-sample of the corpus with the
        same d / k / query shape and QPS scaled linearly in N — stated in `sample`."""
        import torch
        from oracle import oracle
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        d, k, m = self.d, self.k, self.m
        g = torch.Generator().manual_seed(0)
        table = torch.randn(self.V, d, generator=g) * 0.02  # fp32 table, as the reference library path keeps it
        qn = min(self.Q, 1000)
        ids, offsets = make_queries(qn, 1, self.V, self.pad)
        w = m or d
        probe = torch.randn(4096, w)
        qprobe = torch.randn(qn, w)
        t = time.time()
        (qprobe @ probe.T).topk(min(k, 4096), dim=1)
        rate = 4096 / max(time.time() - t, 1e-4)  # corpus rows per second at this query batch
        n_s = int(min(self.N, max(20_000, min(400_000, rate * seconds))))
        corpus = torch.nn.functional.normalize(torch.randn(n_s, d, generator=g)[:, :w], dim=-1)
        times = []
        for _ in range(warmup + steps):
            t0 = time.time()
            qv = oracle.embbag_encode(ids, offsets, table, self.pad, m, True)
            oracle.flatip_topk_fast(qv, corpus, min(k, n_s))
            times.append(time.time() - t0)
        t_step = statistics.mean(times[warmup:])
        qps_sample = qn / t_step
        full = n_s == self.N and qn == self.Q
        qps_full = qps_sample * n_s / self.N
        shape = {"queries": qn, "docs": n_s, "dim": w, "k": min(k, n_s), "extrapolated": not full}
        return {"value": qps_full, "unit": self.unit, "cores": cores, "kind": "port",
                "sample": (f"{qn} queries x {n_s} of {self.N} docs, d={w}, k={k}, fp32 torch EmbeddingBag+matmul+topk (faiss absent); "
                           + ("full size, not extrapolated" if full else
                              f"measured {qps_sample:.1f} q/s on the sample, scaled by {n_s}/{self.N}")),
                "ms_per_step_sample": t_step * 1e3, "ms_per_step_full": self.units_per_step / qps_full * 1e3,
                "threads": torch.get_num_threads(), "sample_shape": shape}


# =================================================================================================== K4 sparse scoring
class SparseScoreWorkload:
    """C4 scoring side: query token counts x document impact vectors (K4), exact integer scores, top-k."""

    unit = "queries/s"
    higher_is_better = True
    dtype = "int32"
    scaling = "strong"
    V, NNZ = 128256, 256

    def __init__(self, name, args):
        self.name, self.dist_kind = name, SPARSE[name]
        self.N = args.docs or 8_800_000
        self.Q = args.queries or 10_000
        self.k = args.topk or 100
        self.units_per_step = self.Q
        self.n_batches = 4
        self.parity_rows = min(args.parity_rows, 32)
        self.requests_per_step = 0
        self.metric = f"QPS (sparse impact scoring, exact top-{self.k}, {self.N / 1e6:.3g}M docs x {self.NNZ} postings, {self.dist_kind} tokens)"

    def config(self, world):
        return {"workload": (f"{self.name}: query token counts (<= {MAX_TOK} tokens) x doc impact vectors ({self.NNZ} postings per doc, "
                             f"impacts U{{1..400}} u16, {self.dist_kind} tokens over V={self.V}), exact integer top-{self.k}"),
                "queries_per_step": self.Q, "docs": self.N, "vocab": self.V, "postings_per_doc": self.NNZ, "k": self.k,
                "token_distribution": "Zipf(1.0) rank-frequency over a shuffled vocabulary" if self.dist_kind == "zipf" else "uniform",
                "sharding": f"documents sharded over {world} GPU(s), per-shard inverted index",
                "l2": "inputs larger than L2 (the postings of a batch exceed L2 and are re-streamed every step)"}

    def _tokens(self, n, gen, dev):
        torch = self.torch
        if self.dist_kind == "uniform":
            return torch.randint(0, self.V, (n,), generator=gen, device=dev, dtype=torch.int32)
        # Zipf(1.0): p(rank r) ~ 1/r, inverse-CDF sampling on the harmonic numbers; ranks mapped through a fixed permutation
        u = torch.rand(n, generator=gen, device=dev, dtype=torch.float64)
        return self.perm[torch.searchsorted(self.cdf, u).clamp_max(self.V - 1)].to(torch.int32)

    def setup(self, dev, rank, world):
        import torch
        import lightretriever_b200 as lr
        from lightretriever_b200.sharded import shard_range
        self.lr, self.torch, self.dev, self.rank, self.world = lr, torch, dev, rank, world
        w = 1.0 / torch.arange(1, self.V + 1, dtype=torch.float64, device=dev)
        self.cdf = torch.cumsum(w / w.sum(), 0)
        self.perm = torch.randperm(self.V, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
        self.lo, self.hi = shard_range(self.N, rank, world)
        self.index = lr.ImpactIndex(self.V, device=dev, id_offset=self.lo)
        chunk = 1 << 17
        for c0 in range((self.lo // chunk) * chunk, self.hi, chunk):
            gc = torch.Generator(device=dev).manual_seed(2000 + c0 // chunk)
            tok = self._tokens(chunk * self.NNZ, gc, dev).view(chunk, self.NNZ)
            imp = torch.randint(1, 401, (chunk, self.NNZ), generator=gc, device=dev, dtype=torch.int32)
            a, b = max(c0, self.lo), min(c0 + chunk, self.hi)
            self.index.add_dense_rows(tok[a - c0:b - c0], imp[a - c0:b - c0])
            del tok, imp
        self.post = self.index.build()
        self.df = (self.post[0][1:] - self.post[0][:-1])
        self.host_batches, self.dev_batches = [], []
        for i in range(self.n_batches):
            gq = torch.Generator(device=dev).manual_seed(300 + i)
            lens = torch.randint(1, MAX_TOK + 1, (self.Q,), generator=gq, device=dev)
            qt = self._tokens(int(lens.sum()), gq, dev)
            # distinct tokens per query with counts: Counter(ids) (exact_search_base.py:371-435)
            qid = torch.repeat_interleave(torch.arange(self.Q, device=dev), lens)
            key = torch.unique(qid.to(torch.int64) * self.V + qt.to(torch.int64), return_counts=True)
            uq, cnt = key
            q_of, tok = uq // self.V, (uq % self.V).to(torch.int32)
            indptr = torch.zeros(self.Q + 1, dtype=torch.int32, device=dev)
            indptr[1:] = torch.cumsum(torch.bincount(q_of, minlength=self.Q), 0).to(torch.int32)
            b = (indptr, tok.contiguous(), cnt.to(torch.int32).contiguous())
            self.dev_batches.append(b)
            self.host_batches.append(tuple(x.cpu().pin_memory() for x in b))
        self.out_s_host = torch.empty((self.Q, self.k), dtype=torch.float32).pin_memory()
        self.out_i_host = torch.empty((self.Q, self.k), dtype=torch.int64).pin_memory()

    def step(self, qi, qt, qc, record=False):
        lr = self.lr
        if self.world == 1:
            return self.index.search_device(qi, qt, qc, self.k)
        from lightretriever_b200.sharded import exchange_candidates
        keys = self.index.search_device(qi, qt, qc, self.k, return_keys=True)[2]
        return lr.topk_merge(exchange_candidates(keys), self.k, score_kind=lr._C.LR_SCORE_U32)

    def step_e2e(self, i):
        b = self.host_batches[i % self.n_batches]
        s_, i_ = self.step(*(x.to(self.dev, non_blocking=True) for x in b))
        self.out_s_host.copy_(s_, non_blocking=True)
        self.out_i_host.copy_(i_, non_blocking=True)

    def io_bytes(self):
        h2d = int(statistics.mean(sum(x.numel() * 4 for x in b) for b in self.host_batches))
        return h2d, self.Q * self.k * 12

    def roofline(self, kern_ms, step_ms, lib, peaks):
        qt = self.dev_batches[0][1]
        nbytes = float(self.df[qt.long()].sum().item()) * 6.0   # SURVEY §8d: sum over query terms of df(t) * 6 B
        ach = nbytes / (kern_ms * 1e-3) / 1e9
        traffic, tsrc = load_traffic(self.name, self.world)
        return {"kernel": "sparse_score kernels of one lr_sparse_score_topk call (postings -> shared-memory accumulators -> top-k)",
                "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                "peak_source": f"{peaks['source']} MEASURED_PEAKS.json hbm_gbs (copy bandwidth)", "bytes_per_launch": nbytes,
                "algorithmic": "sum_t df(t) * 6 B (i32 doc + u16 impact) over the query terms of one batch; accumulators live in shared memory",
                "kernel_ms": kern_ms, "traffic": traffic, "traffic_source": tsrc, "kernel_share_of_step": kern_ms / step_ms}

    outputs = DenseWorkload.outputs  # the same (scores, ids) result, integer-valued scores

    def parity(self, res, batch_index, dist):
        """Integer scores: sampled rows of the timed (merged) result vs a dense int64 recomputation on device — bit-exact
        scores and ids (ties by ascending id), only matching documents returned."""
        torch = self.torch
        s_got, i_got = res
        dev, k = self.dev, self.k
        qi, qt, qc = self.dev_batches[batch_index]
        post_indptr, post_doc, post_imp = self.post[0], self.post[1], self.post[2]
        g = torch.Generator().manual_seed(11)
        rows = torch.unique(torch.cat([torch.tensor([0, self.Q - 1]), torch.randint(0, self.Q, (self.parity_rows,), generator=g)]))
        bad = {"score_mismatch": 0, "id_mismatch": 0}
        n_local = self.hi - self.lo
        for r in rows.tolist():
            acc = torch.zeros(n_local, dtype=torch.int64, device=dev)
            for j in range(int(qi[r]), int(qi[r + 1])):
                t, c = int(qt[j]), int(qc[j])
                a, b = int(post_indptr[t]), int(post_indptr[t + 1])
                acc.index_add_(0, post_doc[a:b].long(), (post_imp[a:b].to(torch.int32) & 0xFFFF).long() * c)
            # exact top-k of the shard: (score desc, id asc) via a combined key
            key = acc * (1 << 32) + ((1 << 32) - 1 - (torch.arange(n_local, device=dev) + self.lo))
            key = torch.where(acc > 0, key, torch.zeros_like(key))
            top = torch.topk(key, min(k, n_local)).values
            if self.world > 1:
                parts = [torch.empty_like(top) for _ in range(self.world)]
                dist.all_gather(parts, top)
                top = torch.topk(torch.cat(parts), k).values
            es = torch.where(top > 0, (top >> 32).float(), torch.full_like(top, float("-inf"), dtype=torch.float32))
            ei = torch.where(top > 0, (1 << 32) - 1 - (top & 0xFFFFFFFF), torch.full_like(top, -1))
            kk = es.numel()
            bad["score_mismatch"] += int((s_got[r, :kk] != es).sum())
            bad["id_mismatch"] += int((i_got[r, :kk] != ei).sum())
        return {"checked": "rows of the last TIMED step's result" + (" (cross-GPU merged)" if self.world > 1 else ""),
                "rows": int(rows.numel()), "k": k, "rule": "integer scores and ids bit-exact (ties by ascending id)",
                "violations": bad, "ok": not any(bad.values())}

    def cpu_sample(self, seconds, steps=1, warmup=0):
        """Reference CPU path = Anserini (JVM, absent) -> scipy CSR product + argpartition on the host cores (SURVEY §8d),
        on a document sub-sample; QPS scaled linearly in N."""
        import numpy as np
        import scipy.sparse as sp
        cores = os.cpu_count() or 1
        rng = np.random.default_rng(0)
        n_s, qn = min(self.N, 200_000), min(self.Q, 1000)

        def toks(n):
            if self.dist_kind == "uniform":
                return rng.integers(0, self.V, n)
            w = 1.0 / np.arange(1, self.V + 1)
            return np.searchsorted(np.cumsum(w / w.sum()), rng.random(n)).clip(max=self.V - 1)
        D = sp.csr_matrix((rng.integers(1, 401, n_s * self.NNZ).astype(np.int32), toks(n_s * self.NNZ),
                           np.arange(0, n_s * self.NNZ + 1, self.NNZ)), shape=(n_s, self.V))
        D.sum_duplicates()
        Dt = D.T.tocsr()
        lens = rng.integers(1, MAX_TOK + 1, qn)
        Qm = sp.csr_matrix((np.ones(lens.sum(), np.int32), toks(lens.sum()), np.concatenate([[0], np.cumsum(lens)])),
                           shape=(qn, self.V))
        Qm.sum_duplicates()
        times = []
        for _ in range(warmup + steps):
            t0 = time.time()
            for q0 in range(0, qn, 100):
                S = (Qm[q0:q0 + 100] @ Dt).toarray()
                idx = np.argpartition(-S, self.k, axis=1)[:, :self.k]
                np.take_along_axis(S, idx, 1)
            times.append(time.time() - t0)
        t_step = statistics.mean(times[warmup:])
        qps_s = qn / t_step
        qps = qps_s * n_s / self.N
        return {"value": qps, "unit": self.unit, "cores": 1, "kind": "port",
                "sample": (f"{qn} queries x {n_s} of {self.N} docs x {self.NNZ} postings, scipy CSR product + argpartition top-{self.k} "
                           f"(Anserini/JVM absent; scipy's product is single-threaded); measured {qps_s:.1f} q/s, scaled by {n_s}/{self.N}"),
                "ms_per_step_sample": t_step * 1e3, "ms_per_step_full": self.Q / qps * 1e3, "threads": 1,
                "sample_shape": {"queries": qn, "docs": n_s, "extrapolated": n_s != self.N}, "host_cores": cores}


# =================================================================================================== K3 sparse head
class SparseHeadWorkload:
    """C4 document side: hidden states -> log1p(relu(max over valid tokens of lm_head . h)) -> top-k sparsify -> quantise."""

    unit = "docs/s"
    higher_is_better = True
    dtype = "bf16"
    scaling = "weak"
    V, d, S, TOPK = 128256, 4096, 512, 256

    def __init__(self, name, args):
        self.name = name
        self.B = args.queries or 64
        self.units_per_step = self.B
        self.n_batches = 2
        self.requests_per_step = 0
        self.metric = f"docs/s (sparse head: lm_head max-pool over <= {self.S} tokens + relu/log1p + top-{self.TOPK} + quantise, V={self.V}, d={self.d})"

    def config(self, world):
        return {"workload": (f"{self.name}: {self.B} documents per step per GPU, lengths U{{16..{self.S}}} (mean 264 valid tokens), hidden "
                             f"[B,{self.S},{self.d}] bf16, lm_head [{self.V},{self.d}] bf16, relu+log1p, top_k_psg={self.TOPK}, quantise x100"),
                "docs_per_step_per_gpu": self.B, "seq_len": self.S, "dim": self.d, "vocab": self.V, "top_k": self.TOPK,
                "sharding": f"data-parallel over {world} GPU(s) (documents are independent, no exchange)",
                "l2": "inputs larger than L2 (lm_head is 1.05 GB and is streamed every step)"}

    def setup(self, dev, rank, world):
        import torch
        import lightretriever_b200 as lr
        self.lr, self.torch, self.dev, self.rank, self.world = lr, torch, dev, rank, world
        g = torch.Generator(device=dev).manual_seed(0)
        self.W = (torch.randn(self.V, self.d, generator=g, device=dev) * 0.02).bfloat16()
        self.host_batches, self.dev_batches = [], []
        for i in range(self.n_batches):
            gb = torch.Generator(device=dev).manual_seed(400 + 16 * rank + i)
            h = torch.randn(self.B, self.S, self.d, generator=gb, device=dev).bfloat16()
            lens = torch.randint(16, self.S + 1, (self.B,), generator=gb, device=dev)
            mask = torch.arange(self.S, device=dev)[None] < lens[:, None]
            mask[:, 0] = False  # bos (get_sparse_attention_mask, sparse_pooling.py:23-41)
            self.dev_batches.append((h, mask, int(mask.sum())))  # the host owns the attention mask: it knows the count
            self.host_batches.append((h.cpu().pin_memory(), mask.cpu().pin_memory(), int(mask.sum())))
        self.valid_tokens = float(statistics.mean(float(m.sum()) for _, m, _ in self.dev_batches))

    def step(self, h, mask, total, record=False):
        return self.lr.sparse_head(h, self.W, None, mask, sparse_top_k=self.TOPK, valid_tokens=total)

    def step_e2e(self, i):
        h, mask, total = self.host_batches[i % self.n_batches]
        indptr, tok, imp = self.step(h.to(self.dev, non_blocking=True), mask.to(self.dev, non_blocking=True), total)
        self._host = (indptr.cpu(), tok.cpu(), imp.cpu())

    def io_bytes(self):
        h2d = self.B * self.S * (self.d * 2 + 1)
        return h2d, self.B * (4 + self.TOPK * 6)

    def roofline(self, kern_ms, step_ms, lib, peaks):
        flops = 2.0 * self.valid_tokens_all() * self.d * self.V
        ach = flops / (kern_ms * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        traffic, tsrc = load_traffic(self.name, self.world)
        return {"kernel": "umma_gemm_kernel<EPI_MAXTOK> (tcgen05 bf16 GEMM, masked max over tokens + relu/log1p epilogue)",
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "peak_source": f"{peaks['source']} MEASURED_PEAKS.json bf16_tflops_sustained",
                "flop_per_launch": flops, "algorithmic": "2 * sum_b S_b * d * V over the document tokens the kernel has to read (SURVEY §8d)",
                "kernel_ms": kern_ms, "traffic": traffic, "traffic_source": tsrc, "kernel_share_of_step": kern_ms / step_ms}

    def valid_tokens_all(self):
        # every token up to a document's length is multiplied (the mask removes bos / eos / prompt afterwards)
        return float(statistics.mean(float((m.float().cumsum(1).argmax(1) + 1).sum()) for _, m, _ in self.dev_batches))

    def outputs(self, res):
        """The CSR a caller receives, as one row per document in CSR order: token ids (-1 after the document's last
        entry) and their uint16 impacts (0 there)."""
        torch = self.torch
        indptr, tok, imp = (x.cpu().long() for x in res)
        n = indptr[1:] - indptr[:-1]
        doc = torch.repeat_interleave(torch.arange(n.numel()), n)
        col = torch.arange(tok.numel()) - indptr[doc]
        tokens = torch.full((n.numel(), max(int(n.max()), 1)), -1.0, dtype=torch.float64)
        impacts = torch.zeros(tokens.shape, dtype=torch.float32)
        tokens[doc, col] = tok.double()
        impacts[doc, col] = (imp & 0xFFFF).float()
        return {"tokens": tokens, "impacts": impacts}

    def parity(self, res, batch_index, dist):
        """4 documents of the timed step against the fp32 oracle (max over valid tokens -> relu -> log1p -> top-k with ties
        -> round-half-even x100): integer impacts within the documented band |d| <= max(1, 1e-2*impact) (SURVEY §8c trap 7),
        token sets equal outside the tie band."""
        torch = self.torch
        indptr, tok, imp = res
        h, mask, _ = self.dev_batches[batch_index]
        bad = {"impact_off": 0, "tokens_outside_band": 0}
        for b in (0, 1, self.B // 2, self.B - 1):
            hv = h[b][mask[b]].float()
            logits = torch.cat([(hv @ self.W[v0:v0 + 16384].float().T).max(dim=0).values for v0 in range(0, self.V, 16384)])
            x = torch.log1p(torch.relu(logits))
            kth = torch.topk(x, self.TOPK).values[-1]
            ref_q = torch.round(x * 100.0)
            a, e = int(indptr[b]), int(indptr[b + 1])
            t = tok[a:e].long()
            got = (imp[a:e].to(torch.int32) & 0xFFFF).float()
            bad["impact_off"] += int(((got - ref_q[t]).abs() > torch.maximum(torch.ones_like(got), 1e-2 * ref_q[t])).sum())
            band = 1e-2 * float(kth) + 1e-5
            bad["tokens_outside_band"] += int((x[t] < kth - band).sum())
            must = torch.nonzero((x > kth + band) & (ref_q > 0)).flatten()
            bad["tokens_outside_band"] += int((~torch.isin(must, t)).sum())
        return {"checked": "4 documents of the last TIMED step's CSR result", "rows": 4,
                "rule": "impacts within max(1, 1e-2*impact) of the fp32 oracle; token sets equal outside the tie band",
                "violations": bad, "ok": not any(bad.values())}

    def cpu_sample(self, seconds, steps=1, warmup=0):
        import torch
        from oracle import oracle
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        g = torch.Generator().manual_seed(0)
        Bs, Ss = 2, 64
        W = torch.randn(self.V, self.d, generator=g) * 0.02
        h = torch.randn(Bs, Ss, self.d, generator=g)
        mask = torch.ones(Bs, Ss, dtype=torch.bool)
        times = []
        for _ in range(warmup + steps):
            t0 = time.time()
            out = oracle.max_linear_map(h, W.T, None, mask)
            oracle.get_sparse_emb(out, top_k=self.TOPK)
            times.append(time.time() - t0)
        t_step = statistics.mean(times[warmup:])
        docs_s = Bs / t_step * Ss / 264.0
        return {"value": docs_s, "unit": self.unit, "cores": cores, "kind": "port",
                "sample": (f"{Bs} documents x {Ss} tokens, fp32 torch port of max_linear_mapping (python loop over tokens) + "
                           f"relu/log1p/top-k; scaled by {Ss}/264 tokens per document"),
                "ms_per_step_sample": t_step * 1e3, "ms_per_step_full": self.B / docs_s * 1e3, "threads": torch.get_num_threads(),
                "sample_shape": {"docs": Bs, "tokens": Ss, "extrapolated": True}}


def dump_outputs(arrays, out_dir):
    """Write `arrays` (name -> CPU tensor, one row per query or document) as out_dir/<name>.npy, and rows.npy with the row
    numbers written.  Above DUMP_BYTES the rows are a fixed, seeded sample: the same rows for every build."""
    import numpy as np
    import torch
    n = next(iter(arrays.values())).shape[0]
    row_bytes = 8 + sum(a[0].numel() * a.element_size() for a in arrays.values())
    keep = min(n, (DUMP_BYTES - 4096) // row_bytes)  # 4 KB for the .npy headers
    rows = torch.arange(n)
    if keep < n:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), rows.double().numpy())
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows].numpy())


def make_workload(args):
    if args.config in DENSE:
        return DenseWorkload(args.config, args)
    if args.config in SPARSE:
        return SparseScoreWorkload(args.config, args)
    return SparseHeadWorkload(args.config, args)


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = make_workload(args)
    cb = wl.cpu_sample(seconds=max(5.0, args.cpu_seconds), steps=max(args.steps, 1), warmup=min(args.warmup, 1))
    cfg = wl.config(max(int(args.gpus), 1))  # the B200 arm's config for the same N
    cfg["sample"] = cb["sample_shape"]       # ... and the shape this arm actually ran
    line = {
        "impl": "reference", "metric": wl.metric, "value": cb["value"], "unit": wl.unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step_full"],
        "ms_per_step_sample": cb["ms_per_step_sample"], "higher_is_better": True,
        "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {k_: cb[k_] for k_ in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import lightretriever_b200 as lr
    lib = lr._C.load()
    wl = make_workload(args)
    wl.setup(dev, rank, world)
    steps, warmup = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # profile events around the dominant kernel of every timed step
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in kev:
        a.record()
        b.record()  # materialise the cudaEvent_t handles
    torch.cuda.synchronize()

    # ---- warm-up
    for w in range(warmup):
        wl.step(*wl.dev_batches[w % wl.n_batches])
    barrier()

    # ---- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    sev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    barrier()
    launches0 = lib.lr_kernel_launches()
    t_wall0 = time.time()
    sev[0].record()
    res = None
    for s in range(steps):
        if not wl.requests_per_step:
            lib.lr_set_profile_events(ctypes.c_void_p(kev[s][0].cuda_event), ctypes.c_void_p(kev[s][1].cuda_event))
        res = wl.step(*wl.dev_batches[s % wl.n_batches], record=True)
        sev[s + 1].record()
    lib.lr_set_profile_events(None, None)
    barrier()
    t_wall1 = time.time()
    launches = lib.lr_kernel_launches() - launches0
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    step_ms = [sev[s].elapsed_time(sev[s + 1]) for s in range(steps)]
    total_ms = sev[0].elapsed_time(sev[steps])
    if args.dump_outputs and rank == 0:  # before anything else runs: online configs return buffers their graph reuses
        dump_outputs(wl.outputs(res), args.dump_outputs)
    last_batch = (steps - 1) % wl.n_batches
    req_ms = sorted(a.elapsed_time(b) for a, b in getattr(wl, "req_events", []))
    if wl.requests_per_step:
        # graph replays cannot carry the profile events: time the dominant kernel in one eager request after the timed region
        lib.lr_set_profile_events(ctypes.c_void_p(kev[0][0].cuda_event), ctypes.c_void_p(kev[0][1].cuda_event))
        wl.search(wl.encode(*wl.dev_batches[last_batch]))
        lib.lr_set_profile_events(None, None)
        torch.cuda.synchronize()
        kern_ms = [kev[0][0].elapsed_time(kev[0][1])]
        launches = launches  # graph replays re-run the captured kernels: counted below from the captured step
    else:
        kern_ms = [a.elapsed_time(b) for a, b in kev]

    # ---- timed region 2: end to end through the public API with host buffers
    for w in range(2):
        wl.step_e2e(w)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        wl.step_e2e(s)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    h2d, d2h = wl.io_bytes()

    # ---- max over ranks
    t = torch.tensor([total_ms, e2e_ms, statistics.mean(kern_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, kern_ms_mean = t.tolist()

    # ---- parity of the timed result (outside the timed region; collective under N > 1)
    parity = wl.parity(res, last_batch, dist)

    if wl.requests_per_step:  # kernels per request, from one eager request
        l0 = lib.lr_kernel_launches()
        wl.search(wl.encode(*wl.dev_batches[last_batch]))
        launches = (lib.lr_kernel_launches() - l0) * wl.requests_per_step * steps

    ok = True
    if rank == 0:
        peaks = load_peaks()
        n_units = wl.units_per_step * (world if wl.scaling == "weak" else 1)
        line = {
            "metric": wl.metric, "value": n_units * steps / (total_ms * 1e-3), "unit": wl.unit, "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
            "higher_is_better": wl.higher_is_better, "scaling": wl.scaling, "vs_baseline": None, "dtype": wl.dtype,
            "data": "synthetic", "config": wl.config(world),
            "p50_ms_per_step": statistics.median(step_ms),
            "e2e": {"value": n_units * steps / (e2e_ms * 1e-3), "unit": wl.unit, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / steps},
            "gpu_launches": int(launches),
            "roofline": wl.roofline(kern_ms_mean, total_ms / steps, lib, peaks),
            "parity": parity,
            "clocks": clocks,
        }
        if req_ms:
            line["latency_ms"] = {"requests": len(req_ms), "batch": wl.Q, "p50": req_ms[len(req_ms) // 2],
                                  "p99": req_ms[min(len(req_ms) - 1, int(len(req_ms) * 0.99))], "min": req_ms[0],
                                  "what": "one CUDA-graph replay per request: K1 encode + K2 search (+ NCCL all-gather + merge), rank 0"}
        if not args.no_cpu_baseline and world == 1:
            cb = wl.cpu_sample(seconds=args.cpu_seconds)
            line["cpu_baseline"] = {k_: cb[k_] for k_ in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
        ok = bool(parity["ok"])
        if not ok:
            print(f"PARITY VIOLATION in the timed result: {parity['violations']}", file=sys.stderr, flush=True)
    if world > 1:
        dist.barrier()
        if wl.requests_per_step:
            # The online configs hold CUDA graphs that captured NCCL collectives; tearing the communicator down under them
            # hung at 8 GPUs (c5b32: every rank had printed / passed the barrier, torchrun never returned).  Leave the
            # teardown to process exit.
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0 if ok else 1)
        dist.destroy_process_group()
    if not ok:
        sys.exit(1)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
