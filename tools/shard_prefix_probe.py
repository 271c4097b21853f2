"""Shard shape of the 8-GPU headline run (10k queries x 1.1M x 4096, top-100): warm-start prefix size sweep."""
import os, sys, json, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lightretriever_b200 as lr
N, d, Q, k = 1_100_000, 4096, 10000, 100
c = torch.nn.functional.normalize(torch.randn(N, d, device="cuda"), dim=-1).bfloat16()
q = torch.nn.functional.normalize(torch.randn(Q, d, device="cuda"), dim=-1).bfloat16()
def t(fn, it=8):
    for _ in range(3): fn()
    torch.cuda.synchronize(); a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(it): fn()
    b.record(); torch.cuda.synchronize(); return a.elapsed_time(b) / it
for rep in range(2):
    for docs in (32768, 16384, 24576, 49152):
        os.environ["LR_FLATIP_PREFIX_DOCS"] = str(docs)
        lr._C.reload_env()
        print(json.dumps({"prefix_docs": docs, "ms": round(t(lambda: lr.flatip_topk(q, c, k)), 3)}), flush=True)
