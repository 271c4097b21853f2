"""Worker of tests/test_online_hybrid.py::test_online_hybrid_over_nccl: one process per GPU under torch.distributed.run
(NCCL).  Every rank holds its dense and sparse shard (shard_range) of the same seeded documents and serves requests
through OnlineHybridSearcher: results must be identical on all ranks, the sparse half bit-exact against the unsharded
oracle, the dense half within the tie rule, the fusion bit-exact against oracle fusion of the merged lists, and each
step must exchange candidates exactly once.  The process ends as bench.py's online configs do (barrier, flush,
os._exit): the captured graphs hold NCCL collectives, and the communicator is not torn down under them."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    rank, local, world = (int(os.environ[k]) for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import lightretriever_b200 as lr
    from lightretriever_b200 import online
    from lightretriever_b200.sparse_search import json_to_csr
    from oracle import oracle

    N, d, V, k, B = 30_001, 256, 3000, 100, 8
    gen = torch.Generator().manual_seed(13)  # same data on every rank
    table = (torch.randn(V, d, generator=gen) * 0.02).bfloat16().to(dev)
    corpus = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16()
    rng = np.random.default_rng(14)
    steps = rng.integers(1, 150, (N, 16)).cumsum(1)
    tok = (rng.integers(0, V, (N, 1)) + steps) % V
    imp = rng.integers(1, 400, (N, 16))
    docs = [dict(zip(t.tolist(), m.tolist())) for t, m in zip(tok, imp)]
    lo, hi = lr.shard_range(N, rank, world)
    index = lr.ImpactIndex(V, device=dev, id_offset=lo)
    index.add_csr(*json_to_csr(docs[lo:hi]))
    shard = corpus[lo:hi].to(dev)
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)

    calls = []
    real_exchange = online.exchange_candidates

    def counting_exchange(keys, group=None):
        calls.append(tuple(keys.shape))
        return real_exchange(keys, group)

    hgen = torch.Generator().manual_seed(15)
    for method in ("linear", "rrf"):
        srv = lr.OnlineHybridSearcher(bag, shard, index, k, batch=B, max_tokens=B * 32, id_offset=lo, method=method)
        for n in (8, 3):
            lens = torch.randint(1, 33, (n,), generator=hgen)
            ids = torch.randint(0, V - 1, (int(lens.sum()),), generator=hgen)
            offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0)
            (ds, di), (ss, si), (fi, fs, fc) = (tuple(t.clone() for t in part)
                                                for part in srv.search(ids.to(dev), offs.to(dev)))
            # exactly one exchange per step (eager path, same staged request)
            online.exchange_candidates = counting_exchange
            try:
                calls.clear()
                eager = srv._step()
            finally:
                online.exchange_candidates = real_exchange
            assert calls == [(2, B, k)], calls
            assert torch.equal(eager[0][1][:n], di) and torch.equal(eager[1][1][:n], si)
            # identical on every rank
            mine = torch.cat([ds.double().flatten(), di.double().flatten(), ss.double().flatten(), si.double().flatten(),
                              fi.double().flatten(), fs.flatten(), fc.double()])
            other = mine.clone()
            dist.broadcast(other, src=0)
            assert torch.equal(mine.nan_to_num(), other.nan_to_num()), "ranks disagree"
            # dense: tie rule against the unsharded fp32 reference
            qv = bag.encode(ids.to(dev), offs.to(dev), normalize=True).float().cpu()
            ref = (qv @ corpus.float().T).numpy()
            oracle.check_topk_parity(ds.cpu().numpy(), di.cpu().numpy(), ref, k, rtol=1e-2)
            # sparse: bit-exact against the unsharded oracle
            ends = offs.tolist()[1:] + [ids.numel()]
            qs = [oracle.query_counts(ids[a:b].tolist()) for a, b in zip(offs.tolist(), ends)]
            es, ei = oracle.impact_topk(qs, docs, k)
            assert (si.cpu().numpy() == ei).all() and (ss.cpu().numpy() == es).all()
            # fusion: bit-exact against oracle fusion of the merged lists
            for q in range(n):
                systems = []
                for s_, i_ in ((ds[q].cpu().numpy(), di[q].cpu().numpy()), (ss[q].cpu().numpy(), si[q].cpu().numpy())):
                    keep = i_ >= 0
                    if not keep.any():
                        systems.append({})
                    elif method == "linear":
                        systems.append({"q": {str(a): float(b) for a, b in zip(i_[keep], s_[keep])}})
                    else:
                        systems.append({"q": {str(a): -float(r) for r, a in enumerate(i_[keep])}})
                fref = (oracle.fuse_linear(systems, weights=[0.7, 0.3]) if method == "linear"
                        else oracle.fuse_rrf(systems)).get("q", {})
                m = int(fc[q])
                assert m == len(fref)
                got = {str(a): b for a, b in zip(fi[q, :m].tolist(), fs[q, :m].tolist())}
                assert got == fref, (method, q)
        del srv

    dist.barrier()
    if rank == 0:
        print(f"nccl hybrid worker OK world={world}", flush=True)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == "__main__":
    main()
