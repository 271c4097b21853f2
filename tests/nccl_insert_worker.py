"""Worker of tests/test_online_inserts.py::test_inserts_over_nccl: one process per GPU under torch.distributed.run (NCCL).
Every rank holds its dense and sparse shard of the same seeded documents, a delta segment with its own id range
(n_total + rank * cap) and inserts its own documents.  Every rank must return the same fused result, equal bit for bit
to the public single-GPU calls over all documents (main shards + both deltas, unfilled slots deleted)."""
import os
import sys

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
    from lightretriever_b200.filters import doc_bitmap

    N, d, V, L, k, B, cap = 30_001, 256, 3000, 16, 100, 8, 512
    gen = torch.Generator().manual_seed(13)  # same data on every rank
    table = (torch.randn(V, d, generator=gen) * 0.02).bfloat16().to(dev)
    corpus = F.normalize(torch.randn(N, d, generator=gen), dim=-1).bfloat16().to(dev)
    tok = torch.randint(0, V, (N, L), generator=gen, dtype=torch.int32).to(dev)
    imp = torch.randint(1, 401, (N, L), generator=gen, dtype=torch.int32).to(dev)
    n_ins = (300, 200)
    new_rows = [F.normalize(torch.randn(n, d, generator=gen), dim=-1).bfloat16().to(dev) for n in n_ins]
    new_tok = [torch.randint(0, V, (n, L), generator=gen, dtype=torch.int32).to(dev) for n in n_ins]
    new_imp = [torch.randint(1, 2001, (n, L), generator=gen, dtype=torch.int32).to(dev) for n in n_ins]

    def csr(t, m):
        return torch.arange(0, t.numel() + 1, t.shape[1], dtype=torch.int64), t.reshape(-1), m.reshape(-1)

    lo, hi = lr.shard_range(N, rank, world)
    index = lr.ImpactIndex(V, device=dev, id_offset=lo)
    index.add_csr(*csr(tok[lo:hi], imp[lo:hi]))
    bag = lr.B200EmbeddingBag.from_pretrained(table, padding_idx=V - 1)
    srv = lr.OnlineHybridSearcher(bag, corpus[lo:hi], index, k, batch=B, max_tokens=B * 32, id_offset=lo,
                                  live=doc_bitmap(N + world * cap, torch.arange(N), device=dev), insert_capacity=cap,
                                  insert_id_base=N + rank * cap)
    ids = srv.insert(new_rows[rank], *csr(new_tok[rank], new_imp[rank]))
    assert ids.tolist() == list(range(N + rank * cap, N + rank * cap + n_ins[rank]))

    # single-GPU oracle: every document at its global id, the unfilled delta slots deleted
    full = torch.zeros((N + world * cap, d), dtype=torch.bfloat16, device=dev)
    ftok = torch.zeros((N + world * cap, L), dtype=torch.int32, device=dev)
    fimp = torch.zeros_like(ftok)
    full[:N], ftok[:N], fimp[:N] = corpus, tok, imp
    filled = [torch.arange(N)]
    for r in range(world):
        a = N + r * cap
        full[a:a + n_ins[r]], ftok[a:a + n_ins[r]], fimp[a:a + n_ins[r]] = new_rows[r], new_tok[r], new_imp[r]
        filled.append(torch.arange(a, a + n_ins[r]))
    live = doc_bitmap(N + world * cap, torch.cat(filled), device=dev)
    oindex = lr.ImpactIndex(V, device=dev)
    oindex.add_csr(*csr(ftok, fimp))

    hgen = torch.Generator().manual_seed(15)
    for n in (8, 3):
        lens = torch.randint(1, 33, (n,), generator=hgen)
        qids = torch.randint(0, V - 1, (int(lens.sum()),), generator=hgen).to(dev)
        offs = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.long), lens[:-1]]), 0).to(dev)
        got = tuple(tuple(t.clone() for t in part) for part in srv.search(qids, offs))
        mine = torch.cat([t.double().flatten() for part in got for t in part])
        other = mine.clone()
        dist.broadcast(other, src=0)
        assert torch.equal(mine.nan_to_num(), other.nan_to_num()), "ranks disagree"
        qv = bag.encode(qids, offs, normalize=True)
        dense = lr.flatip_topk(qv, full, k, live=live)
        sparse = oindex.search_device(*lr.query_token_counts(qids, offs, V), k, live=live)
        fused = lr.fuse_topk_device(*dense, *sparse, method="linear", weights=(0.7, 0.3))
        for a, b in zip(got, (dense, sparse, fused)):
            assert all(torch.equal(x, y) for x, y in zip(a, b)), n
        assert (got[1][1] >= N).any(), "no inserted document reached the sparse top-k"
    del srv

    dist.barrier()
    if rank == 0:
        print(f"nccl insert worker OK world={world}", flush=True)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == "__main__":
    main()
