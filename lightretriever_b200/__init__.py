"""lightretriever_b200 — B200-native serving-side retrieval hot path of caskcsg/lightretriever.

Hand-written sm_100a CUDA kernels (csrc/) behind a C ABI (include/lr_b200.h, liblr_b200.so), driven by a thin Python
host layer that keeps the reference's encode / index / retrieve_with_emb / search interfaces.  No CPU fallback.
"""
from . import _C  # noqa: F401  (ctypes binding; `_C.load()` builds/loads liblr_b200.so)
from .encode import (B200EmbeddingBag, construct_embedding_bag, emb_bag_inputs, flatten_token_ids, lasttoken_head,
                     tokenize_nonctx_qry_emb_bag)
from .search import (FlatIPIndex, FlatIPSearch, decode_keys, drop_identical, encode_keys, flatip_scores, flatip_topk,
                     flatip_topk_sharded, merge_keys, topk_merge)
from .sharded import ShardedFlatIPIndex, ShardedImpactIndex, exchange_candidates, shard_range
from .sparse_head import (aggregate, convert_sparse_reps_to_json, csr_to_json, get_sparse_attention_mask,
                          max_linear_mapping, max_linear_mapping_packed, pack_tokens, sparse_head, sparsify_quantize,
                          top_p_sampling)
from .sparse_search import ImpactIndex, ImpactSearch, query_token_counts
from .online import OnlineHybridSearcher, OnlineSearcher
from .hybrid import HybridSearch, fuse_scores_linear, fuse_scores_rrf, fuse_topk_device

__version__ = "0.1.0"
