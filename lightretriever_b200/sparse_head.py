"""Document sparse head (K3) — host side, seam S3.

Mirrors
  * ``get_sparse_attention_mask`` (reference finetune/sparse_pooling.py:23-59) — host logic on torch tensors;
  * ``max_linear_mapping(input, weight[d,V], bias, attention_mask)`` (utils/max_linear_map.py:175-188) and
    ``aggregate(hidden_states, lm_head, sparse_attention_mask)`` (finetune/sparse_pooling.py:244-278);
  * ``HybridModel.get_sparse_emb`` relu / log1p / top-k (finetune/modeling_hybrid.py:183-201,
    finetune/sparse_pooling.py:89-106);
  * ``convert_sparse_reps_to_json`` (finetune/sparse_converter_mixin.py:25-60; rounding follows the in-repo
    torch twin :103-160 — the Rust converter's rounding is not pinned by the reference).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _C
from ._util import Workspace, require_cuda, stream_ptr

_WS = Workspace()


def get_prompt_mask(input_ids: torch.Tensor, sep_token_id: int) -> torch.Tensor:
    """sparse_pooling.py:43-59."""
    assert input_ids.ndim == 2
    if not bool((input_ids == sep_token_id).any()):
        return torch.zeros_like(input_ids, dtype=torch.bool)
    positions = torch.argmax((input_ids == sep_token_id).int(), dim=-1)
    if bool(torch.all(positions == input_ids.shape[-1] - 1)):
        return torch.zeros_like(input_ids, dtype=torch.bool)
    col = torch.arange(input_ids.shape[-1], device=input_ids.device).unsqueeze(0)
    return col <= positions.unsqueeze(1)


def get_sparse_attention_mask(input_ids: torch.Tensor, attention_mask: torch.Tensor, sep_token_id: int,
                              remove_prompt: bool = False) -> torch.Tensor:
    """Valid-token mask: attention mask minus position 0, minus the last valid position, minus the prompt
    (sparse_pooling.py:23-41)."""
    mask = attention_mask.bool().clone()
    if remove_prompt:
        mask = mask.masked_fill(get_prompt_mask(input_ids, sep_token_id), False)
    bs = torch.arange(attention_mask.shape[0], device=attention_mask.device)
    last = attention_mask.sum(dim=1) - 1
    mask[bs, 0] = False
    mask[bs, last] = False
    return mask


def pack_tokens(hidden: torch.Tensor, mask: torch.Tensor, total: Optional[int] = None):
    """hidden [B,S,d] bf16 + mask [B,S] -> (packed [T,d], cu_seqlens int32 [B+1], T): the valid tokens of every document,
    concatenated.  ``total`` = number of valid tokens when the host already knows it (it owns the attention mask before
    the backbone runs); otherwise one 4-byte device->host read."""
    h = require_cuda(hidden, "hidden")
    B, S, d = h.shape
    m = require_cuda(mask, "mask").to(torch.uint8).contiguous()
    cap = int(total) if total is not None else B * S
    packed = torch.empty((max(cap, 1), d), dtype=torch.bfloat16, device=h.device)
    cu = torch.empty(B + 1, dtype=torch.int32, device=h.device)
    lib = _C.load()
    with torch.cuda.device(h.device):
        _C.check(lib.lr_pack_tokens(h.data_ptr(), m.data_ptr(), B, S, d, packed.data_ptr(), cap, cu.data_ptr(),
                                    stream_ptr(h.device)))
    T = int(total) if total is not None else int(cu[-1].item())
    return packed[:max(T, 1)], cu, T


def max_linear_mapping_packed(packed: torch.Tensor, cu_seqlens: torch.Tensor, total: int, weight_vd: torch.Tensor,
                              bias: Optional[torch.Tensor] = None, relu: bool = False, log1p: bool = False) -> torch.Tensor:
    """The same operator over packed tokens: ``packed`` [T, d] bf16 holds only valid tokens, document b = rows
    ``cu_seqlens[b]:cu_seqlens[b+1]``; ``weight_vd`` = ``lm_head.weight`` [V, d].  No padding token is multiplied."""
    h = require_cuda(packed, "packed")
    W = require_cuda(weight_vd, "weight").to(torch.bfloat16).contiguous()
    cu = require_cuda(cu_seqlens, "cu_seqlens").to(torch.int32).contiguous()
    B = cu.numel() - 1
    V, d = W.shape
    if h.dtype != torch.bfloat16 or h.ndim != 2 or h.shape[1] != d or not h.is_contiguous():
        raise ValueError("packed must be a contiguous [T, d] bfloat16 tensor")
    b = None if bias is None else require_cuda(bias, "bias").to(torch.float32).contiguous()
    out = torch.empty((B, V), dtype=torch.float32, device=h.device)
    if total <= 0:  # no valid token at all: every document is the empty-document value (max_linear_map.py:27)
        x = torch.full((B, V), float(torch.finfo(torch.bfloat16).min), dtype=torch.float32, device=h.device)
        if relu:
            x = torch.relu_(x)
        return torch.log1p_(x) if log1p else x
    lib = _C.load()
    ws = _WS.get(lib.lr_sparse_head_packed_workspace_bytes(int(total), V), h.device)
    with torch.cuda.device(h.device):
        _C.check(lib.lr_sparse_head_max_packed(h.data_ptr(), W.data_ptr(), None if b is None else b.data_ptr(),
                                               cu.data_ptr(), B, int(total), d, V, int(relu), int(log1p), out.data_ptr(),
                                               ws.data_ptr(), ws.numel(), stream_ptr(h.device)))
    return out


def max_linear_mapping(input: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                       attention_mask: Optional[torch.Tensor] = None, relu: bool = False, log1p: bool = False,
                       weight_is_vd: bool = False, packed: Optional[bool] = None,
                       valid_tokens: Optional[int] = None) -> torch.Tensor:
    """``max_t (input[b,t] @ weight + bias)`` over valid t -> [B, V] float32 (max_linear_map.py:175-188).

    weight is [d, V] as in the reference (``lm_head.weight.T``); pass ``weight_is_vd=True`` to hand over
    ``lm_head.weight`` ([V, d]) directly and skip the transpose copy.  With a mask the valid tokens are packed first
    (``packed=None``: whenever a mask is given) so that padding is never multiplied; ``valid_tokens`` = ``mask.sum()``
    when the host knows it already.  ``packed=False`` keeps the padded [B, S] layout (mask applied in the epilogue).
    """
    h = require_cuda(input, "input")
    if h.ndim != 3:
        raise ValueError("input must be [B, S, d]")
    B, S, d = h.shape
    W = require_cuda(weight, "weight")
    Wvd = W if weight_is_vd else W.t()
    if Wvd.shape[1] != d:
        raise ValueError("weight shape does not match the hidden size")
    V = Wvd.shape[0]
    h = h.to(torch.bfloat16).contiguous()
    Wvd = Wvd.to(torch.bfloat16).contiguous()
    if attention_mask is not None and attention_mask.shape != (B, S):
        raise ValueError("attention_mask must be [B, S]")
    if packed is None:
        packed = attention_mask is not None
    if packed and attention_mask is not None:
        hp, cu, T = pack_tokens(h, attention_mask, valid_tokens)
        return max_linear_mapping_packed(hp, cu, T, Wvd, bias, relu=relu, log1p=log1p)
    if attention_mask is None:
        mask = torch.ones((B, S), dtype=torch.uint8, device=h.device)
    else:
        mask = require_cuda(attention_mask, "attention_mask").to(torch.uint8).contiguous()
    b = None if bias is None else require_cuda(bias, "bias").to(torch.float32).contiguous()
    out = torch.empty((B, V), dtype=torch.float32, device=h.device)
    lib = _C.load()
    with torch.cuda.device(h.device):
        _C.check(lib.lr_sparse_head_max(h.data_ptr(), Wvd.data_ptr(), None if b is None else b.data_ptr(),
                                        mask.data_ptr(), B, S, d, V, int(relu), int(log1p), out.data_ptr(),
                                        stream_ptr(h.device)))
    return out


def aggregate(hidden_states: torch.Tensor, lm_head, sparse_attention_mask: torch.Tensor,
              sparse_use_max_aggregation: bool = True) -> torch.Tensor:
    """sparse_pooling.py:244-278 for an ``nn.Linear``-like lm_head (``.weight`` [V, d], optional ``.bias``)."""
    if not sparse_use_max_aggregation:
        raise NotImplementedError("mean aggregation is the reference's memory-inefficient ablation; not on the hot path")
    return max_linear_mapping(hidden_states, lm_head.weight, getattr(lm_head, "bias", None), sparse_attention_mask,
                              weight_is_vd=True)


def top_p_sampling(scores: torch.Tensor, top_p: float, filter_value: float = 0.0, min_tokens_to_keep: int = 1,
                   inplace: bool = False) -> torch.Tensor:
    """``top_p_sampling`` (sparse_pooling.py:64-87) on device: entries whose cumulative softmax probability, taken in
    ascending order, stays <= 1 - top_p are set to 0; the ``min_tokens_to_keep`` largest always stay.  Returns a new
    tensor like the reference unless ``inplace``.  Only the reference's ``filter_value = 0`` is built.

    ``min_tokens_to_keep = 0`` keeps every entry: the reference unremoves ``remove[..., -min_tokens_to_keep:]``, and
    ``-0:`` selects every column.  A negative value would make that slice keep all but the first few sorted entries, a
    meaning no caller wants: it raises ``ValueError``."""
    if min_tokens_to_keep < 0:
        raise ValueError(f"top_p_sampling: min_tokens_to_keep ({min_tokens_to_keep}) must be >= 0")
    if top_p <= 0 or top_p >= 1:
        return scores
    if filter_value != 0.0:
        raise NotImplementedError("top_p_sampling: the reference only ever filters to 0")
    x = require_cuda(scores, "scores")
    if x.dtype != torch.float32 or not x.is_contiguous() or not inplace:
        x = x.to(torch.float32).contiguous().clone() if not inplace else x.to(torch.float32).contiguous()
    x2 = x.view(-1, x.shape[-1])
    lib = _C.load()
    with torch.cuda.device(x.device):
        _C.check(lib.lr_top_p_filter(x2.data_ptr(), x2.shape[0], x2.shape[1], float(top_p), int(min_tokens_to_keep),
                                     stream_ptr(x.device)))
    return x


def sparsify_quantize(reps: torch.Tensor, top_k: int = 0, min_tokens_to_keep: int = 8, quantization_factor: float = 100.0,
                      cap: Optional[int] = None):
    """top_k_sampling + clamp/round quantiser -> CSR (indptr int32 [B+1], token ids int32, impacts uint16)."""
    x = require_cuda(reps, "reps").to(torch.float32).contiguous()
    B, V = x.shape
    dev = x.device
    lib = _C.load()
    if cap is None:
        k_eff = max(top_k, min_tokens_to_keep) if top_k > 0 else V
        cap = B * min(V, max(2 * k_eff, k_eff + 1024)) if top_k > 0 else B * V
    indptr = torch.empty(B + 1, dtype=torch.int32, device=dev)
    tok = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    imp = torch.empty(max(cap, 1), dtype=torch.int16, device=dev)  # uint16 bit pattern
    scratch = torch.empty(lib.lr_sparsify_scratch_bytes(B, V), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.lr_sparsify_quantize(x.data_ptr(), B, V, int(top_k), int(min_tokens_to_keep), float(quantization_factor),
                                      indptr.data_ptr(), tok.data_ptr(), imp.data_ptr(), cap, scratch.data_ptr(),
                                      stream_ptr(dev))
    if rc == _C.LR_EWORKSPACE:  # ties at the threshold can exceed any a-priori bound: retry with the exact size
        nnz = int(indptr[-1].item())
        return sparsify_quantize(reps, top_k, min_tokens_to_keep, quantization_factor, cap=nnz)
    _C.check(rc)
    nnz = int(indptr[-1].item())
    return indptr, tok[:nnz], imp[:nnz]


def sparse_head(hidden_states: torch.Tensor, lm_head_weight: torch.Tensor, bias: Optional[torch.Tensor],
                sparse_attention_mask: torch.Tensor, sparse_use_relu: bool = True,
                sparse_use_log_saturation: bool = True, sparse_top_k: int = 0, sparse_min_tokens_to_keep: int = 8,
                quantization_factor: float = 100.0, valid_tokens: Optional[int] = None, sparse_top_p: float = 1.0):
    """hidden [B,S,d] -> CSR of integer impacts: aggregate + get_sparse_emb + convert_sparse_reps_to_json on the device:
    pack the valid tokens, GEMM with max/relu/log1p epilogue over the packed tokens, (top-p,) select/quantise
    (modeling_hybrid.py:183-201 order: relu, log1p, top-p, top-k).
    ``valid_tokens`` = ``sparse_attention_mask.sum()`` when the host knows it (saves a 4-byte read-back)."""
    reps = max_linear_mapping(hidden_states, lm_head_weight, bias, sparse_attention_mask, relu=sparse_use_relu,
                              log1p=sparse_use_log_saturation, weight_is_vd=True, valid_tokens=valid_tokens)
    reps = top_p_sampling(reps, sparse_top_p, min_tokens_to_keep=sparse_min_tokens_to_keep, inplace=True)
    return sparsify_quantize(reps, sparse_top_k, sparse_min_tokens_to_keep, quantization_factor)


def csr_to_json(indptr: torch.Tensor, tok: torch.Tensor, imp: torch.Tensor) -> list[dict[str, int]]:
    """CSR -> the reference's ``list[dict[str(token_id) -> int]]``; an empty document becomes ``{"-1": 1}``
    (sparse_converter_mixin.py:150-156)."""
    ip = indptr.cpu().tolist()
    t = tok.cpu().tolist()
    v = (imp.cpu().to(torch.int32) & 0xFFFF).tolist()
    out = []
    for b in range(len(ip) - 1):
        d = {str(t[i]): int(v[i]) for i in range(ip[b], ip[b + 1])}
        out.append(d if d else {"-1": 1})
    return out


def convert_sparse_reps_to_json(reps: torch.Tensor, quantization_factor: int = 100,
                                convert_id_to_token: bool = False, vocab_dict=None) -> list[dict[str, int]]:
    """sparse_converter_mixin.py:25-60 on device (dense [B,V] in, list of dicts out)."""
    if reps.ndim == 1:
        reps = reps.unsqueeze(0)
    indptr, tok, imp = sparsify_quantize(reps, top_k=0, quantization_factor=float(quantization_factor))
    res = csr_to_json(indptr, tok, imp)
    if convert_id_to_token:
        if vocab_dict is None:
            raise ValueError("vocab_dict is required when convert_id_to_token=True")
        res = [{("[PAD]" if k == "-1" else vocab_dict[int(k)]): v for k, v in d.items()} for d in res]
    return res
