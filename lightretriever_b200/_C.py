"""ctypes binding of liblr_b200.so (the C ABI declared in include/lr_b200.h).

There is no CPU fallback: if the shared object is missing the import of any compute wrapper raises, and every
compute call on a box without a CUDA device raises RuntimeError (the library returns LR_ECUDA).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "liblr_b200.so"

LR_OK, LR_EINVAL, LR_ECUDA, LR_EWORKSPACE = 0, -1, -2, -3
LR_F32, LR_BF16 = 0, 1
LR_SCORE_F32, LR_SCORE_U32 = 0, 1

_vp, _i64, _i32, _sz, _f32 = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_float

# name -> (restype, argtypes); must list every function declared in include/lr_b200.h
PROTOTYPES = {
    "lr_last_error": (C.c_char_p, []),
    "lr_version": (_i32, []),
    "lr_device_sm_count": (_i32, []),
    "lr_reload_env": (_i32, []),
    "lr_embbag_encode": (_i32, [_vp, _vp, _i64, _i64, _vp, _i32, _i64, _i64, _i64, _i64, _i32, _vp, _i32, _vp, _vp]),
    "lr_lasttoken_head": (_i32, [_vp, _i32, _vp, _i64, _i64, _i64, _i64, _i32, _vp, _i32, _vp, _vp]),
    "lr_flatip_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "lr_flatip_workspace_bytes_for": (_sz, [_i64, _i64, _i32, _i64]),
    "lr_flatip_topk": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lr_flatip_workspace_bytes_sharded": (_sz, [_i64, _i64, _i32, _i64, _i32]),
    "lr_flatip_topk_begin": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "lr_flatip_topk_finish": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp,
                                     _vp, _sz, _vp]),
    "lr_flatip_plan_passes_sharded": (_i32, [_i64, _i64, _i32, _i64, _i32, _vp, _i32, _vp]),
    "lr_flatip_scores": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "lr_flatip_last_plan": (_i32, [_vp]),
    "lr_flatip_last_plan_passes": (_i32, [_vp, _i32]),
    "lr_kernel_launches": (C.c_ulonglong, []),
    "lr_flatip_plan": (_i32, [_i64, _i64, _i32, _vp]),
    "lr_flatip_plan_passes": (_i32, [_i64, _i64, _i32, _i64, _vp, _i32, _vp]),
    "lr_set_profile_events": (_i32, [_vp, _vp]),
    "lr_topk_merge": (_i32, [_vp, _vp, _i32, _i64, _i64, _i32, _i32, _i32, _i64, _vp, _vp, _vp, _vp]),
    "lr_encode_keys": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "lr_fuse_topk": (_i32, [_vp, _vp, _i32, _vp, _vp, _i32, _i64, _i32, C.c_double, C.c_double, C.c_double, C.c_double,
                            _vp, _vp, _vp, _vp]),
    "lr_fuse_topk_f64": (_i32, [_vp, _vp, _i32, _vp, _vp, _i32, _i64, _i32, C.c_double, C.c_double, C.c_double, C.c_double,
                                _vp, _vp, _vp, _vp]),
    "lr_sparse_head_max": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _vp, _vp]),
    "lr_sparse_head_packed_workspace_bytes": (_sz, [_i64, _i64]),
    "lr_sparse_head_packed_plan": (_i32, [_i64, _i64, _vp]),
    "lr_sparse_head_max_packed": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    "lr_top_p_filter": (_i32, [_vp, _i64, _i64, _f32, _i32, _vp]),
    "lr_pack_tokens": (_i32, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp]),
    "lr_sparsify_scratch_bytes": (_sz, [_i64, _i64]),
    "lr_sparsify_quantize": (_i32, [_vp, _i64, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _i64, _vp, _vp]),
    "lr_sparse_block_docs": (_i32, []),
    "lr_sparse_build_blockptr": (_i32, [_vp, _vp, _i64, _i64, _vp, _vp]),
    "lr_sparse_score_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "lr_sparse_score_plan": (_i32, [_i64, _i64, _i32, _vp]),
    "lr_sparse_score_topk": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lr_flatip_topk_filtered": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i32, _vp, _vp, _vp,
                                       _vp, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "lr_flatip_topk_begin_filtered": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i32, _i32, _vp,
                                             _vp, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "lr_flatip_topk_finish_filtered": (_i32, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i32, _i32, _vp,
                                              _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "lr_sparse_score_topk_filtered": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _vp, _vp,
                                             _vp, _vp, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "lr_doc_bitmap_update": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp]),
    "lr_query_token_counts_scratch_bytes": (_sz, [_i64, _i64]),
    "lr_query_token_counts": (_i32, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
}

_lib = None


def load(build_if_missing: bool | None = None) -> C.CDLL:
    """Load the shared object (building it in-tree with nvcc when stale and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing is None:
        build_if_missing = os.environ.get("LR_B200_NO_BUILD", "0") != "1"
    if build_if_missing:
        from . import build as _build
        if _build.is_stale():
            try:
                _build.build()
            except Exception as e:
                # never run kernels that do not match the sources silently: a stale library is an error unless the
                # caller explicitly accepts it (LR_B200_ALLOW_STALE=1, e.g. a box without nvcc)
                if not LIB_PATH.exists():
                    raise RuntimeError(f"liblr_b200.so is missing and could not be built: {e}") from e
                if os.environ.get("LR_B200_ALLOW_STALE", "0") != "1":
                    raise RuntimeError(f"liblr_b200.so is older than its sources and the rebuild failed "
                                       f"(set LR_B200_ALLOW_STALE=1 to load it anyway): {e}") from e
                import warnings
                warnings.warn(f"loading a STALE liblr_b200.so (rebuild failed: {e})", RuntimeWarning)
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m lightretriever_b200.build` "
            "(there is no CPU/PyTorch fallback for the retrieval kernels)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def reload_env() -> None:
    """Make the library re-read its LR_* experiment knobs (they are cached after the first call)."""
    load().lr_reload_env()


def last_error() -> str:
    return load().lr_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Map the C ABI's return codes onto the exceptions the reference raises (ValueError / RuntimeError)."""
    if rc == LR_OK:
        return
    msg = last_error()
    if rc in (LR_EINVAL, LR_EWORKSPACE):
        raise ValueError(msg)
    raise RuntimeError(msg)
