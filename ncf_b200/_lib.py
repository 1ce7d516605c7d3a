"""ctypes binding of the C ABI declared in include/ncf_b200.h.

This is the stub a reference maintainer would add (see INTEGRATION.md): plain pointers and sizes,
`tensor.data_ptr()` for device memory and `torch.cuda.current_stream().cuda_stream` for the stream.
There is no CPU fallback — a missing library or a failing call raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

NCF_MAX_LAYERS = 8
NCF_GMF, NCF_MLP, NCF_NEUMF = 0, 1, 2
MODEL_TYPES = {"GMF": NCF_GMF, "MLP": NCF_MLP, "NeuMF-end": NCF_NEUMF, "NeuMF-pre": NCF_NEUMF}

_f = C.c_void_p  # device pointers travel as integers


class NcfModel(C.Structure):
    _fields_ = [
        ("model_type", C.c_int32), ("factor_num", C.c_int32), ("num_layers", C.c_int32),
        ("mlp_dim", C.c_int32), ("tower_math", C.c_int32), ("reserved", C.c_int32),
        ("user_num", C.c_int64), ("item_num", C.c_int64),
        ("embed_user_gmf", _f), ("embed_item_gmf", _f), ("embed_user_mlp", _f), ("embed_item_mlp", _f),
        ("mlp_w", _f * NCF_MAX_LAYERS), ("mlp_b", _f * NCF_MAX_LAYERS),
        ("predict_w", _f), ("predict_b", _f),
    ]


class NcfGrads(C.Structure):
    _fields_ = [
        ("g_user_gmf", _f), ("g_item_gmf", _f), ("g_user_mlp", _f), ("g_item_mlp", _f),
        ("g_tower", _f), ("user_flag", _f), ("item_flag", _f), ("user_list", _f), ("item_list", _f),
        ("touched_count", _f),
    ]


class NcfAdamState(C.Structure):
    _fields_ = [
        ("m_user_gmf", _f), ("v_user_gmf", _f), ("m_item_gmf", _f), ("v_item_gmf", _f),
        ("m_user_mlp", _f), ("v_user_mlp", _f), ("m_item_mlp", _f), ("v_item_mlp", _f),
        ("m_tower", _f), ("v_tower", _f), ("user_last_step", _f), ("item_last_step", _f), ("step", _f),
    ]


class NcfAdamHyper(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float)]


_P = C.POINTER
_i64, _i32, _u64, _vp, _fl = C.c_int64, C.c_int32, C.c_uint64, C.c_void_p, C.c_float

# name -> (restype, argtypes); the single source of truth for the exported surface, checked
# against include/ncf_b200.h by tests/test_abi.py.
SIGNATURES = {
    "ncf_version": (C.c_int, []),
    "ncf_last_error": (C.c_char_p, []),
    "ncf_last_tile_path": (C.c_int, []),
    "ncf_wait_embedding_grads": (C.c_int, [_vp]),
    "ncf_profile_enable": (C.c_int, [_i32]),
    "ncf_profile_read": (C.c_int, [_vp, _vp, _i32, _i32]),
    "ncf_tower_param_count": (_i64, [_i32, _i32, _i32]),
    "ncf_csr_workspace_bytes": (_i64, [_i64, _i64]),
    "ncf_csr_build": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ncf_text_workspace_bytes": (_i64, [_i64]),
    "ncf_text_line_starts": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp]),
    "ncf_text_parse_ints": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "ncf_split_workspace_bytes": (_i64, [_i64, _i64]),
    "ncf_leave_one_out_split": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ncf_eval_negatives": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i32, _u64, _vp, _vp, _vp]),
    "ncf_sample_neg": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i32, _i64, _u64, _u64, _vp, _vp]),
    "ncf_shuffle_epoch": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _u64, _u64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "ncf_forward_workspace_bytes": (_i64, [_P(NcfModel), _i64]),
    "ncf_forward": (C.c_int, [_P(NcfModel), _vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "ncf_loss_grad": (C.c_int, [_vp, _vp, _vp, _fl, _i64, _vp, _vp, _vp]),
    "ncf_loss_grad_kd": (C.c_int, [_vp, _vp, _vp, _fl, _fl, _fl, _i32, _i64, _vp, _vp, _vp]),
    "ncf_feature_kd": (C.c_int, [_P(NcfModel), _P(NcfModel), _P(NcfGrads), _vp, _vp, _i64, _i32, _vp, _vp, _fl, _vp, _vp]),
    "ncf_train_workspace_bytes": (_i64, [_P(NcfModel), _i64]),
    "ncf_train_step_grads": (C.c_int, [_P(NcfModel), _P(NcfGrads), _vp, _vp, _vp, _vp, _fl, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ncf_train_step_grads_norm": (C.c_int, [_P(NcfModel), _P(NcfGrads), _vp, _vp, _vp, _vp, _fl, _i64, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ncf_mark_rows_side": (C.c_int, [_P(NcfModel), _P(NcfGrads), _vp, _i64, _i32, _vp]),
    "ncf_adam_catchup": (C.c_int, [_P(NcfModel), _P(NcfGrads), _P(NcfAdamState), NcfAdamHyper, _vp]),
    "ncf_bucket_by_owner": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ncf_permute_i64": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "ncf_permute_f32": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "ncf_gather_rows": (C.c_int, [_vp, _vp, _i64, _i32, _i64, _vp, _vp]),
    "ncf_scatter_add_rows": (C.c_int, [_vp, _vp, _i64, _i32, _i64, _vp, _vp]),
    "ncf_shard_request": (C.c_int, [_vp, _i64, _i32, _i32, _i64, _i64, _vp, _vp, _vp, _vp]),
    "ncf_shard_mark_requests": (C.c_int, [_P(NcfModel), _P(NcfGrads), _vp, _vp, _i32, _i64, _vp]),
    "ncf_shard_push_rows": (C.c_int, [_P(NcfModel), _vp, _vp, _i32, _i64, _vp, _vp, _vp]),
    "ncf_shard_push_grads": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "ncf_backward": (C.c_int, [_P(NcfModel), _P(NcfGrads), _vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "ncf_mark_rows": (C.c_int, [_P(NcfModel), _P(NcfGrads), _vp, _vp, _i64, _vp]),
    "ncf_adam_prepare": (C.c_int, [_P(NcfModel), _P(NcfGrads), _P(NcfAdamState), NcfAdamHyper, _vp, _vp, _i64, _vp]),
    "ncf_adam_step": (C.c_int, [_P(NcfModel), _P(NcfGrads), _P(NcfAdamState), NcfAdamHyper, _vp]),
    "ncf_adam_step_dense": (C.c_int, [_P(NcfModel), _P(NcfGrads), _P(NcfAdamState), NcfAdamHyper, _vp]),
    "ncf_adam_step_dense_range": (C.c_int, [_P(NcfModel), _P(NcfGrads), _P(NcfAdamState), NcfAdamHyper, _i64, _i64, _i32, _vp]),
    "ncf_adam_range": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, NcfAdamHyper, _vp]),
    "ncf_adam_finish_dense": (C.c_int, [_P(NcfModel), _P(NcfGrads), _P(NcfAdamState), _vp]),
    "ncf_adam_p2p": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32, _fl, _vp, NcfAdamHyper, _vp]),
    "ncf_peer_barrier": (C.c_int, [_vp, _i32, _i32, _vp, _vp]),
    "ncf_peer_alloc": (C.c_int, [_i64, _vp]),
    "ncf_peer_free": (C.c_int, [_vp]),
    "ncf_ipc_export": (C.c_int, [_vp, _vp]),
    "ncf_ipc_open": (C.c_int, [_vp, _vp]),
    "ncf_ipc_close": (C.c_int, [_vp]),
    "ncf_adam_flush": (C.c_int, [_P(NcfModel), _P(NcfAdamState), NcfAdamHyper, _vp]),
    "ncf_sgd_step": (C.c_int, [_P(NcfModel), _P(NcfGrads), _fl, _vp]),
    "ncf_eval_rank": (C.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ncf_eval_workspace_bytes": (_i64, [_P(NcfModel), _i64, _i32]),
    "ncf_eval_users": (C.c_int, [_P(NcfModel), _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ncf_mask_items": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp]),
    "ncf_topk_rows_workspace_bytes": (_i64, [_i64, _i64, _i32]),
    "ncf_topk_rows": (C.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ncf_recommend_workspace_bytes": (_i64, [_P(NcfModel), _i64, _i32]),
    "ncf_recommend": (C.c_int, [_P(NcfModel), _vp, _i64, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp]),
}

LIB_PATH = Path(__file__).resolve().parent / "libncf_b200.so"
_lib = None


class NcfError(RuntimeError):
    """A C-ABI call returned a non-zero status."""


def load(build_if_missing: bool = True) -> C.CDLL:
    """Loads (building first if needed) the in-tree CUDA library.  Never falls back to CPU."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise NcfError(f"{LIB_PATH} is missing: run `python -m ncf_b200.build`")
        from . import build as _build
        _build.build()
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError => the library does not match the header
        fn.restype = res
        fn.argtypes = args
    if lib.ncf_version() != 1:
        raise NcfError(f"ABI version mismatch: library reports {lib.ncf_version()}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().ncf_last_error().decode(errors="replace")
        raise NcfError(f"{what} failed with status {rc}: {msg}")


def ptr(t) -> int:
    """Device pointer of a tensor (None -> NULL).  Refuses non-CUDA / non-contiguous tensors."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NcfError("ncf_b200 kernels need CUDA tensors; there is no CPU path")
    if not t.is_contiguous():
        raise NcfError("ncf_b200 kernels need contiguous tensors")
    return t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
