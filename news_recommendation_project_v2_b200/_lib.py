"""ctypes binding of libnrb200.so (the C ABI declared in include/nrb200.h).

There is no fallback: if the library is missing, or a compute call is made
without a B200, this raises.  torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NRB200_LIB") or os.path.join(_PKG, "libnrb200.so")  # NRB200_LIB: A/B experiments only

F32, BF16 = 0, 1
POOL_FINAL_ATTENTION, POOL_MEAN_L2 = 0, 1
EPI_NONE, EPI_RELU, EPI_EXP, EPI_RESIDUAL, EPI_GEGLU, EPI_SOFTMAX = 0, 1, 2, 3, 4, 5
RECOMMEND_MAX_K = 32  # longest list nrb_recommend returns per user

_c_void_p, _i64, _i32, _f32, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t


class LatentWeights(C.Structure):
    """struct nrb_latent_weights (include/nrb200.h)."""

    _fields_ = [
        ("precision", C.c_int), ("dim", C.c_int), ("heads", C.c_int), ("num_latents", C.c_int),
        ("latents_padded", C.c_int),
        ("a", C.c_void_p), ("b", C.c_void_p),
        ("ln1_w", C.c_void_p), ("ln1_b", C.c_void_p), ("ln2_w", C.c_void_p), ("ln2_b", C.c_void_p),
        ("w_ff1", C.c_void_p), ("b_ff1", C.c_void_p), ("w_ff2", C.c_void_p), ("b_ff2", C.c_void_p),
    ]


class PushSeg(C.Structure):
    """struct nrb_push_seg (include/nrb200.h)."""

    _fields_ = [("src", C.c_void_p), ("src_dtype", C.c_int), ("src_stride", C.c_int64), ("mc_dst", C.c_void_p),
                ("dst_dtype", C.c_int), ("dst_stride", C.c_int64), ("dst_row_offset", C.c_int64),
                ("n_rows", C.c_int64), ("dim", C.c_int)]


# name -> (restype, argtypes); must list EVERY symbol of include/nrb200.h (tests check this)
PROTOTYPES = {
    "nrb_version": (C.c_char_p, []),
    "nrb_last_error": (C.c_char_p, []),
    "nrb_check_device": (_i32, [_i32]),
    "nrb_sm_count": (_i32, [_i32]),
    "nrb_kernel_launches": (C.c_longlong, []),
    "nrb_dense_rank": (_i32, [_c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p]),
    "nrb_dense_rank_f64": (_i32, [_c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p]),
    "nrb_narrow_ranks": (_i32, [_c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p]),
    "nrb_topk_order": (_i32, [_c_void_p, _c_void_p, _i64, _i32, _c_void_p, _c_void_p]),
    "nrb_gather_collate": (_i32, [_c_void_p, _i32, _i64, _i32, _i64, _c_void_p, _c_void_p, _i64, _i32,
                                  _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "nrb_mask_to_csr": (_i32, [_c_void_p, _i64, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "nrb_score_rank": (_i32, [_i32, _i32, _i32, _i64, _c_void_p, _c_void_p, _i64, _c_void_p, _i64, _c_void_p, _f32,
                              _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i64,
                              _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "nrb_convert_rows": (_i32, [_c_void_p, _i32, _i64, _c_void_p, _i32, _i64, _i64, _i32, _c_void_p]),
    "nrb_layer_norm": (_i32, [_c_void_p, _i32, _i64, _c_void_p, _c_void_p, _f32, _c_void_p, _i32, _i64, _i64, _i32,
                              _c_void_p]),
    "nrb_linear": (_i32, [_i32, _i32, _i32, _c_void_p, _i64, _c_void_p, _i64, _c_void_p, _c_void_p, _i64,
                          _c_void_p, _i64, _i64, _i32, _i32, _i32, _i32, _c_void_p]),
    "nrb_final_attention_rows_workspace_bytes": (_sz, [_i32, _i64, _i32, _i32]),
    "nrb_final_attention_rows": (_i32, [_i32, _i32, _c_void_p, _i64, _i64, _i32, _i32,
                                        _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                                        _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i64,
                                        _c_void_p, _sz, _c_void_p]),
    "nrb_split_rows": (_i32, [_c_void_p, _i64, _c_void_p, _i64, _i64, _i32, _i32, _c_void_p]),
    "nrb_final_attention_rows_split_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "nrb_final_attention_rows_split": (_i32, [_c_void_p, _i64, _i64, _i32, _i32] + [_c_void_p] * 9 +
                                       [_c_void_p, _c_void_p, _i64, _c_void_p, _sz, _c_void_p]),
    "nrb_latent_fold_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "nrb_latent_fold": (_i32, [_i32, _i32, _i32, _i32, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                               _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _sz, _c_void_p]),
    "nrb_latent_forward_workspace_bytes": (_sz, [C.POINTER(LatentWeights), _i64]),
    "nrb_mind_metrics": (_i32, [_c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p]),
    "nrb_push_rows": (_i32, [_c_void_p, _i32, _i64, _i64, _i32, C.POINTER(C.c_void_p), _i32, _i32, _i64, _i64,
                             _c_void_p]),
    "nrb_push_bytes": (_i32, [_c_void_p, _i64, C.POINTER(C.c_void_p), _i32, _i64, _c_void_p]),
    "nrb_push_attach": (_i32, [C.POINTER(PushSeg), _i32, _i32]),
    "nrb_push_flush": (_i32, [_c_void_p]),
    "nrb_push_cancel": (None, []),
    "nrb_host_copy": (_i32, [_c_void_p, _c_void_p, _i64, _i32]),
    "nrb_csr_build": (_c_void_p, [C.c_char_p, _i64, C.c_char_p, _i64, _i64]),
    "nrb_csr_sizes": (_i32, [_c_void_p, C.POINTER(_i64)]),
    "nrb_csr_export": (_i32, [_c_void_p] * 8),
    "nrb_csr_news_ids": (_i64, [_c_void_p, _c_void_p, _i64]),
    "nrb_csr_free": (None, [_c_void_p]),
    "nrb_latent_forward_packed": (_i32, [C.POINTER(LatentWeights), _c_void_p, _i32, _i64, _c_void_p, _i64,
                                         _c_void_p, _c_void_p, _sz, _c_void_p]),
    "nrb_latent_forward": (_i32, [C.POINTER(LatentWeights), _c_void_p, _i32, _i64, _i32, _c_void_p,
                                  _c_void_p, _c_void_p, _c_void_p, _sz, _i64, C.POINTER(_i64), _c_void_p]),
    "nrb_recommend_workspace_bytes": (_sz, [_i32, _i32, _i64, _i64, _i64, _i32]),
    "nrb_recommend": (_i32, [_i32, _i32, _i64, _c_void_p, _i64, _c_void_p, _i64, _c_void_p, _i64, _i64,
                             _c_void_p, _c_void_p, _i64, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _sz,
                             _c_void_p]),
    "nrb_recommend_pool_blend_workspace_bytes": (_sz, [_i32, _i32, _i64, _i64, _i64, _i32, _i64]),
    "nrb_recommend_pool_blend": (_i32, [_i32, _i32, _i64, _c_void_p, _i64, _c_void_p, _i64, _c_void_p, _i64, _i64,
                                        _c_void_p, _c_void_p, _i64, _i32, _c_void_p, _i64, _c_void_p, _f32,
                                        _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _sz, _c_void_p]),
}

_lock = threading.Lock()
_lib = None


class NrbError(RuntimeError):
    pass


def load():
    """dlopen libnrb200.so and bind every prototype.  Loud failure, no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NrbError(
                f"{LIB_PATH} is missing: build it with `python -m news_recommendation_project_v2_b200.build` "
                "(there is no CPU / PyTorch fallback for the hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().nrb_last_error().decode(errors="replace")
        raise NrbError(f"{what or 'nrb200'} failed (code {rc}): {msg}")


_device_ok: dict[int, bool] = {}


def require_device(device: torch.device | None = None) -> torch.device:
    """Return the CUDA device to run on; raise unless it is a B200-class (sm_100) GPU."""
    if not torch.cuda.is_available():
        raise NrbError("no CUDA device visible: the nrb200 hot path has no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise NrbError(f"nrb200 needs a CUDA device, got {dev}")
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx not in _device_ok:
        check(load().nrb_check_device(idx), "nrb_check_device")
        _device_ok[idx] = True
    return torch.device("cuda", idx)


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise NrbError(f"unsupported dtype {dt} (float32 or bfloat16)")


def torch_dtype(code: int) -> torch.dtype:
    return torch.float32 if code == F32 else torch.bfloat16


def ptr(t: torch.Tensor | None) -> int | None:
    if t is None:
        return None
    return t.data_ptr()
