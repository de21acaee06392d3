"""ctypes binding of the C ABI declared in ``include/mae_clip_b200.h``.

PyTorch is only the owner of device memory and streams: every call below passes raw device
pointers (``tensor.data_ptr()``), sizes and the current ``cudaStream_t``.  There is NO fallback:
if the shared library is missing, or the device is not sm_100, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
# MAE_CLIP_B200_LIB: load another build of the same ABI (A/B timing of kernel variants); never a fallback
LIB_PATH = os.environ.get("MAE_CLIP_B200_LIB") or os.path.join(_PKG, "libmae_clip_b200.so")

GEMM_SIMT_FP32 = 0
GEMM_TC_F16X3 = 1
GEMM_TC_F16 = 2
GEMM_MODES = {"simt_fp32": GEMM_SIMT_FP32, "tc_f16x3": GEMM_TC_F16X3, "tc_f16": GEMM_TC_F16}

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_f = C.c_float
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors include/mae_clip_b200.h one to one
SIGNATURES = {
    "mc_version": (_i, []),
    "mc_last_error_string": (C.c_char_p, []),
    "mc_device_supported": (_i, [_i]),
    "mc_kernel_launch_count": (C.c_ulonglong, []),
    "mc_soft_ce_workspace_bytes": (_sz, [_i, _i]),
    "mc_soft_ce_fwd": (_i, [_p, _i64, _i64, _p, _i64, _i64, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "mc_soft_ce_bwd": (_i, [_p, _i64, _i64, _p, _i64, _i64, _i, _i, _p, _p, _p, _p, _i64, _i64, _p,
                            _i64, _i64, _p]),
    "mc_clip_loss_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mc_clip_planes_bytes": (_sz, [_i, _i, _i]),
    "mc_clip_prepare": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "mc_clip_amax": (_i, [_p, _p, _i, _i, _p, _p, _p, _p]),
    "mc_clip_push_shards": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "mc_clip_prepare_peers": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "mc_peer_alloc": (_i, [_sz, _p, _p]),
    "mc_peer_open": (_i, [_p, _p]),
    "mc_peer_close": (_i, [_p]),
    "mc_peer_free": (_i, [_p]),
    "mc_peer_barrier": (_i, [_p, _i, _i, _p, C.c_double, _p]),
    "mc_peer_publish": (_i, [_p, _i, _i, _i64, _p, _i64, _i64, _i, _p]),
    "mc_peer_reduce": (_i, [_p, _i, _sz, _p, _p, _p]),
    "mc_clip_tile_flags_bytes": (_sz, [_i, _i, _i, _i]),
    "mc_clip_flags_finalize": (_i, [_p, _i, _i, _i, _p, _p]),
    "mc_clip_stats": (_i, [_p, _p, _p, _i, _i, _i, _i, _f, _i, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mc_clip_stats_colpart_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mc_clip_stats_colpart": (_i, [_p, _i, _i, _i, _i, _f, _i, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mc_clip_colpart_merge": (_i, [_p, _i, _i64, _i, _p, _p]),
    "mc_clip_rowloss": (_i, [_p, _p, _p, _i, _i, _i, _i, _f, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mc_clip_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _f, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz,
                         _p]),
    "mc_clip_stored_weights_bytes": (_sz, [_i, _i]),
    "mc_clip_bwd_cols_workspace_bytes": (_sz, [_i, _i]),
    "mc_clip_bwd_gate": (_i, [_p, _sz, _p, _p]),
    "mc_clip_bwd_rows": (_i, [_p, _i, _i, _i, _i, _f, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz,
                              _p]),
    "mc_clip_bwd_cols": (_i, [_p, _i, _i, _f, _i, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "mc_clip_loss_fused_workspace_bytes": (_sz, [_i, _i, _i]),
    "mc_clip_loss_fwd_bwd": (_i, [_p, _p, _i, _i, _f, _i, _p, _p, _p, _p, _sz, _p]),
    "mc_clip_loss_host_workspace_bytes": (_sz, [_i, _i, _i]),
    "mc_clip_loss_fwd_bwd_host": (_i, [_p, _p, _i, _i, _f, _i, _p, _p, _p, _p, _sz, _p]),
    "mc_proj_head_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mc_proj_head_fwd": (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _f, _f, _i, _p, _p, _p, _p,
                              _p, _p, _p, _p, _p, _sz, _p]),
    "mc_proj_head_bwd": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _f, _i, _p, _p, _p, _p, _p, _p, _p,
                              _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mc_tc_gemm_workspace_bytes": (_sz, [_i, _i, _i]),
    "mc_tc_gemm": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "mc_head_gemm_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mc_head_gemm": (_i, [_i, _p, _p, _i, _i, _i, _p, _p, _p, _i, _p, _sz, _p]),
    "mc_random_masking": (_i, [_p, _i, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "mc_random_masking_bwd": (_i, [_p, _i, _p, _p, _i, _i, _i, _i, _p, _p]),
    "mc_masked_mse_workspace_bytes": (_sz, [_i, _i]),
    "mc_masked_mse_fwd": (_i, [_p, _i, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _sz, _p]),
    "mc_masked_mse_bwd": (_i, [_p, _i, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p]),
    "mc_patchify": (_i, [_p, _i, _i, _i, _i, _i, _p, _p]),
    "mc_restore_tokens_bwd_workspace_bytes": (_sz, [_i, _i, _i]),
    "mc_restore_tokens_bwd": (_i, [_p, _i, _i, _p, _i, _i, _i, _i, _p, _p, _p, _sz, _p]),
    "mc_similarity_topk_workspace_bytes": (_sz, [_i, C.c_longlong, _i]),
    "mc_similarity_topk": (_i, [_p, _i, _p, C.c_longlong, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "mc_retrieval_ranks_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mc_retrieval_ranks": (_i, [_p, _i, _p, _i, _i, _p, _i, _p, _p, _p, _sz, _p]),
    "mc_retrieval_topk_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "mc_retrieval_topk": (_i, [_p, _i, _p, _i, _i, _i, _i, _p, _p, _p, _sz, _p]),
    "mc_gather_token_rows": (_i, [_p, _p, _i64, _i, _p, _i, _p, _p, _p, _p]),
    "mc_normalize_images": (_i, [_p, _i, _i, _i, _p, _p, _f, _p, _p]),
    "mc_adamw_step": (_i, [_i, _p, _p, _p, _p, _p, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _i, _p,
                           _p]),
    "mc_restore_tokens": (_i, [_p, _i, _p, _p, _i, _i, _i, _i, _p, _p]),
}

_lock = threading.Lock()
_lib = None


class MaeClipB200Error(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise MaeClipB200Error(
                f"{LIB_PATH} is missing: build it with `python -m mae_clip_b200._build` "
                "(there is no CPU or PyTorch fallback for this path)")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)  # AttributeError here = header/library out of sync
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().mc_last_error_string()
        raise MaeClipB200Error(f"{what or 'mae_clip_b200'} failed (status {rc}): "
                               f"{msg.decode() if msg else ''}")


def ptr(t):
    """Raw device pointer of a tensor (or NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def cur_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise MaeClipB200Error(
                "mae_clip_b200 runs on B200 (sm_100a) CUDA tensors only; got a "
                f"{t.device} tensor - there is no CPU fallback for this path")


_ws_cache = {}


def workspace(nbytes: int, device):
    """Grow-only scratch buffer per (device, stream); safe because all uses are stream-ordered."""
    import torch
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf
