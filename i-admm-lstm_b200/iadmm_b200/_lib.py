"""ctypes binding of libiadmm_b200.so (the C ABI declared in include/iadmm.h).

There is no CPU or PyTorch fallback: if the library is missing, or the current device is not a B200,
every compute call raises.  torch is used only for device memory, streams and (in training) NCCL.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_size_t, c_void_p, POINTER

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IADMM_B200_LIB") or os.path.join(_HERE, "libiadmm_b200.so")   # the override is a development aid (A/B of two builds)

GATES_SIMT_FP32 = 0
GATES_TC_3XFP16 = 1
GATES_TC_1XFP16 = 2
GATES_TC_F16F8 = 3
GATES_TC_F16F8U = 4
GATE_MODES = {"simt_fp32": GATES_SIMT_FP32, "tc_3xfp16": GATES_TC_3XFP16, "tc_1xfp16": GATES_TC_1XFP16, "tc_f16f8": GATES_TC_F16F8,
              "tc_f16f8u": GATES_TC_F16F8U}

F_ZERO_STATE = 1
F_SKIP_FINAL_RESID = 2
F_STREAMING = 4
F_KEEP_PLANES = 8
F_RESUME = 16
F_RESUME_ODD = 32
TRAIN_RECOMPUTE_GATES = 1

# every symbol include/iadmm.h declares, with its argument types
_P, _I, _F, _Z = c_void_p, c_int, c_float, c_size_t
SIGNATURES = {
    "iadmm_abi_version": ([], c_int),
    "iadmm_last_error": ([], c_char_p),
    "iadmm_device_check": ([], c_int),
    "iadmm_weights_bytes": ([_I, _I, POINTER(_Z)], c_int),
    "iadmm_pack_weights": ([_P] * 16 + [_I, _I, _P, _P], c_int),
    "iadmm_ruiz_workspace_bytes": ([_I, _I, _I, POINTER(_Z)], c_int),
    "iadmm_ruiz": ([_P] * 13 + [_I, _I, _I, _I, _P, _Z, _P], c_int),
    "iadmm_solve_workspace_bytes": ([_I, _I, _I, _I, _I, POINTER(_Z)], c_int),
    "iadmm_solve_state_resumable": ([_I, _I, _I, _I, _I, POINTER(_I)], c_int),
    "iadmm_solve": ([_P] * 20 + [_I] * 8 + [_F, _I, _I, _P, _Z, _P], c_int),
    "iadmm_sparse_bytes": ([_I, _I, _I, _Z, POINTER(_Z)], c_int),
    "iadmm_sparse_pack": ([_P, _I, _I, _I, _Z, _P, _Z, _P, _P], c_int),
    "iadmm_block_mask_bytes": ([_I, _I, _I, POINTER(_Z)], c_int),
    "iadmm_block_mask": ([_P, _I, _I, _I, _P, _Z, _P, _P], c_int),
    "iadmm_solve_sparse": ([_P, _P, _P, _Z, _P, _P, _P, _P, _Z, _P] + [_P] * 16 + [_I] * 8 + [_F, _I, _I, _P, _Z, _P], c_int),
    "iadmm_residuals_workspace_bytes": ([_I, _I, _I, POINTER(_Z)], c_int),
    "iadmm_residuals": ([_P] * 8 + [_I, _I, _I, _P, _Z, _P], c_int),
    "iadmm_build_kkt": ([_P] * 10 + [_I] * 7 + [_F, _P], c_int),
    "iadmm_kkt_penalty_diagonal": ([_P, _P] + [_I] * 7 + [_P], c_int),
    "iadmm_lu_factor": ([_P] * 4 + [_I, _I, _P], c_int),
    "iadmm_lu_solve": ([_P] * 3 + [_I, _I, _P], c_int),
    "iadmm_lu_factor_blocked_workspace_bytes": ([_I, _I, POINTER(_Z)], c_int),
    "iadmm_lu_factor_blocked": ([_P] * 4 + [_I, _I, _P, _Z, _P], c_int),
    "iadmm_param_count": ([_I, _I, POINTER(_Z)], c_int),
    "iadmm_train_workspace_bytes": ([_I, _I, _I, _I, POINTER(_Z)], c_int),
    "iadmm_step_fwd": ([_P] * 21 + [_I] * 7 + [_F, _I, _P, _Z, _P], c_int),
    "iadmm_step_bwd": ([_P] * 30 + [_I] * 7 + [_F, _P, _Z, _P], c_int),
    "iadmm_window_workspace_bytes": ([_I] * 6 + [POINTER(_Z)], c_int),
    "iadmm_train_window": ([_P] * 14 + [_I] * 8 + [_F, _F, _I, _I, _P, _Z, _P], c_int),
    "iadmm_residuals_train_workspace_bytes": ([_I, _I, _I, POINTER(_Z)], c_int),
    "iadmm_residuals_fwd": ([_P] * 10 + [_I, _I, _I, _P, _Z, _P], c_int),
    "iadmm_residuals_bwd": ([_P] * 11 + [_I, _I, _I, _P, _Z, _P], c_int),
    "iadmm_allreduce_grads": ([_P, _Z, _F, _P, _P], c_int),
    "iadmm_nccl_unique_id": ([_P], c_int),
    "iadmm_nccl_comm_init": ([POINTER(c_void_p), _I, _P, _I], c_int),
    "iadmm_nccl_comm_destroy": ([_P], c_int),
    "iadmm_profile_begin": ([_I], c_int),
    "iadmm_profile_end": ([POINTER(ctypes.c_double)] * 3 + [POINTER(_I)], c_int),
    "iadmm_profile_end_kinds": ([POINTER(ctypes.c_double), POINTER(_I), _I], c_int),
}


class IadmmError(RuntimeError):
    pass


_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IadmmError(f"{LIB_PATH} not found: build it with `python i-admm-lstm_b200/build.py` "
                             "(there is no fallback path)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (argtypes, restype) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise IadmmError(f"libiadmm_b200 error {rc}: {lib().iadmm_last_error().decode()}")


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise IadmmError("libiadmm_b200 takes CUDA tensors only: there is no CPU path "
                             f"(got a tensor on {t.device})")


def ptr(t):
    """Device pointer of a contiguous fp32 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise IadmmError("libiadmm_b200 takes CUDA tensors only (no CPU path)")
    if not t.is_contiguous():
        raise IadmmError("tensor must be contiguous")
    return c_void_p(t.data_ptr())


def f32(t, device=None):
    """Contiguous fp32 view/copy of `t` (host glue: the reference passes fp32 everywhere)."""
    if t is None:
        return None
    if device is not None and t.device != device:
        t = t.to(device)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def stream_ptr():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
