"""ctypes binding of libddm_b200.so (see include/ddm_b200.h).

There is deliberately no fallback: if the shared object is missing, or CUDA is not
available, every entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

PKG = os.path.dirname(os.path.abspath(__file__))
# DDM_B200_LIB overrides the location (kernel-variant sweeps); the default is the in-tree build
LIB_PATH = os.environ.get("DDM_B200_LIB") or os.path.join(PKG, "_lib", "libddm_b200.so")

DDM_OK, DDM_ERR_INVALID, DDM_ERR_CUDA, DDM_ERR_STATE = 0, -1, -2, -3
WS_QUEUE, WS_USEFUL_STEPS, WS_GENERIC_ROWS, WS_LANE_STEPS, WS_ERROR, WS_WORDS = 0, 1, 2, 3, 4, 8
MAX_PEERS = 15

_i64, _u64, _f32, _i32 = ctypes.c_int64, ctypes.c_uint64, ctypes.c_float, ctypes.c_int
_ptr = ctypes.c_void_p

_SIGNATURES = {
    "ddm_abi_version": (ctypes.c_int, []),
    "ddm_last_error": (ctypes.c_char_p, []),
    "ddm_device_info": (ctypes.c_int, [_i32, _ptr, _ptr, _ptr, _ptr]),
    "ddm_probe_launch_blocking": (ctypes.c_int, [_i64, _ptr]),
    "ddm_pack_simd_bits": (ctypes.c_int, []),
    "ddm_sim_set_stream_timeout_us": (ctypes.c_int, [_i64]),
    "ddm_sim_set_small_batch_max": (ctypes.c_int, [_i64]),
    "ddm_sim_workspace_bytes": (ctypes.c_size_t, []),
    "ddm_sim_f32": (ctypes.c_int, [_ptr, _i64, _ptr, _i64, _i64, _i64, _i64, _i64, _f32, _f32, _f32, _f32,
                                   _u64, _u64, _ptr, _i64, _i32, _ptr, _ptr, _ptr, _ptr]),
    "ddm_sim_gather_f32": (ctypes.c_int, [_ptr, _i64, _ptr, _i64, _i64, _i64, _i64, _i64, _f32, _f32, _f32, _f32,
                                          _u64, _u64, _i32, _ptr, _ptr, _i32, _ptr, _ptr]),
    "ddm_sim_stream_f32": (ctypes.c_int, [_ptr, _i64, _ptr, _i64, _i64, _i64, _i64, _i64, _f32, _f32, _f32, _f32,
                                          _u64, _u64, _i32, _ptr, _ptr, _ptr, _ptr]),
    "ddm_pack_z_host": (ctypes.c_int64, [_ptr, _i64, _i64, _i64, _ptr, _i32]),
    "ddm_pack_z_dev": (ctypes.c_int, [_ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
    "ddm_unpack_z_host": (ctypes.c_int, [_ptr, _i64, _i64, _ptr, _i64, _i32]),
    "ddm_ingest_packed": (ctypes.c_int, [_ptr, _i64, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _i32, _ptr, _ptr]),
    "ddm_sim_packed_f32": (ctypes.c_int, [_ptr, _i64, _i64, _i64, _f32, _f32, _f32, _f32, _u64, _u64, _i32, _ptr, _ptr,
                                          _ptr, _ptr, _ptr]),
    "ddm_philox_normals_f32": (ctypes.c_int, [_u64, _u64, _i64, _i64, _ptr, _i64, _ptr]),
    "ddm_philox_words_u32": (ctypes.c_int, [_u64, _u64, _i64, _i64, _ptr, _i64, _ptr]),
    "ddm_pulses_pcg64": (ctypes.c_int, [_u64, _u64, _u64, _u64, _u64, _i64, _i64, _u64, _ptr, _i64, _ptr]),
    "ddm_pcg64_advance": (ctypes.c_int, [_ptr, _ptr, _u64, _u64, _u64]),
    "ddm_slice_propose_f32": (ctypes.c_int, [_ptr, _ptr, _ptr, _ptr, _ptr]),
    "ddm_slice_update_f32": (ctypes.c_int, [_ptr, _ptr, _ptr, _ptr, _ptr]),
    "mnle_packed_floats": (ctypes.c_size_t, [_i32]),
    "mnle_create": (ctypes.c_int, [_ptr, ctypes.c_size_t, _i32, _ptr]),
    "mnle_destroy": (ctypes.c_int, [_ptr]),
    "mnle_log_prob_rows_f32": (ctypes.c_int, [_ptr, _ptr, _ptr, _i64, _i64, _ptr, _ptr]),
    "mnle_log_prob_rows_precise_f32": (ctypes.c_int, [_ptr, _ptr, _ptr, _i64, _i64, _ptr, _ptr]),
    "mnle_log_prob_rows_tc_f32": (ctypes.c_int, [_ptr, _ptr, _ptr, _i64, _i64, _ptr, _ptr]),
    "mnle_loglik_workspace_floats": (ctypes.c_size_t, [_i64, _i64]),
    "mnle_loglik_tc_workspace_floats": (ctypes.c_size_t, [_i64, _i64]),
    "mnle_loglik_sum_tc_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
    "mnle_loglik_batched_tc_workspace_floats": (ctypes.c_size_t, [_i64, _i64, _i64]),
    "mnle_loglik_sum_batched_tc_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
    "mnle_loglik_sessions_tc_workspace_floats": (ctypes.c_size_t, [_i64, _i64, _i64]),
    "mnle_loglik_sum_sessions_tc_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _ptr, _i64, _i64, _i64, _ptr, _ptr,
                                                       _ptr]),
    "mnle_loglik_sessions_tc64_workspace_floats": (ctypes.c_size_t, [_i32, _i64, _i64, _i64]),
    "mnle_loglik_sum_sessions_tc64_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _ptr, _i64, _i64, _i64, _ptr,
                                                         _ptr, _ptr]),
    "mnle_loglik_grad_workspace_floats": (ctypes.c_size_t, [_i64, _i64]),
    "mnle_loglik_sum_grad_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr]),
    "mnle_loglik_tc64_workspace_floats": (ctypes.c_size_t, [_i32, _i64, _i64]),
    "mnle_loglik_sum_tc64_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
    "mnle_loglik_grad_tc_workspace_floats": (ctypes.c_size_t, [_i32, _i64, _i64]),
    "mnle_loglik_sum_grad_tc_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr]),
    "mnle_sample_tc_workspace_floats": (ctypes.c_size_t, [_i32, _i64, _i64]),
    "mnle_sample_tc_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _i64, _i64, _u64, _u64, _ptr, _ptr, _ptr, _ptr]),
    "mnle_train_workspace_floats": (ctypes.c_size_t, [_i32, _i64]),
    "mnle_train_nll_grad_f32": (ctypes.c_int, [_ptr, _i32, _ptr, _ptr, _i64, _ptr, _i64, _ptr, _ptr, _ptr, _i32, _ptr]),
    "mnle_train_adam_f32": (ctypes.c_int, [_ptr, _ptr, _ptr, _ptr, _i32, _ptr, _f32, _f32, _f32, _f32, _i64, _f32, _ptr]),
    "mnle_tc_set_trace": (ctypes.c_int, [_ptr]),
    "mnle_tc_selftest": (ctypes.c_int, [_ptr, _ptr, _i32, _i32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, _ptr, _ptr]),
    "mnle_loglik_sum_simt_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
    "mnle_loglik_sum_precise_f32": (ctypes.c_int, [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
}

_lib: Optional[ctypes.CDLL] = None


class NativeLibraryMissing(RuntimeError):
    pass


def exported_symbols():
    return sorted(_SIGNATURES)


def lib() -> ctypes.CDLL:
    """Load the library once; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} is missing. Build it with `python -m sbi_for_diffusion_models_b200.build` "
                "(needs nvcc; targets sm_100a). There is no CPU or PyTorch fallback for this path.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the ABI drifted
            fn.restype, fn.argtypes = res, args
        if L.ddm_abi_version() != 1:
            raise NativeLibraryMissing(f"{LIB_PATH}: ABI version {L.ddm_abi_version()} != 1, rebuild")
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc == DDM_OK:
        return
    msg = lib().ddm_last_error().decode("utf-8", "replace")
    if rc == DDM_ERR_INVALID:
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what}: {msg} (code {rc})")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError(
            "sbi_for_diffusion_models_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch
