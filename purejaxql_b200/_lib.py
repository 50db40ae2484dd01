"""ctypes binding of libpqn_b200.so (the C ABI in include/pqn_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` /
``python -m purejaxql_b200.build``.  Loading fails loudly when it is missing:
there is no fallback implementation.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_longlong, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpqn_b200.so")


class EnvInfo(Structure):
    _fields_ = [("state_words", c_int32), ("obs_dim", c_int32), ("obs_shape", c_int32 * 3),
                ("num_actions", c_int32), ("max_steps", c_int32), ("binary_obs", c_int32),
                ("packed_obs_words", c_int32)]


class EnvParams(Structure):
    _fields_ = [("max_steps", c_int32), ("memory_length", c_int32)]


class NetDesc(Structure):
    _fields_ = [("kind", c_int32), ("in_c", c_int32), ("hidden", c_int32), ("layers", c_int32),
                ("num_actions", c_int32), ("norm_type", c_int32), ("norm_input", c_int32)]


NORM_TYPES = {"layer_norm": 0, "batch_norm": 1}          # any other string: no normalisation (pqn_minatar.py:35-36)


class NetLayout(Structure):
    _fields_ = [(n, c_int64) for n in (
        "total", "bn_scale", "bn_bias", "conv_w", "conv_b", "ln0_scale", "ln0_bias", "d0_w", "d0_b",
        "ln1_scale", "ln1_bias", "d1_w", "d1_b", "head_w", "head_b",
        "gru_ir_w", "gru_ir_b", "gru_iz_w", "gru_iz_b", "gru_in_w", "gru_in_b", "gru_hr_w", "gru_hz_w", "gru_hn_w",
        "gru_hn_b")]


class PqnError(RuntimeError):
    pass


_SIGS = {
    "pqn_last_error": (c_char_p, []),
    "pqn_version": (c_int, []),
    "pqn_launch_count": (c_longlong, []),
    "pqn_num_kernels": (c_int, []),
    "pqn_kernel_name": (c_char_p, [c_int]),
    "pqn_profile_enable": (c_int, [c_int]),
    "pqn_profile_read": (c_int, [POINTER(c_double), POINTER(c_longlong), c_int]),
    "pqn_env_info": (c_int, [c_int, POINTER(EnvInfo)]),
    "pqn_rng_split": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int, c_void_p]),
    "pqn_threefry2x32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "pqn_rng_bits": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int, c_void_p]),
    "pqn_set_permutation_bucket_log2": (c_int, [c_int]),
    "pqn_permutation_workspace_bytes": (c_int64, [c_int64, c_int]),
    "pqn_permutation": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "pqn_env_reset": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "pqn_env_reset_params": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, POINTER(EnvParams), c_int,
                                     c_void_p]),
    "pqn_env_step": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "pqn_env_obs_packed": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "pqn_env_obs": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "pqn_eps_greedy": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int, c_void_p]),
    "pqn_rollout_act_step": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int32, c_int32,
                                     c_int32, c_int32, c_int, c_float, c_int, c_void_p]),
    "pqn_rollout_keys": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int, c_void_p]),
    "pqn_qlambda": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32,
                            c_float, c_float, c_void_p]),
    "pqn_net_layout": (c_int, [POINTER(NetDesc), POINTER(NetLayout)]),
    "pqn_net_stats_floats": (c_int64, [POINTER(NetDesc)]),
    "pqn_net_workspace_bytes": (c_int64, [POINTER(NetDesc), c_int32, c_int64]),
    "pqn_net_init": (c_int, [POINTER(NetDesc), c_void_p, c_void_p, c_int32, c_void_p]),
    "pqn_qnet_forward": (c_int, [POINTER(NetDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int32,
                                 c_int64, c_void_p, c_void_p]),
    "pqn_qnet_loss_grad": (c_int, [POINTER(NetDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                   c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64,
                                   c_void_p, c_void_p]),
    "pqn_rnn_step": (c_int, [POINTER(NetDesc), c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                             c_int32, c_int32, c_void_p, c_void_p]),
    "pqn_rnn_loss_grad": (c_int, [POINTER(NetDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float, c_float,
                                  c_void_p, c_void_p]),
    "pqn_radam_clip_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                    c_int64, c_float, c_float, c_float, c_float, c_void_p]),
    "pqn_bn_stats_update": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int64, c_float, c_float, c_void_p]),
    "pqn_set_tensor_core_path": (c_int, [c_int]),
    "pqn_set_conv_mma_path": (c_int, [c_int]),
    "pqn_tc_split_lo": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "pqn_tc_split16": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_float, c_void_p]),
    "pqn_tc_gemm16_test": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32,
                                   c_int32, c_int, c_int, c_float, c_void_p]),
    "pqn_tc_debug": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pqn_tc_gemm_test": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32,
                                 c_int32, c_int, c_int, c_int, c_void_p]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def lib():
    """The loaded library (raises PqnError with build instructions if absent)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PqnError(
                f"{LIB_PATH} is not built. Run `python -m purejaxql_b200.build` (needs nvcc). "
                "purejaxql_b200 has no CPU fallback.")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)  # AttributeError here == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().pqn_last_error().decode("utf-8", "replace")
        raise PqnError(f"{what or 'libpqn_b200'} failed (rc={rc}): {msg}")


def p(t):
    """Device pointer of a torch tensor (or None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise PqnError("libpqn_b200 takes CUDA tensors only (no CPU fallback); got a CPU tensor")
    if not t.is_contiguous():
        raise PqnError("libpqn_b200 takes contiguous tensors")
    return c_void_p(t.data_ptr())


def raw(t):
    """Device pointer of a (possibly strided) CUDA tensor view; the caller passes the strides."""
    if t is None:
        return None
    if not t.is_cuda:
        raise PqnError("libpqn_b200 takes CUDA tensors only (no CPU fallback); got a CPU tensor")
    return c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def profile_read(reset=True):
    """{kernel name: (total ms, launches)} from the library's CUDA-event spans."""
    l = lib()
    n = l.pqn_num_kernels()
    ms = (c_double * n)()
    cnt = (c_longlong * n)()
    check(l.pqn_profile_read(ms, cnt, 1 if reset else 0), "pqn_profile_read")
    return {l.pqn_kernel_name(i).decode(): (ms[i], int(cnt[i])) for i in range(n) if cnt[i]}
