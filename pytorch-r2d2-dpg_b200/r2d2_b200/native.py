"""ctypes binding of libr2d2_b200.so (C ABI declared in include/r2d2_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this module raises.
torch is used only for device memory and streams; every pointer handed to the library is a raw
device address taken from a contiguous float32 / int64 CUDA tensor.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, byref, c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("R2D2_B200_LIB") or os.path.join(os.path.dirname(_HERE), "libr2d2_b200.so")  # env: dev builds

GEMM_NT, GEMM_NN, GEMM_TN = 0, 1, 2
EPI_NONE, EPI_TANH, EPI_MUL_DTANH, EPI_ADD_Z = 0, 1, 2, 3


class NativeError(RuntimeError):
    pass


class NetShape(Structure):
    _fields_ = [("obs_size", c_int), ("n_actions", c_int), ("hidden", c_int), ("is_critic", c_int)]


class ReplayConfig(Structure):
    _fields_ = [("obs_size", c_int), ("n_actions", c_int), ("hidden", c_int), ("burn_in", c_int),
                ("learning", c_int), ("n_step", c_int), ("capacity_rows", c_longlong),
                ("max_sequences", c_longlong)]


class ReplayStats(Structure):
    _fields_ = [("n_episodes", c_longlong), ("n_rows_used", c_longlong), ("sequence_counter", c_longlong),
                ("capacity_rows", c_longlong), ("tree_levels", c_longlong), ("tree_nodes", c_longlong),
                ("last_row_start", c_longlong), ("total_priority", c_double)]


class LearnerConfig(Structure):
    _fields_ = [("obs_size", c_int), ("n_actions", c_int), ("hidden", c_int), ("batch", c_int),
                ("burn_in", c_int), ("learning", c_int), ("n_step", c_int), ("gamma", c_float),
                ("actor_lr", c_float), ("critic_lr", c_float), ("eta", c_float),
                ("target_update_interval", c_int),
                ("actor_params", c_void_p), ("critic_params", c_void_p), ("target_actor_params", c_void_p),
                ("target_critic_params", c_void_p), ("actor_grads", c_void_p), ("critic_grads", c_void_p),
                ("actor_exp_avg", c_void_p), ("actor_exp_avg_sq", c_void_p), ("critic_exp_avg", c_void_p),
                ("critic_exp_avg_sq", c_void_p)]


class PeerLayout(Structure):
    _fields_ = [(k, c_size_t) for k in ("bytes", "off_critic_grads", "off_actor_grads", "off_critic_sums",
                                        "off_actor_sums")]


class LearnerBuffers(Structure):
    _fields_ = [(k, c_void_p) for k in ("obs", "act", "rew", "term", "states", "leaf_idx", "uniforms",
                                        "q_value", "target_q_value", "td_sq", "priority", "losses")]


# name -> (restype, argtypes); every symbol include/r2d2_b200.h declares
SIGNATURES = {
    "r2d2_version": (c_int, []),
    "r2d2_arch": (c_char_p, []),
    "r2d2_last_error": (c_char_p, []),
    "r2d2_device_sm_count": (c_int, [POINTER(c_int)]),
    "r2d2_gemm_f32": (c_int, [c_int, c_int, c_int, c_int, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                              c_longlong, c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_void_p, c_void_p,
                              c_longlong, c_int, c_int, c_void_p]),
    "r2d2_net_param_count": (c_size_t, [POINTER(NetShape)]),
    "r2d2_net_workspace_floats": (c_size_t, [POINTER(NetShape), c_int, c_int, c_int]),
    "r2d2_lstm_net_forward": (c_int, [POINTER(NetShape), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                      c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "r2d2_lstm_net_backward": (c_int, [POINTER(NetShape), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                       c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "r2d2_lstm_scan_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "r2d2_lstm_scan_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                        c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "r2d2_debug_scan_forward_trace": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                              c_void_p, c_void_p]),
    "r2d2_debug_scan_backward_trace": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                               c_int, c_void_p, c_void_p]),
    "r2d2_debug_max_active_clusters": (c_int, [c_int, c_int, c_int]),
    "r2d2_set_gemm_impl": (c_int, [c_int]),
    "r2d2_get_gemm_impl": (c_int, []),
    "r2d2_set_scan_impl": (c_int, [c_int]),
    "r2d2_get_scan_impl": (c_int, []),
    "r2d2_scan_status": (c_int, [POINTER(c_int), c_void_p]),
    "r2d2_td_priority": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                                 c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "r2d2_nstep_rewards": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "r2d2_actor_priorities": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                      c_float, c_float, c_int, c_void_p, c_void_p]),
    "r2d2_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_float, c_float, c_float,
                               c_float, c_float, c_void_p]),
    "r2d2_replay_create": (c_int, [POINTER(c_void_p), POINTER(ReplayConfig)]),
    "r2d2_replay_destroy": (c_int, [c_void_p]),
    "r2d2_replay_add_episodes": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "r2d2_replay_add_episode": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                        c_void_p, c_int, c_void_p]),
    "r2d2_replay_sample": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "r2d2_replay_gather": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "r2d2_replay_update_priorities": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "r2d2_replay_stats": (c_int, [c_void_p, POINTER(ReplayStats), c_void_p]),
    "r2d2_replay_decode": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "r2d2_replay_tree_level": (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_longlong)]),
    "r2d2_learner_create": (c_int, [POINTER(c_void_p), POINTER(LearnerConfig)]),
    "r2d2_learner_destroy": (c_int, [c_void_p]),
    "r2d2_learner_buffers_get": (c_int, [c_void_p, POINTER(LearnerBuffers)]),
    "r2d2_learner_critic_phase": (c_int, [c_void_p, c_void_p]),
    "r2d2_learner_actor_forward": (c_int, [c_void_p, c_void_p]),
    "r2d2_learner_actor_phase": (c_int, [c_void_p, c_float, c_void_p]),
    "r2d2_learner_finish_phase": (c_int, [c_void_p, c_float, c_void_p]),
    "r2d2_learner_step_count": (c_int, [c_void_p]),
    "r2d2_learner_set_step_count": (c_int, [c_void_p, c_int]),
    "r2d2_learner_set_overlap_actor_inputs": (c_int, [c_void_p, c_int]),
    "r2d2_learner_buffers_get_slot": (c_int, [c_void_p, c_int, POINTER(LearnerBuffers)]),
    "r2d2_learner_select_batch": (c_int, [c_void_p, c_int]),
    "r2d2_learner_target_phase": (c_int, [c_void_p, c_int, c_void_p]),
    "r2d2_learner_discard_prefetch": (c_int, [c_void_p, c_void_p]),
    "r2d2_peer_layout_for": (c_int, [c_longlong, c_longlong, c_int, POINTER(PeerLayout)]),
    "r2d2_learner_peer_layout": (c_int, [c_void_p, c_int, POINTER(PeerLayout)]),
    "r2d2_learner_attach_peers": (c_int, [c_void_p, c_int, c_int, POINTER(c_void_p)]),
    "r2d2_learner_peer_counters": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "r2d2_learner_peer_status": (c_int, [c_void_p, POINTER(c_int), c_void_p]),
    "r2d2_learner_launches_per_iteration": (c_int, [c_void_p]),
    "r2d2_act_create": (c_int, [POINTER(c_void_p), POINTER(NetShape), c_int]),
    "r2d2_act_destroy": (c_int, [c_void_p]),
    "r2d2_act_load": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "r2d2_act_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "r2d2_act_status": (c_int, [c_void_p, POINTER(c_int), c_void_p]),
}

_lib = None


def lib():
    """Load the shared library once; raise (no fallback) if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NativeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(make -C pytorch-r2d2-dpg_b200/csrc); there is no CPU fallback")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int):
    if rc != 0:
        raise NativeError(f"libr2d2_b200 error {rc}: {lib().r2d2_last_error().decode()}")


def dptr(t, dtype=torch.float32):
    """Raw device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise NativeError("expected a CUDA tensor")
    if t.dtype != dtype or not t.is_contiguous():
        raise NativeError(f"expected contiguous {dtype}, got {t.dtype} contiguous={t.is_contiguous()}")
    return c_void_p(t.data_ptr())


def current_stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


class _RawView:
    """__cuda_array_interface__ adapter so torch can view library-owned device memory."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(int(s) for s in shape), "typestr": typestr,
                                         "data": (int(ptr), False), "version": 2, "strides": None}


def view_f32(ptr, shape, device):
    return torch.as_tensor(_RawView(ptr, shape, "<f4"), device=device)


def view_i64(ptr, shape, device):
    return torch.as_tensor(_RawView(ptr, shape, "<i8"), device=device)


def host_f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(c_void_p)


__all__ = ["lib", "check", "dptr", "current_stream", "NativeError", "NetShape", "ReplayConfig", "ReplayStats",
           "LearnerConfig", "LearnerBuffers", "SIGNATURES", "view_f32", "view_i64", "host_f32", "byref"]
