"""ctypes binding of libspo.so (the C-ABI declared in include/spo.h).

PyTorch is used only as the owner of device memory and streams: every call passes
``tensor.data_ptr()`` and the current CUDA stream handle.  There is no fallback: if the
shared library is missing or a call fails, a ``SpoError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libspo.so")


class SpoError(RuntimeError):
    pass


class Dims(C.Structure):
    _fields_ = [("obs_dim", C.c_int), ("act_dim", C.c_int), ("hidden", C.c_int)]


_fp = C.c_void_p


class Rollout(C.Structure):
    _fields_ = [("obs", _fp), ("act", _fp), ("reward", _fp), ("cost", _fp), ("value_r", _fp), ("value_c", _fp),
                ("logp", _fp), ("seg_end", _fp), ("boot_r", _fp), ("boot_c", _fp),
                ("num_envs", C.c_int), ("steps", C.c_int)]


class Batch(C.Structure):
    _fields_ = [("obs", _fp), ("act", _fp), ("logp", _fp), ("target_r", _fp), ("target_c", _fp), ("adv", _fp),
                ("old_mean", _fp), ("old_std", _fp), ("count", C.c_int64)]


class HParams(C.Structure):
    _fields_ = [("lr_actor", C.c_float), ("lr_reward", C.c_float), ("lr_cost", C.c_float),
                ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("max_grad_norm", C.c_float), ("critic_l2", C.c_float),
                ("clip_lo", C.c_float), ("clip_hi", C.c_float),
                ("focops_lam", C.c_float), ("focops_kl", C.c_float), ("value_coef", C.c_float)]


class Comm(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("grad_bufs", C.c_void_p), ("flags", C.c_void_p),
                ("seq_base", C.c_ulonglong), ("spin_limit", C.c_uint)]


# numpy view of spo_update_ctrl (64 bytes): see include/spo.h
CTRL_BYTES = 64
CTRL_DTYPE = [("loss_sum", "<f8", 3), ("kl_sum", "<f8"), ("steps", "<i8"), ("stop", "<i4"), ("passes", "<i4"),
              ("final_kl", "<f4"), ("ticket", "<u4"), ("extra_sumsq", "<f4"), ("pad", "<i4")]
CTRL_EXTRA_SUMSQ_F32_INDEX = 14  # byte offset 56
CTRL_KL_SUM_F64_INDEX = 3        # byte offset 24

LOSS_PPO_CLIP, LOSS_FOCOPS, LOSS_CRITIC_ONLY, LOSS_PG, LOSS_CUP_PROJECTION = 0, 1, 2, 3, 4

_i, _i64, _f, _d, _u64, _p = C.c_int, C.c_int64, C.c_float, C.c_double, C.c_uint64, C.c_void_p
_pi, _PD = C.POINTER(C.c_int), C.POINTER(Dims)

# Every entry point of include/spo.h: name -> (argtypes, whether a call counts as a kernel launch in LAUNCHES).
# spo_conjugate_gradient launches 2 * iters + 1 kernels; its caller counts them.
_ABI = {
    "spo_version": ([], False),
    "spo_last_error": ([], False),
    "spo_sync_check": ([_p], False),
    "spo_param_count": ([_PD, _pi, _pi, _pi], False),
    "spo_param_offsets": ([_PD, _i] + [_pi] * 7, False),
    "spo_policy_step": ([_PD, _p, _p, _p, _u64, _u64, _i, _i, _p, _p, _p, _p, C.POINTER(Rollout), _i, _p], True),
    "spo_critic_values": ([_PD, _p, _p, _i, _p, _p, _p], True),
    "spo_store_transition": ([C.POINTER(Rollout), _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p], True),
    "spo_gae_dual": ([_p, _p, _p, _p, _p, _p, _p, _f, _d, _d, _p, _p, _p, _p, _i, _i, _i, _p], True),
    "spo_adv_stats": ([_p, _p, _i64, _p, _p], True),
    "spo_adv_apply": ([_p, _p, _i64, _p, _i, _i, _f, _f, _p, _p], True),
    "spo_pg_update": ([_PD, _p, _p, _p, _p, C.POINTER(Batch), _p, _i64, _i, _i, C.POINTER(HParams), _p, _p], True),
    "spo_comm_slot_floats": ([_PD, _pi], False),
    "spo_pg_update_dp": ([_PD, _p, _p, _p, _p, C.POINTER(Batch), _p, _i64, _i, _i, C.POINTER(HParams), _p, C.POINTER(Comm), _p],
                         True),
    "spo_comm_alloc": ([C.c_size_t, C.POINTER(_p)], False),
    "spo_comm_free": ([_p], False),
    "spo_comm_export": ([_p, C.c_char_p], False),
    "spo_comm_import": ([C.c_char_p, C.POINTER(_p)], False),
    "spo_comm_close": ([_p], False),
    "spo_actor_kl_accumulate": ([_PD, _p, _p, _p, _p, _i64, _p, _p], True),
    "spo_kl_finalize": ([_p, _d, _f, _p], True),
    "spo_actor_forward": ([_PD, _p, _p, _i64, _p, _p], True),
    "spo_actor_kl": ([_PD, _p, _p, _p, _p, _i64, _i, _f, _p, _p], True),
    "spo_surrogate_grad": ([_PD, _p, _p, _p, _p, _p, _i64, _p, _p, _p], True),
    "spo_fvp": ([_PD, _p, _p, _i64, _p, _f, _p, _p], True),
    "spo_linesearch_eval": ([_PD, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p], True),
    "spo_conjugate_gradient": ([_PD, _p, _p, _i64, _p, _i, _f, _f, _f, _p, _p, _p], False),
    "spo_cg_begin": ([_PD, _p, _p, _p, _p], True),
    "spo_cg_update": ([_PD, _p, _p, _f, _f, _p], True),
    "spo_obs_normalize": ([_p, _i, _i, _p, _p, _d, _p, _i, _d, _p, _p], True),
    "spo_action_rescale": ([_p, _i, _i, _p, _p, _f, _f, _p, _p], True),
    "spo_gae_masked": ([_p, _p, _p, _f, _f, _f, _d, _p, _i, _i, _p], True),
    "spo_ma_mlp_layer": ([_p, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p], True),
    "spo_ma_head": ([_p, _i, _i, _p, _p, _i, _p, _f, _f, _p, _p, _p, _p], True),
    "spo_ma_mlp_layer_train": ([_p, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p], True),
    "spo_ma_ln_elu_bwd": ([_p, _p, _p, _i, _i, _p, _p, _p], True),
    "spo_ma_ln_in_bwd": ([_p, _p, _i, _i, _p, _p], True),
    "spo_ma_partial_reduce": ([_p, _i, _i, _i, _i, _p, _p, _p, _f, _p], True),
    "spo_ma_gemm_nn": ([_p, _p, _p, _i, _i, _i, _p], True),
    "spo_ma_gemm_tn": ([_p, _p, _p, _i, _i, _i, _i, _p], True),
    "spo_ma_actor_loss": ([_p, _i, _i, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _f, _f, _f, _f, _p, _p, _p, _p], True),
    "spo_ma_actor_finalize": ([_p, _i, _i, _p, _i, _f, _f, _f, _p, _p, _p, _p], True),
    "spo_ma_value_loss": ([_p, _p, _p, _p, _i, _f, _f, _f, _p, _p, _p], True),
    "spo_ma_popart_normalize": ([_p, _i, _p, _d, _f, _p, _p], True),
    "spo_ma_lagrange_step": ([_p, _p, _p, _i, _f, _d, _f, _p, _p], True),
    "spo_ma_clip_adam": ([_p, _p, _p, _p, _i, _f, _d, _d, _d, _d, _d, _i, _p, _p, _p], True),
    "spo_ma_ln_in_jvp": ([_p, _i, _i, _p, _p, _p, _p], True),
    "spo_ma_gemm_nt_pair": ([_p, _p, _i, _p, _p, _i, _p, _p, _i, _i, _p], True),
    "spo_ma_ln_elu_jvp": ([_p, _p, _p, _p, _p, _i, _i, _p], True),
    "spo_ma_fvp_head": ([_p, _i, _i, _p, _f, _f, _p, _p, _p], True),
    "spo_ma_fvp_finish": ([_p, _p, _i, _i, _i, _p, _f, _f, _f, _p, _p], True),
    "spo_ma_dot": ([_p, _p, _i, _p, _p, _p], True),
    "spo_ma_cg_begin": ([_p, _p, _p, _p, _i, _p, _p, _p], True),
    "spo_ma_cg_update": ([_p, _p, _p, _p, _i, _p, _p, _f, _p], True),
    "spo_ma_axpby": ([_p, _f, _p, _f, _p, _i, _p], True),
    "spo_ma_clip_norm": ([_p, _i, _f, _p, _p, _p], True),
    "spo_ma_linesearch_eval": ([_p, _i, _i, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _f, _f, _p, _p, _p], True),
}
EXPORTS = tuple(_ABI)
_KERNEL_CALLS = frozenset(name for name, (_, launch) in _ABI.items() if launch)

# number of libspo kernels launched so far (bench.py reports the delta over its timed region)
LAUNCHES = {"n": 0}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SpoError(f"{LIB_PATH} not found: build it with `python safe-policy-optimization_b200/build.py` "
                           "(there is no CPU / PyTorch fallback for the hot path)")
        _lib = C.CDLL(LIB_PATH)
        for name, (argtypes, _) in _ABI.items():
            fn = getattr(_lib, name)
            fn.argtypes = argtypes
            fn.restype = C.c_int
        _lib.spo_last_error.restype = C.c_char_p
    return _lib


def check(rc, what):
    if what in _KERNEL_CALLS:
        LAUNCHES["n"] += 1
    if rc != 0:
        raise SpoError(f"{what} failed ({rc}): {lib().spo_last_error().decode()}")


def call(name, *args):
    """Call entry point ``name`` of the library, count it in LAUNCHES if it is a kernel, raise SpoError on failure."""
    check(getattr(lib(), name)(*args), name)


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Tensors must be contiguous CUDA tensors."""
    if t is None:
        return None
    if not t.is_cuda:
        raise SpoError("libspo needs CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise SpoError("libspo needs contiguous tensors")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def dims(obs_dim, act_dim, hidden=64):
    return Dims(int(obs_dim), int(act_dim), int(hidden))


def param_count(d):
    a, c, t = C.c_int(), C.c_int(), C.c_int()
    call("spo_param_count", C.byref(d), C.byref(a), C.byref(c), C.byref(t))
    return a.value, c.value, t.value


def param_offsets(d, net):
    out = [C.c_int() for _ in range(7)]
    call("spo_param_offsets", C.byref(d), net, *[C.byref(o) for o in out])
    return dict(zip(("log_std", "w1", "b1", "w2", "b2", "w3", "b3"), (o.value for o in out)))
