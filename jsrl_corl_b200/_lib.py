"""ctypes binding of the C-ABI in include/iql_b200.h.

The shared library is built in-tree (``python -m jsrl_corl_b200.build``) and is
the only compute path of the package: there is no CPU or eager fallback.  A
missing library raises at import of this module's ``lib()``; a missing CUDA
device raises when an engine or buffer is constructed.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libiql_b200.so")
if os.environ.get("IQL_B200_DEBUG") and os.environ.get("IQL_B200_LIB"):  # A/B builds of the library (debug only)
    LIB_PATH = os.environ["IQL_B200_LIB"]

IQL_OK, IQL_ERR_INVALID, IQL_ERR_CUDA, IQL_ERR_STATE, IQL_ERR_SHAPE = 0, 1, 2, 3, 4
MATH_FP32_SIMT, MATH_TF32_TCGEN05 = 0, 1
SAMPLE_PHILOX, SAMPLE_INDICES, SAMPLE_PRELOADED, SAMPLE_MT19937 = 0, 1, 2, 3
MT_STATE_WORDS = 626  # IQL_MT_STATE_WORDS: key[624] | pos | pad
NET_Q1, NET_Q2, NET_V, NET_ACTOR = 0, 1, 2, 3
KIND_WEIGHT, KIND_BIAS, KIND_LOG_STD = 0, 1, 2
OPT_STEP_PATH, OPT_KEEP_GRADS = 1, 2
INFO_TENSOR_CORE_PATH, INFO_FUSED_FORWARD, INFO_CHAINED_BACKWARD, INFO_CHAINED_BACKWARD_GRADS = 1, 2, 3, 4
STEP_PATHS = {"auto": 0, "phases": 1, "chain": 2, "chain_grads": 4}
ACT_SKIP, ACT_LEARNER, ACT_LEARNER_DIST, ACT_GUIDE, ACT_LEARNER_DROPOUT, ACT_LEARNER_DIST_DROPOUT = 0, 1, 2, 3, 4, 5
ACT_SOURCES = {"skip": ACT_SKIP, "learner": ACT_LEARNER, "learner_dist": ACT_LEARNER_DIST, "guide": ACT_GUIDE,
               "learner_dropout": ACT_LEARNER_DROPOUT, "learner_dist_dropout": ACT_LEARNER_DIST_DROPOUT}


class Config(C.Structure):
    _fields_ = [
        ("n_members", C.c_int32), ("state_dim", C.c_int32), ("action_dim", C.c_int32),
        ("hidden_dim", C.c_int32), ("n_hidden", C.c_int32), ("batch_size", C.c_int32),
        ("deterministic", C.c_int32), ("math_mode", C.c_int32), ("max_steps_per_call", C.c_int32),
        ("reserved", C.c_int32 * 7),
    ]


class HParams(C.Structure):
    _fields_ = [
        ("beta", C.c_double), ("iql_tau", C.c_double), ("discount", C.c_double), ("tau", C.c_double),
        ("vf_lr", C.c_double), ("qf_lr", C.c_double), ("actor_lr", C.c_double),
        ("actor_dropout", C.c_double),
        ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double),
        ("lr_eta_min", C.c_double),
        ("cosine_t_max", C.c_int64), ("seed", C.c_uint64),
    ]


class Counters(C.Structure):
    _fields_ = [
        ("v_step", C.c_int64), ("q_step", C.c_int64), ("actor_step", C.c_int64),
        ("sched_epoch", C.c_int64), ("total_it", C.c_int64), ("sample_step", C.c_int64),
    ]


class RowLayout(C.Structure):
    _fields_ = [
        ("state_dim", C.c_int32), ("action_dim", C.c_int32), ("row_floats", C.c_int32),
        ("off_state", C.c_int32), ("off_action", C.c_int32), ("off_next_state", C.c_int32),
        ("off_reward", C.c_int32), ("off_done", C.c_int32),
    ]


class Layout(C.Structure):
    _fields_ = [
        ("param_floats", C.c_int64), ("q_floats", C.c_int64),
        ("v_begin", C.c_int64), ("v_end", C.c_int64),
        ("actor_begin", C.c_int64), ("actor_end", C.c_int64),
        ("workspace_bytes", C.c_int64),
        ("n_tensors", C.c_int32), ("reserved", C.c_int32),
        ("row", RowLayout),
    ]


class TensorInfo(C.Structure):
    _fields_ = [
        ("net", C.c_int32), ("layer", C.c_int32), ("kind", C.c_int32),
        ("rows", C.c_int32), ("cols", C.c_int32), ("ld", C.c_int32),
        ("offset", C.c_int64),
    ]


_P = C.c_void_p
# every symbol include/iql_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "iql_version": (C.c_char_p, []),
    "iql_last_error": (C.c_char_p, [_P]),
    "iql_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "iql_destroy": (None, [_P]),
    "iql_get_layout": (C.c_int, [_P, C.POINTER(Layout)]),
    "iql_tensor_at": (C.c_int, [_P, C.c_int32, C.POINTER(TensorInfo)]),
    "iql_bind_state": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_size_t]),
    "iql_set_hparams": (C.c_int, [_P, C.c_int32, C.POINTER(HParams)]),
    "iql_set_counters": (C.c_int, [_P, C.c_int32, C.POINTER(Counters)]),
    "iql_set_option": (C.c_int, [_P, C.c_int32, C.c_int64]),
    "iql_get_info": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int64)]),
    "iql_get_counters": (C.c_int, [_P, C.c_int32, C.POINTER(Counters), _P]),
    "iql_set_batch_sizes": (C.c_int, [_P, _P]),
    "iql_get_batch_sizes": (C.c_int, [_P, _P]),
    "iql_set_active_members": (C.c_int, [_P, C.c_int32, _P]),
    "iql_get_active_members": (C.c_int, [_P, _P]),
    "iql_sync_target": (C.c_int, [_P, C.c_int32, _P]),
    "iql_replay_row_layout": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(RowLayout)]),
    "iql_replay_pack": (C.c_int, [_P, C.POINTER(RowLayout), C.c_int64, C.c_int64, _P, _P, _P, _P, _P, _P]),
    "iql_replay_ingest": (C.c_int, [_P, C.POINTER(RowLayout), C.c_int64, C.c_int64, _P, _P, _P, _P, _P, C.c_int32, C.c_float,
                                    _P, _P, C.c_float, C.c_float, C.c_float, _P]),
    "iql_replay_insert": (C.c_int, [_P, C.POINTER(RowLayout), C.c_int64, _P, _P]),
    "iql_replay_insert_host": (C.c_int, [_P, C.POINTER(RowLayout), C.c_int64, _P, _P, C.c_float, _P, C.c_float, _P]),
    "iql_replay_sample": (C.c_int, [_P, C.POINTER(RowLayout), C.c_int64, C.c_int64, _P, C.c_uint64, C.c_uint64,
                                    _P, _P, _P, _P, _P, _P, _P]),
    "iql_replay_sample_host": (C.c_int, [_P, C.POINTER(RowLayout), C.c_int64, C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "iql_bind_replay": (C.c_int, [_P, C.c_int32, _P, C.c_int64, C.c_int64]),
    "iql_set_replay_size": (C.c_int, [_P, C.c_int32, C.c_int64]),
    "iql_load_batch": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "iql_train_steps": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "iql_train_host_step": (C.c_int, [_P, _P, _P, _P, _P]),
    "iql_train_host_step_mt19937": (C.c_int, [_P, _P, _P, _P]),
    "iql_bind_index_streams": (C.c_int, [_P, _P, _P]),
    "iql_mt19937_randint": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int64, _P]),
    "iql_host_step_wait": (C.c_int, [_P, _P, _P]),
    "iql_act": (C.c_int, [_P, C.c_int32, _P, C.c_int64, C.c_float, _P, _P]),
    "iql_act_host": (C.c_int, [_P, C.c_int32, _P, C.c_float, _P, _P, _P]),
    "iql_act_host_gaussian": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P]),
    "iql_bind_guide": (C.c_int, [_P, _P]),
    "iql_act_host_members": (C.c_int, [_P, _P, _P, C.c_float, _P, _P, _P, _P]),
    "iql_get_act_steps": (C.c_int, [_P, _P]),
    "iql_set_act_steps": (C.c_int, [_P, _P]),
    "iql_replay_insert_members_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "iql_last_launch_count": (C.c_int64, [_P]),
    "iql_debug_fused_trace": (C.c_int, [_P, C.c_int32]),
    "iql_debug_chain_trace": (C.c_int, [_P, C.c_int32]),
    "iql_debug_step_trace": (C.c_int, [_P, C.c_int32, _P, C.c_int32, _P]),
    "iql_profile_step": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_int32), _P, _P, _P, _P, _P]),
    "iql_selftest_umma_gemm": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, _P, C.c_int32,
                                          _P, C.c_int32, _P, C.c_size_t, _P]),
}

_LIB = None


def lib() -> C.CDLL:
    """Load (once) and return the engine library; raise loudly if it is absent."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA engine is the only compute path of jsrl_corl_b200 "
                "(no CPU fallback). Build it with `python -m jsrl_corl_b200.build`."
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _LIB = handle
    return _LIB


def check(rc: int, handle=None, what: str = ""):
    """Map C status codes to the exception types the reference raises."""
    if rc == IQL_OK:
        return
    msg = lib().iql_last_error(handle)
    msg = msg.decode() if msg else ""
    text = f"{what}: {msg}" if what else msg
    if rc == IQL_ERR_INVALID:
        raise ValueError(text)
    raise RuntimeError(text)


_torch_C = torch._C  # looked up once: call_on_device runs on every host-driven launch


def call_on_device(dev_index: int, device: torch.device, handle, what: str, fn, *args):
    """``fn(*args, stream)`` with ``stream`` the raw handle of torch's current stream on ``device``, run with that device
    current (the caller may sit on another one), a non-zero status raised through ``check`` as ``what``.  ``fn`` is a
    C entry point, or a callable that issues several under the one device switch and returns the last status.
    The host-driven loops call this once per env step or update: the common same-device case enters no context
    manager and uses the raw ``torch._C`` calls (``torch.cuda.current_device()`` costs ~1.5 us of Python,
    ``torch.cuda.current_stream()`` ~7 us)."""
    if _torch_C._cuda_getDevice() == dev_index:
        rc = fn(*args, _torch_C._cuda_getCurrentRawStream(dev_index))
    else:
        with torch.cuda.device(device):
            rc = fn(*args, _torch_C._cuda_getCurrentRawStream(dev_index))
    if rc:
        check(rc, handle, what)


def require_cuda(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda" or not torch.cuda.is_available():
        raise RuntimeError(
            f"jsrl_corl_b200 runs only on a CUDA device (B200, sm_100a); got device={device!r}, "
            f"cuda available={torch.cuda.is_available()}. There is no CPU fallback."
        )
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev
