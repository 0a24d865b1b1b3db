"""Host-side checks of the training-mode act with actor dropout (no GPU): the source codes 4 / 5 and their refusals, the
act counter entry points, the oracle's act masks, and the opt-in of ensemble_train_loop, all of which run before any
device work."""
import ctypes as C

import numpy as np
import pytest

from jsrl_corl_b200 import _lib
from act_mask_oracle import STREAM_ACT_DROPOUT_BASE, philox_act_dropout_mask
from oracle.philox import dropout_threshold, philox4x32_10, philox_dropout_mask


def _handle(S=3, det=0):
    L = _lib.lib()
    h = C.c_void_p()
    cfg = _lib.Config(S, 5, 2, 32, 2, 8, det, 0, 4)
    assert L.iql_create(C.byref(cfg), C.byref(h)) == 0
    return L, h


def _act(L, h, codes, std=True):
    S = len(codes)
    states = np.zeros((S, 5), np.float32)
    src = np.asarray(codes, np.int8)
    out = np.zeros((S, 2), np.float32)
    sd = np.zeros((S, 2), np.float32)
    return L.iql_act_host_members(h, states.ctypes.data, src.ctypes.data, 1.0, out.ctypes.data,
                                  sd.ctypes.data if std else None, None, None)


def test_new_symbols_and_codes_are_exported():
    L = _lib.lib()
    for name in ("iql_get_act_steps", "iql_set_act_steps"):
        assert name in _lib.SYMBOLS and getattr(L, name)
    text = open(_lib.os.path.join(_lib._HERE, "..", "include", "iql_b200.h")).read()
    assert f"#define IQL_ACT_LEARNER_DROPOUT {_lib.ACT_LEARNER_DROPOUT} " in text
    assert f"#define IQL_ACT_LEARNER_DIST_DROPOUT {_lib.ACT_LEARNER_DIST_DROPOUT} " in text
    assert (_lib.ACT_LEARNER_DROPOUT, _lib.ACT_LEARNER_DIST_DROPOUT) == (4, 5)
    assert _lib.ACT_SOURCES["learner_dropout"] == 4 and _lib.ACT_SOURCES["learner_dist_dropout"] == 5


def test_source_code_refusals():
    L, h = _handle(det=1)
    try:
        assert _act(L, h, [0, 5, 0]) == _lib.IQL_ERR_INVALID  # distribution code on a deterministic policy
        assert b"deterministic" in L.iql_last_error(h)
        assert _act(L, h, [0, 7, 0]) == _lib.IQL_ERR_INVALID
        assert b"unknown source" in L.iql_last_error(h)
        assert _act(L, h, [6, 0, 0]) == _lib.IQL_ERR_INVALID
        assert _act(L, h, [-1, 0, 0]) == _lib.IQL_ERR_INVALID
        assert _act(L, h, [0, 4, 0]) == _lib.IQL_ERR_STATE  # a valid code: refused only because nothing is bound
        steps = np.full(3, 99, np.uint64)
        assert L.iql_get_act_steps(h, steps.ctypes.data) == _lib.IQL_OK
        assert steps.tolist() == [0, 0, 0]  # refused calls move no counter
    finally:
        L.iql_destroy(h)
    L, h = _handle(det=0)
    try:
        assert _act(L, h, [5, 0, 0], std=False) == _lib.IQL_ERR_INVALID  # distribution members need the std array
        assert b"null std" in L.iql_last_error(h)
        assert _act(L, h, [5, 2, 4]) == _lib.IQL_ERR_STATE
    finally:
        L.iql_destroy(h)


def test_act_steps_round_trip_and_argument_checks():
    L, h = _handle(S=4)
    try:
        v = np.array([0, 7, 2 ** 40 + 3, 2 ** 64 - 1], np.uint64)
        assert L.iql_set_act_steps(h, v.ctypes.data) == _lib.IQL_OK
        got = np.zeros(4, np.uint64)
        assert L.iql_get_act_steps(h, got.ctypes.data) == _lib.IQL_OK
        assert np.array_equal(got, v)
        assert L.iql_get_act_steps(h, None) == _lib.IQL_ERR_INVALID
        assert L.iql_set_act_steps(h, None) == _lib.IQL_ERR_INVALID
        assert L.iql_get_act_steps(None, got.ctypes.data) == _lib.IQL_ERR_INVALID
        assert L.iql_set_act_steps(None, got.ctypes.data) == _lib.IQL_ERR_INVALID
    finally:
        L.iql_destroy(h)


def test_engine_set_act_steps_refuses_wrong_length_and_negative_values():
    from jsrl_corl_b200.engine import EnsembleEngine

    L, h = _handle(S=3)
    eng = object.__new__(EnsembleEngine)  # the host-side part of an engine; no device is touched
    eng._L, eng._h, eng.n_members = L, h, 3
    eng.set_act_steps([1, 2, 3])
    assert eng.act_steps.tolist() == [1, 2, 3] and eng.act_steps.dtype == np.uint64
    for bad in ([1, 2], [1, 2, 3, 4], []):
        with pytest.raises(ValueError, match="one act counter per member"):
            eng.set_act_steps(bad)
    with pytest.raises(ValueError, match="non-negative"):
        eng.set_act_steps([1, -2, 3])
    with pytest.raises(ValueError, match="non-negative"):
        eng.set_act_steps([1.0, 2.0, 3.0])
    assert eng.act_steps.tolist() == [1, 2, 3]  # nothing changed by the refused calls


def test_oracle_act_mask_formula():
    seed, step, layer, n, p = (5 << 40) | 17, (3 << 32) | 11, 1, 256, 0.1
    mask = philox_act_dropout_mask(seed, step, layer, n, p)
    x, y, z, w = philox4x32_10(np.arange(n // 4), step & 0xFFFFFFFF, step >> 32, STREAM_ACT_DROPOUT_BASE + layer,
                               seed & 0xFFFFFFFF, seed >> 32)
    words = np.stack([x, y, z, w], 1).reshape(-1)
    assert np.array_equal(mask, (words >= dropout_threshold(p)).astype(np.uint8))
    assert philox_act_dropout_mask(seed, step, layer, n, 0.0).all()
    # n not a multiple of 4: the leading units of the last quad
    assert np.array_equal(philox_act_dropout_mask(seed, step, layer, 10, p), mask[:10])
    # the act stream is not the update's: different masks for the same key, counter and layer
    assert not np.array_equal(mask, philox_dropout_mask(seed, step, layer, n, p))


def _configs(n=3, **over):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig

    cfgs = [JsrlTrainConfig(device="cuda", env="Point-v0", seed=m, eval_freq=10, n_episodes=1, offline_iterations=20,
                            online_iterations=20, batch_size=8, beta=1.0 + m, tolerance=0.1 * (m + 1)) for m in range(n)]
    for c in cfgs:
        for k, v in over.items():
            setattr(c, k, v)
    return cfgs


@pytest.mark.parametrize("det", [False, True])
def test_ensemble_loop_dropout_needs_the_opt_in(det):
    from jsrl_corl_b200.jsrl_w_iql import check_ensemble_configs, ensemble_train_loop

    cfgs = _configs(actor_dropout=0.1, iql_deterministic=det)
    with pytest.raises(NotImplementedError, match="philox_act_dropout=True"):
        check_ensemble_configs(cfgs)
    with pytest.raises(NotImplementedError, match="dropout"):
        ensemble_train_loop(cfgs, [None] * 3, [None] * 3, None, 3, 2, 1.0, 20)
    check_ensemble_configs(cfgs, philox_act_dropout=True)
    check_ensemble_configs(_configs(), philox_act_dropout=True)  # the opt-in without dropout changes nothing
    # the dropout rate is still one value for every member
    cfgs[1].actor_dropout = 0.2
    with pytest.raises(ValueError, match="actor_dropout"):
        check_ensemble_configs(cfgs, philox_act_dropout=True)
