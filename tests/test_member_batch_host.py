"""Host-side checks of per-member batch sizes (no GPU): the argument checks of iql_set_batch_sizes /
iql_get_batch_sizes and of IQLEnsemble(batch_sizes=...), which run before any device work, and that the JSRL ensemble
loop keeps requiring one batch size for all members."""
import ctypes as C

import numpy as np
import pytest

from jsrl_corl_b200 import _lib


def _handle(S=3, B=8):
    L = _lib.lib()
    h = C.c_void_p()
    cfg = _lib.Config(S, 5, 2, 32, 2, B, 0, 0, 4)
    assert L.iql_create(C.byref(cfg), C.byref(h)) == 0
    return L, h


def _get(L, h, S=3):
    out = np.full(S, -7, np.int32)
    assert L.iql_get_batch_sizes(h, out.ctypes.data) == _lib.IQL_OK
    return out.tolist()


def test_batch_sizes_default_to_the_engine_batch_and_round_trip():
    L, h = _handle()
    try:
        assert _get(L, h) == [8, 8, 8]
        sizes = np.array([1, 5, 8], np.int32)
        assert L.iql_set_batch_sizes(h, sizes.ctypes.data) == _lib.IQL_OK
        assert _get(L, h) == [1, 5, 8]
        # hyper-parameters are set separately and leave the batch sizes alone
        hp = _lib.HParams(beta=1.0, iql_tau=0.7, discount=0.99, tau=0.005, vf_lr=1e-4, qf_lr=1e-4, actor_lr=1e-4,
                          adam_beta1=0.9, adam_beta2=0.999, adam_eps=1e-8, cosine_t_max=10, seed=3)
        assert L.iql_set_hparams(h, 1, C.byref(hp)) == _lib.IQL_OK
        assert _get(L, h) == [1, 5, 8]
    finally:
        L.iql_destroy(h)


@pytest.mark.parametrize("bad", [[0, 8, 8], [8, 9, 8], [8, 8, -1]])
def test_set_batch_sizes_refuses_sizes_out_of_range_and_changes_nothing(bad):
    L, h = _handle()
    try:
        good = np.array([2, 3, 4], np.int32)
        assert L.iql_set_batch_sizes(h, good.ctypes.data) == _lib.IQL_OK
        arr = np.array(bad, np.int32)
        rc = L.iql_set_batch_sizes(h, arr.ctypes.data)
        assert rc == _lib.IQL_ERR_INVALID
        assert b"batch size" in L.iql_last_error(h)
        with pytest.raises(ValueError):
            _lib.check(rc, h, "iql_set_batch_sizes")
        assert _get(L, h) == [2, 3, 4]
    finally:
        L.iql_destroy(h)


def test_batch_size_entry_points_refuse_null_pointers():
    L, h = _handle()
    sizes = np.full(3, 4, np.int32)
    try:
        assert L.iql_set_batch_sizes(h, None) == _lib.IQL_ERR_INVALID
        assert L.iql_get_batch_sizes(h, None) == _lib.IQL_ERR_INVALID
        assert L.iql_set_batch_sizes(None, sizes.ctypes.data) == _lib.IQL_ERR_INVALID
        assert L.iql_get_batch_sizes(None, sizes.ctypes.data) == _lib.IQL_ERR_INVALID
        assert _get(L, h) == [8, 8, 8]
    finally:
        L.iql_destroy(h)


@pytest.mark.parametrize("sizes,what", [([256, 256], "one entry per member"), ([256, 128, 64, 32], "one entry per member"),
                                        ([256, 0, 64], r"\[1, batch_size=256\]"), ([256, 257, 64], r"\[1, batch_size=256\]")])
def test_ensemble_refuses_bad_batch_sizes_before_touching_a_device(sizes, what):
    from jsrl_corl_b200 import IQLEnsemble

    with pytest.raises(ValueError, match=what):
        IQLEnsemble(3, 17, 6, 256, 2, 256, batch_sizes=sizes, device="cuda")


def test_ensemble_loop_still_requires_one_batch_size():
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    cfgs = [JsrlTrainConfig(device="cuda", env="Point-v0", seed=m, eval_freq=10, n_episodes=1, offline_iterations=20,
                            online_iterations=20, batch_size=8 * (m + 1)) for m in range(3)]
    with pytest.raises(ValueError, match="batch_size"):
        ensemble_train_loop(cfgs, [None] * 3, [None] * 3, None, 3, 2, 1.0, 20)
