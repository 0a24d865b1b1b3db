"""Host-side checks of early stopping (no GPU): the ASHA rule of jsrl_corl_b200.asha on hand-worked report sequences,
the argument checks of iql_set_active_members / iql_get_active_members, which run before any device work, and the
config checks of ensemble_train_loop with mixed batch sizes and a scheduler."""
import ctypes as C
import math

import numpy as np
import pytest

from jsrl_corl_b200 import _lib
from jsrl_corl_b200.asha import ASHAScheduler


def _run(sched, reports):
    """reports: [(member, t, score)] -> the decision of each, in order."""
    return [sched.on_result(m, t, s) for m, t, s in reports]


def test_rungs_follow_max_t_grace_period_and_reduction_factor():
    assert ASHAScheduler().milestones == [64, 16, 4, 1]  # Ray's defaults: max_t 100, grace 1, rf 4
    assert ASHAScheduler(max_t=64, reduction_factor=4).milestones == [64, 16, 4, 1]
    assert ASHAScheduler(max_t=50, reduction_factor=4).milestones == [16, 4, 1]  # not a power of rf
    assert ASHAScheduler(max_t=10, grace_period=2, reduction_factor=3).milestones == [6, 2]
    assert ASHAScheduler(max_t=100, grace_period=3, reduction_factor=3).milestones == [81, 27, 9, 3]


def test_rf4_first_rung_by_hand():
    # cutoffs (75th percentile of what the rung holds): -, 5, 4.5, 6.5, 5.75
    s = ASHAScheduler(reduction_factor=4)
    assert _run(s, [(0, 1, 5.0), (1, 1, 3.0), (2, 1, 8.0), (3, 1, 1.0), (4, 1, 6.0)]) == \
        ["continue", "stop", "continue", "stop", "continue"]
    assert s.rungs[-1][1] == {0: 5.0, 1: 3.0, 2: 8.0, 3: 1.0, 4: 6.0}  # recorded either way
    assert sorted(s.stopped) == [1, 3] and s.stopped[1] == (1, None)


def test_rf3_first_rung_by_hand():
    # cutoffs (66.7th percentile): -, 4, 3.333, 5.667
    s = ASHAScheduler(reduction_factor=3)
    assert _run(s, [(0, 1, 4.0), (1, 1, 2.0), (2, 1, 9.0), (3, 1, 3.0)]) == ["continue", "stop", "continue", "stop"]


def test_ties_continue_and_nan_scores_are_ignored():
    s = ASHAScheduler()
    assert _run(s, [(0, 1, 5.0), (1, 1, 5.0)]) == ["continue", "continue"]  # equal to the cutoff is not below it
    s = ASHAScheduler()
    # NaN never stops (NaN < x is false); the rung's only record NaN gives a NaN cutoff (nobody stops); later cutoffs skip it
    assert _run(s, [(0, 1, math.nan), (1, 1, 2.0), (2, 1, 1.0), (3, 1, 1.5)]) == ["continue", "continue", "stop", "stop"]
    assert math.isnan(s.rungs[-1][1][0])


def test_mode_min_negates_the_score():
    s = ASHAScheduler(mode="min")
    # negated: -5, -3, -8; cutoffs -, -5, -3.5: the largest loss stops
    assert _run(s, [(0, 1, 5.0), (1, 1, 3.0), (2, 1, 8.0)]) == ["continue", "continue", "stop"]
    assert s.rungs[-1][1] == {0: -5.0, 1: -3.0, 2: -8.0}


def test_walk_uses_the_highest_rung_not_yet_recorded():
    s = ASHAScheduler()  # rungs 64, 16, 4, 1
    assert _run(s, [(0, 1, 1.0), (1, 1, 2.0)]) == ["continue", "continue"]
    assert s.on_result(0, 2, 0.0) == "continue"  # rung 1 already holds member 0, rung 4 not reached: nothing recorded
    assert [len(r) for _, r in s.rungs] == [0, 0, 0, 2]
    assert s.on_result(1, 4, 7.0) == "continue"  # first at rung 4
    assert s.on_result(0, 4, 3.0) == "stop"  # cutoff at rung 4 = 7
    assert s.rungs[2][1] == {1: 7.0, 0: 3.0}
    # a member that skipped lower rungs is compared at the highest one it reached
    assert s.on_result(5, 20, 1.0) == "continue" and s.rungs[1][1] == {5: 1.0}


def test_max_t_stops_and_grace_period_delays_the_first_rung():
    s = ASHAScheduler(max_t=4, grace_period=1, reduction_factor=4)
    assert s.milestones == [4, 1]
    assert s.on_result(0, 4, 1e9, total_it=123) == "stop"
    assert s.stopped[0] == (4, 123)
    s = ASHAScheduler(max_t=100, grace_period=3, reduction_factor=3)
    assert _run(s, [(0, 1, 5.0), (1, 1, 1.0), (0, 2, 5.0), (1, 2, 1.0)]) == ["continue"] * 4  # before the first rung
    assert all(not r for _, r in s.rungs)
    assert _run(s, [(0, 3, 5.0), (1, 3, 1.0)]) == ["continue", "stop"]


def test_scheduler_refuses_bad_arguments():
    for kw in (dict(mode="best"), dict(grace_period=0), dict(max_t=2, grace_period=3), dict(reduction_factor=1)):
        with pytest.raises(ValueError):
            ASHAScheduler(**kw)


def _handle(S=4, B=8):
    L = _lib.lib()
    h = C.c_void_p()
    cfg = _lib.Config(S, 5, 2, 32, 2, B, 0, 0, 4)
    assert L.iql_create(C.byref(cfg), C.byref(h)) == 0
    return L, h


def _mask(L, h, S=4):
    out = np.full(S, -7, np.int8)
    assert L.iql_get_active_members(h, out.ctypes.data) == _lib.IQL_OK
    return out.tolist()


@pytest.mark.parametrize("ids,what", [([], b"at least one"), ([0, 4], b"out of range"), ([-1], b"out of range"),
                                      ([1, 2, 1], b"listed twice"), ([0, 1, 2, 3, 0], b"listed twice")])
def test_set_active_members_refuses_bad_lists_and_changes_nothing(ids, what):
    L, h = _handle()
    try:
        assert _mask(L, h) == [1, 1, 1, 1]  # default: every member trains
        arr = np.array(ids + [0], np.int32)  # (never an empty buffer)
        rc = L.iql_set_active_members(h, len(ids), arr.ctypes.data)
        assert rc == _lib.IQL_ERR_INVALID
        assert what in L.iql_last_error(h)
        assert _mask(L, h) == [1, 1, 1, 1]
    finally:
        L.iql_destroy(h)


def test_active_members_entry_points_before_bind_and_with_null_pointers():
    L, h = _handle()
    try:
        ids = np.array([0, 2], np.int32)
        assert L.iql_set_active_members(h, 2, ids.ctypes.data) == _lib.IQL_ERR_STATE  # a valid list, but nothing bound
        assert b"not bound" in L.iql_last_error(h)
        assert _mask(L, h) == [1, 1, 1, 1]
        assert L.iql_set_active_members(h, 2, None) == _lib.IQL_ERR_INVALID
        assert L.iql_get_active_members(h, None) == _lib.IQL_ERR_INVALID
        assert L.iql_set_active_members(None, 2, ids.ctypes.data) == _lib.IQL_ERR_INVALID
        assert L.iql_get_active_members(None, ids.ctypes.data) == _lib.IQL_ERR_INVALID
    finally:
        L.iql_destroy(h)


def _configs(sizes, **over):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig

    cfgs = [JsrlTrainConfig(device="cuda", env="Point-v0", seed=m, eval_freq=10, n_episodes=1, offline_iterations=20,
                            online_iterations=20, batch_size=b, beta=1.0 + m) for m, b in enumerate(sizes)]
    for k, v in over.items():
        for c in cfgs:
            setattr(c, k, v)
    return cfgs


def test_ensemble_configs_accept_mixed_batch_sizes_on_request_and_a_scheduler():
    from jsrl_corl_b200.jsrl_w_iql import ENSEMBLE_SHARED_FIELDS, check_ensemble_configs

    assert "batch_size" not in ENSEMBLE_SHARED_FIELDS
    check_ensemble_configs(_configs([8, 16, 32]), mixed_batch_sizes=True)
    check_ensemble_configs(_configs([8, 16, 32]), scheduler=ASHAScheduler(max_t=4), mixed_batch_sizes=True)
    check_ensemble_configs(_configs([256, 1]), scheduler=ASHAScheduler(mode="min"), mixed_batch_sizes=True)
    check_ensemble_configs(_configs([32, 32]), scheduler=ASHAScheduler())
    # without the request one batch size for all members stays the rule, scheduler or not
    for sched in (None, ASHAScheduler()):
        with pytest.raises(ValueError, match="mixed_batch_sizes=True"):
            check_ensemble_configs(_configs([8, 16]), scheduler=sched)


@pytest.mark.parametrize("sizes", [[8, 0, 16], [8, -4], [8, 2.5], [8, True]])
def test_ensemble_configs_refuse_batch_sizes_the_engine_cannot_run(sizes):
    from jsrl_corl_b200.jsrl_w_iql import check_ensemble_configs, ensemble_train_loop

    with pytest.raises(ValueError, match="positive integer"):
        check_ensemble_configs(_configs(sizes), mixed_batch_sizes=True)
    with pytest.raises(ValueError, match="positive integer"):  # before any device work
        ensemble_train_loop(_configs(sizes), [None] * len(sizes), [None] * len(sizes), None, 3, 2, 1.0, 20,
                            mixed_batch_sizes=True)


def test_ensemble_configs_refuse_a_scheduler_without_on_result():
    from jsrl_corl_b200.jsrl_w_iql import check_ensemble_configs

    with pytest.raises(ValueError, match="on_result"):
        check_ensemble_configs(_configs([8, 8]), scheduler=object())
