"""Host-side checks of the ensemble online path (no GPU): argument and call-order errors of the batched act / ring
insert / guide entry points, and the config checks of ensemble_train_loop, which run before any device work."""
import ctypes as C

import numpy as np
import pytest

from jsrl_corl_b200 import _lib


def _handle(S=3, det=0):
    L = _lib.lib()
    h = C.c_void_p()
    cfg = _lib.Config(S, 5, 2, 32, 2, 8, det, 0, 4)
    assert L.iql_create(C.byref(cfg), C.byref(h)) == 0
    return L, h


def test_batched_entry_points_refuse_before_binding_and_on_null_pointers():
    L, h = _handle()
    S = 3
    states = np.zeros((S, 5), np.float32)
    src = np.ones(S, np.int8)
    out = np.zeros((S, 2), np.float32)
    r = np.zeros(S, np.float32)
    ptr = np.zeros(S, np.int64)
    try:
        rc = L.iql_act_host_members(h, states.ctypes.data, src.ctypes.data, 1.0, out.ctypes.data, None, None, None)
        assert rc == _lib.IQL_ERR_STATE and b"not bound" in L.iql_last_error(h)
        rc = L.iql_replay_insert_members_host(h, states.ctypes.data, out.ctypes.data, r.ctypes.data, states.ctypes.data,
                                              r.ctypes.data, ptr.ctypes.data, None, None)
        assert rc == _lib.IQL_ERR_STATE and b"not bound" in L.iql_last_error(h)
        assert L.iql_act_host_members(h, None, src.ctypes.data, 1.0, out.ctypes.data, None, None, None) == _lib.IQL_ERR_INVALID
        assert L.iql_act_host_members(h, states.ctypes.data, None, 1.0, out.ctypes.data, None, None, None) == _lib.IQL_ERR_INVALID
        assert L.iql_act_host_members(h, states.ctypes.data, src.ctypes.data, 1.0, None, None, None, None) == _lib.IQL_ERR_INVALID
        for k in range(6):
            args = [states.ctypes.data, out.ctypes.data, r.ctypes.data, states.ctypes.data, r.ctypes.data, ptr.ctypes.data]
            args[k] = None
            assert L.iql_replay_insert_members_host(h, *args, None, None) == _lib.IQL_ERR_INVALID
        assert L.iql_bind_guide(h, 4) == _lib.IQL_ERR_INVALID  # unaligned arena
        assert b"aligned" in L.iql_last_error(h)
        assert L.iql_bind_guide(h, None) == _lib.IQL_OK  # unbinding is always allowed
        assert L.iql_bind_guide(None, None) == _lib.IQL_ERR_INVALID
        assert L.iql_act_host_members(None, states.ctypes.data, src.ctypes.data, 1.0, out.ctypes.data, None, None, None) == _lib.IQL_ERR_INVALID
        assert L.iql_replay_insert_members_host(None, *([None] * 8)) == _lib.IQL_ERR_INVALID
    finally:
        L.iql_destroy(h)


def test_act_source_codes_match_the_header():
    text = open(_lib.os.path.join(_lib._HERE, "..", "include", "iql_b200.h")).read()
    for name, code in (("SKIP", _lib.ACT_SKIP), ("LEARNER", _lib.ACT_LEARNER), ("LEARNER_DIST", _lib.ACT_LEARNER_DIST),
                       ("GUIDE", _lib.ACT_GUIDE)):
        assert f"#define IQL_ACT_{name} {code} " in text


def _configs(n=3, **over):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig

    cfgs = [JsrlTrainConfig(device="cuda", env="Point-v0", seed=m, eval_freq=10, n_episodes=1, offline_iterations=20,
                            online_iterations=20, batch_size=8, beta=1.0 + m, tolerance=0.1 * (m + 1)) for m in range(n)]
    for k, v in over.items():
        setattr(cfgs[-1], k, v)
    return cfgs


@pytest.mark.parametrize("field,value", [("batch_size", 16), ("offline_iterations", 21), ("online_iterations", 5),
                                         ("eval_freq", 5), ("n_episodes", 2), ("horizon_fn", "agent_type"),
                                         ("iql_deterministic", True), ("actor_dropout", 0.1), ("new_online_buffer", False)])
def test_ensemble_loop_rejects_differing_shared_fields(field, value):
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    with pytest.raises(ValueError, match=field):
        ensemble_train_loop(_configs(**{field: value}), [None] * 3, [None] * 3, None, 3, 2, 1.0, 20)


@pytest.mark.parametrize("over,what", [({"guide_heuristic_fn": "h"}, "heuristic"), ({"pretrained_policy_path": "x.pt"}, "pretrained"),
                                       ({"horizon_fn": "variance"}, "variance"), ({"actor_dropout": 0.1}, "dropout")])
def test_ensemble_loop_rejects_out_of_scope_options(over, what):
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    cfgs = _configs()
    for c in cfgs:  # the same value for every member, so only the scope check can refuse it
        for k, v in over.items():
            setattr(c, k, v)
    with pytest.raises(NotImplementedError, match=what):
        ensemble_train_loop(cfgs, [None] * 3, [None] * 3, None, 3, 2, 1.0, 20)


def test_ensemble_loop_accepts_per_member_fields():
    from jsrl_corl_b200.jsrl_w_iql import check_ensemble_configs

    cfgs = _configs()
    cfgs[1].n_curriculum_stages, cfgs[2].expl_noise, cfgs[0].qf_lr = 1, 0.2, 1e-3
    check_ensemble_configs(cfgs)
