"""JSRL curriculum / arbitration host logic (SURVEY.md section 8 f-1): hand-derived cases, the documented
quirks, and a differential run against the reference's own jsrl_utils.py when the tree is present."""
import importlib.util
import os
import sys
import types
from collections import deque
from types import SimpleNamespace

import numpy as np
import pytest

from jsrl_corl_b200 import jsrl_utils as J


def _cfg(**kw):
    base = dict(n_curriculum_stages=5, tolerance=0.05, rolling_mean_n=3, horizon_fn="time_step", no_agent_types=True,
                ep_agent_type=0.0, offline_iterations=0)
    base.update(kw)
    return SimpleNamespace(**base)


def test_prepare_finetuning_stage_tables():
    c = J.prepare_finetuning(40, _cfg())
    assert np.allclose(c.all_curriculum_stages, [40, 30, 20, 10, 0])  # time_step: max -> 0
    assert np.allclose(c.all_agent_types, 1) and c.curriculum_stage_idx == 0 and c.curriculum_stage == 40
    assert c.best_eval_score == -np.inf and isinstance(c.rolling_mean_rews, deque) and c.rolling_mean_rews.maxlen == 3
    c = J.prepare_finetuning(8.0, _cfg(horizon_fn="goal_dist", no_agent_types=False))
    assert np.allclose(c.all_curriculum_stages, [0, 2, 4, 6, 8])  # other horizons: 0 -> max
    assert np.allclose(c.all_agent_types, [0, .25, .5, .75, 1]) and c.agent_type_stage == 0
    c = J.prepare_finetuning(8.0, _cfg(n_curriculum_stages=1, no_agent_types=False))
    assert c.agent_type_stage == 1


def test_horizon_update_callback_quirks(capsys):
    c = J.prepare_finetuning(40, _cfg())
    for r in (10.0, 10.0):  # window not full: no advance even though best = -inf
        J.horizon_update_callback(c, r)
        assert c.curriculum_stage_idx == 0
    J.horizon_update_callback(c, 10.0)  # full window, bar = -inf
    assert c.curriculum_stage_idx == 1 and c.best_eval_score == 10.0 and c.curriculum_stage == 30
    J.horizon_update_callback(c, 7.0)  # window (10,10,7) mean 9.0 < 9.5: stay
    assert c.curriculum_stage_idx == 1
    J.horizon_update_callback(c, 12.0)  # window (10,7,12) mean 9.67 >= 9.5: advance, best may DEcrease
    assert c.curriculum_stage_idx == 2 and abs(c.best_eval_score - 29 / 3) < 1e-12
    # the window is not cleared on advance: the very next eval can advance again
    J.horizon_update_callback(c, 12.0)
    assert c.curriculum_stage_idx == 3
    J.horizon_update_callback(c, 50.0)
    assert c.curriculum_stage_idx == 4 and c.curriculum_stage == 0
    best = c.best_eval_score
    J.horizon_update_callback(c, 1000.0)  # last stage: early return, nothing changes but the window
    assert c.curriculum_stage_idx == 4 and c.best_eval_score == best and len(c.rolling_mean_rews) == 3
    # negative returns: the bar best - tol*best is ABOVE best
    c = J.prepare_finetuning(40, _cfg(rolling_mean_n=1))
    J.horizon_update_callback(c, -100.0)
    assert c.curriculum_stage_idx == 1 and c.best_eval_score == -100.0
    J.horizon_update_callback(c, -97.0)  # bar = -100 + 5 = -95 > -97: no advance although the return improved
    assert c.curriculum_stage_idx == 1
    J.horizon_update_callback(c, -95.0)
    assert c.curriculum_stage_idx == 2


def test_horizon_functions():
    c = J.prepare_finetuning(40, _cfg())
    assert J.timestep_horizon(39, None, None, c) == (False, 39)
    assert J.timestep_horizon(40, None, None, c) == (True, 40)
    c.curriculum_stage = np.nan  # offline-phase evaluation: the learner always acts
    assert J.timestep_horizon(0, None, None, c) == (True, 0)
    c = J.prepare_finetuning(40, _cfg(no_agent_types=False))
    c.ep_agent_type = 0.5  # above agent_type_stage 0: the guide keeps control even past the horizon
    assert J.timestep_horizon(100, None, None, c)[0] is False
    c.curriculum_stage_idx = c.n_curriculum_stages - 1
    c.agent_type_stage = 1.0
    assert J.timestep_horizon(0, None, None, c)[0] is True  # last stage: learner from step 0
    env = SimpleNamespace(spec=SimpleNamespace(id="antmaze-umaze-v2"), target_goal=(3.0, 4.0), get_xy=lambda: (0.0, 0.0))
    g = J.prepare_finetuning(10.0, _cfg(horizon_fn="goal_dist"))
    g.curriculum_stage = 5.0
    assert J.goal_distance_horizon(0, None, env, g) == (True, 5.0)
    g.curriculum_stage = 4.9
    assert J.goal_distance_horizon(0, None, env, g)[0] is False
    assert J.max_accumulator([1, 3, 2]) == 3 and J.mean_accumulator([1, 3]) == 2 and J.static_accumulator([9]) == 1
    J.horizon_str = "goal_dist"
    assert J.accumulate([1, 5, 2]) == 5


def test_learner_or_guide_action_arbitration():
    J.horizon_str = "time_step"
    c = J.prepare_finetuning(10, _cfg())
    learner = lambda env, s: np.array([1.0, 1.0])  # noqa: E731  heuristic-style callables
    guide = lambda env, s: np.array([-1.0, -1.0])  # noqa: E731
    a, use, h = J.learner_or_guide_action(np.zeros(3), 3, None, learner, guide, c, "cpu", eval=True)
    assert use is False and h == 3 and np.all(a == -1)
    a, use, h = J.learner_or_guide_action(np.zeros(3), 10, None, learner, guide, c, "cpu", eval=True)
    assert use is True and np.all(a == 1)
    a, use, _ = J.learner_or_guide_action(np.zeros(3), 0, None, learner, None, c, "cpu", eval=True)
    assert use is True  # no guide: the learner always acts
    a, use, _ = J.learner_or_guide_action(np.zeros(3), 0, None, learner, guide, c, "cpu", eval=False)
    import torch
    assert isinstance(a, torch.Tensor) and a.dim() == 1


def test_jsrl_config_fields_and_metrics():
    cfg = J.JsrlTrainConfig()
    for name, default in dict(n_curriculum_stages=10, tolerance=0.05, rolling_mean_n=5, horizon_fn="time_step",
                              new_online_buffer=True, online_buffer_size=10000, max_init_horizon=False,
                              guide_heuristic_fn=None, no_agent_types=True, variance_learn_frac=0.9,
                              downloaded_dataset=None, pretrained_policy_path=None).items():
        assert getattr(cfg, name) == default
    assert cfg.name.startswith("IQL-antmaze-umaze-v2-") and len(cfg.name.split("-")[-1]) == 8
    cfg.curriculum_stage_idx, cfg.curriculum_stage, cfg.best_eval_score = 2, 5.0, 1.5
    cfg.mean_horizon_reached, cfg.eval_mean_agent_type = 3.0, 0.5
    log = J.add_jsrl_metrics({}, cfg)
    assert log["eval/jsrl/curriculum_stage"] == 5.0 and len(log) == 5


def _load_reference_jsrl():
    from oracle.ref_loader import REFERENCE_ROOT, _install_stubs, reference_available

    if not reference_available():
        return None
    _install_stubs()
    fin = os.path.join(REFERENCE_ROOT, "algorithms", "finetune")
    for name in ("stable_baselines3", "matplotlib", "matplotlib.pyplot", "h5py", "ray", "gymnasium_robotics"):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    sb3 = sys.modules["stable_baselines3"]
    if not hasattr(sb3, "SAC"):
        sb3.SAC = object
        sb3.sac = types.ModuleType("stable_baselines3.sac")
        sb3.sac.policies = types.ModuleType("stable_baselines3.sac.policies")
        sb3.sac.policies.Actor = type("Actor", (), {})
    sys.path.insert(0, fin)
    try:
        spec = importlib.util.spec_from_file_location("_ref_jsrl_utils", os.path.join(fin, "jsrl_utils.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    except Exception:
        return None
    finally:
        sys.path.remove(fin)
        for m in ("iql", "goal_horizon_fns", "guide_heuristics", "variance_learner"):
            sys.modules.pop(m, None)


def test_curriculum_differential_against_reference(capsys):
    ref = _load_reference_jsrl()
    if ref is None:
        pytest.skip("needs the original jsrl-CORL finetune/jsrl_utils.py importable under JSRL_REFERENCE_ROOT; "
                    "no stored outputs of it exist for this comparison")
    rng = np.random.RandomState(0)
    for trial in range(40):
        kw = dict(n_curriculum_stages=int(rng.randint(1, 8)), tolerance=float(rng.choice([0.0, 0.05, 0.3])),
                  rolling_mean_n=int(rng.randint(1, 6)), horizon_fn=str(rng.choice(["time_step", "goal_dist", "agent_type"])),
                  no_agent_types=bool(rng.randint(2)))
        init_h = float(rng.uniform(1, 100))
        a, b = J.prepare_finetuning(init_h, _cfg(**kw)), ref.prepare_finetuning(init_h, _cfg(**kw))
        assert np.array_equal(a.all_curriculum_stages, b.all_curriculum_stages)
        assert np.array_equal(a.all_agent_types, b.all_agent_types) and a.agent_type_stage == b.agent_type_stage
        for r in rng.normal(rng.choice([-50, 0, 50]), 20, size=30):
            J.horizon_update_callback(a, float(r))
            ref.horizon_update_callback(b, float(r))
            assert (a.curriculum_stage_idx, a.best_eval_score, list(a.rolling_mean_rews)) == \
                   (b.curriculum_stage_idx, b.best_eval_score, list(b.rolling_mean_rews))
            assert a.curriculum_stage == b.curriculum_stage and a.agent_type_stage == b.agent_type_stage
            for step in (0, 5, 50):
                a.ep_agent_type = b.ep_agent_type = float(rng.uniform())
                np.random.seed(trial)
                ra = J.HORIZON_FNS[kw["horizon_fn"]]["horizon_fn"](step, np.zeros(8), SimpleNamespace(spec=SimpleNamespace(id="LunarLander-v2")), a)
                np.random.seed(trial)
                rb = ref.HORIZON_FNS[kw["horizon_fn"]]["horizon_fn"](step, np.zeros(8), SimpleNamespace(spec=SimpleNamespace(id="LunarLander-v2")), b)
                assert bool(ra[0]) == bool(rb[0]) and ra[1] == rb[1]
