"""Offline -> online JSRL driver loop on the B200 IQL engine: the host-side mirror of
``algorithms/finetune/jsrl_w_iql.py:62-263, 432-606`` of the reference for continuous-action envs.

Kept from the reference: guide-only evaluation to find the initial horizon, the fresh online learner
and the 10k-row online ring, ``ep_agent_type`` bookkeeping, exploration noise / sampling of learner
actions, ``real_done`` excluding time-outs, the update gate on the GLOBAL iteration counter
(``t >= batch_size`` with a new online buffer), evaluation every ``eval_freq`` iterations, the
curriculum callback and checkpoints named ``checkpoint_{t}.pt``.  Replaced: wandb / ray.tune by a
``log`` callable; env construction, D4RL download and dataset normalisation stay with the caller.
Discrete-action heuristics guides (LunarLander / CartPole) are out of scope.
"""
from __future__ import annotations

import os
from typing import Callable, Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib as _lib_codes
from . import jsrl_utils as jsrl
from .iql import (DeterministicPolicy, GaussianPolicy, ReplayBuffer, is_goal_reached, modify_reward_online)


def _is_gymnasium(env) -> bool:
    return "gymnasium" in str(type(env))


def _reset(env, seed=None):
    if _is_gymnasium(env):
        state, _ = env.reset(seed=seed) if seed is not None else env.reset()
        return state
    if seed is not None and hasattr(env, "seed"):
        env.seed(seed)
    state = env.reset()
    return state[0] if isinstance(state, tuple) else state


def _step(env, action):
    out = env.step(action)
    if len(out) == 5:
        state, reward, term, trunc, info = out
        return state, reward, bool(term or trunc), info
    return out


@torch.no_grad()
def eval_actor(env, learner, guide, config) -> Tuple[np.ndarray, float, float, float]:
    """n_episodes mixed guide/learner rollouts; returns (returns, success rate, horizon, mean agent type).
    With ``guide is None`` the "learner" is the guide being probed for the initial horizon."""
    is_module = isinstance(learner, (GaussianPolicy, DeterministicPolicy))
    if is_module:
        learner.eval()
    returns, successes, horizons, agent_types = [], [], [], []
    for ep in range(config.n_episodes):
        state = _reset(env, config.seed if ep == 0 else None)
        done, ts, ep_ret, goal = False, 0, 0.0, False
        ep_horizons, ep_types = [], []
        while not done:
            config.ep_agent_type = 0 if ts == 0 else np.mean(ep_types)
            action, use_learner, horizon = jsrl.learner_or_guide_action(state, ts, env, learner, guide, config,
                                                                        config.device, eval=True)
            ep_horizons.append(horizon)
            ep_types.append(1 if use_learner else 0)
            state, reward, done, info = _step(env, action)
            ep_ret += reward
            ts += 1
            goal = goal or is_goal_reached(reward, info)
        successes.append(float(goal))
        returns.append(ep_ret)
        probing = guide is None and config.max_init_horizon
        horizons.append(np.max(ep_horizons) if probing else jsrl.accumulate(ep_horizons))
        agent_types.append(np.mean(ep_types))
    horizon = np.max(horizons) if (guide is None and config.max_init_horizon) else np.mean(horizons)
    if is_module:
        learner.train()
    return np.asarray(returns), float(np.mean(successes)), horizon, float(np.mean(agent_types))


def jsrl_online_actor(config, env, trainer, state_dim, action_dim, max_action, heuristics=None):
    """Switch to the online phase: evaluate the guide alone for the initial horizon, then build the learner."""
    config.curriculum_stage = np.nan
    guide, guide_trainer = jsrl.get_guide_agent(config, trainer, state_dim, action_dim, max_action, heuristics)
    _, _, init_horizon, _ = eval_actor(env, guide, None, config)
    trainer, config = jsrl.get_learning_agent(config, guide_trainer, init_horizon, state_dim, action_dim, max_action)
    return trainer, guide, config


def make_offline_buffer(config, dataset: Dict[str, np.ndarray], state_dim: int, action_dim: int, max_episode_steps: int = 1000):
    """Dataset -> device replay buffer the way the reference driver does it (jsrl_w_iql.py:344-368), with the
    arithmetic on the GPU: ``return_reward_range`` (host scan, as in the reference) gives the locomotion reward range,
    ``ReplayBuffer.ingest_d4rl_dataset`` computes the state statistics, normalises, rescales rewards and packs.
    Returns (replay_buffer, state_mean, state_std, reward_mod_dict); wrap the envs with the statistics as before."""
    from .iql import return_reward_range

    reward_mod, shift = {}, 0.0
    if config.normalize_reward:
        if any(s in config.env for s in ("halfcheetah", "hopper", "walker2d")):
            lo, hi = return_reward_range(dataset, max_episode_steps)
            reward_mod = {"max_ret": hi, "min_ret": lo, "max_episode_steps": max_episode_steps}
        elif "antmaze" in config.env:
            shift = 1.0
    rb = ReplayBuffer(state_dim, action_dim, config.buffer_size, config.device)
    mean, std = rb.ingest_d4rl_dataset(dataset, normalize=bool(config.normalize), eps=1e-3, reward_mod=reward_mod or None,
                                       reward_shift=shift)
    return rb, mean, std, reward_mod


def train_loop(config, env, eval_env, replay_buffer: Optional[ReplayBuffer], state_dim: int, action_dim: int,
               max_action: float, max_steps: int, log: Optional[Callable[[Dict, int], None]] = None,
               reward_mod_dict: Optional[Dict] = None, heuristics=None, is_env_with_goal: bool = False):
    """Run ``offline_iterations`` updates on ``replay_buffer`` then ``online_iterations`` env steps with one
    update each.  Returns (trainer, config, history of eval logs)."""
    log = log or (lambda d, step: None)
    config.discrete = False
    jsrl.horizon_str = config.horizon_fn
    if config.pretrained_policy_path is not None:
        config.offline_iterations = 0  # reference quirk: a pretrained guide skips the offline phase
    trainer = actor = guide = None
    if config.offline_iterations > 0 or config.pretrained_policy_path is None:
        trainer = jsrl.make_actor(config, state_dim, action_dim, max_action, max_steps=config.offline_iterations)
        actor = trainer.actor
    if config.checkpoints_path is not None:
        os.makedirs(config.checkpoints_path, exist_ok=True)
    state = _reset(env, config.seed)
    ep_ret, ep_step, goal = 0.0, 0, False
    eval_successes, train_successes, history = [], [], []
    online_buffer, ep_types = None, []
    for t in range(int(config.offline_iterations) + int(config.online_iterations)):
        if t == config.offline_iterations:
            trainer, guide, config = jsrl_online_actor(config, env, trainer, state_dim, action_dim, max_action, heuristics)
            actor = trainer.actor
            online_buffer = jsrl.get_online_buffer(config, replay_buffer, state_dim, action_dim)
            state = _reset(env)
        online_log = {}
        if t >= config.offline_iterations:
            if ep_step == 0:
                ep_types = []
                config.ep_agent_type = 0
            else:
                config.ep_agent_type = np.mean(ep_types)
            action, use_learner, _ = jsrl.learner_or_guide_action(state, ep_step, env, actor, guide, config, config.device,
                                                                  as_numpy=True)
            ep_types.append(1 if use_learner else 0)
            if isinstance(action, np.ndarray):
                # engine-backed policies hand back numpy: the exploration noise still comes from torch's CPU generator
                # (what `torch.randn_like` of the reference's CPU action tensor draws from), everything else stays numpy
                if use_learner and config.iql_deterministic:
                    noise = (torch.randn(action.shape[0]) * config.expl_noise).clamp(-config.noise_clip, config.noise_clip)
                    action = action + noise.numpy()
                action = np.clip(max_action * action, -max_action, max_action).astype(np.float32).flatten()
            else:
                if use_learner and config.iql_deterministic:
                    noise = (torch.randn_like(action) * config.expl_noise).clamp(-config.noise_clip, config.noise_clip)
                    action = action + noise
                action = torch.clamp(max_action * action, -max_action, max_action).cpu().numpy().flatten()
            next_state, reward, done, info = _step(env, action)
            ep_step += 1
            goal = goal or is_goal_reached(reward, info)
            ep_ret += reward
            real_done = bool(done and ep_step < max_steps)  # time-outs are not terminals
            if config.normalize_reward and reward_mod_dict is not None:
                reward = modify_reward_online(reward, config.env, **reward_mod_dict)
            online_buffer.add_transition(state, action, reward, next_state, real_done)
            state = next_state
            if done:
                state = _reset(env)
                if is_env_with_goal:
                    train_successes.append(goal)
                    online_log["train/regret"] = float(np.mean(1 - np.array(train_successes)))
                    online_log["train/is_success"] = float(goal)
                online_log.update({"train/episode_return": ep_ret, "train/mean_ep_agent_type": float(np.mean(ep_types)),
                                   "train/episode_length": ep_step})
                ep_ret, ep_step, goal = 0.0, 0, False
        if t >= config.batch_size or not config.new_online_buffer:
            buf = online_buffer if t >= config.offline_iterations else replay_buffer
            log_dict = trainer.train(buf.sample(config.batch_size))
            if t < config.offline_iterations:
                log_dict["offline_iter"] = t
            else:
                log_dict["online_iter"] = t - config.offline_iterations
            log_dict.update(online_log)
            log(log_dict, trainer.total_it)
            if (t + 1) % config.eval_freq == 0:
                if t < config.offline_iterations:
                    guide = None
                if guide is None:
                    config.curriculum_stage = np.nan
                scores, success, config.mean_horizon_reached, config.eval_mean_agent_type = eval_actor(eval_env, actor, guide, config)
                score = float(scores.mean())
                # reference jsrl_w_iql.py:573-592: with normalize_reward the curriculum callback and the log see the
                # D4RL-normalised score (an affine rescale changes when `best - tol * best` is reached)
                norm_fn = getattr(eval_env, "get_normalized_score", None) if config.normalize_reward else None
                if norm_fn is not None:
                    score = float(norm_fn(score))  # the callback sees this value; the log 100x it (reference :587)
                eval_log = {}
                if is_env_with_goal:
                    eval_successes.append(success)
                    eval_log["eval/regret"] = float(np.mean(1 - np.array(eval_successes)))
                    eval_log["eval/success_rate"] = success
                if t >= config.offline_iterations:
                    config = jsrl.horizon_update_callback(config, score)
                    eval_log = jsrl.add_jsrl_metrics(eval_log, config)
                if norm_fn is not None:
                    eval_log["eval/d4rl_normalized_score"] = score * 100.0
                else:
                    eval_log["eval/score"] = score
                if config.checkpoints_path is not None:
                    torch.save(trainer.state_dict(), os.path.join(config.checkpoints_path, f"checkpoint_{t}.pt"))
                log(eval_log, trainer.total_it)
                history.append(dict(eval_log, t=t))
    return trainer, config, history


# ---------------------------------------------------------------------------
# S members through the whole JSRL run at once (the reference's process-per-seed launchers, ray_trainer.py)
# ---------------------------------------------------------------------------
# fields every member of an ensemble run must share: the loop runs all members in lockstep (iteration counts,
# evaluation points), `horizon_fn` is a module global of jsrl_utils, and the policy type / dropout / online buffer rule
# fix the engine shape and the update gate.  `batch_size` is checked on its own: it must be the same for every member
# unless the caller asks for per-member batch sizes (`mixed_batch_sizes=True`); then the engine runs the largest,
# member m trains on its own B_m rows (IQLEnsemble(batch_sizes=...)) and its gate `t >= B_m` keeps it inactive until it
# opens.  `actor_dropout` > 0 needs `philox_act_dropout=True`: the learners' training-mode acts then draw their dropout
# masks from the engine's Philox stream, not from torch's, so the loop asks the caller to say so.
ENSEMBLE_SHARED_FIELDS = ("offline_iterations", "online_iterations", "eval_freq", "n_episodes", "horizon_fn",
                          "iql_deterministic", "actor_dropout", "new_online_buffer")


def check_ensemble_configs(configs, scheduler=None, mixed_batch_sizes: bool = False, philox_act_dropout: bool = False):
    """Refuse (ValueError) configs whose shared fields differ, whose batch sizes differ without ``mixed_batch_sizes``
    or are not positive integers, a scheduler without ``on_result``, and (NotImplementedError) the options the
    ensemble loop does not cover, actor dropout without ``philox_act_dropout``.  Touches no device."""
    if len(configs) == 0:
        raise ValueError("ensemble_train_loop needs at least one config")
    for f in ENSEMBLE_SHARED_FIELDS:
        vals = [getattr(c, f) for c in configs]
        if any(v != vals[0] for v in vals[1:]):
            raise ValueError(f"ensemble_train_loop: `{f}` must be the same for every member, got {vals}")
    sizes = [c.batch_size for c in configs]
    if any(not isinstance(b, (int, np.integer)) or isinstance(b, bool) or b < 1 for b in sizes):
        raise ValueError(f"ensemble_train_loop: every `batch_size` must be a positive integer, got {sizes}")
    if not mixed_batch_sizes and any(b != sizes[0] for b in sizes[1:]):
        raise ValueError(f"ensemble_train_loop: `batch_size` must be the same for every member, got {sizes} (pass "
                         "mixed_batch_sizes=True to train each member on its own batch size)")
    if scheduler is not None and not callable(getattr(scheduler, "on_result", None)):
        raise ValueError("ensemble_train_loop: the scheduler needs an on_result(member, t, score, total_it) method "
                         "(jsrl_corl_b200.asha.ASHAScheduler)")
    c0 = configs[0]
    for c in configs:
        if getattr(c, "guide_heuristic_fn", None) is not None:
            raise NotImplementedError("ensemble_train_loop: heuristic guides are host functions of one env; the ensemble's "
                                      "guides are its offline members (use train_loop)")
        if getattr(c, "pretrained_policy_path", None) is not None:
            raise NotImplementedError("ensemble_train_loop: pretrained guides (pretrained_policy_path) are not supported; "
                                      "the guides are the members trained in the offline phase")
    if c0.horizon_fn == "variance":
        raise NotImplementedError("ensemble_train_loop: the `variance` horizon needs a value network per member on the host")
    if c0.horizon_fn not in jsrl.HORIZON_FNS:
        raise ValueError(f"unknown horizon_fn {c0.horizon_fn!r}")
    if c0.actor_dropout and not philox_act_dropout:
        raise NotImplementedError("ensemble_train_loop: training-mode act with active actor dropout has no engine kernel "
                                  "(the single-learner path falls back to stock torch there); pass philox_act_dropout=True "
                                  "to draw the learners' act masks in the engine's act kernel from its Philox stream")


def member_networks(config, state_dim: int, action_dim: int, max_action: float):
    """Initial networks of one member: ``torch.manual_seed(config.seed)``, then the offline TwinQ / ValueFunction /
    policy and the online learner's, in the reference's construction order (jsrl_utils.py:219-282), the learner's
    drawn right after the offline ones.  The global torch RNG is left as it was.  Returns ((q, v, actor), (q, v,
    actor)) as CPU modules with the class-default 2x256 networks of ``make_actor``."""
    from .iql import TwinQ, ValueFunction

    cls = DeterministicPolicy if config.iql_deterministic else GaussianPolicy
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(config.seed)
        nets = []
        for _ in range(2):
            nets.append((TwinQ(state_dim, action_dim), ValueFunction(state_dim),
                         cls(state_dim, action_dim, max_action, dropout=config.actor_dropout)))
    return nets[0], nets[1]


def _member_hparams(c, t_max: int) -> Dict:
    return dict(beta=c.beta, iql_tau=c.iql_tau, discount=c.discount, tau=c.tau, vf_lr=c.vf_lr, qf_lr=c.qf_lr,
                actor_lr=c.actor_lr, cosine_t_max=int(t_max))


def _build_ensemble(configs, nets, state_dim, action_dim, t_max, device, learner: bool = False):
    """``learner`` (with actor dropout): the members' Philox keys get bit 63 set, so that a learner's masks -- of its
    updates and of its training-mode acts -- never repeat those its guide (the offline member of the same seed) drew."""
    from .ensemble import IQLEnsemble

    c0 = configs[0]
    sizes = [int(c.batch_size) for c in configs]
    p = float(c0.actor_dropout or 0.0)
    keys = [int(c.seed) | (1 << 63) if learner and p > 0.0 else c.seed for c in configs]
    ens = IQLEnsemble(len(configs), state_dim, action_dim, 256, 2, max(sizes), deterministic=c0.iql_deterministic,
                      actor_dropout=p, device=device, max_steps_per_call=max(1, min(256, int(c0.eval_freq))), seeds=keys,
                      hparams=[_member_hparams(c, t_max) for c in configs], init=False,
                      batch_sizes=sizes if len(set(sizes)) > 1 else None)
    for m, (q, v, actor) in enumerate(nets):
        ens.engine.load_params(m, {"qf": q.state_dict(), "vf": v.state_dict(), "actor": actor.state_dict()},
                               dropout_keys=p > 0.0)
    return ens


def _sync_active(ens, want: np.ndarray):
    """Make the members in ``want`` (bool [S], not all False) the ones that train; no call when nothing changes."""
    if not np.array_equal(ens.active, want):
        ens.engine.set_active(np.flatnonzero(want))


@torch.no_grad()
def ensemble_eval_actor(envs, ensemble, use_guide: bool, configs, max_action: float, members=None):
    """``eval_actor`` for every member at once (for those whose ``members`` entry is true, when given; the others get
    None): member m plays ``n_episodes`` episodes on ``envs[m]`` with
    ``ensemble``'s member m as the learner and, with ``use_guide``, the guide bound by ``set_guide`` as the guide.
    All members step in lockstep with one act launch per step; members whose episodes are over are skipped.  Each
    member's episodes are exactly those ``eval_actor`` plays for it alone (the horizon function reads and
    ``config.ep_agent_type`` is written per member).  Returns one (returns, success rate, horizon, mean agent type)
    tuple per member."""
    S = len(configs)
    hfn = jsrl.HORIZON_FNS[jsrl.horizon_str]["horizon_fn"]
    n_ep = configs[0].n_episodes
    states = np.zeros((S, ensemble.engine.state_dim), dtype=np.float32)
    source = np.zeros(S, dtype=np.int8)
    out = np.zeros((S, ensemble.engine.action_dim), dtype=np.float32)
    ep = [0] * S
    chosen = [True] * S if members is None else [bool(x) for x in members]
    live = [n_ep > 0 and chosen[m] for m in range(S)]
    fresh = [True] * S
    raw_state = [None] * S
    acc = [dict(returns=[], successes=[], horizons=[], agent_types=[]) for _ in range(S)]
    cur = [None] * S
    while any(live):
        for m in range(S):
            source[m] = 0
            if not live[m]:
                continue
            c = configs[m]
            if fresh[m]:
                raw_state[m] = _reset(envs[m], c.seed if ep[m] == 0 else None)
                cur[m] = dict(ts=0, ret=0.0, goal=False, horizons=[], types=[])
                fresh[m] = False
            e = cur[m]
            c.ep_agent_type = 0 if e["ts"] == 0 else np.mean(e["types"])
            use_learner, horizon = hfn(e["ts"], raw_state[m], envs[m], c)
            if not use_guide:
                use_learner = True
            e["horizons"].append(horizon)
            e["types"].append(1 if use_learner else 0)
            states[m] = np.asarray(raw_state[m], dtype=np.float32).reshape(-1)
            source[m] = _lib_codes.ACT_LEARNER if use_learner else _lib_codes.ACT_GUIDE
        ensemble.act(states, source, max_action, out=out)
        for m in range(S):
            if not source[m]:
                continue
            c, e = configs[m], cur[m]
            raw_state[m], reward, done, info = _step(envs[m], out[m].copy())
            e["ret"] += reward
            e["ts"] += 1
            e["goal"] = e["goal"] or is_goal_reached(reward, info)
            if done:
                a = acc[m]
                a["successes"].append(float(e["goal"]))
                a["returns"].append(e["ret"])
                probing = (not use_guide) and c.max_init_horizon
                a["horizons"].append(np.max(e["horizons"]) if probing else jsrl.accumulate(e["horizons"]))
                a["agent_types"].append(np.mean(e["types"]))
                ep[m] += 1
                fresh[m] = True
                live[m] = ep[m] < n_ep
    results = []
    for m in range(S):
        if not chosen[m]:
            results.append(None)
            continue
        a, c = acc[m], configs[m]
        horizon = np.max(a["horizons"]) if ((not use_guide) and c.max_init_horizon) else np.mean(a["horizons"])
        results.append((np.asarray(a["returns"]), float(np.mean(a["successes"])), horizon, float(np.mean(a["agent_types"]))))
    return results


def ensemble_train_loop(configs, envs, eval_envs, replay_buffers, state_dim: int, action_dim: int, max_action: float,
                        max_steps: int, log: Optional[Callable[[int, Dict, int], None]] = None, reward_mod_dicts=None,
                        is_env_with_goal: bool = False, scheduler=None, mixed_batch_sizes: bool = False,
                        philox_act_dropout: bool = False):
    """``train_loop`` for S members at once, one ``JsrlTrainConfig`` per member (seed, IQL / Adam hyper-parameters,
    curriculum, tolerance, noise and checkpoint path may differ; ``ENSEMBLE_SHARED_FIELDS`` may not; ``batch_size``
    may differ with ``mixed_batch_sizes=True``, the batch-size axis of a search).

    Offline: one ``IQLEnsemble`` (cosine schedule with T_max = offline_iterations) trained in K-step calls that end at
    the evaluation points, on indices drawn from each member's own ``np.random.RandomState(seed)``.  Switch: a
    guide-only evaluation gives each member's initial horizon, the offline ensemble becomes the guide (``set_guide``,
    its arena read zero-copy) and a fresh learner ensemble starts (no schedule, total_it = offline_iterations, the
    guide's networks copied when there is a single curriculum stage), each member with its own online ring.  Online,
    per env step for all members: the horizon functions on the host, ONE act launch, exploration noise or the
    Gaussian sample from each member's own ``torch.Generator(seed)``, S env steps, ONE ring-insert launch and ONE
    logged update.  ``train_loop``'s quirks are kept per member; a member whose update gate (``t >= batch_size`` with
    a new online buffer) is still closed does not train (``IQLEnsemble.retire``).  ``log(member, dict, step)``
    receives what ``train_loop``'s ``log`` receives.

    ``scheduler`` (e.g. ``asha.ASHAScheduler``): every evaluation of both phases reports each evaluated member's score
    (the value ``horizon_update_callback`` sees) as ``on_result(member, n_reports, score, total_it)``; a member it
    stops gets no act, env step, insert, update, evaluation, log or checkpoint from then on and costs no GPU time.
    Members stopped offline skip the guide probe and start the online phase retired.  The run ends when every member
    has stopped.  Returns (learner ensemble, configs, one eval history per member); the guide ensemble is
    ``learner.guide``.

    ``philox_act_dropout``: runs configs with ``actor_dropout`` > 0 (refused without it).  The learner's env steps act
    in training mode as the reference's do, with dropout after every hidden ReLU, in the batched act kernel
    (IQL_ACT_LEARNER_DIST_DROPOUT / IQL_ACT_LEARNER_DROPOUT): member m's masks come from the engine's Philox stream
    keyed by ``seed | 1 << 63`` at its act counter (``learner.engine.act_steps[m]``, one per learner env step), so they
    are reproducible but are not torch's ``nn.Dropout`` draws.  Guide acts and evaluations run without dropout.
    Checkpoints carry the reference's dropout-policy keys."""
    check_ensemble_configs(configs, scheduler, mixed_batch_sizes, philox_act_dropout)
    S = len(configs)
    if not (len(envs) == len(eval_envs) == S):
        raise ValueError("need one env and one eval env per member")
    if isinstance(replay_buffers, ReplayBuffer):
        replay_buffers = [replay_buffers] * S
    if len(replay_buffers) != S:
        raise ValueError("need one replay buffer or one per member")
    reward_mod_dicts = reward_mod_dicts if reward_mod_dicts is not None else [None] * S
    if not configs[0].new_online_buffer:
        rows = [rb.rows.data_ptr() for rb in replay_buffers]
        if len(set(rows)) != S:
            raise ValueError("new_online_buffer=False: every member needs its own buffer (members must not see each "
                             "other's transitions)")
    log = log or (lambda m, d, step: None)
    c0 = configs[0]
    Bm = [int(c.batch_size) for c in configs]
    off, on, eval_freq = int(c0.offline_iterations), int(c0.online_iterations), int(c0.eval_freq)
    gated = bool(c0.new_online_buffer)  # train_loop's update gate `t >= batch_size` on the global t
    gaussian = not c0.iql_deterministic
    jsrl.horizon_str = c0.horizon_fn
    device = c0.device
    for c in configs:
        c.discrete = False
        if c.checkpoints_path is not None:
            os.makedirs(c.checkpoints_path, exist_ok=True)
    nets = [member_networks(c, state_dim, action_dim, max_action) for c in configs]
    index_rng = [np.random.RandomState(c.seed) for c in configs]
    noise_rng = [torch.Generator().manual_seed(int(c.seed)) for c in configs]
    histories = [[] for _ in range(S)]
    eval_successes = [[] for _ in range(S)]
    states = [_reset(envs[m], configs[m].seed) for m in range(S)]
    live = np.ones(S, dtype=bool)  # not stopped by the scheduler
    reports = [0] * S

    def evaluate(t, ens, use_guide, total_it, members):
        if not use_guide:
            for m in np.flatnonzero(members):
                configs[m].curriculum_stage = np.nan
        results = ensemble_eval_actor(eval_envs, ens, use_guide, configs, max_action, members)
        for m in np.flatnonzero(members):
            c = configs[m]
            scores, success, c.mean_horizon_reached, c.eval_mean_agent_type = results[m]
            score = float(scores.mean())
            norm_fn = getattr(eval_envs[m], "get_normalized_score", None) if c.normalize_reward else None
            if norm_fn is not None:
                score = float(norm_fn(score))
            eval_log = {}
            if is_env_with_goal:
                eval_successes[m].append(success)
                eval_log["eval/regret"] = float(np.mean(1 - np.array(eval_successes[m])))
                eval_log["eval/success_rate"] = success
            if t >= off:
                configs[m] = c = jsrl.horizon_update_callback(c, score)
                eval_log = jsrl.add_jsrl_metrics(eval_log, c)
            if norm_fn is not None:
                eval_log["eval/d4rl_normalized_score"] = score * 100.0
            else:
                eval_log["eval/score"] = score
            if c.checkpoints_path is not None:
                torch.save(ens.member_state_dict(m), os.path.join(c.checkpoints_path, f"checkpoint_{t}.pt"))
            log(m, eval_log, total_it[m])
            histories[m].append(dict(eval_log, t=t))
            if scheduler is not None:
                reports[m] += 1
                if scheduler.on_result(int(m), reports[m], score, int(total_it[m])) == "stop":
                    live[m] = False
        if live.any() and not np.array_equal(ens.active, ens.active & live):
            _sync_active(ens, ens.active & live)  # stopped members are retired at once

    # ---- offline phase: K-step calls between evaluation points and gate openings ----
    offline = _build_ensemble(configs, [n[0] for n in nets], state_dim, action_dim, off, device)
    offline.bind_replay(list(replay_buffers))
    first = np.array([min(b, off) if gated else 0 for b in Bm])  # the first offline step of each member
    done_steps = [0] * S
    t = int(first.min())
    while t < off and live.any():
        stop = min(off, (t // eval_freq + 1) * eval_freq, t + offline.engine.max_steps_per_call)
        opening = first[first > t]
        if opening.size:
            stop = min(stop, int(opening.min()))
        K = stop - t
        train = live & (first <= t)
        if not train.any():  # the members still running have not reached their gates yet
            t = stop
            continue
        _sync_active(offline, train)
        idx = np.zeros((S, K, max(Bm)), dtype=np.int64)
        for m in np.flatnonzero(train):
            high = replay_buffers[m]._high()
            for k in range(K):
                idx[m, k, :Bm[m]] = index_rng[m].randint(0, high, size=Bm[m])
        losses = offline.train_steps(K, mode="indices", indices=torch.from_numpy(idx)).cpu().numpy()
        for k in range(K):
            for m in np.flatnonzero(train):
                done_steps[m] += 1
                log(m, {"value_loss": float(losses[m, k, 0]), "q_loss": float(losses[m, k, 1]),
                        "actor_loss": float(losses[m, k, 2]), "offline_iter": t + k}, done_steps[m])
        t = stop
        if t % eval_freq == 0:
            evaluate(t - 1, offline, False, done_steps, train)
    if on <= 0 or not live.any():
        return offline, configs, histories

    # ---- switch to online: guide-only probe, guide binding, fresh learners, online rings ----
    for m in np.flatnonzero(live):
        configs[m].curriculum_stage = np.nan
    probe = ensemble_eval_actor(envs, offline, False, configs, max_action, live)
    learner = _build_ensemble(configs, [n[1] for n in nets], state_dim, action_dim, 0, device, learner=True)
    for m, c in enumerate(configs):
        if c.n_curriculum_stages == 1:  # the guide's trained networks, fresh optimizers (get_learning_agent)
            learner.engine.load_params(m, offline.engine.param_views(m))
        learner.engine.set_counters(m, total_it=off)
    learner.set_guide(offline)
    for m in np.flatnonzero(live):
        configs[m] = jsrl.prepare_finetuning(probe[m][2], configs[m])
    # stopped members keep the offline buffer bound: they never sample from it
    online_buffers = [jsrl.get_online_buffer(c, replay_buffers[m], state_dim, action_dim) if live[m] else replay_buffers[m]
                      for m, c in enumerate(configs)]
    learner.bind_replay(online_buffers)
    if not live.all():
        _sync_active(learner, live)
    states = [_reset(envs[m]) if live[m] else None for m in range(S)]

    hfn = jsrl.HORIZON_FNS[jsrl.horizon_str]["horizon_fn"]
    A = action_dim
    obs = np.zeros((S, state_dim), dtype=np.float32)
    next_obs = np.zeros((S, state_dim), dtype=np.float32)
    act_out = np.zeros((S, A), dtype=np.float32)
    act_std = np.zeros((S, A), dtype=np.float32) if gaussian else None
    actions = np.zeros((S, A), dtype=np.float32)
    rewards = np.zeros(S, dtype=np.float32)
    real_dones = np.zeros(S, dtype=np.float32)
    source = np.zeros(S, dtype=np.int8)
    if c0.actor_dropout:  # training mode: dropout active in the learner's act (checked: philox_act_dropout)
        learner_code = _lib_codes.ACT_LEARNER_DIST_DROPOUT if gaussian else _lib_codes.ACT_LEARNER_DROPOUT
    else:
        learner_code = _lib_codes.ACT_LEARNER_DIST if gaussian else _lib_codes.ACT_LEARNER
    use = [False] * S
    ep_ret, ep_step, goal = [0.0] * S, [0] * S, [False] * S
    ep_types = [[] for _ in range(S)]
    train_successes = [[] for _ in range(S)]
    total_it = [off] * S
    idx = np.zeros((S, max(Bm)), dtype=np.int64)
    for t in range(off, off + on):
        if not live.any():
            break
        members = np.flatnonzero(live)
        online_logs = [{} for _ in range(S)]
        for m in members:
            c = configs[m]
            if ep_step[m] == 0:
                ep_types[m] = []
                c.ep_agent_type = 0
            else:
                c.ep_agent_type = np.mean(ep_types[m])
            use[m], _ = hfn(ep_step[m], states[m], envs[m], c)
            obs[m] = np.asarray(states[m], dtype=np.float32).reshape(-1)
            source[m] = learner_code if use[m] else _lib_codes.ACT_GUIDE
        source[~live] = _lib_codes.ACT_SKIP
        learner.act(obs, source, max_action, out=act_out, std=act_std)
        for m in members:
            c = configs[m]
            ep_types[m].append(1 if use[m] else 0)
            a = act_out[m].copy()
            if use[m] and gaussian:  # GaussianPolicy.act in training mode: mean + std * N(0, 1), scaled and clipped
                sample = a + act_std[m] * torch.randn(A, generator=noise_rng[m]).numpy()
                a = np.clip(max_action * sample, -max_action, max_action).astype(np.float32)
            elif use[m]:  # deterministic learner: exploration noise
                noise = (torch.randn(A, generator=noise_rng[m]) * c.expl_noise).clamp(-c.noise_clip, c.noise_clip)
                a = a + noise.numpy()
            a = np.clip(max_action * a, -max_action, max_action).astype(np.float32).flatten()
            next_state, reward, done, info = _step(envs[m], a)
            ep_step[m] += 1
            goal[m] = goal[m] or is_goal_reached(reward, info)
            ep_ret[m] += reward
            real_dones[m] = float(bool(done and ep_step[m] < max_steps))  # time-outs are not terminals
            if c.normalize_reward and reward_mod_dicts[m] is not None:
                reward = modify_reward_online(reward, c.env, **reward_mod_dicts[m])
            actions[m] = a
            rewards[m] = reward
            next_obs[m] = np.asarray(next_state, dtype=np.float32).reshape(-1)
            states[m] = next_state
            if done:
                states[m] = _reset(envs[m])
                lg = online_logs[m]
                if is_env_with_goal:
                    train_successes[m].append(goal[m])
                    lg["train/regret"] = float(np.mean(1 - np.array(train_successes[m])))
                    lg["train/is_success"] = float(goal[m])
                lg.update({"train/episode_return": ep_ret[m], "train/mean_ep_agent_type": float(np.mean(ep_types[m])),
                           "train/episode_length": ep_step[m]})
                ep_ret[m], ep_step[m], goal[m] = 0.0, 0, False
        learner.add_transitions(obs, actions, rewards, next_obs, real_dones, mask=live)
        train = live & np.array([t >= b or not gated for b in Bm])
        if not train.any():
            continue
        _sync_active(learner, train)
        for m in np.flatnonzero(train):
            idx[m, :Bm[m]] = index_rng[m].randint(0, online_buffers[m]._high(), size=Bm[m])
        losses = learner.train_step_logged(idx)
        for m in np.flatnonzero(train):
            total_it[m] += 1
            log_dict = {"value_loss": float(losses[m, 0]), "q_loss": float(losses[m, 1]), "actor_loss": float(losses[m, 2]),
                        "online_iter": t - off}
            log_dict.update(online_logs[m])
            log(m, log_dict, total_it[m])
        if (t + 1) % eval_freq == 0:
            evaluate(t, learner, True, total_it, train)
    return learner, configs, histories
