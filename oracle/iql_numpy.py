"""TEST INFRASTRUCTURE ONLY -- CPU restatement (numpy) of the reference IQL update.

This module is the *oracle* of the repo: a plain numpy restatement of the hot
path of LaurenYTaylor/jsrl-CORL, used as the checker by ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs
of ``bench.py``.  Nothing in the product path (``jsrl_corl_b200``) imports it.

Parity status: PINNED against the live reference.  ``oracle/gen_golden.py``
runs the unmodified reference classes (``/root/reference/algorithms/finetune/iql.py``,
imported through ``oracle/ref_loader.py``) and stores their outputs under
``tests/golden/``; ``tests/test_oracle.py`` checks this restatement against
those fixtures (and against the live reference when the tree is present).
The reference itself ships no golden vectors or tests for this path
(SURVEY.md section 4), so the fixtures generated from it are the pin.

Reference lines followed (all relative to /root/reference/algorithms/finetune/iql.py;
the offline variant algorithms/offline/iql.py:255-537 has identical math):
  * asymmetric_l2_loss                      iql.py:301-302
  * MLP layer order / dropout placement      iql.py:314-344
  * GaussianPolicy / DeterministicPolicy     iql.py:347-413  (+ torch Normal.log_prob)
  * TwinQ / ValueFunction                    iql.py:416-442
  * ImplicitQLearning._update_v              iql.py:482-495
  * ImplicitQLearning._update_q + soft_update iql.py:497-515, 72-74
  * ImplicitQLearning._update_policy         iql.py:517-540
  * ImplicitQLearning.train (op order)       iql.py:542-563
  * torch.optim.Adam (defaults) as called at jsrl_utils.py:263-265 / offline/iql.py:595-597
  * CosineAnnealingLR(actor_optimizer, max_steps)  iql.py:470-473 (recursive form)
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

EXP_ADV_MAX = 100.0  # iql.py:26
LOG_STD_MIN = -20.0  # iql.py:27
LOG_STD_MAX = 2.0  # iql.py:28
HALF_LOG_2PI = math.log(math.sqrt(2 * math.pi))  # torch Normal.log_prob constant


@dataclass
class OracleConfig:
    state_dim: int
    action_dim: int
    hidden_dim: int = 256
    n_hidden: int = 2
    deterministic: bool = False
    actor_dropout: float = 0.0
    iql_tau: float = 0.7
    beta: float = 3.0
    discount: float = 0.99
    tau: float = 0.005
    vf_lr: float = 3e-4
    qf_lr: float = 3e-4
    actor_lr: float = 3e-4
    max_steps: Optional[int] = 1000000  # CosineAnnealingLR T_max; None = no schedule
    adam_betas: tuple = (0.9, 0.999)
    adam_eps: float = 1e-8
    lr_eta_min: float = 0.0  # CosineAnnealingLR eta_min


def mlp_layer_names(n_hidden: int, dropout: bool) -> List[int]:
    """Sequential indices of the nn.Linear modules (iql.py:328-341): with
    dropout>0 a Dropout follows every ReLU, shifting the indices to 0,3,6,..."""
    stride = 3 if dropout else 2
    return [stride * i for i in range(n_hidden + 1)]


class _Adam:
    """torch.optim.Adam with default flags (no weight decay / amsgrad), the
    single-tensor formulas: lerp, mul+addcmul, sqrt/bias_correction2_sqrt+eps,
    addcdiv.  Scalars are formed in Python floats (float64) exactly like torch
    does and enter tensor ops as scalars of the tensor dtype."""

    def __init__(self, params: Dict[str, np.ndarray], lr: float, betas, eps: float, dtype):
        self.params = params
        self.lr = lr
        self.beta1, self.beta2 = betas
        self.eps = eps
        self.dtype = dtype
        self.step_count = 0
        self.exp_avg = {k: np.zeros_like(v) for k, v in params.items()}
        self.exp_avg_sq = {k: np.zeros_like(v) for k, v in params.items()}

    def step(self, grads: Dict[str, np.ndarray]):
        dt = self.dtype
        self.step_count += 1
        t = self.step_count
        bc1 = 1 - self.beta1 ** t
        bc2 = 1 - self.beta2 ** t
        step_size = self.lr / bc1
        bc2_sqrt = bc2 ** 0.5
        w1 = dt(1 - self.beta1)
        for k, p in self.params.items():
            g = grads[k].astype(dt, copy=False)
            m = self.exp_avg[k]
            v = self.exp_avg_sq[k]
            if self.beta1 > 0.5:  # lerp_: torch evaluates weights >= 0.5 from the end point (exact g at beta1 = 0)
                m += w1 * (g - m)
            else:
                m[...] = g - (g - m) * (dt(1) - w1)
            v *= dt(self.beta2)
            v += dt(1 - self.beta2) * g * g  # addcmul_
            denom = np.sqrt(v) / dt(bc2_sqrt) + dt(self.eps)
            p += dt(-step_size) * (m / denom)  # addcdiv_


class NumpyIQL:
    """Single-member IQL learner restated in numpy.

    ``params`` uses the checkpoint layout of the reference:
    ``{"qf": {"q1.net.0.weight": ..}, "vf": {"v.net.0.weight": ..},
    "actor": {"log_std": .., "net.net.0.weight": ..}}`` (iql.py:565-579).
    """

    def __init__(self, cfg: OracleConfig, params: Dict[str, Dict[str, np.ndarray]], dtype=np.float32):
        self.cfg = cfg
        self.dtype = np.dtype(dtype).type
        dt = self.dtype
        self.qf = {k: np.array(v, dtype=dt) for k, v in params["qf"].items()}
        self.vf = {k: np.array(v, dtype=dt) for k, v in params["vf"].items()}
        self.actor = {k: np.array(v, dtype=dt) for k, v in params["actor"].items()}
        src_t = params.get("q_target", params["qf"])  # iql.py:464 deep copy
        self.q_target = {k: np.array(v, dtype=dt) for k, v in src_t.items()}
        self.q_opt = _Adam(self.qf, cfg.qf_lr, cfg.adam_betas, cfg.adam_eps, dt)
        self.v_opt = _Adam(self.vf, cfg.vf_lr, cfg.adam_betas, cfg.adam_eps, dt)
        self.a_opt = _Adam(self.actor, cfg.actor_lr, cfg.adam_betas, cfg.adam_eps, dt)
        self.sched_epoch = 0  # CosineAnnealingLR.last_epoch
        self.total_it = 0
        self.q_idx = mlp_layer_names(cfg.n_hidden, False)
        self.a_idx = mlp_layer_names(cfg.n_hidden, cfg.actor_dropout > 0.0)

    # ---- MLP helpers -------------------------------------------------
    def _mlp_forward(self, p, prefix, idx, x, masks=None, keep_scale=None):
        """Returns (output, list of layer inputs H_0..H_L)."""
        hs = [x]
        h = x
        for li, i in enumerate(idx[:-1]):
            z = h @ p[f"{prefix}{i}.weight"].T + p[f"{prefix}{i}.bias"]
            h = np.maximum(z, 0)
            if masks is not None:
                h = h * masks[li].astype(self.dtype) * keep_scale
            hs.append(h)
        i = idx[-1]
        y = h @ p[f"{prefix}{i}.weight"].T + p[f"{prefix}{i}.bias"]
        return y, hs

    def _mlp_backward(self, p, prefix, idx, hs, gy, keep_scale=None):
        """gy = dL/d(output of last Linear). Returns dict of grads."""
        grads = {}
        g = gy
        for li in range(len(idx) - 1, -1, -1):
            i = idx[li]
            grads[f"{prefix}{i}.weight"] = g.T @ hs[li]
            grads[f"{prefix}{i}.bias"] = g.sum(0)
            if li > 0:
                gh = g @ p[f"{prefix}{i}.weight"]
                on = (hs[li] > 0).astype(self.dtype)
                if keep_scale is not None:
                    on = on * keep_scale
                g = gh * on
        return grads

    # ---- the step (iql.py:542-563) ------------------------------------
    def train(self, batch, dropout_masks=None) -> Dict[str, float]:
        cfg, dt = self.cfg, self.dtype
        obs, act, rew, nobs, done = [np.asarray(b, dtype=dt) for b in batch]
        B = obs.shape[0]
        self.total_it += 1
        rew = rew.reshape(B)
        done = done.reshape(B)
        sa = np.concatenate([obs, act], 1)  # iql.py:428

        # A. next_v with the old V (iql.py:552-553)
        next_v, _ = self._mlp_forward(self.vf, "v.net.", self.q_idx, nobs)
        next_v = next_v[:, 0]

        # B. V update (iql.py:482-495)
        tq1, _ = self._mlp_forward(self.q_target, "q1.net.", self.q_idx, sa)
        tq2, _ = self._mlp_forward(self.q_target, "q2.net.", self.q_idx, sa)
        target_q = np.minimum(tq1[:, 0], tq2[:, 0])
        v, v_hs = self._mlp_forward(self.vf, "v.net.", self.q_idx, obs)
        v = v[:, 0]
        adv = target_q - v
        w = np.abs(dt(cfg.iql_tau) - (adv < 0).astype(dt))  # iql.py:302
        v_loss = np.mean(w * adv * adv)
        g_v = -(w * dt(1.0 / B)) * (dt(2) * adv)
        v_grads = self._mlp_backward(self.vf, "v.net.", self.q_idx, v_hs, g_v[:, None])

        # C. Q forward uses the pre-update Q (iql.py:506-508)
        targets = rew + (dt(1.0) - done) * dt(cfg.discount) * next_v
        q1, q1_hs = self._mlp_forward(self.qf, "q1.net.", self.q_idx, sa)
        q2, q2_hs = self._mlp_forward(self.qf, "q2.net.", self.q_idx, sa)
        q1, q2 = q1[:, 0], q2[:, 0]
        q_loss = (np.mean((q1 - targets) ** 2) + np.mean((q2 - targets) ** 2)) / dt(2)
        g_q1 = (q1 - targets) * dt(2.0 / B) * dt(0.5)
        g_q2 = (q2 - targets) * dt(2.0 / B) * dt(0.5)
        q_grads = {}
        q_grads.update(self._mlp_backward(self.qf, "q1.net.", self.q_idx, q1_hs, g_q1[:, None]))
        q_grads.update(self._mlp_backward(self.qf, "q2.net.", self.q_idx, q2_hs, g_q2[:, None]))

        # D. policy forward uses the pre-update actor and the old adv (iql.py:517-534)
        with np.errstate(over="ignore"):
            exp_adv = np.minimum(np.exp(dt(cfg.beta) * adv), dt(EXP_ADV_MAX))
        p = cfg.actor_dropout
        keep_scale = dt(1.0 / (1.0 - p)) if p > 0.0 else None
        if p > 0.0 and dropout_masks is None:
            raise ValueError("actor_dropout > 0 needs injected dropout masks for parity")
        z, a_hs = self._mlp_forward(self.actor, "net.net.", self.a_idx, obs,
                                    masks=dropout_masks if p > 0.0 else None, keep_scale=keep_scale)
        mu = np.tanh(z)
        a_grads = {}
        if not cfg.deterministic:
            ls = np.clip(self.actor["log_std"], dt(LOG_STD_MIN), dt(LOG_STD_MAX))
            std = np.exp(ls)
            var = std * std
            log_scale = np.log(std)
            diff = act - mu
            logp = -(diff * diff) / (dt(2) * var) - log_scale - dt(HALF_LOG_2PI)
            bc = -logp.sum(-1)
            # d bc / d mu = -(a-mu)/var ; d bc / d log_std = 1 - (a-mu)^2/var (inside the clamp)
            e_over_b = exp_adv * dt(1.0 / B)
            g_mu = -(e_over_b[:, None]) * diff / var
            in_range = ((self.actor["log_std"] >= dt(LOG_STD_MIN)) & (self.actor["log_std"] <= dt(LOG_STD_MAX))).astype(dt)
            a_grads["log_std"] = in_range * (e_over_b[:, None] * (dt(1) - diff * diff / var)).sum(0)
        else:
            if mu.shape != act.shape:
                raise RuntimeError("Actions shape missmatch")  # iql.py:530
            diff = mu - act
            bc = (diff * diff).sum(1)
            g_mu = (exp_adv * dt(1.0 / B))[:, None] * (dt(2) * diff)
        actor_loss = np.mean(exp_adv * bc)
        g_z = g_mu * (dt(1) - mu * mu)
        a_grads.update(self._mlp_backward(self.actor, "net.net.", self.a_idx, a_hs, g_z, keep_scale=keep_scale))

        # optimiser steps, in the reference's order: V, Q (+Polyak with the NEW Q), actor
        self.v_opt.step(v_grads)
        self.q_opt.step(q_grads)
        tau = cfg.tau
        for k in self.q_target:  # soft_update iql.py:72-74: (1-tau)*t + tau*s
            self.q_target[k] = dt(1 - tau) * self.q_target[k] + dt(tau) * self.qf[k]
        self.a_opt.step(a_grads)
        if cfg.max_steps is not None:  # CosineAnnealingLR.step(), recursive form
            self.sched_epoch += 1
            self.a_opt.lr = cosine_recursive_lr(self.a_opt.lr, cfg.actor_lr, self.sched_epoch, cfg.max_steps, cfg.lr_eta_min)
        return {"value_loss": float(v_loss), "q_loss": float(q_loss), "actor_loss": float(actor_loss)}

    def state(self) -> Dict[str, Dict[str, np.ndarray]]:
        return {"qf": self.qf, "vf": self.vf, "actor": self.actor, "q_target": self.q_target}


def cosine_recursive_lr(prev_lr: float, base_lr: float, last_epoch: int, t_max: int, eta_min: float = 0.0) -> float:
    """torch.optim.lr_scheduler.CosineAnnealingLR.get_lr (chainable / recursive form)."""
    if last_epoch == 0:
        return base_lr
    if (last_epoch - 1 - t_max) % (2 * t_max) == 0:
        return prev_lr + (base_lr - eta_min) * (1 - math.cos(math.pi / t_max)) / 2
    return (1 + math.cos(math.pi * last_epoch / t_max)) / (1 + math.cos(math.pi * (last_epoch - 1) / t_max)) * (
        prev_lr - eta_min
    ) + eta_min


def cosine_closed_form_lr(base_lr: float, last_epoch: int, t_max: int, eta_min: float = 0.0) -> float:
    return eta_min + (base_lr - eta_min) * (1 + math.cos(math.pi * last_epoch / t_max)) / 2


# ---------------------------------------------------------------------------
# synthetic data of the BASELINE.json shapes (BASELINE.md section 3)
# ---------------------------------------------------------------------------
def synthetic_dataset(n: int, state_dim: int, action_dim: int, seed: int = 0, antmaze_rewards: bool = False):
    rng = np.random.RandomState(seed)
    obs = rng.standard_normal((n, state_dim)).astype(np.float32)
    nobs = rng.standard_normal((n, state_dim)).astype(np.float32)
    act = rng.uniform(-1.0, 1.0, (n, action_dim)).astype(np.float32)
    if antmaze_rewards:
        rew = -(rng.uniform(size=n) < 0.98).astype(np.float32)  # in {-1, 0}
    else:
        rew = rng.standard_normal(n).astype(np.float32)
    term = (rng.uniform(size=n) < 1e-3)
    return {
        "observations": obs,
        "actions": act,
        "rewards": rew,
        "next_observations": nobs,
        "terminals": term,
    }
