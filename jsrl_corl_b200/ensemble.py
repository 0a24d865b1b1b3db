"""S independent IQL learners (seeds / hyper-parameter configs) trained by one
engine on one GPU -- the B200 replacement for the reference's process-per-seed
Ray launchers (algorithms/finetune/ray_trainer.py:8-31, ray_hyperparam.py:35-50).

Every member has the reference's semantics exactly (``S=1, K=1`` reproduces
``ReplayBuffer.sample`` + ``ImplicitQLearning.train`` call for call); members
never exchange data, so an ensemble shards across GPUs by plain range
partition (``shard_members``) with no collective on the update path.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .engine import EnsembleEngine
from .iql import (DeterministicPolicy, GaussianPolicy, ReplayBuffer, TwinQ, ValueFunction)


def shard_members(n_members: int, world_size: int, rank: int) -> range:
    """Contiguous block partition of ensemble members over ranks (SURVEY.md 8e)."""
    base, rem = divmod(n_members, world_size)
    lo = rank * base + min(rank, rem)
    return range(lo, lo + base + (1 if rank < rem else 0))


def reference_init(seed: int, state_dim: int, action_dim: int, hidden_dim: int, n_hidden: int, deterministic: bool,
                   actor_dropout: float = 0.0, max_action: float = 1.0, offline_variant: bool = False):
    """Initial weights of one member, drawn exactly like the reference scripts:
    ``torch.manual_seed(seed)`` then TwinQ, ValueFunction, policy in that order
    (jsrl_utils.py:252-262, offline/iql.py:584-594).  Returns CPU modules."""
    torch.manual_seed(seed)
    q = TwinQ(state_dim, action_dim, hidden_dim, n_hidden)
    v = ValueFunction(state_dim, hidden_dim, n_hidden)
    cls = DeterministicPolicy if deterministic else GaussianPolicy
    actor = cls(state_dim, action_dim, max_action, hidden_dim, n_hidden, dropout=actor_dropout,
                dropout_when_not_none=offline_variant)
    return q, v, actor


class IQLEnsemble:
    def __init__(self, n_members: int, state_dim: int, action_dim: int, hidden_dim: int = 256, n_hidden: int = 2,
                 batch_size: int = 256, deterministic: bool = False, actor_dropout: float = 0.0,
                 math_mode: str = "tf32", device="cuda", max_steps_per_call: int = 256,
                 seeds: Optional[Sequence[int]] = None, hparams: Optional[Sequence[Dict[str, Any]]] = None,
                 init: bool = True, step_path: str = "auto", batch_sizes: Optional[Sequence[int]] = None):
        """``batch_size`` is the engine's batch B: it sizes the workspace and picks the kernels.  ``batch_sizes``: one
        batch size per member, each in [1, B] (default: all B); member m then trains on B_m rows of every batch, as if
        it were an ensemble of batch B_m, while the kernels still run B rows (see ``EnsembleEngine.set_batch_sizes``)."""
        if batch_sizes is not None:
            batch_sizes = [int(b) for b in batch_sizes]
            if len(batch_sizes) != n_members:
                raise ValueError(f"batch_sizes needs one entry per member ({n_members}), got {len(batch_sizes)}")
            bad = [b for b in batch_sizes if not 1 <= b <= batch_size]
            if bad:
                raise ValueError(f"batch_sizes must lie in [1, batch_size={batch_size}], got {bad}")
        self.engine = EnsembleEngine(n_members, state_dim, action_dim, hidden_dim, n_hidden, batch_size,
                                     deterministic, math_mode, device, max_steps_per_call, step_path=step_path)
        if batch_sizes is not None:
            self.engine.set_batch_sizes(batch_sizes)
        self.n_members = n_members
        self.actor_dropout = actor_dropout
        self.guide: Optional["IQLEnsemble"] = None  # set_guide
        self.seeds = list(seeds) if seeds is not None else list(range(n_members))
        if len(self.seeds) != n_members:
            raise ValueError("need one seed per member")
        for m in range(n_members):
            kw = dict(seed=self.seeds[m], actor_dropout=actor_dropout)
            if hparams is not None:
                kw.update(hparams[m])
            self.engine.set_hparams(m, **kw)
        if init:
            for m in range(n_members):
                self.init_member(m, self.seeds[m])

    @property
    def device(self):
        return self.engine.device

    def init_member(self, m: int, seed: int):
        e = self.engine
        q, v, actor = reference_init(seed, e.state_dim, e.action_dim, e.hidden_dim, e.n_hidden, e.deterministic,
                                     self.actor_dropout)
        state = {"qf": q.state_dict(), "vf": v.state_dict(), "actor": actor.state_dict()}
        e.load_params(m, state, dropout_keys=self.actor_dropout > 0.0)

    def bind_replay(self, buffers):
        """One ReplayBuffer shared by all members, or one per member."""
        if isinstance(buffers, ReplayBuffer):
            buffers = [buffers] * self.n_members
        if len(buffers) != self.n_members:
            raise ValueError("need one buffer or one per member")
        self._buffers = list(buffers)
        for m, rb in enumerate(buffers):
            self.engine.bind_replay(m, rb.rows, rb._high())

    def refresh_replay_sizes(self):
        for m, rb in enumerate(self._buffers):
            self.engine.set_replay_size(m, rb._high())

    def train_steps(self, k_steps: int, **kw) -> torch.Tensor:
        """K fused sample+update steps for every member; losses [S, K, 3] on device."""
        return self.engine.train_steps(k_steps, **kw)

    def train_step_logged(self, indices: Optional[np.ndarray] = None) -> np.ndarray:
        """ONE update step of every member with the losses on the host when it returns ([S, 3] float32:
        value_loss, q_loss, actor_loss) -- the ensemble form of the reference's `log_dict = trainer.train(batch)`
        (offline/iql.py:631-635), for loops that log or branch on the losses every step.  ``indices``: [S, B] int64 rows of
        the bound buffers (member m's first B_m drawn here with numpy, like `ReplayBuffer.sample(B_m)`, when omitted;
        entries past B_m are ignored).  Runs through `iql_train_host_step`: one graph launch, the call returns while the
        backward of the step is still running."""
        e = self.engine
        if indices is None:
            indices = np.zeros((e.n_members, e.batch_size), dtype=np.int64)
            for m in np.flatnonzero(e.active):  # inactive members draw nothing; their losses come back NaN
                indices[m, :e._batch_sizes[m]] = np.random.randint(0, self._buffers[m]._high(), size=e._batch_sizes[m])
        idx = np.ascontiguousarray(indices, dtype=np.int64)
        if idx.shape != (e.n_members, e.batch_size):
            raise ValueError(f"indices must be [{e.n_members}, {e.batch_size}]")
        return np.asarray(e.host_step(host_indices=idx.ctypes.data), dtype=np.float32).reshape(e.n_members, 3)

    # ---- early stopping: members that no longer train ----------------------
    @property
    def active(self) -> np.ndarray:
        """[n_members] bool: the members that train in ``train_steps`` / ``train_step_logged``."""
        return self.engine.active

    def retire(self, members):
        """Stop training ``members`` (a stopped trial of a search): they cost no GPU time in later steps, keep their
        state bit for bit, still act, insert and checkpoint, and read NaN losses.  At least one member must stay."""
        self.engine.set_active(np.flatnonzero(self.active & ~_member_mask(members, self.n_members)))

    def resume(self, members):
        """Train ``members`` again from where they stopped (their counters, schedules and Philox streams continue)."""
        self.engine.set_active(np.flatnonzero(self.active | _member_mask(members, self.n_members)))

    # ---- the online phase: guide, batched act, batched ring insert ------------
    def set_guide(self, other: Optional["IQLEnsemble"]):
        """Make ``other``'s members the guides of this ensemble's members (JSRL's guide policy, jsrl_utils.py:285-323):
        member m's guide is ``other``'s member m, read zero-copy from its parameter arena.  Shapes, policy type and
        parameter layout must be identical.  Keeps a reference to ``other``; None unbinds."""
        if other is None:
            self.engine.bind_guide(None)
            self.guide = None
            return
        a, b = self.engine, other.engine
        shape = lambda e: (e.n_members, e.state_dim, e.action_dim, e.hidden_dim, e.n_hidden, e.deterministic)  # noqa: E731
        if shape(a) != shape(b):
            raise ValueError(f"guide ensemble shape {shape(b)} differs from this ensemble's {shape(a)} "
                             "(members, state_dim, action_dim, hidden_dim, n_hidden, deterministic)")
        lay = lambda e: (e.layout.param_floats, [(t.net, t.layer, t.kind, t.rows, t.cols, t.ld, t.offset) for t in e.tensors])  # noqa: E731
        if lay(a) != lay(b):
            raise ValueError("guide ensemble has a different parameter layout")
        if b.device != a.device:
            raise ValueError("guide ensemble lives on another device")
        a.bind_guide(b.params)
        self.guide = other

    def act(self, states: np.ndarray, source, max_action: float = 1.0, out: Optional[np.ndarray] = None,
            std: Optional[np.ndarray] = None):
        """Every member's action for one env step in one launch: ``source[m]`` is "skip", "learner" (eval-mode
        action), "learner_dist" (Gaussian mean and std, sampled by the caller) or "guide" (eval-mode action of the
        guide set with ``set_guide``), or the matching IQL_ACT_* code.  Returns ``(out, std)`` as
        ``EnsembleEngine.act_members_host``."""
        return self.engine.act_members_host(states, source, max_action, out, std)

    def add_transitions(self, states, actions, rewards, next_states, dones, mask=None):
        """``ReplayBuffer.add_transition`` (iql.py:180-196) for every member whose ``mask`` entry is true (all when
        None), into the member's own bound buffer, in one launch.  Advances each buffer's ``_pointer`` / ``_size`` as
        ``add_transition`` does and raises its IndexError for a buffer loaded to the brim -- before anything is
        written.  Members sharing one buffer cannot insert in the same call."""
        S = self.n_members
        bufs = getattr(self, "_buffers", None)
        if bufs is None:
            raise RuntimeError("add_transitions: no replay buffers bound (bind_replay)")
        mask = np.ones(S, dtype=bool) if mask is None else np.asarray(mask, dtype=bool).reshape(S)
        pointers = np.full(S, -1, dtype=np.int64)
        for m in np.flatnonzero(mask):
            rb = bufs[m]
            if not 0 <= rb._pointer < rb._buffer_size:
                raise IndexError(f"index {rb._pointer} is out of bounds for dimension 0 with size {rb._buffer_size}")
            pointers[m] = rb._pointer
        self.engine.insert_members_host(states, actions, rewards, next_states, dones, pointers)
        for m in np.flatnonzero(mask):
            rb = bufs[m]
            rb._pointer = (rb._pointer + 1) % rb._buffer_size
            rb._size = min(rb._size + 1, rb._buffer_size)

    # ---- checkpoints in the reference layout --------------------------------
    def member_state_dict(self, m: int) -> Dict[str, Any]:
        """Checkpoint of member ``m`` with the keys and tensor layout of
        ``ImplicitQLearning.state_dict()`` (reference iql.py:565-579), loadable
        by the reference class (optimizer dicts are stock Adam state dicts)."""
        e = self.engine
        drop = self.actor_dropout > 0.0
        params = e.param_views(m, drop)
        m1, m2 = e.moment_views(m, drop)
        c = e.get_counters(m)
        hp = e.get_hparams(m)
        t_max = int(hp.cosine_t_max)
        actor_lr_now = cosine_lr(hp.actor_lr, c.sched_epoch, t_max, hp.lr_eta_min) if t_max > 0 else hp.actor_lr

        def opt_state(grp, lr, step, initial_lr=None):
            names = list(params[grp].keys())
            state = {}
            if step > 0:
                for i, n in enumerate(names):
                    state[i] = {"step": torch.tensor(float(step)), "exp_avg": m1[grp][n].clone(),
                                "exp_avg_sq": m2[grp][n].clone()}
            group = {"lr": lr, "betas": (hp.adam_beta1, hp.adam_beta2), "eps": hp.adam_eps, "weight_decay": 0,
                     "amsgrad": False, "maximize": False, "foreach": None, "capturable": False,
                     "differentiable": False, "fused": None, "decoupled_weight_decay": False,
                     "params": list(range(len(names)))}
            if initial_lr is not None:
                group["initial_lr"] = initial_lr
            return {"state": state, "param_groups": [group]}

        sched = {}
        if t_max > 0:
            sched = {"T_max": t_max, "eta_min": hp.lr_eta_min, "base_lrs": [hp.actor_lr],
                     "last_epoch": int(c.sched_epoch), "_step_count": int(c.sched_epoch) + 1,
                     "_is_initial": False, "_get_lr_called_within_step": False, "_last_lr": [actor_lr_now]}
        return {
            "qf": {k: v.clone() for k, v in params["qf"].items()},
            "q_optimizer": opt_state("qf", hp.qf_lr, c.q_step),
            "vf": {k: v.clone() for k, v in params["vf"].items()},
            "v_optimizer": opt_state("vf", hp.vf_lr, c.v_step),
            "actor": {k: v.clone() for k, v in params["actor"].items()},
            "actor_optimizer": opt_state("actor", actor_lr_now, c.actor_step, hp.actor_lr if t_max > 0 else None),
            "actor_lr_schedule": sched,
            "total_it": int(c.total_it),
        }

    def load_member_state_dict(self, m: int, sd: Dict[str, Any]):
        """Inverse of ``member_state_dict``; also accepts checkpoints written by
        the reference.  As in the reference (iql.py:584) the target network is
        re-cloned from qf.  The Adam betas and eps come from the optimizer groups,
        which the engine requires to agree (one set per member)."""
        groups = [sd[key]["param_groups"][0] for key in ("q_optimizer", "v_optimizer", "actor_optimizer")]
        if any(tuple(g["betas"]) != tuple(groups[0]["betas"]) or g["eps"] != groups[0]["eps"] for g in groups[1:]):
            raise NotImplementedError("the three Adam optimizers must share betas and eps")
        e = self.engine
        drop = self.actor_dropout > 0.0
        e.load_params(m, {"qf": sd["qf"], "vf": sd["vf"], "actor": sd["actor"]}, dropout_keys=drop, sync_target=True)
        params = e.param_views(m, drop)
        m1, m2 = e.moment_views(m, drop)
        steps = {}
        for grp, key in (("qf", "q_optimizer"), ("vf", "v_optimizer"), ("actor", "actor_optimizer")):
            st = sd[key]["state"]
            step = 0
            for i, n in enumerate(params[grp].keys()):
                if i in st:
                    m1[grp][n].copy_(st[i]["exp_avg"].to(m1[grp][n]))
                    m2[grp][n].copy_(st[i]["exp_avg_sq"].to(m2[grp][n]))
                    step = int(float(st[i]["step"]))
                else:
                    m1[grp][n].zero_()
                    m2[grp][n].zero_()
            steps[grp] = step
        sched = sd.get("actor_lr_schedule") or {}
        kw = dict(qf_lr=groups[0]["lr"], vf_lr=groups[1]["lr"], adam_beta1=float(groups[0]["betas"][0]),
                  adam_beta2=float(groups[0]["betas"][1]), adam_eps=float(groups[0]["eps"]))
        if sched:
            kw.update(actor_lr=sched["base_lrs"][0], cosine_t_max=int(sched["T_max"]), lr_eta_min=float(sched["eta_min"]))
        else:
            kw.update(actor_lr=sd["actor_optimizer"]["param_groups"][0]["lr"], cosine_t_max=0)
        e.set_hparams(m, **kw)
        e.set_counters(m, q_step=steps["qf"], v_step=steps["vf"], actor_step=steps["actor"],
                       sched_epoch=int(sched.get("last_epoch", 0)), total_it=int(sd["total_it"]))


def _member_mask(members, n: int) -> np.ndarray:
    ids = np.asarray(list(members), dtype=np.int64).reshape(-1)
    if ids.size and (ids.min() < 0 or ids.max() >= n):
        raise ValueError(f"member index out of range [0, {n}): {ids.tolist()}")
    mask = np.zeros(n, dtype=bool)
    mask[ids] = True
    return mask


def cosine_lr(base_lr: float, epoch: int, t_max: int, eta_min: float = 0.0) -> float:
    """Closed form of CosineAnnealingLR (the engine evaluates the same formula in fp64)."""
    import math
    return eta_min + (base_lr - eta_min) * (1.0 + math.cos(math.pi * epoch / t_max)) / 2.0
