"""Drop-in surface of ``algorithms/finetune/iql.py`` (and ``offline/iql.py``) of
LaurenYTaylor/jsrl-CORL, backed by the B200 engine.

Same names, signatures, checkpoint layout and exception types as the reference
(SURVEY.md section 8b): ``TrainConfig``, ``ReplayBuffer``, ``MLP``, ``TwinQ``,
``ValueFunction``, ``GaussianPolicy``, ``DeterministicPolicy``,
``ImplicitQLearning`` and the small helpers around them.  The network classes
are ordinary ``nn.Module`` containers: they define the parameter names/shapes
(= the checkpoint contract) and serve ``actor.act`` in stock torch; once handed
to ``ImplicitQLearning`` their parameters alias the engine's flat arena and
every update runs in ``libiql_b200.so``.  There is no CPU / eager fallback for
the update or for replay sampling.
"""
from __future__ import annotations

import copy
import math
import weakref
import os
import random
import uuid
from dataclasses import dataclass
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple, Union

import ctypes as C
import numpy as np
import torch
import torch.nn as nn
from torch.distributions import Normal
from torch.optim.lr_scheduler import CosineAnnealingLR

from . import _lib
from .engine import EnsembleEngine, linear_indices

TensorBatch = List[torch.Tensor]

# constants of the reference module (iql.py:26-29)
EXP_ADV_MAX = 100.0
LOG_STD_MIN = -20.0
LOG_STD_MAX = 2.0
ENVS_WITH_GOAL = ("antmaze", "pen", "door", "hammer", "relocate", "Adroit")


# ---------------------------------------------------------------------------
# configuration (field names/defaults = reference iql.py:32-69; pyrallis-compatible)
# ---------------------------------------------------------------------------
@dataclass
class TrainConfig:
    # experiment
    device: str = "cuda"
    env: str = "antmaze-umaze-v2"
    seed: int = 0
    eval_seed: int = 0
    eval_freq: int = int(5e4)
    n_episodes: int = 100
    offline_iterations: int = int(1e6)
    online_iterations: int = int(1e6)
    checkpoints_path: Optional[str] = None
    load_model: str = ""
    # IQL
    actor_dropout: float = 0.0
    buffer_size: int = 2_000_000
    batch_size: int = 256
    discount: float = 0.99
    tau: float = 0.005
    beta: float = 3.0
    iql_tau: float = 0.7
    expl_noise: float = 0.03
    noise_clip: float = 0.5
    iql_deterministic: bool = False
    normalize: bool = True
    normalize_reward: bool = False
    vf_lr: float = 3e-4
    qf_lr: float = 3e-4
    actor_lr: float = 3e-4
    # wandb
    project: str = "jsrl-CORL-adroit"
    group: str = "IQL-D4RL"
    name: str = "IQL"

    def __post_init__(self):
        # the reference decorates the run name and nests the checkpoint dir under it
        self.name = "-".join([self.name, self.env, str(uuid.uuid4())[:8]])
        if self.checkpoints_path is not None:
            self.checkpoints_path = os.path.join(self.checkpoints_path, self.name)


@dataclass
class OfflineTrainConfig:
    """Field set of ``algorithms/offline/iql.py:30-85`` (max_timesteps instead
    of offline/online iterations, Optional actor_dropout, different eval cadence)."""
    project: str = "jsrl-CORL"
    group: str = "IQL-D4RL"
    name: str = "IQL"
    env: str = "halfcheetah-medium-expert-v2"
    discount: float = 0.99
    tau: float = 0.005
    beta: float = 3.0
    iql_tau: float = 0.7
    iql_deterministic: bool = False
    max_timesteps: int = int(1e6)
    buffer_size: int = 2_000_000
    batch_size: int = 256
    normalize: bool = True
    normalize_reward: bool = False
    vf_lr: float = 3e-4
    qf_lr: float = 3e-4
    actor_lr: float = 3e-4
    actor_dropout: Optional[float] = None
    eval_freq: int = int(5e3)
    n_episodes: int = 10
    checkpoints_path: Optional[str] = None
    load_model: str = ""
    seed: int = 0
    device: str = "cuda"

    def __post_init__(self):
        self.name = "-".join([self.name, self.env, str(uuid.uuid4())[:8]])
        if self.checkpoints_path is not None:
            self.checkpoints_path = os.path.join(self.checkpoints_path, self.name)


# ---------------------------------------------------------------------------
# small helpers with reference semantics
# ---------------------------------------------------------------------------
def soft_update(target: nn.Module, source: nn.Module, tau: float):
    """Polyak step on module parameters (iql.py:72-74).  Inside ``train`` the
    engine fuses this into the Adam kernel; this torch version exists for
    callers that use it directly."""
    with torch.no_grad():
        for t, s in zip(target.parameters(), source.parameters()):
            t.copy_((1 - tau) * t + tau * s)


def compute_mean_std(states: np.ndarray, eps: float) -> Tuple[np.ndarray, np.ndarray]:
    return states.mean(0), states.std(0) + eps


def normalize_states(states: np.ndarray, mean: np.ndarray, std: np.ndarray):
    return (states - mean) / std


def asymmetric_l2_loss(u: torch.Tensor, tau: float) -> torch.Tensor:
    weight = torch.abs(tau - (u < 0).float())
    return (weight * u.pow(2)).mean()


def set_seed(seed: int, env=None, deterministic_torch: bool = False):
    if env is not None:
        env.seed(seed)
        env.action_space.seed(seed)
    os.environ["PYTHONHASHSEED"] = str(seed)
    np.random.seed(seed)
    random.seed(seed)
    torch.manual_seed(seed)
    torch.use_deterministic_algorithms(deterministic_torch)


def return_reward_range(dataset: Dict, max_episode_steps: int) -> Tuple[float, float]:
    returns, lengths = [], []
    acc, n = 0.0, 0
    for r, d in zip(dataset["rewards"], dataset["terminals"]):
        acc += float(r)
        n += 1
        if d or n == max_episode_steps:
            returns.append(acc)
            lengths.append(n)
            acc, n = 0.0, 0
    lengths.append(n)
    assert sum(lengths) == len(dataset["rewards"])
    return min(returns), max(returns)


def modify_reward(dataset: Dict, env_name: str, max_episode_steps: int = 1000) -> Dict:
    if any(s in env_name for s in ("halfcheetah", "hopper", "walker2d")):
        lo, hi = return_reward_range(dataset, max_episode_steps)
        dataset["rewards"] /= hi - lo
        dataset["rewards"] *= max_episode_steps
        return {"max_ret": hi, "min_ret": lo, "max_episode_steps": max_episode_steps}
    if "antmaze" in env_name:
        dataset["rewards"] -= 1.0
    return {}


def modify_reward_online(reward: float, env_name: str, **kwargs) -> float:
    if any(s in env_name for s in ("halfcheetah", "hopper", "walker2d")):
        reward /= kwargs["max_ret"] - kwargs["min_ret"]
        reward *= kwargs["max_episode_steps"]
    elif "antmaze" in env_name:
        reward -= 1.0
    return reward


def is_goal_reached(reward: float, info: Dict) -> bool:
    if "goal_achieved" in info:
        return info["goal_achieved"]
    if "success" in info:
        return info["success"]
    return reward > 0


# ---------------------------------------------------------------------------
# replay buffer (iql.py:122-196) on packed device rows
# ---------------------------------------------------------------------------
_N_SLOTS = 8
# id(observations tensor) -> slot, for the cached output tensors of every live buffer: `ImplicitQLearning.train(batch)`
# recognises a batch that came straight out of `ReplayBuffer.sample` (same tensor objects, untouched since) and lets the
# engine gather the rows itself from the host-drawn indices instead of re-packing the five dense tensors
_SAMPLED: "weakref.WeakValueDictionary[int, _SampleSlot]" = weakref.WeakValueDictionary()


class _SampleSlot:
    """One set of output tensors of ``ReplayBuffer.sample`` + the host indices that filled it."""
    __slots__ = ("rb", "B", "out", "ptrs", "ver", "idx_host", "high", "__weakref__")

    def __init__(self, rb: "ReplayBuffer", B: int):
        S, A = rb._state_dim, rb._action_dim
        # one allocation carved into the five dense outputs
        flat = torch.empty(B * (2 * S + A + 2), dtype=torch.float32, device=rb._device)
        s, a, r, s2, d = flat.split((B * S, B * A, B, B * S, B))
        self.rb, self.B = weakref.ref(rb), B
        self.out = [s.view(B, S), a.view(B, A), r.view(B, 1), s2.view(B, S), d.view(B, 1)]
        self.ptrs = tuple(t.data_ptr() for t in self.out)
        self.ver = None
        self.idx_host = None
        self.high = 0

    def untouched(self, batch) -> bool:
        """`batch` is exactly this slot's tensors and nobody has written to them in place since the gather."""
        o, v = self.out, self.ver
        return (batch[0] is o[0] and batch[1] is o[1] and batch[2] is o[2] and batch[3] is o[3] and batch[4] is o[4]
                and v is not None and o[0]._version == v[0] and o[1]._version == v[1] and o[2]._version == v[2]
                and o[3]._version == v[3] and o[4]._version == v[4])


class ReplayBuffer:
    """Same API as the reference buffer; storage is ONE device tensor of packed
    transition rows ``[buffer_size, row_floats]`` (include/iql_b200.h
    ``iql_row_layout``).  ``_states/_actions/_rewards/_next_states/_dones`` are
    strided views into it with the reference's shapes.

    ``sampler="numpy"`` (default) draws indices exactly like the reference
    (``np.random.randint`` on the global MT19937 stream, iql.py:172) and gathers
    them with the CUDA kernel; ``sampler="philox"`` draws them in-kernel.
    ``offline_semantics=True`` reproduces ``offline/iql.py:173``
    (``high=min(_size, _pointer)``)."""

    def __init__(self, state_dim: int, action_dim: int, buffer_size: int, device: str = "cpu",
                 sampler: str = "numpy", seed: int = 0, offline_semantics: bool = False, fresh_outputs: bool = False):
        self._device = _lib.require_cuda(device)
        self._L = _lib.lib()
        if sampler not in ("numpy", "philox"):
            raise ValueError("sampler must be 'numpy' or 'philox'")
        self._buffer_size = int(buffer_size)
        self._pointer = 0
        self._size = 0
        self._state_dim, self._action_dim = state_dim, action_dim
        self._sampler, self._seed, self._sample_calls = sampler, int(seed), 0
        self._offline_semantics = offline_semantics
        self._lay = _lib.RowLayout()
        _lib.check(self._L.iql_replay_row_layout(state_dim, action_dim, C.byref(self._lay)))
        lay = self._lay
        self._rows = torch.zeros((self._buffer_size, lay.row_floats), dtype=torch.float32, device=self._device)
        self._states = self._rows[:, lay.off_state:lay.off_state + state_dim]
        self._actions = self._rows[:, lay.off_action:lay.off_action + action_dim]
        self._rewards = self._rows[:, lay.off_reward:lay.off_reward + 1]
        self._next_states = self._rows[:, lay.off_next_state:lay.off_next_state + state_dim]
        self._dones = self._rows[:, lay.off_done:lay.off_done + 1]
        # add_transition: two pinned staging rows used alternately, each guarded by an event recorded after its
        # host->device copy, so an insert never waits for the whole stream (only, rarely, for its own slot)
        self._stage = [torch.zeros(lay.row_floats, dtype=torch.float32, device=self._device) for _ in range(2)]
        self._stage_host = [torch.zeros(lay.row_floats, dtype=torch.float32).pin_memory() for _ in range(2)]
        self._stage_ev = [None, None]
        self._stage_i = 0
        # sample: ring of cached output tensor sets; `fresh_outputs=True` allocates new tensors every call instead
        self._fresh_outputs = bool(fresh_outputs)
        self._slots: List["_SampleSlot"] = []
        self._slot_i = 0
        self._last_indices = None  # host int64 array of the last sample() call (numpy sampler)
        self._lay_ref = C.byref(self._lay)
        self._dev_index = self._device.index

    @property
    def rows(self) -> torch.Tensor:
        return self._rows

    @property
    def row_layout(self) -> _lib.RowLayout:
        return self._lay

    def _dataset_tensors(self, data: Dict[str, np.ndarray]):
        """The five arrays of a D4RL-style dataset as float32 device tensors, once it is known to fit this buffer."""
        if self._size != 0:
            raise ValueError("Trying to load data into non-empty replay buffer")
        if data["observations"].shape[0] > self._buffer_size:
            raise ValueError("Replay buffer is smaller than the dataset you are trying to load!")
        # torch.tensor keeps the strides of a non-C-order array (Fortran order, a transposed view); the pack reads row-major
        s, a, r, s2, d = [torch.tensor(data[k], dtype=torch.float32, device=self._device).contiguous()
                          for k in ("observations", "actions", "rewards", "next_observations", "terminals")]
        if s.shape[1] != self._state_dim or a.shape[1] != self._action_dim:
            raise ValueError("dataset dims do not match the buffer")
        return s, a, r.reshape(-1), s2, d.reshape(-1)

    def load_d4rl_dataset(self, data: Dict[str, np.ndarray]):
        s, a, r, s2, d = self._dataset_tensors(data)
        n = s.shape[0]
        _lib.call_on_device(self._dev_index, self._device, None, "iql_replay_pack", self._L.iql_replay_pack,
                            self._rows.data_ptr(), self._lay_ref, 0, n, s.data_ptr(), a.data_ptr(), r.data_ptr(),
                            s2.data_ptr(), d.data_ptr())
        torch.cuda.current_stream(self._device).synchronize()  # inputs are temporaries
        self._size += n
        self._pointer = min(self._size, n)
        print(f"Dataset size: {n}")

    def ingest_d4rl_dataset(self, data: Dict[str, np.ndarray], normalize: bool = True, eps: float = 1e-3,
                            reward_mod: Optional[Dict[str, float]] = None, reward_shift: float = 0.0):
        """The reference's preprocessing + load in one device pass (jsrl_w_iql.py:344-368): state mean / std with
        numpy's summation order (bit-exact against ``compute_mean_std``, iql.py:77-80), ``normalize_states`` of
        observations and next observations, the reward rescaling of ``modify_reward`` (``reward_mod`` = its return
        value for locomotion tasks; ``reward_shift=1`` for antmaze), then the pack.  ``data`` is NOT modified.
        Returns ``(state_mean, state_std)`` as numpy arrays (``(0, 1)`` when ``normalize`` is off), which the caller
        hands to ``wrap_env`` exactly as with the reference functions."""
        s, a, r, s2, d = self._dataset_tensors(data)
        n = s.shape[0]
        mean = torch.zeros(self._state_dim, dtype=torch.float32, device=self._device)
        std = torch.ones(self._state_dim, dtype=torch.float32, device=self._device)
        rdiv = rmul = 1.0
        if reward_mod:
            rdiv = float(np.float32(reward_mod["max_ret"] - reward_mod["min_ret"]))
            rmul = float(reward_mod["max_episode_steps"])
        _lib.call_on_device(self._dev_index, self._device, None, "iql_replay_ingest", self._L.iql_replay_ingest,
                            self._rows.data_ptr(), self._lay_ref, 0, n, s.data_ptr(), a.data_ptr(), r.data_ptr(),
                            s2.data_ptr(), d.data_ptr(), int(bool(normalize)), float(eps), mean.data_ptr(), std.data_ptr(),
                            rdiv, rmul, float(reward_shift))
        torch.cuda.current_stream(self._device).synchronize()
        self._size += n
        self._pointer = min(self._size, n)
        print(f"Dataset size: {n}")
        if not normalize:
            return 0, 1
        return mean.cpu().numpy(), std.cpu().numpy()

    def _high(self) -> int:
        return min(self._size, self._pointer) if self._offline_semantics else self._size

    def _out_slot(self, B: int) -> "_SampleSlot":
        """Next set of cached output tensors (ring of ``_N_SLOTS``; a batch returned by ``sample`` is overwritten by the
        ``_N_SLOTS``-th call after it -- construct the buffer with ``fresh_outputs=True`` for the reference's
        one-allocation-per-call behaviour)."""
        ring = self._slots
        if not ring or ring[0].B != B:
            for sl in ring:
                _SAMPLED.pop(id(sl.out[0]), None)
            ring = self._slots = [_SampleSlot(self, B) for _ in range(_N_SLOTS)]
            for sl in ring:
                _SAMPLED[id(sl.out[0])] = sl
            self._slot_i = 0
        sl = ring[self._slot_i]
        self._slot_i = (self._slot_i + 1) % _N_SLOTS
        return sl

    def sample(self, batch_size: int) -> TensorBatch:
        B = int(batch_size)
        high = self._high()
        if self._sampler == "numpy":
            idx_host = np.random.randint(0, high, size=B)  # raises ValueError on an empty buffer, like the reference
        elif high <= 0:
            raise ValueError("low >= high")
        sl = _SampleSlot(self, B) if self._fresh_outputs else self._out_slot(B)
        s, a, r, s2, d = sl.ptrs
        if self._sampler == "numpy":
            # the indices ride in the kernel parameters: no staging buffer, no host->device copy
            _lib.call_on_device(self._dev_index, self._device, None, "iql_replay_sample_host", self._L.iql_replay_sample_host,
                                self._rows.data_ptr(), self._lay_ref, high, B, idx_host.__array_interface__["data"][0],
                                s, a, r, s2, d)
            sl.idx_host, sl.high = idx_host, high
            self._last_indices = idx_host
        else:
            sl.idx_host = None
            _lib.call_on_device(self._dev_index, self._device, None, "iql_replay_sample", self._L.iql_replay_sample,
                                self._rows.data_ptr(), self._lay_ref, high, B, None, self._seed, self._sample_calls,
                                s, a, r, s2, d, None)
        self._sample_calls += 1
        out = sl.out
        sl.ver = (out[0]._version, out[1]._version, out[2]._version, out[3]._version, out[4]._version)
        return list(out)

    def add_transition(self, state: np.ndarray, action: np.ndarray, reward: float, next_state: np.ndarray, done: bool):
        lay = self._lay
        st = np.ascontiguousarray(state, dtype=np.float32).reshape(-1)
        ac = np.ascontiguousarray(action, dtype=np.float32).reshape(-1)
        ns = np.ascontiguousarray(next_state, dtype=np.float32).reshape(-1)
        if st.size != self._state_dim or ns.size != self._state_dim or ac.size != self._action_dim:
            raise ValueError("transition dims do not match the buffer")
        if not 0 <= self._pointer < self._buffer_size:
            # a buffer loaded to the brim leaves _pointer == buffer_size (iql.py:168); the reference's
            # `self._states[self._pointer] = ...` raises IndexError there too
            raise IndexError(f"index {self._pointer} is out of bounds for dimension 0 with size {self._buffer_size}")
        if lay.row_floats <= 960:
            # the packed row rides in the kernel parameters: one launch, no staging row, no copy
            _lib.call_on_device(self._dev_index, self._device, None, "iql_replay_insert_host", self._L.iql_replay_insert_host,
                                self._rows.data_ptr(), self._lay_ref, self._pointer, st.ctypes.data, ac.ctypes.data,
                                float(reward), ns.ctypes.data, float(done))
        else:
            _lib.call_on_device(self._dev_index, self._device, None, "iql_replay_insert", self._insert_staged,
                                st, ac, reward, ns, done)
        self._pointer = (self._pointer + 1) % self._buffer_size
        self._size = min(self._size + 1, self._buffer_size)

    def _insert_staged(self, st, ac, reward, ns, done, cur) -> int:
        # two pinned staging rows used alternately, each guarded by an event recorded after its host->device copy
        lay = self._lay
        i = self._stage_i
        self._stage_i = i ^ 1
        if self._stage_ev[i] is not None:
            self._stage_ev[i].synchronize()  # this slot's previous host->device copy (two inserts ago) has run
        h = self._stage_host[i].numpy()
        h[:] = 0.0
        h[lay.off_state:lay.off_state + self._state_dim] = st
        h[lay.off_action:lay.off_action + self._action_dim] = ac
        h[lay.off_reward] = float(reward)
        h[lay.off_next_state:lay.off_next_state + self._state_dim] = ns
        h[lay.off_done] = float(done)
        self._stage[i].copy_(self._stage_host[i], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self._device))
        self._stage_ev[i] = ev
        return self._L.iql_replay_insert(self._rows.data_ptr(), self._lay_ref, self._pointer, self._stage[i].data_ptr(), cur)


# ---------------------------------------------------------------------------
# network containers (parameter names/shapes = checkpoint contract, iql.py:305-442)
# ---------------------------------------------------------------------------
class Squeeze(nn.Module):
    def __init__(self, dim=-1):
        super().__init__()
        self.dim = dim

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return x.squeeze(dim=self.dim)


class MLP(nn.Module):
    """Linear/ReLU[/Dropout] stack in one ``nn.Sequential`` called ``net``.
    ``dropout_when_not_none`` selects the offline variant's rule (a Dropout
    module is inserted whenever dropout is not None, offline/iql.py:287-288)."""

    def __init__(self, dims: Sequence[int], activation_fn: Callable[[], nn.Module] = nn.ReLU,
                 output_activation_fn: Callable[[], nn.Module] = None, squeeze_output: bool = False,
                 dropout: Optional[float] = 0.0, dropout_when_not_none: bool = False):
        super().__init__()
        if len(dims) < 2:
            raise ValueError("MLP requires at least two dims (input and output)")
        use_dropout = (dropout is not None) if dropout_when_not_none else (dropout is not None and dropout > 0.0)
        mods: List[nn.Module] = []
        for fan_in, fan_out in zip(dims[:-2], dims[1:-1]):
            mods += [nn.Linear(fan_in, fan_out), activation_fn()]
            if use_dropout:
                mods.append(nn.Dropout(dropout))
        mods.append(nn.Linear(dims[-2], dims[-1]))
        if output_activation_fn is not None:
            mods.append(output_activation_fn())
        if squeeze_output:
            if dims[-1] != 1:
                raise ValueError("Last dim must be 1 when squeezing")
            mods.append(Squeeze(-1))
        self.net = nn.Sequential(*mods)
        self.has_dropout_modules = use_dropout
        self.dropout_p = float(dropout) if dropout is not None else 0.0

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.net(x)


def _aliases_arena(eng: EnsembleEngine, weight: torch.Tensor, log_std: Optional[torch.Tensor] = None) -> bool:
    """The parameters an engine act reads still point into ``eng.params``; False once they were re-pointed (module
    moved / re-initialised), and the stock torch path serves the call."""
    lo = eng.params.data_ptr()
    hi = lo + eng.params.numel() * 4
    return weight.device == eng.device and lo <= weight.data_ptr() < hi and (log_std is None or lo <= log_std.data_ptr() < hi)


class _PolicyBase(nn.Module):
    def __init__(self, state_dim, act_dim, max_action, hidden_dim, n_hidden, dropout, dropout_when_not_none):
        super().__init__()
        self.net = MLP([state_dim] + [hidden_dim] * n_hidden + [act_dim], output_activation_fn=nn.Tanh,
                       dropout=dropout, dropout_when_not_none=dropout_when_not_none)
        self.state_dim, self.act_dim = state_dim, act_dim
        self.hidden_dim, self.n_hidden = hidden_dim, n_hidden
        self.max_action = max_action
        self._engine_ref = None  # (EnsembleEngine, member) once the parameters alias an engine arena

    def _engine_act(self, state: np.ndarray) -> Optional[np.ndarray]:
        """clamp(max_action * tanh(MLP(s))) from the engine's fused act kernel (reads the arena the parameters
        alias) instead of 2 n_hidden + 3 stock torch launches; None when the module is not engine-backed."""
        ref = self._engine_ref
        if ref is None:
            return None
        eng, member = ref
        if not _aliases_arena(eng, self.net.net[0].weight):
            return None
        return eng.act_host(member, state, float(self.max_action))

    def __deepcopy__(self, memo):
        ref, self._engine_ref = self._engine_ref, None  # a copy owns its parameters, not the arena
        try:
            cls = self.__class__
            new = cls.__new__(cls)
            memo[id(self)] = new
            for k, v in self.__dict__.items():
                setattr(new, k, copy.deepcopy(v, memo))
        finally:
            self._engine_ref = ref
        return new

    def _clip(self, action: torch.Tensor) -> np.ndarray:
        scaled = torch.clamp(self.max_action * action, -self.max_action, self.max_action)
        return scaled.cpu().data.numpy().flatten()


class GaussianPolicy(_PolicyBase):
    def __init__(self, state_dim: int, act_dim: int, max_action: float, hidden_dim: int = 256, n_hidden: int = 2,
                 dropout: Optional[float] = 0.0, dropout_when_not_none: bool = False):
        super().__init__(state_dim, act_dim, max_action, hidden_dim, n_hidden, dropout, dropout_when_not_none)
        self.log_std = nn.Parameter(torch.zeros(act_dim, dtype=torch.float32))

    def forward(self, obs: torch.Tensor) -> Normal:
        std = self.log_std.clamp(LOG_STD_MIN, LOG_STD_MAX).exp()
        return Normal(self.net(obs), std)

    @torch.no_grad()
    def act(self, state: np.ndarray, device: str = "cpu"):
        if not self.training:  # eval mode: the mean action, one fused kernel on the engine
            a = self._engine_act(state)
            if a is not None:
                return a
        elif not (self.net.has_dropout_modules and self.net.dropout_p > 0.0):
            # training mode, no active dropout (the learner's env steps of the online loop): the engine kernel returns the
            # distribution's mean and std, the sample `mean + std * N(0, 1)` is drawn on the host from torch's CPU generator
            # (the reference draws it from the generator of the policy's device: same distribution, seeded by the same
            # torch.manual_seed, not the same stream -- sampled actions are not part of the parity contract)
            ms = self._engine_gaussian(state)
            if ms is not None:
                mean, std = ms
                sample = mean + std * torch.randn(mean.shape[0]).numpy()
                return np.clip(self.max_action * sample, -self.max_action, self.max_action).astype(np.float32)
        obs = torch.tensor(state.reshape(1, -1), device=device, dtype=torch.float32)
        dist = self(obs)
        return self._clip(dist.sample() if self.training else dist.mean)

    def _engine_gaussian(self, state: np.ndarray):
        ref = self._engine_ref
        if ref is None:
            return None
        eng, member = ref
        if not _aliases_arena(eng, self.net.net[0].weight, self.log_std):
            return None
        return eng.act_host_gaussian(member, state)


class DeterministicPolicy(_PolicyBase):
    def __init__(self, state_dim: int, act_dim: int, max_action: float, hidden_dim: int = 256, n_hidden: int = 2,
                 dropout: Optional[float] = 0.0, dropout_when_not_none: bool = False):
        super().__init__(state_dim, act_dim, max_action, hidden_dim, n_hidden, dropout, dropout_when_not_none)

    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        return self.net(obs)

    @torch.no_grad()
    def act(self, state: np.ndarray, device: str = "cpu"):
        if not (self.training and self.net.has_dropout_modules and self.net.dropout_p > 0.0):
            a = self._engine_act(state)  # no active dropout: the deterministic action, one fused kernel
            if a is not None:
                return a
        obs = torch.tensor(state.reshape(1, -1), device=device, dtype=torch.float32)
        return self._clip(self(obs))


class TwinQ(nn.Module):
    def __init__(self, state_dim: int, action_dim: int, hidden_dim: int = 256, n_hidden: int = 2):
        super().__init__()
        widths = [state_dim + action_dim] + [hidden_dim] * n_hidden + [1]
        self.q1 = MLP(widths, squeeze_output=True)
        self.q2 = MLP(widths, squeeze_output=True)
        self.state_dim, self.action_dim = state_dim, action_dim
        self.hidden_dim, self.n_hidden = hidden_dim, n_hidden

    def both(self, state: torch.Tensor, action: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        sa = torch.cat([state, action], 1)
        return self.q1(sa), self.q2(sa)

    def forward(self, state: torch.Tensor, action: torch.Tensor) -> torch.Tensor:
        return torch.min(*self.both(state, action))


class ValueFunction(nn.Module):
    def __init__(self, state_dim: int, hidden_dim: int = 256, n_hidden: int = 2):
        super().__init__()
        self.v = MLP([state_dim] + [hidden_dim] * n_hidden + [1], squeeze_output=True)
        self.state_dim, self.hidden_dim, self.n_hidden = state_dim, hidden_dim, n_hidden

    def forward(self, state: torch.Tensor) -> torch.Tensor:
        return self.v(state)


# ---------------------------------------------------------------------------
# the learner
# ---------------------------------------------------------------------------
_COUNTER_OF = {"qf": "q", "vf": "v", "actor": "actor"}  # module group -> its optimizer's step counter in `_steps`


def _adam_group(opt: torch.optim.Optimizer) -> dict:
    if not isinstance(opt, torch.optim.Adam) or len(opt.param_groups) != 1:
        raise NotImplementedError("the engine implements torch.optim.Adam with a single param group")
    g = opt.param_groups[0]
    if g.get("weight_decay", 0) != 0 or g.get("amsgrad", False) or g.get("maximize", False):
        raise NotImplementedError("Adam with weight_decay / amsgrad / maximize is not implemented by the engine")
    return g


class ImplicitQLearning:
    """Same constructor, attributes and methods as the reference trainer
    (iql.py:445-606); ``train`` runs one fused update on the GPU engine.

    Keyword-only extras: ``math_mode`` ("tf32" tensor-core path or "fp32" SIMT
    validation path) and ``seed`` (Philox key for in-kernel dropout masks)."""

    def __init__(self, max_action: float, actor: nn.Module, actor_optimizer: torch.optim.Optimizer,
                 q_network: nn.Module, q_optimizer: torch.optim.Optimizer, v_network: nn.Module,
                 v_optimizer: torch.optim.Optimizer, iql_tau: float = 0.7, beta: float = 3.0,
                 max_steps: Optional[int] = 1000000, discount: float = 0.99, tau: float = 0.005,
                 device: str = "cpu", *, math_mode: str = "tf32", seed: int = 0, step_path: str = "auto"):
        self.device = _lib.require_cuda(device)
        if not isinstance(q_network, TwinQ) or not isinstance(v_network, ValueFunction) or \
                not isinstance(actor, (GaussianPolicy, DeterministicPolicy)):
            raise TypeError("ImplicitQLearning needs jsrl_corl_b200 TwinQ / ValueFunction / *Policy modules")
        self.max_action = max_action
        self.qf = q_network.to(self.device)
        self.q_target = copy.deepcopy(self.qf).requires_grad_(False).to(self.device)
        self.vf = v_network.to(self.device)
        self.actor = actor.to(self.device)
        self.v_optimizer, self.q_optimizer, self.actor_optimizer = v_optimizer, q_optimizer, actor_optimizer
        self.actor_lr_schedule = CosineAnnealingLR(self.actor_optimizer, max_steps) if max_steps is not None else None
        self.iql_tau, self.beta, self.discount, self.tau = iql_tau, beta, discount, tau
        self._math_mode, self._seed, self._step_path = math_mode, int(seed), step_path
        self._engine: Optional[EnsembleEngine] = None
        self._pushed = None
        self._total_it = 0
        self._steps = {"v": 0, "q": 0, "actor": 0}
        self._step_tensors: Dict[str, torch.Tensor] = {}
        self._step_views: Dict[str, np.ndarray] = {}
        self._bound_rows: Optional[torch.Tensor] = None
        self._path_counts = [0, 0]  # train() calls served by [engine-side gather of sample()'s indices, staged dense batch]
        self._published = False
        self._moment_cache = None
        self._loss_buf: Optional[torch.Tensor] = None
        S, A, H, L = self.qf.state_dim, self.qf.action_dim, self.qf.hidden_dim, self.qf.n_hidden
        if (self.vf.state_dim, self.vf.hidden_dim, self.vf.n_hidden) != (S, H, L) or \
                (self.actor.state_dim, self.actor.hidden_dim, self.actor.n_hidden) != (S, H, L):
            raise ValueError("q / v / actor networks must share state_dim, hidden_dim and n_hidden")
        if self.actor.act_dim != A:
            raise RuntimeError("Actions shape missmatch")
        self._dims = (S, A, H, L)

    # ---- counters ------------------------------------------------------
    @property
    def total_it(self) -> int:
        return self._total_it

    @total_it.setter
    def total_it(self, v: int):
        self._total_it = int(v)
        if self._engine is not None:
            self._engine.set_counters(0, total_it=int(v))

    # ---- engine adoption -------------------------------------------------
    def _modules(self):
        return {"qf": self.qf, "vf": self.vf, "actor": self.actor}

    def _optimizers(self):
        return {"qf": self.q_optimizer, "vf": self.v_optimizer, "actor": self.actor_optimizer}

    def _ensure_engine(self, batch_size: int) -> EnsembleEngine:
        if self._engine is not None and self._engine.batch_size == batch_size:
            return self._engine
        S, A, H, L = self._dims
        old = self._engine
        if old is not None:  # batch size changed: migrate the state to a new engine
            self._pull_counters()
            self._publish_optimizer_state()
        eng = EnsembleEngine(1, S, A, H, L, batch_size, isinstance(self.actor, DeterministicPolicy),
                             self._math_mode, self.device, max_steps_per_call=64, step_path=self._step_path)
        drop_keys = self.actor.net.has_dropout_modules
        views = eng.param_views(0, drop_keys)
        m_views, v_views = eng.moment_views(0, drop_keys)
        with torch.no_grad():
            for grp, mod in self._modules().items():
                opt = self._optimizers()[grp]
                for name, view in views[grp].items():
                    p = mod.get_parameter(name)
                    view.copy_(p.data)
                    st = opt.state.get(p, None)
                    if st and "exp_avg" in st:
                        m_views[grp][name].copy_(st["exp_avg"])
                        v_views[grp][name].copy_(st["exp_avg_sq"])
                        self._steps[_COUNTER_OF[grp]] = int(float(st["step"]))
                    p.data = view  # module parameters now alias the engine arena
            for name, view in eng.target_views(0).items():
                p = self.q_target.get_parameter(name)
                view.copy_(p.data)
                p.data = view
        self._engine = eng
        self._bound_rows = None
        self.actor._engine_ref = (eng, 0)
        self._pushed = None
        self._published = False
        self._push_counters()
        self._publish_optimizer_state()
        return eng

    def _push_counters(self):
        sched = self.actor_lr_schedule
        self._engine.set_counters(0, v_step=self._steps["v"], q_step=self._steps["q"], actor_step=self._steps["actor"],
                                  sched_epoch=sched.last_epoch if sched is not None else 0, total_it=self._total_it)

    def _pull_counters(self):
        c = self._engine.get_counters(0)
        self._steps = {"v": c.v_step, "q": c.q_step, "actor": c.actor_step}

    def _publish_optimizer_state(self):
        """Expose the arena moments through the torch optimizers so that
        ``optimizer.state_dict()`` has the stock Adam layout (step/exp_avg/exp_avg_sq)."""
        eng = self._engine
        drop_keys = self.actor.net.has_dropout_modules
        if getattr(self, "_moment_cache", None) is None or self._moment_cache[0] is not eng:
            self._moment_cache = (eng,) + tuple(eng.moment_views(0, drop_keys))  # one set of view objects per engine
        _, m_views, v_views = self._moment_cache
        attached = 0
        for grp, mod in self._modules().items():
            opt = self._optimizers()[grp]
            steps = self._steps[_COUNTER_OF[grp]]
            if steps == 0:
                continue  # torch creates Adam state lazily at the first step
            # one CPU step tensor per optimizer, shared by its parameters and updated in place after every
            # update, so `optimizer.state_dict()` is current even when called directly on the optimizer
            step_t = self._step_tensors.setdefault(grp, torch.tensor(0.0))
            step_t.fill_(float(steps))
            self._step_views[grp] = step_t.numpy()  # shares memory: train() updates the count without a torch op
            for name in m_views[grp]:
                p = mod.get_parameter(name)
                st = opt.state.get(p)
                if st is None or st.get("exp_avg") is not m_views[grp][name] or st.get("step") is not step_t:
                    opt.state[p] = {"step": step_t, "exp_avg": m_views[grp][name], "exp_avg_sq": v_views[grp][name]}
            attached += 1
        # true only when all three optimizers really hold arena views (a checkpoint with empty optimizer state
        # loaded into a stepped trainer resets this through load_state_dict)
        self._published = attached == 3

    def _push_hparams(self):
        groups = getattr(self, "_adam_groups", None)
        if groups is None or groups[0] is not self.q_optimizer.param_groups[0]:
            # validated once per optimizer object: the param-group dicts are stable, later calls only read them
            gq, gv, ga = _adam_group(self.q_optimizer), _adam_group(self.v_optimizer), _adam_group(self.actor_optimizer)
            self._adam_groups = (gq, gv, ga)
        gq, gv, ga = self._adam_groups
        for g in (gv, ga):
            if g["betas"] != gq["betas"] or g["eps"] != gq["eps"]:
                raise NotImplementedError("the three Adam optimizers must share betas and eps")
        sched = self.actor_lr_schedule
        if sched is not None:
            actor_lr, t_max, eta_min = sched.base_lrs[0], int(sched.T_max), float(sched.eta_min)
        else:
            actor_lr, t_max, eta_min = ga["lr"], 0, 0.0
        p = self.actor.net.dropout_p if self.actor.net.has_dropout_modules else 0.0
        key = (self.beta, self.iql_tau, self.discount, self.tau, gv["lr"], gq["lr"], actor_lr, p,
               tuple(gq["betas"]), gq["eps"], eta_min, t_max, self._seed)
        if key != self._pushed:
            self._engine.set_hparams(0, beta=self.beta, iql_tau=self.iql_tau, discount=self.discount, tau=self.tau,
                                     vf_lr=gv["lr"], qf_lr=gq["lr"], actor_lr=actor_lr, actor_dropout=p,
                                     adam_beta1=gq["betas"][0], adam_beta2=gq["betas"][1], adam_eps=gq["eps"],
                                     lr_eta_min=eta_min, cosine_t_max=t_max, seed=self._seed)
            self._pushed = key

    def _advance_schedule(self, k: int):
        """Host mirror of CosineAnnealingLR.step() (recursive form, like torch)."""
        sched = self.actor_lr_schedule
        if sched is None:
            return
        group = self.actor_optimizer.param_groups[0]
        base, t_max, eta_min = sched.base_lrs[0], sched.T_max, sched.eta_min
        lr, e = group["lr"], sched.last_epoch
        for _ in range(k):
            e += 1
            if (e - 1 - t_max) % (2 * t_max) == 0:
                lr = lr + (base - eta_min) * (1 - math.cos(math.pi / t_max)) / 2
            else:
                lr = (1 + math.cos(math.pi * e / t_max)) / (1 + math.cos(math.pi * (e - 1) / t_max)) * (lr - eta_min) + eta_min
        group["lr"] = lr
        sched.last_epoch = e
        sched._last_lr = [lr]
        if hasattr(sched, "_step_count"):
            sched._step_count += k

    # ---- the update -------------------------------------------------------
    def train(self, batch: TensorBatch) -> Dict[str, float]:
        observations, actions, rewards, next_observations, dones = batch
        if actions.dim() != 2 or actions.shape[1] != self._dims[1]:
            raise RuntimeError("Actions shape missmatch")
        eng = self._ensure_engine(int(observations.shape[0]))
        self._push_hparams()
        slot = _SAMPLED.get(id(observations))
        rb = slot.rb() if slot is not None else None
        if rb is not None and slot.idx_host is not None and rb._device == eng.device and slot.untouched(batch):
            # the batch is what ReplayBuffer.sample just returned: the engine gathers the same rows itself from the
            # host-drawn indices (identical values, no re-pack of the five dense tensors)
            if self._bound_rows is not rb._rows:
                eng.bind_replay(0, rb._rows, max(rb._size, 1))
                self._bound_rows = rb._rows
            eng.host_step(host_indices=slot.idx_host.__array_interface__["data"][0], wait=False)
            self._path_counts[0] += 1
        else:
            eng.host_step(batch=(observations, actions, rewards, next_observations, dones), wait=False)
            self._path_counts[1] += 1
        # (the step is running: the host-side mirrors of the counters / schedule are updated meanwhile)
        self._total_it += 1
        st = self._steps
        st["v"] += 1
        st["q"] += 1
        st["actor"] += 1
        if self._published:
            sv = self._step_views
            sv["qf"][...] = st["q"]
            sv["vf"][...] = st["v"]
            sv["actor"][...] = st["actor"]
        else:
            self._publish_optimizer_state()
        self._advance_schedule(1)
        v_loss, q_loss, a_loss = eng.host_step_wait()
        return {"value_loss": v_loss, "q_loss": q_loss, "actor_loss": a_loss}

    # ---- checkpoints (iql.py:565-606) --------------------------------------
    def state_dict(self) -> Dict[str, Any]:
        if self._engine is not None:
            self._publish_optimizer_state()
        sched = self.actor_lr_schedule
        return {
            "qf": self.qf.state_dict(),
            "q_optimizer": self.q_optimizer.state_dict(),
            "vf": self.vf.state_dict(),
            "v_optimizer": self.v_optimizer.state_dict(),
            "actor": self.actor.state_dict(),
            "actor_optimizer": self.actor_optimizer.state_dict(),
            "actor_lr_schedule": sched.state_dict() if sched is not None else {},
            "total_it": self.total_it,
        }

    def _absorb_optimizer(self, grp: str):
        """After optimizer.load_state_dict: copy its moments into the arena."""
        opt, mod = self._optimizers()[grp], self._modules()[grp]
        key = _COUNTER_OF[grp]
        step = 0
        if self._engine is None:
            for st in opt.state.values():
                if "step" in st:
                    step = int(float(st["step"]))
            self._steps[key] = step
            return
        m_views, v_views = self._engine.moment_views(0, self.actor.net.has_dropout_modules)
        with torch.no_grad():
            for name in m_views[grp]:
                p = mod.get_parameter(name)
                st = opt.state.get(p, None)
                if st and "exp_avg" in st:
                    m_views[grp][name].copy_(st["exp_avg"])
                    v_views[grp][name].copy_(st["exp_avg_sq"])
                    step = int(float(st["step"]))
                else:
                    m_views[grp][name].zero_()
                    v_views[grp][name].zero_()
        self._steps[key] = step

    def _reset_target(self):
        if self._engine is not None:
            self._engine.sync_target(0)
        else:
            self.q_target = copy.deepcopy(self.qf)

    def load_state_dict(self, state_dict: Dict[str, Any]):
        self.qf.load_state_dict(state_dict["qf"])
        self.q_optimizer.load_state_dict(state_dict["q_optimizer"])
        self._absorb_optimizer("qf")
        self._reset_target()
        self.vf.load_state_dict(state_dict["vf"])
        self.v_optimizer.load_state_dict(state_dict["v_optimizer"])
        self._absorb_optimizer("vf")
        self.actor.load_state_dict(state_dict["actor"])
        self.actor_optimizer.load_state_dict(state_dict["actor_optimizer"])
        self._absorb_optimizer("actor")
        if self.actor_lr_schedule is not None:
            self.actor_lr_schedule.load_state_dict(state_dict["actor_lr_schedule"])
        self._total_it = state_dict["total_it"]
        self._pushed = None
        self._published = False
        if self._engine is not None:
            self._push_counters()
            self._publish_optimizer_state()

    def partial_load_state_dict(self, state_dict: Dict[str, Any]):
        """Networks + schedule + total_it, no optimizers (iql.py:595-606)."""
        self.qf.load_state_dict(state_dict["qf"])
        self._reset_target()
        self.vf.load_state_dict(state_dict["vf"])
        self.actor.load_state_dict(state_dict["actor"])
        if self.actor_lr_schedule is not None:
            self.actor_lr_schedule.load_state_dict(state_dict["actor_lr_schedule"])
        self._total_it = state_dict["total_it"]
        self._pushed = None
        if self._engine is not None:
            self._push_counters()
