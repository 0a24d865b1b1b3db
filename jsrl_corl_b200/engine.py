"""Python handle over the C-ABI engine: S independent IQL learners on one GPU.

torch is plumbing here: it allocates the flat device arenas (parameters, Adam
moments, target network, gradients, workspace), hands their pointers to the
engine and exposes zero-copy views with the reference's ``state_dict`` key
layout (algorithms/finetune/iql.py:565-579).  All arithmetic of the update runs
inside ``libiql_b200.so``.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib
from ._lib import Config, Counters, HParams, Layout, TensorInfo

NET_NAMES = {_lib.NET_Q1: "q1", _lib.NET_Q2: "q2", _lib.NET_V: "v", _lib.NET_ACTOR: "actor"}
MATH_MODES = {"fp32": _lib.MATH_FP32_SIMT, "tf32": _lib.MATH_TF32_TCGEN05}


def linear_indices(n_hidden: int, dropout: bool) -> List[int]:
    """nn.Sequential indices of the Linear modules of the reference MLP
    (iql.py:328-341): a Dropout after every ReLU shifts them to 0,3,6,..."""
    stride = 3 if dropout else 2
    return [stride * i for i in range(n_hidden + 1)]


def query_layout(n_members, state_dim, action_dim, hidden_dim, n_hidden, batch_size, deterministic,
                 math_mode="fp32", max_steps_per_call=1):
    """Host-only: create a handle, read its layout and tensor table, destroy it.
    Works without a GPU (used by CPU tests and by shape planning)."""
    L = _lib.lib()
    cfg = Config(n_members, state_dim, action_dim, hidden_dim, n_hidden, batch_size, int(bool(deterministic)),
                 MATH_MODES[math_mode], max_steps_per_call)
    h = C.c_void_p()
    _lib.check(L.iql_create(C.byref(cfg), C.byref(h)), None, "iql_create")
    try:
        lay, tensors = _read_layout(L, h)
    finally:
        L.iql_destroy(h)
    return lay, [(t.net, t.layer, t.kind, t.rows, t.cols, t.offset, t.ld) for t in tensors]


def _read_layout(L, h):
    """The handle's arena layout and its tensor table ([TensorInfo], in table order)."""
    lay = Layout()
    _lib.check(L.iql_get_layout(h, C.byref(lay)), h)
    tensors = []
    for i in range(lay.n_tensors):
        t = TensorInfo()
        _lib.check(L.iql_tensor_at(h, i, C.byref(t)), h)
        tensors.append(t)
    return lay, tensors


def index_state_rows(rngs) -> np.ndarray:
    """[len(rngs), IQL_MT_STATE_WORDS] uint32: each ``np.random.RandomState``'s generator in the device layout of
    ``iql_bind_index_streams`` -- the key and pos of ``get_state()``, then a pad word."""
    rows = np.zeros((len(rngs), _lib.MT_STATE_WORDS), dtype=np.uint32)
    for i, rng in enumerate(rngs):
        if not isinstance(rng, np.random.RandomState):
            raise ValueError(f"index streams are np.random.RandomState objects, got {type(rng).__name__}")
        name, key, pos, _, _ = rng.get_state()
        if name != "MT19937":
            raise ValueError(f"index stream {i} is a {name} generator, not MT19937")
        rows[i, :624] = key
        rows[i, 624] = pos
    return rows


def load_index_state_rows(rngs, rows: np.ndarray) -> None:
    """Inverse of ``index_state_rows``: key and pos go back into each RandomState (``set_state``); its cached Gaussian
    (``has_gauss`` / ``cached_gaussian``), which the index draws never touch, is kept."""
    for rng, row in zip(rngs, rows):
        _, _, _, has_gauss, cached = rng.get_state()
        rng.set_state(("MT19937", np.array(row[:624], dtype=np.uint32), int(row[624]), has_gauss, cached))


class EnsembleEngine:
    """S-member IQL update engine bound to one CUDA device."""

    def __init__(self, n_members: int, state_dim: int, action_dim: int, hidden_dim: int = 256, n_hidden: int = 2,
                 batch_size: int = 256, deterministic: bool = False, math_mode: str = "tf32",
                 device="cuda", max_steps_per_call: int = 256, step_path: str = "auto", strict_tf32: bool = False):
        self.device = _lib.require_cuda(device)
        self._L = _lib.lib()
        if math_mode not in MATH_MODES:
            raise ValueError(f"math_mode must be one of {sorted(MATH_MODES)}")
        self.n_members, self.state_dim, self.action_dim = n_members, state_dim, action_dim
        self.hidden_dim, self.n_hidden, self.batch_size = hidden_dim, n_hidden, batch_size
        self.deterministic, self.math_mode = bool(deterministic), math_mode
        self.max_steps_per_call = max_steps_per_call
        cfg = Config(n_members, state_dim, action_dim, hidden_dim, n_hidden, batch_size, int(self.deterministic),
                     MATH_MODES[math_mode], max_steps_per_call)
        self._h = C.c_void_p()
        _lib.check(self._L.iql_create(C.byref(cfg), C.byref(self._h)), None, "iql_create")
        if step_path not in _lib.STEP_PATHS:
            raise ValueError(f"step_path must be one of {sorted(_lib.STEP_PATHS)}")
        _lib.check(self._L.iql_set_option(self._h, _lib.OPT_STEP_PATH, _lib.STEP_PATHS[step_path]), self._h, "iql_set_option")
        self.step_path = step_path
        self.layout, self.tensors = _read_layout(self._L, self._h)
        P, PQ = self.layout.param_floats, self.layout.q_floats
        with torch.cuda.device(self.device):
            f32 = dict(dtype=torch.float32, device=self.device)
            self.params = torch.zeros(n_members, P, **f32)
            self.exp_avg = torch.zeros(n_members, P, **f32)
            self.exp_avg_sq = torch.zeros(n_members, P, **f32)
            self.grads = torch.zeros(n_members, P, **f32)
            self.target = torch.zeros(n_members, PQ, **f32)
            self.workspace = torch.zeros(self.layout.workspace_bytes, dtype=torch.uint8, device=self.device)
            # dedicated stream: CUDA-graph capture is not allowed on the legacy default stream
            self.stream = torch.cuda.Stream(device=self.device)
            # inside the guard: the engine creates its side stream / events on the CURRENT device and sets
            # per-device kernel attributes (engines on cuda:N while the process sits on cuda:0 must work)
            _lib.check(self._L.iql_bind_state(self._h, self.params.data_ptr(), self.exp_avg.data_ptr(),
                                              self.exp_avg_sq.data_ptr(), self.target.data_ptr(), self.grads.data_ptr(),
                                              self.workspace.data_ptr(), self.workspace.numel()), self._h, "iql_bind_state")
        # which kernels serve this shape: math_mode="tf32" outside the tcgen05 shapes (batch % 128, hidden % 256) runs the
        # FP32 CUDA-core kernels -- reported here, and refused when the caller insists on tensor cores
        self.paths = self._read_paths()
        if math_mode == "tf32" and strict_tf32 and not self.paths["tensor_cores"]:
            raise ValueError(f"math_mode='tf32' with strict_tf32: batch {batch_size} / hidden {hidden_dim} is outside the tcgen05 "
                             "kernels (batch % 128 == 0 and hidden % 256 == 0 required); the FP32 kernels would run")
        self.act_calls = 0
        # host buffers of act_host / act_host_gaussian (observation in; action or mean, std out)
        self._act_in = np.zeros(state_dim, dtype=np.float32)
        self._act_out = np.zeros(action_dim, dtype=np.float32)
        self._act_std = np.zeros(action_dim, dtype=np.float32)
        self._act_ptrs = (self._act_in.ctypes.data, self._act_out.ctypes.data, self._act_std.ctypes.data)
        self._hparams = [self._default_hparams(m) for m in range(n_members)]
        self._batch_sizes = [batch_size] * n_members
        self._replay_refs: Dict[int, torch.Tensor] = {}
        self._idx_stage: Dict[int, torch.Tensor] = {}
        self._host_losses = None
        self._dev_index = self.device.index
        self._stream_raw = self.stream.cuda_stream
        self._mt_states = self._mt_indices = None  # numpy index streams, allocated by the first set_index_states

    # ------------------------------------------------------------------
    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                self._L.iql_destroy(h)
            except Exception:
                pass
            self._h = None

    def _default_hparams(self, m: int) -> HParams:
        return HParams(beta=3.0, iql_tau=0.7, discount=0.99, tau=0.005, vf_lr=3e-4, qf_lr=3e-4, actor_lr=3e-4,
                       actor_dropout=0.0, adam_beta1=0.9, adam_beta2=0.999, adam_eps=1e-8, lr_eta_min=0.0,
                       cosine_t_max=1000000, seed=m)

    def _read_paths(self) -> Dict[str, bool]:
        return {"tensor_cores": bool(self.info(_lib.INFO_TENSOR_CORE_PATH)),
                "fused_forward": bool(self.info(_lib.INFO_FUSED_FORWARD)),
                "chained_backward": bool(self.info(_lib.INFO_CHAINED_BACKWARD)),
                "chained_backward_grads": bool(self.info(_lib.INFO_CHAINED_BACKWARD_GRADS))}

    def info(self, key: int) -> int:
        out = C.c_int64(0)
        _lib.check(self._L.iql_get_info(self._h, key, C.byref(out)), self._h, "iql_get_info")
        return int(out.value)

    def keep_grads(self, on: bool = True):
        """The chained backward consumes weight gradients in its epilogue; with this on it also stores them to `grads`."""
        _lib.check(self._L.iql_set_option(self._h, _lib.OPT_KEEP_GRADS, int(bool(on))), self._h, "iql_set_option")

    def set_hparams(self, member: int, **kw):
        hp = self._hparams[member]
        for k, v in kw.items():
            if not hasattr(hp, k):
                raise ValueError(f"unknown hyper-parameter {k}")
            setattr(hp, k, v)
        _lib.check(self._L.iql_set_hparams(self._h, member, C.byref(hp)), self._h, "iql_set_hparams")

    def get_hparams(self, member: int) -> HParams:
        return self._hparams[member]

    def set_batch_sizes(self, sizes):
        """Per-member batch sizes B_m, 1 <= B_m <= batch_size (`iql_set_batch_sizes`): member m trains on rows
        [0, B_m) of every sampled batch, and index entries past B_m are ignored.  Takes effect at the next call, also
        on an already captured graph."""
        arr = np.ascontiguousarray(sizes, dtype=np.int32).reshape(-1)
        if arr.shape != (self.n_members,):
            raise ValueError(f"need one batch size per member ({self.n_members}), got {arr.shape[0]}")
        _lib.check(self._L.iql_set_batch_sizes(self._h, arr.ctypes.data), self._h, "iql_set_batch_sizes")
        self._batch_sizes = arr.tolist()

    @property
    def batch_sizes(self) -> List[int]:
        """The members' batch sizes B_m (a copy; the per-step host loop reads it without a library call)."""
        return list(self._batch_sizes)

    def set_active(self, members):
        """Train only ``members`` (indices, any non-empty subset; `iql_set_active_members`).  The others launch no work
        in later steps and keep their parameters, optimizer state, target and counters bit for bit; their loss rows
        read NaN.  Calling it again with a member resumes it where it stopped.  Re-encodes the tensor maps (host
        milliseconds) and drops the captured graphs, so call it at evaluation points rather than every step."""
        ids = np.ascontiguousarray(sorted(int(m) for m in members), dtype=np.int32)
        _lib.check(self._L.iql_set_active_members(self._h, int(ids.size), ids.ctypes.data if ids.size else None), self._h,
                   "iql_set_active_members")
        self._active = None
        self.paths = self._read_paths()

    @property
    def active(self) -> np.ndarray:
        """[n_members] bool: the members that train."""
        if getattr(self, "_active", None) is None:
            mask = np.zeros(self.n_members, dtype=np.int8)
            _lib.check(self._L.iql_get_active_members(self._h, mask.ctypes.data), self._h, "iql_get_active_members")
            self._active = mask.astype(bool)
        return self._active.copy()

    def get_counters(self, member: int) -> Counters:
        c = Counters()
        _lib.check(self._L.iql_get_counters(self._h, member, C.byref(c), None), self._h)
        return c

    def set_counters(self, member: int, **kw):
        c = self.get_counters(member)
        for k, v in kw.items():
            if not hasattr(c, k):
                raise ValueError(f"unknown counter {k}")
            setattr(c, k, int(v))
        _lib.check(self._L.iql_set_counters(self._h, member, C.byref(c)), self._h)

    # ------------------------------------------------------------------
    # zero-copy views in the reference's checkpoint layout
    # ------------------------------------------------------------------
    def _views(self, arena: torch.Tensor, member: int, nets, dropout_keys: bool, limit: Optional[int] = None):
        out: Dict[str, Dict[str, torch.Tensor]] = {}
        a_idx = linear_indices(self.n_hidden, dropout_keys)
        q_idx = linear_indices(self.n_hidden, False)
        block = arena[member]
        for t in self.tensors:
            if t.net not in nets:
                continue
            if limit is not None and t.offset >= limit:
                continue
            if t.kind == _lib.KIND_WEIGHT:
                # rows are padded to a multiple of 4 floats (16-byte aligned rows for TMA); the view hides the padding
                v = block[t.offset:t.offset + t.rows * t.ld].view(t.rows, t.ld)[:, :t.cols]
            else:
                v = block[t.offset:t.offset + t.rows]
            if t.net in (_lib.NET_Q1, _lib.NET_Q2):
                grp, key = "qf", f"q{1 if t.net == _lib.NET_Q1 else 2}.net.{q_idx[t.layer]}."
            elif t.net == _lib.NET_V:
                grp, key = "vf", f"v.net.{q_idx[t.layer]}."
            else:
                grp, key = "actor", f"net.net.{a_idx[t.layer]}."
            if t.kind == _lib.KIND_LOG_STD:
                name = "log_std"
            else:
                name = key + ("weight" if t.kind == _lib.KIND_WEIGHT else "bias")
            out.setdefault(grp, {})[name] = v
        return out

    def param_views(self, member: int = 0, dropout_keys: bool = False):
        """{"qf": {...}, "vf": {...}, "actor": {...}} views aliasing the parameter arena."""
        return self._views(self.params, member, (0, 1, 2, 3), dropout_keys)

    def moment_views(self, member: int = 0, dropout_keys: bool = False):
        return (self._views(self.exp_avg, member, (0, 1, 2, 3), dropout_keys),
                self._views(self.exp_avg_sq, member, (0, 1, 2, 3), dropout_keys))

    def grad_views(self, member: int = 0, dropout_keys: bool = False):
        return self._views(self.grads, member, (0, 1, 2, 3), dropout_keys)

    def target_views(self, member: int = 0):
        return self._views(self.target, member, (0, 1), False)["qf"]

    def load_params(self, member: int, state: Dict[str, Dict[str, "np.ndarray | torch.Tensor"]], dropout_keys=False,
                    sync_target: bool = True):
        """Copy a {"qf","vf","actor"[, "q_target"]} dict of arrays into the arena."""
        views = self.param_views(member, dropout_keys)
        for grp in ("qf", "vf", "actor"):
            for k, v in views[grp].items():
                v.copy_(torch.as_tensor(np.asarray(state[grp][k]) if not torch.is_tensor(state[grp][k]) else state[grp][k]).to(v))
        if "q_target" in state:
            for k, v in self.target_views(member).items():
                src = state["q_target"][k]
                v.copy_(torch.as_tensor(np.asarray(src) if not torch.is_tensor(src) else src).to(v))
        elif sync_target:
            self.sync_target(member)

    def sync_target(self, member: int):
        """q_target <- qf (copy.deepcopy(self.qf), iql.py:464,584,598)."""
        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream(self.device)
            _lib.check(self._L.iql_sync_target(self._h, member, cur.cuda_stream), self._h)

    # ------------------------------------------------------------------
    def bind_replay(self, member: int, rows: torch.Tensor, size: int):
        if rows.device != self.device or rows.dtype != torch.float32 or not rows.is_contiguous():
            raise ValueError("replay rows must be a contiguous float32 tensor on the engine's device")
        if rows.shape[1] != self.layout.row.row_floats:
            raise ValueError("replay rows have the wrong packed width for this engine")
        self._replay_refs[member] = rows
        _lib.check(self._L.iql_bind_replay(self._h, member, rows.data_ptr(), rows.shape[0], int(size)), self._h)

    def set_replay_size(self, member: int, size: int):
        _lib.check(self._L.iql_set_replay_size(self._h, member, int(size)), self._h)

    def _bind_index_streams(self):
        if self._mt_states is None:
            S, K, B = self.n_members, self.max_steps_per_call, self.batch_size
            self._mt_states = torch.zeros(S, _lib.MT_STATE_WORDS, dtype=torch.int32, device=self.device)
            self._mt_indices = torch.zeros(S, K, B, dtype=torch.int64, device=self.device)
            _lib.check(self._L.iql_bind_index_streams(self._h, self._mt_states.data_ptr(), self._mt_indices.data_ptr()),
                       self._h, "iql_bind_index_streams")

    def set_index_states(self, rngs):
        """Start every member's numpy index stream (``mode="numpy"`` / ``host_step(numpy_streams=True)``) where the
        ``np.random.RandomState`` ``rngs[m]`` stands: the next draws of member m are ``rngs[m].randint(0, high_m, ...)``.
        The objects are read, not kept or advanced."""
        if len(rngs) != self.n_members:
            raise ValueError(f"need one RandomState per member ({self.n_members}), got {len(rngs)}")
        rows = torch.from_numpy(index_state_rows(rngs).view(np.int32))
        self._bind_index_streams()
        with self._on_stream():
            self._mt_states.copy_(rows.to(self.device))

    def get_index_states(self, rngs):
        """Write every member's device stream back into ``rngs[m]`` (key and pos; the cached Gaussian is kept), so that
        ``rngs[m].randint`` continues where the device left off.  Waits for the engine's queued work."""
        if self._mt_states is None:
            raise RuntimeError("no index streams: call set_index_states first")
        if len(rngs) != self.n_members:
            raise ValueError(f"need one RandomState per member ({self.n_members}), got {len(rngs)}")
        with self._on_stream():
            rows = self._mt_states.cpu().numpy().view(np.uint32)
        load_index_state_rows(rngs, rows)

    def load_batch(self, member: int, batch):
        s, a, r, s2, d = self._dense_batch(batch)
        with self._on_stream() as st:
            _lib.check(self._L.iql_load_batch(self._h, member, s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(),
                                              d.data_ptr(), st.cuda_stream), self._h)
        self._keep = (s, a, r, s2, d)

    def train_on_batch(self, batch, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """S = 1 drop-in step: stage an externally sampled batch and run one update, under a single stream
        hand-over (the `ImplicitQLearning.train(batch)` path).  Returns losses [1, 1, 3] on the device."""
        s, a, r, s2, d = self._dense_batch(batch)
        if out is None:
            out = torch.empty(self.n_members, 1, 3, dtype=torch.float32, device=self.device)
        with self._on_stream() as st:
            _lib.check(self._L.iql_load_batch(self._h, 0, s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(),
                                              d.data_ptr(), st.cuda_stream), self._h, "iql_load_batch")
            _lib.check(self._L.iql_train_steps(self._h, 1, _lib.SAMPLE_PRELOADED, None, None, out.data_ptr(), None,
                                               st.cuda_stream), self._h, "iql_train_steps")
        self._keep = (s, a, r, s2, d)
        return out

    def host_step_wait(self) -> List[float]:
        """Losses of the step `host_step(..., wait=False)` launched."""
        rc = self._L.iql_host_step_wait(self._h, self._host_losses_ptr, self._stream_raw)
        if rc:
            _lib.check(rc, self._h, "iql_host_step_wait")
        return self._host_losses.tolist()

    def host_step(self, batch=None, host_indices: Optional[int] = None, wait: bool = True,
                  numpy_streams: bool = False) -> Optional[List[float]]:
        """One update step for a host-driven loop (`iql_train_host_step`): `host_indices` is the ADDRESS of S x B int64
        indices in host memory (rows of the bound replay buffers), or `batch` the five dense tensors of an externally
        built batch (S = 1), or `numpy_streams` draws each member's B_m indices on the device from its numpy index
        stream (`set_index_states`) at its replay size (`iql_train_host_step_mt19937`).  One CUDA-graph launch; returns the step's [S * 3] losses as Python floats as soon as the
        loss kernel has written them to pinned host memory -- the backward / optimizer launches of the step are still
        running then, stream-ordered before anything the caller enqueues next."""
        if self._host_losses is None:
            self._host_losses = np.zeros(3 * self.n_members, dtype=np.float32)
            self._host_losses_ptr = self._host_losses.ctypes.data
        losses = self._host_losses_ptr if wait else None
        if numpy_streams:
            _lib.call_on_device(self._dev_index, self.device, self._h, "iql_train_host_step_mt19937",
                                self._L.iql_train_host_step_mt19937, self._h, losses, self._stream_raw)
        elif host_indices is not None:
            _lib.call_on_device(self._dev_index, self.device, self._h, "iql_train_host_step", self._L.iql_train_host_step,
                                self._h, host_indices, losses, self._stream_raw)
        else:
            _lib.call_on_device(self._dev_index, self.device, self._h, "iql_train_host_step", self._load_and_step,
                                self._dense_batch(batch), losses)
        return self._host_losses.tolist() if wait else None

    def _load_and_step(self, batch, losses, cur) -> int:
        # the batch is staged on the caller's stream, the stream the step runs on: plain stream order
        s, a, r, s2, d = batch
        rc = self._L.iql_load_batch(self._h, 0, s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), cur)
        if rc:
            _lib.check(rc, self._h, "iql_load_batch")
        self._keep = batch
        return self._L.iql_train_host_step(self._h, None, losses, self._stream_raw, cur)

    def _dense(self, t: torch.Tensor) -> torch.Tensor:
        if t.device == self.device and t.dtype == torch.float32 and t.is_contiguous():
            return t
        return t.to(device=self.device, dtype=torch.float32).contiguous()

    def _dense_batch(self, batch):
        """The five tensors of an externally built batch (S = 1), dense float32 on the engine's device, shapes checked."""
        s, a, r, s2, d = [self._dense(b) for b in batch]
        B = self.batch_size
        if s.shape != (B, self.state_dim) or s2.shape != (B, self.state_dim):
            raise ValueError(f"states must be [{B}, {self.state_dim}]")
        if a.shape != (B, self.action_dim):
            raise RuntimeError("Actions shape missmatch")  # iql.py:530
        if r.numel() != B or d.numel() != B:
            raise ValueError("rewards / dones must have batch_size elements")
        return s, a, r, s2, d

    @contextlib.contextmanager
    def _on_stream(self):
        """Every C-ABI call that launches runs inside this: the engine's device is made current (the engine may
        live on cuda:N while the process's current device is another) and the engine stream is ordered after / before
        the caller's current stream on that device."""
        switch = torch.cuda.current_device() != self.device.index
        with torch.cuda.device(self.device) if switch else contextlib.nullcontext():
            cur = torch.cuda.current_stream()
            self.stream.wait_stream(cur)
            try:
                yield self.stream
            finally:
                cur.wait_stream(self.stream)

    def train_steps(self, k_steps: int, mode: str = "philox", indices: Optional[torch.Tensor] = None,
                    dropout_masks: Optional[torch.Tensor] = None, return_indices: bool = False,
                    out: Optional[torch.Tensor] = None):
        """Run K update steps for the active members; returns losses [S, K, 3]
        (value_loss, q_loss, actor_loss) on the device, asynchronously, NaN in the rows of inactive members.
        `indices` [S, K, B]: entries past a member's batch size B_m, and the rows of inactive members, are ignored;
        `return_indices` gives -1 there.  ``mode="numpy"``: member m draws ``randint(0, size_m, size=K * B_m)`` from its
        numpy index stream (`set_index_states`) on the device, step k taking draws [k B_m, (k + 1) B_m)."""
        S, B = self.n_members, self.batch_size
        smode = {"philox": _lib.SAMPLE_PHILOX, "indices": _lib.SAMPLE_INDICES, "preloaded": _lib.SAMPLE_PRELOADED,
                 "numpy": _lib.SAMPLE_MT19937}[mode]
        idx_ptr = None
        if smode == _lib.SAMPLE_INDICES:
            if indices is None:
                raise ValueError("mode='indices' needs an int64 tensor [S, K, B]")
            if indices.numel() != S * k_steps * B:
                raise ValueError("indices must have S*K*B elements")
            # stage into a persistent device buffer (one per K): the engine's CUDA graph is keyed by this pointer,
            # and host (pinned) index tensors are uploaded straight into it on the engine's stream
            stage = self._idx_stage.get(k_steps)
            if stage is None:
                stage = self._idx_stage[k_steps] = torch.empty(S * k_steps * B, dtype=torch.int64, device=self.device)
            src = indices.reshape(-1)
            if src.dtype != torch.int64:
                src = src.to(torch.int64)
            with torch.cuda.device(self.device):
                self.stream.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(self.stream):
                    stage.copy_(src, non_blocking=True)
            indices = stage
            idx_ptr = stage.data_ptr()
        mask_ptr = None
        if dropout_masks is not None:
            dropout_masks = dropout_masks.to(device=self.device, dtype=torch.uint8).contiguous()
            if dropout_masks.numel() != S * k_steps * self.n_hidden * B * self.hidden_dim:
                raise ValueError("dropout_masks must be [S, K, n_hidden, B, H]")
            mask_ptr = dropout_masks.data_ptr()
        if out is None:
            out = torch.empty(S, k_steps, 3, dtype=torch.float32, device=self.device)
        idx_out = torch.empty(S, k_steps, B, dtype=torch.int64, device=self.device) if return_indices else None
        with self._on_stream() as st:
            _lib.check(self._L.iql_train_steps(self._h, k_steps, smode, idx_ptr, mask_ptr, out.data_ptr(),
                                               idx_out.data_ptr() if idx_out is not None else None, st.cuda_stream),
                       self._h, "iql_train_steps")
        # keep argument tensors alive until the stream has consumed them
        self._keep2 = (indices, dropout_masks)
        return (out, idx_out) if return_indices else out

    def profile_step(self, reps: int = 5):
        """Per-kernel CUDA-event timing of the update step (measurement hook).  Returns a list of dicts
        {label, ms, flops, bytes} in launch order; advances the learners by `reps` steps."""
        n = C.c_int32(0)
        cap = 64
        ms = (C.c_float * cap)()
        fl = (C.c_double * cap)()
        by = (C.c_double * cap)()
        labels = C.create_string_buffer(32 * cap)
        with self._on_stream() as st:
            _lib.check(self._L.iql_profile_step(self._h, reps, cap, C.byref(n), ms, fl, by, labels, st.cuda_stream),
                       self._h, "iql_profile_step")
        out = []
        for i in range(n.value):
            out.append({"label": labels.raw[32 * i:32 * (i + 1)].split(b"\0")[0].decode(), "ms": float(ms[i]),
                        "flops": float(fl[i]), "bytes": float(by[i])})
        return out

    def last_launch_count(self) -> int:
        return int(self._L.iql_last_launch_count(self._h))

    def act(self, member: int, states: torch.Tensor, max_action: float = 1.0) -> torch.Tensor:
        """Eval-mode policy actions.  member >= 0: states [n, S] -> [n, A].  member == -1: every member acts on
        its own rows, states [n_members, n, S] -> [n_members, n, A] (one launch, vectorised envs)."""
        if member < 0:
            states = self._dense(states).view(self.n_members, -1, self.state_dim)
            n = states.shape[1]
            out = torch.empty(self.n_members, n, self.action_dim, dtype=torch.float32, device=self.device)
        else:
            states = self._dense(states).view(-1, self.state_dim)
            n = states.shape[0]
            out = torch.empty(n, self.action_dim, dtype=torch.float32, device=self.device)
        with self._on_stream() as st:
            _lib.check(self._L.iql_act(self._h, member, states.data_ptr(), n, float(max_action),
                                       out.data_ptr(), st.cuda_stream), self._h, "iql_act")
        self.act_calls += 1
        return out

    def act_host(self, member: int, state: np.ndarray, max_action: float = 1.0) -> np.ndarray:
        """One env step of ``policy.act`` (iql.py:371-379, 403-413) through the engine's act kernel: the observation
        rides in the kernel parameters, the kernel reads the policy weights straight from the parameter arena, the
        action comes back through pinned host memory the host spins on (`iql_act_host`: one launch, no copies, no
        stream synchronisation).  Returns the flat numpy action (scaled and clamped by max_action)."""
        self._act_in[:] = np.asarray(state, dtype=np.float32).reshape(-1)
        p_in, p_out, _ = self._act_ptrs
        _lib.call_on_device(self._dev_index, self.device, self._h, "iql_act_host", self._L.iql_act_host,
                            self._h, member, p_in, float(max_action), p_out, self._stream_raw)
        self.act_calls += 1
        return self._act_out.copy()

    def act_host_gaussian(self, member: int, state: np.ndarray):
        """(mean, std) of the Gaussian policy's action distribution for one host observation (`iql_act_host_gaussian`):
        mean = tanh(MLP(state)) unscaled, std = exp(clamp(log_std)); the caller samples on the host."""
        self._act_in[:] = np.asarray(state, dtype=np.float32).reshape(-1)
        p_in, p_out, p_std = self._act_ptrs
        _lib.call_on_device(self._dev_index, self.device, self._h, "iql_act_host_gaussian", self._L.iql_act_host_gaussian,
                            self._h, member, p_in, p_out, p_std, self._stream_raw)
        self.act_calls += 1
        return self._act_out.copy(), self._act_std.copy()

    # ------------------------------------------------------------------
    # online phase of an ensemble: every member's act / ring insert of one env step in one launch each
    # ------------------------------------------------------------------
    def bind_guide(self, params: Optional[torch.Tensor]):
        """Bind a [n_members, param_floats] parameter arena with this engine's layout as the members' guides
        (`iql_bind_guide`; the engine reads it zero-copy and never writes it).  None unbinds."""
        if params is None:
            _lib.check(self._L.iql_bind_guide(self._h, None), self._h, "iql_bind_guide")
            self._guide_ref = None
            return
        if params.device != self.device or params.dtype != torch.float32 or not params.is_contiguous() or \
                tuple(params.shape) != (self.n_members, self.layout.param_floats):
            raise ValueError(f"the guide arena must be a contiguous float32 [{self.n_members}, {self.layout.param_floats}] "
                             "tensor on the engine's device")
        _lib.check(self._L.iql_bind_guide(self._h, params.data_ptr()), self._h, "iql_bind_guide")
        self._guide_ref = params

    def act_members_host(self, states: np.ndarray, source, max_action: float = 1.0, out: Optional[np.ndarray] = None,
                         std: Optional[np.ndarray] = None):
        """One env step of every member's policy in one launch (`iql_act_host_members`).  ``states`` [S, state_dim],
        ``source`` [S] IQL_ACT_* codes (int) or names ("skip", "learner", "learner_dist", "guide", "learner_dropout",
        "learner_dist_dropout").  Returns ``(out, std)``: out [S, action_dim] holds the eval-mode action of "learner" /
        "guide" members, the training-mode action (actor dropout active) of "learner_dropout" members and the unscaled
        mean of "learner_dist" / "learner_dist_dropout" members, std [S, action_dim] the std of the latter (None when
        there are none).  Rows of skipped members are left as they were in ``out`` / ``std`` (NaN when the arrays are
        allocated here).  Each dropout member draws its masks at its act counter (``act_steps``), which then advances
        by one."""
        S, A = self.n_members, self.action_dim
        src = np.asarray([_lib.ACT_SOURCES[s] if isinstance(s, str) else int(s) for s in source], dtype=np.int8) \
            if not (isinstance(source, np.ndarray) and source.dtype == np.int8) else source
        if src.shape != (S,):
            raise ValueError(f"source must have one entry per member ({S})")
        st = np.ascontiguousarray(states, dtype=np.float32)
        if st.shape != (S, self.state_dim):
            raise ValueError(f"states must be [{S}, {self.state_dim}]")
        if out is None:
            out = np.full((S, A), np.nan, dtype=np.float32)
        if std is None and ((src == _lib.ACT_LEARNER_DIST) | (src == _lib.ACT_LEARNER_DIST_DROPOUT)).any():
            std = np.full((S, A), np.nan, dtype=np.float32)
        for arr in (out, std):
            if arr is not None and (arr.shape != (S, A) or arr.dtype != np.float32 or not arr.flags.c_contiguous):
                raise ValueError(f"out / std must be C-contiguous float32 [{S}, {A}]")
        _lib.call_on_device(self._dev_index, self.device, self._h, "iql_act_host_members", self._L.iql_act_host_members,
                            self._h, st.ctypes.data, src.ctypes.data, float(max_action), out.ctypes.data,
                            std.ctypes.data if std is not None else None, self._stream_raw)
        self.act_calls += 1
        return out, std

    @property
    def act_steps(self) -> np.ndarray:
        """[n_members] uint64: the act counters at which the members' next training-mode dropout acts draw their masks
        (`iql_get_act_steps`; a copy)."""
        out = np.zeros(self.n_members, dtype=np.uint64)
        _lib.check(self._L.iql_get_act_steps(self._h, out.ctypes.data), self._h, "iql_get_act_steps")
        return out

    def set_act_steps(self, steps):
        """Set every member's act counter (`iql_set_act_steps`): one non-negative integer per member."""
        arr = np.asarray(steps).reshape(-1)
        if arr.shape != (self.n_members,):
            raise ValueError(f"need one act counter per member ({self.n_members}), got {arr.shape[0]}")
        if arr.dtype.kind not in "ui" or (arr.dtype.kind == "i" and (arr < 0).any()):
            raise ValueError("act counters must be non-negative integers")
        arr = np.ascontiguousarray(arr, dtype=np.uint64)
        _lib.check(self._L.iql_set_act_steps(self._h, arr.ctypes.data), self._h, "iql_set_act_steps")

    def insert_members_host(self, states: np.ndarray, actions: np.ndarray, rewards: np.ndarray, next_states: np.ndarray,
                            dones: np.ndarray, pointers: np.ndarray):
        """`ReplayBuffer.add_transition` of every member in one launch (`iql_replay_insert_members_host`): member m's
        transition goes to row ``pointers[m]`` of the rows bound to m (``-1``: no insert).  Host arrays [S, state_dim],
        [S, action_dim], [S], [S, state_dim], [S]; the call copies them, so they may be reused when it returns.  Only
        the engine-side write happens here -- ``IQLEnsemble.add_transitions`` keeps the buffers' pointers."""
        S = self.n_members
        f = lambda x, shape: np.ascontiguousarray(x, dtype=np.float32).reshape(shape)  # noqa: E731
        s, a = f(states, (S, self.state_dim)), f(actions, (S, self.action_dim))
        r, s2, d = f(rewards, (S,)), f(next_states, (S, self.state_dim)), f(dones, (S,))
        p = np.ascontiguousarray(pointers, dtype=np.int64).reshape(S)
        _lib.call_on_device(self._dev_index, self.device, self._h, "iql_replay_insert_members_host",
                            self._L.iql_replay_insert_members_host, self._h, s.ctypes.data, a.ctypes.data, r.ctypes.data,
                            s2.ctypes.data, d.ctypes.data, p.ctypes.data, self._stream_raw)
