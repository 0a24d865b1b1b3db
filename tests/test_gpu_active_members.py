"""Members that stop training (iql_set_active_members): the problem tables, tensor maps and chain tasks are rebuilt over
the active members, so a retired member launches no CTA, keeps every bit of its state and resumes where it stopped, and
the active members compute exactly what a fresh engine holding only them computes.  Then the ASHA search of
ensemble_train_loop on the toy env, and members with their own batch sizes in that loop.

Shape of the engine tests: halfcheetah (obs 17, act 6, hidden 256, batch 256), a 4096-row synthetic buffer.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer  # noqa: E402
from jsrl_corl_b200.asha import ASHAScheduler  # noqa: E402
from jsrl_corl_b200.synthetic import synthetic_dataset  # noqa: E402

S_DIM, A_DIM, H, B, N_ROWS = 17, 6, 256, 256, 4096
_RB = []


def replay():
    if not _RB:
        rb = ReplayBuffer(S_DIM, A_DIM, N_ROWS, "cuda")
        rb.load_d4rl_dataset(synthetic_dataset(N_ROWS, S_DIM, A_DIM, 3))
        _RB.append(rb)
    return _RB[0]


def seed_of(m):
    return 900 + 11 * m


def make(members, math="tf32", step_path="auto", L=2, det=False, drop=0.0, sizes=None, max_k=8):
    """An ensemble of the given members (their seeds, their batch sizes when `sizes` is given)."""
    members = list(members)
    ens = IQLEnsemble(len(members), S_DIM, A_DIM, H, L, B, deterministic=det, actor_dropout=drop, math_mode=math,
                      max_steps_per_call=max_k, seeds=[seed_of(m) for m in members], step_path=step_path,
                      batch_sizes=None if sizes is None else [sizes[m] for m in members])
    ens.bind_replay(replay())
    return ens


def rows(ens, m, grads=True):
    e = ens.engine
    out = [e.params[m].clone(), e.exp_avg[m].clone(), e.exp_avg_sq[m].clone(), e.target[m].clone()]
    if grads:
        out.append(e.grads[m].clone())
    c = e.get_counters(m)
    return out, tuple(getattr(c, f) for f, _ in type(c)._fields_)


def same_rows(a, b):
    return all(torch.equal(x, y) for x, y in zip(a[0], b[0])) and a[1] == b[1]


def test_retired_members_are_frozen_and_report_nan():
    ens = make(range(12))
    ens.train_steps(8)
    retired = [1, 4, 7, 10]
    ens.retire(retired)
    assert ens.active.tolist() == [m not in retired for m in range(12)]
    torch.cuda.synchronize()
    before = {m: rows(ens, m) for m in range(12)}
    losses, idx = ens.engine.train_steps(8, return_indices=True)
    torch.cuda.synchronize()
    losses, idx = losses.cpu(), idx.cpu()
    for m in range(12):
        if m in retired:
            assert same_rows(rows(ens, m), before[m]), m
            assert torch.isnan(losses[m]).all() and (idx[m] == -1).all()
        else:
            assert not torch.equal(ens.engine.params[m], before[m][0][0]) and torch.isfinite(losses[m]).all()
            assert (idx[m] >= 0).all() and rows(ens, m)[1][4] == before[m][1][4] + 8  # total_it
    # the host-step path: NaN losses, counters untouched
    lo = ens.train_step_logged()
    assert np.isnan(lo[retired]).all() and np.isfinite(np.delete(lo, retired, axis=0)).all()
    torch.cuda.synchronize()
    assert all(same_rows(rows(ens, m), before[m]) for m in retired)
    # a retired member still acts, checkpoints and syncs its target
    st = np.random.RandomState(0).standard_normal((12, S_DIM)).astype(np.float32)
    out, _ = ens.act(st, ["learner"] * 12)
    assert np.isfinite(out).all()
    assert ens.member_state_dict(4)["total_it"] == before[4][1][4]


# (id, math, step_path, n_hidden, deterministic, dropout, batch sizes)
MATRIX = [
    ("fp32", "fp32", "auto", 2, False, 0.0, None),
    ("tf32-phases", "tf32", "phases", 2, False, 0.0, None),
    ("tf32-chain_grads", "tf32", "chain_grads", 2, False, 0.0, None),
    ("tf32-chain", "tf32", "chain", 2, False, 0.0, None),
    ("tf32-3x256-det", "tf32", "auto", 3, True, 0.0, None),
    ("tf32-dropout", "tf32", "auto", 2, False, 0.25, None),
    ("tf32-mixed-B", "tf32", "auto", 2, False, 0.0, (1, 7, 33, 128, 200, 256, 256, 64, 17, 256, 100, 250)),
]


@pytest.mark.parametrize("keep", [(0, 2, 3, 5, 6, 8, 9, 11), (1, 6, 10)], ids=["8of12", "3of12"])
@pytest.mark.parametrize("row", MATRIX, ids=[r[0] for r in MATRIX])
def test_compaction_equals_a_fresh_engine_of_the_active_members(row, keep, monkeypatch):
    _, math, step_path, L, det, drop, sizes = row
    big = make(range(12), math, step_path, L, det, drop, sizes)
    big.retire([m for m in range(12) if m not in keep])
    if len(keep) <= 4:  # the 12-member engine chose lb_splits = 1 at creation; so must the fresh one
        monkeypatch.setenv("IQL_B200_NO_LASTBWD_SPLIT", "1")
    fresh = make(keep, math, step_path, L, det, drop, sizes)
    monkeypatch.delenv("IQL_B200_NO_LASTBWD_SPLIT", raising=False)
    assert big.engine.paths == fresh.engine.paths
    for call in range(2):
        if drop:
            g = torch.Generator().manual_seed(call)
            masks = (torch.rand(12, 8, L, B, H, generator=g) >= drop).to(torch.uint8)
            lb = big.engine.train_steps(8, dropout_masks=masks)
            lf = fresh.engine.train_steps(8, dropout_masks=masks[list(keep)].contiguous())
        else:
            lb, lf = big.train_steps(8), fresh.train_steps(8)
        torch.cuda.synchronize()
        assert torch.equal(lb[list(keep)], lf), call
    for i, m in enumerate(keep):
        assert same_rows(rows(big, m, grads=False), rows(fresh, i, grads=False)), m


def test_pause_and_resume_continue_as_if_no_time_had_passed():
    ref, run = make(range(4), max_k=4), make(range(4), max_k=4)
    ref.train_steps(4)
    ref.train_steps(4)
    torch.cuda.synchronize()
    want = rows(ref, 2)
    run.train_steps(4)
    run.retire([2])
    run.train_steps(4)
    run.train_steps(4)
    run.resume([2])
    assert run.active.all()
    run.train_steps(4)
    torch.cuda.synchronize()
    assert same_rows(rows(run, 2), want)


def test_active_set_changes_between_graph_replays_match_the_eager_run(monkeypatch):
    graphs = make(range(6))
    monkeypatch.setenv("IQL_B200_GRAPHS", "0")
    eager = make(range(6))
    monkeypatch.delenv("IQL_B200_GRAPHS")
    for ens in (graphs, eager):
        ens.train_steps(4)
        ens.engine.set_active([0, 3, 4])
        ens.train_steps(4)
        ens.engine.set_active([1, 2, 3, 4, 5])
        ens.train_steps(4)
        ens.engine.set_active(range(6))
        ens.train_steps(4)
    torch.cuda.synchronize()
    for m in range(6):
        assert same_rows(rows(graphs, m, grads=False), rows(eager, m, grads=False)), m


def test_host_steps_with_retired_members_equal_one_k_step_call_and_ignore_their_indices():
    K, retired = 4, [0, 5]
    rng = np.random.RandomState(4)
    idx = rng.randint(0, N_ROWS, size=(6, K, B)).astype(np.int64)
    junk = idx.copy()
    junk[0] = -1
    junk[5] = 1 << 40
    host, call, clean = make(range(6)), make(range(6)), make(range(6))
    for ens in (host, call, clean):
        ens.retire(retired)
    host_lo = np.stack([host.train_step_logged(junk[:, k]) for k in range(K)], axis=1)
    call_lo = call.train_steps(K, mode="indices", indices=torch.from_numpy(junk)).cpu().numpy()
    clean.train_steps(K, mode="indices", indices=torch.from_numpy(idx))
    torch.cuda.synchronize()
    assert np.array_equal(host_lo, call_lo, equal_nan=True) and np.isnan(call_lo[retired]).all()
    for m in range(6):
        assert same_rows(rows(host, m, grads=False), rows(call, m, grads=False)), m
        assert same_rows(rows(clean, m, grads=False), rows(call, m, grads=False)), m


def test_paths_follow_the_active_count():
    ens = make(range(12), max_k=1)
    assert ens.engine.paths["chained_backward_grads"]  # 2x256 auto: chained backward from 8 members on
    for n, chained in ((7, False), (8, True), (1, False), (12, True)):
        ens.engine.set_active(range(n))
        assert ens.engine.paths["chained_backward_grads"] is chained, n
        labels = [r["label"] for r in ens.engine.profile_step(reps=1)]
        assert ("bwd_chain_grads" in labels) is chained, (n, labels)


# ---------------------------------------------------------------------------
# ASHA in ensemble_train_loop (toy env, batch 32: the FP32 kernels)
# ---------------------------------------------------------------------------
class PointEnv:
    """gym-style toy env: 3-dim state (x, y, t/T), 2-dim action, reward = -|pos|, T = 20 steps."""
    T = 20

    def __init__(self, seed=0):
        self.rng = np.random.RandomState(seed)
        self.spec = type("Spec", (), {"id": "Point-v0"})()

    def seed(self, s):
        self.rng = np.random.RandomState(s)

    def reset(self):
        self.pos = self.rng.uniform(-1, 1, 2)
        self.t = 0
        return self._obs()

    def _obs(self):
        return np.array([self.pos[0], self.pos[1], self.t / self.T], dtype=np.float32)

    def step(self, action):
        self.pos = np.clip(self.pos + 0.1 * np.asarray(action, dtype=np.float64).reshape(-1)[:2], -2, 2)
        self.t += 1
        return self._obs(), float(-np.linalg.norm(self.pos)), self.t >= self.T, {}


OFF, ON, EVAL = 60, 80, 20


def _configs(tmp, tag, sizes, members=None):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig

    members = range(len(sizes)) if members is None else members
    return [JsrlTrainConfig(device="cuda", env="Point-v0", seed=10 + 7 * m, eval_freq=EVAL, n_episodes=2,
                            offline_iterations=OFF, online_iterations=ON, batch_size=sizes[m], n_curriculum_stages=1 + m % 3,
                            rolling_mean_n=1, tolerance=0.3, horizon_fn="time_step", online_buffer_size=100,
                            checkpoints_path=os.path.join(str(tmp), f"{tag}{m}"), beta=1.0 + m, qf_lr=3e-4 * (1 + m % 2))
            for m in members]


def _offline_buffer():
    rng = np.random.RandomState(1)
    n = 500
    data = {"observations": rng.uniform(-1, 1, (n, 3)).astype(np.float32), "actions": rng.uniform(-1, 1, (n, 2)).astype(np.float32),
            "rewards": rng.uniform(-1, 0, n).astype(np.float32), "next_observations": rng.uniform(-1, 1, (n, 3)).astype(np.float32),
            "terminals": np.zeros(n, bool)}
    rb = ReplayBuffer(3, 2, n, "cuda")
    rb.load_d4rl_dataset(data)
    return rb


def _loop(configs, members, scheduler=None, mixed=False):
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    logs = {i: [] for i in range(len(configs))}
    learner, cfgs, hist = ensemble_train_loop(configs, [PointEnv(100 + m) for m in members], [PointEnv(200 + m) for m in members],
                                              _offline_buffer(), 3, 2, 1.0, max_steps=PointEnv.T,
                                              log=lambda i, d, step: logs[i].append((step, d)), scheduler=scheduler,
                                              mixed_batch_sizes=mixed)
    torch.cuda.synchronize()
    return learner, hist, logs


def _same(a, b):
    if torch.is_tensor(a) or torch.is_tensor(b):
        return torch.is_tensor(a) and torch.is_tensor(b) and a.shape == b.shape and \
            bool(torch.equal(torch.nan_to_num(a, nan=1.5e38), torch.nan_to_num(b, nan=1.5e38)))
    if isinstance(a, dict):
        return isinstance(b, dict) and list(a) == list(b) and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return repr(a) == repr(b)


def test_asha_loop_stops_members_and_leaves_the_others_untouched(tmp_path):
    S = 6
    sizes = [32] * S
    base_cfgs = _configs(tmp_path, "base", sizes)  # (the config nests its checkpoint directory under its run name)
    base_l, base_h, base_logs = _loop(base_cfgs, range(S))
    sched = ASHAScheduler(max_t=100, grace_period=1, reduction_factor=2)  # rungs at 1, 2, 4 of the 7 evaluations
    l, h, logs = _loop(_configs(tmp_path, "asha", sizes), range(S), sched)
    stopped = dict(sched.stopped)
    assert stopped and 0 not in stopped  # the rule stops some members; the first to reach every rung runs on
    for m in range(S):
        if m not in stopped:  # never stopped: bit for bit the run without a scheduler
            assert _same(h[m], base_h[m]) and _same(logs[m], base_logs[m]), m
            assert _same(l.member_state_dict(m), base_l.member_state_dict(m)), m
            continue
        n, total_it = stopped[m]
        assert len(h[m]) == n and _same(h[m], base_h[m][:n]), m  # the history ends at the stop
        assert logs[m][-1][0] == total_it and _same(logs[m], base_logs[m][:len(logs[m])]), m
        # frozen from the stop on: the state is the checkpoint the stopping evaluation wrote
        t_stop = h[m][-1]["t"]
        ck = torch.load(os.path.join(base_cfgs[m].checkpoints_path, f"checkpoint_{t_stop}.pt"), weights_only=False)
        ens = l if t_stop >= OFF else l.guide
        assert _same(ens.member_state_dict(m), ck), m
        assert not l.active[m]
    # the recorded scores replayed through the rule on the CPU give the same decisions
    replay_s = ASHAScheduler(max_t=100, grace_period=1, reduction_factor=2)
    n_rep = [0] * S
    for t in sorted({e["t"] for hm in h for e in hm}):
        for m in range(S):
            for e in h[m]:
                if e["t"] == t:
                    n_rep[m] += 1
                    replay_s.on_result(m, n_rep[m], e["eval/score"], None)
    assert {m: v[0] for m, v in replay_s.stopped.items()} == {m: v[0] for m, v in stopped.items()}


def test_mixed_batch_sizes_open_each_gate_and_match_single_member_runs(tmp_path):
    sizes = [16, 32, 48]
    _, h, logs = _loop(_configs(tmp_path, "mix", sizes), range(3), mixed=True)
    for m, bm in enumerate(sizes):
        first = next(d for _, d in logs[m] if "offline_iter" in d)
        assert first["offline_iter"] == bm  # train_loop's gate `t >= batch_size`, per member
        one_l, one_h, one_logs = _loop(_configs(tmp_path, f"one{m}_", sizes, [m]), [m])
        assert len(one_logs[0]) == len(logs[m]) and [s for s, _ in one_logs[0]] == [s for s, _ in logs[m]]
        for (_, a), (_, b) in zip(one_logs[0], logs[m]):
            for k in ("value_loss", "q_loss", "actor_loss"):
                if k in a:
                    assert abs(a[k] - b[k]) <= 1e-4 * max(1.0, abs(a[k])), (m, k, a, b)
        assert [e["t"] for e in one_h[0]] == [e["t"] for e in h[m]]
