"""The online phase of an ensemble: one act launch (learner / Gaussian distribution / guide / skip per member), one
ring-insert launch and one logged update per env step for all members, and the vectorised JSRL loop built on them.

Every check here is bit for bit: the batched act runs the single-observation act body unchanged, the batched insert
writes the rows add_transition writes, and each member of the loop is the single-learner JSRL run of its config."""
import copy
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer  # noqa: E402
from jsrl_corl_b200 import _lib  # noqa: E402
from jsrl_corl_b200.synthetic import synthetic_dataset  # noqa: E402

SKIP, LEARNER, DIST, GUIDE = _lib.ACT_SKIP, _lib.ACT_LEARNER, _lib.ACT_LEARNER_DIST, _lib.ACT_GUIDE


def _ensemble(S, Sd, A, L, det, seed0, B=256):
    return IQLEnsemble(S, Sd, A, 256, L, B, deterministic=det, seeds=[seed0 + m for m in range(S)], max_steps_per_call=4)


# ---------------------------------------------------------------------------
# 1. batched act == per-member act
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("S,Sd,A,L,det", [(1, 17, 6, 2, False), (5, 17, 6, 2, True), (64, 17, 6, 2, False),
                                         (5, 29, 8, 3, False), (64, 29, 8, 3, True), (2, 45, 24, 2, False)])
def test_batched_act_equals_per_member_act(S, Sd, A, L, det):
    import contextlib
    import io

    learner = _ensemble(S, Sd, A, L, det, 0)
    guide = _ensemble(S, Sd, A, L, det, 1000)
    rb = ReplayBuffer(Sd, A, 4096, "cuda")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(synthetic_dataset(4096, Sd, A, 0))
    learner.bind_replay(rb)
    rng = np.random.RandomState(S * 100 + Sd)
    for _ in range(3):  # the weights move; the last step is still in flight when the act call is issued
        learner.train_step_logged(rng.randint(0, 4096, size=(S, 256)))
    learner.set_guide(guide)
    codes = [SKIP, LEARNER, GUIDE] + ([] if det else [DIST])
    src = rng.choice(codes, size=S).astype(np.int8)
    if S > 1:
        src[:len(codes)] = codes[:S]  # every code present
    states = rng.randn(S, Sd).astype(np.float32)
    out = np.full((S, A), np.nan, np.float32)
    std = np.full((S, A), np.nan, np.float32)
    learner.act(states, src, 0.8, out=out, std=None if det else std)
    for m in range(S):
        if src[m] == SKIP:
            assert np.isnan(out[m]).all() and np.isnan(std[m]).all()
        elif src[m] == LEARNER:
            assert np.array_equal(out[m], learner.engine.act_host(m, states[m], 0.8)), m
        elif src[m] == GUIDE:
            assert np.array_equal(out[m], guide.engine.act_host(m, states[m], 0.8)), m
        else:
            mean, sd = learner.engine.act_host_gaussian(m, states[m])
            assert np.array_equal(out[m], mean) and np.array_equal(std[m], sd), m
        if src[m] != DIST:
            assert np.isnan(std[m]).all()
    # refused: guide code with no guide, distribution code on a deterministic policy, unknown codes
    learner.set_guide(None)
    with pytest.raises(ValueError, match="no guide"):
        learner.act(states, np.full(S, GUIDE, np.int8))
    if det:
        with pytest.raises(ValueError, match="deterministic"):
            learner.act(states, np.full(S, DIST, np.int8))
    with pytest.raises(ValueError, match="unknown source"):
        learner.act(states, np.full(S, 7, np.int8))
    with pytest.raises(ValueError):  # a guide of another shape
        learner.set_guide(_ensemble(S, Sd, A + 1, L, det, 0))
    # all skipped: nothing launched, nothing written
    out2 = np.full((S, A), np.nan, np.float32)
    learner.act(states, np.zeros(S, np.int8), out=out2)
    assert np.isnan(out2).all()


# ---------------------------------------------------------------------------
# 2. batched insert == per-member add_transition
# ---------------------------------------------------------------------------
def _insert_run(Sd, A, caps, calls, seed):
    S = len(caps)
    ens = IQLEnsemble(S, Sd, A, 256, 2, 32, init=False)
    mine = [ReplayBuffer(Sd, A, c, "cuda") for c in caps]
    ref = [ReplayBuffer(Sd, A, c, "cuda") for c in caps]
    ens.bind_replay(mine)
    rng = np.random.RandomState(seed)
    for i in range(calls):
        s, a = rng.randn(S, Sd).astype(np.float32), rng.randn(S, A).astype(np.float32)
        r, s2 = rng.randn(S).astype(np.float32), rng.randn(S, Sd).astype(np.float32)
        d = (rng.rand(S) < 0.3).astype(np.float32)
        mask = rng.rand(S) < 0.7
        ens.add_transitions(s, a, r, s2, d, mask=mask)
        for m in np.flatnonzero(mask):
            ref[m].add_transition(s[m], a[m], float(r[m]), s2[m], bool(d[m]))
    torch.cuda.synchronize()
    for m in range(S):
        assert torch.equal(mine[m].rows, ref[m].rows), m  # every float of every row, padding included
        assert (mine[m]._pointer, mine[m]._size) == (ref[m]._pointer, ref[m]._size)
    return ens, mine


@pytest.mark.parametrize("Sd,A", [(17, 6), (45, 24)])
def test_batched_insert_equals_add_transition(Sd, A):
    caps = [7, 10, 3, 16, 5]
    ens, mine = _insert_run(Sd, A, caps, 40, 0)  # more inserts than capacity: every ring wraps
    assert all(rb._size == rb._buffer_size for rb in mine)
    S = len(caps)
    z = np.zeros((S, Sd), np.float32)
    za, zr = np.zeros((S, A), np.float32), np.zeros(S, np.float32)
    # refused: a pointer outside the ring, an unbound member, two members sharing one ring
    p = np.full(S, -1, np.int64)
    p[2] = caps[2]
    with pytest.raises(ValueError, match="outside"):
        ens.engine.insert_members_host(z, za, zr, z, zr, p)
    fresh = IQLEnsemble(S, Sd, A, 256, 2, 32, init=False)
    with pytest.raises(ValueError, match="no replay binding"):
        fresh.engine.insert_members_host(z, za, zr, z, zr, np.zeros(S, np.int64))
    shared = ReplayBuffer(Sd, A, 8, "cuda")
    fresh.bind_replay([shared] * S)
    with pytest.raises(ValueError, match="share one ring"):
        fresh.add_transitions(z, za, zr, z, zr, mask=[True, True, False, False, False])
    assert shared._pointer == 0
    fresh.add_transitions(z, za, zr, z, zr, mask=[False, True, False, False, False])  # one of them at a time is fine
    assert shared._pointer == 1
    # a buffer loaded to the brim raises add_transition's IndexError, before anything is written
    full = ReplayBuffer(Sd, A, 4, "cuda")
    full.load_d4rl_dataset(synthetic_dataset(4, Sd, A, 1))
    fresh.bind_replay([full] + [ReplayBuffer(Sd, A, 4, "cuda") for _ in range(S - 1)])
    with pytest.raises(IndexError):
        fresh.add_transitions(z, za, zr, z, zr)
    assert all(rb._pointer == 0 for rb in fresh._buffers[1:])


def test_back_to_back_inserts_without_host_sync():
    """1,000 calls with no synchronisation in between: the two pinned input slots are reused every other call, so a
    missing or broken consumed-flag guard would let a call overwrite rows a queued launch has not read yet."""
    _insert_run(17, 6, [300, 1000, 257, 64], 1000, 3)


# ---------------------------------------------------------------------------
# 3 + 4. the vectorised JSRL loop
# ---------------------------------------------------------------------------
class PointEnv:
    """gym-style (4-tuple) toy env: 3-dim state (x, y, t/T), 2-dim action, reward = -|pos|, T = 20 steps."""
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


OFF, ON, B, EVAL = 40, 160, 32, 50


def _member_configs(det, tmp):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig

    out = []
    for m, (beta, tol, stages, noise) in enumerate([(3.0, 0.5, 3, 0.03), (1.0, 0.05, 1, 0.3), (10.0, 0.2, 2, 0.0),
                                                    (0.5, 1.0, 3, 0.1)]):
        out.append(JsrlTrainConfig(device="cuda", env="Point-v0", seed=10 + 7 * m, eval_freq=EVAL, n_episodes=2,
                                   offline_iterations=OFF, online_iterations=ON, batch_size=B, n_curriculum_stages=stages,
                                   rolling_mean_n=1, tolerance=tol, horizon_fn="time_step", online_buffer_size=100,
                                   checkpoints_path=str(tmp / f"m{m}"), iql_deterministic=det, beta=beta,
                                   expl_noise=noise, noise_clip=0.5 if m % 2 == 0 else 0.05, qf_lr=3e-4 * (1 + m)))
    return out


def _offline_buffer():
    rng = np.random.RandomState(1)
    n = 500
    data = {"observations": rng.uniform(-1, 1, (n, 3)).astype(np.float32), "actions": rng.uniform(-1, 1, (n, 2)).astype(np.float32),
            "rewards": rng.uniform(-1, 0, n).astype(np.float32), "next_observations": rng.uniform(-1, 1, (n, 3)).astype(np.float32),
            "terminals": np.zeros(n, bool)}
    rb = ReplayBuffer(3, 2, n, "cuda")
    rb.load_d4rl_dataset(data)
    return rb


def _run(configs, member_ids, rb, record=None):
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    logs = {m: [] for m in range(len(configs))}
    envs = [PointEnv(100 + i) for i in member_ids]
    eval_envs = [PointEnv(200 + i) for i in member_ids]
    learner, cfgs, hist = ensemble_train_loop(configs, envs, eval_envs, rb, 3, 2, 1.0, max_steps=PointEnv.T,
                                              log=lambda m, d, step: logs[m].append((step, d)))
    torch.cuda.synchronize()
    return learner, cfgs, hist, logs


def _same(a, b):
    """Exact equality of nested logs / checkpoints: tensors element for element, NaN equal to NaN."""
    if torch.is_tensor(a) or torch.is_tensor(b):
        return torch.is_tensor(a) and torch.is_tensor(b) and a.dtype == b.dtype and a.shape == b.shape and \
            bool(torch.equal(a, b) or torch.equal(torch.nan_to_num(a, nan=1.5e38), torch.nan_to_num(b, nan=1.5e38)))
    if isinstance(a, dict):
        return isinstance(b, dict) and list(a) == list(b) and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return type(a) is type(b) and len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return repr(a) == repr(b)


@pytest.fixture(scope="module", params=[False, True], ids=["gaussian", "deterministic"])
def loop_runs(request, tmp_path_factory):
    det = request.param
    tmp = tmp_path_factory.mktemp("det" if det else "gauss")
    rb = _offline_buffer()
    rec = {"insert": [], "step": [], "offline": []}
    orig_add, orig_step, orig_k = IQLEnsemble.add_transitions, IQLEnsemble.train_step_logged, IQLEnsemble.train_steps

    def add(self, *a, **k):
        rec["insert"].append([np.array(x, copy=True) for x in a])
        return orig_add(self, *a, **k)

    def step(self, indices=None):
        rec["step"].append(np.array(indices, copy=True))
        return orig_step(self, indices)

    def ksteps(self, k, **kw):
        rec["offline"].append(kw["indices"].numpy().copy())
        return orig_k(self, k, **kw)

    IQLEnsemble.add_transitions, IQLEnsemble.train_step_logged, IQLEnsemble.train_steps = add, step, ksteps
    try:
        ens_cfgs = _member_configs(det, tmp / "ens")
        init_cfgs = copy.deepcopy(ens_cfgs)
        ens = _run(ens_cfgs, range(4), rb)
    finally:
        IQLEnsemble.add_transitions, IQLEnsemble.train_step_logged, IQLEnsemble.train_steps = orig_add, orig_step, orig_k
    singles = []
    for m in range(4):
        c = copy.deepcopy(init_cfgs[m])
        c.checkpoints_path = os.path.join(str(tmp / "single"), os.path.basename(c.checkpoints_path))
        singles.append(_run([c], [m], rb))
    return dict(det=det, rb=rb, ens=ens, singles=singles, rec=rec, init_cfgs=init_cfgs)


def test_members_are_independent(loop_runs):
    learner, cfgs, hist, logs = loop_runs["ens"]
    for m in range(4):
        l1, c1, h1, g1 = loop_runs["singles"][m]
        assert _same(logs[m], g1[0]), m  # per-step losses, episode logs, eval logs, steps
        assert _same(hist[m], h1[0]), m
        for f in ("curriculum_stage_idx", "curriculum_stage", "best_eval_score", "agent_type_stage", "mean_horizon_reached"):
            assert _same(getattr(cfgs[m], f), getattr(c1[0], f)), (m, f)
        assert _same(list(cfgs[m].all_curriculum_stages), list(c1[0].all_curriculum_stages))
        assert torch.equal(learner._buffers[m].rows, l1._buffers[0].rows)
        assert learner._buffers[m]._pointer == l1._buffers[0]._pointer
        for arena in ("params", "exp_avg", "exp_avg_sq", "target"):
            assert torch.equal(getattr(learner.engine, arena)[m], getattr(l1.engine, arena)[0]), (m, arena)
            assert torch.equal(getattr(learner.guide.engine, arena)[m], getattr(l1.guide.engine, arena)[0]), (m, arena)
        names = sorted(os.listdir(cfgs[m].checkpoints_path))
        assert names == sorted(os.listdir(c1[0].checkpoints_path)) and len(names) == (OFF + ON) // EVAL
        for n in names:
            a = torch.load(os.path.join(cfgs[m].checkpoints_path, n), map_location="cpu")
            b = torch.load(os.path.join(c1[0].checkpoints_path, n), map_location="cpu")
            assert _same(a, b), (m, n)


def test_each_member_is_the_single_learner_jsrl_step(loop_runs):
    """Member m's recorded transitions and indices, replayed through ReplayBuffer.add_transition and an
    ImplicitQLearning trained on the same indices, give the same losses and parameters bit for bit."""
    import jsrl_corl_b200 as J
    from jsrl_corl_b200.jsrl_w_iql import member_networks

    learner, cfgs, hist, logs = loop_runs["ens"]
    rec, rb, det = loop_runs["rec"], loop_runs["rb"], loop_runs["det"]
    offline_idx = np.concatenate(rec["offline"], axis=1)  # [S, OFF - B, B]
    assert offline_idx.shape[1] == OFF - B
    for m in range(4):
        c = loop_runs["init_cfgs"][m]
        (q, v, actor), (q2, v2, actor2) = member_networks(c, 3, 2, 1.0)

        def trainer(q, v, actor, max_steps):
            return J.ImplicitQLearning(1.0, actor, torch.optim.Adam(actor.parameters(), lr=c.actor_lr), q,
                                       torch.optim.Adam(q.parameters(), lr=c.qf_lr), v, torch.optim.Adam(v.parameters(), lr=c.vf_lr),
                                       beta=c.beta, iql_tau=c.iql_tau, discount=c.discount, tau=c.tau, max_steps=max_steps,
                                       device="cuda")
        off_tr = trainer(q, v, actor, OFF)
        np.random.seed(c.seed)  # ReplayBuffer.sample draws from the global stream what the loop drew from RandomState(seed)
        off_logs = [d for _, d in logs[m] if "offline_iter" in d]
        assert len(off_logs) == OFF - B  # the update gate uses the global t
        for k, d in enumerate(off_logs):
            got = off_tr.train(rb.sample(B))
            assert np.array_equal(rb._last_indices, offline_idx[m, k])
            assert all(got[key] == d[key] for key in ("value_loss", "q_loss", "actor_loss")), (m, k)
        on_tr = trainer(q2, v2, actor2, None)
        if c.n_curriculum_stages == 1:
            on_tr.partial_load_state_dict(off_tr.state_dict())
        on_tr.total_it = OFF
        ring = J.ReplayBuffer(3, 2, c.online_buffer_size, "cuda")
        on_logs = [d for _, d in logs[m] if "online_iter" in d]
        assert len(on_logs) == ON
        for k in range(ON):
            s, a, r, s2, d = [x[m] for x in rec["insert"][k][:5]]
            ring.add_transition(s, a, float(r), s2, bool(d))
            got = on_tr.train(ring.sample(B))
            assert np.array_equal(ring._last_indices, rec["step"][k][m])
            assert all(got[key] == on_logs[k][key] for key in ("value_loss", "q_loss", "actor_loss")), (m, k)
        torch.cuda.synchronize()
        assert on_tr.total_it == OFF + ON and on_tr.actor_lr_schedule is None
        assert learner.engine.get_hparams(m).cosine_t_max == 0 and learner.engine.get_counters(m).total_it == OFF + ON
        views = learner.engine.param_views(m)
        for grp, mod in (("qf", on_tr.qf), ("vf", on_tr.vf), ("actor", on_tr.actor)):
            for name, t in mod.state_dict().items():
                assert torch.equal(views[grp][name], t), (m, grp, name)
        assert torch.equal(ring.rows, learner._buffers[m].rows)
        # structure of train_loop: evaluation times, curriculum, episode logs, checkpoints
        assert [h["t"] for h in hist[m]] == [49, 99, 149, 199]
        assert all("eval/jsrl/curriculum_stage" in h for h in hist[m] if h["t"] >= OFF)
        assert len(cfgs[m].all_curriculum_stages) == c.n_curriculum_stages
        episodes = [d for d in on_logs if "train/episode_length" in d]
        assert len(episodes) == ON // PointEnv.T and all(d["train/episode_length"] == PointEnv.T for d in episodes)
        sd = torch.load(os.path.join(cfgs[m].checkpoints_path, "checkpoint_199.pt"), map_location="cuda")
        assert sd["total_it"] == OFF + ON and sd["actor_lr_schedule"] == {}
        sd0 = torch.load(os.path.join(cfgs[m].checkpoints_path, "checkpoint_49.pt"), map_location="cuda")
        assert sd0["total_it"] == 49 + 1  # online steps t = 40..49 continue the offline count
