"""The learner's training-mode act with actor dropout (iql_act_host_members codes 4 / 5) and the ensemble loop that uses it
(ensemble_train_loop(..., philox_act_dropout=True)).

Kernel checks: p = 0 is codes 1 / 2 bit for bit; p > 0 matches a float64 forward with the oracle's act masks; the act
counter is the only state the masks depend on besides the key; the masks the kernel draws, read back exactly through a
probe actor, are the oracle's and keep 1 - p of the units.  Loop checks: as in test_gpu_ensemble_online, each member is
its single-config run and replays through ImplicitQLearning bit for bit, now with dropout actors."""
import copy
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer  # noqa: E402
from jsrl_corl_b200 import _lib  # noqa: E402
from jsrl_corl_b200.synthetic import synthetic_dataset  # noqa: E402
from act_mask_oracle import philox_act_dropout_mask  # noqa: E402
from oracle.philox import philox_dropout_mask  # noqa: E402
from test_gpu_ensemble_online import B, EVAL, OFF, ON, PointEnv, _member_configs, _offline_buffer, _same  # noqa: E402

SKIP, LEARNER, DIST, GUIDE = _lib.ACT_SKIP, _lib.ACT_LEARNER, _lib.ACT_LEARNER_DIST, _lib.ACT_GUIDE
DROP, DIST_DROP = _lib.ACT_LEARNER_DROPOUT, _lib.ACT_LEARNER_DIST_DROPOUT


def _ensemble(S, Sd, A, L, det, p, seeds, **kw):
    return IQLEnsemble(S, Sd, A, 256, L, 256, deterministic=det, actor_dropout=p, math_mode="fp32", seeds=seeds, **kw)


def _actor_tensors(eng, m):
    """Member m's actor as float64 numpy arrays: weights [L+1], biases [L+1], log_std (None: deterministic)."""
    P = eng.params[m].detach().double().cpu()
    L = eng.n_hidden
    W, b, log_std = [None] * (L + 1), [None] * (L + 1), None
    for t in eng.tensors:
        if t.net != _lib.NET_ACTOR:
            continue
        if t.kind == _lib.KIND_WEIGHT:
            W[t.layer] = P[t.offset:t.offset + t.rows * t.ld].view(t.rows, t.ld)[:, :t.cols].numpy()
        elif t.kind == _lib.KIND_BIAS:
            b[t.layer] = P[t.offset:t.offset + t.rows].numpy()
        else:
            log_std = P[t.offset:t.offset + t.rows].numpy()
    return W, b, log_std


def _set_actor(eng, m, layer, kind, value):
    for t in eng.tensors:
        if t.net == _lib.NET_ACTOR and t.layer == layer and t.kind == kind:
            block = eng.params[m]
            if kind == _lib.KIND_WEIGHT:
                block[t.offset:t.offset + t.rows * t.ld].view(t.rows, t.ld)[:, :t.cols] = torch.as_tensor(value, dtype=torch.float32)
            else:
                block[t.offset:t.offset + t.rows] = torch.as_tensor(value, dtype=torch.float32)
            return
    raise KeyError((layer, kind))


def _forward64(eng, m, state, seed, step, p, code, max_action):
    """The float64 forward of code 4 (action) or 5 (mean, std) with the oracle's act masks at counter `step`."""
    W, b, log_std = _actor_tensors(eng, m)
    L = eng.n_hidden
    h = np.asarray(state, np.float64)
    for l in range(L):
        keep = philox_act_dropout_mask(seed, step, l, eng.hidden_dim, p).astype(np.float64)
        h = np.maximum(W[l] @ h + b[l], 0.0) * keep / (1.0 - p)
    y = np.tanh(W[L] @ h + b[L])
    if code == DIST_DROP:
        return y, np.exp(np.clip(log_std, -20.0, 2.0))
    return np.clip(max_action * y, -max_action, max_action), None


def _replay(S, Sd, A):
    import contextlib
    import io

    rb = ReplayBuffer(Sd, A, 4096, "cuda")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(synthetic_dataset(4096, Sd, A, 0))
    return rb


# ---------------------------------------------------------------------------
# 1. p = 0: the dropout codes are the eval / distribution codes
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("det", [False, True])
def test_p0_is_codes_1_and_2_bit_for_bit(det):
    S, Sd, A = 4, 17, 6
    ens = _ensemble(S, Sd, A, 2, det, 0.0, [3, 4, 5, 6])
    states = np.random.RandomState(0).randn(S, Sd).astype(np.float32)
    pairs = [(LEARNER, DROP)] + ([] if det else [(DIST, DIST_DROP)])
    for k, (plain, drop) in enumerate(pairs):
        ref, ref_std = ens.act(states, np.full(S, plain, np.int8), 0.7)
        before = ens.engine.act_steps
        got, got_std = ens.act(states, np.full(S, drop, np.int8), 0.7)
        assert np.array_equal(got, ref)
        assert (got_std is None and ref_std is None) or np.array_equal(got_std, ref_std)
        assert np.array_equal(ens.engine.act_steps, before + 1)  # one draw per call, whatever p is
    assert np.array_equal(ens.engine.act_steps, np.full(S, len(pairs), np.uint64))


# ---------------------------------------------------------------------------
# 2. p > 0 against a float64 forward with the oracle's masks
# ---------------------------------------------------------------------------
SHAPES = [(11, 3, 2), (45, 24, 2), (39, 28, 2), (29, 8, 3), (512, 6, 2)]  # hopper, pen, door, antmaze 3x256, widest state


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("Sd,A,L", SHAPES, ids=["hopper", "pen", "door", "antmaze", "state512"])
@pytest.mark.parametrize("det", [False, True], ids=["gaussian", "deterministic"])
def test_dropout_act_matches_float64_forward(det, Sd, A, L, p):
    S, ma = 4, 0.8
    seeds = [11, (1 << 63) | 11, 2 ** 40 + 5, 7]
    ens = _ensemble(S, Sd, A, L, det, p, seeds)
    eng = ens.engine
    eng.set_act_steps([0, 5, 2 ** 32 - 1, 2 ** 33 + 9])  # the high counter word takes part
    rng = np.random.RandomState(Sd * 10 + A)
    src = np.array([DROP, DROP, DROP, DROP] if det else [DIST_DROP, DROP, DIST_DROP, DROP], np.int8)
    for call in range(3):
        states = rng.randn(S, Sd).astype(np.float32)
        steps = eng.act_steps
        out, std = ens.act(states, src, ma)
        assert np.array_equal(eng.act_steps, steps + 1)
        for m in range(S):
            ref, ref_std = _forward64(eng, m, states[m], seeds[m], int(steps[m]), p, int(src[m]), ma)
            np.testing.assert_allclose(out[m], ref, rtol=1e-5, atol=1e-6, err_msg=f"member {m} call {call}")
            if src[m] == DIST_DROP:
                assert np.array_equal(std[m], eng.act_host_gaussian(m, states[m])[1])  # code 2's std
                np.testing.assert_allclose(std[m], ref_std, rtol=1e-6)


# ---------------------------------------------------------------------------
# 3. the act counter
# ---------------------------------------------------------------------------
def test_counter_rewind_reproduces_and_other_codes_leave_it():
    S, Sd, A = 5, 17, 6
    ens = _ensemble(S, Sd, A, 2, False, 0.3, [1, 2, 3, 4, 5])
    guide = _ensemble(S, Sd, A, 2, False, 0.3, [9, 8, 7, 6, 5])
    ens.set_guide(guide)
    ens.bind_replay(_replay(S, Sd, A))
    eng = ens.engine
    states = np.random.RandomState(1).randn(S, Sd).astype(np.float32)
    src = np.array([DIST_DROP, DROP, DIST_DROP, SKIP, DROP], np.int8)
    eng.set_act_steps([10, 20, 30, 40, 50])
    a0, s0 = ens.act(states, src)
    assert eng.act_steps.tolist() == [11, 21, 31, 40, 51]  # the skipped member's counter stays
    a1, _ = ens.act(states, src)
    assert eng.act_steps.tolist() == [12, 22, 32, 40, 52]
    assert not np.array_equal(a0[[0, 1, 2, 4]], a1[[0, 1, 2, 4]])  # a new draw
    eng.set_act_steps([10, 20, 30, 40, 50])
    r0, rs0 = ens.act(states, src)
    assert np.array_equal(np.nan_to_num(r0), np.nan_to_num(a0)) and np.array_equal(np.nan_to_num(rs0), np.nan_to_num(s0))
    before = eng.act_steps
    for code in (SKIP, LEARNER, DIST, GUIDE):
        ens.act(states, np.full(S, code, np.int8))
    ens.retire([1, 3])
    ens.train_step_logged(np.random.RandomState(2).randint(0, 4096, size=(S, 256)))
    ens.resume([1, 3])
    ens.train_step_logged(np.random.RandomState(3).randint(0, 4096, size=(S, 256)))
    torch.cuda.synchronize()
    assert np.array_equal(eng.act_steps, before)
    # the weights moved, the counter did not: the draw at 11 of the moved weights is the oracle's draw at 11
    a2, _ = ens.act(states, src)
    for m in (0, 1, 2, 4):
        ref, _ = _forward64(eng, m, states[m], m + 1, int(before[m]), 0.3, int(src[m]), 1.0)
        np.testing.assert_allclose(a2[m], ref, rtol=1e-5, atol=1e-6)


def test_one_64_member_call_equals_64_single_member_calls():
    S, Sd, A = 64, 29, 8
    ens = _ensemble(S, Sd, A, 3, False, 0.1, [1000 + 3 * m for m in range(S)])
    eng = ens.engine
    rng = np.random.RandomState(64)
    start = rng.randint(0, 2 ** 40, size=S).astype(np.uint64)
    src = rng.choice([DROP, DIST_DROP], size=S).astype(np.int8)
    states = rng.randn(S, Sd).astype(np.float32)
    eng.set_act_steps(start)
    full, full_std = ens.act(states, src)
    after = eng.act_steps
    eng.set_act_steps(start)
    for m in range(S):
        one = np.full(S, SKIP, np.int8)
        one[m] = src[m]
        out, std = ens.act(states, one)
        assert np.array_equal(out[m], full[m]), m
        if src[m] == DIST_DROP:
            assert np.array_equal(std[m], full_std[m]), m
    assert np.array_equal(eng.act_steps, after) and np.array_equal(after, start + 1)


def test_equal_keys_and_counters_draw_equal_masks_and_permutation_permutes():
    S, Sd, A, p = 6, 39, 28, 0.5
    seeds = [21, 22, 23, 24, 25, 26]
    ens = _ensemble(S, Sd, A, 2, False, p, seeds)
    eng = ens.engine
    eng.load_params(5, eng.param_views(0))  # member 5 is member 0: same weights, key and counter, other slot
    eng.set_hparams(5, seed=seeds[0])
    steps = np.array([7, 8, 9, 10, 11, 7], np.uint64)
    eng.set_act_steps(steps)
    rng = np.random.RandomState(6)
    states = rng.randn(S, Sd).astype(np.float32)
    states[5] = states[0]
    src = np.array([DIST_DROP, DROP, DIST_DROP, DROP, DIST_DROP, DIST_DROP], np.int8)
    out, std = ens.act(states, src)
    assert np.array_equal(out[5], out[0]) and np.array_equal(std[5], std[0])
    # the same members in another order: the results follow them
    perm = [3, 5, 0, 4, 1, 2]
    keys = [eng.get_hparams(j).seed for j in perm]
    other = _ensemble(S, Sd, A, 2, False, p, keys, init=False)
    for i, j in enumerate(perm):
        other.engine.load_params(i, eng.param_views(j))
    other.engine.set_act_steps(steps[perm])
    out2, std2 = other.act(states[perm], src[perm])
    for i, j in enumerate(perm):
        assert np.array_equal(out2[i], out[j]), (i, j)
        if src[j] == DIST_DROP:
            assert np.array_equal(std2[i], std[j]), (i, j)


# ---------------------------------------------------------------------------
# 4. the masks themselves: read back exactly through probe actors
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_masks_read_back_are_the_oracle_masks_and_keep_1_minus_p(p):
    """Probe actors make the action a readout of the masks: an all-zero weight with bias 1 in front of a hidden layer
    makes its pre-activation 1 everywhere, and output a reads units 4a .. 4a+3 with weights c * 2^k, so
    atanh(action_a) / (c * scale) is the 4-bit number of their keep decisions.  Member 2i reads layer 1 alone; member
    2i+1 (layer 0 fed by ones, layer 1 the identity) reads keep0 & keep1.  Both share key and counter."""
    S, Sd, A, H, L, pairs, calls = 64, 5, 64, 256, 2, 32, 64
    seeds = [[5000 + i] * 2 for i in range(pairs)]
    seeds = [s for pair in seeds for s in pair]
    ens = _ensemble(S, Sd, A, L, True, p, seeds, init=False)
    eng = ens.engine
    c = 0.01
    W2 = np.zeros((A, H))
    for a in range(A):
        W2[a, 4 * a:4 * a + 4] = c * 2.0 ** np.arange(4)
    for m in range(S):
        eng.params[m].zero_()
        _set_actor(eng, m, 2, _lib.KIND_WEIGHT, W2)
        if m % 2 == 0:
            _set_actor(eng, m, 1, _lib.KIND_BIAS, np.ones(H))
        else:
            _set_actor(eng, m, 0, _lib.KIND_BIAS, np.ones(H))
            _set_actor(eng, m, 1, _lib.KIND_WEIGHT, np.eye(H))
    scale = float(np.float32(1.0 / (1.0 - p)))
    states = np.zeros((S, Sd), np.float32)
    src = np.full(S, DROP, np.int8)
    kept = np.zeros(2, np.int64)  # layer 0 (counted where layer 1 keeps), layer 1
    seen = np.zeros(2, np.int64)
    for k in range(calls):
        out, _ = ens.act(states, src, 1.0)
        z = np.arctanh(out.astype(np.float64)) / c
        for i in range(pairs):
            seed = seeds[2 * i]
            x1, x01 = z[2 * i] / scale, z[2 * i + 1] / scale ** 2
            k1, k01 = np.rint(x1).astype(np.int64), np.rint(x01).astype(np.int64)
            assert np.abs(x1 - k1).max() < 0.01 and np.abs(x01 - k01).max() < 0.01  # the readout is exact
            keep1 = ((k1[:, None] >> np.arange(4)) & 1).reshape(-1).astype(np.uint8)
            keep01 = ((k01[:, None] >> np.arange(4)) & 1).reshape(-1).astype(np.uint8)
            assert np.array_equal(keep1, philox_act_dropout_mask(seed, k, 1, H, p)), (i, k)
            ref0 = philox_act_dropout_mask(seed, k, 0, H, p)
            assert np.array_equal(keep01, ref0 & keep1), (i, k)
            # the act stream is not the update stream: the training mask of row 0 at actor_step k differs
            assert not np.array_equal(keep1, philox_dropout_mask(seed, k, 1, H, p)[:H])
            kept += [int(keep01.sum()), int(keep1.sum())]
            seen += [int(keep1.sum()), H]
    assert np.array_equal(eng.act_steps, np.full(S, calls, np.uint64))
    assert pairs * calls >= 2000  # draws per layer
    for layer in range(2):
        n, x = int(seen[layer]), int(kept[layer])
        sigma = np.sqrt(n * p * (1 - p))
        assert abs(x - n * (1 - p)) <= 5 * sigma, (layer, x / n, 1 - p)


# ---------------------------------------------------------------------------
# 5. the vectorised JSRL loop with dropout actors
# ---------------------------------------------------------------------------
P_DROP = 0.1


class _StopMember:
    """A scheduler (the on_result protocol of asha.ASHAScheduler) that stops one member at its second report."""

    def __init__(self, member):
        self.member, self.stopped = member, {}

    def on_result(self, m, n, score, total_it):
        if m == self.member and n == 2:
            self.stopped[m] = (n, total_it)
            return "stop"
        return "continue"


def _configs(det, tmp):
    cfgs = _member_configs(det, tmp)
    for c in cfgs:
        c.actor_dropout = P_DROP
    return cfgs


def _run(configs, member_ids, rb, scheduler=None):
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    logs = {m: [] for m in range(len(configs))}
    envs = [PointEnv(100 + i) for i in member_ids]
    eval_envs = [PointEnv(200 + i) for i in member_ids]
    learner, cfgs, hist = ensemble_train_loop(configs, envs, eval_envs, rb, 3, 2, 1.0, max_steps=PointEnv.T,
                                              log=lambda m, d, step: logs[m].append((step, d)), scheduler=scheduler,
                                              philox_act_dropout=True)
    torch.cuda.synchronize()
    return learner, cfgs, hist, logs


@pytest.fixture(scope="module", params=[False, True], ids=["gaussian", "deterministic"])
def dropout_runs(request, tmp_path_factory):
    det = request.param
    tmp = tmp_path_factory.mktemp("drop_det" if det else "drop_gauss")
    rb = _offline_buffer()
    rec = {"insert": [], "step": [], "offline": [], "source": []}
    orig = IQLEnsemble.add_transitions, IQLEnsemble.train_step_logged, IQLEnsemble.train_steps, IQLEnsemble.act

    def add(self, *a, **k):
        rec["insert"].append([np.array(x, copy=True) for x in a])
        return orig[0](self, *a, **k)

    def step(self, indices=None):
        rec["step"].append(np.array(indices, copy=True))
        return orig[1](self, indices)

    def ksteps(self, k, **kw):
        rec["offline"].append(kw["indices"].numpy().copy())
        return orig[2](self, k, **kw)

    def act(self, states, source, *a, **k):
        rec["source"].append(np.array(source, copy=True))
        return orig[3](self, states, source, *a, **k)

    IQLEnsemble.add_transitions, IQLEnsemble.train_step_logged, IQLEnsemble.train_steps, IQLEnsemble.act = add, step, ksteps, act
    try:
        ens_cfgs = _configs(det, tmp / "ens")
        init_cfgs = copy.deepcopy(ens_cfgs)
        ens = _run(ens_cfgs, range(4), rb)
    finally:
        IQLEnsemble.add_transitions, IQLEnsemble.train_step_logged, IQLEnsemble.train_steps, IQLEnsemble.act = orig
    singles = []
    for m in range(4):
        c = copy.deepcopy(init_cfgs[m])
        c.checkpoints_path = os.path.join(str(tmp / "single"), os.path.basename(c.checkpoints_path))
        singles.append(_run([c], [m], rb))
    return dict(det=det, rb=rb, ens=ens, singles=singles, rec=rec, init_cfgs=init_cfgs, tmp=tmp)


def test_dropout_loop_members_are_independent(dropout_runs):
    learner, cfgs, hist, logs = dropout_runs["ens"]
    for m in range(4):
        l1, c1, h1, g1 = dropout_runs["singles"][m]
        assert _same(logs[m], g1[0]), m
        assert _same(hist[m], h1[0]), m
        assert torch.equal(learner._buffers[m].rows, l1._buffers[0].rows)
        for arena in ("params", "exp_avg", "exp_avg_sq", "target"):
            assert torch.equal(getattr(learner.engine, arena)[m], getattr(l1.engine, arena)[0]), (m, arena)
            assert torch.equal(getattr(learner.guide.engine, arena)[m], getattr(l1.guide.engine, arena)[0]), (m, arena)
        assert learner.engine.act_steps[m] == l1.engine.act_steps[0] > 0
        names = sorted(os.listdir(cfgs[m].checkpoints_path))
        assert names == sorted(os.listdir(c1[0].checkpoints_path)) and len(names) == (OFF + ON) // EVAL
        for n in names:
            a = torch.load(os.path.join(cfgs[m].checkpoints_path, n), map_location="cpu")
            b = torch.load(os.path.join(c1[0].checkpoints_path, n), map_location="cpu")
            assert _same(a, b), (m, n)


def test_dropout_loop_act_codes_and_counters(dropout_runs):
    learner, cfgs, hist, logs = dropout_runs["ens"]
    det = dropout_runs["det"]
    code = DROP if det else DIST_DROP
    # the online acts of the learner ensemble (evaluations act with codes 1 / 3 and never with the dropout codes)
    src = np.array([s for s in dropout_runs["rec"]["source"]])
    learner_steps = (src == code).sum(axis=0)
    assert np.array_equal(learner.engine.act_steps, learner_steps.astype(np.uint64))
    assert (learner_steps > 0).all() and not np.isin(src, [DIST] if not det else [DIST_DROP]).any()
    assert np.array_equal(learner.guide.engine.act_steps, np.zeros(4, np.uint64))  # the guides never act in training mode
    assert [learner.engine.get_hparams(m).seed for m in range(4)] == [c.seed | (1 << 63) for c in dropout_runs["init_cfgs"]]
    assert [learner.guide.engine.get_hparams(m).seed for m in range(4)] == [c.seed for c in dropout_runs["init_cfgs"]]


def test_dropout_loop_member_is_the_single_learner_jsrl_step(dropout_runs):
    """Member m's recorded transitions and indices, replayed through ImplicitQLearning with dropout actors keyed like
    the loop's (the offline member by its seed, the learner by seed | 1 << 63), give the same losses and parameters."""
    import jsrl_corl_b200 as J
    from jsrl_corl_b200.jsrl_w_iql import member_networks

    learner, cfgs, hist, logs = dropout_runs["ens"]
    rec, rb, det = dropout_runs["rec"], dropout_runs["rb"], dropout_runs["det"]
    offline_idx = np.concatenate(rec["offline"], axis=1)
    for m in range(4):
        c = dropout_runs["init_cfgs"][m]
        (q, v, actor), (q2, v2, actor2) = member_networks(c, 3, 2, 1.0)
        assert actor.net.has_dropout_modules and actor.net.dropout_p == P_DROP

        def trainer(q, v, actor, max_steps, key):
            return J.ImplicitQLearning(1.0, actor, torch.optim.Adam(actor.parameters(), lr=c.actor_lr), q,
                                       torch.optim.Adam(q.parameters(), lr=c.qf_lr), v, torch.optim.Adam(v.parameters(), lr=c.vf_lr),
                                       beta=c.beta, iql_tau=c.iql_tau, discount=c.discount, tau=c.tau, max_steps=max_steps,
                                       device="cuda", seed=key)
        off_tr = trainer(q, v, actor, OFF, c.seed)
        np.random.seed(c.seed)
        off_logs = [d for _, d in logs[m] if "offline_iter" in d]
        assert len(off_logs) == OFF - B
        for k, d in enumerate(off_logs):
            got = off_tr.train(rb.sample(B))
            assert np.array_equal(rb._last_indices, offline_idx[m, k])
            assert all(got[key] == d[key] for key in ("value_loss", "q_loss", "actor_loss")), (m, k)
        on_tr = trainer(q2, v2, actor2, None, c.seed | (1 << 63))
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
        views = learner.engine.param_views(m, True)
        for grp, mod in (("qf", on_tr.qf), ("vf", on_tr.vf), ("actor", on_tr.actor)):
            for name, t in mod.state_dict().items():
                assert torch.equal(views[grp][name], t), (m, grp, name)


def test_dropout_loop_checkpoints_load_into_dropout_modules(dropout_runs):
    from jsrl_corl_b200.iql import DeterministicPolicy, GaussianPolicy, TwinQ, ValueFunction

    learner, cfgs, hist, logs = dropout_runs["ens"]
    cls = DeterministicPolicy if dropout_runs["det"] else GaussianPolicy
    for m in range(4):
        for n in sorted(os.listdir(cfgs[m].checkpoints_path)):
            sd = torch.load(os.path.join(cfgs[m].checkpoints_path, n), map_location="cpu")
            actor = cls(3, 2, 1.0, dropout=P_DROP)
            assert actor.net.has_dropout_modules
            actor.load_state_dict(sd["actor"], strict=True)
            TwinQ(3, 2).load_state_dict(sd["qf"], strict=True)
            ValueFunction(3).load_state_dict(sd["vf"], strict=True)


def test_dropout_loop_scheduler_stop_leaves_the_others_untouched(dropout_runs):
    learner, cfgs, hist, logs = dropout_runs["ens"]
    sched = _StopMember(1)
    cfg2 = _configs(dropout_runs["det"], dropout_runs["tmp"] / "sched")
    l2, c2, h2, g2 = _run(cfg2, range(4), dropout_runs["rb"], sched)
    assert list(sched.stopped) == [1]
    for m in (0, 2, 3):
        assert _same(g2[m], logs[m]) and _same(h2[m], hist[m]), m
        assert _same(l2.member_state_dict(m), learner.member_state_dict(m)), m
        assert l2.engine.act_steps[m] == learner.engine.act_steps[m]
    assert len(h2[1]) == 2 and not l2.active[1]
    assert l2.engine.act_steps[1] < learner.engine.act_steps[1]
