"""Pins the numpy oracle (oracle/iql_numpy.py) against fixtures generated from
the live reference (oracle/gen_golden.py), and against the reference itself
when /root/reference is present."""
import numpy as np
import pytest

from helpers import Golden, batch_from, network_errors_vs_floor, tree_max_rel
from oracle.iql_numpy import NumpyIQL


def _run(g, steps, dtype=np.float32, masks=None):
    orc = NumpyIQL(g.oracle_config(), g.init_tree(), dtype)
    data, idx = g.dataset(), g.indices()
    losses = []
    for t in range(steps):
        lo = orc.train(batch_from(data, idx[t]), dropout_masks=None if masks is None else masks[t])
        losses.append([lo["value_loss"], lo["q_loss"], lo["actor_loss"]])
    return orc, np.array(losses)


@pytest.mark.parametrize("name,steps", [("small_gauss", 40), ("small_det", 20), ("halfcheetah_2x256", 30),
                                        ("antmaze_3x256", 30)])
def test_oracle_matches_reference_trajectory(name, steps):
    g = Golden(name)
    orc, losses = _run(g, steps)
    # short horizon: before the chaotic amplification documented in DESIGN.md sets in
    np.testing.assert_allclose(losses, g.losses[:steps], rtol=2e-5, atol=1e-8)
    worst, where = tree_max_rel(orc.state(), g.tree(f"step{steps}"))
    assert worst < 1e-5, (worst, where)


def test_oracle_dropout_with_injected_masks():
    g = Golden("small_dropout")
    orc, losses = _run(g, 12, masks=g.dropout_masks())
    np.testing.assert_allclose(losses, g.losses[:12], rtol=2e-5, atol=1e-8)
    worst, where = tree_max_rel(orc.state(), g.tree("step12"))
    assert worst < 1e-5, (worst, where)


def test_oracle_adam_moments_and_target():
    g = Golden("small_gauss")
    orc, _ = _run(g, 20)
    opt = g.opt("step20")
    for grp, o in (("qf", orc.q_opt), ("vf", orc.v_opt), ("actor", orc.a_opt)):
        for name, (m, v) in opt[grp].items():
            np.testing.assert_allclose(o.exp_avg[name], m, rtol=1e-4, atol=1e-9)
            np.testing.assert_allclose(o.exp_avg_sq[name], v, rtol=1e-4, atol=1e-12)
    tgt = g.tree("step20")["q_target"]
    for k, v in tgt.items():
        np.testing.assert_allclose(orc.q_target[k], v, rtol=1e-5, atol=1e-7)
    assert abs(orc.a_opt.lr - float(g.z["step20/actor_lr"])) < 1e-15


@pytest.mark.slow
def test_oracle_1000_steps_within_reference_noise_floor():
    """After 1,000 free-running steps the trajectory is chaotic: the reference in
    fp64 differs from the reference in fp32 by `noise/*` (4-9e-2).  The oracle
    (a different summation order) must stay within 2x that floor."""
    g = Golden("hopper_1000")
    orc, losses = _run(g, 1000)
    for grp, (err, floor) in network_errors_vs_floor(g, orc.state(), "step1000").items():
        assert err <= 2.0 * floor, (grp, err, floor)
    # loss curves agree in the mean over the last 100 steps
    a, b = losses[-100:].mean(0), g.losses[-100:].astype(np.float64).mean(0)
    np.testing.assert_allclose(a, b, rtol=0.05)
    # and tightly over the first 30 steps
    np.testing.assert_allclose(losses[:30], g.losses[:30], rtol=2e-5, atol=1e-8)


def test_oracle_against_live_reference():
    from oracle.ref_loader import load_reference_iql, reference_available

    if not reference_available():
        pytest.skip("needs the original jsrl-CORL source under JSRL_REFERENCE_ROOT; no stored outputs of it exist for this comparison")
    import torch

    ref = load_reference_iql("offline")
    S, A, H, L, B = 7, 3, 48, 2, 24
    torch.manual_seed(3)
    q, v = ref.TwinQ(S, A, H, L), ref.ValueFunction(S, H, L)
    actor = ref.GaussianPolicy(S, A, 1.0, H, L)
    opts = [torch.optim.Adam(m.parameters(), lr=1e-3) for m in (v, q, actor)]
    tr = ref.ImplicitQLearning(1.0, actor, opts[2], q, opts[1], v, opts[0], iql_tau=0.8, beta=5.0, max_steps=50,
                               discount=0.95, tau=0.01, device="cpu")
    from oracle.iql_numpy import OracleConfig

    sd = {k: {kk: vv.detach().numpy().copy() for kk, vv in m.state_dict().items()} for k, m in (("qf", q), ("vf", v), ("actor", actor))}
    orc = NumpyIQL(OracleConfig(S, A, H, L, False, 0.0, 0.8, 5.0, 0.95, 0.01, 1e-3, 1e-3, 1e-3, 50), sd)
    rng = np.random.RandomState(0)
    for _ in range(15):
        batch = [rng.standard_normal((B, S)).astype(np.float32), rng.uniform(-1, 1, (B, A)).astype(np.float32),
                 rng.standard_normal((B, 1)).astype(np.float32), rng.standard_normal((B, S)).astype(np.float32),
                 (rng.uniform(size=(B, 1)) < 0.1).astype(np.float32)]
        lr = tr.train([torch.from_numpy(b) for b in batch])
        lo = orc.train(batch)
        for k in lr:
            assert abs(lr[k] - lo[k]) <= 2e-5 * abs(lr[k]) + 1e-8


@pytest.mark.parametrize("betas,eps", [((0.8, 0.99), 1e-8), ((0.0, 0.999), 1e-8), ((0.9, 0.999), 1e-6)])
def test_oracle_adam_non_default_settings_match_torch(betas, eps):
    """The oracle's Adam with betas / eps other than torch's defaults (ensemble members may each have their own)
    against torch.optim.Adam (single-tensor path), float64, 20 steps with fixed per-step gradients."""
    import torch
    from oracle.iql_numpy import _Adam

    rng = np.random.RandomState(4)
    shapes = {"w": (5, 3), "b": (5,)}
    init = {k: rng.standard_normal(s) for k, s in shapes.items()}
    grads = [{k: rng.standard_normal(s) * 10.0 ** rng.uniform(-4, 1) for k, s in shapes.items()} for _ in range(20)]
    params = {k: v.copy() for k, v in init.items()}
    orc = _Adam(params, 1e-3, betas, eps, np.float64)
    tp = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in init.items()}
    opt = torch.optim.Adam(list(tp.values()), lr=1e-3, betas=betas, eps=eps, foreach=False)
    for g in grads:
        orc.step(g)
        for k, t in tp.items():
            t.grad = torch.from_numpy(g[k])
        opt.step()
        for k, t in tp.items():
            st = opt.state[t]
            np.testing.assert_allclose(params[k], t.detach().numpy(), rtol=1e-12, atol=0)
            np.testing.assert_allclose(orc.exp_avg[k], st["exp_avg"].numpy(), rtol=1e-12, atol=0)
            np.testing.assert_allclose(orc.exp_avg_sq[k], st["exp_avg_sq"].numpy(), rtol=1e-12, atol=0)
    assert orc.step_count == 20


def test_oracle_cosine_schedule_with_eta_min_matches_torch():
    """CosineAnnealingLR(T_max=3, eta_min=1e-5) over 10 epochs (past T_max twice, through the recursive form's
    special branch) against the oracle's recursive form, standalone and as NumpyIQL applies it after each step."""
    import torch
    from oracle.iql_numpy import OracleConfig, cosine_recursive_lr

    base, t_max, eta_min = 3e-4, 3, 1e-5
    p = torch.zeros(1, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([p], lr=base)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=t_max, eta_min=eta_min)
    S, A, H, L, B = 3, 2, 8, 2, 4
    rng = np.random.RandomState(0)
    init = {
        "qf": {f"q{i}.net.{j}.{w}": rng.standard_normal(s) * 0.3 for i in (1, 2) for j, s_w, s_b in
               ((0, (H, S + A), (H,)), (2, (H, H), (H,)), (4, (1, H), (1,))) for w, s in (("weight", s_w), ("bias", s_b))},
        "vf": {f"v.net.{j}.{w}": rng.standard_normal(s) * 0.3 for j, s_w, s_b in
               ((0, (H, S), (H,)), (2, (H, H), (H,)), (4, (1, H), (1,))) for w, s in (("weight", s_w), ("bias", s_b))},
        "actor": {"log_std": np.zeros(A), **{f"net.net.{j}.{w}": rng.standard_normal(s) * 0.3 for j, s_w, s_b in
                  ((0, (H, S), (H,)), (2, (H, H), (H,)), (4, (A, H), (A,))) for w, s in (("weight", s_w), ("bias", s_b))}},
    }
    orc = NumpyIQL(OracleConfig(S, A, H, L, actor_lr=base, max_steps=t_max, lr_eta_min=eta_min), init, np.float64)
    lr = base
    for epoch in range(1, 11):
        opt.step()
        sched.step()
        lr = cosine_recursive_lr(lr, base, epoch, t_max, eta_min)
        want = opt.param_groups[0]["lr"]
        assert abs(lr - want) <= 1e-12 * abs(want), (epoch, lr, want)
        batch = [rng.standard_normal((B, S)), rng.uniform(-1, 1, (B, A)), rng.standard_normal((B, 1)),
                 rng.standard_normal((B, S)), np.zeros((B, 1))]
        orc.train(batch)
        assert orc.sched_epoch == epoch and abs(orc.a_opt.lr - want) <= 1e-12 * abs(want), (epoch, orc.a_opt.lr, want)


@pytest.mark.parametrize("name", ["hopper_late_999", "antmaze_late_999"])
def test_oracle_one_step_from_late_reference_snapshot(name):
    """Late-trajectory regime (Adam step 1000, bias corrections ~ 1, cosine LR ~ 0, saturated exp(beta adv) clamp for
    antmaze): ONE oracle step from the reference's own state at step 999 reproduces the reference's step 1000."""
    from helpers import LateSnapshot

    g = LateSnapshot(name)
    orc = g.load_into_oracle(np.float32)
    lo = orc.train(batch_from(g.dataset(), g.next_indices))
    got = np.array([lo["value_loss"], lo["q_loss"], lo["actor_loss"]])
    np.testing.assert_allclose(got, g.next_losses, rtol=1e-5)
    post = g.post_sampled()
    state = orc.state()
    for grp, d in post.items():
        for k, want in d.items():
            have = np.asarray(state[grp][k]).reshape(-1)[::16]
            np.testing.assert_allclose(have, want, rtol=1e-5, atol=1e-7, err_msg=f"{grp}/{k}")
    assert abs(orc.a_opt.lr - float(g.z[f"step{g.at + 1}/actor_lr"])) < 1e-15
