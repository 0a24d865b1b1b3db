"""Checkpoint interchange in the other direction: a checkpoint written by the B200 engine's drop-in trainer
(tools/write_engine_checkpoint.py, run on a B200; fixture committed under tests/golden/) must be loadable by the
UNMODIFIED reference trainer, which must continue with the same losses.

Without the reference tree this is checked against stored reference data: the engine's checkpoint has exactly the
structure of reference_checkpoint_19.pt (written by the reference trainer itself, oracle/gen_golden.py), and the numpy
oracle -- pinned to the reference by the stored trajectories of test_oracle.py -- continues from its weights, Adam moments,
step counts and LR schedule with the engine's losses.  Where the reference tree is present, the reference trainer is
run as well."""
import os

import numpy as np
import torch

from helpers import GOLDEN, batch_from


def _structure(obj):
    """Nested keys (in order), tensor shapes / dtypes and value types: key order carries the optimizer's index order."""
    if isinstance(obj, dict):
        return [(k, _structure(v)) for k, v in obj.items()]
    if isinstance(obj, (list, tuple)):
        return [_structure(v) for v in obj]
    if torch.is_tensor(obj):
        return ("tensor", tuple(obj.shape), str(obj.dtype))
    return type(obj).__name__


def _skip_first_draws(n_rows, B, n=20):
    np.random.seed(1)
    for _ in range(n):
        np.random.randint(0, n_rows, size=B)


def _oracle_from_checkpoint(sd, S, A, H, L):
    """The reference's load_state_dict applied to the oracle: weights, Adam moments and step counts, scheduler epoch
    and LR, total_it; q_target re-cloned from qf (iql.py:584)."""
    from oracle.iql_numpy import NumpyIQL, OracleConfig

    tree = {g: {k: t.numpy() for k, t in sd[g].items()} for g in ("qf", "vf", "actor")}
    orc = NumpyIQL(OracleConfig(S, A, H, L, max_steps=sd["actor_lr_schedule"]["T_max"]), tree, np.float32)
    for grp, opt, key in (("qf", orc.q_opt, "q_optimizer"), ("vf", orc.v_opt, "v_optimizer"), ("actor", orc.a_opt, "actor_optimizer")):
        state = sd[key]["state"]
        for i, name in enumerate(sd[grp]):  # optimizer index order == state_dict order (no buffers in these modules)
            opt.exp_avg[name][...] = state[i]["exp_avg"].numpy()
            opt.exp_avg_sq[name][...] = state[i]["exp_avg_sq"].numpy()
        opt.step_count = int(state[0]["step"])
        opt.lr = float(sd[key]["param_groups"][0]["lr"])
    orc.sched_epoch = int(sd["actor_lr_schedule"]["last_epoch"])
    orc.total_it = int(sd["total_it"])
    return orc


def _reference_continuation(ref, sd, data, z):
    """The unmodified reference trainer loads the engine's checkpoint and continues with the engine's losses."""
    S, A, H, L, B, n_rows = [int(x) for x in z["dims"]]
    torch.manual_seed(99)
    q, v, actor = ref.TwinQ(S, A, H, L), ref.ValueFunction(S, H, L), ref.GaussianPolicy(S, A, 1.0, H, L)
    vo, qo, ao = (torch.optim.Adam(m.parameters(), lr=3e-4) for m in (v, q, actor))
    tr = ref.ImplicitQLearning(1.0, actor, ao, q, qo, v, vo, max_steps=40, device="cpu")
    assert list(sd.keys()) == list(tr.state_dict().keys())
    tr.load_state_dict(sd)
    assert tr.total_it == 20 and tr.actor_lr_schedule.last_epoch == 20
    assert float(qo.state_dict()["state"][0]["step"]) == 20.0
    import contextlib, io
    rb = ref.ReplayBuffer(S, A, n_rows, "cpu")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(data)
    _skip_first_draws(n_rows, B)
    losses = []
    for _ in range(5):
        log = tr.train(rb.sample(B))
        losses.append([log["value_loss"], log["q_loss"], log["actor_loss"]])
    np.testing.assert_allclose(np.array(losses), z["losses"], rtol=2e-5, atol=1e-8)


def test_reference_trainer_loads_engine_checkpoint():
    from oracle.iql_numpy import synthetic_dataset
    from oracle.ref_loader import load_reference_iql, reference_available

    sd = torch.load(os.path.join(GOLDEN, "engine_checkpoint_19.pt"), map_location="cpu")
    ref_sd = torch.load(os.path.join(GOLDEN, "reference_checkpoint_19.pt"), map_location="cpu")
    z = np.load(os.path.join(GOLDEN, "engine_checkpoint_next_losses.npz"))
    S, A, H, L, B, n_rows = [int(x) for x in z["dims"]]
    assert _structure(sd) == _structure(ref_sd)
    assert sd["total_it"] == 20 and sd["actor_lr_schedule"]["last_epoch"] == 20
    assert float(sd["q_optimizer"]["state"][0]["step"]) == 20.0
    for key in ("q_optimizer", "v_optimizer", "actor_optimizer"):
        assert sd[key]["param_groups"] == ref_sd[key]["param_groups"]
    assert sd["actor_lr_schedule"] == ref_sd["actor_lr_schedule"]

    data = synthetic_dataset(n_rows, S, A, 0)
    orc = _oracle_from_checkpoint(sd, S, A, H, L)
    _skip_first_draws(n_rows, B)
    losses = []
    for _ in range(5):
        lo = orc.train(batch_from(data, np.random.randint(0, n_rows, size=B)))
        losses.append([lo["value_loss"], lo["q_loss"], lo["actor_loss"]])
    np.testing.assert_allclose(np.array(losses), z["losses"], rtol=2e-5, atol=1e-8)

    if reference_available():
        _reference_continuation(load_reference_iql("finetune"), sd, data, z)
