"""Chained backward in gradient-only mode (step_path="chain_grads"): bwd_chain.cu computes the hidden-layer and
input-layer weight gradients of every (member, net) task in one launch and stores them to the gradient arena;
adam_polyak_kernel then runs as on the per-phase path.  The gradients are the same GEMM tiles on the same operands
and the same optimizer kernel consumes them, so every arena matches the per-phase path bit for bit."""
import pytest
import torch

from helpers import Golden

pytestmark = pytest.mark.gpu

ARENAS = ("params", "exp_avg", "exp_avg_sq", "target", "grads")


def _make(g, n_members, step_path):
    from jsrl_corl_b200 import EnsembleEngine, ReplayBuffer

    m = g.meta
    eng = EnsembleEngine(n_members, m["S"], m["A"], m["H"], m["L"], m["B"], bool(m["det"]), "tf32", "cuda", 8,
                         step_path=step_path)
    rb = ReplayBuffer(m["S"], m["A"], m["n_rows"], "cuda")
    rb.load_d4rl_dataset(g.dataset())
    init = g.init_tree()
    for i in range(n_members):
        eng.load_params(i, init, dropout_keys=m["dropout"] > 0)
        eng.set_hparams(i, beta=m["beta"], iql_tau=m["iql_tau"], discount=m["discount"], tau=m["tau"], vf_lr=m["lr"],
                        qf_lr=m["lr"], actor_lr=m["lr"], actor_dropout=m["dropout"], cosine_t_max=m["max_steps"], seed=i)
        eng.bind_replay(i, rb.rows, m["n_rows"])
    return eng, rb


@pytest.mark.parametrize("name,members", [("halfcheetah_2x256", 8),   # the flagship shape, one task per CTA pair
                                          ("halfcheetah_2x256", 32),  # 128 tasks: CTA pairs run several; the
                                                                      # per-phase dgrad runs one CTA per problem
                                          ("antmaze_3x256", 4),       # 3 hidden layers: two dZ hand-overs per task
                                          ("antmaze_3x256", 1),       # single learner: row-split output-layer backward
                                          ("pen_2x256_dropout", 4)])  # dropout actor (masked dgrad of the policy)
def test_chain_grads_bit_identical_to_per_phase_path(name, members):
    """K = 6 fused steps (one CUDA graph, the next step's gather beside the optimizer) on both paths from the same
    state: losses and every arena are equal."""
    g = Golden(name)
    a, _ = _make(g, members, "phases")
    b, _ = _make(g, members, "chain_grads")
    assert not a.paths["chained_backward_grads"] and not a.paths["chained_backward"]
    assert b.paths["chained_backward_grads"] and not b.paths["chained_backward"]
    la, lb = a.train_steps(6), b.train_steps(6)
    torch.cuda.synchronize()
    assert torch.isfinite(la).all()
    assert torch.equal(la, lb)
    for arena in ARENAS:
        assert torch.equal(getattr(a, arena), getattr(b, arena)), arena


def test_chain_grads_k_fusion_and_launch_count():
    """8 members x K = 6 in one call == six calls of one step (bit-identical).  Per step: fused forward, loss,
    output-layer backward, chain, adam_polyak and the gather (the next step's rides beside the optimizer); the
    counter advance is folded into the last optimizer launch."""
    g = Golden("halfcheetah_2x256")
    one, _ = _make(g, 8, "chain_grads")
    six, _ = _make(g, 8, "chain_grads")
    l6 = six.train_steps(6)
    assert six.last_launch_count() == 6 * 6
    l1 = torch.cat([one.train_steps(1) for _ in range(6)], dim=1)
    assert one.last_launch_count() == 6
    assert torch.equal(l1, l6)
    for arena in ARENAS:
        assert torch.equal(getattr(one, arena), getattr(six, arena)), arena
    assert not torch.equal(l6[0], l6[1])  # members have their own Philox streams
    c = six.get_counters(0)
    assert (c.v_step, c.q_step, c.actor_step, c.total_it) == (6, 6, 6, 6)


def test_auto_selects_chain_grads_by_members_and_depth():
    """auto: a two-layer single learner keeps the per-phase backward, the 64-member ensemble and a three-layer single
    learner run the gradient-only chain; a shape the chain does not support (batch, input width, action width) stays
    per-phase under auto and is refused when a chain is asked for."""
    from jsrl_corl_b200 import EnsembleEngine

    single = EnsembleEngine(1, 17, 6, 256, 2, 256, False, "tf32", "cuda", 4)
    assert not single.paths["chained_backward_grads"] and not single.paths["chained_backward"]
    ens = EnsembleEngine(64, 17, 6, 256, 2, 256, False, "tf32", "cuda", 4)
    assert ens.paths["chained_backward_grads"] and not ens.paths["chained_backward"]
    deep = EnsembleEngine(1, 29, 8, 256, 3, 256, False, "tf32", "cuda", 4)
    assert deep.paths["chained_backward_grads"] and not deep.paths["chained_backward"]
    wide = EnsembleEngine(64, 11, 3, 256, 2, 512, True, "tf32", "cuda", 4)  # batch 512: no chain
    assert not wide.paths["chained_backward_grads"]
    with pytest.raises(ValueError, match="chained backward"):
        EnsembleEngine(2, 11, 3, 256, 2, 512, True, "tf32", "cuda", 4, step_path="chain_grads")
    # input width past one 256-column wgrad tile (K0 = 257, 306) and output-layer heads past the skinny backward (the
    # adroit door / hammer / relocate shapes, A = 26..30): per-phase under auto, refused when a chain is asked for
    for S_dim, A in ((251, 6), (300, 6), (39, 28), (46, 26), (39, 30)):
        assert not EnsembleEngine(64, S_dim, A, 256, 2, 256, False, "tf32", "cuda", 4).paths["chained_backward_grads"]
        for step_path in ("chain_grads", "chain"):
            with pytest.raises(ValueError, match="action_dim <= 24, state_dim \\+ action_dim <= 256"):
                EnsembleEngine(8, S_dim, A, 256, 2, 256, False, "tf32", "cuda", 4, step_path=step_path)
