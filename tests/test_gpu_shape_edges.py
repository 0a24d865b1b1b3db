"""Shape edges of the kernel dispatch table: every threshold the engine branches on (input width K0 = state_dim +
action_dim, action width A, hidden width H, batch B, depth L), on both sides, against the numpy oracle.

The named workloads pin only a handful of shapes; the C-ABI accepts any state_dim, any action_dim (up to 64 for Gaussian
actors), any hidden_dim % 4 == 0 and any batch.  Each row of the tables below names the branch it is there for.  The
adroit trio (door 39/28, hammer 46/26, relocate 39/30) are real shapes of this port that sit in the A = 25..32 band.

Bars are the suite's (tests/test_gpu_parity.py): FP32 gradients 2e-5 norm-wise against fp64, FP32 losses 2e-5 (5e-5
with dropout, as the pen test) and tensors 1e-5 against the fp32 oracle over 3 steps; TF32 losses 1e-3 (the depth /
width scaling of test_tcgen05_path_general_shapes_match_oracle on the L = 5 and H = 1024 rows) and tensors 6e-3.  The
TF32 step-1 gradient bars are wider than the late-snapshot test's 3e-2; TF32_GRAD_TOL and TF32_HIDDEN_BIAS_GRAD_TOL
below say why, with the measured values.
On top of the norm-wise bars every output row of every weight gradient and every input column of dW_0 is judged on its
own (slices under SLICE_FLOOR of the tensor norm skipped): a dropped 32-column block or a wrong tail element is ~1 there,
while it can hide in a norm over tens of thousands of elements."""
from collections import namedtuple

import numpy as np
import pytest
import torch

from helpers import batch_from, rel_err, tree_max_rel

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
TF32_TOL = 1e-3
TF32_W30_TOL = 6e-3
GRAD_TOL = 2e-5          # fp64 oracle, FP32 kernels (test_gradients_single_step_against_oracle)
# fp64 oracle, TF32 kernels, step 1 from reference_init.  Wider than the 3e-2 of test_one_step_from_late_reference_snapshot:
# a weight gradient is a batch sum over TF32-rounded dZ rows that partly cancel, and on these fresh states it measured up
# to 4.0e-2 (hammer, 8 members, one member's q2 layer-1 weight; 3.3e-2 for the L = 5 actor's input layer) on one B200
# (1,000 W), with the other rows and members between 8e-3 and 2.6e-2.  The FP32 kernels give <= 1.1e-5 on the same rows.
TF32_GRAD_TOL = 6e-2
SLICE_FLOOR = 1e-3       # slices below this fraction of the tensor norm are not judged on their own
FP32_SLICE_TOL = 1e-3    # one row / column of an FP32 gradient
# one input column of a TF32 dW_0 (measured <= 7.7e-2): a column never written reads 1.0, one taken from another ~1.4
TF32_SLICE_TOL = 0.25
# Bias gradients of the hidden layers on the TF32 path: db_l is the batch sum of dZ_l, whose rows carry the TF32 rounding
# of the hidden dgrad GEMMs and largely cancel in the sum, so the sum's relative error is a multiple of dZ_l's.  Measured
# on one B200 (1,000 W) up to 6.0e-2 (hammer, 8 members, q2 layer 1), where the weight gradients of the same runs reach
# 4.0e-2 and the FP32 kernels give <= 1.1e-5.
TF32_HIDDEN_BIAS_GRAD_TOL = 0.1
N_ROWS, STEPS, DROP = 3000, 3, 0.1

Row = namedtuple("Row", "id S A H L B det members dropout why", defaults=(256, 2, 256, False, 2, 0.0, ""))

FP32_ROWS = [
    Row("k0_24", 20, 4, why="K0 = 24: top of the first skinny input-layer bucket (kpad 24)"),
    Row("k0_25", 21, 4, why="K0 = 25: bottom of the kpad-40 bucket"),
    Row("k0_40", 34, 6, why="K0 = 40: top of the kpad-40 bucket"),
    Row("k0_41", 35, 6, why="K0 = 41: bottom of the kpad-72 bucket"),
    Row("hammer", 46, 26, why="K0 = 72: top of the last skinny bucket; A = 26: out_fwd<64>, output-layer backward on simt_gemm"),
    Row("k0_73", 67, 6, why="K0 = 73: input-layer forward and weight gradient on the generic simt_gemm_kernel"),
    Row("a1", 11, 1, why="A = 1: out_fwd<1>, last_bwd_v4 with a one-wide actor head"),
    Row("a7", 11, 7, why="A = 7: out_fwd<8> / last_bwd_v4<8> with a partial bucket"),
    Row("a9", 11, 9, why="A = 9: bottom of out_fwd<24> and of last_bwd_kernel<24> for the actor"),
    Row("a25", 11, 25, why="A = 25: first width past the skinny output-layer backward (two simt_gemm, loss on the main stream)"),
    Row("a64", 11, 64, why="A = 64: top of out_fwd<64> and of the loss kernel's LOSS_MAX_A log_std slots"),
    Row("a65_det", 11, 65, det=True, why="A = 65 (deterministic): output-layer forward on simt_gemm"),
    Row("s300", 300, 6, why="state_dim 300, K0 = 306: generic input layer, rows of 77 float4"),
    Row("h100_b33", 11, 3, H=100, B=33, why="H = 100, B = 33: tails of every SIMT grid (H not a multiple of 32, B of 16)"),
    Row("b1", 11, 3, B=1, why="B = 1: one batch row"),
    Row("b100_s1", 11, 3, B=100, members=1, why="B = 100, one member: row-split output-layer backward, two 50-row splits"),
    Row("l5", 11, 3, L=5, why="L = 5: deeper than the fused forward and the chain"),
]

TF32_ROWS = [
    Row("a1", 11, 1, why="A = 1: policy head fused into the forward's epilogue"),
    Row("a7", 11, 7, why="A = 7: fused policy head, partial 8-wide bucket"),
    Row("a9", 11, 9, why="A = 9: first width of the two-pass tcgen05 policy head"),
    Row("a32", 11, 32, why="A = 32: top of the two-pass tcgen05 policy head"),
    Row("a33", 11, 33, why="A = 33: policy head on out_fwd<64>"),
    Row("a64", 11, 64, why="A = 64: top of out_fwd<64> and of LOSS_MAX_A"),
    Row("a65_det", 11, 65, det=True, why="A = 65 (deterministic): policy head on simt_gemm"),
    Row("a28_b128", 39, 28, B=128, why="B = 128: single-CTA fused forward feeding the two-pass head"),
    Row("h1024_a28", 39, 28, H=1024, why="H = 1024, A = 28: out_ok false by width (64 x 1024 x 4 B > 200 KB), simt_gemm head"),
    Row("l5", 11, 3, L=5, why="L = 5: per-layer forward and per-phase backward"),
]

ADROIT = [("door", 39, 28), ("hammer", 46, 26), ("relocate", 39, 30)]
ADROIT_ROWS = [Row(f"{n}_S{s}", sd, a, members=s, dropout=DROP, why=f"adroit {n} at full shape, p = 0.1, injected masks")
               for n, sd, a in ADROIT for s in (1, 8)]


def _cpu_tree(views):
    return {g: {k: v.detach().cpu().numpy().copy() for k, v in d.items()} for g, d in views.items()}


def _flat(tree):
    return {k: v for g in ("qf", "vf", "actor") for k, v in tree[g].items()}


_DATA = {}


def dataset(S, A):
    from oracle.iql_numpy import synthetic_dataset

    if (S, A) not in _DATA:
        _DATA[(S, A)] = synthetic_dataset(N_ROWS, S, A, 4)
    return _DATA[(S, A)]


def oracle_config(row):
    from oracle.iql_numpy import OracleConfig

    return OracleConfig(row.S, row.A, row.H, row.L, row.det, row.dropout, max_steps=50)


def oracle_step1_grads(row, init, batch, mask):
    """Gradients of the first step from the fp64 oracle (its Adam spied on, as in test_row_split_output_layer_backward)."""
    import oracle.iql_numpy as onp

    grads = {}

    class Spy(onp._Adam):
        def step(self, gr):
            grads.update(gr)
            super().step(gr)

    orc = onp.NumpyIQL(oracle_config(row), init, np.float64)
    for o in (orc.q_opt, orc.v_opt, orc.a_opt):
        o.__class__ = Spy
    orc.train(batch, dropout_masks=mask)
    return grads


_RUNS = {}


def run_row(row, math_mode):
    """One step, then two more, from reference_init weights on Philox-drawn indices; the same steps on the oracle."""
    key = (row, math_mode)
    if key in _RUNS:
        return _RUNS[key]
    from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer
    from oracle.iql_numpy import NumpyIQL
    from oracle.philox import philox_indices

    S, drop = row.members, row.dropout > 0
    data = dataset(row.S, row.A)
    rb = ReplayBuffer(row.S, row.A, N_ROWS, "cuda")
    rb.load_d4rl_dataset(data)
    seeds = [40 + m for m in range(S)]
    ens = IQLEnsemble(S, row.S, row.A, row.H, row.L, row.B, deterministic=row.det, actor_dropout=row.dropout,
                      math_mode=math_mode, seeds=seeds, max_steps_per_call=4, hparams=[dict(cosine_t_max=50)] * S)
    ens.bind_replay(rb)
    eng = ens.engine
    init = [_cpu_tree(eng.param_views(m, drop)) for m in range(S)]
    idx = np.stack([[philox_indices(s, k, N_ROWS, row.B) for k in range(STEPS)] for s in seeds]).astype(np.int64)
    masks = None
    if drop:
        rs = np.random.RandomState(11)
        masks = (rs.uniform(size=(S, STEPS, row.L, row.B, row.H)) < 1.0 - row.dropout).astype(np.uint8)

    def call(k0, k1):
        mk = torch.from_numpy(masks[:, k0:k1].copy()) if drop else None
        return eng.train_steps(k1 - k0, mode="indices", indices=torch.from_numpy(idx[:, k0:k1].copy()),
                               dropout_masks=mk).cpu().numpy()

    l1 = call(0, 1)
    grads = [_flat(_cpu_tree(eng.grad_views(m, drop))) for m in range(S)]
    losses = np.concatenate([l1, call(1, STEPS)], axis=1)
    params = [_cpu_tree(eng.param_views(m, drop)) for m in range(S)]
    ref_grads, ref_losses, ref_state = [], [], []
    for m in range(S):
        mask = (lambda k: masks[m, k].astype(bool)) if drop else (lambda k: None)
        ref_grads.append(oracle_step1_grads(row, init[m], batch_from(data, idx[m, 0]), mask(0)))
        orc = NumpyIQL(oracle_config(row), init[m], np.float32)
        lo = [orc.train(batch_from(data, idx[m, k]), dropout_masks=mask(k)) for k in range(STEPS)]
        ref_losses.append([[d["value_loss"], d["q_loss"], d["actor_loss"]] for d in lo])
        ref_state.append(orc.state())
    out = dict(paths=dict(eng.paths), losses=losses, grads=grads, params=params, ref_grads=ref_grads,
               ref_losses=np.array(ref_losses, dtype=np.float64), ref_state=ref_state)
    _RUNS[key] = out
    return out


def slice_errors(got, ref, columns):
    """Worst relative error over the output rows of a weight gradient and, with `columns` (input layers), over its input
    columns; slices whose reference norm is below SLICE_FLOOR of the tensor's are skipped."""
    g, r = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    total = np.linalg.norm(r)
    worst = 0.0
    for axis in ((1, 0) if columns else (1,)):
        num, den = np.linalg.norm(g - r, axis=axis), np.linalg.norm(r, axis=axis)
        keep = den >= SLICE_FLOOR * total
        if keep.any():
            worst = max(worst, float((num[keep] / den[keep]).max()))
    return worst


def grad_errors(grads, ref_grads, rows=True, keys=lambda k, ref: True):
    """(worst norm-wise error, where), (worst slice error, where) over the gradient tensors of one member that `keys`
    selects.  Slices: the input columns of every dW_0 and, with `rows`, the output rows of every weight gradient."""
    norm, sl = (0.0, None), (0.0, None)
    for k, ref in ref_grads.items():
        if not keys(k, ref):
            continue
        e = rel_err(grads[k], ref)
        if e > norm[0]:
            norm = (e, k)
        first = k.endswith("net.0.weight")
        if ref.ndim == 2 and (rows or first):
            e = slice_errors(grads[k], ref, first) if rows else slice_errors(grads[k].T, ref.T, False)
            if e > sl[0]:
                sl = (e, k)
    return norm, sl


def _loss_errors(losses, ref):
    return np.abs(losses - ref) / np.maximum(np.abs(ref), 1e-30)


def _report(label, row, values):
    print(f"{label} {row.id}: " + ", ".join(f"{k} {v:.2e}" for k, v in values.items()))


# ---------------------------------------------------------------------------
# 1. FP32 kernels: gradients against fp64, trajectory against fp32
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("row", FP32_ROWS + ADROIT_ROWS, ids=lambda r: r.id)
def test_fp32_shape_edges_against_oracle(row):
    """Worst measured on one B200 over every row and member: gradients 1.1e-5 norm-wise (hammer, 8 members), one row or
    column 1.3e-5 (B = 1), losses 1.7e-5 (B = 1: each loss is one sample), tensors 1.1e-6 (state_dim 300)."""
    r = run_row(row, "fp32")
    assert not r["paths"]["tensor_cores"]
    ltol = 5 * FP32_TOL if row.dropout > 0 else 2 * FP32_TOL
    for m in range(row.members):
        (gn, gk), (gs, sk) = grad_errors(r["grads"][m], r["ref_grads"][m])
        le = _loss_errors(r["losses"][m], r["ref_losses"][m]).max()
        pw, pk = tree_max_rel(r["params"][m], r["ref_state"][m])
        _report("fp32", row, dict(grad=gn, slice=gs, loss=le, param=pw))
        assert gn < GRAD_TOL, (m, gk, gn)
        assert gs < FP32_SLICE_TOL, (m, sk, gs)
        assert le < ltol, (m, r["losses"][m], r["ref_losses"][m])
        assert pw < FP32_TOL, (m, pk, pw)


# ---------------------------------------------------------------------------
# 2. TF32 (tcgen05) kernels against the oracle
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("row", TF32_ROWS + ADROIT_ROWS, ids=lambda r: r.id)
def test_tf32_shape_edges_against_oracle(row):
    """Losses of the 3 steps, every tensor after them, step-1 gradients against fp64 and every input column of dW_0.
    Worst measured on one B200 over every row and member: losses 1.0e-3 (H = 1024, bar 3e-3), tensors 2.6e-3 (L = 5),
    gradients 4.0e-2 and hidden-layer bias gradients 6.0e-2 (hammer, 8 members), one dW_0 column 7.7e-2 (hammer)."""
    r = run_row(row, "tf32")
    assert r["paths"]["tensor_cores"]
    if row.L > 2 or row.H > 256:  # one more TF32 GEMM per layer, wider sums: the general-shape test's scaling
        ltol = TF32_TOL * max(1, row.L - 1) * max(1.0, (row.H / 256) ** 0.5) * 1.5
    else:
        ltol = TF32_TOL
    def hidden_bias(k, ref):
        return ref.ndim == 1 and k.endswith("bias") and ref.size == row.H

    for m in range(row.members):
        (gn, gk), (gs, sk) = grad_errors(r["grads"][m], r["ref_grads"][m], False, lambda k, ref: not hidden_bias(k, ref))
        (bn, bk), _ = grad_errors(r["grads"][m], r["ref_grads"][m], False, hidden_bias)
        # relative error with the 1e-7 absolute floor of the pen bar (|d| <= 1e-7 + ltol |ref|  <=>  le <= ltol)
        le = (np.abs(r["losses"][m] - r["ref_losses"][m]) / (np.abs(r["ref_losses"][m]) + 1e-7 / ltol)).max()
        pw, pk = tree_max_rel(r["params"][m], r["ref_state"][m])
        _report("tf32", row, dict(grad=gn, hidden_bias=bn, column=gs, loss=le, param=pw))
        assert gn < TF32_GRAD_TOL, (m, gk, gn)
        assert bn < TF32_HIDDEN_BIAS_GRAD_TOL, (m, bk, bn)
        assert gs < TF32_SLICE_TOL, (m, sk, gs)
        assert le < ltol, (m, r["losses"][m], r["ref_losses"][m])
        assert pw < TF32_W30_TOL, (m, pk, pw)


# ---------------------------------------------------------------------------
# 3. chained backward against the per-phase path at the input-layer tile edges
# ---------------------------------------------------------------------------
CHAIN_ROWS = [Row(f"k0_{k0}", k0 - 6, 6, members=8, why=f"K0 = {k0}: input-layer wgrad tile {64 if k0 <= 64 else 128 if k0 <= 128 else 256}"
                  if k0 <= 256 else f"K0 = {k0}: wider than one 256-column tile, the chain refuses") for k0 in (64, 65, 128, 129, 256, 257, 306)]
CHAIN_ROWS += [Row("door_S8", 39, 28, members=8, why="A = 28: output-layer backward on simt_gemm, the chain refuses")]
ARENAS = ("params", "exp_avg", "exp_avg_sq", "target", "grads")


def _ensemble(row, step_path="auto", math_mode="tf32"):
    from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer

    rb = ReplayBuffer(row.S, row.A, N_ROWS, "cuda")
    rb.load_d4rl_dataset(dataset(row.S, row.A))
    ens = IQLEnsemble(row.members, row.S, row.A, row.H, row.L, row.B, deterministic=row.det, actor_dropout=row.dropout,
                      math_mode=math_mode, seeds=[40 + m for m in range(row.members)], max_steps_per_call=4,
                      hparams=[dict(cosine_t_max=50)] * row.members, step_path=step_path)
    ens.bind_replay(rb)
    return ens


def chain_serves(row):
    return row.A <= 24 and row.S + row.A <= 256


@pytest.mark.parametrize("row", CHAIN_ROWS, ids=lambda r: r.id)
def test_chain_grads_bit_identical_at_input_width_edges(row):
    """8 members, 2x256, batch 256: auto takes the gradient-only chain exactly where it serves the shape, and there the
    3-step result equals the per-phase path's in every arena, bit for bit."""
    auto = _ensemble(row)
    assert auto.engine.paths["chained_backward_grads"] == chain_serves(row), auto.engine.paths
    if not chain_serves(row):
        return
    phases = _ensemble(row, "phases")
    la, lb = phases.train_steps(3), auto.train_steps(3)
    torch.cuda.synchronize()
    assert torch.isfinite(la).all()
    assert torch.equal(la, lb)
    for arena in ARENAS:
        assert torch.equal(getattr(phases.engine, arena), getattr(auto.engine, arena)), arena


# ---------------------------------------------------------------------------
# 4. the reported paths are the paths that run
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("row", TF32_ROWS + ADROIT_ROWS + CHAIN_ROWS[:-1], ids=lambda r: r.id)
def test_reported_paths_match_profiled_kernels(row):
    """`paths` against the kernel labels of profile_step; the gradient-only chain with a fused policy head (A <= 8)
    takes 6 launches per step (test_chain_grads_k_fusion_and_launch_count)."""
    ens = _ensemble(row)
    paths = ens.engine.paths
    labels = {p["label"] for p in ens.engine.profile_step(reps=2)}
    assert paths["chained_backward_grads"] == ("bwd_chain_grads" in labels), (paths, labels)
    assert paths["chained_backward"] == ("bwd_chain" in labels), (paths, labels)
    assert paths["fused_forward"] == ("fused_fwd" in labels), (paths, labels)
    if paths["chained_backward_grads"] and row.A <= 8 and row.L == 2:
        ens.train_steps(3)
        assert ens.engine.last_launch_count() == 3 * 6


# ---------------------------------------------------------------------------
# 5. act at the wide shapes
# ---------------------------------------------------------------------------
def _policy64(eng, m):
    import jsrl_corl_b200 as J

    cls = J.DeterministicPolicy if eng.deterministic else J.GaussianPolicy
    pol = cls(eng.state_dim, eng.action_dim, 1.0, eng.hidden_dim, eng.n_hidden)
    pol.load_state_dict({k: v.cpu() for k, v in eng.param_views(m)["actor"].items()})
    return pol.double().eval()


def _act64(eng, m, states, max_action):
    with torch.no_grad():
        out = _policy64(eng, m)(torch.as_tensor(states, dtype=torch.float64))
    out = out if eng.deterministic else out.mean
    return torch.clamp(max_action * out, -max_action, max_action).numpy()


@pytest.mark.parametrize("Sd", [1, 300, 512])
@pytest.mark.parametrize("A,det", [(1, False), (28, False), (64, False), (65, True)])
def test_act_paths_at_wide_shapes(Sd, A, det):
    """Batched device act, per-member device act, act_host and act_members_host: bit-equal to each other (one act body)
    and within the act tests' bar (rtol 1e-5, atol 1e-6) of a float64 forward of the same actor."""
    from jsrl_corl_b200 import IQLEnsemble

    S, n, ma = 3, 4, 0.8
    ens = IQLEnsemble(S, Sd, A, 256, 2, 256, deterministic=det, math_mode="fp32", seeds=[7, 8, 9])
    eng = ens.engine
    states = np.random.RandomState(Sd + A).randn(S, n, Sd).astype(np.float32)
    dev = eng.act(-1, torch.from_numpy(states).cuda(), ma).cpu().numpy()
    members, _ = eng.act_members_host(states[:, 0], ["learner"] * S, ma)
    for m in range(S):
        one = eng.act(m, torch.from_numpy(states[m]).cuda(), ma).cpu().numpy()
        assert np.array_equal(one, dev[m]), m
        host = eng.act_host(m, states[m, 0], ma)
        assert np.array_equal(host, dev[m, 0]) and np.array_equal(members[m], host), m
        np.testing.assert_allclose(dev[m], _act64(eng, m, states[m], ma), rtol=1e-5, atol=1e-6)


def test_act_state_dim_513_device_path_only():
    """One float past the by-value observation of iql_act_host: refused there, served by the device act and by the
    batched host act (observations in pinned memory), both within the bar of a float64 forward."""
    from jsrl_corl_b200 import IQLEnsemble

    S, Sd, A, ma = 2, 513, 6, 1.0
    ens = IQLEnsemble(S, Sd, A, 256, 2, 256, math_mode="fp32", seeds=[3, 4])
    eng = ens.engine
    states = np.random.RandomState(513).randn(S, 2, Sd).astype(np.float32)
    with pytest.raises(ValueError, match="state_dim"):
        eng.act_host(0, states[0, 0], ma)
    dev = eng.act(-1, torch.from_numpy(states).cuda(), ma).cpu().numpy()
    members, _ = eng.act_members_host(states[:, 0], ["learner"] * S, ma)
    for m in range(S):
        assert np.array_equal(members[m], dev[m, 0]), m
        np.testing.assert_allclose(dev[m], _act64(eng, m, states[m], ma), rtol=1e-5, atol=1e-6)
