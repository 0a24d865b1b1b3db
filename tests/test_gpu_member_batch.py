"""Ensemble members with their own batch sizes B_m <= B (iql_set_batch_sizes).

The engine keeps running every kernel on all B rows of every member; the gather writes zero rows past B_m, and the loss
kernel and the output-layer backward that restates the loss gradients (loss_row_grads) average over B_m rows and give
the pad rows exact-zero gradients.  Each member must therefore follow the numpy oracle run at its own batch size, with
its own first B_m indices, and members whose B_m == B must not change by a bit.

Shape: halfcheetah (obs 17, act 6, hidden 256), a 4096-row synthetic buffer, default hyper-parameters with one seed per
member, Philox sampling (the production path: each K-step call is a captured CUDA graph).
"""
import numpy as np
import pytest
import torch

from helpers import batch_from, rel_err

pytestmark = pytest.mark.gpu

S_DIM, A_DIM, H, N_ROWS = 17, 6, 256, 4096
FP32_LOSS, FP32_TENSOR, FP32_GRAD = 2e-5, 1e-5, 2e-5
TF32_LOSS5, TF32_TENSOR = 1e-3, 6e-3
SIZES_256 = (1, 7, 33, 128, 200, 256)

# (id, math, step_path, B, n_hidden, deterministic, dropout, batch sizes, engine.paths it must report)
MATRIX = [
    ("fp32", "fp32", "auto", 256, 2, False, 0.0, SIZES_256, dict(tensor_cores=False)),
    ("fp32-det", "fp32", "auto", 256, 2, True, 0.0, (7, 200, 256), dict(tensor_cores=False)),
    ("tf32-phases", "tf32", "phases", 256, 2, False, 0.0, SIZES_256,
     dict(tensor_cores=True, chained_backward=False, chained_backward_grads=False)),
    ("tf32-chain_grads", "tf32", "chain_grads", 256, 2, False, 0.0, SIZES_256, dict(tensor_cores=True, chained_backward_grads=True)),
    ("tf32-chain", "tf32", "chain", 256, 2, False, 0.0, SIZES_256, dict(tensor_cores=True, chained_backward=True)),
    ("tf32-B512", "tf32", "auto", 512, 2, False, 0.0, (128, 300, 512), dict(tensor_cores=True, chained_backward_grads=False)),
    ("tf32-3x256-det", "tf32", "auto", 256, 3, True, 0.0, (33, 200, 256), dict(tensor_cores=True, chained_backward_grads=True)),
    ("tf32-dropout", "tf32", "auto", 256, 2, False, 0.25, (7, 128, 256), dict(tensor_cores=True)),
    ("fp32-dropout", "fp32", "auto", 256, 2, False, 0.25, (1, 128, 256), dict(tensor_cores=False)),
]
ROW_IDS = [r[0] for r in MATRIX]
ROWS = {r[0]: r for r in MATRIX}

_DATA = []


def dataset():
    if not _DATA:
        from oracle.iql_numpy import synthetic_dataset

        _DATA.append(synthetic_dataset(N_ROWS, S_DIM, A_DIM, 3))
    return _DATA[0]


_RB = []


def replay():
    from jsrl_corl_b200 import ReplayBuffer

    if not _RB:
        rb = ReplayBuffer(S_DIM, A_DIM, N_ROWS, "cuda")
        rb.load_d4rl_dataset(dataset())
        _RB.append(rb)
    return _RB[0]


def seed_of(m):
    return 700 + 13 * m


def build(math, step_path, B, L, det, drop, sizes, seeds=None, max_k=8):
    """An ensemble of len(sizes) members, member j initialised with reference_init(seeds[j]); `sizes` None leaves the
    batch sizes at their default (no iql_set_batch_sizes call)."""
    from jsrl_corl_b200 import IQLEnsemble

    S = len(seeds) if seeds else len(sizes)
    seeds = seeds or [seed_of(m) for m in range(S)]
    ens = IQLEnsemble(S, S_DIM, A_DIM, H, L, B, deterministic=det, actor_dropout=drop, math_mode=math, max_steps_per_call=max_k,
                      seeds=seeds, step_path=step_path, batch_sizes=None if sizes is None else list(sizes))
    ens.bind_replay(replay())
    return ens


def init_tree(seed, L, det, drop):
    from jsrl_corl_b200.ensemble import reference_init

    q, v, actor = reference_init(seed, S_DIM, A_DIM, H, L, det, drop)
    return {g: {k: t.detach().numpy().astype(np.float32).copy() for k, t in mod.state_dict().items()}
            for g, mod in (("qf", q), ("vf", v), ("actor", actor))}


def oracle(seed, L, det, drop, dtype=np.float32):
    from oracle.iql_numpy import NumpyIQL, OracleConfig

    return NumpyIQL(OracleConfig(S_DIM, A_DIM, H, L, det, drop), init_tree(seed, L, det, drop), dtype)


def oracle_steps(orc, seed, bm, B, k0, n, masks=None):
    """n oracle steps at Philox positions k0 .. k0 + n - 1 on the member's first bm rows; masks [n][L][B][H] or None."""
    from oracle.philox import philox_indices

    out = []
    for i, k in enumerate(range(k0, k0 + n)):
        idx = philox_indices(seed, k, N_ROWS, B)[:bm]
        lo = orc.train(batch_from(dataset(), idx), dropout_masks=None if masks is None else masks[i][:, :bm])
        out.append([lo["value_loss"], lo["q_loss"], lo["actor_loss"]])
    return np.array(out)


def snapshot(eng, j, drop=False):
    params = {g: {k: v.cpu().numpy() for k, v in d.items()} for g, d in eng.param_views(j, drop).items()}
    params["q_target"] = {k: v.cpu().numpy() for k, v in eng.target_views(j).items()}
    m1, m2 = eng.moment_views(j, drop)
    mom = {g: {k: (m1[g][k].cpu().numpy(), m2[g][k].cpu().numpy()) for k in m1[g]} for g in m1}
    c = eng.get_counters(j)
    return params, mom, {f: getattr(c, f) for f, _ in type(c)._fields_}


def worst_tensor(params, orc):
    ref = dict(orc.state(), q_target=orc.q_target)
    worst = (0.0, None)
    for g in ("qf", "vf", "actor", "q_target"):
        for k, r in ref[g].items():
            if np.linalg.norm(r) > 0:
                worst = max(worst, (rel_err(params[g][k], r), f"{g}/{k}"), key=lambda t: t[0])
    return worst


def tf32_loss_errors(losses, ref, bm, B):
    """Loss errors of a TF32 member over its first five steps, in units of the suite's 1e-3 bar (pass: < 1).

    At B_m == B: relative to each loss.  At B_m < B: relative to the member's mean loss of that kind over the window, and
    the bar grows as sqrt(B / B_m).  The 1e-3 bar is for a mean over B = 256 rows, which averages 256 independent TF32
    rounding errors; a mean over B_m rows averages B_m of them, so its relative error grows as 1 / sqrt(B_m).  And the
    value loss of a handful of rows, a mean of wt * (q_target - v)^2, can nearly cancel at one step, where an error
    relative to that one loss says nothing about the arithmetic.  Measured on one B200 at 1,000 W: at most 0.47 of the
    bar for any member; B_m = 1 at 1.4e-3 of the window mean (7.0e-3 in the graph-replay test, 0.44 of its bar), where
    the error relative to each loss reached 2.2e-2.  A pad row leaking into a mean gives errors of order one."""
    le = np.abs(losses[:5] - ref[:5])
    if bm == B:
        return le / np.abs(ref[:5]) / TF32_LOSS5
    return le / np.abs(ref[:5]).mean(axis=0) / (TF32_LOSS5 * np.sqrt(B / bm))


def masks_for(S, K, L, B, seed=5):
    return (np.random.RandomState(seed).rand(S, K, L, B, H) >= 0.25).astype(np.uint8)


_RUNS = {}


def run_row(row):
    """K steps of the row's mixed-size ensemble (cached by row): (paths, losses [S, K, 3], snapshots, masks)."""
    if row not in _RUNS:
        _, math, step_path, B, L, det, drop, sizes, _ = ROWS[row]
        K = 4 if math == "fp32" else 5
        ens = build(math, step_path, B, L, det, drop, sizes)
        masks = masks_for(len(sizes), K, L, B) if drop > 0 else None
        losses = ens.train_steps(K, dropout_masks=None if masks is None else torch.from_numpy(masks)).cpu().numpy()
        torch.cuda.synchronize()
        _RUNS[row] = (ens.engine.paths, losses, [snapshot(ens.engine, j, drop > 0) for j in range(len(sizes))], masks)
    return _RUNS[row]


# ---------------------------------------------------------------------------------------------------------------------
# 1. every member against the oracle run at its own batch size
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("row", ROW_IDS)
def test_every_member_matches_the_oracle_at_its_own_batch_size(row):
    _, math, _, B, L, det, drop, sizes, paths = ROWS[row]
    got_paths, losses, snaps, masks = run_row(row)
    for k, v in paths.items():
        assert got_paths[k] == v, (row, got_paths)
    assert np.isfinite(losses).all()
    K = losses.shape[1]
    worst = []
    for m, bm in enumerate(sizes):
        orc = oracle(seed_of(m), L, det, drop)
        ref = oracle_steps(orc, seed_of(m), bm, B, 0, K, None if masks is None else masks[m])
        le = np.abs(losses[m] - ref) / np.maximum(np.abs(ref), 1e-30)
        we, where = worst_tensor(snaps[m][0], orc)
        worst.append((bm, float(le.max()), we, where))
        if math == "fp32":
            assert le.max() < FP32_LOSS, (row, m, bm, le)
            assert we < FP32_TENSOR, (row, m, bm, we, where)
        else:
            le = tf32_loss_errors(losses[m], ref, bm, B)
            worst[-1] = (bm, float(le.max()), we, where)
            assert le.max() < 1.0 and we < TF32_TENSOR, (row, m, bm, le, ref, we, where)
        assert snaps[m][2]["sample_step"] == K and snaps[m][2]["actor_step"] == K
    print(f"\n[{row}] (B_m, worst loss error (TF32: in units of its bar), worst tensor error, where): {worst}")


@pytest.mark.parametrize("sizes", [SIZES_256, (256, 200, 1)])
def test_fp32_gradients_at_each_batch_size_against_fp64_oracle(sizes):
    """Step 1: every member's gradient arena against the fp64 oracle at its own B_m (the output-layer gradients come from
    loss_row_grads, the log_std gradient from loss_kernel)."""
    import oracle.iql_numpy as onp

    ens = build("fp32", "auto", 256, 2, False, 0.0, sizes)
    ens.train_steps(1)
    torch.cuda.synchronize()
    for m, bm in enumerate(sizes):
        orc = oracle(seed_of(m), 2, False, 0.0, np.float64)
        grads = {}

        class Spy(onp._Adam):
            def step(self, gr):
                grads.update(gr)
                super().step(gr)

        for o in (orc.q_opt, orc.v_opt, orc.a_opt):
            o.__class__ = Spy
        oracle_steps(orc, seed_of(m), bm, 256, 0, 1)
        gv = ens.engine.grad_views(m)
        flat = {k: v.cpu().numpy() for d in gv.values() for k, v in d.items()}
        for k, ref in grads.items():
            if np.linalg.norm(ref) > 0:
                assert rel_err(flat[k], ref) < FP32_GRAD, (m, bm, k, rel_err(flat[k], ref))


def test_tf32_chain_gradients_with_keep_grads():
    """The chained backward (optimizer in its epilogue) stores the gradients with keep_grads: step 1 at B_m < B against
    the fp64 oracle at the suite's single-step TF32 gradient bar."""
    import oracle.iql_numpy as onp

    sizes = (33, 200, 256)
    ens = build("tf32", "chain", 256, 2, False, 0.0, sizes)
    ens.engine.keep_grads(True)
    ens.train_steps(1)
    torch.cuda.synchronize()
    for m, bm in enumerate(sizes):
        orc = oracle(seed_of(m), 2, False, 0.0, np.float64)
        grads = {}

        class Spy(onp._Adam):
            def step(self, gr):
                grads.update(gr)
                super().step(gr)

        for o in (orc.q_opt, orc.v_opt, orc.a_opt):
            o.__class__ = Spy
        oracle_steps(orc, seed_of(m), bm, 256, 0, 1)
        flat = {k: v.cpu().numpy() for d in ens.engine.grad_views(m).values() for k, v in d.items()}
        g_all = np.concatenate([flat[k].ravel() for k in grads])
        r_all = np.concatenate([np.asarray(grads[k]).ravel() for k in grads])
        assert rel_err(g_all, r_all) < 3e-2, (m, bm, rel_err(g_all, r_all))


# ---------------------------------------------------------------------------------------------------------------------
# 2. bit-exact invariants
# ---------------------------------------------------------------------------------------------------------------------
def _state(ens):
    e = ens.engine
    torch.cuda.synchronize()
    return {a: getattr(e, a).clone() for a in ("params", "exp_avg", "exp_avg_sq", "target")}, \
        [snapshot(e, j)[2] for j in range(e.n_members)]


def _member_equal(sa, sb, j, i):
    for a in sa[0]:
        assert torch.equal(sa[0][a][j], sb[0][a][i]), (a, j, i)
    assert sa[1][j] == sb[1][i], (j, i)


PATHS = [("fp32", "auto"), ("tf32", "phases"), ("tf32", "chain_grads"), ("tf32", "chain")]


@pytest.mark.parametrize("math,step_path", PATHS)
def test_full_sizes_and_one_changed_member(math, step_path):
    """Every B_m = B set explicitly equals never calling the API; setting one member's B_m changes only that member."""
    S, K = 4, 3
    runs = {}
    for tag, sizes in (("default", None), ("explicit", [256] * S), ("one", [256, 64, 256, 256])):
        ens = build(math, step_path, 256, 2, False, 0.0, sizes, seeds=[seed_of(m) for m in range(S)])
        assert ens.engine.batch_sizes == (sizes or [256] * S)
        losses = ens.train_steps(K).cpu().numpy()
        runs[tag] = (losses, _state(ens))
    assert np.array_equal(runs["default"][0], runs["explicit"][0])
    for j in range(S):
        _member_equal(runs["default"][1], runs["explicit"][1], j, j)
    for j in (0, 2, 3):
        assert np.array_equal(runs["default"][0][j], runs["one"][0][j]), j
        _member_equal(runs["default"][1], runs["one"][1], j, j)
    assert not np.array_equal(runs["default"][0][1], runs["one"][0][1])


def test_permuting_members_with_their_sizes_permutes_results():
    _, math, step_path, B, L, det, drop, sizes, _ = ROWS["tf32-chain_grads"]
    perm = [3, 0, 5, 1, 4, 2]
    _, losses, snaps, _ = run_row("tf32-chain_grads")
    ens = build(math, step_path, B, L, det, drop, [sizes[m] for m in perm], seeds=[seed_of(m) for m in perm])
    pl = ens.train_steps(losses.shape[1]).cpu().numpy()
    for j, m in enumerate(perm):
        assert np.array_equal(pl[j], losses[m]), (j, m)
        params, mom, c = snapshot(ens.engine, j)
        assert c == snaps[m][2]
        for g in params:
            for k in params[g]:
                assert np.array_equal(params[g][k], snaps[m][0][g][k]), (j, m, g, k)
        for g in mom:
            for k in mom[g]:
                assert np.array_equal(mom[g][k][0], snaps[m][1][g][k][0]) and np.array_equal(mom[g][k][1], snaps[m][1][g][k][1])


def test_pad_index_entries_are_ignored():
    """Garbage past B_m in given indices (K-step call and host step) is neither read nor refused."""
    S, K, B = 3, 3, 256
    sizes = [7, 128, 256]
    rng = np.random.RandomState(4)
    idx = rng.randint(0, N_ROWS, size=(S, K, B)).astype(np.int64)
    results = []
    for fill in (None, -1, 2 ** 40):
        x = idx.copy()
        if fill is not None:
            for m, bm in enumerate(sizes):
                x[m, :, bm:] = fill
        ens = build("tf32", "auto", B, 2, False, 0.0, sizes)
        la = ens.train_steps(K, mode="indices", indices=torch.from_numpy(x)).cpu().numpy()
        lb = np.stack([ens.train_step_logged(x[:, k]) for k in range(K)], axis=1)
        results.append((la, lb, _state(ens)))
    for la, lb, st in results[1:]:
        assert np.array_equal(la, results[0][0]) and np.array_equal(lb, results[0][1])
        for j in range(S):
            _member_equal(st, results[0][2], j, j)


def test_host_steps_equal_one_k_step_call_with_mixed_sizes():
    S, K, B = 6, 4, 256
    rng = np.random.RandomState(8)
    idx = rng.randint(0, N_ROWS, size=(S, K, B)).astype(np.int64)
    a = build("tf32", "auto", B, 2, False, 0.0, SIZES_256)
    b = build("tf32", "auto", B, 2, False, 0.0, SIZES_256)
    la = np.stack([a.train_step_logged(idx[:, k]) for k in range(K)], axis=1)
    lb = b.train_steps(K, mode="indices", indices=torch.from_numpy(idx)).cpu().numpy()
    assert np.array_equal(la, lb)
    sa, sb = _state(a), _state(b)
    for j in range(S):
        _member_equal(sa, sb, j, j)


def test_logged_step_draws_each_member_its_own_batch():
    """Without indices, member m draws B_m indices with np.random.randint, as ReplayBuffer.sample(B_m) would."""
    sizes = (7, 128, 256)
    ens = build("fp32", "auto", 256, 2, False, 0.0, sizes)
    np.random.seed(3)
    losses = ens.train_step_logged()
    np.random.seed(3)
    for m, bm in enumerate(sizes):
        idx = np.random.randint(0, N_ROWS, size=bm)
        lo = oracle(seed_of(m), 2, False, 0.0).train(batch_from(dataset(), idx))
        ref = np.array([lo["value_loss"], lo["q_loss"], lo["actor_loss"]])
        assert (np.abs(losses[m] - ref) / np.abs(ref)).max() < FP32_LOSS, (m, losses[m], ref)


@pytest.mark.parametrize("math,step_path", [("fp32", "auto"), ("tf32", "chain_grads")])
def test_size_change_between_graph_replays_takes_effect(math, step_path):
    S, K1, B = 3, 4, 256
    first, second = [256, 33, 200], [64, 256, 1]
    ens = build(math, step_path, B, 2, False, 0.0, first)
    la = ens.train_steps(K1).cpu().numpy()
    ens.engine.set_batch_sizes(second)
    lb = ens.train_steps(K1).cpu().numpy()  # same K and mode: replays the graph the first call captured
    torch.cuda.synchronize()
    losses = np.concatenate([la, lb], axis=1)
    for m in range(S):
        orc = oracle(seed_of(m), 2, False, 0.0)
        ref = np.concatenate([oracle_steps(orc, seed_of(m), first[m], B, 0, K1),
                              oracle_steps(orc, seed_of(m), second[m], B, K1, K1)])
        le = np.abs(losses[m] - ref) / np.abs(ref)
        we, where = worst_tensor(snapshot(ens.engine, m)[0], orc)
        if math == "fp32":
            assert le.max() < FP32_LOSS and we < FP32_TENSOR, (m, le, we, where)
        else:
            # the second call starts at step 5 with the new sizes: its own five-step window
            for w in (slice(0, K1), slice(K1, 2 * K1)):
                bm = (first if w.start == 0 else second)[m]
                e = tf32_loss_errors(losses[m][w], ref[w], bm, B)
                assert e.max() < 1.0 and we < TF32_TENSOR, (m, bm, e, ref[w], we, where)


def test_philox_idx_out_and_load_batch_refusal():
    from oracle.philox import philox_indices

    S, K, B = 3, 2, 256
    sizes = [1, 100, 256]
    ens = build("fp32", "auto", B, 2, False, 0.0, sizes)
    _, idx = ens.train_steps(K, return_indices=True)
    idx = idx.cpu().numpy()
    for m, bm in enumerate(sizes):
        for k in range(K):
            assert np.array_equal(idx[m, k, :bm], philox_indices(seed_of(m), k, N_ROWS, B)[:bm]), (m, k)
            assert (idx[m, k, bm:] == -1).all(), (m, k)
    batch = [torch.zeros(B, S_DIM), torch.zeros(B, A_DIM), torch.zeros(B), torch.zeros(B, S_DIM), torch.zeros(B)]
    ens.engine.load_batch(2, batch)  # B_m == B: accepted
    with pytest.raises(RuntimeError, match="batch size"):
        ens.engine.load_batch(0, batch)
