"""numpy's RandomState.randint index stream drawn on the device (IQL_SAMPLE_MT19937): the handle-free sampler against
numpy over the bound, block and position edges; the engine's mode="numpy" against mode="indices" fed by the same
RandomState objects on every step path; host steps, retired members, replay-size changes, state uploads; and
ensemble_train_loop with device_index_streams against the host draws.

Shape of the engine tests: halfcheetah (obs 17, act 6, hidden 256, batch 256), a 4096-row synthetic buffer.
"""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import mt19937_oracle as mt  # noqa: E402
from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer, _lib  # noqa: E402
from jsrl_corl_b200.synthetic import synthetic_dataset  # noqa: E402

S_DIM, A_DIM, H, B, N_ROWS = 17, 6, 256, 256, 4096
_RB = []


def replay():
    if not _RB:
        rb = ReplayBuffer(S_DIM, A_DIM, N_ROWS, "cuda")
        rb.load_d4rl_dataset(synthetic_dataset(N_ROWS, S_DIM, A_DIM, 5))
        _RB.append(rb)
    return _RB[0]


# ---------------------------------------------------------------------------
# 1. the handle-free sampler against numpy
# ---------------------------------------------------------------------------
def device_randint(rows, highs, counts):
    """Run iql_mt19937_randint over len(highs) streams; returns (draws per stream, new state rows)."""
    n = len(highs)
    states = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.uint32).view(np.int32)).cuda()
    stride = max(max(counts), 1)
    out = torch.full((n, stride), -7, dtype=torch.int64, device="cuda")
    hi = np.ascontiguousarray(highs, dtype=np.int64)
    cnt = np.ascontiguousarray(counts, dtype=np.int64)
    rc = _lib.lib().iql_mt19937_randint(states.data_ptr(), n, hi.ctypes.data, cnt.ctypes.data, out.data_ptr(), stride,
                                        torch.cuda.current_stream().cuda_stream)
    assert rc == _lib.IQL_OK
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert all((o[i, counts[i]:] == -7).all() for i in range(n))  # nothing past the count is written
    return [o[i, :counts[i]] for i in range(n)], states.cpu().numpy().view(np.uint32)


def rng_at(seed, pos):
    """A RandomState whose generator stands at word `pos` of its current key block (a fresh one stands at 624)."""
    r = np.random.RandomState(seed)
    if pos != 624:
        r.set_state(("MT19937", r.get_state()[1], pos))
    return r


HIGHS = [1, 2, 3, 10 ** 6, 2 ** 31 + 1, 2 ** 32] + [2 ** k for k in (4, 13, 16, 24, 31)] + [2 ** k + 1 for k in (4, 13, 16, 24)]


@pytest.mark.parametrize("pos", [0, 623, 624])
def test_sampler_matches_numpy_at_every_edge(pos):
    cases = [(h, n) for h in HIGHS for n in (1, 255, 1500)]  # counts within one block and across several
    cases += [(2 ** 32, 624 - pos if pos < 624 else 624), (2 ** 32, 1)]  # ends exactly on word 623 (pos = 624)
    refs = [rng_at(100 + i, pos) for i in range(len(cases))]
    rows = np.stack([mt.state_row(r) for r in refs])
    for call in range(2):  # a second call continues the stream
        got, rows = device_randint(rows, [h for h, _ in cases], [n for _, n in cases])
        for i, (h, n) in enumerate(cases):
            want = refs[i].randint(0, h, size=n)
            assert np.array_equal(got[i], want), (call, h, n, pos)
            _, key, p, _, _ = refs[i].get_state()
            assert np.array_equal(rows[i, :624], key) and int(rows[i, 624]) == p, (call, h, n, pos)


@pytest.mark.parametrize("n", [1, 2, 37, 256, 300])
def test_sampler_runs_many_streams_at_once(n):
    g = np.random.RandomState(n)
    highs = [int(x) for x in g.choice([1, 7, 10000, 65537, 2 ** 31 + 1, 2 ** 32], size=n)]
    counts = [int(x) for x in g.randint(0, 2000, size=n)]
    refs = [np.random.RandomState(7 * i + 1) for i in range(n)]
    for i, r in enumerate(refs):
        r.randint(0, 5, size=i % 700)  # every starting position
    got, rows = device_randint(np.stack([mt.state_row(r) for r in refs]), highs, counts)
    for i in range(n):
        assert np.array_equal(got[i], refs[i].randint(0, highs[i], size=counts[i])), i
        assert np.array_equal(rows[i], mt.state_row(refs[i])), i


# ---------------------------------------------------------------------------
# 2. the engine: mode="numpy" == mode="indices" on the same RandomStates
# ---------------------------------------------------------------------------
def make(S, math="tf32", step_path="auto", sizes=None, max_k=8, seed0=300):
    ens = IQLEnsemble(S, S_DIM, A_DIM, H, 2, B, math_mode=math, max_steps_per_call=max_k, step_path=step_path,
                      seeds=[seed0 + 13 * m for m in range(S)], batch_sizes=sizes)
    ens.bind_replay(replay())
    return ens


def host_indices(rngs, ens, K, highs=None):
    """What ensemble_train_loop draws on the host for one K-step call of `ens`'s active members."""
    e = ens.engine
    idx = np.zeros((e.n_members, K, e.batch_size), dtype=np.int64)
    for m in np.flatnonzero(e.active):
        high = ens._buffers[m]._high() if highs is None else highs[m]
        for k in range(K):
            idx[m, k, :e.batch_sizes[m]] = rngs[m].randint(0, high, size=e.batch_sizes[m])
    return torch.from_numpy(idx)


def snapshot(ens):
    e = ens.engine
    torch.cuda.synchronize()
    counters = [tuple(getattr(e.get_counters(m), f) for f, _ in _lib.Counters._fields_) for m in range(e.n_members)]
    return [t.clone() for t in (e.params, e.exp_avg, e.exp_avg_sq, e.target)], counters


def same_tensor(a, b):
    return torch.equal(torch.nan_to_num(a, nan=1.5e38), torch.nan_to_num(b, nan=1.5e38))


def assert_same_run(a, b):
    (ta, ca), (tb, cb) = snapshot(a), snapshot(b)
    assert ca == cb
    for x, y, name in zip(ta, tb, ("params", "exp_avg", "exp_avg_sq", "target")):
        assert torch.equal(x, y), name


def assert_same_streams(ens, rngs):
    probe = [np.random.RandomState(0) for _ in rngs]
    ens.engine.get_index_states(probe)
    for m, (p, r) in enumerate(zip(probe, rngs)):
        assert np.array_equal(mt.state_row(p), mt.state_row(r)), m


def run_pair(S, K, math, path, sizes=None, calls=3):
    """Same members trained by `calls` K-step calls twice: device streams vs host draws of the same RandomStates."""
    dev, host = make(S, math, path, sizes, max_k=K), make(S, math, path, sizes, max_k=K)
    rd = [np.random.RandomState(40 + m) for m in range(S)]
    rh = copy.deepcopy(rd)
    dev.set_index_streams(rd)
    for call in range(calls):
        logged = call == 0  # the first call reports its indices (no graph); the others replay the captured graph
        ld = dev.train_steps(K, mode="numpy", return_indices=logged)
        lh = host.train_steps(K, mode="indices", indices=host_indices(rh, host, K), return_indices=logged)
        if logged:
            (ld, id_), (lh, ih) = ld, lh
            assert torch.equal(id_, ih)
        assert same_tensor(ld, lh), call
    assert_same_run(dev, host)
    assert_same_streams(dev, rh)
    return dev, host, rd, rh


@pytest.mark.parametrize("math,path", [("fp32", "phases"), ("tf32", "phases"), ("tf32", "chain_grads"), ("tf32", "chain")])
@pytest.mark.parametrize("S,K", [(1, 1), (3, 7)])
def test_numpy_mode_equals_host_indices(math, path, S, K):
    run_pair(S, K, math, path)


@pytest.mark.parametrize("S,K", [(64, 256), (1, 256), (3, 7)])
def test_numpy_mode_equals_host_indices_auto(S, K):
    run_pair(S, K, "tf32", "auto", calls=2)


def test_numpy_mode_with_member_batch_sizes():
    run_pair(4, 7, "tf32", "auto", sizes=[256, 100, 17, 1])
    run_pair(3, 5, "fp32", "phases", sizes=[3, 256, 128])


def test_retired_members_draw_nothing_and_resume():
    dev, host, rd, rh = run_pair(5, 6, "tf32", "auto", calls=1)
    for ens in (dev, host):
        ens.retire([1, 3])
    torch.cuda.synchronize()
    frozen = dev.engine._mt_states.clone()
    for _ in range(2):
        dev.train_steps(6, mode="numpy")
        host.train_steps(6, mode="indices", indices=host_indices(rh, host, 6))
    torch.cuda.synchronize()
    assert torch.equal(dev.engine._mt_states[[1, 3]], frozen[[1, 3]])  # every bit of a retired stream stays
    assert not torch.equal(dev.engine._mt_states[0], frozen[0])
    for ens in (dev, host):
        ens.resume([1, 3])
    dev.train_steps(6, mode="numpy")
    host.train_steps(6, mode="indices", indices=host_indices(rh, host, 6))
    lo_d = dev.train_step_logged(numpy_streams=True)
    lo_h = host.train_step_logged(host_indices(rh, host, 1)[:, 0].numpy())
    assert np.array_equal(lo_d, lo_h)
    assert_same_run(dev, host)
    assert_same_streams(dev, rh)


def test_host_steps_equal_one_k_step_call():
    K = 7
    steps, call = make(3, sizes=[256, 64, 200], max_k=K), make(3, sizes=[256, 64, 200], max_k=K)
    steps.set_index_streams([np.random.RandomState(m) for m in range(3)])
    call.set_index_streams([np.random.RandomState(m) for m in range(3)])
    logged = np.stack([steps.train_step_logged(numpy_streams=True) for _ in range(K)], axis=1)  # [S, K, 3]
    ref = call.train_steps(K, mode="numpy").cpu().numpy()
    assert np.array_equal(logged, ref)
    assert_same_run(steps, call)
    assert torch.equal(steps.engine._mt_states, call.engine._mt_states)


def test_replay_size_change_between_graph_replays():
    dev, host, rd, rh = run_pair(2, 4, "tf32", "auto", calls=2)  # the graph is captured and replayed
    for ens in (dev, host):
        ens.engine.set_replay_size(0, 1000)
        ens.engine.set_replay_size(1, 3)
    for _ in range(2):
        dev.train_steps(4, mode="numpy")
        host.train_steps(4, mode="indices", indices=host_indices(rh, host, 4, highs=[1000, 3]))
    dev.engine.set_replay_size(1, 1)  # randint(0, 1): zeros, no word consumed
    host.engine.set_replay_size(1, 1)
    dev.train_steps(4, mode="numpy")
    host.train_steps(4, mode="indices", indices=host_indices(rh, host, 4, highs=[1000, 1]))
    assert_same_run(dev, host)
    assert_same_streams(dev, rh)


def test_uploaded_state_repeats_draws_and_refusals_draw_nothing():
    ens = make(2, max_k=4)
    with pytest.raises(RuntimeError, match="no index streams"):
        ens.train_steps(4, mode="numpy")
    with pytest.raises(RuntimeError, match="no index streams"):
        ens.train_step_logged(numpy_streams=True)
    start = [np.random.RandomState(8), np.random.RandomState(9)]
    ens.set_index_streams(copy.deepcopy(start))
    _, first = ens.train_steps(4, mode="numpy", return_indices=True)
    ens.set_index_streams(copy.deepcopy(start))
    _, again = ens.train_steps(4, mode="numpy", return_indices=True)
    assert torch.equal(first, again)
    torch.cuda.synchronize()
    before = ens.engine._mt_states.clone()
    ens.engine.set_replay_size(1, 0)
    with pytest.raises(ValueError, match="replay size 0"):
        ens.train_steps(4, mode="numpy")
    with pytest.raises(ValueError, match="replay size 0"):
        ens.train_step_logged(numpy_streams=True)
    ens.retire([1])  # a retired member's size is not checked
    ens.train_steps(4, mode="numpy")
    torch.cuda.synchronize()
    assert torch.equal(ens.engine._mt_states[1], before[1]) and not torch.equal(ens.engine._mt_states[0], before[0])


# ---------------------------------------------------------------------------
# 3. ensemble_train_loop on the device streams
# ---------------------------------------------------------------------------
def test_loop_on_device_streams_equals_host_draws(tmp_path):
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop
    from test_gpu_ensemble_online import B as LB, OFF, ON, PointEnv, _member_configs, _offline_buffer, _same

    rb = _offline_buffer()
    runs = []
    for device in (False, True):
        cfgs = _member_configs(False, tmp_path / f"dev{int(device)}")
        logs = {m: [] for m in range(4)}
        learner, cfgs, hist = ensemble_train_loop(cfgs, [PointEnv(100 + i) for i in range(4)],
                                                  [PointEnv(200 + i) for i in range(4)], rb, 3, 2, 1.0,
                                                  max_steps=PointEnv.T, log=lambda m, d, step: logs[m].append((step, d)),
                                                  device_index_streams=device)
        torch.cuda.synchronize()
        runs.append((learner, cfgs, hist, logs))
    (la, _, ha, ga), (lb, cfgs, hb, gb) = runs
    for m in range(4):
        assert _same(ga[m], gb[m]) and _same(ha[m], hb[m]), m
        for arena in ("params", "exp_avg", "exp_avg_sq", "target"):
            assert torch.equal(getattr(la.engine, arena)[m], getattr(lb.engine, arena)[m]), (m, arena)
        # the run's final RandomState: a host replay of its draws (offline at the dataset's size, online at the ring's)
        ref = np.random.RandomState(cfgs[m].seed)
        for _ in range(OFF - LB):
            ref.randint(0, rb._high(), size=LB)
        for k in range(ON):
            ref.randint(0, min(k + 1, cfgs[m].online_buffer_size), size=LB)
        assert np.array_equal(mt.state_row(lb.index_streams[m]), mt.state_row(ref)), m
