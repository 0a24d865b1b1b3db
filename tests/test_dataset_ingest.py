"""SURVEY.md section 8 (f-4): dataset ingest + normalisation.

CPU: the facade's ``compute_mean_std`` / ``normalize_states`` / ``return_reward_range`` / ``modify_reward`` /
``modify_reward_online`` against the reference's own functions (finetune/iql.py:77-84, 262-306) on episodic synthetic data.
GPU: ``ReplayBuffer.ingest_d4rl_dataset`` (mean / std / normalise / reward rescale / pack in one device pass) bit-exact
against that numpy pipeline followed by ``load_d4rl_dataset``."""
import numpy as np
import pytest


def _episodic(n=5000, S=7, A=3, seed=0, p_term=0.004):
    rng = np.random.RandomState(seed)
    return {"observations": (rng.randn(n, S) * rng.uniform(0.1, 5, S) + rng.uniform(-3, 3, S)).astype(np.float32),
            "actions": rng.uniform(-1, 1, (n, A)).astype(np.float32),
            "rewards": rng.uniform(-1, 2, n).astype(np.float32),
            "next_observations": (rng.randn(n, S) * 2).astype(np.float32),
            "terminals": rng.uniform(size=n) < p_term}


def _copy(d):
    return {k: v.copy() for k, v in d.items()}


def test_preprocessing_functions_match_the_reference():
    from oracle.ref_loader import load_reference_iql, reference_available

    if not reference_available():
        pytest.skip("needs the original jsrl-CORL source under JSRL_REFERENCE_ROOT; no stored outputs of it exist for this comparison")
    ref = load_reference_iql("finetune")
    from jsrl_corl_b200 import iql as ours

    data = _episodic()
    m1, s1 = ref.compute_mean_std(data["observations"], eps=1e-3)
    m2, s2 = ours.compute_mean_std(data["observations"], eps=1e-3)
    np.testing.assert_array_equal(m1, m2)
    np.testing.assert_array_equal(s1, s2)
    np.testing.assert_array_equal(ref.normalize_states(data["observations"], m1, s1), ours.normalize_states(data["observations"], m2, s2))
    for steps in (1000, 137):
        assert ref.return_reward_range(data, steps) == ours.return_reward_range(data, steps)
    for env in ("hopper-medium-v2", "halfcheetah-medium-replay-v2", "walker2d-expert-v2", "antmaze-umaze-v2", "pen-human-v1"):
        a, b = _copy(data), _copy(data)
        ka, kb = ref.modify_reward(a, env), ours.modify_reward(b, env)
        assert ka == kb
        np.testing.assert_array_equal(a["rewards"], b["rewards"])
        for r in (0.0, 1.0, -0.3):
            assert ref.modify_reward_online(r, env, **ka) == ours.modify_reward_online(r, env, **kb)
    assert ref.ENVS_WITH_GOAL == ours.ENVS_WITH_GOAL and ref.EXP_ADV_MAX == ours.EXP_ADV_MAX


@pytest.mark.gpu
@pytest.mark.parametrize("env,normalize,normalize_reward", [("hopper-medium-v2", True, True), ("antmaze-umaze-v2", True, True),
                                                            ("pen-human-v1", False, False), ("halfcheetah-medium-v2", True, False)])
def test_device_ingest_bit_exact_against_numpy_pipeline(env, normalize, normalize_reward):
    import torch

    from jsrl_corl_b200 import ReplayBuffer
    from jsrl_corl_b200 import iql as ours
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from jsrl_corl_b200.jsrl_w_iql import make_offline_buffer

    data = _episodic(n=20011, S=11, A=3, seed=3)
    # the reference pipeline on the host (jsrl_w_iql.py:344-368), then the plain load
    host = _copy(data)
    mod = ours.modify_reward(host, env) if normalize_reward else {}
    mean, std = ours.compute_mean_std(host["observations"], eps=1e-3) if normalize else (0, 1)
    host["observations"] = ours.normalize_states(host["observations"], mean, std)
    host["next_observations"] = ours.normalize_states(host["next_observations"], mean, std)
    want = ReplayBuffer(11, 3, 30000, "cuda")
    want.load_d4rl_dataset(host)
    cfg = JsrlTrainConfig(device="cuda", env=env, normalize=normalize, normalize_reward=normalize_reward, buffer_size=30000)
    before = _copy(data)
    got, gmean, gstd, gmod = make_offline_buffer(cfg, data, 11, 3)
    for k in data:
        np.testing.assert_array_equal(data[k], before[k])  # the caller's dataset is left alone
    assert gmod == mod
    if normalize:
        np.testing.assert_array_equal(gmean, mean)
        np.testing.assert_array_equal(gstd, std)
    else:
        assert (gmean, gstd) == (0, 1)
    assert got._size == want._size == 20011 and got._pointer == want._pointer
    assert torch.equal(got.rows, want.rows)


def _fortran(d):
    """The same dataset with every 2-D array in Fortran order and the 1-D ones as strided column views."""
    out = {k: np.asfortranarray(v) for k, v in d.items()}
    for k in ("rewards", "terminals"):
        out[k] = np.asfortranarray(np.stack([d[k], d[k]], 1))[:, :1]
    return out


def test_dataset_tensors_are_dense_for_non_c_order_arrays():
    import torch

    from jsrl_corl_b200.iql import ReplayBuffer

    rb = object.__new__(ReplayBuffer)  # the host-side part of a buffer; no device is touched
    rb._device, rb._size, rb._buffer_size, rb._state_dim, rb._action_dim = torch.device("cpu"), 0, 100, 7, 3
    data = _episodic(n=50)
    got = rb._dataset_tensors(_fortran(data))
    for t, k in zip(got, ("observations", "actions", "rewards", "next_observations", "terminals")):
        assert t.is_contiguous(), k
        np.testing.assert_array_equal(t.numpy().reshape(data[k].shape), data[k].astype(np.float32))


@pytest.mark.gpu
def test_non_c_order_dataset_loads_like_c_order():
    import torch

    from jsrl_corl_b200 import ReplayBuffer

    data = _episodic(n=3001, S=11, A=3, seed=5)
    want, got = ReplayBuffer(11, 3, 4000, "cuda"), ReplayBuffer(11, 3, 4000, "cuda")
    want.load_d4rl_dataset(data)
    got.load_d4rl_dataset(_fortran(data))
    assert torch.equal(got.rows, want.rows)
    want, got = ReplayBuffer(11, 3, 4000, "cuda"), ReplayBuffer(11, 3, 4000, "cuda")
    m1, s1 = want.ingest_d4rl_dataset(data)
    m2, s2 = got.ingest_d4rl_dataset(_fortran(data))
    np.testing.assert_array_equal(m1, m2)
    np.testing.assert_array_equal(s1, s2)
    assert torch.equal(got.rows, want.rows)
