"""CPU checks of the drop-in boundary: the C-ABI library loads, exports every
symbol include/iql_b200.h declares, rejects bad arguments with the documented
codes, and lays parameters out in the reference's checkpoint order/shapes.
No kernel is launched here."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from jsrl_corl_b200 import _lib
from jsrl_corl_b200.engine import linear_indices, query_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "iql_b200.h")).read()
    declared = set(re.findall(r"\b(iql_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    L = _lib.lib()
    for name in declared:
        assert hasattr(L, name)
    assert b"sm_100a" in L.iql_version()


def test_struct_sizes_match_header_expectations():
    assert C.sizeof(_lib.Config) == 16 * 4
    assert C.sizeof(_lib.HParams) == 12 * 8 + 16
    assert C.sizeof(_lib.Counters) == 6 * 8
    assert C.sizeof(_lib.RowLayout) == 8 * 4
    assert C.sizeof(_lib.TensorInfo) == 6 * 4 + 8


def test_create_rejects_bad_config_with_value_error():
    L = _lib.lib()
    h = C.c_void_p()
    for bad in (dict(n_members=0), dict(hidden_dim=30), dict(n_hidden=0), dict(math_mode=7), dict(batch_size=0)):
        kw = dict(n_members=1, state_dim=3, action_dim=2, hidden_dim=32, n_hidden=2, batch_size=8, deterministic=0,
                  math_mode=0, max_steps_per_call=4)
        kw.update(bad)
        cfg = _lib.Config(**kw)
        rc = L.iql_create(C.byref(cfg), C.byref(h))
        assert rc == _lib.IQL_ERR_INVALID
        with pytest.raises(ValueError):
            _lib.check(rc, None, "iql_create")
    assert L.iql_create(None, C.byref(h)) == _lib.IQL_ERR_INVALID


def test_calls_before_bind_fail_loudly():
    L = _lib.lib()
    h = C.c_void_p()
    cfg = _lib.Config(1, 3, 2, 32, 2, 8, 0, 0, 4)
    assert L.iql_create(C.byref(cfg), C.byref(h)) == 0
    try:
        rc = L.iql_train_steps(h, 1, 0, None, None, None, None, None)
        assert rc == _lib.IQL_ERR_STATE
        assert b"not bound" in L.iql_last_error(h)
        hp = _lib.HParams(actor_dropout=1.5)
        assert L.iql_set_hparams(h, 0, C.byref(hp)) == _lib.IQL_ERR_INVALID
        assert L.iql_set_hparams(h, 3, C.byref(hp)) == _lib.IQL_ERR_INVALID
        assert L.iql_bind_replay(h, 0, None, 10, 0) == _lib.IQL_ERR_INVALID
    finally:
        L.iql_destroy(h)


@pytest.mark.parametrize("S,A,H,L,det,dropout", [(11, 3, 256, 2, True, 0.0), (29, 8, 256, 3, False, 0.0),
                                                 (45, 24, 256, 2, False, 0.1), (11, 3, 1024, 4, True, 0.0)])
def test_layout_follows_reference_checkpoint_order(S, A, H, L, det, dropout):
    import jsrl_corl_b200 as J

    lay, tensors = query_layout(1, S, A, H, L, 256, det)
    q = J.TwinQ(S, A, H, L)
    v = J.ValueFunction(S, H, L)
    actor = (J.DeterministicPolicy if det else J.GaussianPolicy)(S, A, 1.0, H, L, dropout=dropout)
    expected = []  # optimizer parameter order == module.parameters() order (log_std first for the Gaussian actor)
    for mod in (q, v, actor):
        expected += [tuple(p.shape) for p in mod.parameters()]
    got = [(r, c) if kind == _lib.KIND_WEIGHT else (r,) for (_, _, kind, r, c, _, _) in tensors]
    assert all(ld % 4 == 0 and ld >= c for (_, _, kind, r, c, _, ld) in tensors if kind == _lib.KIND_WEIGHT)
    assert got == expected
    offs = [t[5] for t in tensors]
    assert offs == sorted(offs) and all(o % 32 == 0 for o in offs)  # 128-byte aligned tensors
    assert lay.q_floats == lay.v_begin and lay.v_end == lay.actor_begin and lay.actor_end == lay.param_floats
    n_q = sum(p.numel() for p in q.parameters())
    assert lay.q_floats >= n_q and lay.q_floats - n_q < (32 + 3 * H) * len(list(q.parameters()))
    # dropout shifts the Sequential indices to 0,3,6 (reference iql.py:329-333)
    idx = linear_indices(L, dropout > 0)
    assert [k for k in actor.state_dict() if k.endswith("weight")] == [f"net.net.{i}.weight" for i in idx]


def test_row_layout_is_16_byte_segmented():
    L = _lib.lib()
    for S, A, rf in ((11, 3, 32), (17, 6, 44), (29, 8, 72), (45, 24, 120)):
        lay = _lib.RowLayout()
        assert L.iql_replay_row_layout(S, A, C.byref(lay)) == 0
        assert lay.row_floats == rf and lay.row_floats % 4 == 0 and lay.off_next_state % 4 == 0
        assert lay.off_action == S and lay.off_reward == lay.off_next_state + S and lay.off_done == lay.off_reward + 1
    assert L.iql_replay_row_layout(0, 3, C.byref(lay)) == _lib.IQL_ERR_INVALID


def test_product_path_fails_loudly_without_cuda():
    import jsrl_corl_b200 as J

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        J.ReplayBuffer(3, 2, 10, "cpu")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        J.EnsembleEngine(1, 3, 2, 32, 2, 8)
    q, v, a = J.TwinQ(3, 2, 32), J.ValueFunction(3, 32), J.GaussianPolicy(3, 2, 1.0, 32)
    opts = [torch.optim.Adam(m.parameters()) for m in (a, q, v)]
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        J.ImplicitQLearning(1.0, a, opts[0], q, opts[1], v, opts[2], device="cpu")


def test_product_package_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "jsrl_corl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                for pat in (r"^\s*(from|import)\s+oracle", r"oracle[./]_build", r"libphilox_ref", r"iql_numpy"):
                    assert not re.search(pat, text, flags=re.M), (f, pat)


def test_synthetic_dataset_matches_oracle_copy():
    from jsrl_corl_b200.synthetic import synthetic_dataset as a
    from oracle.iql_numpy import synthetic_dataset as b

    for kw in (dict(n=100, state_dim=5, action_dim=2, seed=3), dict(n=50, state_dim=29, action_dim=8, seed=0, antmaze_rewards=True)):
        x, y = a(**kw), b(**kw)
        for k in x:
            assert np.array_equal(x[k], y[k])


def test_train_config_fields_match_reference_dataclasses():
    """TrainConfig / OfflineTrainConfig / JsrlTrainConfig keep the reference's field names and defaults
    (iql.py:32-69, offline/iql.py:30-80, jsrl_w_iql.py:46-60)."""
    import dataclasses

    import jsrl_corl_b200 as J
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from oracle.ref_loader import load_reference_iql, reference_available

    def fields(cls):
        return {f.name: f.default for f in dataclasses.fields(cls) if f.default is not dataclasses.MISSING}

    assert set(fields(J.TrainConfig)) < set(f.name for f in dataclasses.fields(JsrlTrainConfig))
    # offline variant: a Dropout module exists whenever dropout is not None (even 0.0): keys 0,3,6
    pol = J.GaussianPolicy(4, 2, 1.0, 16, 2, dropout=0.0, dropout_when_not_none=True)
    assert [k for k in pol.state_dict() if k.endswith("weight")] == ["net.net.0.weight", "net.net.3.weight", "net.net.6.weight"]
    if not reference_available():
        pytest.skip("needs the original jsrl-CORL source under JSRL_REFERENCE_ROOT; no stored outputs of it exist for this comparison")
    assert fields(J.TrainConfig) == fields(load_reference_iql("finetune").TrainConfig)
    assert fields(J.OfflineTrainConfig) == fields(load_reference_iql("offline").TrainConfig)
    ref_pol = load_reference_iql("offline").GaussianPolicy(4, 2, 1.0, 16, 2, dropout=0.0)
    assert list(pol.state_dict().keys()) == list(ref_pol.state_dict().keys())
    ref_fin = load_reference_iql("finetune").GaussianPolicy(4, 2, 1.0, 16, 2, dropout=0.0)
    assert list(J.GaussianPolicy(4, 2, 1.0, 16, 2, dropout=0.0).state_dict().keys()) == list(ref_fin.state_dict().keys())


def test_options_and_path_info_without_a_gpu():
    """iql_set_option / iql_get_info (include/iql_b200.h): argument checking and the pre-bind answers; the step path must
    be chosen before the state is bound, unknown keys are refused, the tensor-core answer follows the shape rule."""
    L = _lib.lib()

    def handle(batch, hidden, math):
        h = C.c_void_p()
        cfg = _lib.Config(1, 17, 6, hidden, 2, batch, 0, math, 4)
        _lib.check(L.iql_create(C.byref(cfg), C.byref(h)), None, "iql_create")
        return h

    h = handle(256, 256, _lib.MATH_TF32_TCGEN05)
    try:
        out = C.c_int64(-1)
        assert L.iql_get_info(h, _lib.INFO_TENSOR_CORE_PATH, C.byref(out)) == _lib.IQL_OK and out.value == 1
        assert L.iql_get_info(h, _lib.INFO_CHAINED_BACKWARD, C.byref(out)) == _lib.IQL_OK and out.value == 0  # not bound yet
        assert L.iql_get_info(h, 99, C.byref(out)) == _lib.IQL_ERR_INVALID
        assert L.iql_get_info(h, _lib.INFO_FUSED_FORWARD, None) == _lib.IQL_ERR_INVALID
        for v in (0, 1, 2):
            assert L.iql_set_option(h, _lib.OPT_STEP_PATH, v) == _lib.IQL_OK
        assert L.iql_set_option(h, _lib.OPT_STEP_PATH, 3) == _lib.IQL_ERR_INVALID
        assert b"IQL_OPT_STEP_PATH" in L.iql_last_error(h)
        assert L.iql_set_option(h, 77, 1) == _lib.IQL_ERR_INVALID
        assert L.iql_set_option(h, _lib.OPT_KEEP_GRADS, 1) == _lib.IQL_OK
    finally:
        L.iql_destroy(h)
    for batch, hidden, math, want in ((100, 256, _lib.MATH_TF32_TCGEN05, 0), (256, 64, _lib.MATH_TF32_TCGEN05, 0),
                                      (256, 256, _lib.MATH_FP32_SIMT, 0), (4096, 1024, _lib.MATH_TF32_TCGEN05, 1)):
        h = handle(batch, hidden, math)
        try:
            out = C.c_int64(-1)
            assert L.iql_get_info(h, _lib.INFO_TENSOR_CORE_PATH, C.byref(out)) == _lib.IQL_OK and out.value == want, (batch, hidden)
        finally:
            L.iql_destroy(h)


def test_replay_ingest_rejects_bad_arguments():
    L = _lib.lib()
    lay = _lib.RowLayout()
    assert L.iql_replay_row_layout(11, 3, C.byref(lay)) == _lib.IQL_OK
    assert L.iql_replay_ingest(None, C.byref(lay), 0, 4, None, None, None, None, None, 1, 1e-3, None, None, 1.0, 1.0, 0.0, None) == _lib.IQL_ERR_INVALID
    bad = _lib.RowLayout()
    assert L.iql_replay_ingest(1, C.byref(bad), 0, 4, 1, 1, 1, 1, 1, 0, 1e-3, None, None, 1.0, 1.0, 0.0, None) == _lib.IQL_ERR_INVALID
    # n == 0 is a no-op that succeeds (an empty dataset), before any pointer is dereferenced
    assert L.iql_replay_ingest(1, C.byref(lay), 0, 0, None, None, None, None, None, 0, 1e-3, None, None, 1.0, 1.0, 0.0, None) == _lib.IQL_OK


def test_host_step_and_host_sample_reject_bad_arguments():
    """iql_train_host_step / iql_replay_sample_host (the per-step host loop of offline/iql.py:631-635) check their
    arguments before touching the GPU."""
    L = _lib.lib()
    out = (C.c_float * 3)()
    assert L.iql_train_host_step(None, None, out, None, None) == _lib.IQL_ERR_INVALID
    cfg = _lib.Config(1, 11, 3, 256, 2, 256, 1, _lib.MATH_FP32_SIMT, 4)
    h = C.c_void_p()
    assert L.iql_create(C.byref(cfg), C.byref(h)) == _lib.IQL_OK
    try:
        assert L.iql_train_host_step(h, None, out, 1, 1) == _lib.IQL_ERR_STATE  # nothing bound yet
        assert b"not bound" in L.iql_last_error(h)
    finally:
        L.iql_destroy(h)
    lay = _lib.RowLayout()
    assert L.iql_replay_row_layout(11, 3, C.byref(lay)) == _lib.IQL_OK
    idx = (C.c_int64 * 4)(0, 1, 2, 3)
    assert L.iql_replay_sample_host(None, C.byref(lay), 10, 4, idx, 1, 1, 1, 1, 1, None) == _lib.IQL_ERR_INVALID
    assert L.iql_replay_sample_host(1, C.byref(lay), 0, 4, idx, 1, 1, 1, 1, 1, None) == _lib.IQL_ERR_INVALID  # empty buffer
    assert L.iql_replay_sample_host(1, C.byref(lay), 10, 4, None, 1, 1, 1, 1, 1, None) == _lib.IQL_ERR_INVALID
    assert L.iql_replay_sample_host(1, C.byref(lay), 3, 4, idx, 1, 1, 1, 1, 1, None) == _lib.IQL_ERR_INVALID  # index 3 >= size 3
    assert L.iql_replay_sample_host(1, C.byref(lay), 10, 0, None, None, None, None, None, None, None) == _lib.IQL_OK


def test_debug_hooks_are_inert_without_their_switches():
    """The trace hooks (fused forward, chained backward, step timeline) report 'off' unless their debug switches are set."""
    L = _lib.lib()
    buf = (C.c_ulonglong * 64)()
    assert L.iql_debug_step_trace(None, 0, buf, 64, None) < 0
    cfg = _lib.Config(1, 11, 3, 256, 2, 256, 1, _lib.MATH_FP32_SIMT, 4)
    h = C.c_void_p()
    assert L.iql_create(C.byref(cfg), C.byref(h)) == _lib.IQL_OK
    try:
        assert L.iql_debug_step_trace(h, 1, None, 0, None) < 0  # no stamp buffer: IQL_STEP_TRACE is not set
        assert L.iql_host_step_wait(h, (C.c_float * 3)(), None) == _lib.IQL_ERR_STATE  # nothing in flight
        assert L.iql_act_host(h, 0, (C.c_float * 11)(), 1.0, (C.c_float * 3)(), None, None) == _lib.IQL_ERR_STATE  # not bound
        assert L.iql_act_host(h, 5, (C.c_float * 11)(), 1.0, (C.c_float * 3)(), None, None) == _lib.IQL_ERR_INVALID
    finally:
        L.iql_destroy(h)
    lay = _lib.RowLayout()
    assert L.iql_replay_row_layout(600, 8, C.byref(lay)) == _lib.IQL_OK and lay.row_floats > 960
    z = (C.c_float * 600)()
    assert L.iql_replay_insert_host(1, C.byref(lay), 0, z, z, 0.0, z, 0.0, None) == _lib.IQL_ERR_SHAPE  # too wide for the by-value row
    assert L.iql_replay_insert_host(None, C.byref(lay), 0, z, z, 0.0, z, 0.0, None) == _lib.IQL_ERR_INVALID
