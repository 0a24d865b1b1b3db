"""The numpy index stream of IQL_SAMPLE_MT19937 without a GPU: the restatement the device sampler follows, checked
against numpy itself (outputs and get_state()) across the bound and block edges; the get_state() <-> device-layout
round trip; and the argument checks of the new entry points."""
import ctypes as C

import numpy as np
import pytest

from jsrl_corl_b200 import _lib
import mt19937_oracle as mt

EDGE_HIGHS = [1, 2, 3, 10 ** 4, 2 ** 16, 2 ** 16 + 1, 10 ** 6, 2 ** 31, 2 ** 31 + 1, 2 ** 32 - 1, 2 ** 32]


def _same_state(rng_a, row):
    _, key, pos, _, _ = rng_a.get_state()
    return np.array_equal(key, row[:624]) and pos == int(row[624])


@pytest.mark.parametrize("high", EDGE_HIGHS + [2 ** k for k in (1, 5, 12, 20, 27)] + [2 ** k + 1 for k in (1, 5, 12, 20, 27)])
def test_restatement_matches_numpy_over_three_calls(high):
    ref = np.random.RandomState(1234 + high % 97)
    row = mt.state_row(ref)
    for n in (1, 700, 2000):  # crosses 624-word blocks
        want = ref.randint(0, high, size=n)
        got, row = mt.randint(row, high, n)
        assert got.dtype == np.int64 and np.array_equal(got, want)
        assert _same_state(ref, row)


def test_k_calls_equal_one_call():
    a, b = np.random.RandomState(5), np.random.RandomState(5)
    joined = np.concatenate([a.randint(0, 10000, size=256) for _ in range(7)])
    assert np.array_equal(joined, b.randint(0, 10000, size=7 * 256))
    assert _same_state(a, mt.state_row(b))


def test_lazy_twist_ends_on_word_623():
    # high 2^32 accepts every word: 624 - pos draws end exactly on word 623, leaving pos = 624 and the key untwisted
    for start in (0, 100, 623):
        ref = np.random.RandomState(9)
        ref.set_state(("MT19937", ref.get_state()[1], start))  # a fresh RandomState stands at pos 624
        row = mt.state_row(ref)
        key0 = row[:624].copy()
        got, row = mt.randint(row, 2 ** 32, 624 - start)
        assert np.array_equal(got, ref.randint(0, 2 ** 32, size=624 - start))
        assert int(row[624]) == 624 and ref.get_state()[2] == 624 and np.array_equal(row[:624], key0)
        got, row = mt.randint(row, 2 ** 32, 5)  # the next draw twists first
        assert np.array_equal(got, ref.randint(0, 2 ** 32, size=5)) and _same_state(ref, row)


def test_high_one_consumes_nothing():
    ref = np.random.RandomState(3)
    ref.randint(0, 7, size=11)
    row = mt.state_row(ref)
    got, row2 = mt.randint(row, 1, 50)
    assert np.array_equal(got, ref.randint(0, 1, size=50)) and np.array_equal(row, row2) and _same_state(ref, row2)


def test_state_round_trip_keeps_the_cached_gaussian():
    rng = np.random.RandomState(11)
    rng.standard_normal()  # leaves has_gauss = 1 and a cached value
    _, _, _, has_gauss, cached = rng.get_state()
    assert has_gauss == 1
    row = mt.state_row(rng)
    assert row.dtype == np.uint32 and row.shape == (_lib.MT_STATE_WORDS,)
    advanced, row = mt.randint(row, 1000, 900)
    mt.load_row(rng, row)
    st = rng.get_state()
    assert st[3] == has_gauss and st[4] == cached and _same_state(rng, row)
    twin = np.random.RandomState(11)
    twin.standard_normal()
    assert np.array_equal(advanced, twin.randint(0, 1000, size=900))
    assert np.array_equal(rng.randint(0, 1000, size=10), twin.randint(0, 1000, size=10))


def test_facade_state_rows_are_the_oracle_layout():
    from jsrl_corl_b200.engine import index_state_rows, load_index_state_rows

    rngs = [np.random.RandomState(s) for s in (0, 1, 2)]
    rngs[1].randint(0, 5, size=100)
    rows = index_state_rows(rngs)
    assert rows.dtype == np.uint32 and rows.shape == (3, _lib.MT_STATE_WORDS)
    for r, row in zip(rngs, rows):
        assert np.array_equal(row, mt.state_row(r))
    rows[0] = mt.randint(rows[0], 10, 3)[1]
    load_index_state_rows(rngs, rows)
    assert _same_state(rngs[0], rows[0])
    with pytest.raises(ValueError):
        index_state_rows([np.random.default_rng(0)])


def test_entry_points_check_arguments_without_a_device():
    L = _lib.lib()
    hi = (C.c_int64 * 2)(10, 1 << 33)
    cnt = (C.c_int64 * 2)(4, 4)
    # bad bound, null arrays and a stride below a count are refused before anything is launched
    assert L.iql_mt19937_randint(C.c_void_p(256), 2, hi, cnt, C.c_void_p(256), 4, None) == _lib.IQL_ERR_INVALID
    hi[1] = 0
    assert L.iql_mt19937_randint(C.c_void_p(256), 2, hi, cnt, C.c_void_p(256), 4, None) == _lib.IQL_ERR_INVALID
    hi[1] = 10
    assert L.iql_mt19937_randint(None, 2, hi, cnt, C.c_void_p(256), 4, None) == _lib.IQL_ERR_INVALID
    assert L.iql_mt19937_randint(C.c_void_p(256), 2, hi, cnt, C.c_void_p(256), 3, None) == _lib.IQL_ERR_INVALID
    assert L.iql_mt19937_randint(C.c_void_p(256), 0, hi, cnt, None, 0, None) == _lib.IQL_OK
    # a handle before bind: streams may be bound (host pointers only), steps are refused
    cfg = _lib.Config(2, 17, 6, 256, 2, 256, 0, _lib.MATH_FP32_SIMT, 4)
    h = C.c_void_p()
    _lib.check(L.iql_create(C.byref(cfg), C.byref(h)))
    try:
        assert L.iql_bind_index_streams(h, C.c_void_p(256), None) == _lib.IQL_ERR_INVALID
        assert L.iql_bind_index_streams(h, C.c_void_p(260), C.c_void_p(256)) == _lib.IQL_ERR_INVALID
        assert L.iql_bind_index_streams(h, C.c_void_p(256), C.c_void_p(264)) == _lib.IQL_ERR_INVALID
        assert L.iql_bind_index_streams(h, C.c_void_p(256), C.c_void_p(256)) == _lib.IQL_OK
        assert L.iql_bind_index_streams(h, None, None) == _lib.IQL_OK
        assert L.iql_train_steps(h, 1, _lib.SAMPLE_MT19937, None, None, None, None, None) == _lib.IQL_ERR_STATE
        assert L.iql_train_host_step_mt19937(h, None, None, None) == _lib.IQL_ERR_STATE
        assert L.iql_train_host_step_mt19937(None, None, None, None) == _lib.IQL_ERR_INVALID
    finally:
        L.iql_destroy(h)
