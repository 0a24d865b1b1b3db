"""numpy restatement of the legacy ``RandomState.randint(0, high, size=n)`` (int64) stream that the engine's MT19937
sampler reproduces (include/iql_b200.h, IQL_SAMPLE_MT19937), written in the sampler's terms: a lazy twist in three
dependent phases, then every unread word of a key block tempered, masked and tested at once, the accepted words kept
in stream order.  Works on the device state layout: uint32 words [key[624] | pos | pad]."""
import numpy as np

N, M = 624, 397
STATE_WORDS = 626  # IQL_MT_STATE_WORDS


def state_row(rng: np.random.RandomState) -> np.ndarray:
    """The device layout of a RandomState's generator: key[624], pos, pad."""
    name, key, pos, _, _ = rng.get_state()
    assert name == "MT19937"
    row = np.zeros(STATE_WORDS, dtype=np.uint32)
    row[:N] = key
    row[N] = pos
    return row


def load_row(rng: np.random.RandomState, row: np.ndarray) -> None:
    """Write key and pos back into ``rng``; its cached Gaussian (has_gauss, cached_gaussian) is kept."""
    _, _, _, has_gauss, cached = rng.get_state()
    rng.set_state(("MT19937", np.asarray(row[:N], dtype=np.uint32), int(row[N]), has_gauss, cached))


def twist(key: np.ndarray) -> np.ndarray:
    k = key.astype(np.uint32).copy()

    def words(i, nxt, far):
        y = (k[i] & np.uint32(0x80000000)) | (k[nxt] & np.uint32(0x7FFFFFFF))
        return k[far] ^ (y >> np.uint32(1)) ^ np.where(y & np.uint32(1), np.uint32(0x9908B0DF), np.uint32(0))

    i = np.arange(0, N - M)
    k[i] = words(i, i + 1, i + M)
    i = np.arange(N - M, 2 * (N - M))
    k[i] = words(i, i + 1, i - (N - M))
    i = np.arange(2 * (N - M), N)
    k[i] = words(i, (i + 1) % N, i - (N - M))
    return k


def temper(y: np.ndarray) -> np.ndarray:
    y = y.astype(np.uint32)
    y = y ^ (y >> np.uint32(11))
    y = y ^ ((y << np.uint32(7)) & np.uint32(0x9D2C5680))
    y = y ^ ((y << np.uint32(15)) & np.uint32(0xEFC60000))
    return y ^ (y >> np.uint32(18))


def randint(row: np.ndarray, high: int, n: int):
    """(draws int64 [n], new state row) of randint(0, high, size=n) from state ``row``; 1 <= high <= 2^32."""
    if not 1 <= high <= 1 << 32:
        raise ValueError("high must lie in [1, 2^32]")
    row = np.asarray(row, dtype=np.uint32).copy()
    rng = high - 1
    if rng == 0 or n == 0:
        return np.zeros(n, dtype=np.int64), row
    mask = (1 << int(rng).bit_length()) - 1
    key, pos = row[:N], int(row[N])
    out = np.empty(n, dtype=np.int64)
    done = 0
    while done < n:
        if pos == N:
            key = twist(key)
            pos = 0
        v = temper(key[pos:]).astype(np.int64) & mask
        acc = np.flatnonzero(v <= rng)
        take = acc[: n - done]
        out[done:done + take.size] = v[take]
        done += take.size
        pos = pos + int(take[-1]) + 1 if done == n else N
    row[:N] = key
    row[N] = pos
    return out, row
