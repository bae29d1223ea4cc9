"""CPU: the segmented draw of numpy's global stream (oracle/np_stream.py, the algorithm of csrc/nprng.cu) against
np.random.randint itself: values and the generator state numpy is left in."""
import numpy as np
import pytest

from oracle import np_stream as ns

HIGHS = [1, 2, 6, 24, 120, 720, 5040, 40320, 2 ** 31 + 1, 2 ** 32]
POSES = [0, 1, 226, 227, 396, 623, 624]
NS = [0, 1, 623, 624, 625, 9000]


@pytest.fixture(scope="module")
def A():
    return ns.twist_matrix()


def state_at(seed, pos):
    r = np.random.RandomState(seed)
    key = r.randint(0, 2 ** 32, ns.N, dtype=np.uint64).astype(np.uint32)
    return ("MT19937", key, pos, 0, 0.0)


def numpy_draw(state, high, n):
    saved = np.random.get_state()
    try:
        np.random.set_state(state)
        v = np.random.randint(0, high, n)
        return v, np.random.get_state()
    finally:
        np.random.set_state(saved)


def same_state(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3] and a[4] == b[4]


def test_twist_matrix_is_the_twist(A):
    r = np.random.RandomState(3)
    for _ in range(4):
        key = r.randint(0, 2 ** 32, ns.N, dtype=np.uint64).astype(np.uint32)
        assert np.array_equal(ns.apply(A, key), ns.twist(key))


def test_twist_and_temper_are_numpys():
    np.random.seed(11)
    key = np.random.get_state()[1]
    words = np.random.randint(0, 2 ** 32, 2 * ns.N)            # high = 2^32: raw words
    assert np.array_equal(words[:ns.N], ns.temper(ns.twist(key)))
    assert np.array_equal(words[ns.N:], ns.temper(ns.twist(ns.twist(key))))


@pytest.mark.parametrize("high", HIGHS)
@pytest.mark.parametrize("pos", POSES)
def test_restatement_equals_numpy(A, high, pos):
    for j, n in enumerate(NS):
        st = state_at(1000 * high % 997 + 10 * pos + j, pos)
        want, want_state = numpy_draw(st, high, n)
        got, got_state = ns.randint(st, high, n, A)
        assert got.dtype == want.dtype and np.array_equal(got, want), (high, pos, n)
        assert same_state(got_state, want_state), (high, pos, n)


def test_consecutive_calls_and_gauss_cache(A):
    np.random.seed(5)
    np.random.standard_normal()                                 # has_gauss = 1, cached value kept
    st = np.random.get_state()
    assert st[3] == 1
    got_state, got = st, []
    for high, n in [(24, 700), (720, 3000), (2, 1), (6, 5000), (1, 9), (40320, 1300)]:
        v, got_state = ns.randint(got_state, high, n, A)
        got.append(v)
    np.random.set_state(st)
    want = [np.random.randint(0, h, n) for h, n in [(24, 700), (720, 3000), (2, 1), (6, 5000), (1, 9), (40320, 1300)]]
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    assert same_state(got_state, np.random.get_state())


def test_bad_high():
    st = state_at(0, 624)
    for bad in (0, -3, 2 ** 32 + 1):
        with pytest.raises(ValueError):
            ns.randint(st, bad, 4, None)
