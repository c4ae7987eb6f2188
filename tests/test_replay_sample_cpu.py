"""CPU: the formulations hmz_replay_sample evaluates in parallel, restated in oracle/replay_ref.py, against NumPy bit for
bit — the pairwise float32 sum (np.sum), the stretch-wise exact float64 cumulative sum (np.cumsum) and the whole
index / weight chain of ReplayRing.priority_sample (np.random.choice) — and the new entry points' argument checks."""
import ctypes

import numpy as np
import pytest

from oracle import replay_ref as R

SIZES = list(range(1, 301)) + [1023, 1024, 1025, 8191, 8192, 8193, 100003]


def heavy_tailed(rng, n, zero_fraction=0.0):
    """Priorities spanning 1e-12 to 1e3 (log-uniform), a fraction of them zero rows."""
    q = (10.0 ** rng.uniform(-12, 3, n)).astype(np.float32)
    if zero_fraction:
        q[rng.random(n) < zero_fraction] = 0
    return q


def same_bits(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def test_pairwise_sum_matches_np_sum():
    rng = np.random.default_rng(1)
    bad = []
    for n in SIZES:
        for q in (heavy_tailed(rng, n), heavy_tailed(rng, n, 0.3), rng.random(n, dtype=np.float32)):
            if not same_bits(R.pairwise_sum(q), np.sum(q)):
                bad.append(n)
    assert not bad, bad[:10]


def test_pairwise_sum_at_a_million_rows():
    rng = np.random.default_rng(2)
    for n in (1048576, 1048579):
        q = heavy_tailed(rng, n, 0.01)
        assert same_bits(R.pairwise_sum(q), np.sum(q))


def test_exact_cumsum_matches_np_cumsum():
    rng = np.random.default_rng(3)
    bad = []
    for n in SIZES:
        for zf in (0.0, 0.3):
            q = heavy_tailed(rng, n, zf)
            q[: rng.integers(0, 4)] = 0  # leading zero rows
            if not np.sum(q) > 0:
                continue
            x = (q / np.sum(q)).astype(np.float32)
            for chunk in (R.CHUNK, 64):  # also stretches and chunks that end inside each other
                cdf, _ = R.exact_cumsum(x, chunk)
                if not same_bits(cdf, np.cumsum(x.astype(np.float64))):
                    bad.append((n, zf, chunk))
    assert not bad, bad[:10]


@pytest.mark.parametrize("n", [300, 8193, 100003])
def test_constructed_rings_with_ties_and_rounding_up_crossings(n):
    q = R.constructed_ring(n, seed=n)
    s = np.sum(q)
    assert np.frexp(s)[0] == 0.5, "the ring's sum must be a power of two"
    x = (q / s).astype(np.float32)
    assert same_bits(x, (q.astype(np.float64) / float(s)).astype(np.float32))  # q / s scaled every row exactly
    for chunk in (R.CHUNK, 97):
        cdf, info = R.exact_cumsum(x, chunk)
        assert same_bits(cdf, np.cumsum(x.astype(np.float64)))
    assert info["ties"] >= n // 5 and info["roundup"] >= 15 and info["stretches"] >= 20, info
    # a tree-ordered float64 sum does not reproduce these rings
    assert not same_bits(np.add.reduce(x.astype(np.float64)), cdf[-1]) or n < 1000


def numpy_priority_sample(q, size, beta, seed, batch):
    """ReplayRing.priority_sample's NumPy part on host priorities."""
    np.random.seed(seed)
    p = q ** 1
    probs = p / np.sum(p)
    idx = np.random.choice(np.arange(len(q)), size=batch, replace=True, p=probs).astype(np.int64)
    w = ((1.0 / size) / probs[idx]) ** beta
    w /= np.max(w)
    return idx, w.astype(np.float32)


@pytest.mark.parametrize("beta", [0, 0.5])
def test_whole_chain_matches_np_random_choice(beta):
    rng = np.random.default_rng(4)
    for n in (1, 2, 7, 129, 1000, 50000):
        for q in (heavy_tailed(rng, n, 0.2 if n > 2 else 0.0) + np.float32(n <= 2), R.constructed_ring(max(n, 2), n)[:n]):
            if not np.sum(q) > 0:
                continue
            size = n + 17
            idx, w = numpy_priority_sample(q, size, beta, seed=n, batch=256)
            np.random.seed(n)
            u = np.random.random_sample(256)
            idx2, w2 = R.sample(q, size, u, beta)
            assert np.array_equal(idx, idx2), n
            assert same_bits(w, w2), n


def test_uniform_replay_draw_is_randint():
    for num in (1, 5, 50000):
        np.random.seed(num)
        a = np.random.choice(np.arange(num), size=256, replace=True)
        x = np.random.random_sample()
        np.random.seed(num)
        b = np.random.randint(0, num, 256)
        assert np.array_equal(a, b) and np.random.random_sample() == x


@pytest.mark.parametrize("case,message", [
    ("zeros", "probabilities contain NaN"),
    ("nan", "probabilities contain NaN"),
    ("negative", "probabilities are not non-negative"),
    ("overflow", "probabilities do not sum to 1"),
])
def test_rejected_rings_raise_numpys_errors(case, message):
    q = np.linspace(0.1, 1, 100).astype(np.float32)
    if case == "zeros":
        q[:] = 0
    elif case == "nan":
        q[7] = np.nan
    elif case == "negative":
        q[3] = -0.5
    else:
        q[:] = 3e38  # the float32 sum overflows: every probability is 0
    with np.errstate(all="ignore"):
        with pytest.raises(ValueError, match=message):
            numpy_priority_sample(q, 100, 0, 0, 8)
        with pytest.raises(ValueError, match=message):
            R.sample(q, 100, np.random.random_sample(8), 0)


def test_entry_points_reject_bad_arguments_before_any_cuda_call(lib):
    from muzero_hanoi_b200 import _lib

    host = (ctypes.c_double * 64)()
    p = ctypes.cast(host, ctypes.c_void_p)
    assert lib.hmz_replay_sample_workspace_bytes(0) == 0
    assert lib.hmz_replay_sample_workspace_bytes(50000) >= 50000 * 8
    args = dict(priorities=p, num=10, size=10, pexp=1.0, u=p, batch=4, beta=0.0, ws=p, idx=p, w=p, status=p)

    def call(**kw):
        a = {**args, **kw}
        return lib.hmz_replay_sample(a["priorities"], a["num"], a["size"], a["pexp"], a["u"], a["batch"], a["beta"], a["ws"], a["idx"],
                                     a["w"], a["status"], None)

    for bad in (dict(priorities=None), dict(u=None), dict(ws=None), dict(idx=None), dict(w=None), dict(status=None),
                dict(num=0), dict(num=-3), dict(size=9), dict(batch=0), dict(beta=float("nan"))):
        assert call(**bad) == _lib.ERR_INVALID, bad
    assert call(pexp=0.5) == _lib.ERR_UNSUPPORTED and b"exponent" in lib.hmz_last_error()
    assert call(num=(1 << 27) + 1, size=(1 << 27) + 1) == _lib.ERR_UNSUPPORTED
    for bad in ((None, 10, p, p, 4, p), (p, 10, None, p, 4, p), (p, 10, p, None, 4, p), (p, 10, p, p, 4, None), (p, 0, p, p, 4, p),
                (p, 10, p, p, 0, p)):
        assert lib.hmz_replay_set_priorities(*bad, None) == _lib.ERR_INVALID, bad
