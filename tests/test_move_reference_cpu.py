"""oracle/move_ref.py, the restatement the self-play draws and the root policy are checked against on the GPU
(tests/test_move_reference_gpu.py), pinned without a GPU:

* Philox4x32-10 to the published known answers, and the stream layout (words x, y, z, w; c3 = counter bits 32-55 << 8
  plus the block) to the scalar Python restatement;
* the laws to their exact CDFs with scipy: every Dirichlet coordinate against Beta(alpha, 5 alpha), x_i / (x_i + x_j)
  against Beta(alpha, alpha) and the raw gamma draws against Gamma(alpha), over 2^20 rows at nine alphas from 1e-3 to
  30, with Kolmogorov-Smirnov thresholds at p = 1e-6;
* the root policy to port.play_policy / port.sample_action (the reference's own calls) bit for bit at row sums up to
  65,534, and np.power's non-integer powers to mpmath within 2 ulp;
* as sharp: nine plausible kernel bugs, each restated, change at least a stated number of elements of the GPU test's
  own inputs, so a green GPU run rules them out."""
import mpmath
import numpy as np
import pytest
import scipy.stats as ss

from oracle import episode_ref as er
from oracle import move_ref as mr
from oracle import port

KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
LAW_ALPHAS = (1e-3, 0.03, 0.25, 0.5, 0.999, 1.0, 1.001, 3.0, 30.0)
LAW_ROWS = 1 << 20
KS_P = 1e-6


def test_philox_known_answers_and_array_form():
    for c, k, want in KAT:
        assert tuple(mr.philox_host(c, k)) == want
        assert tuple(int(v) for v in mr.philox(*c, *k)) == want
    w = np.random.default_rng(0).integers(0, 2 ** 32, (300, 6), dtype=np.uint64)
    got = np.stack(mr.philox(*w.T), 1)
    for i in range(len(w)):
        assert got[i].tolist() == mr.philox_host(w[i, :4].tolist(), w[i, 4:].tolist())


def _u(hi, lo):
    return ((((hi << 32) | lo) >> 11) + 0.5) * 2.0 ** -53


def test_stream_layout_against_the_scalar_restatement():
    """Uniform k of a stream is words (x, y) or (z, w) of block k // 2, the block number added to c3 = counter bits
    32-55 << 8; the move's uniform is words (x, y) of block (item, counter) under seed ^ "UNIF"; the keyed form is it."""
    seed, item, counter = 0xFEDCBA9876543210, (1 << 63) + 12345, ((1 << 56) - 1) ^ (0x5A << 40)
    s = mr.PhiloxStream(seed, [item], counter)
    ctr = [item & mr.MASK32, item >> 32, counter & mr.MASK32, ((counter >> 32) << 8) & mr.MASK32]
    key = [seed & mr.MASK32, seed >> 32]
    for k in range(12):
        blk = mr.philox_host(ctr[:3] + [ctr[3] + k // 2], key)
        hi, lo = (blk[0], blk[1]) if k % 2 == 0 else (blk[2], blk[3])
        assert s.uniform()[0] == _u(hi, lo)
    assert s.blocks()[0] == 6
    items = np.array([0, 1, (1 << 32) - 1, 1 << 32, (1 << 64) - 1], np.uint64)
    u = mr.uniform01(seed, items, counter)
    for i, it in enumerate(items.tolist()):
        r = mr.philox_host([it & mr.MASK32, it >> 32, counter & mr.MASK32, counter >> 32], [(seed & mr.MASK32) ^ mr.UNIFORM_KEY, seed >> 32])
        assert u[i] == float(((r[0] << 32) | r[1]) >> 11) / 2.0 ** 53
    hi = np.array([5 << 32, 0, 7 << 40, 1 << 63, 0], np.uint64)
    assert np.array_equal(mr.uniform_keyed(seed, hi, 3, items), np.array([mr.uniform01(seed, items[i], int(hi[i]) | 3) for i in range(5)]))
    # the one-hot fallback: int(6 u) on the first uniform of the stream keyed with 7 << 56
    d = mr.dirichlet(3, np.arange(4000, dtype=np.uint64), 11, 1e-4)
    fb = np.nonzero(d.fallback)[0]
    assert len(fb) > 100 and (d.x[fb].sum(1) == 1.0).all() and (d.x[fb].max(1) == 1.0).all()
    s = mr.PhiloxStream(3 ^ mr.DIRICHLET_KEY ^ (7 << 56), fb.astype(np.uint64), 11)
    assert np.array_equal(d.x[fb].argmax(1), (s.uniform() * 6.0).astype(int))


def test_cospi_reduction():
    y = np.concatenate([np.arange(-8, 9) / 4.0, np.random.default_rng(1).random(10_000) * 2.0])
    ref = np.array([float(mpmath.cospi(mpmath.mpf(float(v)))) for v in y])
    assert np.abs(mr.cospi(y) - ref).max() < 4e-16
    assert (mr.cospi(np.array([0.5, 1.5])) == 0.0).all() and (mr.cospi(np.array([0.0, 1.0, 2.0])) == [1.0, -1.0, 1.0]).all()


def _ks_crit(n):
    return ss.kstwo(n).isf(KS_P)


@pytest.mark.parametrize("alpha", LAW_ALPHAS)
def test_dirichlet_and_gamma_laws_against_exact_cdfs(alpha):
    d = mr.dirichlet(2024, np.arange(LAW_ROWS, dtype=np.uint64), 5, alpha)
    assert d.blocks.max() < mr.MAX_BLOCKS and np.isfinite(d.x).all() and np.abs(d.x.sum(1) - 1.0).max() < 1e-15
    crit = _ks_crit(LAW_ROWS)
    stats = {}
    coord = ss.beta(alpha, 5 * alpha)
    for a in range(6):
        # the gammas are normalised after they are drawn (np.random.dirichlet's way): at alpha = 1e-3 the median gamma is
        # about 1e-301, most underflow before the division, and the coordinates are not resolved in float64
        if alpha > 1e-3:
            stats[f"x{a}"] = mr.ks_grid(np.sort(d.x[:, a]), coord.ppf, coord.cdf, ceil=mr.CEIL_01), crit
        g = ss.gamma(alpha)
        stats[f"g{a}"] = mr.ks_grid(np.sort(d.gammas[:, a]), g.ppf, g.cdf), crit
    half = ss.beta(alpha, alpha)
    # at alpha = 1e-3 the median gamma draw is about 1e-301: the ratio of two is not resolved in float64
    for i, j in ((0, 1), (2, 3), (4, 5)) if alpha > 1e-3 else ():
        # the ratio of two gammas is independent of their sum: rows whose pair underflowed to 0 + 0 leave its law as is
        s = d.x[:, i] + d.x[:, j]
        r = np.sort(d.x[s > 0, i] / s[s > 0])
        stats[f"x{i}/(x{i}+x{j})"] = mr.ks_grid(r, half.ppf, half.cdf, ceil=mr.CEIL_01), _ks_crit(len(r))
    print(alpha, {k: round(v[0], 5) for k, v in stats.items()}, "crit", round(crit, 5), "fallback", int(d.fallback.sum()))
    for k, (v, c) in stats.items():
        assert v < c, (alpha, k, v, c)
    if alpha == 1e-3:  # the all-underflow fallback runs at about 1.1 % of the rows
        assert 0.009 < d.fallback.mean() < 0.014


@pytest.mark.parametrize("S", [1, 2, 1554, 1555, 4096, 14000, 65534])
def test_play_policy_and_sampling_equal_port(S):
    rows = mr.root_rows(S, 600, S) if S > 2 else np.array([r for r in np.ndindex(*(3,) * 6) if sum(r) == S], np.int64)
    ri, u = mr.edge_uniforms(rows, 1.0)
    u = np.concatenate([u, np.random.default_rng(S).random(len(rows))])
    ri = np.concatenate([ri, np.arange(len(rows))])
    differ = 0
    for T in (1.0, 0.5, 0.1, 0.0):
        table = mr.numpy_pow_table(S, T)
        pi = mr.play_policy(rows, T)
        assert np.array_equal(mr.play_policy(rows, T, pow_table=table), pi)
        prod = mr.play_policy(rows, T, products=True)
        want = np.stack([port.play_policy(r, T) for r in rows])
        assert np.array_equal(pi, want), (S, T)
        if S <= er.POLICY_EXACT_MAX:
            assert np.array_equal(prod, want)
        differ += int((prod != want).any(1).sum())
        act = mr.sample_action(pi[ri], u)
        assert act.tolist() == [port.sample_action(want[i], x) for i, x in zip(ri, u)], (S, T)
        assert np.array_equal(mr.argmax_action(rows), np.array([np.argmax(r) for r in rows]))
    print(f"S={S}: products != np.power in {differ} rows")


def test_non_integer_powers_within_two_ulp_of_mpmath():
    counts = np.concatenate([np.arange(0, 2000), np.random.default_rng(2).integers(2000, 65536, 3000)]).astype(np.int64)
    mpmath.mp.prec = 120
    for T in (0.4, 0.3):
        ex = mr.exponent_of(T)
        table = mr.numpy_pow_table(65535, T)
        got = table[counts, np.arange(len(counts)) % 6]
        ref = np.array([float(mpmath.power(int(c), mpmath.mpf(ex))) for c in counts])
        ulp = np.spacing(np.maximum(ref, np.finfo(float).tiny))
        assert (np.abs(got - ref) <= 2 * ulp).all(), T


# ---- sharpness: each wrong restatement changes at least MIN elements of the GPU test's inputs ------------------------
SHARP_MIN = dict(sine=300_000, boost_alpha=200_000, shared_stream=300_000, block_not_advanced=200_000, counter_hi_ignored=200_000,
                 sum_order=10_000, searchsorted_left=50_000, last_argmax=20, products_not_table=3_000)
SHARP_ROWS = 4096  # the first rows of the GPU test's large batch


def test_wrong_restatements_change_the_gpu_tests_outputs():
    seen = dict.fromkeys(SHARP_MIN, 0)
    for seed, counter, offset in mr.DIRICHLET_KEYS:
        items = np.uint64(offset) + np.arange(SHARP_ROWS, dtype=np.uint64)
        for alpha in mr.DIRICHLET_ALPHAS:
            good = mr.dirichlet(seed, items, counter, alpha).x

            def count(**wrong):
                return int((mr.dirichlet(seed, items, counter, alpha, **wrong).x != good).sum())

            seen["sine"] += count(trig=mr.sinpi)
            if alpha < 1:
                seen["boost_alpha"] += count(boost_exponent=alpha)
            seen["shared_stream"] += count(shared_stream=True)
            seen["block_not_advanced"] += count(advance=False)
            if counter >> 32:
                seen["counter_hi_ignored"] += count(counter_hi=False)
    for S in mr.ROOT_SUMS:
        rows = mr.root_rows(S, 2000, S)
        table = mr.numpy_pow_table(S, 0.1)
        good = mr.play_policy(rows, 0.1, pow_table=table)
        seen["sum_order"] += int((mr.play_policy(rows, 0.1, pow_table=table, sum_order="right") != good).sum())
        seen["products_not_table"] += int((mr.play_policy(rows, 0.1, products=True) != good).sum())
        ri, u = mr.edge_uniforms(rows, 0.1, table)
        seen["searchsorted_left"] += int((mr.sample_action(good[ri], u, "left") != mr.sample_action(good[ri], u)).sum())
        seen["last_argmax"] += int((mr.argmax_action(rows, last=True) != mr.argmax_action(rows)).sum())
    print({k: (seen[k], SHARP_MIN[k]) for k in seen})
    for k, v in seen.items():
        assert v >= SHARP_MIN[k], (k, v, SHARP_MIN[k])
