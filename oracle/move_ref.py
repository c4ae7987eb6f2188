"""Vectorised NumPy restatement of the random draws and the root policy of one self-play move
(muzero-hanoi_b200/csrc/hmz_selfplay.cu, hmz_env.cu and root_policy_eval in hmz_tree.cuh).

Random draws, Philox4x32-10 (Salmon, Moraes, Dror, Shaw 2011) over uint64 arrays:

* ``PhiloxStream``: counter words (item lo, item hi, counter lo, (counter hi << 8) + block), key (seed lo, seed hi); a
  block's words are consumed x, y, z, w and ``c3`` goes up by one per block.  Every draw takes two words, so uniform k of
  a stream is the word pair (x, y) or (z, w) of block k // 2.  ``uniform()`` = ((hi << 32 | lo) >> 11) + 0.5) * 2^-53;
  ``normal()`` = Box-Muller with cospi (argument reduced exactly here, then libm); ``gamma(alpha)`` = Marsaglia and
  Tsang (2000), for alpha < 1 the draw of alpha + 1 times U^(1/alpha).
* Dirichlet: action a draws its gamma from its own stream, key seed ^ "DIRICHLE" ^ (a + 1) << 56; the six are normalised
  by their left-to-right sum, and a row whose sum is not positive (every gamma underflowed, alpha of a few 1e-3 or less)
  becomes one-hot on action int(6 u), u the first uniform of the stream keyed with 7 << 56.
* The move's sampling uniform (``uniform01``, key word 0 ^ "UNIF"), its per-item keyed form, the random env reset
  (``__umulhi`` of word x over the non-goal states, key word 0 ^ "RESE") and the random env step (lane e & 3 of the block
  of vec4 group e >> 2, a uniform choice among the two or three legal moves; the step itself is oracle/cport.py's).

Every accept / reject test of the gamma loop reports its margin |lhs - rhs| / max(1, |lhs|, |rhs|): the device's libm
(``log``, ``cospi``, ``pow``) and its fused multiply-adds differ from the host's in the last bits, so a row whose
smallest margin is below ``MARGIN_MIN`` may legitimately take the other branch on the device.  The fallback test counts
as one too: a row whose gamma sum is positive but below 16 subnormal ulp gets margin 0.

Root policy (MCTS/mcts.py:112-126), NumPy's way: ``np.power(int64 visits, clamp(1/T, 1, 5))`` or a supplied table,
``/ np.sum`` (left to right for six elements), ``np.random.choice`` with its uniform supplied (cdf / cdf[-1],
``searchsorted(side="right")``) or ``np.argmax``.  ``products=True`` restates the kernel's repeated products instead: they
equal ``np.power`` for every count up to ``episode_ref.POLICY_EXACT_MAX`` = 1,554 and differ above it by design (a
caller that needs NumPy's powers there passes ``pow_table``).

Keyword switches that restate plausible kernel bugs exist so that tests/test_move_reference_cpu.py can show that the GPU
test would catch them.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import cport

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF
MASK64 = (1 << 64) - 1
DIRICHLET_KEY = 0x4449524943484C45  # "DIRICHLE"
UNIFORM_KEY = 0x554E4946            # "UNIF"
RESET_KEY = 0x52455345              # "RESE"
COUNTER_LIMIT = 1 << 56             # hmz_rng_dirichlet / hmz_selfplay_move reject counters from here on
MAX_BLOCKS = 256                    # blocks one (key, item, counter) stream can use before c3 carries into the counter
MARGIN_MIN = 1e-10                  # accept / reject tests closer than this may go either way on the device
TWO_M53 = 1.0 / 9007199254740992.0
SUBNORMAL_SUM = 16 * 2.0 ** -1074   # a positive gamma sum below this may be 0 on the device (and take the fallback)


def philox_host(c, k):
    """Philox4x32-10 of one block with Python integers: counter words c[0..3], key words k[0..1] -> 4 output words."""
    c, k = list(c), list(k)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k[0], p1 & MASK32, (p0 >> 32) ^ c[3] ^ k[1], p0 & MASK32]
        k = [(k[0] + W0) & MASK32, (k[1] + W1) & MASK32]
    return c


def _u64(x):
    return np.asarray(x, dtype=np.uint64) if not isinstance(x, int) else np.uint64(x & MASK64)


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over arrays (broadcast): every argument holds 32-bit words; returns (x, y, z, w) as uint64 arrays."""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*(np.asarray(_u64(v), dtype=np.uint64) for v in (c0, c1, c2, c3, k0, k1)))
    m = np.uint64(MASK32)
    s32 = np.uint64(32)
    k0, k1 = k0.copy(), k1.copy()
    for _ in range(10):
        p0 = np.uint64(M0) * c0
        p1 = np.uint64(M1) * c2
        c0, c1, c2, c3 = (p1 >> s32) ^ c1 ^ k0, p1 & m, (p0 >> s32) ^ c3 ^ k1, p0 & m
        k0 = (k0 + np.uint64(W0)) & m
        k1 = (k1 + np.uint64(W1)) & m
    return c0, c1, c2, c3


def _lo(x):
    return _u64(x) & np.uint64(MASK32)


def _hi(x):
    return _u64(x) >> np.uint64(32)


def cospi(y):
    """cos(pi y) with the argument reduced exactly: y = n / 2 + r, |r| <= 1/4 (both exact in float64), then libm."""
    n = np.rint(2.0 * y)
    r = y - 0.5 * n
    q = n.astype(np.int64) & 3
    s, c = np.sin(np.pi * r), np.cos(np.pi * r)
    return np.select([q == 0, q == 1, q == 2], [c, -s, -c], s)


def sinpi(y):
    return cospi(y - 0.5)


class PhiloxStream:
    """One PhiloxStream per element of ``item`` (hmz_selfplay.cu): sequential uniforms, normals and gammas.

    ``pos`` counts the uniforms each stream has drawn (two 32-bit words each), so the blocks it used are ceil(pos / 2).
    Wrong restatements: ``advance=False`` keeps c3 at its first block; ``counter_hi=False`` drops counter bits 32-55."""

    def __init__(self, seed, item, counter, advance=True, counter_hi=True):
        item = np.atleast_1d(_u64(item))
        self.n = item.size
        counter = np.broadcast_to(_u64(counter), item.shape)
        seed = int(seed) & MASK64
        self.c0, self.c1, self.c2 = _lo(item), _hi(item), _lo(counter)
        hi = _hi(counter) if counter_hi else np.zeros_like(item)
        self.c3 = (hi << np.uint64(8)) & np.uint64(MASK32)
        self.k0, self.k1 = np.uint64(seed & MASK32), np.uint64(seed >> 32)
        self.pos = np.zeros(self.n, np.int64)
        self.advance = advance
        self._blk = np.full(self.n, -1, np.int64)  # the block each stream has in its buffer
        self._buf = np.zeros((self.n, 4), np.uint64)

    def uniform(self, rows=None):
        rows = np.arange(self.n) if rows is None else rows
        k = self.pos[rows]
        blk = k >> 1 if self.advance else np.zeros_like(k)
        new = blk != self._blk[rows]
        r = rows[new]
        self._buf[r] = np.stack(philox(self.c0[r], self.c1[r], self.c2[r], (self.c3[r] + blk[new].astype(np.uint64)) &
                                       np.uint64(MASK32), self.k0, self.k1), 1)
        self._blk[r] = blk[new]
        odd = (k & 1).astype(bool)
        buf = self._buf[rows]
        hi, lo = np.where(odd, buf[:, 2], buf[:, 0]), np.where(odd, buf[:, 3], buf[:, 1])
        self.pos[rows] += 1
        return ((((hi << np.uint64(32)) | lo) >> np.uint64(11)).astype(np.float64) + 0.5) * TWO_M53

    def normal(self, rows, trig=cospi):
        u1 = self.uniform(rows)
        u2 = self.uniform(rows)
        return np.sqrt(-2.0 * np.log(u1)) * trig(2.0 * u2)

    def blocks(self):
        return (self.pos + 1) // 2


def _margin(lhs, rhs):
    return np.abs(lhs - rhs) / np.maximum(1.0, np.maximum(np.abs(lhs), np.abs(rhs)))


def gamma(stream: PhiloxStream, alpha: float, trig=cospi, boost_exponent=None, max_iterations=1000):
    """Marsaglia and Tsang's gamma(alpha) for every stream of ``stream``: (draws, smallest margin of each draw's accept /
    reject tests).  ``boost_exponent`` (wrong restatement) replaces the 1 / alpha of the alpha < 1 boost.  A stream that
    has not accepted after ``max_iterations`` tries (only a broken restatement gets there) draws NaN."""
    alpha = float(alpha)
    a = alpha + 1.0 if alpha < 1.0 else alpha
    d = a - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    out = np.full(stream.n, np.nan)
    margin = np.full(stream.n, np.inf)
    todo = np.arange(stream.n)
    for _ in range(max_iterations):
        if todo.size == 0:
            break
        x = stream.normal(todo, trig)
        t = 1.0 + c * x
        margin[todo] = np.minimum(margin[todo], _margin(t, 0.0))
        ok = t > 0.0
        rows, x, t = todo[ok], x[ok], t[ok]
        t = t * t * t
        u = stream.uniform(rows)
        lhs = np.log(u)
        rhs = 0.5 * x * x + d - d * t + d * np.log(t)
        margin[rows] = np.minimum(margin[rows], _margin(lhs, rhs))
        acc = lhs < rhs
        out[rows[acc]] = d * t[acc]
        todo = np.sort(np.concatenate([todo[~ok], rows[~acc]]))
    if alpha < 1.0:
        ex = 1.0 / alpha if boost_exponent is None else boost_exponent
        out = out * np.power(stream.uniform(), ex)
    return out, margin


@dataclass
class Dirichlet:
    x: np.ndarray         # float64 [n, 6]: the draw
    gammas: np.ndarray    # float64 [n, 6]: the six gamma draws before normalisation
    blocks: np.ndarray    # int64 [n, 6]: Philox blocks each action's stream used
    margin: np.ndarray    # float64 [n]: smallest accept / reject margin of the row
    fallback: np.ndarray  # bool [n]: every gamma underflowed, the row is one-hot


def dirichlet_key(seed: int, a: int) -> int:
    return (int(seed) ^ DIRICHLET_KEY ^ ((a + 1) << 56)) & MASK64


def dirichlet(seed, item, counter, alpha, *, trig=cospi, boost_exponent=None, shared_stream=False, advance=True,
              counter_hi=True) -> Dirichlet:
    """hmz_rng_dirichlet of items ``item`` (uint64 array) at ``counter`` (scalar or per item).  The keywords restate
    wrong kernels: ``trig=sinpi``, ``boost_exponent=alpha``, ``shared_stream`` (one key for all six actions),
    ``advance=False`` (block counter never advanced), ``counter_hi=False`` (counter bits 32-55 ignored)."""
    item = np.atleast_1d(_u64(item))
    n = item.size
    g, blocks, margin = np.empty((n, 6)), np.empty((n, 6), np.int64), np.full(n, np.inf)
    for a in range(6):
        key = dirichlet_key(seed, 0 if shared_stream else a)
        s = PhiloxStream(key, item, counter, advance=advance, counter_hi=counter_hi)
        g[:, a], m = gamma(s, alpha, trig, boost_exponent)
        blocks[:, a] = s.blocks()
        margin = np.minimum(margin, m)
    total = g[:, 0].copy()
    for a in range(1, 6):
        total = total + g[:, a]
    fb = ~(total > 0.0)
    # the fallback test itself: a sum of a few subnormal ulp hangs on the last bits of a subnormal pow()
    margin = np.where(fb | (total >= SUBNORMAL_SUM), margin, 0.0)
    x = g.copy()
    if fb.any():
        s = PhiloxStream((int(seed) ^ DIRICHLET_KEY ^ (7 << 56)) & MASK64, item[fb],
                         np.broadcast_to(_u64(counter), item.shape)[fb], advance=advance, counter_hi=counter_hi)
        pick = (s.uniform() * 6.0).astype(np.int64)
        x[fb] = np.arange(6)[None, :] == pick[:, None]
        total[fb] = 1.0
    return Dirichlet(x / total[:, None], g, blocks, margin, fb)


def uniform01(seed, item, counter):
    """hmz_rng_uniform: the 53 high bits of words (x, y) of the block (item, counter), key (seed lo ^ "UNIF", seed hi)."""
    seed = int(seed) & MASK64
    x, y, _, _ = philox(_lo(item), _hi(item), _lo(counter), _hi(counter), (seed & MASK32) ^ UNIFORM_KEY, seed >> 32)
    return (((x << np.uint64(32)) | y) >> np.uint64(11)).astype(np.float64) * TWO_M53


def uniform_keyed(seed, counter_hi, counter_lo, item):
    """hmz_rng_uniform_keyed: item i draws uniform01(seed, item[i], counter_hi[i] | counter_lo)."""
    return uniform01(seed, item, _u64(counter_hi) | _u64(counter_lo))


def index_to_word(idx, n_disks):
    """Base-3 state index (disk 0 most significant) -> packed env word."""
    idx = np.asarray(idx, np.uint64).copy()
    w = np.zeros(idx.shape, np.uint64)
    for d in range(n_disks - 1, -1, -1):
        w |= (idx % np.uint64(3)) << np.uint64(2 * d)
        idx //= np.uint64(3)
    return w.astype(np.uint32)


def env_random_reset(n, n_disks, goal_peg, seed, counter):
    """hmz_env_random_reset of envs 0..n-1: umulhi(word x, 3^N - 1), skipping the goal index."""
    seed = int(seed) & MASK64
    i = np.arange(n, dtype=np.uint64)
    x, _, _, _ = philox(_lo(i), _hi(i), _lo(counter), _hi(counter), (seed & MASK32) ^ RESET_KEY, seed >> 32)
    n_states = 3 ** n_disks
    goal_index = sum(goal_peg * 3 ** d for d in range(n_disks))
    idx = (x * np.uint64(n_states - 1)) >> np.uint64(32)
    idx += (idx >= np.uint64(goal_index)).astype(np.uint64)
    return index_to_word(idx, n_disks)


def random_step_words(n, seed, step_index):
    """The 32-bit random word of env e in env_step_random_vec4 / env_rollout_random_vec4: lane e & 3 (x, y, z, w) of
    the block (group e >> 2, step_index) under key (seed lo, seed hi)."""
    seed = int(seed) & MASK64
    g = np.arange((n + 3) // 4, dtype=np.uint64)
    blk = np.stack(philox(_lo(g), _hi(g), _lo(step_index), _hi(step_index), seed & MASK32, seed >> 32), 1)
    return blk.reshape(-1)[:n]


def random_actions(words, rnd, n_disks):
    """The legal move step_random_word takes: index umulhi(rnd, n_legal) into (disk 0 -> the next peg, disk 0 -> the
    other peg, the move between the other two pegs), in the env's action numbering."""
    st = np.asarray(words, np.uint64) & np.uint64((1 << 2 * n_disks) - 1)
    pegs = np.stack([(st >> np.uint64(2 * d)) & np.uint64(3) for d in range(n_disks)], 1).astype(np.int64)
    p0 = pegs[:, 0]
    q1, q2 = (p0 + 1) % 3, (p0 + 2) % 3
    big = n_disks  # top disk of an empty peg

    def top(q):
        on = pegs == q[:, None]
        return np.where(on.any(1), on.argmax(1), big)

    t1, t2 = top(q1), top(q2)
    n_legal = 2 + (t1 != t2)
    idx = (np.asarray(rnd, np.uint64) * n_legal.astype(np.uint64)) >> np.uint64(32)
    first = t1 < t2
    f = np.where(idx < 2, p0, np.where(first, q1, q2))
    t = np.where(idx == 0, q1, np.where(idx == 1, q2, np.where(first, q2, q1)))
    return (2 * f + t - (t > f)).astype(np.uint8)


def env_step_random(words, n_disks, max_steps, goal_peg, reset_word, seed, step_index):
    """hmz_env_step_random: (new words, actions, rewards, flags); ``words`` uint32 [n] is not modified."""
    w = np.array(words, np.uint32)
    act = random_actions(w, random_step_words(len(w), seed, step_index), n_disks)
    rw, fl, _ = cport.env_step(w, act, n_disks, max_steps, goal_peg, auto_reset=True, reset_word=reset_word)
    return w, act, rw, fl


def env_rollout_random(words, n_disks, max_steps, goal_peg, reset_word, n_steps, seed, step_index):
    """hmz_env_rollout_random: (new words, counters [steps, goals, truncations, xor fold of the final words])."""
    w = np.array(words, np.uint32)
    goals = truncs = 0
    for k in range(n_steps):
        w, _, _, fl = env_step_random(w, n_disks, max_steps, goal_peg, reset_word, seed, step_index + k)
        goals += int((fl & 4).astype(bool).sum())
        truncs += int((fl & 8).astype(bool).sum())
    q = w.reshape(-1, 4).astype(np.uint64)
    fold = np.bitwise_xor.reduce(((q[:, 0] ^ q[:, 2]) << np.uint64(32)) | (q[:, 1] ^ q[:, 3])) if len(q) else np.uint64(0)
    return w, np.array([4 * len(q) * n_steps, goals, truncs, int(fold)], np.uint64)


@dataclass
class Begin:
    noise: Dirichlet | None
    prior: np.ndarray      # float64 [B, 6]: root_prior
    prior_f32: np.ndarray  # float32 [B, 6]: the priors of node record 0
    uniform: np.ndarray    # float64 [B]: the move's sampling uniform


def selfplay_begin(p0, alpha, eps, seed, counter, game_offset, **wrong) -> Begin:
    """selfplay_begin: the Dirichlet draw of every game (when alpha > 0 and eps > 0), port.mix_dirichlet's float32
    product and float64 sum, the float32 priors of record 0 and the sampling uniform."""
    p0 = np.asarray(p0, np.float32)
    games = np.uint64(game_offset) + np.arange(len(p0), dtype=np.uint64)
    noise = None
    if alpha > 0.0 and eps > 0.0:
        noise = dirichlet(seed, games, counter, alpha, **wrong)
        prior = np.float32(1.0 - eps) * p0 + eps * noise.x  # MCTS/mcts.py:148-150 (port.mix_dirichlet at eps = 0.25)
    else:
        prior = p0.astype(np.float64)
    return Begin(noise, prior, prior.astype(np.float32), uniform01(seed, games, counter))


# ----------------------------------------------------------------------------------------------------- root policy
def exponent_of(temperature: float) -> float:
    return max(1.0, min(5.0, 1.0 / temperature)) if temperature > 0.0 else 1.0


def numpy_pow_table(n_max: int, temperature: float) -> np.ndarray:
    """float64 [n_max + 1, 6]: np.power of every count at every position of a 6-element int64 array, as
    generate_play_policy calls it (hmz_search_root_policy's pow_table)."""
    ex = exponent_of(temperature)
    return np.stack([np.power(np.full(6, n, np.int64), ex) for n in range(n_max + 1)]) if temperature > 0.0 else \
        np.repeat(np.arange(n_max + 1, dtype=np.float64)[:, None], 6, 1)


def play_policy(visits, temperature, *, pow_table=None, products=False, sum_order="left"):
    """generate_play_policy rows: visits int [M, 6] -> float64 [M, 6].  np.power's values (``pow_table`` when given,
    for counts inside it), or with ``products`` the kernel's repeated products for integer exponents.
    ``sum_order="right"`` (wrong restatement): v0 + (v1 + ... + v5)."""
    v = np.asarray(visits).astype(np.int64)
    ex = exponent_of(temperature)
    if products and ex == int(ex):
        x = v.astype(np.float64)
        w = x.copy()
        for _ in range(1, int(ex)):
            w = w * x
    else:
        w = np.power(v, ex) if temperature > 0.0 else v.astype(np.float64)
    if pow_table is not None:
        inside = v < len(pow_table)
        w = np.where(inside, pow_table[np.minimum(v, len(pow_table) - 1), np.arange(6)[None, :]], w)
    if sum_order == "left":
        tot = w[:, 0]
        for a in range(1, 6):
            tot = tot + w[:, a]
    else:
        tot = w[:, 5]
        for a in range(4, 0, -1):
            tot = w[:, a] + tot
        tot = w[:, 0] + tot
    return w / tot[:, None]


def sample_action(pi, u, side="right"):
    """np.random.choice(6, p=pi) with its uniform supplied (port.sample_action): cdf = cumsum, cdf /= cdf[-1], count of
    cdf <= u (``side="left"``, wrong: cdf < u)."""
    cdf = np.cumsum(pi, axis=1)
    cdf = cdf / cdf[:, -1:]
    u = np.asarray(u)[:, None]
    hit = cdf <= u if side == "right" else cdf < u
    return np.minimum(hit.sum(1), 5)


def argmax_action(visits, last=False):
    """np.argmax of the visit counts: the first maximum (``last=True``, wrong: the last one)."""
    v = np.asarray(visits)
    if not last:
        return v.argmax(1)
    return v.shape[1] - 1 - v[:, ::-1].argmax(1)


def sum_orders_differ(visits, temperature, pow_table=None):
    """Rows whose play policy depends on the order of np.sum's six additions."""
    return (play_policy(visits, temperature, pow_table=pow_table) !=
            play_policy(visits, temperature, pow_table=pow_table, sum_order="right")).any(1)


# ------------------------------------------------------------------------------------- laws and the GPU test's inputs
def ks_grid(sorted_x, ppf, cdf, floor=2.2250738585072014e-308, ceil=np.inf, grid=1 << 14):
    """Kolmogorov-Smirnov distance between the sample (sorted, float64) and a continuous law, both clipped to
    [floor, ceil]: below the smallest normal double values carry no precision, and a law on [0, 1] rounds its mass
    within a few ulp of 1 to 1 (pass ceil = CEIL_01).  The largest gap between the empirical CDF and the law at the law's
    own quantiles j / grid and at the two clip points: a lower bound of the exact statistic, short of it by at most
    1 / grid."""
    n = len(sorted_x)
    p = np.arange(1, grid) / grid
    q = ppf(p)
    keep = (q >= floor) & (q < ceil)
    emp = np.searchsorted(sorted_x, q[keep], side="right") / n
    d = np.abs(emp - p[keep]).max(initial=0.0)
    d = max(d, abs(np.searchsorted(sorted_x, floor, side="right") / n - float(cdf(floor))))
    if np.isfinite(ceil):
        d = max(d, abs(np.searchsorted(sorted_x, ceil, side="left") / n - float(cdf(ceil))))
    return d


CEIL_01 = 1.0 - 2.0 ** -50


DIRICHLET_ALPHAS = (1e-3, 0.03, 0.25, 3.0, 30.0)
DIRICHLET_BATCHES = (1, 3, 4, 33, 65536 + 77)
# (seed, counter, item_offset): counter bits 32-55 all set at the largest counter allowed; offsets across 2^32 and
# near 2^63
DIRICHLET_KEYS = ((9, 0, 0), (0x0123456789ABCDEF, (0xABCDEF << 32) | 17, (1 << 32) - 40),
                  (5, COUNTER_LIMIT - 1, (1 << 63) - 20))
ROOT_SUMS = (1554, 1555, 4096, 14000, 65534)


def root_rows(S, n, seed):
    """Visit-count rows [n, 6] summing to S for the root-policy test: Dirichlet(0.3) splits, plus the edges (all visits on
    one child, zero-visit children at the front, middle and end, ties of the maximum)."""
    rng = np.random.default_rng(seed)
    rows = rng.multinomial(S, rng.dirichlet(np.full(6, 0.3), n)).astype(np.int64)
    edge = [[S, 0, 0, 0, 0, 0], [0, 0, 0, 0, 0, S], [0, 0, S - S // 2, S // 2, 0, 0], [0, S // 3, S // 3, 0, S - 2 * (S // 3), 0],
            [S // 2, 0, 0, 0, 0, S - S // 2], [S // 6] * 5 + [S - 5 * (S // 6)], [0, 0, 0, S // 2, 0, S - S // 2]]
    rows[:len(edge)] = edge
    return rows


def edge_uniforms(visits, temperature, pow_table=None):
    """Per row, the uniforms at which np.random.choice changes its answer: 0, every cdf[k] / cdf[5] and the double just
    below it, and the largest double below 1.  Returns (row index, u)."""
    pi = play_policy(visits, temperature, pow_table=pow_table)
    cdf = np.cumsum(pi, axis=1)
    cdf = cdf / cdf[:, -1:]
    rows = np.arange(len(pi))
    us = [np.zeros(len(pi)), np.full(len(pi), np.nextafter(1.0, 0.0))]
    for k in range(6):
        us += [cdf[:, k], np.nextafter(cdf[:, k], 0.0)]
    u = np.concatenate(us)
    return np.tile(rows, len(us)), np.clip(u, 0.0, np.nextafter(1.0, 0.0))
