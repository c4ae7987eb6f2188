"""Vectorised NumPy restatement of the episode post-processing kernels (muzero-hanoi_b200/csrc/hmz_episode.cu).

It reads the episode store the device keeps: struct-of-arrays ``[t_max][B]`` indexed by each game's own step counter,
``ep_len[g] > 0`` marking the games whose episode finished on this move.  It computes what the kernels compute, the
way the reference's own functions do (``port.n_step_returns`` / ``mc_returns`` / ``priorities`` / ``play_policy`` /
``organise_transitions`` and ``Buffer.add``, which ``gen_golden`` checked against the unmodified reference):

* n-step returns: ``sum([discount ** i * r ...])`` with CPython 3.12's float ``sum`` (``0 + first``, then Neumaier
  compensation, then ``if c and isfinite(c)``), host ``discount ** i``, plus ``discount ** n_step * root_value``;
* MC returns: NumPy's ``discount ** np.arange(T)``, the reversed cumulative sum and the division;
* priorities ``|f32(return) - f32(root value)|``;
* the row bases of ``hmz_episode_rows`` (``only_solved``: ``returns[len - 1] > 0``) and the total;
* the ring after the reference's per-episode adds in game order (wrap, ``ptr``, ``is_full``; later rows overwrite
  earlier ones), with the rows of ``organise_transitions``: one-hot states, rewards, actions with the absorbing padding,
  float32 play policies from each step's own exponent, returns and priorities.

Only the finished columns are computed (``Post.cols``), and of the rows only those that survive in the ring, so
B = 524,288 stays cheap.

Play policies: ``np.power(int64, e)`` for the integer exponents 1, 2, 5 is evaluated here as repeated float64
products, as the kernels do.  For every count up to ``POLICY_EXACT_MAX`` = 1,554 the two agree bit for bit (the powers
are exact, or a correctly rounded product of an exact power); above it NumPy's ``pow`` rounds some exact halfway cases
the other way (11,533 of the counts 1,555-65,535 at exponent 5 with NumPy 2.3.5), so the ring's policies above that
bound are the repeated products, not NumPy's powers.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

FLAG_DONE, FLAG_ILLEGAL, FLAG_GOAL, FLAG_TRUNC = 1, 2, 4, 8
N_ACTIONS = 6
POLICY_EXACT_MAX = 1554  # largest visit count at which the products equal np.power(count, 5.0)


def exponent_of(temperature: float) -> int:
    """generate_play_policy's exponent clamp(1/T, 1, 5), 1 for T == 0 (raw counts); integer exponents only."""
    if temperature == 0:
        return 1
    e = max(1.0, min(5.0, 1.0 / temperature))
    if e != int(e):
        raise ValueError(f"temperature {temperature} gives the non-integer exponent {e}")
    return int(e)


def rewards(flags: np.ndarray) -> np.ndarray:
    """The env's reward (python numbers 100, -100/1000, 0) selected by the move's flags, float64."""
    flags = np.asarray(flags)
    return np.where(flags & FLAG_GOAL, 100.0, np.where(flags & FLAG_ILLEGAL, -100 / 1000, 0.0))


def libm_powers(discount: float, n: int) -> np.ndarray:
    """``discount ** i`` for i in [0, n) through the host's float pow (the n-step returns, utils.py:64-69)."""
    return np.array([discount ** i for i in range(n)], dtype=np.float64)


def numpy_powers(discount: float, n: int) -> np.ndarray:
    """``discount ** np.arange(n)``: NumPy's power ufunc (compute_MCreturns)."""
    return float(discount) ** np.arange(n)


def neumaier_rows(terms):
    """CPython 3.12 ``sum()`` of float terms, elementwise over arrays: ``terms`` yields the k-th addend of every sum."""
    it = iter(terms)
    f = 0.0 + next(it)  # int 0 + float
    c = np.zeros_like(f)
    for x in it:
        t = f + x
        c = c + np.where(np.abs(f) >= np.abs(x), (f - t) + x, (x - t) + f)
        f = t
    return np.where((c != 0) & np.isfinite(c), f + c, f)


def plain_rows(terms):
    """A left-to-right float sum (what the reference does NOT do); used to show the checks can tell them apart."""
    it = iter(terms)
    f = 0.0 + next(it)
    for x in it:
        f = f + x
    return f


@dataclass
class Post:
    """Returns and priorities of the finished columns: arrays [L][C] over the columns ``cols`` (L = the longest of
    their episodes); ``mask[t, c]`` = t < lens[c]; entries outside the mask are meaningless."""
    cols: np.ndarray
    lens: np.ndarray
    returns: np.ndarray
    priority: np.ndarray
    mask: np.ndarray

    def last_returns(self, B: int) -> np.ndarray:
        """returns[len - 1] of every finished column, 0 elsewhere (float64 [B])."""
        out = np.zeros(B, np.float64)
        if len(self.cols):
            out[self.cols] = self.returns[self.lens - 1, np.arange(len(self.cols))]
        return out


def _finished(ep_len, t_max):
    ep_len = np.minimum(np.asarray(ep_len, np.int64), t_max)
    cols = np.nonzero(ep_len > 0)[0]
    lens = ep_len[cols]
    L = int(lens.max()) if len(cols) else 0
    mask = np.arange(L)[:, None] < lens[None, :]
    return cols, lens, L, mask


def priorities(returns, root_q):
    """Muzero.py:197-200: |float32(return) - float32(root value)|, the subtraction in float32."""
    return np.abs(np.asarray(returns).astype(np.float32) - np.asarray(root_q).astype(np.float32))


def n_step_returns(flags, root_q, ep_len, n_step, discount, *, summation=neumaier_rows, powers=None) -> Post:
    """compute_n_step_returns + priorities of every finished column (hmz_episode_returns)."""
    T = flags.shape[0]
    cols, lens, L, mask = _finished(ep_len, T)
    pw = libm_powers(discount, n_step + 1) if powers is None else powers
    r = np.where(mask, rewards(flags[:L, cols]), 0.0)
    q = np.where(mask, root_q[:L, cols], 0.0)
    K = min(n_step, L)  # addends past the episode are int 0: x = 0.0 leaves f and c as they are
    r_pad = np.concatenate([r, np.zeros((K, len(cols)))])
    acc = summation(pw[k] * r_pad[k:k + L] for k in range(max(K, 1)))
    boot = np.zeros_like(q)
    if n_step < L:
        boot[:L - n_step] = np.where(mask[n_step:], q[n_step:], 0.0)
    ret = acc + pw[n_step] * boot
    return Post(cols, lens, ret, priorities(ret, root_q[:L, cols]), mask)


def mc_returns(flags, root_q, ep_len, discount, *, powers=None) -> Post:
    """compute_MCreturns + priorities of every finished column (hmz_episode_mc_returns): one sequential float64 sum
    per episode from its end, each partial sum divided by the discount of its step."""
    T = flags.shape[0]
    cols, lens, L, mask = _finished(ep_len, T)
    d = numpy_powers(discount, T) if powers is None else powers
    x = d[:L, None] * rewards(flags[:L, cols])
    ret = np.zeros((L, len(cols)))
    acc = np.zeros(len(cols))
    for t in range(L - 1, -1, -1):
        live = t < lens
        acc = np.where(t == lens - 1, x[t], np.where(live, acc + x[t], acc))
        ret[t] = np.where(live, acc / d[t], 0.0)
    return Post(cols, lens, ret, priorities(ret, root_q[:L, cols]), mask)


def row_bases(ep_len, last_returns, ptr, only_solved):
    """hmz_episode_rows: row_base[g] = ptr + the rows stored before game g (-1 if g stores none), and the total."""
    ep_len = np.asarray(ep_len, np.int64)
    stored = np.where((ep_len > 0) & ((not only_solved) | (np.asarray(last_returns) > 0.0)), ep_len, 0)
    before = np.cumsum(stored) - stored
    return np.where(stored > 0, ptr + before, -1).astype(np.int64), int(stored.sum())


def play_policy(visits, exponent):
    """generate_play_policy rows: visits [M, 6] (integers), exponent int or [M]; float64 [M, 6].  visits ** e as
    repeated products (np.power's values for counts <= POLICY_EXACT_MAX), then np.sum's order for six elements: left to
    right, ((((v0 + v1) + v2) + v3) + v4) + v5 (NumPy 2.3.5 sums arrays shorter than 8 sequentially)."""
    x = np.asarray(visits).astype(np.float64)
    e = np.broadcast_to(np.asarray(exponent).reshape(-1, 1) if np.ndim(exponent) else exponent, (x.shape[0], 1))
    y = x.copy()
    for k in range(2, 6):
        y = np.where(e >= k, y * x, y)
    tot = y[:, 0]
    for a in range(1, 6):
        tot = tot + y[:, a]
    return y / tot[:, None]


def one_hot(words, n_disks):
    """utils.oneHot_encoding of env words: float32 [M, 3 N]."""
    w = np.asarray(words).astype(np.uint32)
    pegs = (w[:, None] >> (2 * np.arange(n_disks, dtype=np.uint32))[None, :]) & 3
    return (pegs[:, :, None] == np.arange(3)[None, None, :]).reshape(len(w), 3 * n_disks).astype(np.float32)


@dataclass
class Store:
    """Host copy of an episode store (the fields of replay.EpisodeStore), [t_max][B] numpy arrays; exp may be None."""
    state: np.ndarray
    action: np.ndarray
    flags: np.ndarray
    visits: np.ndarray
    root_q: np.ndarray
    ep_len: np.ndarray
    exp: np.ndarray | None = None
    n_disks: int = 3

    @property
    def t_max(self):
        return self.state.shape[0]

    @property
    def B(self):
        return self.state.shape[1]


class Ring:
    """buffer.Buffer with NumPy arrays, filled as ReplayRing.add_episodes fills the device ring."""

    FIELDS = ("states", "rwds", "actions", "pi_probs", "mc_returns", "priorities")

    def __init__(self, size, unroll, d_state, fill=0.0, ptr=0, is_full=False):
        self.size, self.unroll, self.ptr, self.is_full = int(size), int(unroll), int(ptr), bool(is_full)
        self.states = np.full((size, d_state), fill, np.float32)
        self.rwds = np.full((size, unroll), fill, np.float32)
        self.actions = np.full((size, unroll), int(fill), np.int64)
        self.pi_probs = np.full((size, unroll, N_ACTIONS), fill, np.float32)
        self.mc_returns = np.full((size, unroll), fill, np.float32)
        self.priorities = np.full(size, fill, np.float32)

    def _advance(self, n):
        if self.ptr + n >= self.size:
            self.is_full = True
        self.ptr = (self.ptr + n) % self.size

    def add_episodes(self, store: Store, post: Post, temperature=1.0, only_solved=True, absorbing=None, *,
                     last_write_wins=True):
        """organise_transitions + one Buffer.add per stored episode, in game order; returns the number of rows."""
        rb, n = row_bases(store.ep_len, post.last_returns(store.B), self.ptr, only_solved)
        if n == 0:
            return 0
        rows = episode_rows(store, post, rb, self.unroll, absorbing, temperature,
                            first_row=self.ptr + max(0, n - self.size) if last_write_wins else None)
        pos = rows["at"] % self.size
        if not last_write_wins:  # keep the first write of every position instead
            pos, first = np.unique(pos, return_index=True)
            rows = {k: v[first] for k, v in rows.items()}
        for k in self.FIELDS:
            getattr(self, k)[pos] = rows[k]
        self._advance(n)
        return n


def episode_rows(store: Store, post: Post, rb, unroll, absorbing, temperature=1.0, first_row=None):
    """The replay rows of every stored episode in game order: ``at`` = row_base + t (before the wrap) and the six
    row arrays.  Rows with at < first_row (overwritten by later rows of the same add) are left out."""
    t_max, B = store.t_max, store.B
    sel = np.nonzero(rb[post.cols] >= 0)[0]  # finished and stored: index into post's columns
    g, lens = post.cols[sel], post.lens[sel]
    start = np.zeros(len(sel), np.int64) if first_row is None else np.clip(first_row - rb[g], 0, lens)
    cnt = lens - start
    c_idx = np.repeat(np.arange(len(sel)), cnt)
    t = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt) + np.repeat(start, cnt)
    pc, gg, L = sel[c_idx], g[c_idx], lens[c_idx]
    M = len(t)
    j = t[:, None] + np.arange(unroll)[None, :]  # [M, K]
    live = j < L[:, None]
    jc = np.minimum(j, L[:, None] - 1)
    G = np.broadcast_to(gg[:, None], j.shape)
    PC = np.broadcast_to(pc[:, None], j.shape)
    if absorbing is None:
        raise ValueError("absorbing actions are required")
    ab = np.asarray(absorbing).astype(np.int64)
    exp = store.exp[jc, G] if store.exp is not None else np.full(j.shape, exponent_of(temperature))
    pi = play_policy(store.visits[jc, G].reshape(M * unroll, 6), exp.reshape(-1)).reshape(M, unroll, 6)
    return dict(
        at=rb[gg] + t,
        states=one_hot(store.state[t, gg], store.n_disks),
        rwds=np.where(live, rewards(store.flags[jc, G]), 0.0).astype(np.float32),
        actions=np.where(live, store.action[jc, G].astype(np.int64), ab[G]),
        pi_probs=np.where(live[:, :, None], pi, np.float64(1.0) / 6).astype(np.float32),
        mc_returns=np.where(live, post.returns[jc, PC], 0.0).astype(np.float32),
        priorities=post.priority[t, pc],
    )


# ---- synthetic episode stores ---------------------------------------------------------------------------------------
V_MAX = 278.6  # |root value| bound of the network's support (33 atoms, signed-parabolic)


def random_root_values(rng, shape):
    """Root values across the network's range with signed zeros, tiny and subnormal values and float32 underflows."""
    q = rng.uniform(-V_MAX, V_MAX, shape)
    pick = rng.random(shape)
    special = np.array([0.0, -0.0, 1e-300, -5e-324, 1e-46, -1e-40, V_MAX, -V_MAX, 2.0 ** -149, 1e-8])
    q = np.where(pick < 0.15, special[rng.integers(0, len(special), shape)], q)
    return np.where((pick >= 0.15) & (pick < 0.25), rng.uniform(-1e-3, 1e-3, shape), q)


def random_visits(rng, M, S):
    """Visit rows summing to S (multinomial over Dirichlet(0.3) probabilities: some rows put almost all on one action)."""
    return rng.multinomial(S, rng.dirichlet(np.full(6, 0.3), M)).astype(np.int16)


def random_store(seed, B, t_max, n_disks=3, *, illegal=0.2, finished=0.7, lengths=None, S=25, exponents=None,
                 boundary_rows=0):
    """A store as the device leaves it after a move: every finished column holds one episode (its last move done,
    goal or truncation at t_max), unfinished columns interleaved; lengths 1 and t_max always occur.  ``exponents``: a
    tuple of per-step exponents mixed within episodes (store.exp), or None.  ``boundary_rows``: that many steps get
    visit counts around POLICY_EXACT_MAX + 1."""
    rng = np.random.default_rng(seed)
    if lengths is None:
        lengths = np.minimum(rng.geometric(min(1.0, 4.0 / t_max), B), t_max)
        lengths[rng.random(B) < 0.05] = t_max
        lengths[rng.random(B) < 0.05] = 1
    lengths = np.asarray(lengths, np.int64)
    if B >= 4:
        lengths[:4] = [1, t_max, 1, t_max]
    done = rng.random(B) < finished
    if B >= 4:
        done[:4] = [True, True, False, True]
    T = np.arange(t_max)[:, None]
    flags = np.where(rng.random((t_max, B)) < illegal, FLAG_ILLEGAL, 0).astype(np.uint8)
    flags[T >= lengths[None, :]] = 0
    last = (T == lengths[None, :] - 1)
    solved = rng.random(B) < 0.5
    end = np.where(solved, FLAG_GOAL | FLAG_DONE, FLAG_TRUNC | FLAG_DONE).astype(np.uint8)
    end = np.where(lengths == t_max, end, FLAG_GOAL | FLAG_DONE)  # only the t_max-th move can truncate
    flags = np.where(last & done[None, :], end[None, :], flags).astype(np.uint8)
    if illegal > 0:  # an illegal move may end the episode by truncation too
        flags = np.where(last & done[None, :] & (end[None, :] & FLAG_TRUNC).astype(bool) & (rng.random((1, B)) < illegal),
                         flags | FLAG_ILLEGAL, flags).astype(np.uint8)
    pegs = np.zeros((t_max, B), np.int64)
    for d in range(n_disks):
        pegs |= rng.integers(0, 3, (t_max, B), dtype=np.int64) << (2 * d)
    state = (pegs | (T.astype(np.int64) << (2 * n_disks))).astype(np.uint32).view(np.int32)
    action = rng.integers(0, 6, (t_max, B)).astype(np.uint8)
    visits = random_visits(rng, t_max * B, S).reshape(t_max, B, 6)
    if boundary_rows:  # the first steps of game 1 and the last ones of game B - 1, both solved at t_max (stored, kept last)
        row = np.array([POLICY_EXACT_MAX + 1, POLICY_EXACT_MAX, 1, 3, 0, 7], np.int16)
        k = min(boundary_rows, t_max)
        rows = np.stack([np.roll(row - (np.arange(6) == 0) * (i % 3 == 0), i) for i in range(k)]).astype(np.int16)
        for g, ts in ((1, np.arange(k)), (B - 1, np.arange(t_max - k, t_max))):
            visits[ts, g] = rows
            flags[:, g] = np.where(np.arange(t_max) == t_max - 1, FLAG_GOAL | FLAG_DONE, flags[:, g] & FLAG_ILLEGAL)
            lengths[g], done[g] = t_max, True
    root_q = random_root_values(rng, (t_max, B))
    ep_len = np.where(done, lengths, 0).astype(np.int32)
    exp = None
    if exponents is not None:
        exp = np.asarray(exponents, np.uint8)[rng.integers(0, len(exponents), (t_max, B))]
    return Store(state, action, flags, visits, root_q, ep_len, exp, n_disks)


# ---- the GPU tests' cases (also the inputs of the CPU sharpness checks) -----------------------------------------------
# (t_max, n_step, discount, B, illegal rate, seed)
RETURN_CASES = [
    (1, 1, 0.8, 300, 0.2, 1),
    (1, 50, 0.99, 300, 0.0, 2),
    (7, 2, 0.5, 2000, 0.5, 3),
    (7, 10, 1.0, 2000, 0.9, 4),
    (200, 1, 0.97, 600, 0.1, 5),
    (200, 10, 0.8, 600, 0.3, 6),
    (200, 50, 0.99, 600, 0.05, 7),
    (200, 250, 0.8, 600, 0.2, 8),
    (1000, 10, 0.97, 120, 0.02, 9),
    (1000, 50, 0.8, 120, 0.2, 10),
    (1000, 1100, 0.99, 60, 0.1, 11),
]
# the grid-stride loops: (t_max, n_step, discount, B, illegal, seed); more than 8 waves of every kernel on a B200
RETURN_CASES_LARGE = [
    (200, 10, 0.8, 16384, 0.2, 12),
    (2, 2, 0.97, 2_600_000, 0.3, 13),
]
# (t_max, n_disks, unroll, exponents or None, temperature, capacity, ptr, force scalar, B, S, only_solved, seed)
UNROLL_CASES = [
    (200, 5, 5, (1, 2, 5), 1.0, 50000, 49990, False, 400, 25, True, 21),
    (279, 3, 8, (1, 2, 5), 1.0, 37, 36, False, 300, 100, False, 22),
    (7, 1, 1, None, 0.0, 37, 0, False, 500, 25, False, 23),
    (200, 12, 5, None, 0.1, 50000, 0, False, 300, 1554, True, 24),
    (255, 12, 8, (5,), 1.0, 37, 17, False, 200, 1554, False, 25),
    (280, 10, 8, (1, 2, 5), 1.0, 50000, 49999, False, 200, 100, False, 26),
    (1000, 3, 5, None, 0.5, 37, 5, False, 60, 25, True, 27),
    (200, 5, 1, (1, 5), 1.0, 37, 30, True, 300, 1554, False, 28),
    (150, 8, 8, None, 0.2, 50000, 123, True, 300, 100, False, 29),
    (50, 5, 5, None, 1.0, 50000, 7, False, 1000, 25, True, 30),
    (200, 3, 5, (1, 2, 5), 1.0, 50000, 31337, False, 40000, 25, False, 31),   # warp form past 8 waves
    (1000, 3, 5, (2, 5), 1.0, 50000, 2, False, 4000, 100, False, 32),         # scalar form past 8 waves
]
UNROLL_N_STEP, UNROLL_DISCOUNT = 10, 0.8


def unroll_case_store(case):
    t_max, n_disks, unroll, exps, temperature, capacity, ptr0, scalar, B, S, only_solved, seed = case
    st = random_store(seed, B, t_max, n_disks, S=S, exponents=exps, boundary_rows=64 if S >= 1554 else 0)
    absorbing = np.random.default_rng(seed + 1000).integers(0, 6, B).astype(np.uint8)
    return st, absorbing

ROWS_BATCHES = [1, 31, 32, 1023, 1024, 1025, 4097, 65613, 524288]
ROWS_CAPACITY = 50000


def rows_case(B, seed, t_max=3):
    """Inputs of hmz_episode_rows: ep_len in [0, t_max] (about a third unfinished) and a store of returns whose
    returns[len - 1] are positive, negative, +0.0 or -0.0."""
    rng = np.random.default_rng(seed)
    ep_len = np.where(rng.random(B) < 0.35, 0, rng.integers(1, t_max + 1, B)).astype(np.int32)
    ret = rng.choice(np.array([1.5, -2.0, 0.0, -0.0, 5e-324, -5e-324, 100.0]), (t_max, B))
    return ep_len, ret


def rows_ptrs(seed):
    """ptr = 0, capacity - 1 and a random position."""
    return [0, ROWS_CAPACITY - 1, int(np.random.default_rng(seed).integers(1, ROWS_CAPACITY - 1))]
