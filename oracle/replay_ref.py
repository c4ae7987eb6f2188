"""NumPy / integer restatement of the device replay sampler (muzero-hanoi_b200/csrc/hmz_replay.cu).

``ReplayRing.priority_sample`` (priority exponent 1) computes, with NumPy:

    s = np.sum(q)                       float32, NumPy's pairwise tree
    x = q / s                           float32
    np.random.choice(num, batch, p=x):  cdf = cumsum(float64(x)); cdf /= cdf[-1]; searchsorted(cdf, u, side="right")
    w = (float32(1 / size) / x[idx]) ** beta;  w /= max(w)

The device evaluates the two sums in parallel but exactly.  This module restates both the way the kernels do, in
vectorised NumPy and integer arithmetic, so that the CPU tests can check the formulations against ``np.sum`` and
``np.cumsum`` bit for bit:

* ``pairwise_sum``: NumPy's pairwise tree laid out as a complete binary tree, each leaf (<= 128 elements, eight
  accumulators) owned by the position whose path ends there, parents formed as left + right where the right child
  exists (replay_sum_leaves / replay_draw);
* ``exact_cumsum``: the stretch-wise cumulative sum: inside one binade of the running sum every addition is an integer
  step on the grid u = ulp(c), decided by the addend alone except at exact half-ulp remainders (ties to even), so each
  row is a map from the incoming parity bit to (increment, outgoing parity); the maps are scanned (Hillis-Steele, as a
  block scan does) chunk by chunk, and a stretch ends at the first row that reaches the next binade.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

LEAF = 128
CHUNK = 8192
TOP = np.uint64(1 << 53)
SAT = np.uint64(1 << 54)
MANT = np.uint64((1 << 52) - 1)
HIDDEN = np.uint64(1 << 52)
SUM_ATOL = float(np.sqrt(np.finfo(np.float32).eps))  # RandomState.choice: max(sqrt(eps64), sqrt(eps32)) for float32 p


# ---- pairwise sum ---------------------------------------------------------------------------------------------------

def pairwise_depth(n: int) -> int:
    d = 0
    while n > LEAF:
        n -= (n // 2) & ~7
        d += 1
    return d


def _leaves(num: int, depth: int):
    """Start, length and ownership of every position of the complete tree of the given depth."""
    t = np.arange(1 << depth, dtype=np.int64)
    a = np.zeros_like(t)
    n = np.full_like(t, num)
    stop = np.full_like(t, depth)  # level at which the walk reaches a leaf
    for level in range(depth):
        split = n > LEAF
        stop = np.where(~split & (stop == depth), level, stop)
        m = (n // 2) & ~7
        right = ((t >> (depth - 1 - level)) & 1).astype(bool)
        a = np.where(split & right, a + m, a)
        n = np.where(split, np.where(right, n - m, m), n)
    assert (n <= LEAF).all(), "tree deeper than pairwise_depth"
    owner = (t & ((np.int64(1) << (depth - stop)) - 1)) == 0
    return a, n, owner


def _leaf_sums(q: np.ndarray, a: np.ndarray, n: np.ndarray) -> np.ndarray:
    """pairwise_sum's leaf (numpy/_core/src/umath/loops_utils.h.src) for many leaves at once, float32 adds."""
    last = len(q) - 1
    at = lambda i: q[np.minimum(a + i, last)]
    res = np.full(len(a), -0.0, np.float32)
    small = n < 8
    for i in range(7):  # n < 8: left to right from -0.0
        res = np.where(small & (i < n), res + at(i), res)
    r = [at(j) for j in range(8)]
    body = n - n % 8
    for i in range(8, LEAF, 8):
        take = i < body
        for j in range(8):
            r[j] = np.where(take, r[j] + at(i + j), r[j])
    big = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for k in range(7):
        big = np.where(k < n % 8, big + at(body + k), big)
    return np.where(small, res, big).astype(np.float32)


def pairwise_sum(q: np.ndarray) -> np.float32:
    """np.sum(q) for a contiguous float32 vector, through the complete-tree layout the device uses."""
    q = np.ascontiguousarray(q, np.float32)
    depth = max(pairwise_depth(len(q)), 8)
    a, n, owner = _leaves(len(q), depth)
    v = np.zeros(len(a), np.float32)
    v[owner] = _leaf_sums(q, a[owner], n[owner])
    ex = owner.copy()
    while len(v) > 1:
        left, right, ex_r = v[0::2], v[1::2], ex[1::2]
        v = np.where(ex_r, left + right, left).astype(np.float32)
        ex = ex[0::2]
    return v[0]


# ---- exact cumulative sum -------------------------------------------------------------------------------------------

def _bits(x: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(x, np.float64).view(np.uint64)


def row_maps(x: np.ndarray, E: int):
    """(inc0, inc1, out0, out1) of every row: adding x >= 0 to c (biased exponent E, c/u of parity b) adds inc_b to c/u
    and leaves parity out_b, while the sum stays in the binade.  Increments saturate at 2^54."""
    xb = _bits(x)
    pos = x > 0
    sh = (xb >> np.uint64(52)).astype(np.int64) - E
    mx = (xb & MANT) | HIDDEN
    k = np.clip(-sh, 1, 63).astype(np.uint64)
    n_low = mx >> k
    rem = mx & ((np.uint64(1) << k) - np.uint64(1))
    half = np.uint64(1) << (k - np.uint64(1))
    cls = np.where(rem > half, 1, np.where(rem == half, 2, 0))
    n = np.where(sh > 0, SAT, np.where(sh == 0, mx, np.where(sh < -60, np.uint64(0), n_low)))
    cls = np.where(sh < 0, np.where(sh < -60, 0, cls), 0)
    n = np.where(pos, n, np.uint64(0))
    cls = np.where(pos, cls, 0)
    fixed = np.minimum(n + (cls == 1).astype(np.uint64), SAT)
    p = (fixed & np.uint64(1)).astype(np.uint8)
    tie = cls == 2
    nb = n & np.uint64(1)
    inc0 = np.where(tie, n + nb, fixed)
    inc1 = np.where(tie, n + (nb ^ np.uint64(1)), fixed)
    out0 = np.where(tie, 0, p).astype(np.uint8)
    out1 = np.where(tie, 0, p ^ 1).astype(np.uint8)
    return inc0, inc1, out0, out1


def compose(f, g):
    """Map f followed by map g (elementwise over arrays of maps)."""
    fi0, fi1, fo0, fo1 = f
    gi0, gi1, go0, go1 = g
    pick = lambda b, a0, a1: np.where(b == 1, a1, a0)
    return (np.minimum(fi0 + pick(fo0, gi0, gi1), SAT), np.minimum(fi1 + pick(fo1, gi0, gi1), SAT),
            pick(fo0, go0, go1).astype(np.uint8), pick(fo1, go0, go1).astype(np.uint8))


def inclusive_scan(maps):
    """Hillis-Steele inclusive scan of row maps (the order of composition a block scan uses)."""
    m = tuple(np.array(a) for a in maps)
    n, d = len(m[0]), 1
    ident = (np.uint64(0), np.uint64(0), np.uint8(0), np.uint8(1))
    while d < n:
        prev = tuple(np.concatenate([np.full(d, e, dtype=a.dtype), a[:-d]]) for e, a in zip(ident, m))
        m = compose(prev, m)
        d *= 2
    return m


def exact_cumsum(x32: np.ndarray, chunk: int = CHUNK):
    """np.cumsum(float64(x32)) for non-negative x32, stretch by stretch.  Returns (cdf, info): info counts the stretches,
    the rows whose addition was an exact half-ulp tie and the stretches that ended by rounding up onto the next binade."""
    x = np.asarray(x32, np.float32).astype(np.float64)
    num = len(x)
    out = np.empty(num, np.float64)
    c, pos, stretches, ties, roundup = 0.0, 0, 0, 0, 0
    while pos < num:
        xs = x[pos:pos + chunk]
        if c == 0.0:  # leading zero rows
            nz = np.flatnonzero(xs > 0)
            if len(nz) == 0:
                out[pos:pos + len(xs)] = 0.0
                pos += len(xs)
                continue
            k = int(nz[0])
            out[pos:pos + k] = 0.0
            out[pos + k] = c = xs[k]
            pos += k + 1
            stretches += 1
            continue
        cb = int(np.float64(c).view(np.uint64))
        E, C0 = cb >> 52, (cb & ((1 << 52) - 1)) | (1 << 52)
        maps = row_maps(xs, E)
        inc0, inc1, _, _ = inclusive_scan(maps)
        val = np.uint64(C0) + (inc1 if C0 & 1 else inc0)
        crossed = np.flatnonzero(val >= TOP)
        k = int(crossed[0]) if len(crossed) else len(xs)
        ties += int(np.count_nonzero(maps[0][:k + 1] != maps[1][:k + 1]))
        grid = ((np.uint64(E) << np.uint64(52)) + val[:k] - HIDDEN).view(np.float64)
        out[pos:pos + k] = grid
        if k == len(xs):
            c = float(grid[-1])
            pos += k
            continue
        prev = float(grid[-1]) if k else c
        if val[k] == TOP:
            c = float(((np.uint64(E) << np.uint64(52)) + val[k] - HIDDEN).view(np.float64))
            roundup += Fraction(prev) + Fraction(float(xs[k])) < Fraction(c)
        else:
            c = prev + float(xs[k])
        out[pos + k] = c
        pos += k + 1
        stretches += 1
    return out, dict(stretches=stretches, ties=ties, roundup=int(roundup))


# ---- the whole draw -------------------------------------------------------------------------------------------------

def sample(q: np.ndarray, size: int, uniforms: np.ndarray, beta=0):
    """priority_sample's indices and weights from the restated sums.  Raises NumPy's ValueErrors."""
    q = np.asarray(q, np.float32)
    s = pairwise_sum(q)
    x = (q / s).astype(np.float32)
    p = x.astype(np.float64)
    with np.errstate(invalid="ignore"):
        if np.isnan(p).any() or (len(p) > 2 and np.isinf(p[:-1]).any()):
            raise ValueError("probabilities contain NaN")
        if (p < 0).any():
            raise ValueError("probabilities are not non-negative")
    cdf, _ = exact_cumsum(x)
    if np.isinf(p[-1]) or abs(cdf[-1] - 1.0) > SUM_ATOL:
        raise ValueError("probabilities do not sum to 1")
    idx = (cdf / cdf[-1]).searchsorted(uniforms, side="right").astype(np.int64)
    w = ((1.0 / size) / x[idx]) ** beta
    return idx, (w / np.max(w)).astype(np.float32)


# ---- constructed rings ----------------------------------------------------------------------------------------------

def _f32_exact(v: float):
    v32 = np.float32(v)
    return v32 if np.isfinite(v32) and v32 > 0 and float(v32) == v else None


def constructed_ring(n: int, seed: int = 0, zeros: int = 3) -> np.ndarray:
    """Float32 priorities whose cumulative sum (after q / np.sum(q)) is hard for any reordered sum: leading zero rows,
    many exact half-ulp ties, and binade crossings that land on the next binade by rounding up (a tie or a remainder
    above one half).  np.sum of the ring is a power of two, so q / s scales every row exactly and keeps those
    properties; the last row balances the sum to that power of two."""
    rng = np.random.default_rng(seed)
    q = np.zeros(n, np.float32)
    i = min(zeros, max(0, n - 2))
    c = 0.0
    pending = []
    while i < n - 1:
        if c == 0.0:
            v = _f32_exact(2.0 ** -40)
        elif pending:
            v = pending.pop(0)
        else:
            u = float(np.spacing(c))
            kind = rng.random()
            v = None
            if kind < 0.45:  # an exact half-ulp tie
                v = _f32_exact((2 * int(rng.integers(0, 8)) + 1) * u / 2)
            elif kind < 0.55 and c < 2.0 ** 10:  # walk to within a few ulps of the binade's top, then round up onto it
                top = 2.0 ** (np.frexp(c)[1])
                a1 = np.float32(top - c)
                if float(a1) > top - c:
                    a1 = np.nextafter(a1, np.float32(0))
                a1 = _f32_exact(float(a1))
                if a1 is not None:
                    c2 = c + float(a1)
                    a2 = np.float32(top - c2)
                    if float(a2) > top - c2:
                        a2 = np.nextafter(a2, np.float32(0))
                    a2 = _f32_exact(float(a2)) if top - c2 > 0 else None
                    c3 = c2 + (float(a2) if a2 is not None else 0.0)
                    k = (top - c3) / float(np.spacing(c3))
                    last = _f32_exact((k - float(rng.choice([0.25, 0.5]))) * float(np.spacing(c3))) if 0 < k < 2 ** 21 else None
                    pending = [x for x in (a2, last) if x is not None]
                    v = a1
            if v is None:  # heavy-tailed, well below the running sum
                v = _f32_exact(float(np.float32(c * 10.0 ** rng.uniform(-14, -5))))
        if v is None:
            continue
        q[i] = v
        c += float(v)
        i += 1
    # balance: the last row brings np.sum to a power of two
    s = np.float32(np.sum(q[:-1])) if n > 1 else np.float32(0)
    for up in (1, 2, 3):
        target = np.float32(2.0 ** (np.frexp(float(s))[1] + up)) if s > 0 else np.float32(1)
        z = np.float32(target - s)
        for _ in range(400):
            q[-1] = z
            t = np.sum(q)
            if t == target:
                return q
            z = np.nextafter(z, np.float32(np.inf) if t < target else np.float32(0))
    raise RuntimeError("could not balance the constructed ring")
