"""oracle/episode_ref.py, the vectorised restatement the episode kernels are checked against on the GPU
(tests/test_episode_reference_gpu.py), pinned without a GPU:

* to the per-episode functions of oracle/port.py that gen_golden checked against the unmodified reference
  (n_step_returns, mc_returns, priorities, play_policy, organise_transitions) plus a literal sequential Buffer.add, bit
  for bit, on thousands of random episodes over the GPU tests' case grid;
* to np.power's play policies for every visit count up to the stated bound, POLICY_EXACT_MAX = 1,554;
* as sharp: seven plausible kernel bugs, each restated, change at least a stated number of elements of the GPU tests'
  own inputs, so a green GPU run rules them out."""
import numpy as np
import pytest

from oracle import episode_ref as er
from oracle import port

TEMPERATURE_OF = {1: 1.0, 2: 0.5, 5: 0.2}  # a temperature with that play-policy exponent


def _port_rewards(flags):
    return [100 if f & er.FLAG_GOAL else (-100 / 1000 if f & er.FLAG_ILLEGAL else 0) for f in flags]


def _cpu_games(t_max, n_step):
    """How many games of a case the per-episode port loops check (they cost t_max * n_step Python steps each)."""
    if t_max >= 1000:
        return 8
    if t_max >= 200:
        return 160 if n_step <= 50 else 40
    return None  # all of them


@pytest.mark.parametrize("case", er.RETURN_CASES, ids=lambda c: f"T{c[0]}-n{c[1]}-d{c[2]}")
def test_returns_and_priorities_equal_port(case):
    t_max, n_step, discount, B, illegal, seed = case
    B = _cpu_games(t_max, n_step) or B
    st = er.random_store(seed, B, t_max, illegal=illegal)
    td = er.n_step_returns(st.flags, st.root_q, st.ep_len, n_step, discount)
    mc = er.mc_returns(st.flags, st.root_q, st.ep_len, discount)
    assert len(td.cols) > B // 2 and {1, t_max} <= set(td.lens.tolist())
    for c, g in enumerate(td.cols):
        L = int(td.lens[c])
        rw, q = _port_rewards(st.flags[:L, g]), [float(x) for x in st.root_q[:L, g]]
        ret = port.n_step_returns(rw, q, n_step, discount)
        assert np.array_equal(td.returns[:L, c], np.array(ret)), (g, L)
        assert np.array_equal(td.priority[:L, c], port.priorities(ret, q)), g
        ret = port.mc_returns(rw, discount)
        assert np.array_equal(mc.returns[:L, c], np.array(ret)), (g, L)
        assert np.array_equal(mc.priority[:L, c], port.priorities(ret, q)), g


def _sequential_ring(case, st, absorbing, only_solved):
    """The reference's own order of operations: per stored episode, port's returns, play policies and
    organise_transitions, then one Buffer.add (buffer.py:47-83) on NumPy arrays."""
    t_max, n_disks, unroll, exps, temperature, capacity, ptr0 = case[:7]
    ring = er.Ring(capacity, unroll, 3 * n_disks, fill=-7.0, ptr=ptr0)
    for g in np.nonzero(st.ep_len)[0]:
        L = int(st.ep_len[g])
        rw, q = _port_rewards(st.flags[:L, g]), [float(x) for x in st.root_q[:L, g]]
        ret = port.n_step_returns(rw, q, er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
        if only_solved and not ret[-1] > 0:
            continue
        temps = [TEMPERATURE_OF[int(e)] for e in st.exp[:L, g]] if st.exp is not None else [temperature] * L
        pis = [port.play_policy(st.visits[t, g].astype(np.int64), temps[t]) for t in range(L)]
        states = [port.one_hot(port.packed_to_state(int(w) & ((1 << 2 * n_disks) - 1), n_disks)) for w in
                  st.state[:L, g].view(np.uint32)]
        s, o_r, o_a, o_p, o_g = port.organise_transitions(states, rw, [int(a) for a in st.action[:L, g]], pis, ret, unroll,
                                                          6, int(absorbing[g]))
        rows = (ring.ptr + np.arange(L)) % capacity
        for name, x in (("states", s), ("rwds", o_r), ("actions", o_a), ("pi_probs", o_p), ("mc_returns", o_g),
                        ("priorities", port.priorities(ret, q))):
            getattr(ring, name)[rows] = x
        ring._advance(L)
    return ring


def _small_unroll_cases():
    return [c for c in er.UNROLL_CASES if c[8] * c[0] <= 100_000]


def _faithful_ring(case, st=None, absorbing=None, **kw):
    t_max, n_disks, unroll, exps, temperature, capacity, ptr0, scalar, B, S, only_solved, seed = case
    if st is None:
        st, absorbing = er.unroll_case_store(case)
    post = er.n_step_returns(st.flags, st.root_q, st.ep_len, er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
    ring = er.Ring(capacity, unroll, 3 * n_disks, fill=-7.0, ptr=ptr0)
    n = ring.add_episodes(st, post, temperature, only_solved, absorbing, **kw)
    return ring, n, st, absorbing, post


@pytest.mark.parametrize("case", _small_unroll_cases(), ids=lambda c: f"T{c[0]}-N{c[1]}-K{c[2]}-cap{c[5]}-s{c[-1]}")
def test_ring_equals_organise_transitions_and_sequential_adds(case):
    """Every array of the ring, ptr and is_full, against port's per-episode functions and sequential adds.  The stores
    here have no visit counts above POLICY_EXACT_MAX (where np.power and the ring part ways by design)."""
    t_max, n_disks, unroll, exps, temperature, capacity, ptr0, scalar, B, S, only_solved, seed = case
    st = er.random_store(seed, B, t_max, n_disks, S=S, exponents=exps)
    absorbing = np.random.default_rng(seed + 1000).integers(0, 6, B).astype(np.uint8)
    ring, n, *_ = _faithful_ring(case, st, absorbing)
    seq = _sequential_ring(case, st, absorbing, only_solved)
    assert n > 0 and (ring.ptr, ring.is_full) == (seq.ptr, seq.is_full)
    for name in er.Ring.FIELDS:
        assert np.array_equal(getattr(ring, name), getattr(seq, name)), name
    if capacity == 37:
        assert n > capacity  # more rows than the ring holds: later rows overwrite earlier ones


@pytest.mark.parametrize("exponent", [1, 2, 5])
def test_play_policy_equals_numpy_for_every_count_up_to_the_bound(exponent):
    """Each count 0..1,554 at every position of the 6-element call, against port.play_policy's own call shape."""
    c = np.arange(er.POLICY_EXACT_MAX + 1, dtype=np.int64)
    rows = np.stack([c, (7 * c + 1) % 1555, er.POLICY_EXACT_MAX - c, (13 * c + 5) % 1555, c // 2, np.full_like(c, 1554)], 1)
    rows = np.concatenate([np.roll(rows, k, axis=1) for k in range(6)])
    got = er.play_policy(rows, exponent)
    for i, r in enumerate(rows):
        assert np.array_equal(got[i], port.play_policy(r, TEMPERATURE_OF[exponent])), (exponent, r)
    if exponent == 5:  # what the bound means: np.power and the products part ways just above it
        x = np.arange(er.POLICY_EXACT_MAX + 1, 65536, dtype=np.int64)
        xf = x.astype(np.float64)
        print(f"np.power(count, 5.0) differs from the repeated products at {int((np.power(x, 5.0) != xf * xf * xf * xf * xf).sum())}"
              f" of the counts {er.POLICY_EXACT_MAX + 1}-65535")


# ---- sharpness: each wrong restatement changes at least MIN elements of the GPU tests' inputs -------------------------
SHARP_MIN = dict(plain_sum=13000, libm_mc_powers=5000, f64_priority=20000, pad_last_action=12000, pad_zero_policy=90000,
                 first_write_wins=2_000_000, only_solved_ignored=500_000, add_temperature=1_000_000)


def test_the_case_grid_reaches_the_powers_that_differ():
    """The MC table is NumPy's power and the n-step table libm's: the grid holds a discount where they differ below
    t_max, so a kernel fed the wrong table fails the GPU returns test."""
    assert any((er.numpy_powers(d, T) != er.libm_powers(d, T)).any() for T, _, d, *_ in er.RETURN_CASES)


def _count(a, b, mask=None):
    d = a != b
    if a.dtype.kind == "f":
        d &= ~(np.isnan(a) & np.isnan(b))
    return int(d[mask].sum() if mask is not None else d.sum())


def test_wrong_restatements_change_the_gpu_tests_outputs():
    seen = dict.fromkeys(SHARP_MIN, 0)
    for t_max, n_step, discount, B, illegal, seed in er.RETURN_CASES:
        st = er.random_store(seed, B, t_max, illegal=illegal)
        td = er.n_step_returns(st.flags, st.root_q, st.ep_len, n_step, discount)
        wrong = er.n_step_returns(st.flags, st.root_q, st.ep_len, n_step, discount, summation=er.plain_rows)
        seen["plain_sum"] += _count(td.returns, wrong.returns, td.mask)
        f64 = np.abs(td.returns - st.root_q[:td.returns.shape[0], td.cols]).astype(np.float32)
        seen["f64_priority"] += _count(td.priority, f64, td.mask)
        mc = er.mc_returns(st.flags, st.root_q, st.ep_len, discount)
        wrong = er.mc_returns(st.flags, st.root_q, st.ep_len, discount, powers=er.libm_powers(discount, t_max))
        seen["libm_mc_powers"] += _count(mc.returns, wrong.returns, mc.mask)
    for B in er.ROWS_BATCHES:
        ep_len, ret = er.rows_case(B, B)
        last = ret[np.maximum(ep_len - 1, 0), np.arange(B)]
        for p in er.rows_ptrs(B):
            seen["only_solved_ignored"] += _count(er.row_bases(ep_len, last, p, True)[0], er.row_bases(ep_len, last, p, False)[0])
    for case in er.UNROLL_CASES:
        ring, n, st, absorbing, post = _faithful_ring(case)
        wrong, *_ = _faithful_ring(case, st, absorbing, last_write_wins=False)
        seen["first_write_wins"] += sum(_count(getattr(ring, k), getattr(wrong, k)) for k in er.Ring.FIELDS)
        if st.exp is not None:
            wrong, *_ = _faithful_ring(case, er.Store(**{**st.__dict__, "exp": None}), absorbing)
            seen["add_temperature"] += _count(ring.pi_probs, wrong.pi_probs)
        # padding slots: rows whose unroll runs past the episode end carry the absorbing action and the uniform policy
        pad = ring.pi_probs[..., 0] == np.float32(1 / 6)
        pad &= (ring.pi_probs == np.float32(1 / 6)).all(-1) & (ring.rwds == 0) & (ring.mc_returns == 0)
        last_action = _last_actions(ring)
        seen["pad_last_action"] += int((pad & (ring.actions != last_action)).sum())
        seen["pad_zero_policy"] += int(pad.sum()) * 6
    print({k: (seen[k], SHARP_MIN[k]) for k in seen})
    for k, v in seen.items():
        assert v >= SHARP_MIN[k], (k, v, SHARP_MIN[k])


def _last_actions(ring):
    """For every padded slot, the action of the last live slot of its row (what padding with the episode's last action
    would write there); -1 where the row has no live slot before it."""
    live = ~((ring.pi_probs == np.float32(1 / 6)).all(-1) & (ring.rwds == 0) & (ring.mc_returns == 0))
    idx = np.where(live, np.arange(ring.unroll)[None, :], -1)
    idx = np.maximum.accumulate(idx, axis=1)
    out = np.take_along_axis(ring.actions, np.maximum(idx, 0), 1)
    return np.where(idx >= 0, out, -1)
