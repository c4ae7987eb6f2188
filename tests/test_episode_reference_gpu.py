"""The episode kernels (hmz_episode.cu: returns, MC returns, priorities, episode_rows, both unroll forms, and the ingest of
gathered move records) against oracle/episode_ref.py, bit for bit, at the shapes training reaches: every n_step /
discount / t_max of the case grid, batches past every kernel's eighth wave (the grid-stride loops), episode_rows' chunk
carry up to 524,288 games, unroll at N = 1-12, K = 1-8, mixed per-step exponents, rings smaller than one move's rows,
and a rank-0 run of 8 x 65,536 games.  Outputs are filled with a sentinel first: what a kernel must not write keeps it.

Play policies at visit counts above 1,554 (episode_ref.POLICY_EXACT_MAX) are the repeated float64 products, not
np.power's values; the stores of the unroll cases with 1,554 simulations carry rows at that boundary."""
import numpy as np
import pytest
import torch

from oracle import episode_ref as er

pytestmark = pytest.mark.gpu
SENT_F64, SENT_F32 = -7.25e300, np.float32(-3.5)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view({8: np.uint64, 4: np.uint32, 2: np.uint16, 1: np.uint8}[a.dtype.itemsize])


def _equal_bits(a, b):
    return a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


def _device_store(st: er.Store):
    from muzero_hanoi_b200.replay import EpisodeStore

    d = EpisodeStore(st.B, st.t_max, st.n_disks)
    for name in ("state", "action", "flags", "visits", "root_q", "ep_len"):
        getattr(d, name).copy_(torch.from_numpy(np.ascontiguousarray(getattr(st, name))))
    if st.exp is not None:
        d.exp = torch.from_numpy(st.exp).cuda()
    d.returns.fill_(SENT_F64)
    d.priority.fill_(float(SENT_F32))
    return d


def _check_post(dev, ref: er.Post, ep_len):
    ret, prio = dev.returns.cpu().numpy(), dev.priority.cpu().numpy()
    L = ref.returns.shape[0]
    assert _equal_bits(ret[:L][:, ref.cols][ref.mask], ref.returns[ref.mask])
    assert _equal_bits(prio[:L][:, ref.cols][ref.mask], ref.priority[ref.mask])
    untouched = np.arange(ret.shape[0])[:, None] >= np.asarray(ep_len)[None, :]  # t >= ep_len, unfinished columns whole
    assert (ret[untouched] == SENT_F64).all() and (prio[untouched] == SENT_F32).all()


@pytest.mark.parametrize("mc", [False, True], ids=["td", "mc"])
@pytest.mark.parametrize("case", er.RETURN_CASES + er.RETURN_CASES_LARGE, ids=lambda c: f"T{c[0]}-n{c[1]}-d{c[2]}-B{c[3]}")
def test_returns_and_priorities_bit_exact(case, mc):
    t_max, n_step, discount, B, illegal, seed = case
    st = er.random_store(seed, B, t_max, illegal=illegal)
    dev = _device_store(st)
    if mc:
        dev.post_process_mc(discount)
        ref = er.mc_returns(st.flags, st.root_q, st.ep_len, discount)
    else:
        dev.post_process(n_step, discount)
        ref = er.n_step_returns(st.flags, st.root_q, st.ep_len, n_step, discount)
    torch.cuda.synchronize()
    _check_post(dev, ref, st.ep_len)


@pytest.mark.parametrize("only_solved", [False, True])
@pytest.mark.parametrize("B", er.ROWS_BATCHES)
def test_episode_rows_exact(B, only_solved):
    from muzero_hanoi_b200._lib import check, current_stream, ptr
    from muzero_hanoi_b200.replay import EpisodeStore

    ep_len, ret = er.rows_case(B, B)
    dev = EpisodeStore(B, ret.shape[0], 1)
    dev.ep_len.copy_(torch.from_numpy(ep_len))
    dev.returns.copy_(torch.from_numpy(ret))
    last = ret[np.maximum(ep_len - 1, 0), np.arange(B)]
    for p in er.rows_ptrs(B):
        dev.row_base.fill_(-12345)
        dev.total.fill_(-12345)
        check(dev.lib.hmz_episode_rows(ptr(dev.ep_len), ptr(dev.returns), B, p, int(only_solved), ptr(dev.row_base),
                                       ptr(dev.total), current_stream()))
        base, total = er.row_bases(ep_len, last, p, only_solved)
        assert np.array_equal(dev.row_base.cpu().numpy(), base), p
        assert int(dev.total.item()) == total, p


def _sentinel_ring(capacity, unroll, d_state, ptr0):
    from muzero_hanoi_b200.replay import ReplayRing

    ring = ReplayRing(capacity, unroll, d_state, 6)
    for name in er.Ring.FIELDS:
        getattr(ring, name).fill_(-7)
    ring.ptr = ptr0
    return ring


def _check_ring(dev, ref: er.Ring):
    assert (dev.ptr, dev.is_full) == (ref.ptr, ref.is_full)
    for name in er.Ring.FIELDS:
        assert _equal_bits(getattr(dev, name).cpu().numpy(), getattr(ref, name)), name


@pytest.mark.parametrize("case", er.UNROLL_CASES, ids=lambda c: f"T{c[0]}-N{c[1]}-K{c[2]}-cap{c[5]}-B{c[8]}-s{c[-1]}")
def test_unroll_into_the_ring_bit_exact(case, monkeypatch):
    """Warp form (t_max <= 279) and scalar form (t_max >= 280, or HMZ_UNROLL_SCALAR=1), against the reference's
    sequential adds: all six arrays, ptr and is_full; rows nothing wrote keep the sentinel."""
    t_max, n_disks, unroll, exps, temperature, capacity, ptr0, scalar, B, S, only_solved, seed = case
    if scalar:
        monkeypatch.setenv("HMZ_UNROLL_SCALAR", "1")
    st, absorbing = er.unroll_case_store(case)
    dev = _device_store(st)
    dev.post_process(er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
    ring = _sentinel_ring(capacity, unroll, 3 * n_disks, ptr0)
    n = ring.add_episodes(dev, temperature=temperature, only_solved=only_solved, absorbing_action=absorbing)
    post = er.n_step_returns(st.flags, st.root_q, st.ep_len, er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
    ref = er.Ring(capacity, unroll, 3 * n_disks, fill=-7.0, ptr=ptr0)
    assert n == ref.add_episodes(st, post, temperature, only_solved, absorbing) > 0
    torch.cuda.synchronize()
    _check_ring(ring, ref)


def test_repeated_calls_are_bit_identical():
    """Two identical calls of every episode kernel give bit-identical outputs."""
    case = er.UNROLL_CASES[1]
    t_max, n_disks, unroll, exps, temperature, capacity, ptr0, scalar, B, S, only_solved, seed = case
    st, absorbing = er.unroll_case_store(case)
    outs = []
    for _ in range(2):
        dev = _device_store(st)
        mc = [x.clone() for x in dev.post_process_mc(0.97)]
        td = dev.post_process(er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
        ring = _sentinel_ring(capacity, unroll, 3 * n_disks, ptr0)
        ring.add_episodes(dev, temperature=temperature, only_solved=False, absorbing_action=absorbing)
        outs.append(mc + [x.clone() for x in td] + [dev.row_base.clone(), dev.total.clone()] +
                    [getattr(ring, k).clone() for k in er.Ring.FIELDS])
    for a, b in zip(*outs):
        assert torch.equal(a.view(torch.uint8) if a.dtype.is_floating_point else a,
                           b.view(torch.uint8) if b.dtype.is_floating_point else b)


def test_rank0_scale_ingest_post_process_and_ring():
    """What rank 0 runs each move at 8 GPUs: 8 x 65,536 games' records (eight rank blocks with their game offsets,
    packed with dist.pack_records), ingest, post_process, add_episodes(only_solved=True).  After every move the
    written store slots, returns and priorities of every finished episode, and the whole 50,000-row ring equal the
    reference; the whole store is compared at the end.  About 4.3 GB of device memory."""
    from muzero_hanoi_b200 import dist as hdist
    from muzero_hanoi_b200.replay import EpisodeStore

    R, per, N, T, K, cap, S, moves = 8, 65536, 3, 200, 5, 50000, 25, 8
    G = R * per
    rng = np.random.default_rng(2024)
    dev = EpisodeStore(G, T, N)
    ring = _sentinel_ring(cap, K, 3 * N, 0)
    ref = er.Store(np.zeros((T, G), np.int32), np.zeros((T, G), np.uint8), np.zeros((T, G), np.uint8),
                   np.ones((T, G, 6), np.int16), np.zeros((T, G)), np.zeros(G, np.int32), np.ones((T, G), np.uint8), N)
    dev.visits.fill_(1)  # slots before a game's first recorded move: a uniform policy rather than 0 / 0
    rring = er.Ring(cap, K, 3 * N, fill=-7.0)
    step = rng.integers(0, T, G)  # games mid-episode at every step counter: long episodes and truncations from move 1
    game_lo = np.tile(np.arange(per, dtype=np.int64), R).astype(np.uint16).view(np.int16)
    seen = dict(stored=0, wraps=0, trunc=0, long=0)
    for m in range(moves):
        temperature = (1.0, 0.5, 0.1)[3 * m // moves]
        pegs = np.zeros(G, np.int64)
        for d in range(N):
            pegs |= rng.integers(0, 3, G) << (2 * d)
        word = (pegs | (step << (2 * N))).astype(np.uint32).view(np.int32)
        flags = np.where(rng.random(G) < 0.2, er.FLAG_ILLEGAL, 0)
        goal = rng.random(G) < 0.12
        flags = np.where(goal, er.FLAG_GOAL | er.FLAG_DONE, np.where(step == T - 1, flags | er.FLAG_TRUNC | er.FLAG_DONE, flags))
        fields = dict(root_q=er.random_root_values(rng, G), state=word, reward=er.rewards(flags).astype(np.float32),
                      visits=er.random_visits(rng, G, S), action=rng.integers(0, 6, G).astype(np.uint8),
                      flags=flags.astype(np.uint8), game_lo=game_lo)
        records = torch.cat([hdist.pack_records({k: torch.from_numpy(np.ascontiguousarray(v[r * per:(r + 1) * per])).cuda()
                                                 for k, v in fields.items()}) for r in range(R)])
        dev.ingest(records, temperature)
        dev.post_process(er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
        absorbing = rng.integers(0, 6, G).astype(np.uint8)
        n = ring.add_episodes(dev, temperature=temperature, only_solved=True, absorbing_action=absorbing)
        # the reference: the ingest's store writes, then the post-processing and the sequential adds
        g = np.arange(G)
        ref.state[step, g], ref.action[step, g], ref.flags[step, g] = word, fields["action"], fields["flags"]
        ref.visits[step, g], ref.root_q[step, g], ref.exp[step, g] = fields["visits"], fields["root_q"], er.exponent_of(temperature)
        ref.ep_len[:] = np.where(flags & er.FLAG_DONE, step + 1, 0)
        post = er.n_step_returns(ref.flags, ref.root_q, ref.ep_len, er.UNROLL_N_STEP, er.UNROLL_DISCOUNT)
        wrapped = rring.ptr
        assert n == rring.add_episodes(ref, post, temperature, True, absorbing), m
        torch.cuda.synchronize()
        assert int(dev.mismatch.item()) == 0
        assert np.array_equal(dev.ep_len.cpu().numpy(), ref.ep_len) and np.array_equal(dev.cur_slot.cpu().numpy(), step)
        slot = torch.from_numpy(step).cuda()[None, :]
        for name in ("state", "action", "flags", "root_q", "exp"):
            assert _equal_bits(getattr(dev, name).gather(0, slot)[0].cpu().numpy(), getattr(ref, name)[step, g]), (m, name)
        assert np.array_equal(dev.visits.gather(0, slot[..., None].expand(1, G, 6))[0].cpu().numpy(), ref.visits[step, g])
        L = post.returns.shape[0]
        cols = torch.from_numpy(post.cols).cuda()
        mask = post.mask
        assert _equal_bits(dev.returns[:L].index_select(1, cols).cpu().numpy()[mask], post.returns[mask]), m
        assert _equal_bits(dev.priority[:L].index_select(1, cols).cpu().numpy()[mask], post.priority[mask]), m
        _check_ring(ring, rring)
        seen["stored"] += n
        seen["wraps"] += int(n >= cap or rring.ptr < wrapped)
        seen["trunc"] += int((flags & er.FLAG_TRUNC).astype(bool).sum())
        seen["long"] += int((post.lens > 150).sum())
        step = np.where(flags & er.FLAG_DONE, 0, step + 1)
    for name in ("state", "action", "flags", "visits", "root_q", "exp"):
        assert _equal_bits(getattr(dev, name).cpu().numpy(), getattr(ref, name)), name
    print(seen)
    assert seen["wraps"] == moves and min(seen.values()) > 0, seen
