"""hmz_episode_ingest / EpisodeStore.ingest: the episode store filled from move records (e.g. the all-gather of every
rank's move) equals, bit for bit, the store hmz_selfplay_move writes itself, and so does every replay row made from it.
The argument checks at the end run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import port

FIELDS = ("state", "action", "flags", "visits", "root_q", "cur_slot", "ep_len", "exp")


def _selfplay(n, max_steps, B, S, mode=0, offset=0, episodes=False, seed=3, start=None):
    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200.engine import PackedWeights, SelfPlay

    w = PackedWeights(port.make_weights(n, 2), n, mode)
    sp = SelfPlay(n, max_steps, B, S, w, seed=seed, latent_dtype=_lib.LATENT_BF16 if mode == _lib.MODE_BF16 else _lib.LATENT_F32,
                  episodes=episodes, game_offset=offset)
    if start is not None:
        sp.env.words.copy_(start)
    return sp


def _assert_stores_equal(a, b, what):
    for k in FIELDS:
        assert torch.equal(getattr(a, k), getattr(b, k)), (what, k)


def _exponent(temperature):
    return 1 if temperature == 0 else int(min(5.0, max(1.0, 1.0 / temperature)))


def _restate_ingest(ref, rec, n_disks, t_max, exponent):
    """NumPy restatement of the ingest of one move into a store of t_max slots (the slot clamp included)."""
    t = np.minimum(rec["state"].view(np.uint32) >> (2 * n_disks), t_max - 1).astype(np.int64)
    g = np.arange(len(t))
    ref["state"][t, g] = rec["state"]
    ref["action"][t, g] = rec["action"]
    ref["flags"][t, g] = rec["flags"]
    ref["visits"][t, g] = rec["visits"]
    ref["root_q"][t, g] = rec["root_q"]
    ref["exp"][t, g] = exponent
    ref["cur_slot"][:] = t
    ref["ep_len"][:] = np.where(rec["flags"] & 1, t + 1, 0)
    return int((rec["state"].view(np.uint32) >> (2 * n_disks) >= t_max).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("n,max_steps,B,moves", [(3, 12, 256, 40), (5, 40, 200, 60)])
def test_ingest_equals_the_selfplay_writer(n, max_steps, B, moves):
    """SelfPlay(episodes=True) writes its store in the move's own kernel; a second store is fed the same move's records.
    After every move all store arrays agree, across goals, truncations, auto-resets and a temperature schedule that
    changes within episodes (1 -> 0.5 -> 0.25: exponents 1, 2, 4).  A store with t_max < max_steps checks the slot clamp
    against a NumPy restatement.  Replay rings built from the two stores are identical."""
    from muzero_hanoi_b200 import dist as hdist
    from muzero_hanoi_b200.engine import VecHanoi
    from muzero_hanoi_b200.replay import EpisodeStore, ReplayRing

    start = VecHanoi(n, max_steps, B)
    start.random_reset(seed=11)  # games start all over the state space: some reach the goal within a few moves
    sp = _selfplay(n, max_steps, B, 16, episodes=True, start=start.words)
    fed = EpisodeStore(B, max_steps, n)
    t_small = max_steps // 3
    clamped = EpisodeStore(B, t_small, n)
    ref = {k: np.zeros(v.shape, v.cpu().numpy().dtype) for k, v in
           (("state", clamped.state), ("action", clamped.action), ("flags", clamped.flags), ("visits", clamped.visits),
            ("root_q", clamped.root_q), ("cur_slot", clamped.cur_slot), ("ep_len", clamped.ep_len))}
    ref["exp"] = np.ones((t_small, B), np.uint8)
    rings = [ReplayRing(20000, 5, 3 * n, 6) for _ in range(2)]
    gen = torch.Generator(device="cuda").manual_seed(5)
    seen = dict(goal=0, trunc=0, clamp=0, mixed=0)
    for m in range(moves):
        sp.temperature = (1.0, 0.5, 0.25)[3 * m // moves]
        t = sp.move()
        fed.ingest(sp.slot(t), sp.temperature)
        clamped.ingest(sp.slot(t), sp.temperature)
        torch.cuda.synchronize()
        _assert_stores_equal(sp.episodes, fed, m)
        rec = {k: v.cpu().numpy() for k, v in hdist.unpack_records(sp.slot(t)).items()}
        seen["clamp"] += _restate_ingest(ref, rec, n, t_small, _exponent(sp.temperature))
        for k in FIELDS:
            assert np.array_equal(getattr(clamped, k).cpu().numpy(), ref[k]), (m, "clamped", k)
        seen["goal"] += int((rec["flags"] & 4).astype(bool).sum())
        seen["trunc"] += int((rec["flags"] & 8).astype(bool).sum())
        absorbing = torch.randint(0, 6, (B,), dtype=torch.uint8, device="cuda", generator=gen)
        for ring, st in zip(rings, (sp.episodes, fed)):
            st.post_process(10, 0.8)
            ring.add_episodes(st, temperature=sp.temperature, only_solved=False, absorbing_action=absorbing)
        _assert_stores_equal(sp.episodes, fed, m)
        assert torch.equal(sp.episodes.returns, fed.returns) and torch.equal(sp.episodes.priority, fed.priority)
        ep_len, exp = fed.ep_len.cpu().numpy(), fed.exp.cpu().numpy()
        seen["mixed"] += sum(len(np.unique(exp[:ep_len[g], g])) > 1 for g in np.nonzero(ep_len)[0])  # finished across a change
    assert min(seen.values()) > 0, seen
    assert int(fed.mismatch.item()) == 0 and int(clamped.mismatch.item()) == 0
    assert len(rings[0]) > 0 and rings[0].ptr == rings[1].ptr and rings[0].is_full == rings[1].is_full
    for name in ("states", "rwds", "actions", "pi_probs", "mc_returns", "priorities"):
        assert torch.equal(getattr(rings[0], name), getattr(rings[1], name)), name


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_sharded_records_ingested_equal_one_selfplay(mode):
    """Three SelfPlay shards with their game offsets (what three ranks play): their records, concatenated in rank order
    as the all-gather leaves them, ingested into one store, equal the store of one SelfPlay over all the games."""
    from muzero_hanoi_b200.engine import VecHanoi
    from muzero_hanoi_b200.replay import EpisodeStore

    n, max_steps, B, S = 4, 30, 96, 20
    start = VecHanoi(n, max_steps, B)
    start.random_reset(seed=4)
    whole = _selfplay(n, max_steps, B, S, mode, episodes=True, start=start.words)
    k = B // 3
    shards = [_selfplay(n, max_steps, k, S, mode, offset=o, start=start.words[o:o + k]) for o in range(0, B, k)]
    store = EpisodeStore(B, max_steps, n)
    for m in range(40):
        temperature = 1.0 if m < 20 else 0.5
        whole.temperature = temperature
        for s in shards:
            s.temperature = temperature
        whole.move()
        gathered = torch.cat([s.slot(s.move()) for s in shards])
        store.ingest(gathered, temperature)
        torch.cuda.synchronize()
        _assert_stores_equal(whole.episodes, store, m)
    assert int(store.mismatch.item()) == 0


@pytest.mark.gpu
def test_records_out_of_order_write_nothing_and_are_counted():
    """Records rolled by one game (or ingested with the wrong game offset) fail the game_lo check: no store row changes
    and every record is counted."""
    from muzero_hanoi_b200.replay import EpisodeStore

    n, max_steps, B = 3, 20, 300
    sp = _selfplay(n, max_steps, B, 8, offset=0)
    store = EpisodeStore(B, max_steps, n)
    t = sp.move()
    store.ingest(sp.slot(t), 1.0)
    torch.cuda.synchronize()
    before = {k: getattr(store, k).clone() for k in FIELDS}
    t = sp.move()
    store.ingest(torch.roll(sp.slot(t), 1, 0), 1.0)
    store.ingest(sp.slot(t), 1.0, game_offset=1)
    torch.cuda.synchronize()
    assert int(store.mismatch.item()) == 2 * B
    for k in FIELDS:
        assert torch.equal(getattr(store, k), before[k]), k
    store.ingest(sp.slot(t), 1.0)  # in order: written, and the count stays
    torch.cuda.synchronize()
    assert int(store.mismatch.item()) == 2 * B and not torch.equal(store.cur_slot, before["cur_slot"])


def test_ingest_argument_validation_without_gpu(lib):
    """Null pointers, negative sizes and a non-integer play-policy exponent are rejected before any CUDA call."""
    from muzero_hanoi_b200 import _lib

    B, T = 4, 8
    rec = (ctypes.c_uint64 * (4 * B + 2))()  # a 16-byte aligned start inside it
    rec_p = ctypes.addressof(rec) + (-ctypes.addressof(rec)) % 16
    bufs = [(ctypes.c_uint64 * (T * B * 2))() for _ in range(9)]
    state, action, flags, visits, root_q, cur_slot, ep_len, exp, mismatch = bufs

    def call(records=rec_p, n=B, t_max=T, temperature=1.0, **null):
        args = dict(state=state, action=action, flags=flags, visits=visits, root_q=root_q, cur_slot=cur_slot, ep_len=ep_len,
                    exp=exp, mismatch=mismatch)
        args.update(null)
        return lib.hmz_episode_ingest(records, n, 0, 3, t_max, temperature, *(args[k] for k in (
            "state", "action", "flags", "visits", "root_q", "cur_slot", "ep_len", "exp", "mismatch")), None)

    for k in ("state", "action", "flags", "visits", "root_q", "cur_slot", "ep_len", "mismatch"):
        assert call(**{k: None}) == _lib.ERR_INVALID, k
    assert call(records=None) == _lib.ERR_INVALID
    assert call(records=rec_p + 8) == _lib.ERR_INVALID and b"aligned" in lib.hmz_last_error()
    assert call(n=-1) == _lib.ERR_INVALID
    assert call(t_max=0) == _lib.ERR_INVALID
    assert call(temperature=1.5) == _lib.ERR_INVALID
    assert call(temperature=0.4) == _lib.ERR_UNSUPPORTED
    assert b"integer play-policy exponents" in lib.hmz_last_error()
    assert call(n=0) == _lib.OK  # nothing to do: no CUDA call either
