"""GPU: throughput-mode randomness and the fused begin / end-of-move kernels of hmz_selfplay_move.

The reference draws np.random.dirichlet (MCTS/mcts.py:149) and np.random.choice (:120) from NumPy's global Mersenne
twister; the batched engine cannot reproduce that stream (parity mode takes the draws as INPUTS instead), so the
on-device generator is validated for what it is: Philox4x32-10 against the published known-answer vectors, the uniform
and Dirichlet moments, and the keying by GLOBAL game id (results invariant to the sharding, SURVEY.md §8e).  Every draw
is also compared element by element with oracle/move_ref.py's restatement, and the laws with their exact CDFs, in
tests/test_move_reference_{cpu,gpu}.py.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cport, port
from oracle.move_ref import philox_host as _philox_host

pytestmark = pytest.mark.gpu


# Random123 kat_vectors, philox4x32 with 10 rounds: (counter, key) -> output
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


def test_philox_known_answers(lib):
    from muzero_hanoi_b200 import _lib

    for c, k, want in KAT:
        assert tuple(_philox_host(c, k)) == want  # the host restatement used below is itself pinned
    rng = np.random.default_rng(0)
    extra = rng.integers(0, 2 ** 32, (500, 6), dtype=np.uint64).astype(np.uint32)
    inp = np.concatenate([np.array([list(c) + list(k) for c, k, _ in KAT], np.uint32), extra])
    d_in = torch.from_numpy(inp.view(np.int32)).cuda()
    d_out = torch.empty(len(inp), 4, dtype=torch.int32, device="cuda")
    _lib.check(lib.hmz_debug_philox(_lib.ptr(d_in), _lib.ptr(d_out), len(inp), _lib.current_stream()))
    got = d_out.cpu().numpy().view(np.uint32)
    for i, (_, _, want) in enumerate(KAT):
        assert tuple(int(x) for x in got[i]) == want
    for i in range(3, len(inp)):
        assert [int(x) for x in got[i]] == _philox_host([int(x) for x in inp[i, :4]], [int(x) for x in inp[i, 4:]])


def _uniform(lib, n, seed, counter, offset):
    from muzero_hanoi_b200 import _lib

    out = torch.empty(n, dtype=torch.float64, device="cuda")
    _lib.check(lib.hmz_rng_uniform(_lib.ptr(out), n, seed, counter, offset, _lib.current_stream()))
    return out.cpu().numpy()


def _dirichlet(lib, n, alpha, seed, counter, offset):
    from muzero_hanoi_b200 import _lib

    out = torch.empty(n, 6, dtype=torch.float64, device="cuda")
    _lib.check(lib.hmz_rng_dirichlet(_lib.ptr(out), n, float(alpha), seed, counter, offset, _lib.current_stream()))
    return out.cpu().numpy()


def test_uniform_is_philox_keyed_by_global_item(lib):
    seed, counter = 0x1234567890ABCDEF, (7 << 32) | 99
    u = _uniform(lib, 4096, seed, counter, 1000)
    for i in (0, 1, 17, 4095):  # bit for bit: 53 high bits of the first two output words of block (item, counter)
        item = 1000 + i
        r = _philox_host([item & 0xFFFFFFFF, item >> 32, counter & 0xFFFFFFFF, counter >> 32],
                         [(seed & 0xFFFFFFFF) ^ 0x554E4946, seed >> 32])
        assert u[i] == float(((r[0] << 32) | r[1]) >> 11) / 2.0 ** 53
    # sharding invariance: items [1000, 5096) drawn as one batch or as two batches with their own offsets
    assert np.array_equal(u, np.concatenate([_uniform(lib, 1500, seed, counter, 1000), _uniform(lib, 2596, seed, counter, 2500)]))
    assert not np.array_equal(u, _uniform(lib, 4096, seed, counter + 1, 1000))
    big = _uniform(lib, 1 << 20, 5, 0, 0)
    assert big.min() >= 0.0 and big.max() < 1.0
    n = len(big)
    assert abs(big.mean() - 0.5) < 5 * np.sqrt(1 / 12 / n) and abs(big.var() - 1 / 12) < 5 * np.sqrt(1 / 180 / n)
    hist = np.histogram(big, bins=64, range=(0, 1))[0]
    assert (np.abs(hist - n / 64) < 6 * np.sqrt(n / 64)).all()


@pytest.mark.parametrize("alpha", [0.25, 1.0, 3.0])
def test_dirichlet_moments_and_keying(lib, alpha):
    """Dirichlet(alpha * 1_6): mean 1/6, Var = (1/6)(5/6) / (6 alpha + 1), Cov = -(1/36) / (6 alpha + 1) — the law of
    np.random.dirichlet at MCTS/mcts.py:148-149 (alpha = 0.25 -> variance (5/36) / 2.5)."""
    n = 400_000
    x = _dirichlet(lib, n, alpha, 77, 3, 0)
    assert np.abs(x.sum(1) - 1.0).max() < 1e-12 and x.min() >= 0.0
    a0 = 6 * alpha
    var, cov = (1 / 6) * (5 / 6) / (a0 + 1), -(1 / 36) / (a0 + 1)
    assert np.abs(x.mean(0) - 1 / 6).max() < 6 * np.sqrt(var / n)
    assert np.abs(x.var(0) / var - 1).max() < 0.02
    c = np.cov(x.T)
    off = c[~np.eye(6, dtype=bool)]
    assert np.abs(off / cov - 1).max() < 0.05
    # third moment of a coordinate ~ Beta(alpha, 5 alpha): E[x^3] = a(a+1)(a+2) / (a0 (a0+1) (a0+2))
    m3 = alpha * (alpha + 1) * (alpha + 2) / (a0 * (a0 + 1) * (a0 + 2))
    assert np.abs((x ** 3).mean(0) / m3 - 1).max() < 0.03
    # keyed by global item: any split of the batch draws the same rows
    assert np.array_equal(x[:5000], np.concatenate([_dirichlet(lib, 1234, alpha, 77, 3, 0), _dirichlet(lib, 3766, alpha, 77, 3, 1234)]))


def _selfplay(n, B, S, mode, offset, seed=9, alpha=0.25, temperature=1.0, words=None):
    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200.engine import PackedWeights, SelfPlay

    w = PackedWeights(port.make_weights(n, 2), n, mode)
    sp = SelfPlay(n, 200, B, S, w, alpha=alpha, temperature=temperature, seed=seed, ring_slots=4,
                  latent_dtype=_lib.LATENT_BF16 if mode == _lib.MODE_BF16 else _lib.LATENT_F32, game_offset=offset)
    if words is not None:
        sp.env.words.copy_(words)
    return sp


@pytest.mark.parametrize("mode", [0, 1])
def test_selfplay_records_do_not_depend_on_the_sharding(mode):
    """96 games played as ONE batch or as two batches of 48 with game_offset 0 / 48 (what two ranks would do): every
    move record (state, action, reward, flags, visit counts, float64 root value, game id) is identical."""
    from muzero_hanoi_b200 import dist as hdist
    from muzero_hanoi_b200.engine import VecHanoi

    n, B, S, moves = 4, 96, 20, 5
    start = VecHanoi(n, 200, B)
    start.random_reset(seed=4)
    whole = _selfplay(n, B, S, mode, 0, words=start.words)
    halves = [_selfplay(n, B // 2, S, mode, off, words=start.words[off:off + B // 2]) for off in (0, B // 2)]
    for _ in range(moves):
        t = whole.move()
        ts = [h.move() for h in halves]
        torch.cuda.synchronize()
        a = hdist.unpack_records(whole.slot(t))
        b = hdist.unpack_records(torch.cat([h.slot(x) for h, x in zip(halves, ts)]))
        for k in hdist.RECORD_FIELDS:
            assert torch.equal(a[k], b[k]), k
        assert torch.equal(a["game_lo"].cpu(), torch.arange(B, dtype=torch.int16))
        assert torch.equal(whole.env.words, torch.cat([h.env.words for h in halves]))


@pytest.mark.parametrize("alpha,temperature", [(0.25, 1.0), (0.0, 0.5), (0.25, 0.1)])
def test_fused_move_kernels_equal_the_split_entry_points(lib, alpha, temperature):
    """hmz_selfplay_move's two fused kernels against the separately exported steps they replace: hmz_rng_dirichlet +
    hmz_rng_uniform + hmz_search_begin_p0 (start of the move) and hmz_search_root_policy + hmz_env_step + the record
    (end of the move); the env part also against the C oracle."""
    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200 import dist as hdist

    n, B, S, offset, seed = 5, 200, 24, 5000, 31
    sp = _selfplay(n, B, S, 0, offset, seed=seed, alpha=alpha, temperature=temperature)
    sp.env.random_reset(seed=8)
    for move in range(3):
        before = sp.env.words.clone()
        t = sp.move()
        torch.cuda.synchronize()
        u = _uniform(lib, B, seed, move, offset)
        assert np.array_equal(sp.uniform.cpu().numpy(), u)
        p0 = sp.p0.cpu().numpy()
        prior = sp.mcts.store.root_prior.cpu().numpy()
        if alpha > 0:
            nz = _dirichlet(lib, B, alpha, seed, move, offset)
            assert np.array_equal(sp.noise.cpu().numpy(), nz)
            assert np.array_equal(prior, port.mix_dirichlet(p0, nz))
        else:
            assert np.array_equal(prior, p0.astype(np.float64))
        visits, root_q, action = sp.mcts.visits.clone(), sp.mcts.root_q.clone(), sp.mcts.action.clone()
        act2, pi2, q2, visits2 = sp.mcts.root_policy(temperature, False, uniforms=sp.uniform)  # same tree, split entry point
        torch.cuda.synchronize()
        assert torch.equal(visits, visits2) and torch.equal(root_q, q2) and torch.equal(action, act2)
        want_pi = np.stack([port.play_policy(v, temperature) for v in visits.cpu().numpy()])
        assert np.array_equal(pi2.cpu().numpy(), want_pi)
        rec = hdist.unpack_records(sp.slot(t))
        words = before.cpu().numpy().view(np.uint32).copy()
        rw, fl, _ = cport.env_step(words, action.cpu().numpy().astype(np.uint8), n, 200, auto_reset=True, reset_word=sp.env.reset_word)
        assert np.array_equal(sp.env.words.cpu().numpy().view(np.uint32), words)
        assert np.array_equal(rec["state"].cpu().numpy(), before.cpu().numpy())
        assert np.array_equal(rec["reward"].cpu().numpy(), rw) and np.array_equal(rec["flags"].cpu().numpy(), fl)
        assert np.array_equal(rec["action"].cpu().numpy(), action.cpu().numpy().astype(np.uint8))
        assert np.array_equal(rec["visits"].cpu().numpy(), visits.cpu().numpy().astype(np.int16))
        assert np.array_equal(rec["root_q"].cpu().numpy(), root_q.cpu().numpy())  # float64 on the wire
        assert np.array_equal(rec["game_lo"].cpu().numpy().view(np.uint16), ((offset + np.arange(B)) & 0xFFFF).astype(np.uint16))
