"""The random draws and the root policy of a self-play move against oracle/move_ref.py, element by element:

* hmz_rng_uniform, hmz_rng_uniform_keyed, hmz_env_random_reset and the random env step / rollout bit for bit, from one
  item to past the eighth wave of their grids, with item / game offsets across 2^32 and near 2^63 and counters whose
  high words are set;
* hmz_rng_dirichlet and selfplay_begin (through SelfPlay.move) at alpha 1e-3 to 30, batches of 1 to 65,613 games,
  within 1e-11 relative of the restatement (plus four subnormal ulp of a gamma that underflowed below the smallest
  normal double, divided by the row's sum); a row may differ only where one of its accept / reject tests has a margin
  below 1e-10 on the host, and at most a handful do.  At alpha = 1e-3 the all-underflow fallback runs hundreds of times.
  On 2^24 device rows: the coordinates' law against Beta(alpha, 5 alpha), and no correlation between adjacent games or
  consecutive moves;
* hmz_search_root_policy, _multi and selfplay_finish bit for bit at root visit sums up to 65,534, where the six powers
  sum past 2^53 and the order of np.sum's additions matters: with a pow_table of np.power's values they equal NumPy's
  generate_play_policy / np.random.choice / np.argmax, without one the kernel's repeated products, at the sampling
  edges (u = 0, u at every cdf boundary and one ulp below it, the largest double below 1, zero-visit children, ties)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import record_metric
from oracle import episode_ref as er
from oracle import move_ref as mr
from oracle import port

pytestmark = pytest.mark.gpu
GATE = 1e-11  # relative, every Dirichlet element
HANDFUL = 3   # rows allowed to differ (each one with a host margin below mr.MARGIN_MIN)
TINY = np.finfo(np.float64).tiny
SUB = 2.0 ** -1074


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _same(a, b):
    return a.shape == b.shape and np.array_equal(_bits(np.asarray(a, np.float64)), _bits(np.asarray(b, np.float64)))


def _waves8(ctas_per_sm):
    """Items past the eighth wave of grid_for(n, 256, ctas_per_sm), where the grid-stride loops take over."""
    return torch.cuda.get_device_properties(0).multi_processor_count * ctas_per_sm * 256 * 8 + 77


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


def _items(offset, n):
    return np.uint64(offset) + np.arange(n, dtype=np.uint64)


# ------------------------------------------------------------------------------------------- uniforms and env draws
def test_uniforms_bit_exact(lib):
    from muzero_hanoi_b200 import _lib

    for n in (1, 5, 12, 4099, _waves8(8)):
        for seed, counter, offset in ((0, 0, 0), (0x0123456789ABCDEF, (0xFFFFFFFF << 32) | 3, (1 << 32) - n // 2 - 1),
                                      (7, (1 << 64) - 1, (1 << 63) - n // 2)):
            assert _same(_uniform(lib, n, seed, counter, offset), mr.uniform01(seed, _items(offset, n), counter)), (n, counter)
    rng = np.random.default_rng(1)
    n = _waves8(8)
    item = rng.integers(0, 2 ** 63, n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    hi = rng.integers(0, 2 ** 32, n, dtype=np.uint64) << np.uint64(32)
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    d_item, d_hi = (torch.from_numpy(x.view(np.int64)).cuda() for x in (item, hi))
    _lib.check(lib.hmz_rng_uniform_keyed(_lib.ptr(out), n, 0xDEADBEEF, _lib.ptr(d_hi), 0x1234, _lib.ptr(d_item), _lib.current_stream()))
    assert _same(out.cpu().numpy(), mr.uniform_keyed(0xDEADBEEF, hi, 0x1234, item))


def test_env_random_reset_step_and_rollout_bit_exact():
    from muzero_hanoi_b200.engine import VecHanoi

    big = _waves8(8) * 4  # the vec4 kernels: groups of four envs past the eighth wave
    cases = [(n_disks, n) for n_disks in (1, 5, 12) for n in (4, 12, 4100)] + [(3, big)]
    for n_disks, n in cases:
        max_steps = 7 if n_disks < 12 else 200
        env = VecHanoi(n_disks, max_steps, n)
        for counter in ((3 << 32) | 9, (1 << 64) - 1):
            env.random_reset(seed=0xC0FFEE, counter=counter)
            assert np.array_equal(env.words.cpu().numpy().view(np.uint32), mr.env_random_reset(n, n_disks, 2, 0xC0FFEE, counter))
        if n_disks == 1:
            for m in (1, 5, 12):  # the reset kernel alone at the smallest counts
                e = VecHanoi(n_disks, max_steps, m)
                e.random_reset(seed=4, counter=1 << 40)
                assert np.array_equal(e.words.cpu().numpy().view(np.uint32), mr.env_random_reset(m, n_disks, 2, 4, 1 << 40))
        words = env.words.cpu().numpy().view(np.uint32).copy()
        for step_index in ((1 << 32) - 1, (5 << 32) | 7):
            acts, rew, fl = env.step_random(seed=11, step_index=step_index)
            w, a, r, f = mr.env_step_random(words, n_disks, max_steps, 2, env.reset_word, 11, step_index)
            assert np.array_equal(acts.cpu().numpy(), a) and np.array_equal(fl.cpu().numpy(), f)
            assert np.array_equal(rew.cpu().numpy(), r) and np.array_equal(env.words.cpu().numpy().view(np.uint32), w)
            words = w
        k = 2 if n == big else 9
        counters = env.rollout_random(k, seed=3, step_index=(1 << 32) - 4).cpu().numpy().view(np.uint64)
        w, want = mr.env_rollout_random(words, n_disks, max_steps, 2, env.reset_word, k, 3, (1 << 32) - 4)
        assert np.array_equal(env.words.cpu().numpy().view(np.uint32), w) and np.array_equal(counters, want), (n_disks, n)


# ------------------------------------------------------------------------------------------------------- Dirichlet
class _Tally:
    """Device Dirichlet rows against the restatement: the 1e-11 gate, rows allowed to differ, ulp errors, fallbacks."""

    def __init__(self):
        self.rows = self.bad = self.small_margin = self.fallback = self.max_blocks = self.subnormal = 0
        self.ulp = 0

    def add(self, dev, ref: mr.Dirichlet, where):
        assert dev.shape == ref.x.shape
        # a gamma below the smallest normal double keeps only its absolute precision (2^-1074) into the division
        total = np.maximum(ref.gammas.sum(1, keepdims=True), TINY)
        bad = (np.abs(dev - ref.x) > GATE * np.abs(ref.x) + 4 * SUB / total).any(1)
        small = ref.margin < mr.MARGIN_MIN
        assert not (bad & ~small).any(), (where, np.nonzero(bad & ~small)[0][:5])
        self.rows += len(dev)
        self.bad += int(bad.sum())
        self.small_margin += int(small.sum())
        self.fallback += int(ref.fallback.sum())
        self.max_blocks = max(self.max_blocks, int(ref.blocks.max()))
        self.subnormal += int(((ref.gammas > 0) & (ref.gammas < TINY)).sum())
        good = ~bad[:, None] & (ref.gammas >= TINY)
        if good.any():
            d = np.abs(_bits(dev).astype(np.int64) - _bits(ref.x).astype(np.int64))
            self.ulp = max(self.ulp, int(d[good].max()))
        # the fallback rows are one-hot on the device too, and every row sums to one
        assert np.array_equal(dev[ref.fallback], ref.x[ref.fallback]), where
        assert np.abs(dev.sum(1) - 1.0).max() < 1e-14 and (dev >= 0).all()

    def check(self, name, min_fallback=0):
        record_metric(name, dict(rows=self.rows, rows_over_gate=self.bad, rows_small_margin=self.small_margin,
                                 fallback_rows=self.fallback, subnormal_gammas=self.subnormal, max_ulp=self.ulp,
                                 max_blocks=self.max_blocks))
        assert self.bad <= HANDFUL and self.max_blocks < mr.MAX_BLOCKS and self.fallback >= min_fallback


def _min_fallback(alpha):
    return 300 if alpha == 1e-3 else 0  # about 1.1 % of 65,613 games per key (740)


@pytest.mark.parametrize("alpha", mr.DIRICHLET_ALPHAS)
def test_dirichlet_matches_the_restatement(lib, alpha):
    tally = _Tally()
    for seed, counter, offset in mr.DIRICHLET_KEYS:
        for B in mr.DIRICHLET_BATCHES:
            tally.add(_dirichlet(lib, B, alpha, seed, counter, offset), mr.dirichlet(seed, _items(offset, B), counter, alpha),
                      (seed, counter, offset, B))
    if alpha == 3.0:  # past the eighth wave of the kernel's grid
        n = _waves8(4)
        tally.add(_dirichlet(lib, n, alpha, 31, 2, 0), mr.dirichlet(31, _items(0, n), 2, alpha), "waves")
    tally.check(f"move_ref_dirichlet_alpha{alpha:g}", _min_fallback(alpha))


def _selfplay(B, alpha, offset, seed=9, S=1, temperature=1.0, episodes=False):
    from muzero_hanoi_b200.engine import PackedWeights, SelfPlay

    w = PackedWeights(port.make_weights(3, 2), 3, 0)
    return SelfPlay(3, 200, B, S, w, alpha=alpha, temperature=temperature, seed=seed, ring_slots=2, game_offset=offset,
                    episodes=episodes)


@pytest.mark.parametrize("alpha", mr.DIRICHLET_ALPHAS + (0.0,))
def test_selfplay_begin_matches_the_restatement(alpha):
    """Eight lanes per game with shuffles: 1, 3, 4 and 33 games leave partial 8-lane groups and warps; alpha = 0 is the
    move without noise."""
    tally = _Tally()
    for k, B in enumerate(mr.DIRICHLET_BATCHES):
        seed, counter, offset = mr.DIRICHLET_KEYS[k % len(mr.DIRICHLET_KEYS)]
        sp = _selfplay(B, alpha, offset, seed)
        sp.moves_done = counter
        sp.move()
        torch.cuda.synchronize()
        p0 = sp.p0.cpu().numpy()
        ref = mr.selfplay_begin(p0, alpha, 0.25, seed, counter, offset)
        assert _same(sp.uniform.cpu().numpy(), ref.uniform)
        prior = sp.mcts.store.root_prior.cpu().numpy()
        rec_prior = sp.mcts.store.records()["prior"][:, 0]
        if alpha > 0:
            noise = sp.noise.cpu().numpy()
            tally.add(noise, ref.noise, (alpha, B))
            assert _same(prior, port.mix_dirichlet(p0, noise))
        else:
            assert _same(prior, ref.prior)
        assert np.array_equal(rec_prior, prior.astype(np.float32))
    if alpha > 0:
        tally.check(f"move_ref_selfplay_begin_alpha{alpha:g}", _min_fallback(alpha))


def test_dirichlet_law_on_the_device(lib):
    """2^24 rows at alpha = 0.25: every coordinate against Beta(alpha, 5 alpha) (Kolmogorov-Smirnov, p = 1e-6), and the
    correlation of a coordinate between adjacent games and between consecutive moves of one game."""
    import scipy.stats as ss

    from muzero_hanoi_b200 import _lib

    alpha, n = 0.25, 1 << 24
    x = torch.empty(n, 6, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)
    for out, counter in ((x, (7 << 32) | 1), (y, (7 << 32) | 2)):
        _lib.check(lib.hmz_rng_dirichlet(_lib.ptr(out), n, alpha, 123, counter, 1 << 40, _lib.current_stream()))
    law = ss.beta(alpha, 5 * alpha)
    crit = ss.kstwo(n).isf(1e-6)
    ks = [mr.ks_grid(torch.sort(x[:, a]).values.cpu().numpy(), law.ppf, law.cdf, ceil=mr.CEIL_01) for a in range(6)]

    def corr(a, b):
        a, b = a - a.mean(), b - b.mean()
        return float((a * b).mean() / (a.std() * b.std()))

    r_games = max(abs(corr(x[:-1, a], x[1:, a])) for a in range(6))
    r_moves = max(abs(corr(x[:, a], y[:, a])) for a in range(6))
    r_actions = abs(corr(x[:, 0], x[:, 1]))  # Dirichlet: -1 / 5 between two coordinates
    record_metric("move_ref_dirichlet_law", dict(ks_max=max(ks), ks_crit=crit, r_games=r_games, r_moves=r_moves, r_actions=r_actions))
    assert max(ks) < crit
    assert r_games < 6 / np.sqrt(n) and r_moves < 6 / np.sqrt(n) and abs(r_actions - 0.2) < 6 / np.sqrt(n)


# ----------------------------------------------------------------------------------------------------- root policy
def _write_counts(nodes, n_records, counts):
    """Visit counts into node record 0 of every search: child a at half a // 3, slot a % 3, the uint16 N."""
    B = len(counts)
    rec = nodes.view(torch.int16).reshape(B, n_records, 64)
    for a in range(6):
        rec[:, 0, (a // 3) * 32 + (a % 3) * 8 + 6] = torch.from_numpy(counts[:, a].astype(np.uint16).view(np.int16)).cuda()


def _power_sum_past_2_53(rows, temperature):
    w = np.power(rows.astype(np.float64), mr.exponent_of(temperature))
    return w.sum(1) > 2.0 ** 53


def test_root_policy_bit_exact_at_large_visit_counts():
    from muzero_hanoi_b200.engine import BatchedMCTS

    rng = np.random.default_rng(7)
    past, differ, rows_total = 0, 0, 0
    for S in mr.ROOT_SUMS:
        base = mr.root_rows(S, 3000, S)
        for T in (1.0, 0.5, 0.1, 0.0):
            table = mr.numpy_pow_table(S, T)
            ri, u = mr.edge_uniforms(base, T, table)
            ri = np.concatenate([ri, np.arange(len(base))])
            u = np.concatenate([u, rng.random(len(base))])
            ri2, u2 = mr.edge_uniforms(base, T)  # the products' own cdf boundaries
            ri, u = np.concatenate([ri, ri2]), np.concatenate([u, u2])
            rows = base[ri]
            B = len(rows)
            mcts = BatchedMCTS(0.8, 0.0, 1, B)
            _write_counts(mcts.store.nodes, 2, rows)
            root_w = rng.normal(size=B) * 100.0
            mcts.store.root_W.copy_(torch.from_numpy(root_w))
            for use_table in (False, True):
                mcts.pow_table = torch.from_numpy(table).cuda() if use_table else None
                act, pi, q, visits = (t.cpu().numpy() for t in mcts.root_policy(T, False, uniforms=u, n_simulations=S))
                want = mr.play_policy(rows, T, pow_table=table) if use_table else mr.play_policy(rows, T, products=True)
                assert np.array_equal(visits, rows) and _same(q, root_w / S)
                assert _same(pi, want), (S, T, use_table)
                assert np.array_equal(act, mr.sample_action(want, u)), (S, T, use_table)
                if use_table or S <= er.POLICY_EXACT_MAX:  # NumPy's own calls, row by row, on a sample
                    for i in range(0, B, 97):
                        assert _same(pi[i], port.play_policy(rows[i], T)) and act[i] == port.sample_action(pi[i], u[i])
                det = mcts.root_policy(T, True, n_simulations=S)[0].cpu().numpy()
                assert np.array_equal(det, mr.argmax_action(rows))
            if T == 0.1:
                past += int(_power_sum_past_2_53(base, T).sum())
                differ += int(mr.sum_orders_differ(base, T, table).sum())
                rows_total += len(base)
                if S >= 4096:
                    assert mr.sum_orders_differ(base, T, table).any(), S
    record_metric("move_ref_root_policy", dict(rows_t01=rows_total, rows_power_sum_past_2_53=past, rows_sum_orders_differ=differ))
    assert past > 0 and differ > 0


def test_root_policy_multi_per_search_budgets(lib):
    from muzero_hanoi_b200 import _lib

    B, n_records = 512, 32768
    rng = np.random.default_rng(11)
    budget = np.concatenate([rng.integers(1, 32768, 256), rng.integers(1, 20001, 256)]).astype(np.int64)
    budget[[0, 255]] = [32767, 1]
    rows = np.stack([rng.multinomial(b, rng.dirichlet(np.full(6, 0.3))) for b in budget]).astype(np.int64)
    hbb = np.array([budget[:256].max(), budget[256:].max()], np.int32)
    nodes = torch.zeros(B * n_records * 128, dtype=torch.uint8, device="cuda")
    _write_counts(nodes, n_records, rows)
    root_w = torch.from_numpy(rng.normal(size=B) * 50.0).cuda()
    small = [torch.zeros(B, 6, dtype=torch.float64, device="cuda"), torch.zeros(B, 2, dtype=torch.float64, device="cuda")]
    sd = _lib.SearchDesc(nodes=nodes.data_ptr(), latents=None, root_prior=small[0].data_ptr(), root_W=root_w.data_ptr(),
                         minmax=small[1].data_ptr(), workspace=None, capture=None, n_searches=B, n_records=n_records,
                         latent_dtype=0, root_prior_is_f64=1, schedule=0)
    block_set = torch.zeros(2, dtype=torch.int16, device="cuda")
    d_budget = torch.from_numpy(budget.astype(np.int16)).cuda()
    md = _lib.MultiDesc(block_set=block_set.data_ptr(), budget=d_budget.data_ptr(), host_block_budget=hbb.ctypes.data,
                        weight_stride=0, n_sets=1, n_disks=3)
    u = np.concatenate([rng.random(B // 2), np.zeros(B // 4), np.full(B - B // 2 - B // 4, np.nextafter(1.0, 0.0))])
    d_u = torch.from_numpy(u).cuda()
    visits = torch.empty(B, 6, dtype=torch.int32, device="cuda")
    pi = torch.empty(B, 6, dtype=torch.float64, device="cuda")
    q = torch.empty(B, dtype=torch.float64, device="cuda")
    act = torch.empty(B, dtype=torch.int32, device="cuda")
    for T in (0.1, 0.5):
        table = mr.numpy_pow_table(int(hbb[0]), T)  # pow_table_len = the first block's budget + 1
        for use_table in (False, True):
            d_table = torch.from_numpy(table).cuda() if use_table else None
            _lib.check(lib.hmz_search_root_policy_multi(C.byref(sd), C.byref(md), T, 0, _lib.ptr(d_u), _lib.ptr(d_table),
                                                        _lib.ptr(visits), _lib.ptr(pi), _lib.ptr(q), _lib.ptr(act),
                                                        _lib.current_stream()))
            torch.cuda.synchronize()
            want = mr.play_policy(rows, T, pow_table=table) if use_table else mr.play_policy(rows, T, products=True)
            assert np.array_equal(visits.cpu().numpy(), rows)
            assert _same(q.cpu().numpy(), root_w.cpu().numpy() / budget)  # each search's own division
            assert _same(pi.cpu().numpy(), want), (T, use_table)
            assert np.array_equal(act.cpu().numpy(), mr.sample_action(want, u))


def test_selfplay_finish_bit_exact_past_the_exact_powers():
    """SelfPlay at S = 2,048 and T = 0.1 (exponent 5): root counts pass 1,554 on their own.  Action, ring record,
    episode store (exponent included) and root_q recomputed from the tree's record 0 and the move's uniform; the first
    move with the kernel's products, the second with np.power's table."""
    from muzero_hanoi_b200 import dist as hdist

    B, S, T = 320, 2048, 0.1
    sp = _selfplay(B, 0.25, 1000, seed=5, S=S, temperature=T, episodes=True)
    table = mr.numpy_pow_table(S, T)
    past = 0
    for move in range(2):
        if move == 1:
            sp.mcts.pow_table = torch.from_numpy(table).cuda()
        before = sp.env.words.cpu().numpy().view(np.uint32).copy()
        t = sp.move()
        torch.cuda.synchronize()
        rec = sp.mcts.store.records()
        n = rec["N"][:, 0].astype(np.int64)
        root_w = sp.mcts.store.root_W.cpu().numpy()
        u = sp.uniform.cpu().numpy()
        pi = mr.play_policy(n, T, pow_table=table) if move == 1 else mr.play_policy(n, T, products=True)
        act = mr.sample_action(pi, u)
        q = root_w / S
        past += int(_power_sum_past_2_53(n, T).sum())
        assert (n.sum(1) == S).all() and (n.max(1) > er.POLICY_EXACT_MAX).any()
        assert np.array_equal(sp.mcts.visits.cpu().numpy(), n) and np.array_equal(sp.mcts.action.cpu().numpy(), act)
        assert _same(sp.mcts.root_q.cpu().numpy(), q)
        if move == 1:
            for i in range(0, B, 7):
                assert port.sample_action(port.play_policy(n[i], T), u[i]) == act[i]
        r = hdist.unpack_records(sp.slot(t))
        assert np.array_equal(r["action"].cpu().numpy(), act.astype(np.uint8))
        assert np.array_equal(r["visits"].cpu().numpy().view(np.uint16), n.astype(np.uint16))
        assert _same(r["root_q"].cpu().numpy(), q) and np.array_equal(r["state"].cpu().numpy().view(np.uint32), before)
        ep = sp.episodes
        slot = np.minimum(before >> 6, ep.t_max - 1).astype(np.int64)  # the counter bits above 2 N = 6 state bits
        g = np.arange(B)
        assert (ep.exp.cpu().numpy()[slot, g] == 5).all()
        assert np.array_equal(ep.action.cpu().numpy()[slot, g], act.astype(np.uint8))
        assert np.array_equal(ep.visits.cpu().numpy()[slot, g].view(np.uint16), n.astype(np.uint16))
        assert _same(ep.root_q.cpu().numpy()[slot, g], q)
    record_metric("move_ref_selfplay_finish", dict(games=B, moves=2, rows_power_sum_past_2_53=past))
    assert past > 0
