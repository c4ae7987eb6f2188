"""GPU: heterogeneous search batches (hmz_multi_t) — several networks and per-search budgets in one launch sequence —
against one ordinary hmz_search_run per (network, budget) segment, bit for bit, and against the C oracle's replay."""
import numpy as np
import pytest
import torch

from oracle import cport, port

pytestmark = pytest.mark.gpu

N = 4
# per block of 256 searches: (weight set, budgets drawn for its searches); block maxima non-increasing, ragged segments
BLOCKS = [(0, (120, 100, 37)), (1, (100, 1, 5, 100)), (2, (60, 2, 17)), (0, (60, 1)), (1, (9,))]


def _nets():
    base = port.make_weights(N, 21)
    return [base, port.lesion_weights(base, ["policy_net"], seed=3), port.lesion_weights(port.make_weights(N, 22), ["value_net", "rwd_net"], seed=4)]


def _batch(blocks, seed=0):
    rng = np.random.default_rng(seed)
    budget = np.concatenate([rng.choice(b, 256) for _, b in blocks]).astype(np.int64)
    for k, (_, b) in enumerate(blocks):  # every listed budget occurs
        budget[k * 256: k * 256 + len(b)] = b
    block_set = np.array([s for s, _ in blocks], np.int64)
    return budget, block_set


def _run_multi(sets, budget, block_set, words, noise, uni, ldt, schedule, capture=False, moves=2):
    from muzero_hanoi_b200.engine import MultiMCTS

    B = len(budget)
    m = MultiMCTS(0.8, 0.25, int(budget.max()), B, latent_dtype=ldt)
    m.store.set_schedule(schedule)
    cap = m.store.enable_capture(int(budget.max())) if capture else None
    bs = torch.as_tensor(block_set, dtype=torch.int16, device="cuda")
    bd = torch.as_tensor(budget, dtype=torch.int16, device="cuda")
    hbb = np.ascontiguousarray(budget.reshape(-1, 256).max(1), dtype=np.int32)
    md = sets.desc(bs, bd, hbb)
    outs = []
    for move in range(moves):
        mm = m.store.minmax.cpu().numpy().copy()
        a, pi, q, v = m.run_mcts(sets, md, B, words=words, temperature=1.0, noise=noise[move], uniforms=uni[move])
        torch.cuda.synchronize()
        outs.append(dict(action=a.cpu().numpy(), pi=pi.cpu().numpy(), q=q.cpu().numpy(), visits=v.cpu().numpy(),
                         p0=m.p0.cpu().numpy(), v0=m.v0.cpu().numpy(), minmax=m.store.minmax.cpu().numpy().copy(), mm_before=mm,
                         root_W=m.store.root_W.cpu().numpy().copy(), prior=m.store.root_prior.cpu().numpy().copy(),
                         nodes=m.store.nodes.cpu().numpy().reshape(B, m.store.n_records, 128).copy(),
                         latents=m.store.latents.view(torch.int16).cpu().numpy().copy(),
                         capture=cap.cpu().numpy().copy() if capture else None))
    return outs


def _setup(mode, B, moves=2):
    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200.engine import VecHanoi

    env = VecHanoi(N, 200, B)
    env.random_reset(seed=7)
    rng = np.random.default_rng(5)
    noise = [torch.as_tensor(rng.dirichlet(np.full(6, 0.25), B), device="cuda") for _ in range(moves)]
    uni = [torch.as_tensor(rng.random(B), device="cuda") for _ in range(moves)]
    ldt = _lib.LATENT_BF16 if mode == _lib.MODE_BF16 else _lib.LATENT_F32
    return env.words, noise, uni, ldt


@pytest.mark.parametrize("schedule", [0, 1, 4])
@pytest.mark.parametrize("mode", [0, 2, 1])
def test_multi_search_equals_one_search_per_segment(mode, schedule):
    """hmz_net_initial_multi + hmz_search_run_multi + hmz_search_root_policy_multi against BatchedMCTS.run_mcts (hmz_net_initial,
    hmz_search_run, hmz_search_root_policy) of every (network, budget) segment alone, over two moves: node records 0..b,
    latents 0..b, root prior, root_W, min/max, p0, v0, visits, pi, root_q and the sampled action, bit for bit."""
    from muzero_hanoi_b200.engine import BatchedMCTS, PackedWeights, WeightSets

    nets = _nets()
    budget, block_set = _batch(BLOCKS)
    B = len(budget)
    words, noise, uni, ldt = _setup(mode, B)
    sets = WeightSets(nets, N, mode)
    got = _run_multi(sets, budget, block_set, words, noise, uni, ldt, schedule)
    game_set = np.repeat(block_set, 256)
    packed = [PackedWeights(sd, N, mode) for sd in nets]
    for k in range(len(nets)):
        for b in np.unique(budget[game_set == k]):
            idx = np.nonzero((game_set == k) & (budget == b))[0]
            it = torch.as_tensor(idx, device="cuda")
            ref = BatchedMCTS(0.8, 0.25, int(b), len(idx), latent_dtype=ldt)
            for move in range(2):
                a, pi, q, v = ref.run_mcts(packed[k], words=words[it].contiguous(), temperature=1.0, noise=noise[move][it].contiguous(),
                                           uniforms=uni[move][it].contiguous())
                torch.cuda.synchronize()
                g = got[move]
                tag = f"set {k} budget {b} move {move}"
                recs = ref.store.nodes.cpu().numpy().reshape(len(idx), b + 1, 128)
                assert np.array_equal(g["nodes"][idx, : b + 1], recs), tag
                assert np.array_equal(g["latents"][idx, : b + 1], ref.store.latents.view(torch.int16).cpu().numpy()), tag
                assert np.array_equal(g["p0"][idx], ref.p0.cpu().numpy()) and np.array_equal(g["v0"][idx], ref.v0.cpu().numpy()), tag
                assert np.array_equal(g["prior"][idx], ref.store.root_prior.cpu().numpy()), tag
                assert np.array_equal(g["root_W"][idx], ref.store.root_W.cpu().numpy()), tag
                assert np.array_equal(g["minmax"][idx], ref.store.minmax.cpu().numpy()), tag
                for key, t in (("visits", v), ("pi", pi), ("q", q), ("action", a)):
                    assert np.array_equal(g[key][idx], t.cpu().numpy()), f"{tag}: {key}"


def test_multi_search_replayed_by_the_oracle():
    """HMZ_MODE_FP32X3, four stream groups, capture on: the C oracle replays every search at its own budget from the captured
    network outputs and reproduces visit counts, root_q and min/max bit for bit."""
    from muzero_hanoi_b200.engine import WeightSets

    budget, block_set = _batch(BLOCKS, seed=1)
    words, noise, uni, ldt = _setup(2, len(budget))
    got = _run_multi(WeightSets(_nets(), N, 2), budget, block_set, words, noise, uni, ldt, 4, capture=True)
    for g in got:
        c = g["capture"]
        for b in np.unique(budget):
            idx = np.nonzero(budget == b)[0]
            mm = np.ascontiguousarray(g["mm_before"][idx])
            sub = lambda j: np.ascontiguousarray(c[:b][:, idx][:, :, j])
            o_visits, o_q, _ = cport.search_injected(np.ascontiguousarray(g["prior"][idx]), True, mm, sub(6),
                                                     np.ascontiguousarray(c[:b][:, idx, :6]), sub(7), 0.8, port.ucb_table(int(b) + 1))
            assert np.array_equal(g["visits"][idx], o_visits), f"budget {b}"
            assert np.array_equal(g["q"][idx], o_q) and np.array_equal(g["minmax"][idx], mm), f"budget {b}"


def test_multi_search_does_not_depend_on_other_blocks_budgets():
    """The per-simulation prefix: the first block's searches give the same results whatever the later blocks' budgets
    (all 1 here, so after simulation 0 only the first block is launched)."""
    from muzero_hanoi_b200.engine import WeightSets

    budget, block_set = _batch(BLOCKS, seed=2)
    words, noise, uni, ldt = _setup(1, len(budget))
    sets = WeightSets(_nets(), N, 1)
    a = _run_multi(sets, budget, block_set, words, noise, uni, ldt, 0, moves=1)[0]
    budget2 = budget.copy()
    budget2[256:] = 1
    b = _run_multi(sets, budget2, block_set, words, noise, uni, ldt, 0, moves=1)[0]
    for key in ("visits", "pi", "q", "action", "root_W", "minmax"):
        assert np.array_equal(a[key][:256], b[key][:256]), key
    assert np.array_equal(a["nodes"][:256], b["nodes"][:256])
    assert (b["visits"][256:].sum(1) == 1).all()
