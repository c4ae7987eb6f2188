"""GPU: device replay sampling (hmz_replay_sample / hmz_replay_set_priorities through ReplayRing) against the host path
it replaces — priority_sample, update_priorities and BatchedMuzero's host-path update — bit for bit."""
import numpy as np
import pytest
import torch

from conftest import record_metric
from oracle import replay_ref as R

pytestmark = pytest.mark.gpu

SIZES = [1, 2, 3, 7, 8, 127, 128, 129, 1000, 8191, 8193, 50000, 100003, 1048579]


def make_ring(q, size, beta=0, seed=0, full=False):
    """A ReplayRing with q as the priorities of its filled rows (all `size` rows when full, the ring then wrapped), and
    random row contents so that gathers are checked too."""
    from muzero_hanoi_b200.replay import ReplayRing

    ring = ReplayRing(size, 5, 9, 6, importance_sampling_exponent=beta)
    g = torch.Generator(device="cuda").manual_seed(seed)
    ring.states.copy_(torch.rand(ring.states.shape, generator=g, device="cuda"))
    ring.rwds.copy_(torch.rand(ring.rwds.shape, generator=g, device="cuda"))
    ring.actions.copy_(torch.randint(0, 6, ring.actions.shape, generator=g, device="cuda"))
    ring.pi_probs.copy_(torch.rand(ring.pi_probs.shape, generator=g, device="cuda"))
    ring.mc_returns.copy_(torch.rand(ring.mc_returns.shape, generator=g, device="cuda"))
    ring.priorities[: len(q)] = torch.from_numpy(np.asarray(q, np.float32)).cuda()
    if full:
        assert len(q) == size
        ring.is_full, ring.ptr = True, size // 3
    else:
        ring.ptr = len(q)
    return ring


def heavy_tailed(rng, n):
    q = (10.0 ** rng.uniform(-12, 3, n)).astype(np.float32)
    q[rng.random(n) < 0.05] = 0
    if not q.any():
        q[-1] = 1
    return q


def compare(ring, seed, batch=256, exact=True, rtol=0.0):
    np.random.seed(seed)
    host = ring.priority_sample(batch)
    after_host = np.random.random_sample()
    np.random.seed(seed)
    dev = ring.priority_sample_device(batch)
    after_dev = np.random.random_sample()
    torch.cuda.synchronize()
    ring.check_status()
    assert after_host == after_dev, "the device path consumed a different number of draws"
    assert np.array_equal(host[5], dev[5].cpu().numpy())
    for a, b in zip(host[:5], dev[:5]):
        assert torch.equal(a, b)
    if exact:
        assert torch.equal(host[6].view(torch.int32), dev[6].view(torch.int32))
    else:
        assert torch.allclose(host[6], dev[6], rtol=rtol, atol=0)
    return (host[6] - dev[6]).abs().div(host[6].abs()).max().item()


@pytest.mark.parametrize("kind", ["trained", "constructed"])
def test_indices_and_weights_are_numpys(kind):
    rng = np.random.default_rng(11)
    for n in SIZES:
        q = heavy_tailed(rng, n) if kind == "trained" else R.constructed_ring(n, seed=n)
        if kind == "constructed" and n >= 300:
            _, info = R.exact_cumsum((q / np.sum(q)).astype(np.float32))
            assert info["ties"] > 0 and info["roundup"] > 0
        compare(make_ring(q, n + 1000, seed=n), seed=n)           # partly filled
        compare(make_ring(q, n, seed=n, full=True), seed=n + 1)   # full, wrapped


def test_batch_sizes_and_repeated_draws():
    rng = np.random.default_rng(12)
    ring = make_ring(heavy_tailed(rng, 50000), 50000, full=True)
    for i, batch in enumerate((1, 255, 256, 1025, 5000)):
        compare(ring, seed=100 + i, batch=batch)


@pytest.mark.parametrize("beta", [0.5, 1, 0.3])
def test_importance_weights_other_than_zero(beta):
    """beta = 0.5 / 1 use NumPy's own fast paths (sqrt / identity) and come out exact; others use CUDA's powf, gated at
    4 float32 ulps (powf's 2 ulps, plus the division by the maximum)."""
    rng = np.random.default_rng(13)
    worst = 0.0
    for n in (129, 50000):
        ring = make_ring(heavy_tailed(rng, n), n, beta=beta, full=True)
        worst = max(worst, compare(ring, seed=n, exact=beta in (0.5, 1), rtol=4 * 2.0 ** -24))
    record_metric(f"replay weights beta={beta}", {"max_rel_err": worst})


@pytest.mark.parametrize("case,message", [
    ("zeros", "probabilities contain NaN"),
    ("nan", "probabilities contain NaN"),
    ("inf", "probabilities contain NaN"),
    ("negative", "probabilities are not non-negative"),
    ("overflow", "probabilities do not sum to 1"),
    ("one_zero", "probabilities contain NaN"),
    ("two_cancel", "probabilities contain NaN"),
])
def test_rings_numpy_rejects_raise_the_same(case, message):
    q = np.linspace(0.1, 1, 100).astype(np.float32)
    if case == "zeros":
        q[:] = 0
    elif case == "nan":
        q[7] = np.nan
    elif case == "inf":
        q[7] = np.inf
    elif case == "negative":
        q[3] = -0.5
    elif case == "overflow":
        q[:] = 3e38
    elif case == "one_zero":
        q = np.zeros(1, np.float32)
    else:
        q = np.array([1, -1], np.float32)
    for ring in (make_ring(q, len(q) + 5), make_ring(q, len(q), full=True)):
        with np.errstate(all="ignore"), pytest.raises(ValueError, match=message):
            ring.priority_sample(16)
        before = ring.priorities.clone()
        ring.priority_sample_device(16)
        with pytest.raises(ValueError, match=message):
            ring.check_status()
        assert torch.equal(before.view(torch.int32), ring.priorities.view(torch.int32))


def test_priority_write_back_is_update_priorities():
    """Duplicates keep their last value, as NumPy's fancy assignment into the reference's priority array does (torch's
    CUDA index assignment leaves the winner of a duplicate unspecified, so the host path is compared where the values of
    a repeated index agree, as the learner's priorities of a row drawn twice do)."""
    rng = np.random.default_rng(14)
    for size, batch in ((1000, 256), (50000, 256), (64, 4096)):
        q = heavy_tailed(rng, size)
        host, dev = make_ring(q, size, full=True), make_ring(q, size, full=True)
        ref = q.copy()
        for _ in range(3):
            indx = rng.integers(0, size, batch).astype(np.int64)
            indx[: batch // 4] = indx[-1]  # duplicates with different values: the last occurrence wins
            new_p = rng.random(batch).astype(np.float32) + np.float32(0.01)
            ref[indx] = new_p
            dev.update_priorities_device(torch.from_numpy(indx).cuda(), torch.from_numpy(new_p).cuda())
            assert np.array_equal(dev.priorities.cpu().numpy(), ref)
        dev.check_status()
        host.priorities.copy_(dev.priorities)
        indx = rng.integers(0, size, batch).astype(np.int64)
        new_p = (rng.random(size).astype(np.float32) + np.float32(0.01))[indx]  # one value per row
        host.update_priorities(indx, new_p)
        dev.update_priorities_device(torch.from_numpy(indx).cuda(), torch.from_numpy(new_p).cuda())
        assert torch.equal(host.priorities, dev.priorities)


@pytest.mark.parametrize("bad", ["nan", "inf", "zeros", "negative"])
def test_priority_write_back_assertion(bad):
    rng = np.random.default_rng(15)
    q = heavy_tailed(rng, 500)
    host, dev = make_ring(q, 500, full=True), make_ring(q, 500, full=True)
    indx = rng.integers(0, 500, 64).astype(np.int64)
    new_p = rng.random(64).astype(np.float32)
    new_p[5] = {"nan": np.nan, "inf": np.inf, "zeros": 0, "negative": -1}[bad]
    if bad in ("zeros", "negative"):
        new_p[:] = new_p[5]
    with pytest.raises(AssertionError, match="Priorities must be finite and positive."):
        host.update_priorities(indx, new_p)
    dev.update_priorities_device(torch.from_numpy(indx).cuda(), torch.from_numpy(new_p).cuda())
    with pytest.raises(AssertionError, match="Priorities must be finite and positive."):
        dev.check_status()
    assert torch.equal(host.priorities, dev.priorities)  # nothing written


# ---- BatchedMuzero: device path against the host path it replaces ---------------------------------------------------

N, MAX_STEPS, GAMES, LOOPS, MIN_REPLAY = 3, 40, 256, 16, 100
RING = ("states", "rwds", "actions", "pi_probs", "mc_returns", "priorities")


def _host_path_trainer_class():
    from muzero_hanoi_b200.trainer import BatchedMuzero

    class HostPath(BatchedMuzero):
        """BatchedMuzero's update as it was before the device path: NumPy draws on a host copy of the priorities,
        Learner.update's read-back, update_priorities' upload."""

        def step(self):
            if self.priority_replay:
                states, rwds, actions, pi_probs, returns, indx, w = self.buffer.priority_sample(self.batch_s)
            else:
                states, rwds, actions, pi_probs, returns = self.buffer.uniform_sample(self.batch_s)
                indx, w = None, None
            new_p, v_loss, r_loss, p_loss = self.learner.update(states, rwds, actions, pi_probs, returns, w)
            self._weights_dirty = True
            self.buffer.update_priorities(indx, new_p)
            return torch.tensor([v_loss, r_loss, p_loss], dtype=torch.float32, device=self.learner.device)

    return HostPath


def _train(cls, priority_replay):
    from muzero_hanoi_b200.networks import MuZeroNet

    torch.manual_seed(7)
    np.random.seed(7)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    mz = cls(net.state_dict(), N, MAX_STEPS, GAMES, n_mcts_simulations=8, batch_s=64, buffer_size=6000, n_update_x_loop=4,
             moves_per_loop=8, priority_replay=priority_replay, seed=5)
    hist = mz.training_loop(LOOPS, MIN_REPLAY)
    torch.cuda.synchronize()
    return dict(hist=np.array(hist, dtype=np.float64), episodes_done=mz.episodes_done, step_index=mz.learner.step_index,
                params=mz.learner.params.cpu(), adam_m=mz.learner.adam_m.cpu(), adam_v=mz.learner.adam_v.cpu(), ptr=mz.buffer.ptr,
                is_full=mz.buffer.is_full, next_draw=np.random.random_sample(), **{k: getattr(mz.buffer, k).cpu() for k in RING})


@pytest.mark.parametrize("priority_replay", [True, False])
def test_training_is_bit_identical_to_the_host_path(priority_replay):
    from muzero_hanoi_b200.trainer import BatchedMuzero

    dev = _train(BatchedMuzero, priority_replay)
    host = _train(_host_path_trainer_class(), priority_replay)
    assert dev["step_index"] >= 4 * 10 and dev["step_index"] == host["step_index"]
    for k in ("params", "adam_m", "adam_v", *RING):
        assert torch.equal(dev[k], host[k]), k
    for k in ("episodes_done", "ptr", "is_full", "next_draw"):
        assert dev[k] == host[k], k
    assert np.array_equal(dev["hist"][:, :2], host["hist"][:, :2], equal_nan=True)
    assert np.allclose(dev["hist"][:, 2:], host["hist"][:, 2:], rtol=1e-5, atol=1e-6, equal_nan=True)
    assert np.isfinite(dev["hist"][:, 2]).sum() >= 10


@pytest.mark.parametrize("priority_replay", [True, False])
def test_a_loops_updates_do_not_synchronise(priority_replay):
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.trainer import BatchedMuzero

    torch.manual_seed(3)
    np.random.seed(3)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    mz = BatchedMuzero(net.state_dict(), N, MAX_STEPS, GAMES, n_mcts_simulations=8, batch_s=64, buffer_size=6000,
                       priority_replay=priority_replay, seed=5)
    mz._refresh_actor(1.0)
    while len(mz.buffer) <= MIN_REPLAY:
        mz.play(8)
    mz.step()  # first-use allocations (workspace, pinned staging)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(8):
            losses = mz.step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    vals, status = mz._read_back(losses)
    assert status == 0 and all(np.isfinite(vals))


def test_an_invalid_ring_raises_at_the_end_of_the_loop():
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.trainer import BatchedMuzero

    torch.manual_seed(3)
    np.random.seed(3)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    mz = BatchedMuzero(net.state_dict(), N, MAX_STEPS, GAMES, n_mcts_simulations=8, batch_s=64, buffer_size=100000, seed=5)
    mz._refresh_actor(1.0)
    while len(mz.buffer) <= MIN_REPLAY:
        mz.play(8)
    mz.buffer.priorities[0] = float("nan")  # the reference's priority_sample raises at the loop's first update
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        mz.training_loop(2, 0)
