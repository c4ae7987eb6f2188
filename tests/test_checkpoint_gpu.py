"""BatchedMuzero.save / load resume a run bit-identically, saving leaves the run unchanged, the file does not depend on the
number of ranks that wrote or reads it, and export_reference writes a file the reference's own MuZeroNet and Adam load and
continue.  Sizes follow test_dist_train_gpu: N = 3, 40 max steps, 256 games, 8 simulations, batch 64, 2 updates per
loop, 14 loops (13 run), saved after 7."""
import datetime
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT  # noqa: F401

pytestmark = pytest.mark.gpu

N, MAX_STEPS, GAMES, LOOPS, SAVE_AT, MIN_REPLAY = 3, 40, 256, 14, 7, 100
RING = ("states", "rwds", "actions", "pi_probs", "mc_returns", "priorities")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _trainer(priority_replay=True, buffer_size=6000, acting_mode=None):
    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.trainer import BatchedMuzero

    torch.manual_seed(7)
    np.random.seed(7)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    return BatchedMuzero(net.state_dict(), N, MAX_STEPS, GAMES, n_mcts_simulations=8, batch_s=64, buffer_size=buffer_size,
                         n_update_x_loop=2, moves_per_loop=8, priority_replay=priority_replay, seed=5,
                         acting_mode=_lib.MODE_FP32 if acting_mode is None else acting_mode)


def _state(mz):
    """What a one-GPU run leaves: learner, ring, self-play (host copies)."""
    torch.cuda.synchronize()
    ln, buf, sp = mz.learner, mz.buffer, mz._selfplay
    return dict(params=ln.params.cpu(), adam_m=ln.adam_m.cpu(), adam_v=ln.adam_v.cpu(), step_index=ln.step_index,
                episodes_done=mz.episodes_done, ptr=buf.ptr, is_full=buf.is_full, status=int(buf.status.item()),
                words=sp.env.words.cpu(), minmax=sp.mcts.store.minmax.cpu(), moves_done=sp.moves_done,
                **{k: getattr(buf, k).cpu() for k in RING})


def _assert_equal(a, b, what):
    """Nested dicts of tensors and scalars: tensors torch.equal, the rest ==."""
    if isinstance(a, dict):
        assert isinstance(b, dict) and set(a) == set(b), (what, sorted(a), sorted(b))
        for k in a:
            _assert_equal(a[k], b[k], f"{what}.{k}")
    elif torch.is_tensor(a):
        assert torch.is_tensor(b) and a.dtype == b.dtype and torch.equal(a, b), what
    else:
        assert a == b, (what, a, b)


def _assert_same_history(a, b, what):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(a[:, :2], b[:, :2], equal_nan=True), what  # loop, mean episode length
    # losses: the loss kernels sum with float32 atomics, so only the summation order may differ
    assert np.allclose(a[:, 2:], b[:, 2:], rtol=1e-5, atol=1e-6, equal_nan=True), what


def _scramble_generators():
    np.random.seed(12345)
    torch.manual_seed(12345)
    np.random.random_sample(17)
    torch.randint(0, 6, (1000,), device="cuda")


VARIANTS = {
    "priority": dict(),
    "uniform": dict(priority_replay=False),
    "before_updates": dict(),  # min_replay_size chosen so that the first update comes after the save
    "wrapped_ring": dict(buffer_size=64),  # with min_replay_size 40
    "bf16_acting": dict(acting_mode="bf16"),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_resume_is_bit_identical(tmp_path, variant):
    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200.trainer import BatchedMuzero, _step_counters

    kw = dict(VARIANTS[variant])
    if kw.get("acting_mode") == "bf16":
        kw["acting_mode"] = _lib.MODE_BF16
    min_replay = 40 if variant == "wrapped_ring" else MIN_REPLAY
    if variant == "before_updates":  # the ring's length after SAVE_AT loops without updates (play does not depend on them)
        probe = _trainer(**kw)
        probe.training_loop(SAVE_AT + 1, 10 ** 9)
        min_replay = len(probe.buffer)
        del probe

    straight = _trainer(**kw)
    hist = straight.training_loop(LOOPS, min_replay)
    want = _state(straight)
    assert want["step_index"] > 0

    mz = _trainer(**kw)
    first = mz.training_loop(SAVE_AT + 1, min_replay)
    assert (mz.learner.step_index == 0) == (variant == "before_updates")
    if variant == "wrapped_ring":
        assert mz.buffer.is_full and 0 < mz.buffer.ptr < mz.buffer.size
    path = tmp_path / "run.pt"
    mz.save(path)
    mz.save(tmp_path / "again.pt")
    ck = torch.load(path)  # default weights_only=True
    _assert_equal(ck, torch.load(tmp_path / "again.pt"), "two saves at the same point")
    # only the slots of the episodes in flight are written
    live = int(_step_counters(ck["selfplay"]["words"], N).sum())
    assert live > 0 and ck["episodes"]["state"].shape[0] == live and ck["episodes"]["visits"].shape == (live, 6)

    # saving has no side effect: the saving run goes on exactly as the straight one
    mz.training_loop(LOOPS - SAVE_AT, min_replay)
    _assert_equal(_state(mz), want, "run that saved vs straight run")

    _scramble_generators()
    resumed = BatchedMuzero.load(path)
    rest = resumed.training_loop(LOOPS - SAVE_AT, min_replay)
    assert [r[0] for r in rest] == list(range(SAVE_AT + 1, LOOPS))  # loop numbering continues
    _assert_same_history(first + rest, hist, "save / load / rest vs straight")
    _assert_equal(_state(resumed), want, "resumed vs straight")


def _worker(rank, world, port, backend, out_dir):
    from muzero_hanoi_b200.trainer import BatchedMuzero

    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            timeout=datetime.timedelta(seconds=300), **(dict(device_id=dev) if backend == "nccl" else {}))
    try:
        mz = _trainer()
        mz.training_loop(SAVE_AT + 1, MIN_REPLAY)
        mz.save(os.path.join(out_dir, "two.pt"))
        for src in ("two", "one"):
            _scramble_generators()
            r = BatchedMuzero.load(os.path.join(out_dir, f"{src}.pt"), device=dev)
            hist = r.training_loop(LOOPS - SAVE_AT, MIN_REPLAY)
            r.save(os.path.join(out_dir, f"end_{src}_on_two.pt"))
            torch.save(np.asarray(hist, dtype=np.float64), os.path.join(out_dir, f"hist_{src}_on_two_rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_file_does_not_depend_on_the_number_of_ranks(tmp_path, backend):
    from muzero_hanoi_b200.trainer import BatchedMuzero

    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip(f"NCCL needs 2 GPUs, found {torch.cuda.device_count()}")
    torch.cuda.set_device(0)
    straight = _trainer()
    hist = np.asarray(straight.training_loop(LOOPS, MIN_REPLAY), dtype=np.float64)
    straight.save(tmp_path / "end_straight.pt")
    want = torch.load(tmp_path / "end_straight.pt")
    one = _trainer()
    one.training_loop(SAVE_AT + 1, MIN_REPLAY)
    one.save(tmp_path / "one.pt")
    del one

    mp.spawn(_worker, args=(2, _free_port(), backend, str(tmp_path)), nprocs=2, join=True)
    _assert_equal(torch.load(tmp_path / "two.pt"), torch.load(tmp_path / "one.pt"), "file of two ranks vs file of one GPU")
    for src in ("two", "one"):
        _assert_equal(torch.load(tmp_path / f"end_{src}_on_two.pt"), want, f"{src}-rank file resumed on two ranks")
        for rank in range(2):
            _assert_same_history(torch.load(tmp_path / f"hist_{src}_on_two_rank{rank}.pt", weights_only=False), hist[SAVE_AT:],
                                 f"{src}-rank file resumed on two ranks, rank {rank}")

    _scramble_generators()
    r = BatchedMuzero.load(tmp_path / "two.pt")
    _assert_same_history(r.training_loop(LOOPS - SAVE_AT, MIN_REPLAY), hist[SAVE_AT:], "two-rank file resumed on one GPU")
    r.save(tmp_path / "end_two_on_one.pt")
    _assert_equal(torch.load(tmp_path / "end_two_on_one.pt"), want, "two-rank file resumed on one GPU")


def test_reference_file_loads_and_continues_in_the_reference_code(tmp_path):
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.trainer import BatchedMuzero

    mz = _trainer()
    mz.training_loop(SAVE_AT + 1, MIN_REPLAY)
    ln = mz.learner
    assert ln.step_index > 0
    path = tmp_path / "muzero_model.pt"
    mz.export_reference(path)
    ck = torch.load(path)
    assert set(ck) == {"Muzero_net", "Net_optim"}
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    net.load_state_dict(ck["Muzero_net"], strict=True)
    net.optimiser.load_state_dict(ck["Net_optim"])
    for (key, p), (key2, q) in zip(net.state_dict().items(), ln.state_dict().items()):
        assert key == key2 and torch.equal(p, q.cpu()), key

    before = dict(params=ln.params.clone(), adam_m=ln.adam_m.clone(), adam_v=ln.adam_v.clone(), step_index=ln.step_index)
    back = BatchedMuzero.from_reference(path, N, MAX_STEPS, GAMES, n_mcts_simulations=8, batch_s=64, n_update_x_loop=2)
    _assert_equal(dict(params=back.learner.params, adam_m=back.learner.adam_m, adam_v=back.learner.adam_v,
                       step_index=back.learner.step_index), before, "from_reference of the exported file")

    # the learner's next step vs the reference's Adam given the same gradient
    states, rwds, actions, pi_probs, returns, indx, w = mz.buffer.priority_sample_device(64)
    ln.step(states, rwds, actions, pi_probs, returns, w)
    torch.cuda.synchronize()
    for p, (key, g) in zip(net.parameters(), ln.grad_dict().items()):
        p.grad = g.cpu().clone()
    net.optimiser.step()
    for (key, p), (_, q) in zip(net.named_parameters(), ln.state_dict().items()):
        d = (p.detach() - q.cpu()).abs()
        assert d.max() <= 1e-4 and d.mean() <= 1e-6, (key, float(d.max()), float(d.mean()))
