"""BatchedMuzero with torch.distributed initialised over two ranks — sharded self-play, every move's records all-gathered
and ingested by the single learner on rank 0, weights broadcast back once per loop — trains bit-identically to
BatchedMuzero on one GPU with the same global number of games.  Over NCCL the two ranks run on two GPUs (skips with
fewer); over gloo they share the GPUs there are (rank r on GPU r % count), which runs the same trainer path on one GPU."""
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

N, MAX_STEPS, GAMES, LOOPS, MIN_REPLAY = 3, 40, 256, 14, 100
RING = ("states", "rwds", "actions", "pi_probs", "mc_returns", "priorities")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _trainer(priority_replay):
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.trainer import BatchedMuzero

    torch.manual_seed(7)
    np.random.seed(7)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    return BatchedMuzero(net.state_dict(), N, MAX_STEPS, GAMES, n_mcts_simulations=8, batch_s=64, buffer_size=6000,
                         n_update_x_loop=2, moves_per_loop=8, priority_replay=priority_replay, seed=5)


def _train(priority_replay):
    """-> what a run leaves: learner state, replay ring, history (host copies)."""
    mz = _trainer(priority_replay)
    hist = mz.training_loop(LOOPS, MIN_REPLAY)
    torch.cuda.synchronize()
    out = dict(hist=np.array(hist, dtype=np.float64), episodes_done=mz.episodes_done,
               params=mz.learner.params.cpu(), step_index=mz.learner.step_index)
    if mz.rank == 0:
        out.update(adam_m=mz.learner.adam_m.cpu(), adam_v=mz.learner.adam_v.cpu(), ptr=mz.buffer.ptr, is_full=mz.buffer.is_full,
                   **{k: getattr(mz.buffer, k).cpu() for k in RING})
    return out


def _worker(rank, world, port, backend, priority_replay, out_dir):
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            timeout=datetime.timedelta(seconds=300), **(dict(device_id=dev) if backend == "nccl" else {}))
    try:
        torch.save(_train(priority_replay), os.path.join(out_dir, f"rank{rank}.pt"))
        # the ordering check on the trainer path: gathered records out of order stop every rank at the end of the loop
        from muzero_hanoi_b200 import dist as hdist

        result = hdist.RecordGather.result
        hdist.RecordGather.result = lambda self, i: torch.roll(result(self, i), 1, 0)
        try:
            _trainer(priority_replay).training_loop(2, MIN_REPLAY)
            raised = False
        except RuntimeError as e:
            raised = "out of order" in str(e)
        finally:
            hdist.RecordGather.result = result
        assert raised, rank
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _assert_same_training(a, b, what):
    assert a["step_index"] == b["step_index"] and a["episodes_done"] == b["episodes_done"], what
    for k in ("params", "adam_m", "adam_v", *RING):
        assert torch.equal(a[k], b[k]), (what, k)
    assert (a["ptr"], a["is_full"]) == (b["ptr"], b["is_full"]), what
    assert np.array_equal(a["hist"][:, :2], b["hist"][:, :2], equal_nan=True), what  # loop, mean episode length
    # losses: the loss kernels sum with float32 atomics, so only the summation order may differ
    assert np.allclose(a["hist"][:, 2:], b["hist"][:, 2:], rtol=1e-5, atol=1e-6, equal_nan=True), what


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_rank_training_is_bit_identical_to_one_gpu(tmp_path, backend):
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip(f"NCCL needs 2 GPUs, found {torch.cuda.device_count()}")
    torch.cuda.set_device(0)
    one = _train(True)
    assert one["step_index"] > 0 and (one["ptr"] > MIN_REPLAY or one["is_full"]) and np.isfinite(one["hist"][:, 2]).any()
    _assert_same_training(one, _train(True), "one GPU, run twice")
    mp.spawn(_worker, args=(2, _free_port(), backend, True, str(tmp_path)), nprocs=2, join=True)
    ranks = [torch.load(tmp_path / f"rank{r}.pt", weights_only=False) for r in range(2)]
    _assert_same_training(one, ranks[0], "one GPU vs rank 0 of two")
    # every rank returns the same history, holds the same weights and counts the same episodes
    assert np.array_equal(ranks[0]["hist"], ranks[1]["hist"], equal_nan=True)
    assert torch.equal(ranks[0]["params"], ranks[1]["params"]) and ranks[0]["episodes_done"] == ranks[1]["episodes_done"]
