"""End-to-end training on the device: batched self-play -> episode post-processing -> replay ring -> learner step,
the loop of the reference's training_main.py / Muzero.training_loop with B games played at once.

    python examples/train_hanoi.py [--disks 3] [--games 512] [--loops 400]
    torchrun --nproc-per-node G examples/train_hanoi.py --games 1024    # G GPUs: self-play on all, one learner on rank 0

--games is the global number of games; under torchrun each GPU plays --games / G of them and the run is bit-identical
to the one-GPU run with the same arguments.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from muzero_hanoi_b200 import dist as hdist
from muzero_hanoi_b200.networks import MuZeroNet
from muzero_hanoi_b200.trainer import BatchedMuzero


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--disks", type=int, default=3)
    ap.add_argument("--games", type=int, default=512)
    ap.add_argument("--loops", type=int, default=400)
    ap.add_argument("--sims", type=int, default=25)
    ap.add_argument("--updates-per-loop", type=int, default=8)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    rank, world, _ = hdist.init_from_env()
    try:
        run(args, rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


def run(args, rank):
    torch.manual_seed(args.seed)
    np.random.seed(args.seed)
    net = MuZeroNet(3 * args.disks, 6, 0.002, "cpu", TD_return=True)  # torch's default init, as training_main.py
    mz = BatchedMuzero(net.state_dict(), args.disks, 200, args.games, n_mcts_simulations=args.sims,
                       n_update_x_loop=args.updates_per_loop, seed=args.seed)
    t0 = time.time()
    hist = mz.training_loop(args.loops, min_replay_size=5000, print_acc=25 if rank == 0 else None)
    if rank != 0:
        return
    lens = [h[1] for h in hist if h[1] == h[1]]
    k = max(1, len(lens) // 10)
    print("mean episode length: first 10%% of loops %.1f, last 10%% %.1f (optimal 7 from the all-on-peg-0 start); "
          "%d episodes, %d updates, %.1f s" % (np.mean(lens[:k]), np.mean(lens[-k:]), mz.episodes_done, mz.learner.step_index,
                                             time.time() - t0))


if __name__ == "__main__":
    main()
