"""The reference's lesion experiment (acting_experiments/acting_ablations.py) on a network trained a moment ago (or
loaded with --checkpoint): train 3-disk Hanoi on the device, then measure the planning error (moves beyond the optimum)
from random starts for several MCTS budgets, intact and with the policy / value / reward heads re-initialised.

    python examples/lesion_eval.py [--loops 300] [--episodes 2048]
    python examples/lesion_eval.py --checkpoint muzero_model.pt      # a trained network instead of training one
"""
import argparse
import copy
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from muzero_hanoi_b200 import acting
from muzero_hanoi_b200.engine import PackedWeights
from muzero_hanoi_b200.learner import split_flat
from muzero_hanoi_b200.networks import MuZeroNet
from muzero_hanoi_b200.trainer import BatchedMuzero, check_checkpoint


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--loops", type=int, default=300)
    ap.add_argument("--episodes", type=int, default=2048)
    ap.add_argument("--checkpoint", metavar="PATH", help="evaluate this network instead of training one: the reference's "
                    "muzero_model.pt (BatchedMuzero.export_reference) or a BatchedMuzero.save file")
    args = ap.parse_args()
    torch.manual_seed(1)
    np.random.seed(1)
    N = 3
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    if args.checkpoint:
        ck = torch.load(args.checkpoint, map_location="cpu")
        if "Muzero_net" in ck:  # the reference's file, loaded as the lesion scripts load it (acting_ablations.py:350-360)
            net.load_state_dict(ck["Muzero_net"])
        else:
            check_checkpoint(ck)
            if ck["config"]["N"] != N:
                raise ValueError(f"{args.checkpoint}: a network of N={ck['config']['N']}, this experiment is N={N}")
            net.load_state_dict(split_flat(ck["learner"]["params"], N))
        print("loaded %s" % args.checkpoint)
    else:
        mz = BatchedMuzero(net.state_dict(), N, 200, 512, n_update_x_loop=8, seed=1)
        hist = mz.training_loop(args.loops, min_replay_size=5000)
        print("trained: mean episode length of the last 20 loops %.1f" % np.mean([h[1] for h in hist[-20:]]))
        net.load_state_dict({k: v.cpu() for k, v in mz.learner.state_dict().items()})
    budgets = [5, 10, 30, 80]
    settings = [("intact", (False, False, False)), ("policy lesion", (True, False, False)), ("value lesion", (False, True, False)),
                ("reward lesion", (False, False, True)), ("policy + value lesion", (True, True, False))]
    # the whole grid (networks x budgets) as one batch of searches; each condition's numbers are those of
    # acting.get_results(weights, N, 200, episodes, [budget], 0.0, seed=3)
    conditions = []
    for _, flags in settings:
        lesioned = acting.ablate_networks(*flags, copy.deepcopy(net))  # acting_ablations.py:29-45
        weights = PackedWeights(lesioned.state_dict(), N)
        conditions += [dict(weights=weights, n_simulations=n, episode=args.episodes) for n in budgets]
    results = acting.get_results_grid(conditions, N, 200, 0.0, seed=3)
    for k, (name, _) in enumerate(settings):
        data = [row for r in results[k * len(budgets):(k + 1) * len(budgets)] for row in r]
        print("%-22s " % name + "  ".join("S=%d: %.2f" % (n, e) for n, e in data))


if __name__ == "__main__":
    main()
