"""Times the lesion-experiment grid run condition by condition (acting.get_results, one call per condition) against the
same grid as one batch (acting.get_results_grid), in one process on the same conditions and seeds, and checks that both
return the same numbers.  Two grids: examples/lesion_eval.py's (5 networks x 4 budgets x 2,048 episodes, random starts) and
the reference's acting_ablations shape (8 ablations x 4 start states x 7 budgets x 100 episodes).  The networks are
lesioned copies of one trained briefly on the device, so episode lengths are those of a planning agent.

    python tools/acting_grid_bench.py [--loops 300] [--out profiles/acting_grid_bench.json]
"""
import argparse
import copy
import itertools
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from muzero_hanoi_b200 import _lib, acting
from muzero_hanoi_b200.engine import PackedWeights
from muzero_hanoi_b200.networks import MuZeroNet
from muzero_hanoi_b200.trainer import BatchedMuzero
from oracle import port

N, MAX_STEPS, T, SEED = 3, 200, 0.0, 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().split("\n")[0]
    name, power, clock = (x.strip() for x in q.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def moves_played(steps):
    """Moves get_results plays for one condition: up to the first multiple of 8 at which all first episodes are over."""
    if (steps == 0).any():
        return MAX_STEPS
    return min(MAX_STEPS, -(-int(steps.max()) // 8) * 8)


def run(name, conds):
    sync = torch.cuda.synchronize
    # warm-up: every kernel and both paths at a small size
    small = [dict(c, episode=8) for c in conds[:3]]
    acting.get_results_grid(small, N, MAX_STEPS, T, seed=SEED)
    for c in small:
        acting.get_results(c["weights"], N, MAX_STEPS, 8, [c["n_simulations"]], T, seed=SEED, start_idx=c.get("start_idx"))
    sync()
    t0 = time.perf_counter()
    seq = [acting.get_results(c["weights"], N, MAX_STEPS, c["episode"], [c["n_simulations"]], T, seed=SEED, start_idx=c.get("start_idx"),
                              return_details=True) for c in conds]
    sync()
    t_seq = time.perf_counter() - t0
    stats = {}
    t0 = time.perf_counter()
    grid = acting.get_results_grid(conds, N, MAX_STEPS, T, seed=SEED, return_details=True, stats=stats)
    sync()
    t_grid = time.perf_counter() - t0
    equal = all(g[0] == s[0] and all(np.array_equal(g[1][0][k], s[1][0][k]) for k in ("steps", "errors", "illegal_moves", "min_moves"))
                for g, s in zip(grid, seq))
    sims_seq = sum(c["episode"] * moves_played(s[1][0]["steps"]) * c["n_simulations"] for c, s in zip(conds, seq))
    useful = sims_seq
    out = dict(grid=name, conditions=len(conds), episodes=sum(c["episode"] for c in conds), outputs_equal=bool(equal),
               sequential=dict(wall_s=t_seq, simulations=sims_seq, simulations_per_s=sims_seq / t_seq),
               batched=dict(wall_s=t_grid, simulations=stats["simulations"], simulations_per_s=stats["simulations"] / t_grid,
                            useful_simulations_per_s=useful / t_grid, searches=stats["searches"], moves=stats["moves"]),
               speedup=t_seq / t_grid, mean_error=[g[0][0] for g in grid])
    print(json.dumps({k: v for k, v in out.items() if k != "mean_error"}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--loops", type=int, default=300)
    ap.add_argument("--episodes", type=int, default=2048)
    ap.add_argument("--out", default=os.path.join("profiles", "acting_grid_bench.json"))
    args = ap.parse_args()
    _lib.require_cuda()
    torch.manual_seed(1)
    np.random.seed(1)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    mz = BatchedMuzero(net.state_dict(), N, MAX_STEPS, 512, n_update_x_loop=8, seed=1)
    t0 = time.perf_counter()
    hist = mz.training_loop(args.loops, min_replay_size=5000)
    train_s = time.perf_counter() - t0
    net.load_state_dict({k: v.cpu() for k, v in mz.learner.state_dict().items()})
    mode = _lib.MODE_BF16

    def lesioned(flags):
        return PackedWeights(acting.ablate_networks(*flags, copy.deepcopy(net)).state_dict(), N, mode)

    results = []
    # examples/lesion_eval.py's grid
    settings = [(False, False, False), (True, False, False), (False, True, False), (False, False, True), (True, True, False)]
    nets = [lesioned(f) for f in settings]
    results.append(run("lesion_eval", [dict(weights=w, n_simulations=b, episode=args.episodes) for w in nets for b in (5, 10, 30, 80)]))
    # acting_ablations' shape: 8 ablations x ES / MS / LS / random starts x 7 budgets x 100 episodes
    dist = {i: port.hanoi_solver(port.index_to_state(i, N)) for i in range(3 ** N)}
    starts = [0, min(i for i in dist if dist[i] == 4), min(i for i in dist if dist[i] == 1), None]
    nets = [lesioned(f) for f in itertools.product((False, True), repeat=3)]
    conds = [dict(weights=w, n_simulations=b, episode=100, **({} if s is None else {"start_idx": s}))
             for w in nets for s in starts for b in (5, 10, 30, 50, 80, 110, 150)]
    results.append(run("reference_shape", conds))
    doc = dict(card=card(), mode="bf16", n_disks=N, max_steps=MAX_STEPS, temperature=T, seed=SEED, train_loops=args.loops, train_s=train_s,
               train_last20_mean_length=float(np.mean([h[1] for h in hist[-20:]])), results=results,
               note="host clocks around work that ends in torch.cuda.synchronize(), after a warm-up of both paths; "
                    "batched simulations include the padding of each network's games to whole 256-search blocks")
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    assert all(r["outputs_equal"] for r in results), "grid and per-condition results differ"


if __name__ == "__main__":
    main()
