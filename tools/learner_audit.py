"""Checks every learner update of a training run against the float64 reference of the step (oracle/learner_ref.py).

    python tools/learner_audit.py [--disks 3] [--games 1024] [--loops 400] [--out profiles/learner_audit_n3_g1024.json]

Trains exactly as examples/train_hanoi.py does with the same arguments (same seeds, torch default init, 25 simulations,
8 updates per loop, min_replay_size 5,000).  Before each Learner.step it snapshots the batch, parameters, Adam moments
and step index; after it, it compares every gradient, the parameters, moments, new priorities and losses with the
one-step float64 reference from that snapshot (float32 yardstick on the CPU) under the gates of
tests/test_learner_reference.py.  Writes one JSON document: the card name and power limit, every update that failed a
gate with its failing tensors, and one row per block of 10 loops: the means of the training history (mean episode
length, the three losses of each loop's last update), the number of updates, hazard rows (learner_ref.hazard_rows) and
failing updates, and per gate category the worst ratio (max of the maximum and 99.9th-percentile ratios) over them.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import learner_ref as lref  # noqa: E402
from test_learner_reference import GATES, LR, snapshot  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--disks", type=int, default=3)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--loops", type=int, default=400)
    ap.add_argument("--sims", type=int, default=25)
    ap.add_argument("--updates-per-loop", type=int, default=8)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.trainer import BatchedMuzero

    torch.manual_seed(args.seed)
    np.random.seed(args.seed)
    net = MuZeroNet(3 * args.disks, 6, LR, "cpu", TD_return=True)
    mz = BatchedMuzero(net.state_dict(), args.disks, 200, args.games, n_mcts_simulations=args.sims,
                       n_update_x_loop=args.updates_per_loop, seed=args.seed)
    # the hook sits on Learner.step, the entry point BatchedMuzero's updates call (Learner.update is step + read-back)
    ln, orig, rows = mz.learner, mz.learner.step, []
    loop = [0]

    def audited(states, rwds, actions, pi_probs, returns, priority_w=None, apply_update=True):
        batch = [t.clone() for t in (states, rwds, actions, pi_probs, returns)]
        w = None if priority_w is None else priority_w.clone()
        before, step_index = snapshot(ln), ln.step_index + 1
        new_p, losses = orig(states, rwds, actions, pi_probs, returns, priority_w, apply_update)
        kern = dict(grads=ln.grad_dict(), **snapshot(ln), priorities=None if new_p is None else new_p.cpu(),
                    losses=np.array(losses.cpu().tolist()))
        stats, ref = lref.compare_update(kern, before, step_index, batch, w, LR, ref_device="cuda")
        worst, bad = lref.check(stats, GATES)
        rows.append(dict(update=step_index, loop=loop[0], hazard_rows=int(lref.hazard_rows(ref).sum()), failing=bad,
                         worst={c: max(v) for c, v in worst.items()}))
        if bad:
            print(f"update {step_index} (loop {loop[0]}): {len(bad)} tensors fail: {bad[:6]}", flush=True)
        return new_p, losses

    ln.step = audited

    def log(msg):
        print(msg, flush=True)

    play = mz.play

    def counted_play(n):
        loop[0] += 1
        return play(n)

    mz.play = counted_play
    t0 = time.time()
    hist = mz.training_loop(args.loops, min_replay_size=5000, print_acc=25, log=log)
    cats, block = list(GATES), 10
    per_block = []  # loops [first, first + block): history means, update counts, worst gate ratio per category
    for first in range(1, len(hist) + 1, block):
        hs = [h for h in hist if first <= h[0] < first + block]
        ups = [r for r in rows if first <= r["loop"] < first + block]
        means = [np.nanmean(col) if not np.isnan(col).all() else None for col in np.array([h[1:] for h in hs], dtype=np.float64).T]
        per_block.append([first, hs[-1][0], *(None if m is None else round(float(m), 4) for m in means), len(ups),
                          sum(r["hazard_rows"] for r in ups), sum(bool(r["failing"]) for r in ups),
                          *(round(max((r["worst"][c] for r in ups if c in r["worst"]), default=0.0), 3) for c in cats)])
    doc = dict(card=card(), args={k: v for k, v in vars(args).items() if k != "out"}, gates={c: list(g) for c, g in GATES.items()},
               seconds=round(time.time() - t0, 1), updates=len(rows), failing_updates=[dict(update=r["update"], loop=r["loop"],
                                                                                            failing=r["failing"]) for r in rows if r["failing"]],
               worst_ratios={c: round(max((r["worst"][c] for r in rows if c in r["worst"]), default=0.0), 3) for c in cats},
               per_block_columns=["first_loop", "last_loop", "mean_episode_length", "value_loss", "reward_loss", "policy_loss", "updates",
                                  "hazard_rows", "failing_updates", *(f"worst_{c}_ratio" for c in cats)])
    out = args.out or os.path.join(ROOT, "profiles", f"learner_audit_n{args.disks}_g{args.games}.json")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:  # one block of loops per line, so that the file reads as a table
        f.write(json.dumps(doc)[:-1] + ',\n "per_block": [\n' + ",\n".join(json.dumps(r) for r in per_block) + "\n ]\n}\n")
    print(json.dumps({k: doc[k] for k in ("card", "updates", "failing_updates", "worst_ratios", "seconds")}))

if __name__ == "__main__":
    main()
