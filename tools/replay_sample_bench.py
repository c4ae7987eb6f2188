"""What drawing a prioritized replay batch on the device saves.

    python tools/replay_sample_bench.py [--out profiles/replay_sample_bench.json] [--quick]

1. Sampling alone, at 50,000 and 1,048,576 rows, for two kinds of priorities: those of a ring after a short training run
   (N = 3, 4,096 games; tiled to the larger size) and a constructed worst case with many exact half-ulp ties and binade
   crossings that land by rounding up (oracle/replay_ref.constructed_ring).  hmz_replay_sample is timed with CUDA events
   over repeated calls; the host ReplayRing.priority_sample with the host clock, each call ending in a device
   synchronise.  Both draw the same indices (checked).  The number of stretches (binades of the running sum the exact
   cumulative sum walks through) is reported per case.
2. Whole training_loop iterations with the host path (the update as it was: NumPy draw on a host copy of the priorities,
   Learner.update's read-back, update_priorities' upload) and the device path, alternated loop by loop in one process,
   at N = 3 with 512 and 4,096 games and 8 and 64 updates per loop.  Each path keeps its own NumPy / torch RNG state, so
   the two runs are the same run; their parameters and Adam moments are asserted identical at the end.
The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from muzero_hanoi_b200._lib import check, current_stream, ptr
from muzero_hanoi_b200.networks import MuZeroNet
from muzero_hanoi_b200.replay import ReplayRing
from muzero_hanoi_b200.trainer import BatchedMuzero
from oracle import replay_ref as R


def card():
    q = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


class HostPath(BatchedMuzero):
    """BatchedMuzero's update as it was before the device path."""

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


def trained_priorities(rows):
    torch.manual_seed(1)
    np.random.seed(1)
    net = MuZeroNet(9, 6, 0.002, "cpu", TD_return=True)
    mz = BatchedMuzero(net.state_dict(), 3, 200, 4096, n_mcts_simulations=25, n_update_x_loop=8, buffer_size=rows, seed=1)
    loops = 0
    while not mz.buffer.is_full and loops < 60:
        mz.training_loop(2, 5000)
        loops += 1
    return mz.buffer.priorities[:len(mz.buffer)].cpu().numpy(), loops


def ring_with(q):
    ring = ReplayRing(len(q), 5, 9, 6)
    ring.priorities.copy_(torch.from_numpy(q).cuda())
    ring.is_full = True
    return ring


def time_sampling(q, batch, reps):
    ring = ring_with(q)
    num = len(q)
    lib = ring.lib
    ws = torch.empty(int(lib.hmz_replay_sample_workspace_bytes(num)), dtype=torch.uint8, device="cuda")
    u = torch.rand(batch, dtype=torch.float64, device="cuda")
    idx = torch.empty(batch, dtype=torch.int64, device="cuda")
    w = torch.empty(batch, dtype=torch.float32, device="cuda")

    def call():
        check(lib.hmz_replay_sample(ptr(ring.priorities), num, num, 1.0, ptr(u), batch, 0.0, ptr(ws), ptr(idx), ptr(w), ptr(ring.status),
                                    current_stream()))

    for _ in range(5):
        call()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        call()
    ev[1].record()
    torch.cuda.synchronize()
    device_ms = ev[0].elapsed_time(ev[1]) / reps
    host = []
    for i in range(max(3, reps // 5) + 2):
        np.random.seed(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ring.priority_sample(batch)
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) * 1e3)
    host = host[2:]
    np.random.seed(123)
    a = ring.priority_sample(batch)[5]
    np.random.seed(123)
    b = ring.priority_sample_device(batch)[5].cpu().numpy()
    ring.check_status()
    assert np.array_equal(a, b)
    _, info = R.exact_cumsum((q / np.sum(q)).astype(np.float32))
    return dict(rows=num, batch=batch, device_ms=round(device_ms, 4), host_ms_median=round(float(np.median(host)), 3),
                host_ms_min=round(float(np.min(host)), 3), speedup=round(float(np.median(host)) / device_ms, 1), **info)


def rng_state():
    return dict(np=np.random.get_state(), cpu=torch.get_rng_state(), cuda=torch.cuda.get_rng_state())


def set_rng_state(s):
    np.random.set_state(s["np"])
    torch.set_rng_state(s["cpu"])
    torch.cuda.set_rng_state(s["cuda"])


def time_training(games, updates, timed_loops, min_replay):
    runs = {}
    for name, cls in (("device", BatchedMuzero), ("host", HostPath)):
        torch.manual_seed(7)
        np.random.seed(7)
        net = MuZeroNet(9, 6, 0.002, "cpu", TD_return=True)
        mz = cls(net.state_dict(), 3, 200, games, n_mcts_simulations=25, n_update_x_loop=updates, seed=5)
        runs[name] = dict(mz=mz, rng=rng_state(), ms=[])
    warm = 0
    while len(runs["device"]["mz"].buffer) <= min_replay or warm < 2:
        for r in runs.values():
            set_rng_state(r["rng"])
            r["mz"].training_loop(2, min_replay)
            r["rng"] = rng_state()
        warm += 1
    for _ in range(timed_loops):
        for r in runs.values():
            set_rng_state(r["rng"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r["mz"].training_loop(2, min_replay)
            torch.cuda.synchronize()
            r["ms"].append((time.perf_counter() - t0) * 1e3)
            r["rng"] = rng_state()
    d, h = runs["device"]["mz"], runs["host"]["mz"]
    for k in ("params", "adam_m", "adam_v"):
        assert torch.equal(getattr(d.learner, k), getattr(h.learner, k)), k
    assert torch.equal(d.buffer.priorities, h.buffer.priorities)
    dm, hm = float(np.median(runs["device"]["ms"])), float(np.median(runs["host"]["ms"]))
    return dict(games=games, updates_per_loop=updates, warmup_loops=warm, timed_loops=timed_loops, replay_rows=len(d.buffer),
                device_loop_ms_median=round(dm, 2), host_loop_ms_median=round(hm, 2),
                device_loop_ms=[round(x, 2) for x in runs["device"]["ms"]], host_loop_ms=[round(x, 2) for x in runs["host"]["ms"]],
                saved_per_update_ms=round((hm - dm) / updates, 3), identical_parameters=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "replay_sample_bench.json"))
    ap.add_argument("--quick", action="store_true", help="fewer repetitions (a rehearsal)")
    args = ap.parse_args()
    reps, timed = (5, 2) if args.quick else (50, 8)
    doc = dict(card=card(), notes="sampling: device = hmz_replay_sample alone (CUDA events, mean over calls, priorities "
               "resident in L2: 4 MB at 1,048,576 rows); host = ReplayRing.priority_sample (host clock, ends in a device "
               "synchronise, median).  training: one training_loop iteration (8 self-play moves of every game + the "
               "updates), host clock ending in a synchronise, the two paths alternated loop by loop; N = 3, 25 simulations, "
               "batch 256, priority replay.")
    t0 = time.time()
    trained, loops = trained_priorities(50000)
    doc["trained_ring"] = dict(rows=len(trained), training_loops=loops, zero_rows=int((trained == 0).sum()),
                               min_nonzero=float(trained[trained > 0].min()), max=float(trained.max()))
    big = np.resize(trained, 1048576).astype(np.float32)
    doc["sampling"] = []
    for kind, q50, q1m in (("trained", trained[:50000] if len(trained) >= 50000 else np.resize(trained, 50000), big),
                           ("constructed_worst_case", R.constructed_ring(50000, 1), R.constructed_ring(1048576, 2))):
        for q in (q50, q1m):
            row = dict(kind=kind, **time_sampling(np.ascontiguousarray(q, np.float32), 256, reps))
            print(json.dumps(row), flush=True)
            doc["sampling"].append(row)
    doc["training"] = []
    for games in (512, 4096):
        for updates in (8, 64):
            row = time_training(games, updates, timed, 1000)
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("loop_ms")}), flush=True)
            doc["training"].append(row)
    doc["seconds"] = round(time.time() - t0, 1)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc["card"]))


if __name__ == "__main__":
    main()
