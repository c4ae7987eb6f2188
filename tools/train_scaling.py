"""Where the time of a distributed training loop goes (BatchedMuzero over torch.distributed: self-play on every rank, the
per-move all-gather of the move records, ONE learner on rank 0, the weight broadcast), at several global game counts.

    torchrun --nproc-per-node G tools/train_scaling.py [--games-per-gpu 4096,65536] [--disks 3,5] [--out FILE]
    python tools/train_scaling.py ...          # G = 1: the one-GPU trainer, for comparison

For every (N, games per GPU) it builds a BatchedMuzero with n_games = G x games per GPU and
  1. times whole loops of training_loop with nothing added (host clock ending in a device synchronise): moves/s and
     finished episodes/s of the whole box;
  2. runs more loops with every phase bracketed by device synchronises (so phases cannot overlap; slower than 1) and
     reports per rank: self-play per move (SelfPlay.move), the all-gather per move (RecordGather.submit, which includes
     waiting for the slowest rank), and on rank 0 the per-move ingest, post_process and add_episodes (whose host
     read-back of the row count is the per-move sync), the learner per update, and broadcast + repack per loop;
  3. times rank 0's hmz_episode_rows alone (CUDA events), the single-block scan inside add_episodes.
Finally rank 0 times EpisodeStore.ingest, post_process and hmz_episode_rows alone (CUDA events) on a store of
--ingest-games games (default 8 x 65,536) filled from synthetic in-order records, the rank-0 work of one move of an
8-GPU box at that size.  Rank 0 writes one JSON document (--out, default profiles/train_scaling_<G>gpu.json) with the card name and power limit
read in the same run.
"""
import argparse
import functools
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from muzero_hanoi_b200 import dist as hdist
from muzero_hanoi_b200.engine import SelfPlay
from muzero_hanoi_b200.networks import MuZeroNet
from muzero_hanoi_b200.replay import EpisodeStore, ReplayRing
from muzero_hanoi_b200.trainer import BatchedMuzero

PHASES = {"selfplay_move": (SelfPlay, "move"), "gather": (hdist.RecordGather, "submit"), "ingest": (EpisodeStore, "ingest"),
          "post_process": (EpisodeStore, "post_process"), "add_episodes": (ReplayRing, "add_episodes"),
          "update": (BatchedMuzero, "update"), "broadcast": (BatchedMuzero, "_end_loop"), "repack": (BatchedMuzero, "_refresh_actor")}


class PhaseClock:
    """Wraps the methods of PHASES so that each call is bracketed by device synchronises and its time accumulated."""

    def __init__(self):
        self.total, self.calls, self.on, self._orig = {}, {}, False, {}
        for name, (cls, attr) in PHASES.items():
            orig = getattr(cls, attr)
            self._orig[name] = orig
            setattr(cls, attr, self._wrap(name, orig))

    def _wrap(self, name, fn):
        @functools.wraps(fn)
        def timed(*a, **k):
            if not self.on:
                return fn(*a, **k)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn(*a, **k)
            torch.cuda.synchronize()
            self.total[name] = self.total.get(name, 0.0) + time.perf_counter() - t0
            self.calls[name] = self.calls.get(name, 0) + 1
            return out
        return timed

    def reset(self):
        self.total, self.calls = {}, {}

    def per_call_ms(self):
        return {k: dict(ms_per_call=1e3 * self.total[k] / self.calls[k], calls=self.calls[k]) for k in self.total}


def card():
    q = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def one_config(clock, n_disks, per_gpu, world, rank, args):
    torch.manual_seed(1)
    np.random.seed(1)
    net = MuZeroNet(3 * n_disks, 6, 0.002, "cpu", TD_return=True)
    mz = BatchedMuzero(net.state_dict(), n_disks, 200, per_gpu * world, n_mcts_simulations=args.sims, n_update_x_loop=args.updates,
                       seed=1)
    mz.training_loop(1 + args.warmup, min_replay_size=args.min_replay)  # builds everything, fills the ring
    # 1. whole loops, nothing added
    torch.cuda.synchronize()
    e0, t0 = mz.episodes_done, time.perf_counter()
    steps0 = mz.learner.step_index
    mz.training_loop(1 + args.loops, min_replay_size=args.min_replay)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    moves = args.loops * mz.moves_per_loop * mz.B
    out = dict(N=n_disks, games_per_gpu=per_gpu, n_games=mz.B, loops=args.loops, moves_per_loop=mz.moves_per_loop,
               sims=args.sims, updates_per_loop=args.updates, s_per_loop=wall / args.loops, game_moves_per_s=moves / wall,
               episodes_per_s=(mz.episodes_done - e0) / wall, updates_in_window=mz.learner.step_index - steps0)
    # 2. phase by phase
    clock.reset()
    clock.on = True
    mz.training_loop(1 + args.loops, min_replay_size=args.min_replay)
    clock.on = False
    out["phases"] = clock.per_call_ms()
    # 3. hmz_episode_rows alone on rank 0's store
    if rank == 0:
        st = mz._episodes if world > 1 else mz._selfplay.episodes
        lib, ring = mz.buffer.lib, mz.buffer
        from muzero_hanoi_b200._lib import check, current_stream, ptr

        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(20):
            check(lib.hmz_episode_rows(ptr(st.ep_len), ptr(st.returns), st.B, ring.ptr, 1, ptr(st.row_base), ptr(st.total),
                                       current_stream()))
        ev[1].record()
        torch.cuda.synchronize()
        out["episode_rows_ms"] = ev[0].elapsed_time(ev[1]) / 20
    per_rank = [None] * world
    if world > 1:
        dist.all_gather_object(per_rank, out["phases"])
    else:
        per_rank = [out["phases"]]
    out["phases"] = per_rank
    del mz
    torch.cuda.empty_cache()
    return out


def ingest_alone(n_games, n_disks=5, t_max=200, reps=20):
    """ms per call of the rank-0 per-move kernels on n_games gathered records (CUDA events)."""
    from muzero_hanoi_b200._lib import check, current_stream, ptr

    g = torch.Generator(device="cuda").manual_seed(0)
    counter = torch.randint(0, t_max, (n_games,), device="cuda", generator=g, dtype=torch.int64)
    flags = torch.where(counter % 37 == 0, 9, 0)  # some episodes end (truncation + done): post_process has work
    rec = hdist.pack_records(dict(state=(counter << (2 * n_disks)).to(torch.int32), action=counter % 6, flags=flags,
                                  visits=torch.ones(n_games, 6, dtype=torch.int16, device="cuda"),
                                  root_q=torch.rand(n_games, dtype=torch.float64, device="cuda", generator=g),
                                  reward=torch.zeros(n_games, device="cuda"),
                                  game_lo=torch.arange(n_games, device="cuda") & 0xFFFF))
    st = EpisodeStore(n_games, t_max, n_disks)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(reps):
            fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / reps

    out = dict(n_games=n_games, N=n_disks, t_max=t_max,
               ingest_ms=timed(lambda: st.ingest(rec, 1.0)),
               post_process_ms=timed(lambda: st.post_process(10, 0.8)),
               episode_rows_ms=timed(lambda: check(st.lib.hmz_episode_rows(ptr(st.ep_len), ptr(st.returns), st.B, 0, 0,
                                                                           ptr(st.row_base), ptr(st.total), current_stream()))))
    assert int(st.mismatch.item()) == 0
    out["bytes_per_ingest"] = n_games * (32 + 4 + 1 + 1 + 12 + 8 + 1 + 4 + 4)  # record in; state..exp, cur_slot, ep_len out
    out["ingest_GB_per_s"] = out["bytes_per_ingest"] / out["ingest_ms"] / 1e6
    del st
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games-per-gpu", default="4096,65536")
    ap.add_argument("--disks", default="3,5")
    ap.add_argument("--sims", type=int, default=25)
    ap.add_argument("--updates", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--loops", type=int, default=3)
    ap.add_argument("--min-replay", type=int, default=256)
    ap.add_argument("--ingest-games", type=int, default=8 * 65536)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world, _ = hdist.init_from_env()
    try:
        clock = PhaseClock()
        results = []
        for n_disks in (int(x) for x in args.disks.split(",")):
            for per_gpu in (int(x) for x in args.games_per_gpu.split(",")):
                r = one_config(clock, n_disks, per_gpu, world, rank, args)
                if rank == 0:
                    print(json.dumps(r), flush=True)
                results.append(r)
        alone = ingest_alone(args.ingest_games) if rank == 0 else None
        if rank == 0:
            print(json.dumps(alone), flush=True)
            path = args.out or os.path.join("profiles", f"train_scaling_{world}gpu.json")
            os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
            with open(path, "w") as f:
                settings = {k: v for k, v in vars(args).items() if k != "out"}  # what was measured, not where it went
                json.dump(dict(world=world, card=card(), args=settings, results=results, rank0_kernels_alone=alone), f, indent=1)
            print("wrote", path)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
