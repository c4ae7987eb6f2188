#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native MuZero/Hanoi acting engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode bf16|fp32|fp32x3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2], the config the metric's targets are quoted on): Tower of Hanoi with 5 disks,
65,536 parallel self-play games x 100 MCTS simulations per move, random-init h/g/f networks, Dirichlet root noise,
temperature 1.  The 65,536 games are GLOBAL: with N GPUs every rank owns 65,536 / N of them (strong scaling, as the
config says: "sharded over 1/2/4/8 B200"); the fixed-games-per-GPU number is carried as the secondary `weak` record.
A "step" is MOVES_PER_STEP = 16 consecutive moves of every game, a move being
root inference -> 100 x (select -> g+f MLP -> expand+backup) -> root policy -> record -> env step,
so the default 20 timed steps cover more than a second of device time.
`value` = MCTS simulations / s over all GPUs with the state resident in HBM; `e2e` = the same steps with, every step,
the env words coming from pinned host memory and the step's results (the 32-byte records of its 16 moves, the new env
words) read back to pinned host memory before the next step starts.
One JSON line on stdout (rank 0); progress goes to stderr.
`--dump-outputs DIR` (rank 0) writes what the last timed step handed its caller -- the move records of its moves and the
env words it left -- as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
REF_ROOT = os.path.join(ROOT, "baseline", "_ref")  # unmodified hot-path files of the reference, vendored by build()

N_DISKS, GLOBAL_GAMES, N_SIMS, MAX_STEPS = 5, 65536, 100, 200
MOVES_PER_STEP = 16
DISCOUNT, ALPHA, EPS, TEMPERATURE = 0.8, 0.25, 0.25, 1.0
FLOP_PER_SIM = 203_776  # SURVEY.md §3.3 / §8d: 101,888 MAC of g + reward/policy/value heads, un-padded
ENV_BYTES_PER_STEP, ENV_BYTES_PER_RANDOM_STEP = 14, 13  # SURVEY.md §8d: word r/w 8 + action 1 + reward 4 + flags 1
METRIC, UNIT = "mcts_simulations_per_second", "sims/s"
DUMP_BUDGET_BYTES = 64_000_000  # --dump-outputs: above this, a fixed, seeded sample of the games is written


def tree_bytes_per_sim(depth, latent_bytes=128):
    """SURVEY.md §8d: select 128 B/level, backup 28 B/node over depth + 1 nodes, min/max 32 B, expansion
    (prior 24 + rwd 4 + 72 zeroed + latent row written + parent latent row read) => 156 d + 160 + 2 x latent row."""
    return 156.0 * depth + 160.0 + 2.0 * latent_bytes


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, for one) print to
    file descriptor 1 from C, so fd 1 is pointed at stderr for the whole run and the JSON line is written
    to a private duplicate of the original stdout at the end."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# --------------------------------------------------------------------------- CPU arms (host cores)
def import_ref():
    """The UNMODIFIED reference (baseline/_ref: env/, MCTS/, networks.py, utils.py copied by __graft_entry__.build())
    behind stub plotting modules (its utils.py imports matplotlib / seaborn at module top; SURVEY.md §8c)."""
    import types

    for name in ("matplotlib", "matplotlib.pyplot", "seaborn"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import env.hanoi as ref_env
    import MCTS.mcts as ref_mcts
    import networks as ref_net

    assert ref_env.__file__.startswith(REF_ROOT) and ref_mcts.__file__.startswith(REF_ROOT), (ref_env.__file__, ref_mcts.__file__)
    return ref_env.TowersOfHanoi, ref_mcts.MCTS, ref_net.MuZeroNet


def ref_available():
    return all(os.path.exists(os.path.join(REF_ROOT, p)) for p in ("env/hanoi.py", "MCTS/mcts.py", "MCTS/node.py", "networks.py", "utils.py"))


def _search_worker(idx, cfg, barrier, out):
    """One host process playing self-play moves with the reference's own MCTS.run_mcts / TowersOfHanoi.step
    (kind "reference") or with the oracle port (kind "port"), for cfg["budget_s"] seconds after cfg["warm_moves"]."""
    import numpy as np
    import torch

    torch.set_num_threads(1)
    torch.manual_seed(1000 + idx)
    np.random.seed(1000 + idx)
    n, S, alpha, T = cfg["n_disks"], cfg["n_sims"], cfg["alpha"], cfg["temperature"]
    if cfg["kind"] == "reference":
        TowersOfHanoi, MCTS, MuZeroNet = import_ref()
        env = TowersOfHanoi(N=n, max_steps=MAX_STEPS)
        net = MuZeroNet(rpr_input_s=3 * n, action_s=6, lr=0.002, device="cpu", TD_return=True)
        for head in cfg["lesion"]:  # acting_ablations.ablate_networks (acting_ablations.py:29-45)
            getattr(net, head).apply(net.reset_param)
        mcts = MCTS(discount=DISCOUNT, root_dirichlet_alpha=alpha, n_simulations=S, batch_s=1, device="cpu")
        state = {"obs": env.random_reset() if cfg["random_start"] else env.reset()}

        def one_move():
            action, _, _ = mcts.run_mcts(state["obs"], net, T, False)
            obs, _, done, _ = env.step(action)
            state["obs"] = (env.random_reset() if cfg["random_start"] else env.reset()) if done else obs
    else:
        from oracle import port

        rng = np.random.default_rng(1000 + idx)
        sd = port.make_weights(n, 0)
        if cfg["lesion"]:
            sd = port.lesion_weights(sd, tuple(cfg["lesion"]), seed=5)
        net, env, mm = port.PortNet(sd), port.PortHanoi(n, MAX_STEPS), port.MinMax()
        state = {"obs": env.reset()}

        def one_move():
            a, _, _, _, _ = port.run_mcts_port(state["obs"], net, port.PortSearch(DISCOUNT, S, mm), T, False, alpha=alpha,
                                               noise=rng.dirichlet(np.full(6, alpha)) if alpha > 0 else None, u=rng.random())
            obs, _, done, _ = env.step(a)
            state["obs"] = env.reset() if done else obs
    for _ in range(cfg["warm_moves"]):
        one_move()
    barrier.wait()
    moves, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < cfg["budget_s"]:
        one_move()
        moves += 1
    out.put((idx, moves * S, moves, time.perf_counter() - t0))


def _env_worker(idx, cfg, barrier, out):
    """Config-4 host equivalent: TowersOfHanoi.step on a uniformly random LEGAL move found by scanning _move_allowed over
    moves (as legal_illegal_preds.py:51 does) — reference env when vendored, else the oracle port."""
    import numpy as np

    n = cfg["n_disks"]
    rng = np.random.default_rng(idx)
    if cfg["kind"] == "reference":
        TowersOfHanoi, _, _ = import_ref()
        env = TowersOfHanoi(N=n, max_steps=MAX_STEPS)
    else:
        from oracle import port

        env = port.PortHanoi(n, MAX_STEPS)
    env.reset()
    draws = rng.random(4096)

    def one_step(k):
        legal = [a for a in range(6) if env._move_allowed(env.moves[a])]
        _, _, done, _ = env.step(legal[int(draws[k & 4095] * len(legal))])
        if done:
            env.reset()
    for k in range(2000):
        one_step(k)
    barrier.wait()
    steps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < cfg["budget_s"]:
        for k in range(256):
            one_step(steps + k)
        steps += 256
    out.put((idx, steps, steps, time.perf_counter() - t0))


def run_host_processes(worker, cfg, n_procs):
    """P forked processes, released together by a barrier, each running for cfg["budget_s"]; the aggregate rate is the
    summed work over the longest elapsed time.  No per-step pool.map: the processes run free for the whole budget."""
    ctx = mp.get_context("fork")
    barrier, out = ctx.Barrier(n_procs), ctx.Queue()
    procs = [ctx.Process(target=worker, args=(i, cfg, barrier, out), daemon=True) for i in range(n_procs)]
    for p in procs:
        p.start()
    res = [out.get(timeout=cfg["budget_s"] * 6 + 600) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    wall = max(r[3] for r in res)
    return sum(r[1] for r in res) / wall, sum(r[2] for r in res) / wall, wall, sum(r[1] for r in res)


def search_cpu_cfg(budget_s, warm_moves=1, n_disks=N_DISKS, n_sims=N_SIMS, alpha=ALPHA, temperature=TEMPERATURE, lesion=(),
                   random_start=False):
    return dict(kind="reference" if ref_available() else "port", n_disks=n_disks, n_sims=n_sims, alpha=alpha,
                temperature=temperature, lesion=list(lesion), random_start=random_start, budget_s=budget_s, warm_moves=warm_moves)


def cpu_baseline_record(cfg, cores, rate, moves_rate, wall, sims):
    src = ("the UNMODIFIED reference (baseline/_ref: MCTS.run_mcts + TowersOfHanoi.step + MuZeroNet, torch CPU, 1 thread per process)"
           if cfg["kind"] == "reference" else "oracle/port.py (numpy tree + 1-row fp32 torch net); baseline/_ref is absent")
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": cfg["kind"], "cpu_model": cpu_model(),
            "sample": f"{cores} processes x {wall:.1f} s of N={cfg['n_disks']}, S={cfg['n_sims']} self-play moves ({sims} simulations) through {src}",
            "env_steps_per_second": moves_rate}


def env_cpu_baseline(cores, budget_s):
    out = {"cores": cores, "cpu_model": cpu_model(), "unit": "env steps/s",
           "what": "TowersOfHanoi.step on a uniformly random legal move found by scanning _move_allowed over the 6 moves "
                   "(env/hanoi.py:47-84, :123-139; BASELINE.json configs[3] host equivalent)"}
    for n in (10, 5):
        cfg = dict(kind="reference" if ref_available() else "port", n_disks=n, budget_s=budget_s)
        rate, _, wall, steps = run_host_processes(_env_worker, cfg, cores)
        out[f"n{n}"] = {"value": rate, "kind": cfg["kind"], "sample": f"{cores} processes x {wall:.1f} s ({steps} steps)"}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (baseline/_ref, unmodified) on every host
    core, same metric / unit / config.  Each of the P processes plays `warmup` moves, then all run free for
    steps x 0.5 s; value = simulations completed / longest elapsed time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    cfg = search_cpu_cfg(budget_s=max(2.0, 0.5 * args.steps), warm_moves=max(1, args.warmup))
    log(f"[bench] reference arm: {cfg['kind']} on {cores} processes for {cfg['budget_s']:.1f} s ...")
    rate, moves_rate, wall, sims = run_host_processes(_search_worker, cfg, cores)
    base = cpu_baseline_record(cfg, cores, rate, moves_rate, wall, sims)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": wall / max(1, args.steps) * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1, "f32 (torch CPU)", None),
        "cpu_baseline": base,
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "env_steps_per_second": moves_rate,
    }
    emit(line)


# ------------------------------------------------------------------------------------ ours
def workload_config(args, world, mode, schedule):
    per_gpu = args.games // world
    return {
        "workload": f"hanoi{N_DISKS}_selfplay_{args.games}games_x{args.sims}sims (BASELINE.json configs[2]), "
                    f"{per_gpu} games per GPU on {world} GPU(s)",
        "n_disks": N_DISKS, "global_games": args.games, "games_per_gpu": per_gpu, "n_simulations": args.sims,
        "moves_per_step": MOVES_PER_STEP, "max_steps": MAX_STEPS, "discount": DISCOUNT, "dirichlet_alpha": ALPHA,
        "temperature": TEMPERATURE, "mode": mode, "search_schedule": schedule,
        "parallelism": f"games sharded over {world} GPU(s); NCCL all-gather of 32-byte move records only, on a side stream",
        "cache": "working set (tree + latents, 26 KB per game) is larger than the 126 MB L2 at >= 8,192 games per GPU; no L2 flush needed",
    }


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML from a thread, every 10 ms; nvidia-smi's
    `-lms` loop buffers its output when piped, which is why round 1's sampler saw nothing on the driver's box)."""

    def __init__(self, gpu_index=0):
        self.rows, self.gpu, self.stop_flag, self.thread, self.err = [], gpu_index, False, None, None
        self.t0 = self.t1 = None

    def start(self):
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    power = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    power = None
                self.rows.append((time.perf_counter(), sm, mx, int(get_reasons(h)), power))
                time.sleep(0.01)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=2)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                "hw_power_brake_slowdown": 0x80}
        inside = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or r[0])]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"no samples ({self.err or 'region too short'})"], "samples": 0}
        sm = sorted(r[1] for r in inside)
        mask = 0
        for r in inside:
            mask |= r[3]
        power = [r[4] for r in inside if r[4] is not None]
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_min_mhz": float(sm[0]), "sm_max_mhz": float(inside[0][2]),
                "reasons": sorted(k for k, b in bits.items() if mask & b), "samples": len(inside),
                "power_w_max": max(power) if power else None}


def mean_leaf_depth(sp, sample=4096):
    """Mean leaf depth of the move just searched, measured from the trees themselves: a simulation whose leaf sits at
    depth d adds one visit to each of the d child slots on its path, so sum(child N over all records) / S = mean depth."""
    import numpy as np
    import torch

    st = sp.mcts.store
    b = min(sample, st.B)
    raw = st.nodes[: b * st.n_records * 128].view(torch.int16).cpu().numpy().view(np.uint16)  # 16-byte blocks = 8 x u16 each
    slots = raw.reshape(b, st.n_records, 2, 4, 8)[:, : sp.S + 1, :, :3, 6]  # N = u16 at byte 12 of child slots 0..2 of each half
    return float(slots.astype(np.int64).sum() / (b * sp.S))


def network_accuracy(net, n, dev, rows=4096):
    """Max relative error (elements with |ref| >= 1e-3) of recurrent_inference in both kernel modes against a float64
    evaluation of the SAME weights through the module's own differentiable forms (networks.py:129-196).  The gate
    against the reference's recorded float32 outputs (tests/golden/net_io.npz) is tests/test_net_gpu.py."""
    import copy

    import torch

    from muzero_hanoi_b200 import _lib
    from muzero_hanoi_b200.engine import PackedWeights

    g = torch.Generator().manual_seed(5)
    h_in = torch.rand(rows, 64, generator=g)
    acts = torch.randint(0, 6, (rows,), generator=g)
    net64 = copy.deepcopy(net).double()
    with torch.no_grad():
        h2, r = net64.dynamics(h_in.double(), torch.nn.functional.one_hot(acts, 6).double())
        logits, v = net64.prediction(h2)
        ref = dict(h=h2, r=r.reshape(-1), p=torch.softmax(logits, -1), v=v.reshape(-1))
    out = {}
    for name, md, ld in (("fp32", _lib.MODE_FP32, _lib.LATENT_F32), ("fp32x3", _lib.MODE_FP32X3, _lib.LATENT_F32),
                         ("bf16", _lib.MODE_BF16, _lib.LATENT_F32)):
        w = PackedWeights(net.state_dict(), n, md, dev)
        h = torch.empty(rows, 64, device=dev)
        rr, vv, pp = torch.empty(rows, device=dev), torch.empty(rows, device=dev), torch.empty(rows, 6, device=dev)
        w.recurrent(rows, latents_in=h_in.to(dev), in_rows_per_item=1, in_row=None, actions=acts.to(torch.uint8).to(dev), latents_out=h,
                    out_rows_per_item=1, out_row=0, latent_dtype=ld, r=rr, p=pp, v=vv)
        torch.cuda.synchronize()
        got = dict(h=h, r=rr, p=pp, v=vv)
        rec = {}
        for k in ("h", "p", "r", "v"):
            d = (got[k].double().cpu() - ref[k]).abs()
            big = ref[k].abs() >= 1e-3
            rec[k + "_max_abs"] = float(d.max())
            rec[k + "_max_rel"] = float((d[big] / ref[k].abs()[big]).max()) if bool(big.any()) else 0.0
        out[name] = rec
    out["reference"] = f"float64 evaluation of the same weights on {rows} random latents; tolerance gates: 1e-5 relative (fp32 = FFMA kernel, fp32x3 = tcgen05 with three bf16 parts per operand), 2e-2 (bf16)"
    return out


def dump_outputs(out_dir, sp, n_moves):
    """Writes the outputs of the last n_moves SelfPlay.move() calls: every field of their move records (dist.unpack_records)
    as [move, game] arrays (visits [move, game, 6]), the env words the last move left ([game]) and the global id of every
    game row (game.npy), all float32 / float64 (exact for every integer field).  Above DUMP_BUDGET_BYTES the rows are a
    fixed, seeded sample of the games.  The record ring must hold n_moves slots."""
    import numpy as np
    import torch

    from muzero_hanoi_b200 import _lib

    assert sp.T >= n_moves
    per_game = n_moves * (8 + 8 + 4 + 6 * 4 + 3 * 4) + 8 + 8
    games = np.arange(sp.B)
    if per_game * sp.B > DUMP_BUDGET_BYTES:
        games = np.sort(np.random.default_rng(0).choice(sp.B, DUMP_BUDGET_BYTES // per_game, replace=False))
    idx = torch.as_tensor(games, device=sp.device)
    slots = torch.as_tensor([(sp.moves_done - n_moves + k) % sp.T for k in range(n_moves)], device=sp.device)
    raw = sp.records.index_select(0, slots).index_select(1, idx).cpu().numpy()  # uint8 [move, game, 32]
    rec = raw.view(np.dtype(_lib.RECORD_DTYPE))[..., 0]
    arrays = {"root_q": rec["root_q"].astype(np.float64), "state": rec["state"].astype(np.float64),
              "reward": rec["reward"].astype(np.float32), "visits": rec["visits"].astype(np.float32),
              "action": rec["action"].astype(np.float32), "flags": rec["flags"].astype(np.float32),
              "game_lo": rec["game_lo"].astype(np.float32),
              "env_words": sp.env.words.index_select(0, idx).cpu().numpy().view(np.uint32).astype(np.float64),
              "game": (sp.game_offset + games).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] wrote {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 1e6:.1f} MB, {len(games)} of {sp.B} games "
        f"x {n_moves} moves) to {out_dir}")


def run_ours(args):
    import ctypes as C

    import numpy as np
    import torch
    import torch.distributed as dist

    # CPU baselines first (rank 0, N=1 only): fork()ing is only safe before CUDA is initialised.
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    cpu_baseline = env_cpu = None
    if world_env == 1 and args.gpus == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        cfg = search_cpu_cfg(budget_s=args.cpu_seconds)
        log(f"[bench] CPU baseline: {cfg['kind']} on {cores} processes for ~{args.cpu_seconds:.0f} s ...")
        rate, moves_rate, wall, sims = run_host_processes(_search_worker, cfg, cores)
        cpu_baseline = cpu_baseline_record(cfg, cores, rate, moves_rate, wall, sims)
        log(f"[bench] CPU baseline: {rate:.1f} sims/s on {cores} cores ({cfg['kind']})")
        env_cpu = env_cpu_baseline(cores, budget_s=max(1.0, args.cpu_seconds / 4))
        log(f"[bench] CPU env baseline: N=10 {env_cpu['n10']['value']:.3e}, N=5 {env_cpu['n5']['value']:.3e} steps/s")

    from muzero_hanoi_b200 import _lib, acting
    from muzero_hanoi_b200 import dist as hdist
    from muzero_hanoi_b200.engine import PackedWeights, SelfPlay, VecHanoi
    from muzero_hanoi_b200.networks import MuZeroNet

    rank, world, local = hdist.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load()
    flags = lib.hmz_build_flags().decode()
    mode = {"bf16": _lib.MODE_BF16, "fp32": _lib.MODE_FP32, "fp32x3": _lib.MODE_FP32X3}[args.mode]
    latent_dtype = _lib.LATENT_BF16 if args.mode == "bf16" else _lib.LATENT_F32
    torch.manual_seed(0)
    net = MuZeroNet(3 * N_DISKS, 6, 0.002, "cpu", TD_return=True)  # random-init h / g / f
    weights = PackedWeights(net.state_dict(), N_DISKS, mode, dev)
    if args.games % world:
        raise SystemExit(f"--games {args.games} is not divisible by {world} ranks")
    B, S = args.games // world, args.sims
    schedule = {"auto": _lib.SCHEDULE_AUTO, "persistent": _lib.SCHEDULE_PERSISTENT, "server": _lib.SCHEDULE_SERVER}.get(args.schedule, None)
    if schedule is None:
        schedule = int(args.schedule)

    # --dump-outputs: a record ring that holds every move of a step, so that the last timed step's records are still there
    ring_slots = max(4, MOVES_PER_STEP) if args.dump_outputs else 4

    def make_selfplay(games, offset, sched=schedule):
        sp_ = SelfPlay(N_DISKS, MAX_STEPS, games, S, weights, DISCOUNT, ALPHA, EPS, TEMPERATURE, seed=1234, ring_slots=ring_slots,
                       device=dev, latent_dtype=latent_dtype, game_offset=offset)
        sp_.mcts.store.set_schedule(sched)
        return sp_

    sp = make_selfplay(B, rank * B)
    gather = hdist.RecordGather(B, world, dev, depth=2) if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def make_step(sp_, gather_):
        def step():
            for _ in range(MOVES_PER_STEP):
                t = sp_.move()
                if gather_ is not None:
                    gather_.submit(sp_.slot(t))
        return step

    step = make_step(sp, gather)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    warm = max(args.warmup, 3)
    log(f"[bench] rank {rank}/{world}: warm-up {warm} steps x {MOVES_PER_STEP} moves (B={B}, S={S}, mode={args.mode}, schedule={args.schedule})")
    for _ in range(warm):
        step()
    barrier()
    launches0 = lib.hmz_launch_count()
    sampler.mark_begin()
    ms = timed(step, args.steps)
    sampler.mark_end()
    launches = lib.hmz_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    moves = args.steps * MOVES_PER_STEP
    sims_per_s = world * B * S * moves / (ms * 1e-3)
    depth = mean_leaf_depth(sp)
    log(f"[bench] {ms / args.steps:.2f} ms/step ({ms / moves:.3f} ms/move) -> {sims_per_s:.3e} sims/s; mean leaf depth {depth:.2f}")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sp, MOVES_PER_STEP)

    # ---- per-kernel device time over one step (CUDA-event pairs recorded by the library on its launch streams)
    def kernel_profile(sp_, sched):
        sp_.mcts.store.set_schedule(sched)
        for _ in range(2):
            sp_.move()
        barrier()
        _lib.check(lib.hmz_prof_begin())
        for _ in range(MOVES_PER_STEP):
            sp_.move()
        ms_cls, n_cls = (C.c_double * 8)(), (C.c_int64 * 8)()
        _lib.check(lib.hmz_prof_end(ms_cls, n_cls))
        sp_.mcts.store.set_schedule(schedule)
        names = ["env_step", "select", "net_recurrent", "backup_select", "net_initial", "move_finish", "move_begin_and_other", "search_persistent"]
        kern = {names[i]: {"ms_total": ms_cls[i], "launches": int(n_cls[i]),
                           "us_per_launch": (ms_cls[i] / n_cls[i] * 1e3) if n_cls[i] else None} for i in range(8) if n_cls[i]}
        total = sum(v["ms_total"] for v in kern.values())
        for v in kern.values():
            v["share"] = v["ms_total"] / total if total else None
        return kern

    peaks = measured_peaks()
    try:  # DRAM traffic per launch from the committed ncu --set full capture of this workload (profiles/)
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            traffic = json.load(f)
    except (OSError, ValueError):
        traffic = {}

    def traffic_of(name, games):
        t = traffic.get(name, {}) if games == GLOBAL_GAMES and S == N_SIMS else {}
        return t.get("dram_bytes_per_launch"), (traffic.get("source") if t else None)

    latent_row = 128 if args.mode == "bf16" else 256
    kern = kernel_profile(sp, schedule)
    rooflines = {}
    bps = tree_bytes_per_sim(depth, latent_row)
    if "search_persistent" in kern:  # one kernel per move: both roles share its duration
        per_launch_s = kern["search_persistent"]["us_per_launch"] * 1e-6
        tr, src = traffic_of("search_persistent", B)
        rooflines["hbm"] = {
            "kernel": "search_persistent (tree CTAs: expand + backup + select; MLP CTAs: g + f on tcgen05; one launch per move)",
            "bound": "hbm", "achieved": bps * B * S / per_launch_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": bps * B * S / per_launch_s / 1e9 / peaks["hbm_gbs"], "traffic": tr, "traffic_source": src,
            "peak_source": peaks["source"],
            "algorithmic": f"(156 d + 160 + 2 x {latent_row}) = {bps:.0f} B/sim (SURVEY §8d, measured mean leaf depth d = {depth:.2f}) x {B} searches x {S} sims per launch",
            "tree_only_frac": (156.0 * depth + 160.0) * B * S / per_launch_s / 1e9 / peaks["hbm_gbs"]}
        ach = FLOP_PER_SIM * B * S / per_launch_s / 1e12
        rooflines["tensor"] = {
            "kernel": "search_persistent, MLP role (fused g + reward/policy/value heads, tcgen05)", "bound": "tensor",
            "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops_sustained"],
            "traffic": None, "peak_source": peaks["source"] + ", sustained bf16",
            "algorithmic": f"{FLOP_PER_SIM} FLOP/sim x {B} searches x {S} sims per launch"}
        roofline, roofline_other = rooflines["hbm"], rooflines["tensor"]
    else:
        def roofline_of(name):
            per_launch_s = kern[name]["us_per_launch"] * 1e-6
            # (the ncu captures are of the bf16 network kernel and of net_x3; the FFMA kernel has none)
            tr, src = traffic_of({"fp32x3": "net_x3_recurrent", "fp32": "net_recurrent_fp32"}.get(args.mode, name) if name == "net_recurrent" else name, B)
            if name == "net_recurrent":
                ach = FLOP_PER_SIM * B / per_launch_s / 1e12
                return {"kernel": "net_tc<recurrent> (fused g + reward/policy/value heads, tcgen05)" if args.mode == "bf16" else ("net_recurrent_fp32 (FFMA)" if args.mode == "fp32" else "net_x3_recurrent (tcgen05, three bf16 parts per float32 operand)"),
                        "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                        "frac": ach / peaks["bf16_tflops_sustained"], "traffic": tr, "traffic_source": src,
                        "peak_source": peaks["source"] + ", sustained bf16", "algorithmic": f"{FLOP_PER_SIM} FLOP/sim x {B} sims per launch",
                        **({"executed_bf16": 7 * ach, "executed_frac": 7 * ach / peaks["bf16_tflops_sustained"],
                            "executed_note": "float32 accuracy from seven exact bf16 x bf16 products per multiply: the tensor cores execute 7 x the algorithmic FLOPs"}
                           if args.mode == "fp32x3" else {})}
            tb = 156.0 * depth + 160.0
            return {"kernel": "search_backup_select (expand + backup + next select)", "bound": "hbm", "achieved": tb * B / per_launch_s / 1e9,
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": tb * B / per_launch_s / 1e9 / peaks["hbm_gbs"], "traffic": tr,
                    "traffic_source": src, "peak_source": peaks["source"],
                    "algorithmic": f"(156 d + 160) = {tb:.0f} B/sim (SURVEY §8d tree bytes, measured mean leaf depth d = {depth:.2f}) x {B} sims per launch"}
        serial = kernel_profile(sp, 1)  # serial launches: clean, non-overlapped per-kernel durations
        kern = serial
        dominant = max(("net_recurrent", "backup_select"), key=lambda k: kern[k]["ms_total"])
        other = "backup_select" if dominant == "net_recurrent" else "net_recurrent"
        roofline, roofline_other = roofline_of(dominant), roofline_of(other)

    # ---- end to end, through the public API (SelfPlay.move) with HOST buffers: every step the env words of all games come
    #      from pinned host memory (H2D) and the step's results — the 32-byte records of its 16 moves and the new env
    #      words — are read back to pinned host memory (D2H), then the host waits for them; the next step starts from the
    #      words the host just received.
    h_words = torch.empty(B, dtype=torch.int32).pin_memory()
    h_words.copy_(sp.env.words.cpu())
    h_rec = torch.empty(MOVES_PER_STEP, B, _lib.RECORD_BYTES, dtype=torch.uint8).pin_memory()
    h_next = torch.empty(B, dtype=torch.int32).pin_memory()

    def e2e_step():
        sp.env.words.copy_(h_words, non_blocking=True)
        for k in range(MOVES_PER_STEP):
            t = sp.move()
            h_rec[k].copy_(sp.slot(t), non_blocking=True)
            if gather is not None:
                gather.submit(sp.slot(t))
        h_next.copy_(sp.env.words, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        h_words.copy_(h_next)  # the host owns the env state between steps

    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    e2e_rate = world * B * S * moves / (ms_e2e * 1e-3)
    h2d, d2h = 4 * B, _lib.RECORD_BYTES * B * MOVES_PER_STEP + 4 * B
    log(f"[bench] e2e {ms_e2e / args.steps:.2f} ms/step -> {e2e_rate:.3e} sims/s")

    # ---- weak-scaling record (N > 1): the fixed-games-per-GPU number of round 1, a few steps
    weak = None
    if world > 1 and not args.no_weak:
        del sp, gather
        torch.cuda.empty_cache()
        spw = make_selfplay(args.games, rank * args.games)
        gw = hdist.RecordGather(args.games, world, dev, depth=2)
        stepw = make_step(spw, gw)
        for _ in range(2):
            stepw()
        kw = max(2, args.steps // 4)
        msw = timed(stepw, kw)
        weak = {"scaling": "weak", "games_per_gpu": args.games, "global_games": args.games * world, "steps": kw,
                "ms_per_step": msw / kw, "ms_per_move": msw / (kw * MOVES_PER_STEP),
                "value": world * args.games * S * kw * MOVES_PER_STEP / (msw * 1e-3), "unit": UNIT}
        gw.drain()
        del spw, gw
        torch.cuda.empty_cache()

    # ---- raw env throughput (BASELINE.json configs[3]: N=10, 2^24 envs, random legal moves; N=5 as well)
    env_line = None
    if not args.no_env:
        env_line = {}
        nenv = 1 << 24
        for n in (10, 5):
            env = VecHanoi(n, 200, nenv, dev)
            env.reset()
            acts = torch.randint(0, 6, (nenv,), dtype=torch.uint8, device=dev)
            k_env = [0]

            def env_step_fixed():
                env.step(acts, want_obs=False)

            def env_step_rand():
                env.step_random(seed=1, step_index=k_env[0])
                k_env[0] += 1

            for f in (env_step_fixed, env_step_rand):
                for _ in range(3):
                    f()
            ms_env = timed(env_step_fixed, 50) / 50
            ms_rand = timed(env_step_rand, 50) / 50
            ms_roll = timed(lambda: env.rollout_random(64, seed=1, step_index=0), 3) / 3
            gbs, gbs_r = ENV_BYTES_PER_STEP * nenv / (ms_env * 1e-3) / 1e9, ENV_BYTES_PER_RANDOM_STEP * nenv / (ms_rand * 1e-3) / 1e9
            env_line[f"n{n}"] = {
                "workload": f"hanoi{n}_2^24envs_per_gpu" + (" (BASELINE.json configs[3])" if n == 10 else ""), "n_envs_per_gpu": nenv,
                "step_given_actions_per_s": world * nenv / (ms_env * 1e-3), "step_random_legal_per_s": world * nenv / (ms_rand * 1e-3),
                "fused_rollout64_random_legal_per_s": world * nenv * 64 / (ms_roll * 1e-3),
                "roofline": {"kernel": "env_step_vec4", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": gbs / peaks["hbm_gbs"], "algorithmic": f"{ENV_BYTES_PER_STEP} B/step x {nenv} steps per launch"},
                "roofline_random": {"kernel": "env_step_random_vec4", "bound": "hbm", "achieved": gbs_r, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": gbs_r / peaks["hbm_gbs"], "algorithmic": f"{ENV_BYTES_PER_RANDOM_STEP} B/step x {nenv} steps per launch"}}
            del env, acts
        if env_cpu is not None:
            env_line["cpu_baseline"] = env_cpu

    # ---- the other BASELINE.json configs and the parity (fp32) mode, each with its own ms per move (N = 1 only)
    sub = None
    if world == 1 and not args.no_configs:
        sub = {}

        def time_moves(sp_, n_moves, warm_moves=3):
            for _ in range(warm_moves):
                sp_.move()
            return timed(lambda: sp_.move(), n_moves) / n_moves

        def sub_record(name, n, games, sims, alpha, temp, heads, modes, n_moves):
            torch.manual_seed(1)
            net_ = MuZeroNet(3 * n, 6, 0.002, "cpu", TD_return=True)
            if heads:  # acting_ablations.ablate_networks (acting_ablations.py:29-45): re-initialised heads
                acting.ablate_networks("policy_net" in heads, "value_net" in heads, "rwd_net" in heads, net_)
            rec = {"workload": name, "n_disks": n, "games": games, "n_simulations": sims, "dirichlet_alpha": alpha, "temperature": temp,
                   "lesioned_heads": list(heads)}
            for m_name in modes:
                md = {"bf16": _lib.MODE_BF16, "fp32": _lib.MODE_FP32, "fp32x3": _lib.MODE_FP32X3}[m_name]
                ld = _lib.LATENT_BF16 if m_name == "bf16" else _lib.LATENT_F32
                w_ = PackedWeights(net_.state_dict(), n, md, dev)
                sp_ = SelfPlay(n, MAX_STEPS, games, sims, w_, DISCOUNT, alpha, EPS, temp, seed=7, ring_slots=4, device=dev, latent_dtype=ld)
                sp_.env.random_reset(seed=3)
                sp_.mcts.store.set_schedule(schedule if m_name == "bf16" else _lib.SCHEDULE_AUTO)
                ms_move = time_moves(sp_, n_moves if m_name == "bf16" else max(2, n_moves // (8 if m_name == "fp32" else 2)))
                rec[m_name] = {"ms_per_step": ms_move, "step": "one move of every game", "value": games * sims / (ms_move * 1e-3), "unit": UNIT,
                               "mean_leaf_depth": mean_leaf_depth(sp_)}
                del sp_, w_
            return rec

        sub["configs_1"] = sub_record("hanoi3_4096searches_x50sims (BASELINE.json configs[1]; fp32 = the bit-exact-gated parity mode)",
                                      3, 4096, 50, ALPHA, 1.0, (), ("fp32", "fp32x3", "bf16"), 64)
        sub["configs_4"] = sub_record("hanoi4_lesion_16384searches_x200sims_T0 (BASELINE.json configs[4], acting_ablations.py lesion mode)",
                                      4, 16384, 200, 0.0, 0.0, ("policy_net", "value_net", "rwd_net"), ("fp32", "fp32x3", "bf16"), 16)
        fp = sub_record("hanoi5_65536games_x100sims in fp32 parity mode (configs[2] workload)", N_DISKS, args.games, S, ALPHA, 1.0, (),
                        ("fp32", "fp32x3"), 16)
        # the parity mode's number is the tensor-core kernel's (HMZ_MODE_FP32X3, same 1e-5 gate); the FFMA kernel's stays beside it
        sub["fp32_mode"] = {"value": fp["fp32x3"]["value"], "unit": UNIT, "ms_per_step": fp["fp32x3"]["ms_per_step"],
                            "kernel": "net_x3_recurrent (tcgen05, every float32 operand as three bf16 parts, fp32 accumulate)",
                            "step": "one move of every game", "mean_leaf_depth": fp["fp32x3"]["mean_leaf_depth"],
                            "ffma_kernel": {"value": fp["fp32"]["value"], "ms_per_step": fp["fp32"]["ms_per_step"]},
                            "accuracy": network_accuracy(net, N_DISKS, dev)}

    # ---- §8f rows (episode post-processing, replay ring, acting harness): measured only on request
    extras = None
    if args.extras and rank == 0:
        extras = measure_extras(dev, weights, peaks, timed)

    if rank == 0:
        line = {
            "metric": METRIC, "value": sims_per_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms / args.steps, "ms_per_move": ms / moves, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "bf16" if args.mode == "bf16" else "f32",
            "data": "synthetic", "config": workload_config(args, world, args.mode, args.schedule), "clocks": clocks,
            "e2e": {"value": e2e_rate, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "roofline": roofline, "roofline_second_kernel": roofline_other, "kernels": kern,
            "mean_leaf_depth": depth, "env_steps_per_second": world * B * moves / (ms * 1e-3), "env": env_line,
            "build_flags": flags, "targets": {"sims_per_s_8gpu": 1e8, "env_steps_per_s_8gpu": 1e9},
        }
        if weak is not None:
            line["weak"] = weak
        if sub is not None:
            line["configs"] = sub
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if extras is not None:
            line["extras"] = extras
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure_extras(dev, weights, peaks, timed):
    """SURVEY §8f rows 1-3 at BASELINE sizes: episode post-processing kernels, replay-ring insertion and the
    batched acting-evaluation harness.  Synthetic finished episodes (random lengths, flags, visit counts)."""
    import numpy as np
    import torch

    from muzero_hanoi_b200 import _lib, acting
    from muzero_hanoi_b200.engine import PackedWeights
    from muzero_hanoi_b200.learner import Learner
    from muzero_hanoi_b200.networks import MuZeroNet
    from muzero_hanoi_b200.replay import EpisodeStore, ReplayRing

    B, T, n = GLOBAL_GAMES, MAX_STEPS, N_DISKS
    st = EpisodeStore(B, T, n, dev)
    g = torch.Generator(device=dev).manual_seed(0)
    st.ep_len.copy_(torch.randint(1, T + 1, (B,), generator=g, device=dev, dtype=torch.int32))
    st.flags.copy_((torch.rand(T, B, generator=g, device=dev) < 0.25).to(torch.uint8) * 2)
    last = (st.ep_len.long() - 1).clamp(min=0)
    st.flags[last, torch.arange(B, device=dev)] = 5  # every episode ends solved: all of them enter the ring
    st.root_q.copy_(torch.randn(T, B, generator=g, device=dev, dtype=torch.float64) * 20)
    st.visits.copy_(torch.randint(1, 40, (T, B, 6), generator=g, device=dev, dtype=torch.int16))
    st.state.copy_(torch.randint(0, 1 << (2 * n), (T, B), generator=g, device=dev, dtype=torch.int32))
    steps = int(st.ep_len.sum().item())
    ms_ret = timed(lambda: st.post_process(10, DISCOUNT), 10) / 10
    ms_mc = timed(lambda: st.post_process_mc(DISCOUNT), 10) / 10
    ring = ReplayRing(steps + 1024, 5, 3 * n, 6, dev)

    def add():
        ring.ptr, ring.is_full = 0, False
        ring.add_episodes(st, temperature=TEMPERATURE, only_solved=True)
    add()
    ms_add = timed(add, 5) / 5
    row_bytes = 4 * 3 * n + 5 * 4 + 5 * 8 + 5 * 6 * 4 + 5 * 4 + 4
    out = {"episodes": B, "transitions": steps, "t_max": T,
           "n_step_returns": {"ms": ms_ret, "transitions_per_s": steps / (ms_ret * 1e-3),
                              "gbs": steps * 21 / (ms_ret * 1e-3) / 1e9, "algorithmic": "21 B / transition (flags 1, root_q 8, return 8, priority 4)"},
           "mc_returns": {"ms": ms_mc, "transitions_per_s": steps / (ms_mc * 1e-3)},
           "replay_add": {"ms": ms_add, "rows_per_s": steps / (ms_add * 1e-3), "gbs": steps * (row_bytes + 30) / (ms_add * 1e-3) / 1e9,
                          "frac_of_hbm": steps * (row_bytes + 30) / (ms_add * 1e-3) / 1e9 / peaks["hbm_gbs"],
                          "algorithmic": f"{row_bytes} B row written + 30 B episode record read per transition; includes the "
                                         "row-assignment scan and one scalar read-back"}}
    # acting harness at BASELINE.json configs[4] semantics (N=4, random starts, S=200, T=0)
    n4, eps, sims = 4, 16384, 200
    torch.manual_seed(2)
    net4 = acting.ablate_networks(True, True, True, MuZeroNet(3 * n4, 6, 0.002, "cpu", TD_return=True))
    w4 = PackedWeights(net4.state_dict(), n4, _lib.MODE_BF16, dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, det = acting.get_results(w4, n4, MAX_STEPS, eps, [sims], 0.0, seed=1, return_details=True)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    moves = int(det[0]["steps"].max())
    # learner step (Muzero._update + Adam) at the reference's default batch (TrainingConfig: batch 256, unroll 5)
    Bl, Kl = 256, 5
    rng = np.random.default_rng(3)
    torch.manual_seed(3)
    netl = MuZeroNet(3 * n, 6, 0.002, "cpu", TD_return=True)
    sd = {k: v.detach().numpy().copy() for k, v in netl.state_dict().items()}
    idx = rng.integers(0, 3 ** n, Bl)
    onehot = np.zeros((Bl, 3 * n), np.float32)
    for i, s_idx in enumerate(idx):
        for d in range(n - 1, -1, -1):
            onehot[i, 3 * d + s_idx % 3] = 1.0
            s_idx //= 3
    batch = (onehot, rng.choice(np.array([0.0, 100.0, -0.1], np.float32), size=(Bl, Kl)).astype(np.float32),
             rng.integers(0, 6, (Bl, Kl)).astype(np.int64), rng.dirichlet(np.ones(6), size=(Bl, Kl)).astype(np.float32),
             rng.normal(0, 20, (Bl, Kl)).astype(np.float32), rng.uniform(0.2, 1.0, Bl).astype(np.float32))
    ln = Learner(sd, n, Kl, device=dev)
    dbatch = [torch.as_tensor(x, device=dev) for x in batch]
    ln.update(*dbatch)
    ms_upd = timed(lambda: ln.update(*dbatch), 20) / 20
    out["learner_step"] = {"workload": f"Muzero._update batch {Bl} x unroll {Kl}, N={n} (TrainingConfig defaults)", "ms": ms_upd,
                           "updates_per_s": 1e3 / ms_upd, "note": "includes the host-side loss read-back of every update"}
    out["acting_harness"] = {"workload": f"hanoi{n4}_{eps}episodes_x{sims}sims_T0, all three heads lesioned (BASELINE.json configs[4])",
                             "wall_s": wall, "moves_played": moves, "sims_per_s": eps * sims * moves / wall,
                             "mean_error": float(det[0]["errors"].mean()), "episodes_per_s": eps / wall}
    return out


def main():
    global MOVES_PER_STEP
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--mode", choices=["bf16", "fp32", "fp32x3"], default=os.environ.get("HMZ_BENCH_MODE", "bf16"))
    ap.add_argument("--games", type=int, default=GLOBAL_GAMES, help="GLOBAL number of games (sharded over the ranks)")
    ap.add_argument("--sims", type=int, default=N_SIMS)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-env", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[1] / configs[4] / fp32-mode sub-records")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the secondary fixed-games-per-GPU record")
    ap.add_argument("--extras", action="store_true", help="also time the SURVEY §8f rows (episode kernels, replay ring, acting harness)")
    ap.add_argument("--moves-per-step", type=int, default=MOVES_PER_STEP, help="moves of every game per timed step (profiling runs use 1)")
    ap.add_argument("--schedule", default=os.environ.get("HMZ_BENCH_SCHEDULE", "auto"),
                    help="hmz_search_t.schedule: auto | persistent | server | k (stream groups, 1..16; 128 + k = server with k tree groups)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (move records, env words) as DIR/<name>.npy, at most 64 MB (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    MOVES_PER_STEP = max(1, args.moves_per_step)
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
