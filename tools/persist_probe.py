"""Timing probe of hmz_search_run's schedules on the self-play move (tooling): ms per move for a list of schedules, and the
persistent kernel's role statistics when the loaded library is the HMZ_PERSIST_STATS variant (HMZ_LIB_PATH) and
HMZ_PERSIST_STATS=1.   B=65536 S=100 SCHEDULES=64,0,1 MOVES=12 python tools/persist_probe.py"""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from muzero_hanoi_b200 import _lib
from muzero_hanoi_b200.engine import PackedWeights, SelfPlay
from muzero_hanoi_b200.networks import MuZeroNet

B, S, n = int(os.environ.get("B", 65536)), int(os.environ.get("S", 100)), int(os.environ.get("N", 5))
moves = int(os.environ.get("MOVES", 12))
lib = _lib.load()
torch.manual_seed(0)
MODE = int(os.environ.get("MODE", _lib.MODE_BF16))  # 0: float32 FFMA, 1: bf16 tcgen05, 2: float32 accuracy on tcgen05
LDT = _lib.LATENT_BF16 if MODE == _lib.MODE_BF16 else _lib.LATENT_F32
w = PackedWeights(MuZeroNet(3 * n, 6, 0.002, "cpu", TD_return=True).state_dict(), n, MODE)
for sched in [int(x) for x in os.environ.get("SCHEDULES", "64").split(",")]:
    sp = SelfPlay(n, 200, B, S, w, seed=1, ring_slots=4, latent_dtype=LDT)
    sp.mcts.store.set_schedule(sched)
    for _ in range(4):
        sp.move()
    torch.cuda.synchronize()
    if os.environ.get("SKIP"):  # time one kernel family alone (HMZ_DEBUG_SKIP, read by the library at every call)
        os.environ["HMZ_DEBUG_SKIP"] = os.environ["SKIP"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(moves):
        sp.move()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / moves
    line = f"B={B} S={S} mode={MODE} schedule={sched}: {ms:.3f} ms/move, {B * S / ms / 1e6:.1f} M sims/s, {ms / S * 1e3:.2f} us/round"
    if sched == 64 and os.environ.get("HMZ_PERSIST_STATS"):
        buf = (C.c_ulonglong * 16)()
        _lib.check(lib.hmz_debug_persist_stats(buf))
        st = list(buf)
        warps, items = max(1, st[7]), max(1, st[2])
        passes = max(1, st[6])
        line += (f"\n    tree: {warps} warps, {items} slices; per warp: wait {st[0] / warps / 1.965e3:.0f} us, work {st[1] / warps / 1.965e3:.0f} us, "
                 f"life {st[3] / warps / 1.965e3:.0f} us; work per slice {st[1] / items / 1.965e3:.2f} us"
                 f"\n    mlp: {passes} passes; waiting for the tree {st[4] / passes / 1.965e3:.2f} us per pass; first->last hand-off per CTA {st[5] / 1.965e3:.0f} us summed over CTAs")
    print(line, flush=True)
    os.environ.pop("HMZ_DEBUG_SKIP", None)
    del sp
