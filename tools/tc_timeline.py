"""Prints the phase timeline (clock64 deltas, CTA 0) of one net_recurrent_tc launch.  HMZ_TC_TIMELINE=1."""
import ctypes as C, os, sys
os.environ["HMZ_TC_TIMELINE"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from muzero_hanoi_b200 import _lib
from muzero_hanoi_b200.engine import PackedWeights
from muzero_hanoi_b200.networks import MuZeroNet
torch.manual_seed(0)
n = int(os.environ.get("N", 65536))
net = MuZeroNet(15, 6, 0.002, "cpu", TD_return=True)
w = PackedWeights(net.state_dict(), 5, 1)
h_in = torch.rand(n, 64, device="cuda").to(torch.bfloat16)
acts = torch.randint(0, 6, (n,), dtype=torch.uint8, device="cuda")
h = torch.empty(n, 64, device="cuda", dtype=torch.bfloat16)
r, v, p = torch.empty(n, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, 6, device="cuda")
if os.environ.get("SERVER"):  # phase marks of one steady-state pass of MLP CTA 0 under the server schedule
    from muzero_hanoi_b200.engine import SelfPlay
    os.environ.setdefault("HMZ_TC_TIMELINE_PASS", "203")
    sp = SelfPlay(5, 200, 65536, 100, w, seed=1, ring_slots=4, latent_dtype=_lib.LATENT_BF16)
    sp.mcts.store.set_schedule(int(os.environ["SERVER"]))
    for _ in range(3):
        sp.move()
    torch.cuda.synchronize()
    READ = _lib.load().hmz_debug_persist_timeline
else:
    READ = _lib.load().hmz_debug_tc_timeline
for _ in range(0 if os.environ.get("SERVER") else 3):
    w.recurrent(n, latents_in=h_in, in_rows_per_item=1, in_row=None, actions=acts, latents_out=h, out_rows_per_item=1,
                out_row=0, latent_dtype=1, r=r, p=p, v=v)
torch.cuda.synchronize()
buf = (C.c_ulonglong * 96)()
_lib.check(READ(buf))
marks = np.array(list(buf), dtype=np.int64)
# two tiles per CTA
names = {60: "CTA: kernel entry", 61: "CTA: barriers + TMEM ready", 62: "CTA: past the PDL wait", 63: "CTA: all warps done",
         64: "T0 hid: pass start", 66: "out: pass published"}
for i, net in enumerate("grvp"):  # network order of a pass: dynamics, reward, value, policy
    for t in range(2):
        names[i * 4 + t] = f"T{t} mma {net}: L1 inputs ready"
        names[i * 4 + 2 + t] = f"T{t} mma {net}: L2 inputs ready (A1 written)"
        names[16 + i * 2 + t] = f"T{t} mma {net}: L1 issue point reached"
for t in range(2):
    names[86 + t * 8] = f"T{t} hid: raw latent published"
    names[44 + t * 8] = f"T{t} hid: saw dynamics L2 complete"
    names[40 + t * 8] = f"T{t} hid: minmax exchanged"
    names[41 + t * 8] = f"T{t} hid: hn tile written"
    names[42 + t * 8] = f"T{t} hid: hn published"
    names[43 + t * 8] = f"T{t} hid: copy-out barrier passed"
    names[80 + t * 8] = f"T{t} hid: gather done"
    for ly, nm in enumerate("grvp"):
        names[81 + t * 8 + ly] = f"T{t} hid {nm}: A1 half 0 written"
    names[85 + t * 8] = f"T{t} hid: latent done"
    for hd, nm in enumerate("rvp"):
        names[70 + hd * 2 + t] = f"T{t} out {nm}: done"
if os.environ.get("SERVER"):
    for k in (60, 61, 62, 63):
        names.pop(k, None)
t0 = min(int(marks[k]) for k in names if marks[k] != 0)
ev = sorted((int(marks[k] - t0), names[k]) for k in names if marks[k] != 0)
prev = 0
for c, nm in ev:
    print(f"{c:8d}  (+{c - prev:6d})  {nm}")
    prev = c
