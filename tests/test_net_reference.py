"""MuZeroNet inference kernels against a float64 reference of the same operation, at the batch sizes where their launch
paths change and at the size bench.py runs.

The reference (``recurrent`` / ``initial`` below) is batched torch float64: cuBLAS DGEMM on the GPU, in chunks of at
most 65,536 rows, or the CPU for the CPU tests.  It never calls libhmz.  Its semantics are those of oracle/port.py:PortNet
(networks.py:71-196): the 33-bin support expectation and the signed parabolic, normalize_h_state with its +1e-8, and a
reward head that reads the raw (un-normalised) latent.

``emulate_bf16=True`` rounds exactly where net_tc (HMZ_MODE_BF16, hmz_net_tc.cu / hmz_net_tc.cuh) rounds, each time
float64 -> float32 -> bf16 with round-to-nearest-even (the host f2bf of the packer, cvt.rn.bf16x2 on the device):
  * every weight, including the six one-hot action columns of dynamic_net.0 and every bias (biases ride in the extra
    K = 16 slice of each weight block as bf16 and multiply a constant 1.0);
  * the input latent (a no-op for bf16 latents);
  * each hidden layer, after the ReLU;
  * the raw latent before the reward head;
  * the normalised latent before the value and policy heads (and before a bf16 store).
Accumulation, the softmaxes and the support transform stay float64.

Gates.  HMZ_MODE_FP32 (FFMA) and HMZ_MODE_FP32X3 are held to the 1e-5 gates of test_net_gpu.py against the plain
reference.  HMZ_MODE_BF16 is held to the emulated reference (statistics e = (kernel - ref) / max(1, |ref|) for r and v,
e = kernel - ref for p and float32-stored h):
  * bf16 latent stores: at least 99.98 % of elements bit-identical to the reference's rounded latent, none more than
    one bf16 ulp plus 1.5e-3 away;
  * 99.9th percentile of |e| (batches of 1,000 rows or more);
  * mean signed e (batches of 10,000 rows or more): a kernel that rounds the wrong way is biased;
  * maximum |e| and, against the plain reference, the 2e-2 gate the mode has always had (except for saturated heads).
The 1e-5 gates compare against a float64 reference here, not the reference network's float32 outputs, so the r / v
floor follows the float32 grid of the signed parabolic, which widens with |v| (see _fp32_failures).
The gate values and what a faithful kernel achieves are given at BF16_GATES."""
import math
from typing import Callable, NamedTuple

import numpy as np
import pytest
import torch

from conftest import record_metric
from oracle import port

CHUNK = 65536
LATENT, ACTIONS, SUPPORT = 64, 6, 33


# ============================================================================ the reference
def bf16_rne(x):
    """float64 -> float32 -> bf16 (round to nearest, ties to even) -> float64."""
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def bf16_trunc(x):
    """float64 -> float32 -> bf16 by truncation (a wrong contract: the sharpness test's mutations)."""
    return (x.to(torch.float32).view(torch.int32) & -65536).view(torch.float32).to(torch.float64)


class Rounding(NamedTuple):
    """Where the bf16 contract rounds and how; FAITHFUL is net_tc's.  The other forms exist only to show that the gates
    reject a kernel that rounds differently."""
    hidden: Callable = bf16_rne
    latent_in: Callable = bf16_rne
    bf16_bias: bool = True


FAITHFUL = Rounding()


def _prepare(sd, emulate, device, rounding):
    W = {}
    for k, t in sd.items():
        t = t.detach() if torch.is_tensor(t) else torch.from_numpy(np.asarray(t))
        t = t.to(device=device, dtype=torch.float64)
        if emulate and (k.endswith("weight") or rounding.bf16_bias):
            t = bf16_rne(t)
        W[k] = t
    return W


def _layer1(W, name, x, extra=None):
    w = W[f"{name}.0.weight"]
    pre = x @ w[:, : x.shape[1]].T + W[f"{name}.0.bias"]
    return torch.relu(pre if extra is None else pre + extra)


def _mlp(W, name, x, hidden_round, extra=None):
    h = _layer1(W, name, x, extra)
    if hidden_round is not None:
        h = hidden_round(h)
    return h @ W[f"{name}.2.weight"].T + W[f"{name}.2.bias"]


def _support_to_scalar(logits, eps=1e-3):
    """networks.py:152-189 in float64: softmax -> expectation over linspace(-16, 16, 33) -> signed parabolic."""
    half = (SUPPORT - 1) // 2
    x = torch.softmax(logits, dim=-1) @ torch.arange(-half, half + 1, dtype=torch.float64, device=logits.device)
    z = torch.sqrt(1 + 4 * eps * (eps + 1 + x.abs())) / 2 / eps - 1 / 2 / eps
    return torch.sign(x) * (z * z - 1)


def _normalize(h):
    lo, hi = h.min(dim=-1, keepdim=True)[0], h.max(dim=-1, keepdim=True)[0]
    return (h - lo) / (hi - lo + 1e-8)


def _prediction(W, hn, emulate, hid):
    x = bf16_rne(hn) if emulate else hn
    p = torch.softmax(_mlp(W, "policy_net", x, hid), dim=-1)
    return p, _support_to_scalar(_mlp(W, "value_net", x, hid))


def recurrent(sd, h_in, actions, emulate_bf16, *, device=None, rounding=FAITHFUL):
    """recurrent_inference of a batch -> (h normalised, r, p, v), float64 on ``device`` (default: h_in's device)."""
    h_in, actions = torch.as_tensor(h_in), torch.as_tensor(actions)
    dev = torch.device(device) if device is not None else h_in.device
    W = _prepare(sd, emulate_bf16, dev, rounding)
    hid = rounding.hidden if emulate_bf16 else None
    act_cols = W["dynamic_net.0.weight"][:, LATENT:].T.contiguous()  # [6, 256]: the one-hot action columns
    out = []
    for lo in range(0, h_in.shape[0], CHUNK):
        x = h_in[lo:lo + CHUNK].to(dev, torch.float64)
        if emulate_bf16:
            x = rounding.latent_in(x)
        a = actions[lo:lo + CHUNK].to(dev, torch.long)
        raw = _mlp(W, "dynamic_net", x, hid, extra=act_cols[a])
        hn = _normalize(raw)
        r = _support_to_scalar(_mlp(W, "rwd_net", bf16_rne(raw) if emulate_bf16 else raw, hid))
        p, v = _prediction(W, hn, emulate_bf16, hid)
        out.append((hn, r, p, v))
    return tuple(torch.cat(t) for t in zip(*out))


def onehot_of_words(words, n):
    """utils.oneHot_encoding of packed env words (2 bits per disk, disk 0 lowest): float64 [B, 3n]."""
    w = torch.as_tensor(words).to(torch.int64)
    pegs = (w[:, None] >> (2 * torch.arange(n, device=w.device))) & 3
    return torch.nn.functional.one_hot(pegs, 3).reshape(w.shape[0], 3 * n).to(torch.float64)


def initial(sd, words_or_onehot, n, emulate_bf16, *, device=None, rounding=FAITHFUL):
    """initial_inference of a batch from packed env words (1-D integer) or observations [B, 3n] -> (h, p, v)."""
    x = torch.as_tensor(words_or_onehot)
    dev = torch.device(device) if device is not None else x.device
    x = x.to(dev)
    obs = onehot_of_words(x, n) if not x.is_floating_point() else x.to(torch.float64)
    assert obs.shape[1] == 3 * n
    W = _prepare(sd, emulate_bf16, dev, rounding)
    hid = rounding.hidden if emulate_bf16 else None
    out = []
    for lo in range(0, obs.shape[0], CHUNK):
        hn = _normalize(_mlp(W, "representation_net", obs[lo:lo + CHUNK], hid))
        p, v = _prediction(W, hn, emulate_bf16, hid)
        out.append((hn, p, v))
    return tuple(torch.cat(t) for t in zip(*out))


# ================================================================================= gates
# HMZ_MODE_FP32 / HMZ_MODE_FP32X3 against the plain reference (test_net_gpu.py, with the reasons for the floors there)
REL, H_ABS, P_ABS, RV_ABS = 1e-5, 1e-6, 1e-7, 2.5e-4
BF16_HALF_ULP = 2.0 ** -8  # largest relative rounding error of a bf16 store (8 significant bits)

# HMZ_MODE_BF16 against the emulated reference: each gate is about 3x the worst value the kernel reached over every case
# of this file on a B200 (1,000 W; the batches of 1,000 rows or more for the percentiles and 10,000 or more for the
# means; saturated heads included).  Measured / gate:
#   bit-identical bf16 latents      >= 0.99993 / 0.9998   (with any of the three mutations of the sharpness test: ~0.72)
#   |kernel - ref| - ulp(ref)       4.9e-4 / 1.5e-3  (one ulp does not bound every element: where a hidden unit's float32
#                                   sum lies within its accumulation error of a bf16 rounding midpoint, the kernel and the
#                                   reference round it differently, which moves the raw latent by ~1e-4 absolute; near 0,
#                                   where a bf16 ulp is tiny, that is up to 171 ulps)
#   p99.9 |e|  h (float32 store) 2.2e-7 / 6.5e-7, p 4.5e-5 / 1.35e-4, r 5.9e-4 / 1.8e-3, v 1.05e-3 / 3.2e-3
#   |mean e|   h 3.1e-8 / 1e-7, r 6.0e-5 / 1.8e-4, v 6.0e-5 / 1.8e-4  (r / v: mostly the float32 constants of the kernel's
#                                   signed parabolic — 0.001f is not 1e-3 — which the float64 reference does not share)
#   max |e|    r 3.8e-3, p 3.8e-4, v 1.3e-2 (saturated heads), h 9.3e-4 / 2e-2
#   plain reference, max: 1.2e-2 / 2e-2 — except saturated heads, where bf16 rounding itself moves v by 3.7e-2 of
#                                   max(1, |v|) (the emulated reference follows the kernel there: p99.9 1.05e-3)
BF16_GATES = dict(
    h_identical=0.9998,  # fraction of bf16 latent elements bit-identical
    h_excess=1.5e-3,     # largest |kernel - ref| - ulp(ref) of a bf16 latent element
    h_q=6.5e-7, p_q=1.35e-4, r_q=1.8e-3, v_q=3.2e-3,  # 99.9th percentile of |e|
    h_mean=1e-7, r_mean=1.8e-4, v_mean=1.8e-4,        # |mean signed e| (not for p: a row's errors of p sum to 0)
    max=2e-2,            # backstop on max |e| (and the plain-reference gate)
)
Q_MIN_ROWS, MEAN_MIN_ROWS = 1000, 10000


def _bf16_ordered(t):
    """bf16 tensor -> int32 keys whose difference counts bf16 ulps (sign-magnitude to two's complement)."""
    b = t.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(b < 0, -(b & 0x7FFF), b)


class Bf16Errors:
    """Error statistics of HMZ_MODE_BF16 outputs against the emulated reference, accumulated over chunks of rows."""

    def __init__(self):
        self.rows = 0
        self.h_n = self.h_same = self.h_ulp = 0
        self.h_excess = 0.0
        self.e = {"h": [], "p": [], "r": [], "v": []}
        self.plain = 0.0

    def add(self, h, r, p, v, ref, plain=None):
        """h: the kernel's stored latents (bf16 or float32), r / p / v float32; ref / plain: (h, r, p, v) float64."""
        self.rows += r.shape[0]
        if h.dtype == torch.bfloat16:
            want = ref[0].to(torch.float32).to(torch.bfloat16)
            d = (_bf16_ordered(h) - _bf16_ordered(want)).abs()
            self.h_n += d.numel()
            self.h_same += int((d == 0).sum())
            self.h_ulp = max(self.h_ulp, int(d.max()))
            want = want.double()
            ulp = torch.ldexp(torch.ones_like(want), torch.frexp(want)[1] - 8) * (want != 0)
            self.h_excess = max(self.h_excess, float(((h.double() - want).abs() - ulp).max()))
        else:
            self.e["h"].append((h.double() - ref[0]).flatten())
        self.e["p"].append((p.double() - ref[2]).flatten())
        for key, got, want in (("r", r, ref[1]), ("v", v, ref[3])):
            self.e[key].append((got.double() - want) / want.abs().clamp(min=1.0))
        if plain is not None:
            for got, want, rel in ((h, plain[0], False), (r, plain[1], True), (p, plain[2], False), (v, plain[3], True)):
                d = (got.double() - want).abs()
                self.plain = max(self.plain, float((d / want.abs().clamp(min=1.0) if rel else d).max()))

    def stats(self):
        s = {"rows": self.rows, "plain_max": self.plain}
        if self.h_n:
            s.update(h_identical=self.h_same / self.h_n, h_ulp=self.h_ulp, h_excess=self.h_excess)
        for key, parts in self.e.items():
            if not parts:
                continue
            e = torch.cat(parts)
            a = e.abs()
            k = max(1, math.ceil(0.999 * a.numel()))
            s.update({f"{key}_q": float(a.kthvalue(k).values), f"{key}_max": float(a.max()), f"{key}_mean": float(e.mean())})
        return s


def bf16_failures(s, gates=BF16_GATES, plain=True):
    """The gates a set of statistics (Bf16Errors.stats) fails, as readable strings; [] = accepted.  plain=False leaves
    out the 2e-2 gate against the plain reference (saturated heads, see BF16_GATES)."""
    bad = []
    if "h_identical" in s:
        if s["h_identical"] < gates["h_identical"]:
            bad.append(f"bit-identical latents {s['h_identical']:.5f} < {gates['h_identical']}")
        if s["h_excess"] > gates["h_excess"]:
            bad.append(f"a latent element {s['h_excess']:.3g} beyond one bf16 ulp (> {gates['h_excess']})")
    for key in ("h", "p", "r", "v"):
        if f"{key}_max" not in s:
            continue
        if s[f"{key}_max"] > gates["max"]:
            bad.append(f"max |e_{key}| {s[f'{key}_max']:.3g} > {gates['max']}")
        if s["rows"] >= Q_MIN_ROWS and s[f"{key}_q"] > gates[f"{key}_q"]:
            bad.append(f"p99.9 |e_{key}| {s[f'{key}_q']:.3g} > {gates[f'{key}_q']}")
        if s["rows"] >= MEAN_MIN_ROWS and f"{key}_mean" in gates and abs(s[f"{key}_mean"]) > gates[f"{key}_mean"]:
            bad.append(f"mean e_{key} {s[f'{key}_mean']:.3g} beyond +-{gates[f'{key}_mean']}")
    if plain and s["plain_max"] > gates["max"]:
        bad.append(f"{s['plain_max']:.3g} from the plain reference > {gates['max']}")
    return bad


def _fp32_failures(h, r, p, v, ref, rec):
    """HMZ_MODE_FP32 / FP32X3 against the plain reference at the 1e-5 gates; a bf16 latent store may add its own
    rounding (half a bf16 ulp).  The achieved maxima are accumulated into ``rec``."""
    bad = []
    h_abs = H_ABS + (BF16_HALF_ULP * ref[0].abs() if h.dtype == torch.bfloat16 else 0.0)
    # r / v: two steps of the float32 grid of the signed parabolic (z = sqrt(..) / 2 / eps - 500, v = z^2 - 1), which the
    # reference network and the kernels evaluate in float32 and this reference in float64: 2.5e-4 at v = 0, growing as
    # dv / dz = 2z = 2 sqrt(1 + |v|) (measured: 3.1e-4 at v = -3.0, where the plain 2.5e-4 floor allows 2.8e-4)
    for key, got, want, floor in (("h", h, ref[0], h_abs), ("p", p, ref[2], P_ABS),
                                  ("r", r, ref[1], RV_ABS * (1 + ref[1].abs()).sqrt()),
                                  ("v", v, ref[3], RV_ABS * (1 + ref[3].abs()).sqrt())):
        d = (got.double() - want).abs()
        excess = d - (REL * want.abs() + floor)
        rec[f"{key}_abs"] = max(rec.get(f"{key}_abs", 0.0), float(d.max()))
        if bool((excess > 0).any()):
            i = int(excess.flatten().argmax())
            bad.append(f"{key}: {int((excess > 0).sum())} elements beyond the 1e-5 gate, worst |d| {float(d.flatten()[i]):.3g} "
                       f"at flat index {i} (ref {float(want.flatten()[i]):.6g})")
    return bad


# ============================================================================ CPU tests
def _close(got, ref, atol):
    return bool(np.all(np.abs(got - ref) <= REL * np.abs(ref) + atol))


@pytest.mark.parametrize("n", [3, 5, 10])
def test_reference_reproduces_the_recorded_network_outputs(golden, n):
    """The plain float64 reference against the outputs recorded from the unmodified reference network
    (tests/golden/net_io.npz), at the 1e-5 gates of test_net_gpu.py: both inference forms, words and one-hot input."""
    g = golden("net_io.npz")
    sd = port.make_weights(n, int(g[f"n{n}_weight_seed"]))
    h, r, p, v = (t.numpy() for t in recurrent(sd, torch.from_numpy(g[f"n{n}_h_in"]), torch.from_numpy(g[f"n{n}_action"]), False))
    assert _close(h, g[f"n{n}_h_out"], H_ABS) and _close(p, g[f"n{n}_p"], P_ABS)
    assert _close(r, g[f"n{n}_r"], RV_ABS) and _close(v, g[f"n{n}_v"], RV_ABS)
    states = [port.index_to_state(int(i), n) for i in g[f"n{n}_state_idx"]]
    words = torch.tensor([port.state_to_packed(s) for s in states], dtype=torch.int32)
    obs = torch.from_numpy(np.stack([port.one_hot(s) for s in states]))
    assert torch.equal(onehot_of_words(words, n), obs)
    for x in (words, obs):
        h0, p0, v0 = (t.numpy() for t in initial(sd, x, n, False))
        assert _close(h0, g[f"n{n}_h0"], H_ABS) and _close(p0, g[f"n{n}_p0"], P_ABS) and _close(v0, g[f"n{n}_v0"], RV_ABS)


def test_emulation_rounds_where_the_contract_says():
    """The emulated reference differs from the plain one by bf16 rounding only: a batch whose every rounded quantity
    is already a bf16 value gives the same outputs in both forms."""
    sd = port.make_weights(3, 2)
    sd = {k: bf16_rne(torch.from_numpy(v).double()).numpy() for k, v in sd.items()}
    sd["dynamic_net.2.weight"][:] = 0.0  # raw latent = the (bf16) bias; hidden units of the heads then see bf16 inputs
    sd["dynamic_net.2.bias"][:] = 0.5  # raw latent 0.5 everywhere, normalised latent exactly 0
    for k in ("rwd_net", "policy_net", "value_net"):
        sd[f"{k}.0.weight"][:] = np.round(sd[f"{k}.0.weight"] * 8) / 8  # hidden sums on a coarse grid: exact in bf16
        sd[f"{k}.0.bias"][:] = 0.25
    h = bf16_rne(torch.rand(40, LATENT, dtype=torch.float64))
    a = torch.arange(40) % ACTIONS
    emu, plain = recurrent(sd, h, a, True), recurrent(sd, h, a, False)
    for x, y in zip(emu, plain):
        assert torch.equal(x, y)
    # and on random weights the two differ, by bf16-sized amounts
    sd = port.make_weights(3, 2)
    emu, plain = recurrent(sd, h, a, True), recurrent(sd, h, a, False)
    d = [float((x - y).abs().max()) for x, y in zip(emu, plain)]
    assert all(0 < e < 2e-2 for e in d), d


# ---- the HMZ_MODE_BF16 weight section, decoded on the host (layout: hmz_net_tc.cuh:13-33)
def _w_bytes(n_out, k_atoms):
    return n_out * 128 * k_atoms + n_out * 32


K_WG1, K_WG2, K_WR1, K_WR2 = 0, 40960, 75776, 116736
K_WP1 = 142848 + 1024 - 512
K_WP2 = K_WP1 + 40960
K_WV1 = K_WP2 + 9216
K_WV2 = K_WV1 + 40960
K_WH1 = K_WV2 + 26112 + 512
K_WH2 = K_WH1 + 40960
K_SECTION = K_WH2 + 34816
# block offset -> (state_dict layer, rows padded to, K-atoms, extra-slice columns k = 0..5 taken from W[:, 64:70])
TC_BLOCKS = {
    K_WG1: ("dynamic_net.0", 256, 1, True), K_WG2: ("dynamic_net.2", 64, 4, False),
    K_WR1: ("rwd_net.0", 256, 1, False), K_WR2: ("rwd_net.2", 48, 4, False),
    K_WP1: ("policy_net.0", 256, 1, False), K_WP2: ("policy_net.2", 16, 4, False),
    K_WV1: ("value_net.0", 256, 1, False), K_WV2: ("value_net.2", 48, 4, False),
    K_WH1: ("representation_net.0", 256, 1, False), K_WH2: ("representation_net.2", 64, 4, False),
}


def _plain_off(row, c):
    return (row >> 3) * 256 + c * 128 + (row & 7) * 16


def _decode_tc_block(u16, covered, off, n_pad, k_atoms):
    """-> (main [n_pad][64 k_atoms], extra [n_pad][16]) uint16 bf16 bits of one block; marks the halfwords read."""
    n = np.arange(n_pad)[:, None, None]
    c = np.arange(8)[None, :, None]
    j = np.arange(8)[None, None, :]
    atoms = []
    for ka in range(k_atoms):  # SWIZZLE_128B K-atom: 16-byte chunk c of row n at n * 128 + ((c ^ (n & 7)) << 4)
        idx = (off + ka * n_pad * 128 + n * 128 + ((c ^ (n & 7)) << 4)) // 2 + j
        atoms.append(u16[idx].reshape(n_pad, 64))
        covered[idx] = True
    x0 = off + n_pad * 128 * k_atoms  # core-matrix K = 16 slice: 8 rows x 16 B, the two K chunks 128 B apart
    c2 = np.arange(2)[None, :, None]
    idx = (x0 + (n >> 3) * 256 + c2 * 128 + (n & 7) * 16) // 2 + j
    covered[idx] = True
    return np.concatenate(atoms, axis=1), u16[idx].reshape(n_pad, 16)


def _bits(x):
    """bf16 bits of the reference's rounding of a float32 array."""
    return bf16_rne(torch.from_numpy(np.asarray(x, np.float32)).double()).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


@pytest.mark.parametrize("n", [1, 5, 12])  # 3N = 3 .. 36 observation columns of representation_net.0
def test_bf16_section_holds_what_the_reference_multiplies(lib, n):
    """hmz_weights_pack(HMZ_MODE_BF16) decoded through the layout net_tc's descriptors read (block offsets kWg1 .. kWh2,
    SWIZZLE_128B K-atoms, the extra K = 16 slice with the action columns at k = 0..5 and the bias at k = 6): every bf16
    value equals the emulated reference's bf16_rne(w) bit for bit, and every padding row, column and gap is zero."""
    import ctypes as C

    from muzero_hanoi_b200.engine import STATE_DICT_ORDER

    sd = port.make_weights(n, 40 + n)
    sd["policy_net.2.bias"][0] = 1.0 + 2.0 ** -8  # an exact tie: even rounding gives 1.0, not 1.0078125
    sd["rwd_net.2.weight"][1, 2] = -(1.0 + 3 * 2.0 ** -8)  # a tie that rounds away from zero
    arrays = [np.ascontiguousarray(sd[k], dtype=np.float32) for k in STATE_DICT_ORDER]
    nbytes = int(lib.hmz_weights_packed_bytes(n, 1))
    fp32_off = (K_SECTION + 1023) // 1024 * 1024
    assert nbytes > fp32_off
    host = np.full(nbytes, 0xA5, np.uint8)
    table = (C.c_void_p * 20)(*[a.ctypes.data for a in arrays])
    assert lib.hmz_weights_pack(table, n, 1, host.ctypes.data) == 0
    u16 = host[:fp32_off].view(np.uint16)
    covered = np.zeros(u16.shape, bool)
    for off, (layer, n_pad, k_atoms, action_cols) in TC_BLOCKS.items():
        assert off % 1024 == 0 and off + _w_bytes(n_pad, k_atoms) <= K_SECTION
        main, extra = _decode_tc_block(u16, covered, off, n_pad, k_atoms)
        w, b = sd[f"{layer}.weight"], sd[f"{layer}.bias"]
        n_out, k_in = w.shape[0], min(w.shape[1], 64 * k_atoms)
        want = np.zeros((n_pad, 64 * k_atoms), np.uint16)
        want[:n_out, :k_in] = _bits(w[:, :k_in])
        assert np.array_equal(main, want), layer
        want = np.zeros((n_pad, 16), np.uint16)
        if action_cols:
            want[:n_out, :ACTIONS] = _bits(w[:, LATENT:LATENT + ACTIONS])
        want[:n_out, 6] = _bits(b)
        assert np.array_equal(extra, want), layer
    assert covered.sum() * 2 == sum(_w_bytes(p, k) for _, p, k, _ in TC_BLOCKS.values())  # blocks do not overlap
    assert not u16[~covered].any()  # gaps between blocks and the tail of the section
    assert _bits(np.float32(1.0 + 2.0 ** -8)) == 0x3F80 and _bits(np.float32(-(1.0 + 3 * 2.0 ** -8))) == 0xBF82


# ============================================================================ GPU grid
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _count(spec):
    """Batch sizes named by the launch path they select (derived from the SM count, 148 on a B200):
    tc_split  = 256 * (SMs // 3): largest batch of net_tc's head split (three CTAs per 256-row tile pair), 12,544
    tc_pass   = 256 * SMs: largest batch with one tile pair per CTA; above it CTAs run two passes, 37,888
    x3_split  = 128 * (SMs // 3): largest batch of net_x3's head split (three CTAs per 128-row tile), 6,272
    x3_tile   = 128 * SMs: largest batch with one tile per CTA, 18,944"""
    sms = _sms()
    base = {"tc_split": 256 * (sms // 3), "tc_pass": 256 * sms, "x3_split": 128 * (sms // 3), "x3_tile": 128 * sms}
    name, _, plus = spec.partition("+")
    return (base[name] if name in base else int(name)) + (int(plus) if plus else 0)


def weight_set(name, n):
    """make: port.make_weights; torch: MuZeroNet's torch-default init (what bench.py packs); lesion: port.lesion_weights
    of the three heads; saturated: second-layer head weights x4 and +12 on one policy bias (|r|, |v| reach the steep end
    of the signed parabolic, p is nearly one-hot); flat_dyn: dynamic_net.2.weight = 0 and equal biases (the raw latent
    is constant, the normalised latent exactly 0)."""
    if name == "torch":
        from muzero_hanoi_b200.networks import MuZeroNet

        torch.manual_seed(0)
        net = MuZeroNet(3 * n, ACTIONS, 0.002, "cpu", TD_return=True)
        return {k: t.detach().numpy().copy() for k, t in net.state_dict().items()}
    sd = {k: np.array(v, copy=True) for k, v in port.make_weights(n, 7 + n).items()}
    if name == "lesion":
        sd = port.lesion_weights(sd, ("rwd_net", "policy_net", "value_net"), 3)
    elif name == "saturated":
        for k in ("rwd_net", "policy_net", "value_net"):
            sd[f"{k}.2.weight"] *= 4
        sd["policy_net.2.bias"][0] += 12
    elif name == "flat_dyn":
        sd["dynamic_net.2.weight"][:] = 0
        sd["dynamic_net.2.bias"][:] = 0.3
    else:
        assert name == "make"
    return sd


E, PAD = 3, 37  # input records per item; output rows beyond the batch


def _latents(count, seed):
    """Min-max-normalised random latents [count, E, 64] as the search produces them, every 97th selected row zero."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(count, E, LATENT, device="cuda", generator=g)
    lo, hi = x.min(-1, keepdim=True)[0], x.max(-1, keepdim=True)[0]
    return (x - lo) / (hi - lo), torch.randint(0, E, (count,), device="cuda", generator=g)


def _sentinel(shape, dtype=torch.float32):
    return torch.full(shape if isinstance(shape, tuple) else (shape,), float("nan"), dtype=dtype, device="cuda")


def run_recurrent(mode, sd, n, count, latent_dtype, seed=0):
    """One PackedWeights.recurrent call as the search makes it: inputs gathered through in_row from E records, the new
    latent scattered to record E of E + 1; every other record and PAD rows past the batch (latents and r / p / v)
    start as NaN and must come back untouched.  -> (h, r, p, v) of the batch, (gathered inputs, actions)."""
    from muzero_hanoi_b200.engine import PackedWeights

    w = PackedWeights(sd, n, mode)
    ldt = torch.bfloat16 if latent_dtype else torch.float32
    lat, in_row = _latents(count, seed)
    lat[torch.arange(0, count, 97, device="cuda"), in_row[::97]] = 0.0
    lat = lat.to(ldt)
    acts = torch.randint(0, ACTIONS, (count,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed + 1),
                         dtype=torch.uint8)
    out = _sentinel((count + PAD, E + 1, LATENT), ldt)
    r, v, p = _sentinel(count + PAD), _sentinel(count + PAD), _sentinel((count + PAD, ACTIONS))
    w.recurrent(count, latents_in=lat, in_rows_per_item=E, in_row=in_row.to(torch.int16), actions=acts, latents_out=out,
                out_rows_per_item=E + 1, out_row=E, latent_dtype=latent_dtype, r=r, p=p, v=v)
    torch.cuda.synchronize()
    assert bool(out[:, :E].isnan().all()) and bool(out[count:].isnan().all()), "latent written outside its rows"
    assert bool(r[count:].isnan().all() and v[count:].isnan().all() and p[count:].isnan().all()), "r / p / v written past the batch"
    h = out[:count, E]
    assert bool(h.isfinite().all() and r[:count].isfinite().all() and p[:count].isfinite().all() and v[:count].isfinite().all())
    return (h, r[:count], p[:count], v[:count]), (lat[torch.arange(count, device="cuda"), in_row.long()], acts)


def run_initial(mode, sd, n, count, latent_dtype, seed=0):
    """One PackedWeights.initial call from packed env words, written to record 0 of E-record items; the other records
    and PAD items past the batch must stay NaN.  -> (h, p, v), words."""
    from muzero_hanoi_b200.engine import PackedWeights, VecHanoi

    w = PackedWeights(sd, n, mode)
    env = VecHanoi(n, 200, count)
    env.random_reset(seed=seed)
    ldt = torch.bfloat16 if latent_dtype else torch.float32
    out = _sentinel((count + PAD, E, LATENT), ldt)
    p0, v0 = _sentinel((count + PAD, ACTIONS)), _sentinel(count + PAD)
    w.initial(count, words=env.words, latents_out=out, out_rows_per_item=E, latent_dtype=latent_dtype, p0=p0, v0=v0)
    torch.cuda.synchronize()
    assert bool(out[:, 1:].isnan().all()) and bool(out[count:].isnan().all()), "latent written outside its rows"
    assert bool(p0[count:].isnan().all() and v0[count:].isnan().all()), "p0 / v0 written past the batch"
    h = out[:count, 0]
    assert bool(h.isfinite().all() and p0[:count].isfinite().all() and v0[:count].isfinite().all())
    return (h, p0[:count], v0[:count]), env.words.clone()


def _check_bf16(name, got, ref, plain, gate_plain=True):
    acc = Bf16Errors()
    acc.add(*got, ref, plain)
    s = acc.stats()
    record_metric(name, s)
    bad = bf16_failures(s, plain=gate_plain)
    assert not bad, f"{name}: " + "; ".join(bad)


BF16_REC_COUNTS = ["1", "129", "255", "257", "tc_split", "tc_split+1", "tc_pass", "tc_pass+1", "65536", "65536+300"]
BF16_REC_CASES = ([(c, ldt, "make") for c in BF16_REC_COUNTS for ldt in (0, 1)]
                  + [(c, ldt, ws) for ws in ("torch", "lesion", "saturated", "flat_dyn") for c in ("257", "65536+300") for ldt in (0, 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("count,latent_dtype,wset", BF16_REC_CASES)
def test_bf16_recurrent_against_emulated_reference(count, latent_dtype, wset):
    """net_tc<recurrent> on both sides of each path change: head split (<= tc_split), one pass per CTA (<= tc_pass),
    two passes, ragged last tile and pair."""
    n, rows = 5, _count(count)
    sd = weight_set(wset, n)
    (h, r, p, v), (x, a) = run_recurrent(1, sd, n, rows, latent_dtype, seed=rows)
    _check_bf16(f"bf16_recurrent_{wset}_x{rows}_ldt{latent_dtype}", (h, r, p, v), recurrent(sd, x, a, True),
                recurrent(sd, x, a, False), gate_plain=wset != "saturated")


BF16_INIT_CASES = ([(c, ldt, 5, "make") for c in ("257", "tc_pass", "tc_pass+1", "65536+300") for ldt in (0, 1)]
                   + [("65536+300", ldt, nd, "make") for nd in (1, 12) for ldt in (0, 1)]
                   + [("65536+300", i % 2, 5, ws) for i, ws in enumerate(("torch", "lesion", "saturated"))])


@pytest.mark.gpu
@pytest.mark.parametrize("count,latent_dtype,n,wset", BF16_INIT_CASES)
def test_bf16_initial_against_emulated_reference(count, latent_dtype, n, wset):
    """net_tc<initial> from packed env words: one pass per CTA (<= tc_pass) and several; narrowest and widest one-hot."""
    rows = _count(count)
    sd = weight_set(wset, n)
    (h, p, v), words = run_initial(1, sd, n, rows, latent_dtype, seed=rows + n)
    zero = torch.zeros_like(v)
    ref, plain = initial(sd, words, n, True), initial(sd, words, n, False)
    _check_bf16(f"bf16_initial_{wset}_n{n}_x{rows}_ldt{latent_dtype}", (h, zero, p, v), (ref[0], zero.double(), ref[1], ref[2]),
                (plain[0], zero.double(), plain[1], plain[2]), gate_plain=wset != "saturated")


FP32_REC_CASES = ([(2, c, ldt, 5, "make") for c in ("x3_split", "x3_split+1", "x3_tile", "x3_tile+1", "65536+77") for ldt in (0, 1)]
                  + [(mode, "65536+77", ldt, nd, "make") for mode in (0, 2) for nd in (1, 12) for ldt in (0, 1)
                     if (mode, nd, ldt) != (2, 5, 0)]
                  + [(mode, "65536+77", 0, 5, ws) for mode in (0, 2) for ws in ("torch", "saturated", "flat_dyn")])


@pytest.mark.gpu
@pytest.mark.parametrize("mode,count,latent_dtype,n,wset", FP32_REC_CASES)
def test_fp32_modes_recurrent_against_reference(mode, count, latent_dtype, n, wset):
    """HMZ_MODE_FP32X3 (mode 2) on both sides of its head split (<= x3_split) and of one tile per CTA (<= x3_tile), and
    both parity modes at a large ragged batch: against the plain float64 reference at the 1e-5 gates."""
    rows = _count(count)
    sd = weight_set(wset, n)
    (h, r, p, v), (x, a) = run_recurrent(mode, sd, n, rows, latent_dtype, seed=rows + mode)
    rec = {}
    bad = _fp32_failures(h, r, p, v, recurrent(sd, x, a, False), rec)
    record_metric(f"mode{mode}_recurrent_{wset}_n{n}_x{rows}_ldt{latent_dtype}", rec)
    assert not bad, "; ".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("n", [1, 12])
@pytest.mark.parametrize("latent_dtype", [0, 1])
def test_fp32_modes_initial_against_reference(mode, n, latent_dtype):
    """Root inference of both parity modes from packed env words at 65,536 + 77 rows (the FFMA kernel on the float32
    copy for mode 0, the tcgen05 kernel for mode 2): against the plain float64 reference at the 1e-5 gates."""
    rows = 65536 + 77
    sd = weight_set("make", n)
    (h, p, v), words = run_initial(mode, sd, n, rows, latent_dtype, seed=n)
    ref = initial(sd, words, n, False)
    zero = torch.zeros_like(v)
    rec = {}
    bad = _fp32_failures(h, zero, p, v, (ref[0], zero.double(), ref[1], ref[2]), rec)
    record_metric(f"mode{mode}_initial_n{n}_x{rows}_ldt{latent_dtype}", rec)
    assert not bad, "; ".join(bad)


# ======================================================= sharpness of the HMZ_MODE_BF16 gate
@pytest.mark.gpu
def test_bf16_gate_rejects_a_kernel_that_rounds_differently():
    """The kernel's outputs of one grid case (bf16 recurrent, 65,536 rows, float32 latents) against references whose
    bf16 contract is wrong in one place each: the gates must reject every mutation and accept the faithful contract.
    (Nothing is injected into the kernel; only the host-side reference changes.)"""
    n, rows = 5, 65536
    sd = weight_set("make", n)
    got, (x, a) = run_recurrent(1, sd, n, rows, 0, seed=rows)
    plain = recurrent(sd, x, a, False)
    verdicts = {}
    for label, rnd in (("faithful", FAITHFUL), ("hidden_truncated", Rounding(hidden=bf16_trunc)),
                       ("input_truncated", Rounding(latent_in=bf16_trunc)), ("bias_float32", Rounding(bf16_bias=False))):
        acc = Bf16Errors()
        acc.add(*got, recurrent(sd, x, a, True, rounding=rnd), plain)
        s = acc.stats()
        verdicts[label] = bf16_failures(s)
        record_metric(f"bf16_sharpness_{label}", {**s, "rejected_by": "; ".join(verdicts[label])})
    assert verdicts.pop("faithful") == []
    for label, bad in verdicts.items():
        assert bad, f"the gates accept a reference with {label.replace('_', ' ')}"


# ============================================== every network evaluation of a full-size search
def _check_search(m, sd, n, words, cap, emulate, name, move):
    """After a move: every evaluation's input recovered from the store (parent latent row, the action that led to the
    node), its outputs (capture row, the node's latent row) against the reference; and the root inference."""
    S, B = m.n_simulations, m.B
    rec = m.store.records()
    parent = torch.from_numpy(rec["parent"].astype(np.int64)).cuda()
    action = torch.from_numpy(rec["parent_action"].astype(np.int64)).cuda()
    lat = m.store.latents
    items = torch.arange(B, device="cuda")
    acc, bad, rec = Bf16Errors(), [], {}
    for e in range(1, S + 1):
        x, a = lat[items, parent[:, e]], action[:, e]
        c = cap[e - 1]
        got = (lat[:, e], c[:, 6], c[:, :6], c[:, 7])
        if emulate:
            acc.add(*got, recurrent(sd, x, a, True), recurrent(sd, x, a, False))
        else:
            bad += [f"node {e}: {b}" for b in _fp32_failures(*got, recurrent(sd, x, a, False), rec)]
    root = (lat[:, 0], torch.zeros_like(m.v0), m.p0, m.v0)
    if emulate:
        s = acc.stats()
        record_metric(f"{name}_move{move}", s)
        bad += bf16_failures(s)
        acc = Bf16Errors()
        ref, plain = initial(sd, words, n, True), initial(sd, words, n, False)
        z = torch.zeros_like(ref[2])
        acc.add(*root, (ref[0], z, ref[1], ref[2]), (plain[0], z, plain[1], plain[2]))
        s = acc.stats()
        record_metric(f"{name}_move{move}_root", s)
        bad += [f"root: {b}" for b in bf16_failures(s)]
    else:
        record_metric(f"{name}_move{move}", rec)
        ref, rec = initial(sd, words, n, False), {}
        bad += [f"root: {b}" for b in _fp32_failures(*root, (ref[0], torch.zeros_like(ref[2]), ref[1], ref[2]), rec)]
        record_metric(f"{name}_move{move}_root", rec)
    assert not bad, f"{name} move {move}: " + "; ".join(bad[:8])


def _search_two_moves(mode, latent_dtype, schedule, B, sd, n, name):
    from muzero_hanoi_b200.engine import BatchedMCTS, PackedWeights, VecHanoi

    S = 100
    w = PackedWeights(sd, n, mode)
    env = VecHanoi(n, 200, B)
    env.random_reset(seed=6)
    rng = np.random.default_rng(17)
    m = BatchedMCTS(0.8, 0.25, S, B, latent_dtype=latent_dtype)
    m.store.set_schedule(schedule)
    cap = m.store.enable_capture(S)
    for move in range(2):
        words = env.words.clone()
        cap.fill_(float("nan"))
        action, _, _, visits = m.run_mcts(w, words=env.words, temperature=1.0, deterministic=False,
                                          noise=rng.dirichlet(np.full(6, 0.25), B), uniforms=rng.random(B))
        torch.cuda.synchronize()
        assert bool(cap.isfinite().all()) and bool((visits.sum(1) == S).all())
        _check_search(m, sd, n, words, cap, mode == 1, name, move)
        env.step(action.to(torch.uint8), want_obs=False)


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", [0, 64, 128])  # automatic (stream groups), SCHEDULE_PERSISTENT, SCHEDULE_SERVER
def test_benchmarked_search_every_evaluation_against_emulated_reference(schedule):
    """The search bench.py times, at the size it times it: HMZ_MODE_BF16 with bf16 latents, torch-default weights,
    65,536 searches x 100 simulations, two moves.  All 6.5 M recurrent evaluations of a move and its root inference are
    checked against the emulated reference at the gates of the grid above.  Unlike the oracle replay (which injects
    the captured outputs), this sees an evaluation that read its parent row or action before the tree wrote it."""
    from muzero_hanoi_b200 import _lib

    n = 5
    _search_two_moves(_lib.MODE_BF16, _lib.LATENT_BF16, schedule, 65536, weight_set("torch", n), n, f"search_bf16_sched{schedule}")


@pytest.mark.gpu
def test_fp32x3_search_every_evaluation_against_reference():
    """The same check for HMZ_MODE_FP32X3 with float32 latents at 32,768 + 300 searches x 100 simulations: every
    evaluation within the 1e-5 gates of the plain float64 reference."""
    from muzero_hanoi_b200 import _lib

    n = 5
    _search_two_moves(_lib.MODE_FP32X3, _lib.LATENT_F32, 0, 32768 + 300, weight_set("make", n), n, "search_fp32x3")
