"""A restatement of the learner step (Muzero._update, reference Muzero.py:209-274, + Adam of networks.py:69) in batched
torch at any precision, with autograd.  It never calls libhmz.  Run in float64 it is the reference ``hmz_learner_step``
is held to; run in float32 on the CPU it is the yardstick: the precision of the reference implementation itself.

Semantics (those of ``tests/test_learner_gpu.py::test_gradients_only_and_uniform_replay_match_torch_autograd``):
  h_0 = normalize(rep(s)), normalize(h) = (h - min) / (max - min + 1e-8) with min / max routed to their FIRST occurrence;
  per unroll step t: pi_t = pol(h_t), v_t = T(val(h_t)), h_raw = dyn([h_t, onehot(a_t)]), r_t = T(rwd(h_raw)),
  h_{t+1} = normalize(h_raw) with its incoming gradient halved;
  loss_b = sum_t (v_t - G_t)^2 + (r_t - R_t)^2 + CE(pi_t, pi*_t);  L = mean_b(w_b loss_b), gradient x 1/K;
  new priorities |v_0 - G_0|; the three reported losses are mean_b sum_t of each term, unweighted.
T is the 33-bin support expectation x = sum_i e_i (i - 16) / sum_i e_i (e_i = exp(l_i - max l)) followed by the signed
parabolic.  Forming x from the unnormalised exponentials makes it exactly 0 on all-equal logits at any precision, as
torch's float32 sum(softmax * linspace) is; there sign(x) = 0 and the row sends no gradient into that head.

``Mutant`` switches each piece of those semantics to a plausible wrong one, so that tests can show their gates reject it.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

MLPS = ("representation_net", "dynamic_net", "rwd_net", "policy_net", "value_net")
KEYS = [f"{m}.{i}.{k}" for m in MLPS for i in ("0", "2") for k in ("weight", "bias")]
SUPPORT = 33
ACTIONS = 6


@dataclass(frozen=True)
class Mutant:
    """Wrong variants of the learner step (all off = the faithful reference)."""
    hook: float = 0.5              # gradient factor on each h_{t+1} (Muzero.py:235)
    detach_minmax: bool = False    # no gradient through min / max of the normalisation
    ties_last: bool = False        # min / max routed to the last occurrence instead of the first
    rwd_on_normalised: bool = False  # reward head on normalize(h_raw) instead of h_raw
    adam_step_off: int = 0         # Adam bias corrections evaluated at step_index + this
    policy_no_tsum: bool = False   # policy gradient softmax - t instead of softmax * sum(t) - t


FAITHFUL = Mutant()


def _normalize(h, mut):
    idx = torch.arange(h.shape[-1], device=h.device)
    big = h.shape[-1]

    def pick(ext):
        eq = h == ext
        if mut.ties_last:
            return torch.where(eq, idx, -1).amax(-1, keepdim=True)
        return torch.where(eq, idx, big).amin(-1, keepdim=True)

    mn = h.gather(-1, pick(h.detach().amin(-1, keepdim=True)))
    mx = h.gather(-1, pick(h.detach().amax(-1, keepdim=True)))
    if mut.detach_minmax:
        mn, mx = mn.detach(), mx.detach()
    return (h - mn) / (mx - mn + 1e-8)


def _support_x(logits):
    support = torch.arange(SUPPORT, device=logits.device, dtype=logits.dtype) - (SUPPORT - 1) // 2
    e = torch.exp(logits - logits.detach().amax(-1, keepdim=True))
    return (e * support).sum(-1) / e.sum(-1)


def _signed_parabolic(x, eps=1e-3):
    z = torch.sqrt(1 + 4 * eps * (eps + 1 + torch.abs(x))) / 2 / eps - 1 / 2 / eps
    return torch.sign(x) * (torch.square(z) - 1)


def _mlp(P, name, x, pre_acts):
    z = x @ P[f"{name}.0.weight"].T + P[f"{name}.0.bias"]
    pre_acts.append(z.detach())
    return torch.relu(z) @ P[f"{name}.2.weight"].T + P[f"{name}.2.bias"]


def as_tensors(params, dtype, device):
    return {k: torch.as_tensor(np.asarray(params[k]) if not torch.is_tensor(params[k]) else params[k]).to(device=device, dtype=dtype)
            for k in KEYS}


@dataclass
class StepResult:
    grads: dict          # key -> tensor (the unscaled-by-lr gradient of L x 1/K)
    losses: np.ndarray   # float64 [3]: value, reward, policy
    priorities: torch.Tensor  # [B] |v_0 - G_0|
    x_min: torch.Tensor  # [B] min over heads and unroll steps of |x| (support expectation before the transform)
    relu_min: torch.Tensor  # [B] min over every hidden unit of |pre-activation|
    gap_min: torch.Tensor   # [B] min over latents of (gap between the two smallest, resp. largest, values) / (max - min)


def forward_backward(params, batch, priority_w=None, dtype=torch.float64, device="cpu", mut=FAITHFUL):
    """Gradients, losses and new priorities of one learner step from ``params`` (key -> array) on ``batch`` =
    (states [B,3N], rwds [B,K], actions [B,K], pi [B,K,6], returns [B,K])."""
    states, rwds, actions, pi, returns = batch
    cvt = lambda a: torch.as_tensor(a if torch.is_tensor(a) else np.asarray(a)).to(device=device, dtype=dtype)  # noqa: E731
    states, rwds, pi, returns = cvt(states), cvt(rwds), cvt(pi), cvt(returns)
    actions = torch.as_tensor(actions if torch.is_tensor(actions) else np.asarray(actions)).to(device=device, dtype=torch.int64)
    B, K = rwds.shape
    P = {k: v.clone().requires_grad_(True) for k, v in as_tensors(params, dtype, device).items()}
    pre, xs, latents = [], [], []

    def T(logits):
        x = _support_x(logits)
        xs.append(x.detach().abs())
        return _signed_parabolic(x)

    h_raw = _mlp(P, "representation_net", states, pre)
    latents.append(h_raw.detach())
    h = _normalize(h_raw, mut)
    lv = lr_ = lp = 0
    v0 = None
    for t in range(K):
        pl = _mlp(P, "policy_net", h, pre)
        v = T(_mlp(P, "value_net", h, pre))
        if t == 0:
            v0 = v.detach()
        onehot = torch.nn.functional.one_hot(actions[:, t], ACTIONS).to(dtype)
        h_raw = _mlp(P, "dynamic_net", torch.cat([h, onehot], dim=-1), pre)
        latents.append(h_raw.detach())
        r = T(_mlp(P, "rwd_net", _normalize(h_raw, mut) if mut.rwd_on_normalised else h_raw, pre))
        h = _normalize(h_raw, mut)
        if mut.hook != 1.0:
            h.register_hook(lambda g, f=mut.hook: g * f)
        lv = lv + (v - returns[:, t]) ** 2
        lr_ = lr_ + (r - rwds[:, t]) ** 2
        if mut.policy_no_tsum:
            lp = lp - (pi[:, t] * pl).sum(-1) + torch.logsumexp(pl, -1)
        else:
            lp = lp - (pi[:, t] * torch.log_softmax(pl, -1)).sum(-1)
    loss = lv + lr_ + lp
    if priority_w is not None:
        loss = loss * cvt(priority_w)
    loss = loss.mean()
    g = torch.autograd.grad(loss, [P[k] for k in KEYS], grad_outputs=torch.tensor(1.0 / K, dtype=dtype, device=device))
    lat = torch.stack(latents)  # [K+1, B, 64]
    srt = lat.sort(-1).values
    span = (srt[..., -1] - srt[..., 0]).clamp_min(1e-30)
    gap = torch.minimum(srt[..., 1] - srt[..., 0], srt[..., -1] - srt[..., -2]) / span
    return StepResult(
        grads=dict(zip(KEYS, g)),
        losses=np.array([lv.detach().mean().item(), lr_.detach().mean().item(), lp.detach().mean().item()]),
        priorities=(v0 - returns[:, 0]).abs(),
        x_min=torch.stack(xs).amin(0),
        relu_min=torch.stack([z.abs().amin(-1) for z in pre]).amin(0),
        gap_min=gap.amin(0),
    )


def adam(params, grads, m, v, step_index, lr=0.002, betas=(0.9, 0.999), eps=1e-8, mut=FAITHFUL):
    """torch.optim.Adam's single-tensor step (no weight decay, amsgrad off) at the dtype of the tensors given:
    m.lerp_(g, 1 - beta1), v = beta2 v + (1 - beta2) g^2, bias corrections and step size in double on the host.
    Returns new (params, m, v) dicts."""
    b1, b2 = betas
    s = int(step_index) + mut.adam_step_off
    bias1, bias2 = 1 - b1 ** s, 1 - b2 ** s
    out_p, out_m, out_v = {}, {}, {}
    for k in KEYS:
        g = grads[k]
        mk = m[k] + (1 - b1) * (g - m[k])
        vk = b2 * v[k] + (1 - b2) * g * g
        denom = vk.sqrt() / (bias2 ** 0.5) + eps
        out_p[k] = params[k] - (lr / bias1) * (mk / denom)
        out_m[k], out_v[k] = mk, vk
    return out_p, out_m, out_v


def step(params, m, v, step_index, batch, priority_w=None, lr=0.002, dtype=torch.float64, device="cpu", mut=FAITHFUL):
    """One whole learner update: forward_backward then adam.  params / m / v: key -> array or tensor."""
    res = forward_backward(params, batch, priority_w, dtype, device, mut)
    P, M, V = (as_tensors(d, dtype, device) for d in (params, m, v))
    p2, m2, v2 = adam(P, res.grads, M, V, step_index, lr=lr, mut=mut)
    return res, p2, m2, v2


# ---- the gate: a kernel's error against float64, element-wise, relative to the yardstick's error --------------------

def error_stats(kernel, yard, ref):
    """|kernel - ref| and |yard - ref| (float64, element-wise): their maxima and 99.9th percentiles."""
    r = torch.as_tensor(ref).double().cpu().reshape(-1)
    ek = (torch.as_tensor(kernel).double().cpu().reshape(-1) - r).abs()
    ey = (torch.as_tensor(yard).double().cpu().reshape(-1) - r).abs()
    q = lambda e: float(torch.quantile(e, 0.999)) if e.numel() <= 16_000_000 else float(e.max())  # noqa: E731
    return dict(k_max=float(ek.max()), y_max=float(ey.max()), k_q=q(ek), y_q=q(ey), ref_max=float(r.abs().max()))


def ratios(s, floor):
    """How many times the yardstick's error (plus an absolute floor) the kernel's error is, at the max and the 99.9th
    percentile.  A gate (c_max, c_q) passes when these are <= c_max and c_q."""
    return s["k_max"] / (s["y_max"] + floor), s["k_q"] / (s["y_q"] + floor)


def compare_update(kernel, before, step_index, batch, priority_w=None, lr=0.002, ref_device="cpu", yard_device="cpu"):
    """Error statistics of one learner update against the float64 reference, next to the float32 yardstick's.

    kernel: dict with grads / params / m / v (key -> tensor), priorities ([B] or None) and losses ([3]); params / m / v
    may be None (no update applied).  before: dict params / m / v (key -> tensor) the update started from.
    Returns (stats {"grad:<key>" | "param:<key>" | "m:<key>" | "v:<key>" | "prio" | "loss:<name>": error_stats},
    the float64 StepResult)."""
    ref, rp, rm, rv = step(before["params"], before["m"], before["v"], step_index, batch, priority_w, lr, torch.float64, ref_device)
    yard, yp, ym, yv = step(before["params"], before["m"], before["v"], step_index, batch, priority_w, lr, torch.float32, yard_device)
    stats = {}
    for k in KEYS:
        stats[f"grad:{k}"] = error_stats(kernel["grads"][k], yard.grads[k], ref.grads[k])
        for name, part, y, r in (("param", "params", yp, rp), ("m", "m", ym, rm), ("v", "v", yv, rv)):
            if kernel.get(part) is not None:
                stats[f"{name}:{k}"] = error_stats(kernel[part][k], y[k], r[k])
    if kernel.get("priorities") is not None:
        stats["prio"] = error_stats(kernel["priorities"], yard.priorities, ref.priorities)
    for i, name in enumerate(("value", "reward", "policy")):
        stats[f"loss:{name}"] = error_stats(torch.tensor([float(kernel["losses"][i])]), torch.tensor([yard.losses[i]]),
                                            torch.tensor([ref.losses[i]]))
    return stats, ref


def check(stats, gates):
    """-> (worst ratios per category {cat: (max ratio, q ratio)}, [names that fail their category's gate]).
    gates: {category: (c_max, c_q, floor)} with category the part of the stats name before ':'."""
    worst, bad = {}, []
    for name, s in stats.items():
        cat = name.split(":")[0]
        c_max, c_q, floor = gates[cat]
        rm, rq = ratios(s, floor)
        w = worst.get(cat, (0.0, 0.0))
        worst[cat] = (max(w[0], rm), max(w[1], rq))
        if rm > c_max or rq > c_q:
            bad.append(name)
    return worst, bad


def hazard_rows(res, x_tol=1e-6, relu_tol=1e-6, gap_tol=1e-6):
    """bool [B]: rows where float32 rounding can flip a discontinuity of the step, so that an exact implementation
    at float32 sends a gradient O(1) away from float64's: |x| of a support head within ``x_tol`` of the jump of sign(x) at
    0, a ReLU pre-activation within ``relu_tol`` of 0, or a latent whose two smallest (largest) values are within
    ``gap_tol`` x (max - min) of each other without being equal (the argmin / argmax can change).  Exact ties are no
    hazard: every precision sees them and routes to the first occurrence."""
    return (res.x_min < x_tol) | (res.relu_min < relu_tol) | ((res.gap_min > 0) & (res.gap_min < gap_tol))
