"""The learner step on the device (SURVEY.md §8f row 4): ``Muzero._update`` + ``MuZeroNet.update`` of the
reference (Muzero.py:209-274, networks.py:118-122) as one libhmz call per batch.

``Learner`` owns the flat float32 parameter / gradient / Adam-moment buffers (the 20 state_dict tensors in
state_dict order, torch ``[out][in]`` layout); ``update`` has the reference's ``_update`` signature and return
values, ``step`` is the same update left on the device (no read-back); ``state_dict`` / ``load_state_dict`` move weights to and from a ``MuZeroNet`` (or a PackedWeights for the
acting kernels).  ``adam_to_torch`` / ``torch_to_adam`` map the flat Adam moments to and from the state dict of the
reference's optimiser (``torch.optim.Adam(MuZeroNet.parameters(), lr)``, networks.py:35).  torch is used for memory only.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr
from .engine import STATE_DICT_ORDER

ADAM_BETAS, ADAM_EPS = (0.9, 0.999), 1e-8  # torch.optim.Adam's defaults, which the reference's optimiser keeps


def param_shapes(n_disks):
    """[(state_dict key, shape)] of the N-disk MuZeroNet the learner trains (TD_return=True, h1_s=256,
    reprs_output_size=64: networks.py:39-67), in state_dict order = MuZeroNet.parameters() order."""
    hidden, latent, support = 256, 64, 33
    io = {"representation_net": (3 * int(n_disks), latent), "dynamic_net": (latent + 6, latent), "rwd_net": (latent, support),
          "policy_net": (latent, 6), "value_net": (latent, support)}
    out = []
    for net, (n_in, n_out) in io.items():
        out += [(f"{net}.0.weight", (hidden, n_in)), (f"{net}.0.bias", (hidden,)), (f"{net}.2.weight", (n_out, hidden)),
                (f"{net}.2.bias", (n_out,))]
    return out


def split_flat(flat, n_disks):
    """Flat parameter-ordered host tensor -> {key: CPU tensor of the key's shape} (each its own copy)."""
    out, at = {}, 0
    for key, shape in param_shapes(n_disks):
        n = math.prod(shape)
        out[key] = flat[at:at + n].reshape(shape).clone()
        at += n
    return out


def adam_to_torch(adam_m, adam_v, step_index, n_disks, lr, betas=ADAM_BETAS, eps=ADAM_EPS):
    """The state dict torch.optim.Adam(MuZeroNet.parameters(), lr, betas, eps) holds after ``step_index`` steps whose
    moments are the flat host tensors adam_m / adam_v: per parameter (in parameters() order) ``step``, ``exp_avg``,
    ``exp_avg_sq``, and torch's own param_groups (weight_decay 0).  Before the first step torch holds no state."""
    shapes = param_shapes(n_disks)
    params = [torch.nn.Parameter(torch.zeros(shape)) for _, shape in shapes]
    groups = torch.optim.Adam(params, lr=float(lr), betas=tuple(betas), eps=float(eps)).state_dict()["param_groups"]
    m, v = split_flat(adam_m, n_disks), split_flat(adam_v, n_disks)
    state = {}
    if step_index > 0:
        for i, (key, _) in enumerate(shapes):
            state[i] = {"step": torch.tensor(float(step_index), dtype=torch.float32), "exp_avg": m[key], "exp_avg_sq": v[key]}
    return {"state": state, "param_groups": groups}


def torch_to_adam(optim_state, n_disks):
    """Inverse of adam_to_torch: a torch.optim.Adam state dict of the N-disk MuZeroNet -> (adam_m, adam_v float32 flat
    host tensors, step_index, lr, betas, eps).  Raises ValueError, naming the field, for anything hmz_learner_step
    (plain Adam, hmz_learner.cu) cannot continue exactly: other keys, shapes or parameter count, weight decay, amsgrad,
    maximize, or parameters at different steps."""
    shapes = param_shapes(n_disks)
    if not isinstance(optim_state, dict) or set(optim_state) != {"state", "param_groups"}:
        got = sorted(optim_state) if isinstance(optim_state, dict) else type(optim_state).__name__
        raise ValueError(f"Net_optim: expected the keys ['param_groups', 'state'] of an optimiser state dict, got {got}")
    groups = optim_state["param_groups"]
    if not isinstance(groups, (list, tuple)) or len(groups) != 1:
        raise ValueError("Net_optim.param_groups: expected one parameter group")
    g = groups[0]
    for key in ("params", "lr", "betas", "eps"):
        if key not in g:
            raise ValueError(f"Net_optim.param_groups[0]: missing '{key}'")
    if list(g["params"]) != list(range(len(shapes))):
        raise ValueError(f"Net_optim.param_groups[0].params: expected the {len(shapes)} MuZeroNet parameters, got {list(g['params'])}")
    if float(g.get("weight_decay", 0.0)) != 0.0:
        raise ValueError(f"Net_optim.param_groups[0].weight_decay={g['weight_decay']}: the learner is plain Adam without weight decay")
    for flag in ("amsgrad", "maximize"):
        if g.get(flag, False):
            raise ValueError(f"Net_optim.param_groups[0].{flag}=True: the learner is plain Adam")
    state = optim_state["state"]
    n = sum(math.prod(s) for _, s in shapes)
    adam_m, adam_v = torch.zeros(n, dtype=torch.float32), torch.zeros(n, dtype=torch.float32)
    step_index = 0
    if state:
        if set(state) != set(range(len(shapes))):
            raise ValueError(f"Net_optim.state: expected entries for parameters 0..{len(shapes) - 1}, got {sorted(state)}")
        steps, at = set(), 0
        for i, (key, shape) in enumerate(shapes):
            s = state[i]
            if set(s) != {"step", "exp_avg", "exp_avg_sq"}:
                raise ValueError(f"Net_optim.state[{i}] ({key}): expected the keys ['exp_avg', 'exp_avg_sq', 'step'], got {sorted(s)}")
            for name, dst in (("exp_avg", adam_m), ("exp_avg_sq", adam_v)):
                t = s[name]
                if not torch.is_tensor(t) or tuple(t.shape) != shape:
                    got = tuple(t.shape) if torch.is_tensor(t) else type(t).__name__
                    raise ValueError(f"Net_optim.state[{i}].{name} ({key}): expected shape {shape}, got {got}")
                dst[at:at + t.numel()] = t.detach().to("cpu", torch.float32).reshape(-1)
            steps.add(float(s["step"]))
            at += math.prod(shape)
        step = min(steps)
        if len(steps) != 1 or step < 1 or step != int(step):
            raise ValueError(f"Net_optim.state[*].step: the learner keeps one step count for all parameters, got {sorted(steps)}")
        step_index = int(step)
    return adam_m, adam_v, step_index, float(g["lr"]), tuple(float(b) for b in g["betas"]), float(g["eps"])


class Learner:
    def __init__(self, state_dict, n_disks, unroll_n_steps, lr=0.002, betas=(0.9, 0.999), eps=1e-8, device="cuda"):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.n_disks, self.unroll, self.lr, self.betas, self.eps = int(n_disks), int(unroll_n_steps), float(lr), betas, float(eps)
        self.device = torch.device(device)
        n = int(self.lib.hmz_learner_param_count(self.n_disks))
        self.params = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.grads = torch.zeros_like(self.params)
        self.adam_m = torch.zeros_like(self.params)
        self.adam_v = torch.zeros_like(self.params)
        self.losses = torch.zeros(3, dtype=torch.float32, device=self.device)
        self.step_index = 0
        self._ws = None
        self._shapes = None
        self.load_state_dict(state_dict)

    # -- weights in / out ---------------------------------------------------------------------------
    def load_state_dict(self, state_dict):
        flat, shapes = [], []
        for key in STATE_DICT_ORDER:
            t = state_dict[key]
            a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
            shapes.append((key, a.shape))
            flat.append(np.ascontiguousarray(a, dtype=np.float32).reshape(-1))
        flat = np.concatenate(flat)
        if flat.size != self.params.numel():
            raise ValueError(f"state_dict has {flat.size} parameters, the N={self.n_disks} network has {self.params.numel()}")
        self._shapes = shapes
        self.params.copy_(torch.from_numpy(flat))

    def _split(self, flat):
        out, at = {}, 0
        for key, shape in self._shapes:
            n = int(np.prod(shape))
            out[key] = flat[at:at + n].reshape(shape)
            at += n
        return out

    def state_dict(self):
        """name -> device tensor views into the flat parameter buffer (MuZeroNet.load_state_dict accepts them)."""
        return self._split(self.params)

    def grad_dict(self):
        return self._split(self.grads)

    def optimizer_state_dict(self):
        """The reference optimiser's state dict of this learner's Adam state (adam_to_torch), on the host."""
        return adam_to_torch(self.adam_m.cpu(), self.adam_v.cpu(), self.step_index, self.n_disks, self.lr, self.betas, self.eps)

    # -- Muzero._update ------------------------------------------------------------------------------
    def step(self, states, rwds, actions, pi_probs, returns, priority_w=None, apply_update=True):
        """Enqueues one hmz_learner_step on the current stream and returns device tensors (new_priorities f32[B] or None,
        losses f32[3] = value, reward, policy loss) without synchronising.  ``losses`` is this Learner's buffer: the next
        step overwrites it."""
        dev = self.device
        states = torch.as_tensor(states, dtype=torch.float32, device=dev).contiguous()
        B = states.shape[0]
        rwds = torch.as_tensor(rwds, dtype=torch.float32, device=dev).contiguous()
        actions = torch.as_tensor(actions, dtype=torch.int64, device=dev).contiguous()
        pi_probs = torch.as_tensor(pi_probs, dtype=torch.float32, device=dev).contiguous()
        returns = torch.as_tensor(returns, dtype=torch.float32, device=dev).contiguous()
        if states.shape != (B, 3 * self.n_disks) or rwds.shape != (B, self.unroll) or actions.shape != (B, self.unroll) or \
                pi_probs.shape != (B, self.unroll, 6) or returns.shape != (B, self.unroll):
            raise ValueError("batch shapes do not match (B, 3N) / (B, unroll) / (B, unroll, 6)")
        w = None if priority_w is None else torch.as_tensor(priority_w, dtype=torch.float32, device=dev).contiguous()
        need = int(self.lib.hmz_learner_workspace_bytes(self.n_disks, B, self.unroll))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        new_p = torch.empty(B, dtype=torch.float32, device=dev) if w is not None else None
        self.step_index += 1 if apply_update else 0
        check(self.lib.hmz_learner_step(ptr(self.params), ptr(self.grads), ptr(self.adam_m), ptr(self.adam_v), ptr(self._ws),
                                        self.n_disks, B, self.unroll, ptr(states), ptr(rwds), ptr(actions), ptr(pi_probs), ptr(returns),
                                        ptr(w), self.lr, self.betas[0], self.betas[1], self.eps, max(1, self.step_index), ptr(new_p),
                                        ptr(self.losses), int(bool(apply_update)), current_stream()))
        return new_p, self.losses

    def update(self, states, rwds, actions, pi_probs, returns, priority_w=None, apply_update=True):
        """-> (new_priorities np.float32[B] or None, value_loss, rwd_loss, policy_loss) like Muzero._update: step() and
        the read-back."""
        new_p, losses = self.step(states, rwds, actions, pi_probs, returns, priority_w, apply_update)
        v_loss, r_loss, p_loss = losses.cpu().tolist()
        return (None if new_p is None else new_p.cpu().numpy()), v_loss, r_loss, p_loss
