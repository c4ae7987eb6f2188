"""The learner step on the device (SURVEY.md §8f row 4): ``Muzero._update`` + ``MuZeroNet.update`` of the
reference (Muzero.py:209-274, networks.py:118-122) as one libhmz call per batch.

``Learner`` owns the flat float32 parameter / gradient / Adam-moment buffers (the 20 state_dict tensors in
state_dict order, torch ``[out][in]`` layout); ``update`` has the reference's ``_update`` signature and return
values, ``step`` is the same update left on the device (no read-back); ``state_dict`` / ``load_state_dict`` move weights to and from a ``MuZeroNet`` (or a PackedWeights for the
acting kernels).  torch is used for memory only.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr
from .engine import STATE_DICT_ORDER


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
