"""Episode store and GPU-resident replay ring (SURVEY.md §8f rows 1-2).

``EpisodeStore`` keeps the per-move lists of ``Muzero._play_game`` (reference Muzero.py:153-207) for B
games in struct-of-arrays form on the device and runs the episode post-processing there: n-step TD
returns (utils.py:28-72), priorities (Muzero.py:197-200) and ``organise_transitions``
(Muzero.py:276-323).  ``ReplayRing`` is ``buffer.Buffer`` (buffer.py) with its arrays resident in HBM:
same constructor, attributes and methods; ``add_episodes`` is the device-side ``add``.
torch is used for memory and index gathers only; every computation is a libhmz kernel.

``priority_sample_device`` / ``uniform_sample_device`` / ``update_priorities_device`` draw a training batch and write the
new priorities back without a host round trip, bit-identical to ``priority_sample`` / ``uniform_sample`` /
``update_priorities`` given the same NumPy global RandomState.  The host draws only the random numbers: the uniforms
of ``np.random.choice``, or ``randint``'s indices.  ``hmz_replay_sample`` runs the rest on the device.  It runs NumPy's
pairwise float32 sum, the division and ``choice``'s checks.  It runs the float64 cumulative sum exactly in parallel:
inside one binade of the running sum every addition is an integer step on the grid ulp(c), decided by the addend
alone except at an exact half-ulp tie, so the rows compose as maps of the parity bit and a block scan gives NumPy's
left-to-right sums (DESIGN §3).  It also runs the search and the importance weights.  Errors NumPy would raise set
bits of ``status`` (a device int32 that only accumulates); ``check_status`` or ``raise_for_status`` raise them with
the reference's exception types and messages.  Priority exponents other than 1 are served by ``priority_sample``
only.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr


def discount_powers(discount: float, n_step: int) -> np.ndarray:
    """``discount ** i`` for i in [0, n_step] with the host's float pow, as utils.py:64-69 evaluates it."""
    return np.array([discount ** i for i in range(n_step + 1)], dtype=np.float64)


class EpisodeStore:
    """[t_max][B] struct-of-arrays of the running episodes; slot = the game's own step counter."""

    def __init__(self, B, t_max, n_disks, device="cuda"):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.B, self.t_max, self.n_disks = int(B), int(t_max), int(n_disks)
        self.device = dev = torch.device(device)
        T = self.t_max
        self.state = torch.zeros(T, B, dtype=torch.int32, device=dev)
        self.action = torch.zeros(T, B, dtype=torch.uint8, device=dev)
        self.flags = torch.zeros(T, B, dtype=torch.uint8, device=dev)
        self.visits = torch.zeros(T, B, 6, dtype=torch.int16, device=dev)
        self.root_q = torch.zeros(T, B, dtype=torch.float64, device=dev)
        self.cur_slot = torch.zeros(B, dtype=torch.int32, device=dev)
        self.ep_len = torch.zeros(B, dtype=torch.int32, device=dev)
        # play-policy exponent in force when each move was played (SelfPlay fills it); None = use add_episodes' temperature
        self.exp = None
        self.mismatch = None  # ingest's count of records that were not the game of their row (int32 [1] on the device)
        self.returns = torch.zeros(T, B, dtype=torch.float64, device=dev)
        self.priority = torch.zeros(T, B, dtype=torch.float32, device=dev)
        self.row_base = torch.full((B,), -1, dtype=torch.int64, device=dev)
        self.total = torch.zeros(1, dtype=torch.int64, device=dev)
        self._pow = None
        self._mc_pow = None

    def record(self, words, action, visits, root_q, action_u8_out=None):
        """Muzero.py:179-183 for every game (before the env step)."""
        check(self.lib.hmz_episode_record(ptr(words), ptr(action), ptr(visits), ptr(root_q), self.n_disks, self.t_max, self.B,
                                          ptr(self.state), ptr(self.action), ptr(self.visits), ptr(self.root_q),
                                          ptr(self.cur_slot), ptr(action_u8_out), current_stream()))

    def close(self, flags):
        """After the env step: ep_len[g] = length of the episode that just finished, else 0."""
        check(self.lib.hmz_episode_close(ptr(flags), ptr(self.cur_slot), self.B, ptr(self.flags), ptr(self.ep_len),
                                         current_stream()))

    def ingest(self, records, temperature, game_offset=0):
        """One move of every game from its move records (uint8 [B, 32], e.g. dist.RecordGather.result(i)): the store
        writes SelfPlay(episodes=True) makes, with ``temperature`` the one the move was played at.  Record i must be global
        game ``game_offset + i``; one whose game_lo says otherwise writes nothing and adds 1 to ``self.mismatch``
        (int32 [1] on the device, never reset here)."""
        if records.dtype != torch.uint8 or tuple(records.shape) != (self.B, _lib.RECORD_BYTES) or not records.is_contiguous() \
                or not records.is_cuda:
            raise ValueError(f"records must be a contiguous uint8 [{self.B}, {_lib.RECORD_BYTES}] device tensor, got "
                             f"{records.dtype} {tuple(records.shape)} on {records.device}")
        if self.exp is None:
            self.exp = torch.ones(self.t_max, self.B, dtype=torch.uint8, device=self.device)
        if self.mismatch is None:
            self.mismatch = torch.zeros(1, dtype=torch.int32, device=self.device)
        check(self.lib.hmz_episode_ingest(ptr(records), self.B, int(game_offset), self.n_disks, self.t_max, float(temperature),
                                          ptr(self.state), ptr(self.action), ptr(self.flags), ptr(self.visits), ptr(self.root_q),
                                          ptr(self.cur_slot), ptr(self.ep_len), ptr(self.exp), ptr(self.mismatch), current_stream()))

    def post_process(self, n_step, discount):
        """compute_n_step_returns + priorities of every finished episode (ep_len > 0)."""
        key = (float(discount), int(n_step))
        if self._pow is None or self._pow[0] != key:
            self._pow = (key, torch.from_numpy(discount_powers(*key)).to(self.device))
        check(self.lib.hmz_episode_returns(ptr(self.flags), ptr(self.root_q), ptr(self.ep_len), self.B, self.t_max,
                                           ptr(self._pow[1]), int(n_step), ptr(self.returns), ptr(self.priority),
                                           current_stream()))
        return self.returns, self.priority

    def post_process_mc(self, discount):
        """compute_MCreturns (utils.py:75-86, TD_return=False) + priorities of every finished episode."""
        if self._mc_pow is None or self._mc_pow[0] != float(discount):
            # the reference evaluates `discount ** np.array(range(T))` with NumPy's power ufunc (not libm's pow)
            self._mc_pow = (float(discount), torch.from_numpy(float(discount) ** np.arange(self.t_max)).to(self.device))
        check(self.lib.hmz_episode_mc_returns(ptr(self.flags), ptr(self.root_q), ptr(self.ep_len), self.B, self.t_max,
                                              ptr(self._mc_pow[1]), ptr(self.returns), ptr(self.priority), current_stream()))
        return self.returns, self.priority


class ReplayRing:
    """buffer.Buffer (reference buffer.py:5-136) with device-resident arrays."""

    def __init__(self, size, unroll_n_steps, d_state, n_action, device="cuda", priority_exponent=1,
                 importance_sampling_exponent=0):
        _lib.require_cuda()
        if n_action != _lib.N_ACTIONS:
            raise ValueError(f"n_action={n_action}: the Hanoi action set has {_lib.N_ACTIONS} moves")
        self.lib = _lib.load()
        self.dev = torch.device(device)
        self._priority_exponent = priority_exponent
        self._importance_sampling_exponent = importance_sampling_exponent
        self.size, self.unroll_n_steps, self.n_action, self.d_state = int(size), int(unroll_n_steps), int(n_action), int(d_state)
        dev = self.dev
        self.states = torch.zeros(size, d_state, dtype=torch.float32, device=dev)
        self.rwds = torch.zeros(size, unroll_n_steps, dtype=torch.float32, device=dev)
        self.actions = torch.zeros(size, unroll_n_steps, dtype=torch.int64, device=dev)
        self.pi_probs = torch.zeros(size, unroll_n_steps, n_action, dtype=torch.float32, device=dev)
        self.mc_returns = torch.zeros(size, unroll_n_steps, dtype=torch.float32, device=dev)
        self.priorities = torch.zeros(size, dtype=torch.float32, device=dev)
        self.ptr = 0
        self.is_full = False
        # device sampling: HMZ_REPLAY_* bits of every error NumPy would have raised since the ring was made (never cleared)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        self._ws = None

    def __len__(self):
        return self.size if self.is_full else self.ptr

    def _advance(self, n):
        if self.ptr + n >= self.size:  # buffer.py:80-82
            self.is_full = True
        self.ptr = (self.ptr + n) % self.size

    # -- device-side add -------------------------------------------------------------------------
    def add_episodes(self, store: EpisodeStore, temperature=1.0, only_solved=True, absorbing_action=None):
        """organise_transitions + Buffer.add for every finished episode of ``store`` (after
        ``store.post_process``).  ``only_solved`` applies training_loop's filter ``returns[-1, 0] > 0``
        (Muzero.py:98).  ``absorbing_action`` uint8 [B]: the padding action of each episode (the
        reference draws one ``np.random.randint(0, n_action)`` per episode, Muzero.py:300-303); drawn
        with torch when omitted.  Returns the number of rows added (one scalar read back)."""
        if self.d_state != 3 * store.n_disks:
            raise ValueError(f"d_state={self.d_state} does not match {store.n_disks} disks")
        if absorbing_action is None:
            absorbing_action = torch.randint(0, self.n_action, (store.B,), dtype=torch.uint8, device=self.dev)
        ab = torch.as_tensor(absorbing_action, dtype=torch.uint8, device=self.dev).contiguous()
        s = current_stream()
        check(self.lib.hmz_episode_rows(ptr(store.ep_len), ptr(store.returns), store.B, self.ptr, int(bool(only_solved)),
                                        ptr(store.row_base), ptr(store.total), s))
        n = int(store.total.item())
        # The reference adds one episode at a time (Muzero.py:98-101 -> buffer.py:47-83), so when the episodes finishing on
        # this move hold more rows than the ring, the earlier rows are overwritten by the later ones: only the last
        # `size` rows (in game order) survive, at the positions sequential adds would have left them.
        first_row = self.ptr + max(0, n - self.size)
        if n:
            check(self.lib.hmz_episode_unroll(ptr(store.state), ptr(store.action), ptr(store.flags), ptr(store.visits),
                                              ptr(store.returns), ptr(store.priority), ptr(store.ep_len), ptr(store.row_base),
                                              ptr(ab), ptr(store.exp), store.B, store.t_max, store.n_disks, self.unroll_n_steps,
                                              float(temperature), self.size, first_row, ptr(self.states), ptr(self.rwds), ptr(self.actions),
                                              ptr(self.pi_probs), ptr(self.mc_returns), ptr(self.priorities), s))
            self._advance(n)
        return n

    # -- reference-shaped host add (buffer.py:47-83) -----------------------------------------------
    def _add(self, buffer, transitions):
        t = torch.as_tensor(np.asarray(transitions), device=self.dev).to(buffer.dtype)
        n = t.shape[0]
        excess = self.ptr + n - self.size
        a, b = (n, 0) if excess <= 0 else (n - excess, excess)
        buffer[self.ptr:self.ptr + a] = t[:a]
        buffer[:b] = t[a:]

    def add(self, states, rwds, actions, pi_probs, mc_returns, priorities):
        n = np.asarray(states).shape[0]
        assert n <= self.size
        for buf, x in ((self.states, states), (self.rwds, rwds), (self.actions, actions), (self.pi_probs, pi_probs),
                       (self.mc_returns, mc_returns), (self.priorities, priorities)):
            self._add(buf, x)
        self._advance(n)

    # -- sampling (buffer.py:85-128) on the host: the index draw is NumPy's, the rows never leave the device -----
    def _sample(self, indx):
        i = torch.as_tensor(indx, dtype=torch.int64, device=self.dev)
        return self.states[i], self.rwds[i], self.actions[i], self.pi_probs[i], self.mc_returns[i]

    def uniform_sample(self, batch_s):
        num = len(self)
        indx = np.random.choice(np.arange(num), size=batch_s, replace=True).astype(np.int64)
        return self._sample(indx)

    def priority_sample(self, batch_s):
        num = len(self)
        priorities = self.priorities[:num].cpu().numpy() ** self._priority_exponent
        priorities_probs = priorities / np.sum(priorities)
        indx = np.random.choice(np.arange(num), size=batch_s, replace=True, p=priorities_probs).astype(np.int64)
        states, rwds, actions, pi_probs, mc_returns = self._sample(indx)
        weights = ((1.0 / self.size) / priorities_probs[indx]) ** self._importance_sampling_exponent
        weights /= np.max(weights)
        weights = torch.from_numpy(weights).to(self.dev, dtype=torch.float32)
        return states, rwds, actions, pi_probs, mc_returns, indx, weights

    def update_priorities(self, indx, new_priorities):
        if indx is not None:
            new_priorities = np.asarray(new_priorities)
            assert np.isfinite(new_priorities).all() and (new_priorities > 0.0).any(), "Priorities must be finite and positive."
            self.priorities[torch.as_tensor(indx, dtype=torch.int64, device=self.dev)] = torch.as_tensor(
                new_priorities, dtype=torch.float32, device=self.dev)

    # -- sampling without a host round trip ------------------------------------------------------------
    # The same draws as uniform_sample / priority_sample / update_priorities, enqueued on the current stream with no
    # synchronisation: the host draws only the random numbers (from NumPy's global RandomState, in the same order) and
    # copies them from pinned memory; hmz_replay_sample runs priority_sample's sum, division, NumPy's checks, the
    # cumulative sum, the search and the weights on the device, bit-exact.  Errors NumPy would raise set bits of
    # self.status instead; check_status() (or raise_for_status on a value read back with other results) raises them.
    def _to_device(self, a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().to(self.dev, non_blocking=True)

    def uniform_sample_device(self, batch_s):
        """uniform_sample with the indices copied to the device without a synchronise (np.random.choice(arange(num),
        batch, replace=True) is np.random.randint(0, num, batch): same indices, same draws)."""
        indx = self._to_device(np.random.randint(0, len(self), int(batch_s)).astype(np.int64))
        return self._sample(indx)

    def priority_sample_device(self, batch_s, uniforms=None):
        """priority_sample with indx and the weights as device tensors.  uniforms: float64 [batch_s], the draw of
        np.random.choice; np.random.random_sample(batch_s) when omitted."""
        num, batch_s = len(self), int(batch_s)
        if uniforms is None:
            uniforms = np.random.random_sample(batch_s)
        u = uniforms if torch.is_tensor(uniforms) else self._to_device(np.asarray(uniforms, dtype=np.float64))
        if u.dtype != torch.float64 or u.numel() != batch_s or not u.is_cuda:
            raise ValueError(f"uniforms must be {batch_s} float64 values")
        u = u.contiguous()
        need = int(self.lib.hmz_replay_sample_workspace_bytes(max(num, 1)))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.dev)
        indx = torch.empty(batch_s, dtype=torch.int64, device=self.dev)
        weights = torch.empty(batch_s, dtype=torch.float32, device=self.dev)
        check(self.lib.hmz_replay_sample(ptr(self.priorities), num, self.size, float(self._priority_exponent), ptr(u), batch_s,
                                         float(self._importance_sampling_exponent), ptr(self._ws), ptr(indx), ptr(weights),
                                         ptr(self.status), current_stream()))
        states, rwds, actions, pi_probs, mc_returns = self._sample(indx)
        return states, rwds, actions, pi_probs, mc_returns, indx, weights

    def update_priorities_device(self, indx, new_priorities):
        """update_priorities from device tensors: duplicates in indx keep their last value; a batch that fails the
        reference's assertion writes nothing and sets REPLAY_PRIORITY in self.status."""
        if indx is None:
            return
        i = torch.as_tensor(indx, dtype=torch.int64, device=self.dev).contiguous()
        p = torch.as_tensor(new_priorities, dtype=torch.float32, device=self.dev).contiguous()
        if i.numel() != p.numel():
            raise ValueError(f"{i.numel()} indices but {p.numel()} priorities")
        check(self.lib.hmz_replay_set_priorities(ptr(self.priorities), self.size, ptr(i), ptr(p), i.numel(), ptr(self.status),
                                                 current_stream()))

    @staticmethod
    def raise_for_status(status: int):
        """The exception the reference would have raised first, for status bits read back from ReplayRing.status."""
        status = int(status)
        if status & _lib.REPLAY_NAN:
            raise ValueError("probabilities contain NaN")
        if status & _lib.REPLAY_NEGATIVE:
            raise ValueError("probabilities are not non-negative")
        if status & _lib.REPLAY_SUM:
            raise ValueError("probabilities do not sum to 1")
        if status & _lib.REPLAY_PRIORITY:
            raise AssertionError("Priorities must be finite and positive.")

    def check_status(self):
        """Reads the status word (one synchronise) and raises what the reference would have raised."""
        self.raise_for_status(int(self.status.item()))
