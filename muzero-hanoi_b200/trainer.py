"""Batched counterpart of the reference's ``Muzero`` class (Muzero.py): self-play, episode post-processing,
replay and the learner step, all on the device, tied together in the shape of ``Muzero.training_loop``
(Muzero.py:80-150).

Differences from the sequential reference, all forced by playing B games at once:
  * one "loop" plays ``moves_per_loop`` moves of all B games instead of ``n_ep_x_loop`` whole episodes; the episodes
    that finish during a loop are post-processed and (if solved, Muzero.py:98) stored;
  * the temperature schedule (utils.adjust_temperature) is driven by the number of finished episodes per game slot;
  * acting uses the weights of the last completed update (repacked for the acting kernels once per loop);
  * the updates of a loop are enqueued without a host round trip (``step``: the replay draw, the learner step and the
    priority write-back on the device, bit-identical to the reference's NumPy draws); the last update's losses and the
    replay ring's status are read back once at the end of the loop, so a ring the reference would reject raises there.
Same hyper-parameters and defaults as training_main.TrainingConfig (training_main.py:17-36).

With ``torch.distributed`` initialised over G > 1 processes (one per GPU, e.g. torchrun) the loop takes the Ape-X /
IMPALA shape: every rank plays n_games / G of the games (global ids rank * n_games / G onwards, so the Philox streams and
hence the moves are those of one GPU playing all n_games), every move's records are all-gathered (dist.RecordGather), and
ONE learner on rank 0 builds the episode store and replay ring from them (EpisodeStore.ingest), samples and updates.  At
the end of each loop rank 0 broadcasts its weights, the episode count and the loop's history row.  Training on G GPUs
is therefore bit-identical to training on one GPU with the same n_games; with G == 1 nothing of this runs.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from . import dist as hdist
from .engine import PackedWeights, SelfPlay
from .learner import Learner
from .replay import EpisodeStore, ReplayRing
from .utils import adjust_temperature


class BatchedMuzero:
    def __init__(self, state_dict, N, max_steps, n_games, discount=0.8, dirichlet_alpha=0.25, n_mcts_simulations=25,
                 unroll_n_steps=5, batch_s=256, n_TD_step=10, lr=0.002, buffer_size=50000, priority_replay=True,
                 n_update_x_loop=1, moves_per_loop=8, acting_mode=_lib.MODE_FP32, seed=0, device="cuda"):
        self.N, self.max_steps, self.B = int(N), int(max_steps), int(n_games)
        self.discount, self.alpha, self.S = discount, dirichlet_alpha, int(n_mcts_simulations)
        self.unroll, self.batch_s, self.n_step = int(unroll_n_steps), int(batch_s), int(n_TD_step)
        self.priority_replay, self.n_update_x_loop, self.moves_per_loop = priority_replay, int(n_update_x_loop), int(moves_per_loop)
        self.acting_mode, self.seed, self.device = acting_mode, int(seed), device
        self.rank, self.world = (dist.get_rank(), dist.get_world_size()) if dist.is_available() and dist.is_initialized() else (0, 1)
        if self.B % self.world:
            raise ValueError(f"n_games={self.B} must be a multiple of the world size {self.world} (equal shards per rank)")
        # every rank keeps a Learner as the holder of the acting weights; only rank 0's ever updates
        self.learner = Learner(state_dict, N, unroll_n_steps, lr=lr, device=device)
        self.buffer = ReplayRing(buffer_size, unroll_n_steps, 3 * N, 6, device) if self.rank == 0 else None
        self.episodes_done = 0
        self._selfplay = None
        self._temperature = None
        self._weights_dirty = False
        self._gather = None      # world > 1: the per-move all-gather of the move records
        self._episodes = None    # world > 1, rank 0: the episode store of all n_games, filled from the gathered records
        self._mismatches = 0     # world > 1, rank 0: gathered records that were not the game of their row (cumulative)
        self._replay_status = 0  # world > 1, rank 0: the replay ring's status word as read at the end of the loop

    def _latent_dtype(self):
        return _lib.LATENT_BF16 if self.acting_mode == _lib.MODE_BF16 else _lib.LATENT_F32

    def _refresh_actor(self, temperature):
        """New acting weights (and a new temperature) take effect; games in flight and their episode store carry on.
        The weights are repacked only after an update has changed them."""
        if self._selfplay is None:
            w = PackedWeights({k: v for k, v in self.learner.state_dict().items()}, self.N, self.acting_mode, self.device)
            if self.world == 1:
                self._selfplay = SelfPlay(self.N, self.max_steps, self.B, self.S, w, self.discount, self.alpha, temperature=temperature,
                                          seed=self.seed, device=self.device, latent_dtype=self._latent_dtype(), episodes=True)
            else:
                shard = self.B // self.world
                self._selfplay = SelfPlay(self.N, self.max_steps, shard, self.S, w, self.discount, self.alpha, temperature=temperature,
                                          seed=self.seed, device=self.device, latent_dtype=self._latent_dtype(), episodes=False,
                                          game_offset=self.rank * shard)
                self._gather = hdist.RecordGather(shard, self.world, self.device)
                if self.rank == 0:
                    self._episodes = EpisodeStore(self.B, self.max_steps, self.N, self.device)
        else:
            if self._weights_dirty:
                self._selfplay.weights = PackedWeights({k: v for k, v in self.learner.state_dict().items()}, self.N, self.acting_mode,
                                                       self.device)
            self._selfplay.temperature = float(temperature)
        self._weights_dirty = False
        self._temperature = temperature

    def play(self, n_moves):
        """n_moves moves of every game; finished episodes are post-processed and, if solved, stored.
        Returns (episodes finished, mean length of those episodes, transitions stored).  With world > 1 every rank must
        call it; those numbers are rank 0's, and the other ranks return (0, nan, 0)."""
        if self.world > 1:
            return self._play_sharded(n_moves)
        sp, st = self._selfplay, self._selfplay.episodes
        stored = 0
        counts = torch.zeros(2, dtype=torch.int64, device=st.ep_len.device)  # episodes finished, sum of their lengths
        for _ in range(n_moves):
            sp.move()
            st.post_process(self.n_step, self.discount)
            stored += self.buffer.add_episodes(st, temperature=self._temperature, only_solved=True)  # the one sync per move
            lens = st.ep_len
            counts[0] += (lens > 0).sum()
            counts[1] += lens.sum()
        finished, length_sum = (int(x) for x in counts.tolist())  # read back once per call
        self.episodes_done += finished
        return finished, (length_sum / finished if finished else float("nan")), stored

    def _play_sharded(self, n_moves):
        """play() over the ranks: each rank plays its shard and submits every move's records to the all-gather; rank 0
        ingests the gathered records of all n_games into its episode store and stores the finished episodes.  The
        ingest's ordering check is read back with the loop's counts and acted on in _end_loop, on every rank."""
        sp, st = self._selfplay, self._episodes
        stored = 0
        counts = torch.zeros(2, dtype=torch.int64, device=sp.device) if self.rank == 0 else None
        for _ in range(n_moves):
            i = self._gather.submit(sp.slot(sp.move()))
            if self.rank == 0:
                st.ingest(self._gather.result(i), self._temperature)
                st.post_process(self.n_step, self.discount)
                stored += self.buffer.add_episodes(st, temperature=self._temperature, only_solved=True)  # the one sync per move
                lens = st.ep_len
                counts[0] += (lens > 0).sum()
                counts[1] += lens.sum()
        if self.rank != 0:
            return 0, float("nan"), 0
        finished, length_sum, self._mismatches = (int(x) for x in torch.cat([counts, st.mismatch.to(torch.int64)]).tolist())
        self.episodes_done += finished
        return finished, (length_sum / finished if finished else float("nan")), stored

    def _end_loop(self, row):
        """world > 1, every rank: rank 0's weights, episode count, whether an update changed the weights, the replay
        ring's status and the loop's history row are broadcast, so that every rank repacks its acting weights when one GPU
        would, returns the same history and raises what rank 0 raises.  Raises if rank 0 found gathered records out of
        order or a replay draw / priority write-back that the reference would have rejected."""
        info = torch.tensor([self.episodes_done, float(self._weights_dirty), self._mismatches, self._replay_status, *row[1:]],
                            dtype=torch.float64, device=self.learner.device)
        dist.broadcast(self.learner.params, 0)
        dist.broadcast(info, 0)
        episodes_done, dirty, mismatches, replay_status, *rest = info.tolist()
        if mismatches:
            raise RuntimeError(f"{int(mismatches)} gathered move records were not the game of their row (game_lo check): the "
                               "all-gathered records are out of order")
        ReplayRing.raise_for_status(int(replay_status))
        self.episodes_done, self._weights_dirty = int(episodes_done), bool(dirty)
        return (row[0], *rest)

    def step(self):
        """One Muzero._update (Muzero.py:104-127) on a batch drawn from the replay ring, enqueued without a host round
        trip: the host draws the random numbers from NumPy's global RandomState exactly as the reference does, the draw
        itself (ReplayRing.priority_sample_device / uniform_sample_device), the learner step and the priority write-back
        run on the device.  Returns the losses (value, reward, policy) as the learner's device buffer, which the next
        update overwrites.  Errors the reference would raise accumulate in self.buffer.status."""
        if self.priority_replay:
            states, rwds, actions, pi_probs, returns, indx, w = self.buffer.priority_sample_device(self.batch_s)
        else:
            states, rwds, actions, pi_probs, returns = self.buffer.uniform_sample_device(self.batch_s)
            indx, w = None, None
        if "update" in vars(self.learner):
            # Learner.update replaced on the instance (a hook that inspects every update): it is driven, read-back included
            new_p, *losses = self.learner.update(states, rwds, actions, pi_probs, returns, w)
            losses = torch.tensor(losses, dtype=torch.float32, device=self.learner.device)
        else:
            new_p, losses = self.learner.step(states, rwds, actions, pi_probs, returns, w)
        self._weights_dirty = True
        self.buffer.update_priorities_device(indx, new_p)
        return losses

    def _read_back(self, losses):
        """(value, reward, policy loss) and the replay ring's status word in one read-back."""
        *vals, status = torch.cat([losses.to(torch.float64), self.buffer.status.to(torch.float64)]).tolist()
        return tuple(vals), int(status)

    def update(self):
        """One update (step) and its read-back: -> (value loss, reward loss, policy loss) as Muzero._update returns them;
        raises what the reference would have raised."""
        losses, status = self._read_back(self.step())
        ReplayRing.raise_for_status(status)
        return losses

    def training_loop(self, n_loops, min_replay_size, print_acc=None, log=print):
        """-> list of (loop, mean episode length of the loop, value loss, reward loss, policy loss)."""
        history = []
        for n in range(1, n_loops):
            self._refresh_actor(adjust_temperature(self.episodes_done // max(1, self.B)))
            finished, mean_len, _ = self.play(self.moves_per_loop)
            losses = (float("nan"),) * 3
            if self.rank == 0 and not self._mismatches and len(self.buffer) > min_replay_size and self.n_update_x_loop > 0:
                for _ in range(self.n_update_x_loop):
                    dev_losses = self.step()
                # the loop's one read-back of its updates: the last update's losses and the replay ring's status word, so
                # a draw the reference would reject raises here, at the end of the loop, rather than at its update
                losses, self._replay_status = self._read_back(dev_losses)
                if self.world == 1:
                    ReplayRing.raise_for_status(self._replay_status)
            row = (n, mean_len, *losses)
            history.append(self._end_loop(row) if self.world > 1 else row)
            mean_len, losses = history[-1][1], history[-1][2:]
            if print_acc and n % print_acc == 0:
                log("Loop %d | episodes %d | steps %.3f | V %.3f | rwd %.3f | Pi %.3f" % (n, self.episodes_done, mean_len, *losses))
        return history
