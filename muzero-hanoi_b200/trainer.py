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

``save`` / ``load`` write and read the whole state of a run at a loop boundary (DESIGN §6), so that a loaded trainer
continues bit-identically; ``export_reference`` / ``from_reference`` write and read the reference's own checkpoint file
(``{"Muzero_net": state_dict, "Net_optim": optimiser state dict}``, training_main.py:save_results).
"""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from . import dist as hdist
from .engine import PackedWeights, SelfPlay, check_env_shape
from .learner import ADAM_BETAS, ADAM_EPS, Learner, param_shapes, split_flat, torch_to_adam
from .replay import EpisodeStore, ReplayRing
from .utils import adjust_temperature

CHECKPOINT_VERSION = 1
# the constructor arguments a checkpoint records (all but the initial weights and the device)
CONFIG_KEYS = ("N", "max_steps", "n_games", "discount", "dirichlet_alpha", "n_mcts_simulations", "unroll_n_steps", "batch_s",
               "n_TD_step", "lr", "buffer_size", "priority_replay", "n_update_x_loop", "moves_per_loop", "acting_mode", "seed")
EPISODE_FIELDS = {"state": torch.int32, "action": torch.uint8, "flags": torch.uint8, "visits": torch.int16,
                  "root_q": torch.float64, "exp": torch.uint8}
RING_FIELDS = ("states", "rwds", "actions", "pi_probs", "mc_returns", "priorities")


def _world():
    return (dist.get_rank(), dist.get_world_size()) if dist.is_available() and dist.is_initialized() else (0, 1)


def _step_counters(words, n_disks):
    """The step counters in the spare bits of env words (int32 [B]) as int64 [B]: the moves of each game's episode in flight."""
    return (words.to(torch.int64) & 0xFFFFFFFF) >> (2 * int(n_disks))


def _field(ck, path, dtype=None, shape=None, kind=None):
    """ck's field at the dotted ``path``, checked to be a CPU tensor of dtype and shape, or an instance of kind."""
    node = ck
    for part in path.split("."):
        if not isinstance(node, dict) or part not in node:
            raise ValueError(f"checkpoint: missing field '{path}'")
        node = node[part]
    if dtype is not None:
        if not torch.is_tensor(node) or node.dtype != dtype or tuple(node.shape) != tuple(shape):
            got = f"{node.dtype} {tuple(node.shape)}" if torch.is_tensor(node) else type(node).__name__
            raise ValueError(f"checkpoint field '{path}': expected {dtype} {tuple(shape)}, got {got}")
    elif kind is not None and (not isinstance(node, kind) or (kind is int and isinstance(node, bool))):
        raise ValueError(f"checkpoint field '{path}': expected {kind.__name__}, got {type(node).__name__}")
    return node


def check_checkpoint(ck):
    """Raises ValueError naming the field if ``ck`` (a loaded BatchedMuzero.save file) is not a checkpoint of this format
    version whose every tensor has the shape its config implies."""
    if not isinstance(ck, dict) or ck.get("version") != CHECKPOINT_VERSION:
        got = ck.get("version") if isinstance(ck, dict) else type(ck).__name__
        raise ValueError(f"checkpoint field 'version': expected format version {CHECKPOINT_VERSION}, got {got!r}")
    cfg = _field(ck, "config", kind=dict)
    if set(cfg) != set(CONFIG_KEYS):
        raise ValueError(f"checkpoint field 'config': expected the keys {sorted(CONFIG_KEYS)}, got {sorted(cfg)}")
    for key in ("N", "max_steps", "n_games", "n_mcts_simulations", "unroll_n_steps", "batch_s", "n_TD_step", "buffer_size",
                "n_update_x_loop", "moves_per_loop", "acting_mode", "seed"):
        _field(ck, f"config.{key}", kind=int)
    for key in ("discount", "dirichlet_alpha", "lr"):
        _field(ck, f"config.{key}", kind=float)
    _field(ck, "config.priority_replay", kind=bool)
    N, T, B, K, size = cfg["N"], cfg["max_steps"], cfg["n_games"], cfg["unroll_n_steps"], cfg["buffer_size"]
    try:
        check_env_shape(N, T)
    except ValueError as e:
        raise ValueError(f"checkpoint field 'config': {e}") from None
    P = sum(int(np.prod(s)) for _, s in param_shapes(N))
    for key in ("params", "adam_m", "adam_v"):
        _field(ck, f"learner.{key}", torch.float32, (P,))
    _field(ck, "learner.step_index", kind=int)
    for key in ("loops_done", "episodes_done", "replay_status"):
        _field(ck, f"trainer.{key}", kind=int)
    _field(ck, "trainer.weights_dirty", kind=bool)
    _field(ck, "trainer.temperature", kind=float)
    _field(ck, "selfplay.moves_done", kind=int)
    _field(ck, "selfplay.minmax", torch.float64, (B, 2))
    steps = _step_counters(_field(ck, "selfplay.words", torch.int32, (B,)), N)
    if B and int(steps.max()) >= T:
        raise ValueError(f"checkpoint field 'selfplay.words': a step counter of {int(steps.max())} with max_steps={T}")
    L = int(steps.sum())
    for key, dtype in EPISODE_FIELDS.items():
        _field(ck, f"episodes.{key}", dtype, (L, 6) if key == "visits" else (L,))
    _field(ck, "episodes.cur_slot", torch.int32, (B,))
    _field(ck, "episodes.ep_len", torch.int32, (B,))
    ptr, is_full = _field(ck, "replay.ptr", kind=int), _field(ck, "replay.is_full", kind=bool)
    _field(ck, "replay.status", kind=int)
    if not 0 <= ptr < max(size, 1):
        raise ValueError(f"checkpoint field 'replay.ptr': {ptr} is outside a ring of {size} rows")
    n = size if is_full else ptr
    shapes = dict(states=(n, 3 * N), rwds=(n, K), actions=(n, K), pi_probs=(n, K, _lib.N_ACTIONS), mc_returns=(n, K),
                  priorities=(n,))
    for key in RING_FIELDS:
        _field(ck, f"replay.{key}", torch.int64 if key == "actions" else torch.float32, shapes[key])
    _field(ck, "rng.numpy.key", torch.int64, (624,))
    for key in ("pos", "has_gauss"):
        _field(ck, f"rng.numpy.{key}", kind=int)
    _field(ck, "rng.numpy.cached_gaussian", kind=float)
    gen = _field(ck, "rng.torch_cuda")
    if not torch.is_tensor(gen) or gen.dtype != torch.uint8 or gen.dim() != 1:
        raise ValueError("checkpoint field 'rng.torch_cuda': expected a uint8 vector (torch.cuda.get_rng_state)")


class BatchedMuzero:
    def __init__(self, state_dict, N, max_steps, n_games, discount=0.8, dirichlet_alpha=0.25, n_mcts_simulations=25,
                 unroll_n_steps=5, batch_s=256, n_TD_step=10, lr=0.002, buffer_size=50000, priority_replay=True,
                 n_update_x_loop=1, moves_per_loop=8, acting_mode=_lib.MODE_FP32, seed=0, device="cuda"):
        self.N, self.max_steps, self.B = int(N), int(max_steps), int(n_games)
        self.discount, self.alpha, self.S = discount, dirichlet_alpha, int(n_mcts_simulations)
        self.unroll, self.batch_s, self.n_step = int(unroll_n_steps), int(batch_s), int(n_TD_step)
        self.priority_replay, self.n_update_x_loop, self.moves_per_loop = priority_replay, int(n_update_x_loop), int(moves_per_loop)
        self.acting_mode, self.seed, self.device = acting_mode, int(seed), device
        self.buffer_size = int(buffer_size)
        self.rank, self.world = _world()
        if self.B % self.world:
            raise ValueError(f"n_games={self.B} must be a multiple of the world size {self.world} (equal shards per rank)")
        # every rank keeps a Learner as the holder of the acting weights; only rank 0's ever updates
        self.learner = Learner(state_dict, N, unroll_n_steps, lr=lr, device=device)
        self.buffer = ReplayRing(buffer_size, unroll_n_steps, 3 * N, 6, device) if self.rank == 0 else None
        self.episodes_done = 0
        self.loops_done = 0       # loops of training_loop run so far, those before a load included
        self._resumed = False     # loaded from a checkpoint: training_loop numbers its loops on from loops_done
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
        """-> list of (loop, mean episode length of the loop, value loss, reward loss, policy loss).  Runs n_loops - 1
        loops numbered from 1, or, on a trainer made by ``load``, numbered on from the loops the saved run had done."""
        history = []
        first = self.loops_done if self._resumed else 0
        for n in range(first + 1, first + n_loops):
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
            self.loops_done += 1
            mean_len, losses = history[-1][1], history[-1][2:]
            if print_acc and n % print_acc == 0:
                log("Loop %d | episodes %d | steps %.3f | V %.3f | rwd %.3f | Pi %.3f" % (n, self.episodes_done, mean_len, *losses))
        return history

    # -- checkpoints ---------------------------------------------------------------------------------
    def _config(self):
        return dict(N=self.N, max_steps=self.max_steps, n_games=self.B, discount=float(self.discount),
                    dirichlet_alpha=float(self.alpha), n_mcts_simulations=self.S, unroll_n_steps=self.unroll, batch_s=self.batch_s,
                    n_TD_step=self.n_step, lr=float(self.learner.lr), buffer_size=self.buffer_size,
                    priority_replay=bool(self.priority_replay), n_update_x_loop=self.n_update_x_loop,
                    moves_per_loop=self.moves_per_loop, acting_mode=int(self.acting_mode), seed=self.seed)

    def _episode_store(self):
        return self._selfplay.episodes if self.world == 1 else self._episodes

    def _live_mask(self, words):
        """bool [B, t_max]: the episode-store slots a later move can still read, those of each game's episode in flight."""
        t = torch.arange(self.max_steps, device=words.device)
        return t[None, :] < _step_counters(words, self.N)[:, None]

    def _rank0_outcome(self, error, what):
        """Every rank learns whether rank 0's part of a collective save / load failed, so that no rank goes on to a
        collective rank 0 will not join; raises rank 0's error there and a RuntimeError on the other ranks."""
        if self.world > 1:
            flag = torch.tensor([0 if error is None else 1], dtype=torch.int32, device=self.learner.device)
            dist.broadcast(flag, 0)
            if error is None and int(flag.item()):
                raise RuntimeError(f"{what} failed on rank 0")
        if error is not None:
            raise error

    def save(self, path):
        """Writes the state of the run to ``path`` (one file, loadable with torch.load(path) and its default
        weights_only=True) so that ``load`` continues it bit-identically.  Call it between two public calls
        (training_loop, play, update).  It synchronises the stream once, draws no random numbers and changes no state
        of the run.  With world > 1 it is collective: every rank calls it and rank 0 writes the file, which does not
        depend on the number of ranks."""
        if self._selfplay is None:  # nothing played yet: build the actor the next training_loop would build first
            self._refresh_actor(adjust_temperature(self.episodes_done // max(1, self.B)))
        sp = self._selfplay
        if self._gather is not None:
            self._gather.drain()
        torch.cuda.current_stream(self.learner.device).synchronize()
        # every game's env word and MinMaxStats, in global game order: int32 + 2 x float64 = 20 bytes per game
        games = torch.cat([sp.env.words.view(torch.uint8).view(-1, 4), sp.mcts.store.minmax.view(torch.uint8).view(-1, 16)], 1)
        if self.world > 1:
            gathered = torch.empty(self.world * games.numel(), dtype=torch.uint8, device=games.device)
            dist.all_gather_into_tensor(gathered, games.reshape(-1))
            games = gathered.view(self.B, 20)
        error = None
        if self.rank == 0:
            try:
                self._write(path, games)
            except Exception as e:  # re-raised on rank 0 once the other ranks know
                error = e
        self._rank0_outcome(error, f"saving {path}")

    def _write(self, path, games):
        ln, buf, st = self.learner, self.buffer, self._episode_store()
        words = games[:, :4].contiguous().view(torch.int32).view(-1)
        mask = self._live_mask(words)
        episodes = {}
        for key in EPISODE_FIELDS:
            t = getattr(st, key)
            # the G > 1 store allocates its exponents at the first ingest; before it no episode is in flight
            episodes[key] = t.transpose(0, 1)[mask].cpu() if t is not None else torch.zeros(0, dtype=torch.uint8)
        n = len(buf)
        _, key, pos, has_gauss, cached = np.random.get_state()
        ck = dict(
            version=CHECKPOINT_VERSION, config=self._config(),
            trainer=dict(loops_done=self.loops_done, episodes_done=self.episodes_done, weights_dirty=bool(self._weights_dirty),
                         replay_status=int(self._replay_status), temperature=float(self._temperature)),
            learner=dict(params=ln.params.cpu(), adam_m=ln.adam_m.cpu(), adam_v=ln.adam_v.cpu(), step_index=int(ln.step_index)),
            selfplay=dict(moves_done=int(self._selfplay.moves_done), words=words.cpu(),
                          minmax=games[:, 4:].contiguous().view(torch.float64).cpu()),
            episodes=dict(episodes, cur_slot=st.cur_slot.cpu(), ep_len=st.ep_len.cpu()),
            replay=dict(**{k: getattr(buf, k)[:n].cpu() for k in RING_FIELDS}, ptr=int(buf.ptr), is_full=bool(buf.is_full),
                        status=int(buf.status.item())),
            rng=dict(numpy=dict(key=torch.from_numpy(key.astype(np.int64)), pos=int(pos), has_gauss=int(has_gauss),
                                cached_gaussian=float(cached)),
                     torch_cuda=torch.cuda.get_rng_state(ln.device)))
        tmp = f"{path}.tmp"  # a run pre-empted while writing leaves the previous file intact
        torch.save(ck, tmp)
        os.replace(tmp, path)

    @classmethod
    def load(cls, path, device="cuda"):
        """A trainer that continues the run ``save`` wrote to ``path``: its further loops are bit-identical to those of
        the run that was saved, and training_loop numbers them on from the saved loop count.  The acting weights are
        rebuilt from the learner's parameters.  Loading sets NumPy's global RandomState and the torch CUDA generator of
        ``device``: the run draws its replay batches from the former and the padding actions of stored episodes from
        the latter, so both are part of its state.  Raises ValueError, naming the field, for a file of another format
        version or with shapes its config does not imply.  With world > 1 it is collective: rank 0 reads the file,
        every rank takes its slice of the games, and only rank 0 restores the learner's Adam state, the episode store,
        the replay ring and the random state; the number of ranks may differ from the run that saved."""
        rank, world = _world()
        dev = torch.device(device)
        ck, error = None, None
        if rank == 0:
            try:
                ck = torch.load(path, map_location="cpu")
                check_checkpoint(ck)
            except Exception as e:
                error = e
        head = None
        if rank == 0 and error is None:
            head = dict(config=ck["config"], trainer=ck["trainer"], moves_done=ck["selfplay"]["moves_done"])
        if world > 1:
            msg = [head]
            dist.broadcast_object_list(msg, 0, device=dev)
            head = msg[0]
        if head is None:
            raise error if error is not None else RuntimeError(f"loading {path} failed on rank 0")
        cfg, tr = head["config"], head["trainer"]
        n_params = sum(int(np.prod(s)) for _, s in param_shapes(cfg["N"]))
        params = ck["learner"]["params"] if rank == 0 else torch.zeros(n_params, dtype=torch.float32)
        mz = cls(split_flat(params, cfg["N"]), **cfg, device=device)
        ln = mz.learner
        if rank == 0:
            games = torch.cat([ck["selfplay"]["words"].view(torch.uint8).view(-1, 4),
                               ck["selfplay"]["minmax"].view(torch.uint8).view(-1, 16)], 1).to(ln.device)
        else:
            games = torch.empty(mz.B, 20, dtype=torch.uint8, device=ln.device)
        if world > 1:
            dist.broadcast(ln.params, 0)
            dist.broadcast(games, 0)
        mz.loops_done, mz.episodes_done, mz._replay_status = tr["loops_done"], tr["episodes_done"], tr["replay_status"]
        mz._resumed = True
        mz._refresh_actor(tr["temperature"])
        mz._weights_dirty = tr["weights_dirty"]
        sp, shard = mz._selfplay, mz.B // world
        mine = games[rank * shard:(rank + 1) * shard]
        sp.env.words.copy_(mine[:, :4].contiguous().view(torch.int32).view(-1))
        sp.mcts.store.minmax.copy_(mine[:, 4:].contiguous().view(torch.float64))
        sp.moves_done = head["moves_done"]
        if rank == 0:
            mz._restore_rank0(ck, games[:, :4].contiguous().view(torch.int32).view(-1))
        torch.cuda.current_stream(ln.device).synchronize()
        return mz

    def _restore_rank0(self, ck, words):
        """The learner's Adam state, the episode store, the replay ring and the random state: rank 0's part of load."""
        ln, buf, st = self.learner, self.buffer, self._episode_store()
        ln.adam_m.copy_(ck["learner"]["adam_m"])
        ln.adam_v.copy_(ck["learner"]["adam_v"])
        ln.step_index = ck["learner"]["step_index"]
        if st.exp is None:
            st.exp = torch.ones(self.max_steps, self.B, dtype=torch.uint8, device=st.device)
        mask = self._live_mask(words)
        for key in EPISODE_FIELDS:
            getattr(st, key).transpose(0, 1)[mask] = ck["episodes"][key].to(st.device)
        st.cur_slot.copy_(ck["episodes"]["cur_slot"])
        st.ep_len.copy_(ck["episodes"]["ep_len"])
        rp = ck["replay"]
        for key in RING_FIELDS:
            getattr(buf, key)[:rp[key].shape[0]].copy_(rp[key])
        buf.ptr, buf.is_full = rp["ptr"], rp["is_full"]
        buf.status.fill_(rp["status"])
        r = ck["rng"]["numpy"]
        np.random.set_state(("MT19937", r["key"].numpy().astype(np.uint32), r["pos"], r["has_gauss"], r["cached_gaussian"]))
        torch.cuda.set_rng_state(ck["rng"]["torch_cuda"], ln.device)

    def export_reference(self, path):
        """Writes the reference's checkpoint file (training_main.py:save_results): {"Muzero_net": the 20 MuZeroNet
        tensors on the CPU, "Net_optim": the state dict torch.optim.Adam(MuZeroNet.parameters(), lr) would hold after the
        learner's step_index steps}.  With world > 1 rank 0, which holds the learner, writes it; other ranks do nothing."""
        if self.rank != 0:
            return
        ln = self.learner
        torch.save({"Muzero_net": split_flat(ln.params.cpu(), self.N), "Net_optim": ln.optimizer_state_dict()}, path)

    @classmethod
    def from_reference(cls, path, N, max_steps, n_games, **kwargs):
        """A trainer that starts from the reference's checkpoint file (``export_reference``, or the reference's own
        muzero_model.pt): its weights, Adam moments and step count.  The learning rate is the file's; ``kwargs`` are the
        other constructor arguments.  Raises ValueError for missing or extra keys, wrong shapes, or an optimiser the
        learner's plain Adam cannot continue (weight decay, amsgrad, maximize, other betas or eps)."""
        ck = torch.load(path, map_location="cpu")
        if not isinstance(ck, dict) or set(ck) != {"Muzero_net", "Net_optim"}:
            got = sorted(ck) if isinstance(ck, dict) else type(ck).__name__
            raise ValueError(f"{path}: expected the keys ['Muzero_net', 'Net_optim'], got {got}")
        sd, shapes = ck["Muzero_net"], param_shapes(N)
        if not isinstance(sd, dict) or set(sd) != {k for k, _ in shapes}:
            got = sorted(set(sd) ^ {k for k, _ in shapes}) if isinstance(sd, dict) else type(sd).__name__
            raise ValueError(f"Muzero_net: missing or extra keys {got}")
        for key, shape in shapes:
            if not torch.is_tensor(sd[key]) or tuple(sd[key].shape) != shape:
                got = tuple(sd[key].shape) if torch.is_tensor(sd[key]) else type(sd[key]).__name__
                raise ValueError(f"Muzero_net.{key}: expected shape {shape} for N={N}, got {got}")
        adam_m, adam_v, step_index, lr, betas, eps = torch_to_adam(ck["Net_optim"], N)
        if betas != ADAM_BETAS or eps != ADAM_EPS:
            raise ValueError(f"Net_optim.param_groups[0]: betas {betas}, eps {eps}; the trainer's Adam has betas {ADAM_BETAS}, "
                             f"eps {ADAM_EPS}")
        mz = cls(sd, N, max_steps, n_games, lr=lr, **kwargs)
        mz.learner.adam_m.copy_(adam_m)
        mz.learner.adam_v.copy_(adam_v)
        mz.learner.step_index = step_index
        return mz
