"""Batched engines over libhmz.so: VecHanoi (env), PackedWeights, BatchedMCTS, SelfPlay.

These are the batched additions SURVEY.md §8b names; the reference-shaped classes in
``env/``, ``MCTS/`` and ``networks.py`` are thin B=1 views over them.  torch is used for device
memory and streams only; every computation is a libhmz kernel.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr

MOVES = ((0, 1), (0, 2), (1, 0), (1, 2), (2, 0), (2, 1))  # env/hanoi.py:39-41


# ----------------------------------------------------------------------- packing helpers
def pack_state(state) -> int:
    """tuple(peg of disk d) -> env word state bits (2 bits per disk, disk 0 lowest)."""
    w = 0
    for d, p in enumerate(state):
        w |= (int(p) & 3) << (2 * d)
    return w


def unpack_state(word: int, n_disks: int) -> tuple:
    return tuple((int(word) >> (2 * d)) & 3 for d in range(n_disks))


def state_index(state) -> int:
    """Index into itertools.product(range(3), repeat=N) (disk 0 most significant)."""
    idx = 0
    for p in state:
        idx = idx * 3 + int(p)
    return idx


def index_state(idx: int, n_disks: int) -> tuple:
    out = [0] * n_disks
    for d in range(n_disks - 1, -1, -1):
        out[d] = idx % 3
        idx //= 3
    return tuple(out)


def check_env_shape(n_disks: int, max_steps: int):
    if not 1 <= n_disks <= _lib.MAX_DISKS:
        raise ValueError(f"N={n_disks} unsupported: the packed env word holds 1..{_lib.MAX_DISKS} disks")
    if not 1 <= max_steps < (1 << (32 - 2 * n_disks)):
        raise ValueError(f"max_steps={max_steps} does not fit the {32 - 2 * n_disks} counter bits of the env word")


class VecHanoi:
    """B Tower-of-Hanoi environments stepped in lock-step on the GPU.

    State lives in one int32 tensor ``words`` (bit layout in include/hmz.h).  Semantics are
    those of TowersOfHanoi.step (reference env/hanoi.py:47-84) per env, bit-exact."""

    def __init__(self, N, max_steps, B, device="cuda", init_state_idx=0, goal_peg=2, auto_reset=True):
        _lib.require_cuda()
        check_env_shape(N, max_steps)
        self.lib = _lib.load()
        self.discs, self.max_steps, self.B, self.goal_peg = N, max_steps, int(B), goal_peg
        self.device = torch.device(device)
        self.init_state_idx = init_state_idx
        self.auto_reset = bool(auto_reset)
        self.words = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        self.rewards = torch.empty(self.B, dtype=torch.float32, device=self.device)
        self.flags = torch.empty(self.B, dtype=torch.uint8, device=self.device)
        self.obs_words = torch.empty(self.B, dtype=torch.int32, device=self.device)
        self.actions = torch.empty(self.B, dtype=torch.uint8, device=self.device)
        self._counters = torch.zeros(4, dtype=torch.int64, device=self.device)

    @property
    def reset_word(self) -> int:
        return pack_state(index_state(self.init_state_idx, self.discs))

    @property
    def goal_word(self) -> int:
        return pack_state((self.goal_peg,) * self.discs)

    def reset(self):
        check(self.lib.hmz_env_reset(ptr(self.words), self.B, self.reset_word, current_stream()))
        return self.words

    def set_state_indices(self, indices):
        idx = torch.as_tensor(indices, dtype=torch.int32, device=self.device).contiguous()
        assert idx.numel() == self.B
        check(self.lib.hmz_env_from_index(ptr(idx), ptr(self.words), self.B, self.discs, current_stream()))
        return self.words

    def state_indices(self):
        out = torch.empty(self.B, dtype=torch.int32, device=self.device)
        check(self.lib.hmz_env_to_index(ptr(self.words), ptr(out), self.B, self.discs, current_stream()))
        return out

    def random_reset(self, seed=0, counter=0):
        check(self.lib.hmz_env_random_reset(ptr(self.words), self.B, self.discs, self.goal_peg, seed, counter,
                                            current_stream()))
        return self.words

    def step(self, actions, want_obs=True):
        """actions: uint8 tensor [B] on the device.  Returns (obs_words|None, rewards, flags)."""
        a = actions if actions.dtype == torch.uint8 else actions.to(torch.uint8)
        check(self.lib.hmz_env_step(ptr(self.words), ptr(a), ptr(self.rewards), ptr(self.flags),
                                    ptr(self.obs_words) if want_obs else None, self.B, self.discs, self.max_steps,
                                    self.goal_peg, int(self.auto_reset), self.reset_word, current_stream()))
        return (self.obs_words if want_obs else None), self.rewards, self.flags

    def step_random(self, seed=0, step_index=0):
        check(self.lib.hmz_env_step_random(ptr(self.words), ptr(self.actions), ptr(self.rewards), ptr(self.flags),
                                           self.B, self.discs, self.max_steps, self.goal_peg, self.reset_word, seed,
                                           step_index, current_stream()))
        return self.actions, self.rewards, self.flags

    def rollout_random(self, n_steps, seed=0, step_index=0):
        """n_steps fused random-legal-move steps; returns the int64[4] device counters
        (steps, goals, truncations, xor checksum), accumulated since construction."""
        check(self.lib.hmz_env_rollout_random(ptr(self.words), self.B, self.discs, self.max_steps, self.goal_peg,
                                              self.reset_word, n_steps, seed, step_index, ptr(self._counters),
                                              current_stream()))
        return self._counters

    def legal_mask(self):
        out = torch.empty(self.B, dtype=torch.uint8, device=self.device)
        check(self.lib.hmz_env_legal_mask(ptr(self.words), ptr(out), self.B, self.discs, current_stream()))
        return out

    def onehot(self, words=None):
        w = self.words if words is None else words
        out = torch.empty(w.numel(), 3 * self.discs, dtype=torch.float32, device=self.device)
        check(self.lib.hmz_env_onehot(ptr(w), ptr(out), w.numel(), self.discs, current_stream()))
        return out

    def solver_distance(self, words=None):
        w = self.words if words is None else words
        out = torch.empty(w.numel(), dtype=torch.int32, device=self.device)
        check(self.lib.hmz_env_solver_distance(ptr(w), ptr(out), w.numel(), self.discs, self.goal_peg,
                                               current_stream()))
        return out

    def states(self):
        """Host view: (state bits [B] uint32, step counters [B])."""
        w = self.words.cpu().numpy().view(np.uint32)
        shift = 2 * self.discs
        return w & ((1 << shift) - 1), w >> shift


# ------------------------------------------------------------------------------- search
def ucb_table(n_max: int) -> np.ndarray:
    """TABLE[n] = (log((n + 19652 + 1)/19652) + 1.25) * sqrt(n) for n in [0, n_max], float64 via the
    host libm in the reference's own evaluation order (MCTS/node.py:114-120); the per-child
    division by (child.N + 1) happens on the device.  Only the integer parent count enters, so a
    host table removes any device-vs-glibc log() ulp question from the bit-exact path."""
    return np.array([(math.log((n + 19652 + 1) / 19652) + 1.25) * math.sqrt(n) for n in range(n_max + 1)],
                    dtype=np.float64)


class SearchStore:
    """Device buffers of B concurrent searches with room for ``n_records`` expanded nodes each
    (struct hmz_search_t).  MinMaxStats state persists until ``reset_minmax``."""

    def __init__(self, B, n_records, device="cuda", latent_dtype=_lib.LATENT_F32):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.B, self.n_records, self.latent_dtype = int(B), int(n_records), latent_dtype
        self.device = torch.device(device)
        dev = self.device
        self.nodes = torch.zeros(max(1, self.B * self.n_records * 128), dtype=torch.uint8, device=dev)
        assert self.nodes.data_ptr() % 128 == 0
        ldt = torch.float32 if latent_dtype == _lib.LATENT_F32 else torch.bfloat16
        self.latents = torch.zeros(self.B, self.n_records, _lib.LATENT, dtype=ldt, device=dev)
        self.root_prior = torch.zeros(self.B, 6, dtype=torch.float64, device=dev)
        self.root_W = torch.zeros(self.B, dtype=torch.float64, device=dev)
        self.minmax = torch.zeros(self.B, 2, dtype=torch.float64, device=dev)
        self.workspace = torch.zeros(int(self.lib.hmz_search_workspace_bytes(self.B)), dtype=torch.uint8, device=dev)
        self.desc = _lib.SearchDesc(
            nodes=self.nodes.data_ptr(), latents=self.latents.data_ptr(), root_prior=self.root_prior.data_ptr(),
            root_W=self.root_W.data_ptr(), minmax=self.minmax.data_ptr(), workspace=self.workspace.data_ptr(),
            capture=None, n_searches=self.B, n_records=self.n_records, latent_dtype=latent_dtype, root_prior_is_f64=0,
            schedule=_lib.SCHEDULE_AUTO)
        self.reset_minmax()

    def reset_minmax(self):
        check(self.lib.hmz_search_minmax_reset(ptr(self.minmax), self.B, current_stream()))

    def set_schedule(self, schedule):
        """How hmz_search_run schedules its kernels (never changes results): 0 = automatic, k in [1, 16] = one launch
        pair per simulation over k concurrent stream groups, _lib.SCHEDULE_PERSISTENT = one persistent kernel,
        _lib.SCHEDULE_SERVER | k = resident network CTAs fed by ordinary tree-kernel launches in k stream groups."""
        self.desc.schedule = int(schedule)

    def enable_capture(self, n_simulations):
        """Parity tests: hmz_search_run records [p0..p5, r, v] of every simulation in the returned float32
        [n_simulations, B, 8] tensor (until disable_capture)."""
        self.capture = torch.zeros(int(n_simulations), self.B, 8, dtype=torch.float32, device=self.device)
        self.desc.capture = self.capture.data_ptr()
        return self.capture

    def disable_capture(self):
        self.capture, self.desc.capture = None, None

    def records(self):
        """Host copy of the node records as a dict of numpy arrays indexed [search, record, action]
        (W, rwd, N, child, prior) and [search, record] (parent, parent_action)."""
        slot = np.dtype([("W", "<f8"), ("rwd", "<f4"), ("N", "<u2"), ("child", "<u2")])
        half = np.dtype([("c", slot, 3), ("prior", "<f4", 3), ("parent", "<u2"), ("parent_action", "u1"), ("pad", "u1")])
        raw = self.nodes.cpu().numpy()[: self.B * self.n_records * 128].view(half).reshape(self.B, self.n_records, 2)
        out = {k: raw["c"][k].reshape(self.B, self.n_records, 6) for k in ("W", "rwd", "N", "child")}
        out["prior"] = raw["prior"].reshape(self.B, self.n_records, 6)
        out["parent"], out["parent_action"] = raw["parent"][:, :, 0], raw["parent_action"][:, :, 0]
        return out


class BatchedMCTS:
    """B independent MCTS searches advanced in lock-step (MCTS.run_mcts, MCTS/mcts.py:34-126)."""

    def __init__(self, discount, root_dirichlet_alpha, n_simulations, B, device="cuda", root_exploration_eps=0.25,
                 latent_dtype=_lib.LATENT_F32, max_simulations=None):
        self.discount = float(discount)
        self.root_dirichlet_alpha = root_dirichlet_alpha
        self.root_exploration_eps = root_exploration_eps
        self.n_simulations = int(n_simulations)
        self.B = int(B)
        cap = max(self.n_simulations, int(max_simulations or 0))
        self.store = SearchStore(B, cap + 1, device, latent_dtype)
        self.lib = self.store.lib
        self.device = self.store.device
        self._table_host = ucb_table(cap + 1)
        self._table = torch.from_numpy(self._table_host).to(self.device)
        dev = self.device
        self.leaf_parent = torch.zeros(self.B, dtype=torch.int16, device=dev)
        self.leaf_action = torch.zeros(self.B, dtype=torch.uint8, device=dev)
        self.leaf_depth = torch.zeros(self.B, dtype=torch.int16, device=dev)
        self.visits = torch.zeros(self.B, 6, dtype=torch.int32, device=dev)
        self.pi = torch.zeros(self.B, 6, dtype=torch.float64, device=dev)
        self.root_q = torch.zeros(self.B, dtype=torch.float64, device=dev)
        self.action = torch.zeros(self.B, dtype=torch.int32, device=dev)

    # -- split phases (used by the injected parity path and by tests) ---------------------------
    def begin(self, root_prior, prior_is_f64):
        rp = torch.as_tensor(np.asarray(root_prior, dtype=np.float64) if not torch.is_tensor(root_prior) else root_prior,
                             dtype=torch.float64, device=self.device).contiguous()
        assert rp.shape == (self.B, 6)
        self.store.desc.root_prior_is_f64 = int(bool(prior_is_f64))
        check(self.lib.hmz_search_begin(C.byref(self.store.desc), ptr(rp), current_stream()))

    def select(self, sim, path_out=None):
        cap = 0 if path_out is None else path_out.shape[1]
        check(self.lib.hmz_search_select(C.byref(self.store.desc), sim, ptr(self._table), self.discount,
                                         ptr(self.leaf_parent), ptr(self.leaf_action), ptr(self.leaf_depth),
                                         ptr(path_out), cap, current_stream()))

    def expand_backup(self, sim, r, p, v):
        check(self.lib.hmz_search_expand_backup(C.byref(self.store.desc), sim, self.discount, ptr(self.leaf_parent),
                                                ptr(self.leaf_action), ptr(r), ptr(p), ptr(v), current_stream()))

    def root_policy(self, temperature, deterministic, uniforms=None, n_simulations=None):
        if not 0.0 <= temperature <= 1.0:  # MCTS/mcts.py:163-166
            raise ValueError(f"Expect `temperature` to be in the range [0.0, 1.0], got {temperature}")
        u = None
        if not deterministic:
            if uniforms is None:
                raise ValueError("sampling the action needs one uniform per search (`uniforms`)")
            u = torch.as_tensor(uniforms, dtype=torch.float64, device=self.device).contiguous()
        n = self.n_simulations if n_simulations is None else n_simulations
        check(self.lib.hmz_search_root_policy(C.byref(self.store.desc), n, float(temperature), int(bool(deterministic)),
                                              ptr(u), ptr(self._pow_table(temperature, n)), ptr(self.visits), ptr(self.pi),
                                              ptr(self.root_q), ptr(self.action), current_stream()))
        return self.action, self.pi, self.root_q, self.visits

    def _pow_table(self, temperature, n):
        """Optional caller-supplied powers for generate_play_policy (hmz_search_root_policy's pow_table): None by default.
        Integer exponents (every temperature of the reference's schedule: 1, 2, 5) are exact on the device and identical to
        NumPy while the power stays below 2^53.  For non-integer exponents NumPy's own np.power is not reproducible to the
        last bit — its SIMD body and scalar head / tail round differently, so the result of the reference's 6-element call
        depends on the array's memory alignment — and the device's pow() (<= 2 ulp) is as close to it as NumPy is to itself;
        ``self.pow_table`` (float64 [n + 1, 6] device tensor) lets a caller pin the powers explicitly."""
        return getattr(self, "pow_table", None)

    def run_injected(self, root_prior, prior_is_f64, r, p, v, want_paths=False):
        """Search with the network outputs of every simulation supplied (parity mode of
        BASELINE.json north_star): r, v float32 [S, B]; p float32 [S, B, 6]."""
        S = self.n_simulations
        dev = self.device
        r = torch.as_tensor(r, dtype=torch.float32, device=dev).contiguous()
        v = torch.as_tensor(v, dtype=torch.float32, device=dev).contiguous()
        p = torch.as_tensor(p, dtype=torch.float32, device=dev).contiguous()
        assert r.shape == (S, self.B) and v.shape == (S, self.B) and p.shape == (S, self.B, 6)
        self.begin(root_prior, prior_is_f64)
        paths = depths = None
        if want_paths:
            paths = torch.full((S, self.B, S + 1), 255, dtype=torch.uint8, device=dev)
            depths = torch.zeros(S, self.B, dtype=torch.int16, device=dev)
        for s in range(S):
            self.select(s, None if paths is None else paths[s])
            if depths is not None:
                depths[s].copy_(self.leaf_depth)
            self.expand_backup(s, r[s], p[s], v[s])
        return paths, depths


# ------------------------------------------------------------------------------ weights
STATE_DICT_ORDER = [f"{net}.{idx}.{kind}" for net in ("representation_net", "dynamic_net", "rwd_net", "policy_net",
                                                      "value_net") for idx in ("0", "2") for kind in ("weight", "bias")]


class PackedWeights:
    """Device blob of a MuZeroNet state_dict in kernel layout (hmz_weights_pack).  Accepts a
    state_dict of torch tensors or numpy arrays with the 20 keys of networks.py:39-67."""

    def __init__(self, state_dict, n_disks, mode=_lib.MODE_FP32, device="cuda"):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.n_disks, self.mode = int(n_disks), int(mode)
        self.device = torch.device(device)
        self.blob = torch.from_numpy(pack_host(state_dict, self.n_disks, self.mode)).to(self.device)
        self.ptr = C.c_void_p(self.blob.data_ptr())

    def initial(self, n, *, words=None, obs=None, latents_out, out_rows_per_item, latent_dtype, p0, v0):
        check(self.lib.hmz_net_initial(self.ptr, self.mode, self.n_disks, ptr(words), ptr(obs), ptr(latents_out),
                                       out_rows_per_item, latent_dtype, ptr(p0), ptr(v0), n, current_stream()))

    def recurrent(self, n, *, latents_in, in_rows_per_item, in_row, actions, latents_out, out_rows_per_item, out_row,
                  latent_dtype, r, p, v):
        check(self.lib.hmz_net_recurrent(self.ptr, self.mode, ptr(latents_in), in_rows_per_item, ptr(in_row),
                                         ptr(actions), ptr(latents_out), out_rows_per_item, out_row, latent_dtype,
                                         ptr(r), ptr(p), ptr(v), n, current_stream()))


def pack_host(state_dict, n_disks, mode):
    """hmz_weights_pack of a MuZeroNet state_dict (torch tensors or numpy arrays): the packed blob as host uint8."""
    lib = _lib.load()
    arrays = []
    for key in STATE_DICT_ORDER:
        t = state_dict[key]
        a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
        arrays.append(np.ascontiguousarray(a, dtype=np.float32))
    expect = {"representation_net.0.weight": (256, 3 * n_disks), "dynamic_net.0.weight": (256, 70),
              "rwd_net.2.weight": (33, 256), "policy_net.2.weight": (6, 256), "value_net.2.weight": (33, 256)}
    for key, shape in expect.items():
        got = arrays[STATE_DICT_ORDER.index(key)].shape
        if got != shape:
            raise ValueError(f"{key}: expected shape {shape}, got {got} (TD_return=True nets with h1_s=256, "
                             "reprs_output_size=64 are supported)")
    nbytes = int(lib.hmz_weights_packed_bytes(int(n_disks), int(mode)))
    if nbytes <= 0:
        raise _lib.HmzError(_lib.ERR_UNSUPPORTED, f"no packed layout for n_disks={n_disks}, mode={mode}")
    host = np.zeros(nbytes, dtype=np.uint8)
    table = (C.c_void_p * 20)(*[a.ctypes.data for a in arrays])
    check(lib.hmz_weights_pack(table, int(n_disks), int(mode), host.ctypes.data))
    return host


class WeightSets:
    """Several networks in ONE blob, set k at byte k * stride (hmz_multi_t): the weights of a search batch whose 256-search
    blocks each play with their own network.  ``nets``: state_dicts and / or PackedWeights of the same n_disks and mode.
    stride = hmz_weights_packed_bytes rounded up to a multiple of 256; the bytes between two sets are zero."""

    def __init__(self, nets, n_disks, mode=_lib.MODE_FP32, device="cuda"):
        self.lib = _lib.load()
        self.n_disks, self.mode, self.n_sets = int(n_disks), int(mode), len(nets)
        if self.n_sets < 1:
            raise ValueError("WeightSets needs at least one network")
        self.device = torch.device(device)
        nbytes = int(self.lib.hmz_weights_packed_bytes(self.n_disks, self.mode))
        if nbytes <= 0:
            raise _lib.HmzError(_lib.ERR_UNSUPPORTED, f"no packed layout for n_disks={n_disks}, mode={mode}")
        self.set_bytes = nbytes
        self.stride = (nbytes + 255) // 256 * 256
        self.blob = torch.zeros(self.n_sets * self.stride, dtype=torch.uint8, device=self.device)
        for k, net in enumerate(nets):
            if isinstance(net, PackedWeights):
                if (net.n_disks, net.mode) != (self.n_disks, self.mode):
                    raise ValueError(f"set {k}: packed for n_disks={net.n_disks}, mode={net.mode}, not {self.n_disks}, {self.mode}")
                src = net.blob
            else:
                src = torch.from_numpy(pack_host(net, self.n_disks, self.mode))
            self.blob[k * self.stride: k * self.stride + nbytes].copy_(src)
        self.ptr = C.c_void_p(self.blob.data_ptr())

    def desc(self, block_set, budget=None, host_block_budget=None):
        """hmz_multi_t over these sets: block_set int16 device [B / 256], budget int16 device [B] (simulations per search),
        host_block_budget int32 numpy [B / 256] (non-increasing).  The caller keeps the arrays alive."""
        return _lib.MultiDesc(block_set=block_set.data_ptr(), budget=budget.data_ptr() if budget is not None else None,
                              host_block_budget=host_block_budget.ctypes.data if host_block_budget is not None else None,
                              weight_stride=self.stride, n_sets=self.n_sets, n_disks=self.n_disks)

    def initial(self, n, md, *, words, latents_out, out_rows_per_item, latent_dtype, p0, v0):
        check(self.lib.hmz_net_initial_multi(self.ptr, C.byref(md), self.mode, ptr(words), ptr(latents_out), out_rows_per_item,
                                             latent_dtype, ptr(p0), ptr(v0), n, current_stream()))


def mix_dirichlet(prior_f32: np.ndarray, noise_f64: np.ndarray, eps=0.25) -> np.ndarray:
    """add_dirichlet_noise arithmetic (MCTS/mcts.py:148-150) with the draw supplied: the
    (1-eps)*prob product stays float32 (weak python scalar), the sum promotes to float64."""
    return (1 - eps) * np.asarray(prior_f32, dtype=np.float32) + eps * np.asarray(noise_f64, dtype=np.float64)


def _run_mcts(self, weights: PackedWeights, *, words=None, obs=None, temperature=1.0, deterministic=False, noise=None,
              uniforms=None):
    """MCTS.run_mcts for B searches (MCTS/mcts.py:34-126): root inference, optional Dirichlet mix
    (noise float64 [B,6] supplied by the caller), n_simulations fused simulations, root policy.
    Returns device tensors (action int32 [B], pi float64 [B,6], root_q float64 [B], visits int32 [B,6])."""
    if not 0.0 <= temperature <= 1.0:
        raise ValueError(f"Expect `temperature` to be in the range [0.0, 1.0], got {temperature}")
    st = self.store
    p0 = torch.empty(self.B, 6, dtype=torch.float32, device=self.device)
    v0 = torch.empty(self.B, dtype=torch.float32, device=self.device)
    weights.initial(self.B, words=words, obs=obs, latents_out=st.latents, out_rows_per_item=st.n_records,
                    latent_dtype=st.latent_dtype, p0=p0, v0=v0)
    use_noise = (not deterministic) and self.root_dirichlet_alpha > 0.0 and self.root_exploration_eps > 0.0
    nz = None
    if use_noise:
        if noise is None:
            raise ValueError("Dirichlet noise is an input of the batched engine (`noise`, float64 [B,6])")
        nz = torch.as_tensor(noise, dtype=torch.float64, device=self.device).contiguous()
        assert nz.shape == (self.B, 6)
    self.p0, self.v0 = p0, v0
    st.desc.root_prior_is_f64 = int(use_noise)
    check(self.lib.hmz_search_begin_p0(C.byref(st.desc), ptr(p0), ptr(nz), float(self.root_exploration_eps),
                                       current_stream()))
    check(self.lib.hmz_search_run(C.byref(st.desc), weights.ptr, weights.mode, self.n_simulations, ptr(self._table),
                                  self.discount, current_stream()))
    return self.root_policy(temperature, deterministic, uniforms)


BatchedMCTS.run_mcts = _run_mcts


class MultiMCTS:
    """B searches (a multiple of 256) over several networks and simulation budgets in ONE launch sequence
    (hmz_search_run_multi): block k of 256 searches plays with weight set block_set[k], search b runs budget[b] simulations.
    Each search computes exactly what BatchedMCTS.run_mcts with its own network and n_simulations = budget[b] computes.
    Searches [0, n) of the store take part in a call, so a caller can drop finished blocks by compacting them away."""

    def __init__(self, discount, root_dirichlet_alpha, max_simulations, B, device="cuda", root_exploration_eps=0.25,
                 latent_dtype=_lib.LATENT_F32):
        if int(B) % _lib.BLOCK:
            raise ValueError(f"B={B} is not a multiple of {_lib.BLOCK}")
        self.discount = float(discount)
        self.root_dirichlet_alpha = root_dirichlet_alpha
        self.root_exploration_eps = root_exploration_eps
        self.max_simulations, self.B = int(max_simulations), int(B)
        self.store = SearchStore(B, self.max_simulations + 1, device, latent_dtype)
        self.lib, self.device = self.store.lib, self.store.device
        self._table = torch.from_numpy(ucb_table(self.max_simulations + 1)).to(self.device)
        dev = self.device
        self.p0 = torch.empty(self.B, 6, dtype=torch.float32, device=dev)
        self.v0 = torch.empty(self.B, dtype=torch.float32, device=dev)
        self.visits = torch.zeros(self.B, 6, dtype=torch.int32, device=dev)
        self.pi = torch.zeros(self.B, 6, dtype=torch.float64, device=dev)
        self.root_q = torch.zeros(self.B, dtype=torch.float64, device=dev)
        self.action = torch.zeros(self.B, dtype=torch.int32, device=dev)

    def run_mcts(self, sets: WeightSets, md, n, *, words, temperature=1.0, deterministic=False, noise=None, uniforms=None,
                 pow_table=None):
        """MCTS.run_mcts for searches [0, n) (n a multiple of 256): root inference with each block's network, optional
        Dirichlet mix, the fused heterogeneous search, root policy with root_q = root_W / budget.  md: sets.desc(...) of the
        n searches.  Returns device views [n] of (action, pi, root_q, visits)."""
        if not 0.0 <= temperature <= 1.0:
            raise ValueError(f"Expect `temperature` to be in the range [0.0, 1.0], got {temperature}")
        n = int(n)
        st = self.store
        st.desc.n_searches = n
        try:
            sets.initial(n, md, words=words, latents_out=st.latents, out_rows_per_item=st.n_records, latent_dtype=st.latent_dtype,
                         p0=self.p0, v0=self.v0)
            use_noise = (not deterministic) and self.root_dirichlet_alpha > 0.0 and self.root_exploration_eps > 0.0
            if use_noise and noise is None:
                raise ValueError("Dirichlet noise is an input of the batched engine (`noise`, float64 [n,6])")
            st.desc.root_prior_is_f64 = int(use_noise)
            check(self.lib.hmz_search_begin_p0(C.byref(st.desc), ptr(self.p0), ptr(noise) if use_noise else None,
                                               float(self.root_exploration_eps), current_stream()))
            check(self.lib.hmz_search_run_multi(C.byref(st.desc), C.byref(md), sets.ptr, sets.mode, ptr(self._table), self.discount,
                                                current_stream()))
            check(self.lib.hmz_search_root_policy_multi(C.byref(st.desc), C.byref(md), float(temperature), int(bool(deterministic)),
                                                        ptr(uniforms), ptr(pow_table), ptr(self.visits), ptr(self.pi),
                                                        ptr(self.root_q), ptr(self.action), current_stream()))
        finally:
            st.desc.n_searches = st.B
        return self.action[:n], self.pi[:n], self.root_q[:n], self.visits[:n]


# ---------------------------------------------------------------------------- self-play
class SelfPlay:
    """B games of Muzero._play_game (reference Muzero.py:153-207) advanced one move at a time,
    entirely on device: root inference -> Dirichlet mix -> n_simulations fused simulations ->
    root policy + sampled action -> trajectory record -> env step with auto-reset.

    Throughput mode: the Dirichlet draw and the sampling uniform come from on-device Philox
    streams (parity mode = BatchedMCTS.run_mcts with those supplied as inputs).  Finished-move
    records land in a [ring_slots, B] struct-of-arrays ring that `gather` all-gathers over NCCL."""

    def __init__(self, N, max_steps, B, n_simulations, weights: PackedWeights, discount=0.8, alpha=0.25, eps=0.25,
                 temperature=1.0, seed=0, ring_slots=8, device="cuda", latent_dtype=_lib.LATENT_F32, episodes=False,
                 game_offset=0):
        self.env = VecHanoi(N, max_steps, B, device)
        self.mcts = BatchedMCTS(discount, alpha, n_simulations, B, device, eps, latent_dtype)
        self.weights, self.temperature, self.seed = weights, float(temperature), int(seed)
        self.B, self.S, self.T = int(B), int(n_simulations), int(ring_slots)
        # global id of this batch's first game: keys the Philox streams, so that a game draws the same noise and
        # uniforms whichever rank (and whichever position in the rank's batch) plays it (SURVEY.md §8e)
        self.game_offset = int(game_offset)
        self.lib, self.device = self.env.lib, self.env.device
        dev = self.device
        self.p0 = torch.empty(B, 6, dtype=torch.float32, device=dev)
        self.v0 = torch.empty(B, dtype=torch.float32, device=dev)
        self.noise = torch.empty(B, 6, dtype=torch.float64, device=dev)
        self.uniform = torch.empty(B, dtype=torch.float64, device=dev)
        # trajectory ring: [slot][game] 32-byte move records (hmz_move_record_t) = the wire format of dist.RecordGather
        self.records = torch.zeros(self.T, B, _lib.RECORD_BYTES, dtype=torch.uint8, device=dev)
        self.moves_done = 0
        # episodes=True additionally keeps whole episodes (slot = the game's own step counter) for the
        # device-side post-processing of replay.EpisodeStore / ReplayRing (SURVEY §8f rows 1-2)
        self.episodes = None
        if episodes:
            from .replay import EpisodeStore

            self.episodes = EpisodeStore(B, max_steps, N, device)
            self.episodes.exp = torch.ones(max_steps, B, dtype=torch.uint8, device=dev)
        self.env.reset()

    def move(self):
        """One move of every game (hmz_selfplay_move: one C call, no host sync); returns the ring slot that was written."""
        env, m, st = self.env, self.mcts, self.mcts.store
        t, ctr = self.moves_done % self.T, self.moves_done
        use_noise = m.root_dirichlet_alpha > 0.0 and m.root_exploration_eps > 0.0
        st.desc.root_prior_is_f64 = int(use_noise)
        ep = self.episodes
        pw = m._pow_table(self.temperature, self.S)
        d = _lib.SelfPlayDesc(
            search=st.desc, weights=self.weights.ptr.value, ucb_table=m._table.data_ptr(), words=env.words.data_ptr(),
            p0=self.p0.data_ptr(), v0=self.v0.data_ptr(), noise=self.noise.data_ptr() if use_noise else None,
            uniform=self.uniform.data_ptr(), visits=m.visits.data_ptr(), root_q=m.root_q.data_ptr(), action=m.action.data_ptr(),
            records=self.records[t].data_ptr(),
            ep_state=ep.state.data_ptr() if ep else None, ep_action=ep.action.data_ptr() if ep else None,
            ep_flags=ep.flags.data_ptr() if ep else None, ep_visits=ep.visits.data_ptr() if ep else None,
            ep_root_q=ep.root_q.data_ptr() if ep else None, ep_cur_slot=ep.cur_slot.data_ptr() if ep else None,
            ep_len=ep.ep_len.data_ptr() if ep else None, ep_exp=ep.exp.data_ptr() if ep else None, pow_table=pw.data_ptr() if pw is not None else None,
            discount=m.discount, dirichlet_alpha=float(m.root_dirichlet_alpha),
            exploration_eps=float(m.root_exploration_eps), temperature=self.temperature, seed=self.seed,
            game_offset=self.game_offset, mode=self.weights.mode,
            n_disks=env.discs, max_steps=env.max_steps, goal_peg=env.goal_peg, n_simulations=self.S,
            ep_t_max=ep.t_max if ep else 0, reset_word=env.reset_word, reserved=0)
        check(self.lib.hmz_selfplay_move(C.byref(d), ctr, current_stream()))
        self.moves_done += 1
        return t

    def record_bytes_per_game(self):
        return _lib.RECORD_BYTES

    def slot(self, t):
        """The move records written by the move that returned ``t``: uint8 [B, 32] (decode with dist.unpack_records)."""
        return self.records[t]
