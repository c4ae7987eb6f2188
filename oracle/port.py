"""TEST INFRASTRUCTURE ONLY — numpy/torch restatement of the reference hot path.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module; the product never does.

Every function cites the reference file:line (under ``/root/reference``) whose
behaviour it restates.  It is written array-first (packed states, flat tree
tables) rather than object-first, so it is *not* a copy of the reference, but it
is checked bit-for-bit against the unmodified reference by ``gen_golden.py`` and
against the committed fixtures by ``tests/test_oracle_golden.py``.

Arithmetic contract reproduced here (SURVEY.md §8a, Appendix A):
  * tree statistics (W, Q, min/max, backed-up value) are IEEE float64,
  * Q and U terms are rounded to float32 before the add and the arg-max,
  * ``prior * w`` is a float32 product when the prior is float32 (NumPy >= 2
    weak-scalar promotion) and a float64 product at a Dirichlet-noised root,
  * network inference is float32 torch on one row at a time.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

# action index -> (from peg, to peg); env/hanoi.py:39-41 (itertools.permutations(range(3), 2))
MOVES = ((0, 1), (0, 2), (1, 0), (1, 2), (2, 0), (2, 1))
N_ACTIONS = 6
PB_C_BASE = 19652  # MCTS/mcts.py:24
PB_C_INIT = 1.25  # MCTS/mcts.py:25
REWARD_GOAL = 100  # env/hanoi.py:66
REWARD_ILLEGAL = -100 / 1000  # env/hanoi.py:72  (python double, != float32(-0.1))

# flag bits returned by step_packed (shared with include/hmz.h)
FLAG_DONE = 1
FLAG_ILLEGAL = 2
FLAG_GOAL = 4
FLAG_TRUNC = 8


# --------------------------------------------------------------------------- env
def state_to_packed(state) -> int:
    """tuple (peg of disk 0 .. N-1, disk 0 smallest) -> 2 bits per disk; env/hanoi.py:19-25."""
    w = 0
    for d, p in enumerate(state):
        w |= int(p) << (2 * d)
    return w


def packed_to_state(word: int, n_disks: int) -> tuple:
    return tuple((word >> (2 * d)) & 3 for d in range(n_disks))


def index_to_state(idx: int, n_disks: int) -> tuple:
    """env/hanoi.py:23-25: states = itertools.product(range(3), repeat=N) — disk 0 is the
    MOST significant base-3 digit of the index."""
    out = [0] * n_disks
    for d in range(n_disks - 1, -1, -1):
        out[d] = idx % 3
        idx //= 3
    return tuple(out)


def state_to_index(state) -> int:
    idx = 0
    for p in state:
        idx = idx * 3 + int(p)
    return idx


def top_disk(state, peg):
    """Smallest disk index on ``peg`` or None; env/hanoi.py:117-121 (+ min() in :135,:144)."""
    for d, p in enumerate(state):
        if p == peg:
            return d
    return None


def move_allowed(state, move) -> bool:
    """env/hanoi.py:123-139."""
    f, t = move
    tf = top_disk(state, f)
    if tf is None:
        return False
    tt = top_disk(state, t)
    return True if tt is None else tt > tf


def legal_mask(state) -> int:
    m = 0
    for a, mv in enumerate(MOVES):
        if move_allowed(state, mv):
            m |= 1 << a
    return m


def one_hot(state, n_pegs=3) -> np.ndarray:
    """utils.py:9-25: float64[3N], disk-major."""
    out = np.zeros((len(state), n_pegs))
    out[np.arange(len(state)), list(state)] = 1
    return out.reshape(-1)


def hanoi_solver(state, goal_peg=2) -> int:
    """env/hanoi_utils.py:4-26: minimal number of moves to stack everything on goal_peg."""
    moves, target = 0, goal_peg
    for i in range(len(state) - 1, -1, -1):
        if state[i] != target:
            moves += 1 << i
            target = 3 - target - state[i]
    return moves


def step_state(state, step_counter, action, max_steps, goal):
    """Pure-function form of TowersOfHanoi.step (env/hanoi.py:47-84).

    Returns (obs_state, stored_state, new_counter, reward, done, illegal, reset_check).
    ``obs_state`` is what the returned one-hot encodes; ``stored_state`` is the env's
    ``c_state`` afterwards (NOT updated when the goal is reached, :65-69)."""
    move = MOVES[action]
    illegal = not move_allowed(state, move)
    step_counter += 1  # :56 — counted for illegal moves too
    reset_check = True
    if not illegal:
        tf = top_disk(state, move[0])
        moved = list(state)
        moved[tf] = move[1]
        moved = tuple(moved)
        if moved != goal:
            rwd, done, stored = 0, False, moved
        else:
            rwd, done, stored = REWARD_GOAL, True, state
            reset_check, step_counter = False, 0
    else:
        rwd, moved, done, stored = REWARD_ILLEGAL, state, False, state
    if step_counter == max_steps:  # :77-80
        done, reset_check, step_counter = True, False, 0
    return moved, stored, step_counter, rwd, done, illegal, reset_check


class PortHanoi:
    """Stateful restatement of env.hanoi.TowersOfHanoi (env/hanoi.py:11-151), same surface."""

    def __init__(self, N, max_steps, init_state_idx=0, goal_peg=2):
        self.discs, self.n_pegs = N, 3
        self.oneH_s_size = 3 * N
        self.goal = (goal_peg,) * N
        self.init_state_idx = init_state_idx
        self.moves = list(MOVES)
        self.max_steps = max_steps
        self.reset_check = False
        self.step_counter = 0

    def reset(self):
        self.reset_check = True
        self.c_state = index_to_state(self.init_state_idx, self.discs)
        self.oneH_c_state = one_hot(self.c_state)
        return self.oneH_c_state

    def random_reset(self, rng=np.random):
        """env/hanoi.py:98-111 — rejection-sample a non-goal state index."""
        self.reset_check = True
        while True:
            idx = rng.randint(3 ** self.discs)
            self.c_state = index_to_state(idx, self.discs)
            if self.c_state != self.goal:
                break
        self.oneH_c_state = one_hot(self.c_state)
        return self.oneH_c_state

    def current_state(self):
        return list(self.c_state)

    def _move_allowed(self, move):
        """env/hanoi.py:123-139 on the current state."""
        return move_allowed(self.c_state, move)

    def step(self, action):
        assert self.reset_check, "Need to reset env before taking a step"
        moved, stored, ctr, rwd, done, illegal, rc = step_state(
            self.c_state, self.step_counter, action, self.max_steps, self.goal
        )
        self.c_state, self.step_counter, self.reset_check = stored, ctr, rc
        return one_hot(moved), rwd, done, illegal


# ----------------------------------------------------------------------- network
def make_weights(n_disks: int, seed: int, hidden=256, latent=64, support=33, actions=6):
    """Deterministic synthetic MuZeroNet weights (state_dict layout of networks.py:39-67).

    Drawn with numpy's Generator (stream-stable across numpy versions) rather than torch's
    default init so that fixtures do not depend on the torch version.  Bounds follow the
    nn.Linear default, U(-1/sqrt(fan_in), 1/sqrt(fan_in))."""
    rng = np.random.default_rng(seed)
    shapes = {
        "representation_net": (3 * n_disks, hidden, latent),
        "dynamic_net": (latent + actions, hidden, latent),
        "rwd_net": (latent, hidden, support),
        "policy_net": (latent, hidden, actions),
        "value_net": (latent, hidden, support),
    }
    sd = {}
    for name, (i, h, o) in shapes.items():
        for idx, (fan_in, fan_out) in (("0", (i, h)), ("2", (h, o))):
            k = 1.0 / math.sqrt(fan_in)
            sd[f"{name}.{idx}.weight"] = rng.uniform(-k, k, (fan_out, fan_in)).astype(np.float32)
            sd[f"{name}.{idx}.bias"] = rng.uniform(-k, k, (fan_out,)).astype(np.float32)
    return sd


def lesion_weights(sd, heads, seed, latent=64):
    """Restates networks.py:201-205 + acting_ablations.py:29-45: re-draw every Linear weight
    and bias of the named heads from U(-k, k), k = sqrt(1/latent) (numpy stream, see above)."""
    rng = np.random.default_rng(seed)
    k = float(np.sqrt(1 / latent))
    out = dict(sd)
    for head in heads:
        for idx in ("0", "2"):
            for kind in ("weight", "bias"):
                key = f"{head}.{idx}.{kind}"
                out[key] = rng.uniform(-k, k, sd[key].shape).astype(np.float32)
    return out


class PortNet:
    """Functional float32 torch restatement of MuZeroNet inference (networks.py:71-196).

    One row at a time through ``torch.nn.functional.linear`` — the same primitive the
    reference's nn.Linear dispatches to — so outputs are bit-identical to the reference in
    the same container (checked by gen_golden.py)."""

    def __init__(self, state_dict, support_size=33):
        import torch

        self.torch = torch
        self.sd = {k: torch.as_tensor(np.asarray(v), dtype=torch.float32) for k, v in state_dict.items()}
        self.support_size = support_size
        self.num_actions = self.sd["policy_net.2.weight"].shape[0]

    def _mlp(self, name, x):
        F = self.torch.nn.functional
        x = F.relu(F.linear(x, self.sd[f"{name}.0.weight"], self.sd[f"{name}.0.bias"]))
        return F.linear(x, self.sd[f"{name}.2.weight"], self.sd[f"{name}.2.bias"])

    def _support_to_scalar(self, logits, eps=1e-3):
        """networks.py:152-189: softmax -> expectation over linspace(-16,16,33) -> signed parabolic."""
        t = self.torch
        if self.support_size == 1:
            return logits
        half = (self.support_size - 1) // 2
        probs = t.softmax(logits, dim=-1)
        support = t.linspace(-half, half, self.support_size).expand_as(probs)
        x = t.sum(probs * support, dim=-1, keepdim=True)
        z = t.sqrt(1 + 4 * eps * (eps + 1 + t.abs(x))) / 2 / eps - 1 / 2 / eps
        return t.sign(x) * (t.square(z) - 1)

    def _normalize(self, h):
        """networks.py:191-196."""
        lo = h.min(dim=-1, keepdim=True)[0]
        hi = h.max(dim=-1, keepdim=True)[0]
        return (h - lo) / (hi - lo + 1e-8)

    def represent(self, x):
        return self._normalize(self._mlp("representation_net", x))

    def dynamics(self, h, a_onehot):
        """networks.py:129-138 — the reward head reads the UN-normalised new latent."""
        raw = self._mlp("dynamic_net", self.torch.cat([h, a_onehot], dim=-1))
        r = self._support_to_scalar(self._mlp("rwd_net", raw))
        return self._normalize(raw), r

    def prediction(self, h):
        return self._mlp("policy_net", h), self._support_to_scalar(self._mlp("value_net", h))

    def initial_inference(self, x):
        """networks.py:71-94 -> (np.f32[64], 0.0, np.f32[6], float)."""
        t = self.torch
        with t.no_grad():
            h = self.represent(x)
            logits, v = self.prediction(h)
            p = t.nn.functional.softmax(logits, dim=-1)
            return h.squeeze(0).numpy(), 0.0, p.squeeze(0).numpy(), v.squeeze(0).item()

    def recurrent_inference(self, h, a_onehot):
        """networks.py:96-116."""
        t = self.torch
        with t.no_grad():
            h2, r = self.dynamics(h, a_onehot)
            logits, v = self.prediction(h2)
            p = t.nn.functional.softmax(logits, dim=-1)
            return h2.squeeze(0).numpy(), r.squeeze(0).item(), p.squeeze(0).numpy(), v.squeeze(0).item()


# ------------------------------------------------------------------------ search
def ucb_table(n_max: int) -> np.ndarray:
    """TABLE[n] = (log((n + c_base + 1)/c_base) + c_init) * sqrt(n), float64 through libm
    exactly as MCTS/node.py:114-120 evaluates it (left to right; the /(child.N+1) comes after)."""
    return np.array(
        [(math.log((n + PB_C_BASE + 1) / PB_C_BASE) + PB_C_INIT) * math.sqrt(n) for n in range(n_max + 1)],
        dtype=np.float64,
    )


@dataclass
class MinMax:
    """MCTS/utils_mcts.py:1-16 — starts at (+inf, -inf), lives as long as its MCTS object."""

    minimum: float = float("inf")
    maximum: float = -float("inf")

    def update(self, v):
        self.maximum = max(self.maximum, v)
        self.minimum = min(self.minimum, v)

    def normalize(self, v):
        if self.maximum > self.minimum:
            return (v - self.minimum) / (self.maximum - self.minimum)
        return v


def play_policy(visits, temperature):
    """MCTS/mcts.py:154-176."""
    if not 0.0 <= temperature <= 1.0:
        raise ValueError(f"Expect `temperature` to be in the range [0.0, 1.0], got {temperature}")
    v = np.asarray(visits, dtype=np.int64)
    if temperature > 0.0:
        v = np.power(v, max(1.0, min(5.0, 1.0 / temperature)))
    return v / np.sum(v)


def sample_action(pi, u):
    """np.random.choice(6, p=pi) with its single uniform draw ``u`` supplied
    (MCTS/mcts.py:120; Generator-free legacy path: cdf = cumsum(p); cdf /= cdf[-1];
    idx = cdf.searchsorted(u, side='right'))."""
    cdf = np.cumsum(pi)
    cdf /= cdf[-1]
    return int(cdf.searchsorted(u, side="right"))


def mix_dirichlet(prior_f32, noise_f64, eps=0.25):
    """MCTS/mcts.py:148-150 with the Dirichlet draw supplied: (1-eps)*prob is a float32
    product (weak python scalar), the sum with eps*noise promotes to float64."""
    return (1 - eps) * prior_f32 + eps * noise_f64


@dataclass
class SearchTrace:
    actions_path: list = field(default_factory=list)  # per simulation: list of actions root->leaf
    r: list = field(default_factory=list)
    p: list = field(default_factory=list)
    v: list = field(default_factory=list)
    h: list = field(default_factory=list)


class PortSearch:
    """Array-based restatement of MCTS.run_mcts + Node (MCTS/mcts.py:34-126, MCTS/node.py:30-136).

    Expanded node e owns 6 child slots; the node expanded by simulation s gets index s+1
    (root = 0), which is also the layout of the GPU tree store.  Tie-break is lowest index
    (the sanctioned parity hook replacing MCTS/node.py:86)."""

    def __init__(self, discount, n_simulations, minmax: MinMax | None = None):
        self.discount = discount
        self.n_simulations = n_simulations
        self.minmax = minmax if minmax is not None else MinMax()

    def run(self, root_prior, root_h, infer, *, injected=None, trace: SearchTrace | None = None):
        """root_prior: np.float32[6] or np.float64[6] (noised).  ``infer(parent_h, action)`` ->
        (h', r, p f32[6], v) is called once per simulation unless ``injected`` =
        (r[S], p[S,6], v[S]) is given.  Returns (child_N int32[6], root_Q, root_W)."""
        S, g, mm = self.n_simulations, self.discount, self.minmax
        E = S + 1
        table = ucb_table(S + 1)
        prior_is_f64 = np.asarray(root_prior).dtype == np.float64
        cN = np.zeros((E, 6), dtype=np.int64)
        cW = np.zeros((E, 6), dtype=np.float64)
        cR = np.zeros((E, 6), dtype=np.float64)  # child.rwd (a float32 value widened)
        cP = np.zeros((E, 6), dtype=np.float64)
        cP[0] = np.asarray(root_prior, dtype=np.float64)
        cE = -np.ones((E, 6), dtype=np.int64)  # expanded-node index of child or -1
        hs = [None] * E
        hs[0] = root_h
        root_N, root_W = 0, 0.0
        for s in range(S):
            e, n_parent, path = 0, root_N, []
            while True:
                best, best_score = 0, None
                for a in range(6):
                    n = int(cN[e, a])
                    if n > 0:
                        q = mm.normalize(cR[e, a] + g * (cW[e, a] / n))  # node.py:99
                    else:
                        q = 0
                    w = table[n_parent] / (n + 1)  # node.py:114-121
                    if e == 0 and prior_is_f64:
                        u = np.float32(cP[e, a] * w)  # float64 product (noised root)
                    else:
                        u = np.float32(np.float32(cP[e, a]) * np.float32(w))  # NEP-50 f32 product
                    score = np.float32(q) + u  # node.py:83 float32 add
                    if best_score is None or score > best_score:
                        best, best_score = a, score
                path.append((e, best))
                nxt = int(cE[e, best])
                if nxt < 0:
                    break
                n_parent = int(cN[e, best])
                e = nxt
            pe, pa = path[-1]
            if injected is None:
                h2, r, p, v = infer(hs[pe], pa)
            else:
                h2, r, p, v = None, float(injected[0][s]), injected[1][s], float(injected[2][s])
            new = s + 1
            hs[new] = h2
            cE[pe, pa] = new
            cR[pe, pa] = float(r)
            cP[new] = np.asarray(p, dtype=np.float64)
            if trace is not None:
                trace.actions_path.append([a for _, a in path])
                trace.r.append(np.float32(r)); trace.p.append(np.asarray(p, dtype=np.float32))
                trace.v.append(np.float32(v)); trace.h.append(h2)
            value = float(v)
            for (e_i, a_i) in reversed(path):  # node.py:62-70, leaf first
                cW[e_i, a_i] += value
                cN[e_i, a_i] += 1
                mm.update(cR[e_i, a_i] + g * (cW[e_i, a_i] / int(cN[e_i, a_i])))
                value = cR[e_i, a_i] + g * value
            root_W += value
            root_N += 1
            mm.update(0.0 + g * (root_W / root_N))  # the root's own rwd is 0.0 (mcts.py:69)
        return cN[0].astype(np.int32), (root_W / root_N if root_N else 0.0), root_W


def run_mcts_port(obs, net: PortNet, search: PortSearch, temperature, deterministic, *, alpha=0.25,
                  eps=0.25, noise=None, u=None, trace=None):
    """MCTS.run_mcts (MCTS/mcts.py:34-126) over PortNet/PortSearch with the sanctioned hooks:
    Dirichlet draw ``noise`` (f64[6]) and sampling uniform ``u`` supplied by the caller."""
    import torch

    x = torch.from_numpy(np.asarray(obs)).to(dtype=torch.float32)
    h0, _, p0, _ = net.initial_inference(x)
    prior = p0
    if not deterministic and alpha > 0.0 and eps > 0.0:
        prior = mix_dirichlet(p0, noise, eps)

    def infer(h, a):
        onehot = torch.zeros(net.num_actions, dtype=torch.float32)
        onehot[a] = 1.0
        return net.recurrent_inference(torch.from_numpy(h).to(dtype=torch.float32), onehot)

    visits, root_q, _ = search.run(prior, h0, infer, trace=trace)
    pi = play_policy(visits, temperature)
    action = int(np.argmax(visits)) if deterministic else sample_action(pi, u)
    return action, pi, root_q, visits, prior


# ------------------------------------------------------- trajectory post-processing (§8f row 1)
def py312_sum(terms):
    """Python >= 3.12 ``sum()`` over floats: the first add goes through the generic int + float path,
    the rest through Neumaier compensated summation (CPython Python/bltinmodule.c) — the reference's
    ``sum([...])`` at utils.py:64-66 therefore is NOT a plain left-to-right float64 sum."""
    if not terms:
        return 0
    f, c = 0 + float(terms[0]), 0.0
    for x in terms[1:]:
        x = float(x)
        t = f + x
        if abs(f) >= abs(x):
            c += (f - t) + x
        else:
            c += (x - t) + f
        f = t
    if c and math.isfinite(c):
        f += c
    return f


def n_step_returns(rwds, root_values, n_step, discount):
    """utils.py:28-72 (n-step TD targets; zeros beyond the end of the episode)."""
    T = len(rwds)
    r = list(rwds) + [0] * n_step
    q = list(root_values) + [0] * n_step
    out = []
    for t in range(T):
        acc = py312_sum([discount ** i * x for i, x in enumerate(r[t:t + n_step])])
        out.append(acc + discount ** n_step * q[t + n_step])
    return out


def mc_returns(rwds, discount):
    """utils.py:75-86 (compute_MCreturns): discounted reward-to-go through NumPy's flip / cumsum / divide."""
    T = len(rwds)
    # np.power(float, int array): NumPy's own (SIMD) pow, which differs from libm pow() in the last bit for some
    # exponents — the table has to come from NumPy itself; element i does not depend on the array length
    disc = [float(x) for x in discount ** np.arange(T)]
    acc, out = 0.0, [0.0] * T
    for t in range(T - 1, -1, -1):  # np.cumsum over the flipped array: sequential float64 adds from the end
        x = disc[t] * float(rwds[t])
        acc = x if t == T - 1 else acc + x
        out[t] = acc / disc[t]
    return out


def priorities(returns, root_values):
    """Muzero.py:197-200: |float32(return) - float32(root value)|."""
    return np.abs(np.array(returns, dtype=np.float32) - np.array(root_values, dtype=np.float32))


def organise_transitions(states, rwds, actions, pi_probs, returns, unroll, n_action, absorbing_action):
    """Muzero.organise_transitions (Muzero.py:276-323): every step gets its next `unroll` rewards /
    actions / policies / returns; beyond the end of the episode the padding is reward 0, return 0,
    the uniform policy and ONE absorbing action (drawn once per call by the caller, :300-303)."""
    n = len(states)
    rwds = list(rwds) + [0] * unroll
    actions = list(actions) + [absorbing_action] * unroll
    returns = list(returns) + [0] * unroll
    uniform = np.ones_like(pi_probs[-1]) / len(pi_probs[-1])
    pi_probs = list(pi_probs) + [uniform] * unroll
    o_r = np.zeros((n, unroll), np.float32)
    o_a = np.zeros((n, unroll), np.int64)
    o_p = np.zeros((n, unroll, n_action), np.float32)
    o_g = np.zeros((n, unroll), np.float32)
    for i in range(n):
        o_r[i] = rwds[i:i + unroll]
        o_a[i] = actions[i:i + unroll]
        o_p[i] = pi_probs[i:i + unroll]
        o_g[i] = returns[i:i + unroll]
    return np.array(states), o_r, o_a, o_p, o_g
