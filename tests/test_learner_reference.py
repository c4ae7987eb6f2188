"""The learner step (hmz_learner_step) against a float64 reference of the same operation (oracle/learner_ref.py), element
by element, at the shapes, weights and optimiser states training reaches.

Every tensor the step produces is compared: the 20 gradients, parameters and both Adam moments after the update, the
new priorities and the three losses.  The float32 yardstick is the same reference code run in float32 on the CPU, the
precision of the reference implementation itself.  Per tensor, the kernel's |error| against float64 must stay within
GATES[c] = (c_max, c_q, floor) times the yardstick's |error| plus an absolute floor, at the maximum and at the 99.9th
percentile: k_max <= c_max (y_max + floor) and k_q999 <= c_q (y_q999 + floor).  The constants are about 3x what the
kernel measured on a B200 (DESIGN.md §4, learner).

Random inputs keep out the rows where float32 rounding can flip a discontinuity of the step (|x| of a support head
near 0, a ReLU pre-activation near 0, a near-tie of the latent's min or max; learner_ref.hazard_rows): they are
resampled until the float64 reference has none.  All-equal head logits (x = 0 exactly) have a test of their own.
"""
import numpy as np
import pytest
import torch

from oracle import learner_ref as lref
from oracle import port

from conftest import record_metric

# category -> (c_max, c_q, floor): about 3x the worst ratio measured on a B200 (1,000 W) over this file's tests and the
# 3,144 updates of tools/learner_audit.py (DESIGN.md §4): grad 5.2, param 11.4, m 5.2, v 7.6, prio 3.4, loss 21.2.
# Parameters after Adam carry the largest ratio: m / sqrt(v) turns float32 noise in a near-zero gradient into a step
# error of up to lr, at elements where kernel and yardstick round differently.  Each loss is a single number, so its
# ratio is the noisiest.
GATES = {
    "grad": (16.0, 16.0, 1e-9),
    "param": (35.0, 35.0, 1e-9),
    "m": (16.0, 16.0, 1e-10),
    "v": (23.0, 23.0, 1e-14),
    "prio": (10.0, 10.0, 1e-6),
    "loss": (64.0, 64.0, 1e-4),
}
LR = 0.002


# ---- inputs --------------------------------------------------------------------------------------------------------

def torch_default_weights(n, seed):
    from muzero_hanoi_b200.networks import MuZeroNet

    torch.manual_seed(seed)
    return {k: v.detach().numpy().copy() for k, v in MuZeroNet(3 * n, 6, LR, "cpu", TD_return=True).state_dict().items()}


def weights(regime, n, seed=7):
    """The weight regimes the step is checked under."""
    sd = torch_default_weights(n, seed) if regime == "torch" else port.make_weights(n, seed)
    if regime == "saturated":  # every head's output layer x 30: softmaxes near one-hot, v / r near +-(16 squared-ish)
        for net in ("rwd_net", "policy_net", "value_net"):
            for kind in ("weight", "bias"):
                sd[f"{net}.2.{kind}"] = sd[f"{net}.2.{kind}"] * 30
    elif regime == "flat":  # a nearly constant latent: max - min ~ 1e-6, so the 1e-8 of normalize matters
        for net in ("representation_net", "dynamic_net"):
            for kind in ("weight", "bias"):
                sd[f"{net}.2.{kind}"] = sd[f"{net}.2.{kind}"] * 1e-6
    elif regime == "ties":  # h_raw = bias exactly: its minimum and its maximum each occur three times
        bias = np.linspace(-0.5, 0.5, 64, dtype=np.float32)
        np.random.default_rng(seed).shuffle(bias)
        lo, hi = int(np.argmin(bias)), int(np.argmax(bias))
        for j in (5, 17, 40):
            bias[j if j not in (lo, hi) else j + 1] = -0.5
        for j in (9, 33, 60):
            bias[j if j not in (lo, hi) else j + 1] = 0.5
        for net in ("representation_net", "dynamic_net"):
            sd[f"{net}.2.weight"] = np.zeros_like(sd[f"{net}.2.weight"])
            sd[f"{net}.2.bias"] = bias.copy()
    elif regime == "dead":  # a quarter of every MLP's hidden units never fire
        for net in lref.MLPS:
            b = sd[f"{net}.0.bias"].copy()
            b[::4] = -100.0
            sd[f"{net}.0.bias"] = b
    return {k: np.ascontiguousarray(v, np.float32) for k, v in sd.items()}


def _rows(rng, n, B, K, pi_sum=1.0):
    states = np.stack([port.one_hot(port.index_to_state(int(i), n)) for i in rng.integers(0, 3 ** n, B)]).astype(np.float32)
    rwds = rng.choice(np.array([0.0, 100.0, -0.1], np.float32), size=(B, K), p=[0.7, 0.1, 0.2]).astype(np.float32)
    actions = rng.integers(0, 6, (B, K)).astype(np.int64)
    pi = (rng.dirichlet(np.ones(6), size=(B, K)) * pi_sum).astype(np.float32)
    returns = rng.normal(0, 20, (B, K)).astype(np.float32)
    return [states, rwds, actions, pi, returns]


def priority_weights(kind, rng, B):
    if kind is None:
        return None
    if kind == "uniform":
        return rng.uniform(0.2, 1.0, B).astype(np.float32)
    if kind == "zeros":
        w = rng.uniform(0.2, 1.0, B).astype(np.float32)
        w[::3] = 0.0
        return w
    return np.ones(B, np.float32)  # "ones": priority_sample with importance-sampling exponent 0


def synthetic_batch(params, n, B, K, seed, pi_sum=1.0, device="cuda"):
    """Golden-style random rows, with the hazard rows of the float64 reference resampled away."""
    rng = np.random.default_rng(seed)
    batch = _rows(rng, n, B, K, pi_sum)
    for _ in range(40):
        bad = lref.hazard_rows(lref.forward_backward(params, batch, None, torch.float64, device)).cpu().numpy()
        if not bad.any():
            return batch
        fresh = _rows(rng, n, int(bad.sum()), K, pi_sum)
        for a, f in zip(batch, fresh):
            a[bad] = f
    raise AssertionError(f"{int(bad.sum())} hazard rows left after resampling")


# ---- the kernel side -----------------------------------------------------------------------------------------------

def snapshot(ln):
    return dict(params={k: v.clone() for k, v in ln.state_dict().items()}, m={k: v.clone() for k, v in ln._split(ln.adam_m).items()},
                v={k: v.clone() for k, v in ln._split(ln.adam_v).items()})


def kernel_update(ln, batch, w, apply_update=True):
    new_p, v_loss, r_loss, p_loss = ln.update(*batch, w, apply_update=apply_update)
    torch.cuda.synchronize()
    out = dict(grads={k: v.clone() for k, v in ln.grad_dict().items()}, priorities=None if new_p is None else torch.from_numpy(new_p),
               losses=np.array([v_loss, r_loss, p_loss]))
    if apply_update:
        out.update(snapshot(ln))
    return out


def check_update(name, ln, batch, w, apply_update=True, **meta):
    """One kernel update from the learner's current state, held to the gates; returns the float64 StepResult."""
    before, step_index = snapshot(ln), ln.step_index + 1
    kern = kernel_update(ln, batch, w, apply_update)
    stats, ref = lref.compare_update(kern, before, step_index, batch, w, LR, ref_device="cuda", yard_device="cpu")
    worst, bad = lref.check(stats, GATES)
    record_metric(name, {**meta, **{f"{c}_ratio_max": v[0] for c, v in worst.items()}, **{f"{c}_ratio_q999": v[1] for c, v in worst.items()},
                         "failing": ",".join(bad)})
    assert not bad, (name, {b: stats[b] for b in bad[:6]})
    return ref


# ---- CPU: the reference is the reference's operation ---------------------------------------------------------------

def test_reference_reproduces_the_recorded_updates(golden):
    """Two consecutive Muzero._update calls of the unmodified reference (tests/golden/learner.npz, torch CPU float32):
    the float32 run of oracle/learner_ref.py reproduces them to float32 summation order, and the recorded float32
    values stand to the float64 run exactly as the yardstick does (the gates the kernel is held to)."""
    g = golden("learner.npz")
    n = int(g["n"])
    runs = {}
    for dt in (torch.float32, torch.float64):
        P = {k: torch.from_numpy(v).to(dt) for k, v in port.make_weights(n, int(g["weight_seed"])).items()}
        M, V = ({k: torch.zeros_like(v) for k, v in P.items()} for _ in range(2))
        res = []
        for i in range(2):
            batch = [g[f"b{i}_{k}"] for k in ("states", "rwds", "actions", "pi", "returns")]
            r, P, M, V = lref.step(P, M, V, i + 1, batch, g[f"b{i}_w"], float(g["lr"]), dt)
            res.append(r)
        runs[dt] = (res, P)
    (r32, p32), (r64, p64) = runs[torch.float32], runs[torch.float64]
    for i in range(2):
        assert np.allclose(r32[i].losses, g[f"b{i}_losses"], rtol=1e-6), (r32[i].losses, g[f"b{i}_losses"])
        assert np.allclose(r32[i].priorities.numpy(), g[f"b{i}_new_priorities"], rtol=1e-6, atol=1e-6)
    for k in lref.KEYS:
        ref = g[f"grad0_{k}"]
        assert np.abs(r32[0].grads[k].numpy() - ref).max() <= 1e-5 * np.abs(ref).max(), k
        assert np.abs(p32[k].numpy() - g[f"param2_{k}"]).max() <= 1e-5, k
    stats = {}
    for k in lref.KEYS:
        stats[f"grad:{k}"] = lref.error_stats(g[f"grad0_{k}"], r32[0].grads[k], r64[0].grads[k])
        stats[f"param:{k}"] = lref.error_stats(g[f"param2_{k}"], p32[k], p64[k])
    for i in range(2):
        stats[f"prio:{i}"] = lref.error_stats(g[f"b{i}_new_priorities"], r32[i].priorities, r64[i].priorities)
        stats[f"loss:{i}"] = lref.error_stats(g[f"b{i}_losses"], r32[i].losses, r64[i].losses)
    worst, bad = lref.check(stats, GATES)
    assert not bad, (bad, worst)


# ---- CPU: the gates are sharp --------------------------------------------------------------------------------------

MUTANTS = [
    ("hook 1.0", lref.Mutant(hook=1.0), "port", 1.0),
    ("min/max detached", lref.Mutant(detach_minmax=True), "port", 1.0),
    ("ties to the last occurrence", lref.Mutant(ties_last=True), "ties", 1.0),
    ("reward head on the normalised latent", lref.Mutant(rwd_on_normalised=True), "port", 1.0),
    ("Adam bias correction one step off", lref.Mutant(adam_step_off=1), "port", 1.0),
    ("policy gradient without sum(target)", lref.Mutant(policy_no_tsum=True), "port", 0.6),
]


@pytest.mark.parametrize("label,mut,regime,pi_sum", MUTANTS, ids=[m[0] for m in MUTANTS])
def test_gates_reject_wrong_learner_steps(label, mut, regime, pi_sum):
    """Each float64 mutant, put in place of the kernel, fails the gates; a faithful float32 step that sums in another
    order (the batch rows permuted) passes them."""
    n, B, K = 3, 64, 5
    params = weights(regime, n)
    batch = synthetic_batch(params, n, B, K, seed=11, pi_sum=pi_sum, device="cpu")
    w = priority_weights("uniform", np.random.default_rng(3), B)
    zeros = {k: torch.zeros_like(torch.from_numpy(v)) for k, v in params.items()}
    before = dict(params={k: torch.from_numpy(v) for k, v in params.items()}, m=zeros, v=zeros)

    def as_kernel(res, p, m, v):
        return dict(grads=res.grads, params=p, m=m, v=v, priorities=res.priorities, losses=res.losses)

    wrong = as_kernel(*lref.step(params, zeros, zeros, 1, batch, w, LR, torch.float64, mut=mut))
    _, bad = lref.check(lref.compare_update(wrong, before, 1, batch, w, LR)[0], GATES)
    assert bad, f"the gates accept the mutant '{label}'"
    perm = np.random.default_rng(5).permutation(B)
    faithful = as_kernel(*lref.step(params, zeros, zeros, 1, [a[perm] for a in batch], w[perm], LR, torch.float32))
    faithful["priorities"] = faithful["priorities"][np.argsort(perm)]
    worst, bad = lref.check(lref.compare_update(faithful, before, 1, batch, w, LR)[0], GATES)
    assert not bad, (bad, worst)
    print(label, "rejected by", len(bad), "tensors")


# ---- GPU: shapes, weights, priority weights ------------------------------------------------------------------------

SHAPES = ([(n, 48, 5, "uniform") for n in (1, 3, 5, 10, 11, 12)]
          + [(3, b, 5, "uniform") for b in (1, 31, 32, 33, 255, 256, 257, 1024, 4096)]
          + [(3, 64, k, "uniform") for k in (1, 2, 8)]
          + [(3, 256, 5, w) for w in (None, "zeros", "ones")])


@pytest.mark.gpu
@pytest.mark.parametrize("n,B,K,wkind", SHAPES, ids=[f"N{n}-B{b}-K{k}-w{w}" for n, b, k, w in SHAPES])
def test_update_matches_float64_across_shapes(n, B, K, wkind):
    from muzero_hanoi_b200.learner import Learner

    params = weights("port", n, seed=n)
    batch = synthetic_batch(params, n, B, K, seed=100 * n + B + K)
    w = priority_weights(wkind, np.random.default_rng(B), B)
    ln = Learner(params, n, K, lr=LR)
    check_update(f"learner_ref shape N={n} B={B} K={K} w={wkind}", ln, batch, w)


REGIMES = ["torch", "port", "saturated", "flat", "ties", "dead"]


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
def test_update_matches_float64_across_weight_regimes(regime):
    from muzero_hanoi_b200.learner import Learner

    n, B, K = 3, 256, 5
    params = weights(regime, n)
    batch = synthetic_batch(params, n, B, K, seed=21)
    w = priority_weights("uniform", np.random.default_rng(2), B)
    ln = Learner(params, n, K, lr=LR)
    check_update(f"learner_ref weights {regime}", ln, batch, w)


@pytest.mark.gpu
def test_consecutive_updates_and_a_loaded_optimiser_state():
    """Four consecutive updates, each checked from the state the kernel left; then one update from a loaded state at
    step_index 1,000 with non-trivial moments."""
    from muzero_hanoi_b200.learner import Learner

    n, B, K = 3, 256, 5
    params = weights("torch", n)
    ln = Learner(params, n, K, lr=LR)
    rng = np.random.default_rng(8)
    for i in range(4):
        batch = synthetic_batch({k: v.cpu() for k, v in ln.state_dict().items()}, n, B, K, seed=300 + i)
        check_update(f"learner_ref consecutive step {ln.step_index + 1}", ln, batch, priority_weights("uniform", rng, B))
    g = torch.Generator().manual_seed(4)
    ln.adam_m.copy_(torch.randn(ln.adam_m.shape, generator=g) * 1e-2)
    ln.adam_v.copy_(torch.rand(ln.adam_v.shape, generator=g) * 1e-4)
    ln.step_index = 999
    batch = synthetic_batch({k: v.cpu() for k, v in ln.state_dict().items()}, n, B, K, seed=400)
    check_update("learner_ref loaded state step 1000", ln, batch, priority_weights("uniform", rng, B))


@pytest.mark.gpu
def test_update_matches_float64_on_replay_rows():
    """Rows of a real ReplayRing filled by SelfPlay: one-hot states, rewards in {0, 100, -0.1}, n-step returns, visit-count
    policies and absorbing padding.  Hazard rows are dropped from the sampled batch."""
    from muzero_hanoi_b200.trainer import BatchedMuzero

    n, K = 3, 5
    params = weights("torch", n, seed=1)
    np.random.seed(1)
    mz = BatchedMuzero(params, n, 200, 256, n_mcts_simulations=25, seed=3)
    mz._refresh_actor(1.0)
    while len(mz.buffer) < 2000:
        mz.play(8)
    for label, sample in (("priority", lambda: mz.buffer.priority_sample(512)), ("uniform", lambda: mz.buffer.uniform_sample(512))):
        out = sample()
        batch, w = [t.cpu().numpy() for t in out[:5]], (out[6].cpu().numpy() if len(out) > 5 else None)
        keep = ~lref.hazard_rows(lref.forward_backward(params, batch, None, torch.float64, "cuda")).cpu().numpy()
        batch, w = [a[keep][:256] for a in batch], (None if w is None else w[keep][:256])
        assert len(batch[0]) == 256 and (batch[4].max() > 50) and set(np.unique(batch[1])) <= {0.0, 100.0, np.float32(-0.1)}
        from muzero_hanoi_b200.learner import Learner

        check_update(f"learner_ref replay rows {label}", Learner(params, n, K, lr=LR), batch, w, dropped=int((~keep).sum()))


# ---- GPU: all-equal head logits (x = 0 exactly) --------------------------------------------------------------------

@pytest.mark.gpu
def test_all_equal_head_logits_send_no_gradient():
    """Value and reward output layers whose 33 rows are equal give all-equal logits in every row.  torch's float32
    sum(softmax * linspace) gives x = 0 there, so v = r = 0, the priorities are |G_0| and neither head gets a gradient.
    The kernel must match that exactly (it used to normalise before summing, get x = -8.9e-8 and send a gradient)."""
    from muzero_hanoi_b200.learner import Learner

    n, B, K = 3, 64, 5
    params = weights("port", n)
    for net in ("value_net", "rwd_net"):
        params[f"{net}.2.weight"] = np.repeat(params[f"{net}.2.weight"][:1], 33, axis=0)
        params[f"{net}.2.bias"] = np.full(33, params[f"{net}.2.bias"][0], np.float32)
    rng = np.random.default_rng(9)
    batch = _rows(rng, n, B, K)
    w = priority_weights("uniform", rng, B)
    yard = lref.forward_backward(params, batch, w, torch.float32)
    assert float(yard.x_min.max()) == 0.0  # the float32 reference's own x is 0 in every row
    ln = Learner(params, n, K, lr=LR)
    kern = kernel_update(ln, batch, w, apply_update=False)
    for k in lref.KEYS:
        if k.startswith(("value_net", "rwd_net")):
            assert not kern["grads"][k].any(), k
            assert not yard.grads[k].any(), k
    assert torch.equal(kern["priorities"], torch.from_numpy(np.abs(batch[4][:, 0])))
    assert np.allclose(kern["losses"][:2], [np.mean((batch[4].astype(np.float64) ** 2).sum(1)), np.mean((batch[1].astype(np.float64) ** 2).sum(1))],
                       rtol=1e-6)
    ln = Learner(params, n, K, lr=LR)
    check_update("learner_ref all-equal head logits", ln, batch, w)


# ---- GPU: the kernel's contract ------------------------------------------------------------------------------------

def _raw_step(ln, batch, w, new_p, apply_update):
    dev = ln.device
    t = [torch.as_tensor(a, device=dev).contiguous() for a in batch]
    w = torch.as_tensor(w, device=dev).contiguous()
    B = t[0].shape[0]
    need = int(ln.lib.hmz_learner_workspace_bytes(ln.n_disks, B, ln.unroll))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    from muzero_hanoi_b200._lib import check, current_stream, ptr

    check(ln.lib.hmz_learner_step(ptr(ln.params), ptr(ln.grads), ptr(ln.adam_m), ptr(ln.adam_v), ptr(ws), ln.n_disks, B, ln.unroll,
                                  *(ptr(x) for x in t), ptr(w), ln.lr, ln.betas[0], ln.betas[1], ln.eps, 1, ptr(new_p),
                                  ptr(ln.losses), int(apply_update), current_stream()))
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_gradients_only_leaves_the_state_and_nothing_is_written_past_the_batch():
    from muzero_hanoi_b200.learner import Learner

    n, B, K = 3, 33, 5
    params = weights("port", n)
    batch = synthetic_batch(params, n, B, K, seed=12)
    w = priority_weights("uniform", np.random.default_rng(1), B)
    ln = Learner(params, n, K, lr=LR)
    ln.adam_m.normal_(0, 1e-3)
    ln.adam_v.uniform_(0, 1e-6)
    before = [x.clone() for x in (ln.params, ln.adam_m, ln.adam_v)]
    new_p = torch.full((B + 64,), float("nan"), device="cuda")
    _raw_step(ln, batch, w, new_p, apply_update=False)
    for a, b in zip(before, (ln.params, ln.adam_m, ln.adam_v)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert torch.isfinite(new_p[:B]).all() and torch.isnan(new_p[B:]).all()
    _raw_step(ln, batch, w, new_p, apply_update=True)
    assert not torch.equal(before[0], ln.params) and torch.isnan(new_p[B:]).all()


@pytest.mark.gpu
def test_repeat_calls_and_a_grown_workspace_are_bit_identical():
    """Two identical calls give bit-identical gradients, parameters, moments and priorities (only the three losses are
    summed with atomics); a Learner whose workspace grew for B = 4,096 gives at B = 33 exactly what a fresh one gives."""
    from muzero_hanoi_b200.learner import Learner

    n, K = 5, 5
    params = weights("torch", n)
    small = synthetic_batch(params, n, 33, K, seed=13)
    big = synthetic_batch(params, n, 4096, K, seed=14)
    w_small = priority_weights("uniform", np.random.default_rng(2), 33)
    runs = []
    for grow in (False, False, True):
        ln = Learner(params, n, K, lr=LR)
        if grow:
            ln.update(*big, priority_weights("uniform", np.random.default_rng(3), 4096), apply_update=False)
            assert ln._ws.numel() >= ln.lib.hmz_learner_workspace_bytes(n, 4096, K)
        out = kernel_update(ln, small, w_small)
        runs.append(out)
    base = runs[0]
    for other in runs[1:]:
        for part in ("grads", "params", "m", "v"):
            for k in lref.KEYS:
                assert torch.equal(base[part][k], other[part][k]), (part, k)
        assert torch.equal(base["priorities"], other["priorities"])
        assert np.allclose(base["losses"], other["losses"], rtol=1e-6)


# ---- GPU: every update of a real training run ----------------------------------------------------------------------

@pytest.mark.gpu
def test_every_update_of_a_training_run_matches_float64():
    """BatchedMuzero on N = 3 with 256 games: each learner update, from a snapshot of its batch, parameters, moments and
    step index, is checked against the one-step float64 reference."""
    from muzero_hanoi_b200.trainer import BatchedMuzero

    torch.manual_seed(1)
    np.random.seed(1)
    mz = BatchedMuzero(torch_default_weights(3, 1), 3, 200, 256, n_mcts_simulations=25, n_update_x_loop=4, seed=1)
    ln, orig, checked = mz.learner, mz.learner.update, []

    def audited(states, rwds, actions, pi_probs, returns, priority_w=None, apply_update=True):
        batch = [t.clone() for t in (states, rwds, actions, pi_probs, returns)]
        w = None if priority_w is None else priority_w.clone()
        before, step_index = snapshot(ln), ln.step_index + 1
        out = orig(states, rwds, actions, pi_probs, returns, priority_w, apply_update)
        kern = dict(grads=ln.grad_dict(), **snapshot(ln), priorities=None if out[0] is None else torch.from_numpy(out[0]),
                    losses=np.array(out[1:]))
        stats, ref = lref.compare_update(kern, before, step_index, batch, w, LR, ref_device="cuda")
        worst, bad = lref.check(stats, GATES)
        checked.append((step_index, worst, bad, int(lref.hazard_rows(ref).sum())))
        return out

    ln.update = audited
    mz.training_loop(40, min_replay_size=1000)
    assert len(checked) >= 100, len(checked)
    worst = {c: tuple(max(r[1][c][i] for r in checked) for i in (0, 1)) for c in checked[0][1]}
    record_metric("learner_ref training run", {"updates": len(checked), "hazard_rows": sum(r[3] for r in checked),
                                                **{f"{c}_ratio_max": v[0] for c, v in worst.items()},
                                                **{f"{c}_ratio_q999": v[1] for c, v in worst.items()}})
    failed = [(s, b, h) for s, _, b, h in checked if b]
    assert not failed, failed[:5]
