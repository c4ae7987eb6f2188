"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.npz by EXECUTING the unmodified
reference (dev container only; needs /root/reference).  Run:  python -m oracle.gen_golden

Each fixture records what the reference itself returned; while generating, the numpy/torch
port (oracle/port.py) is checked bit-for-bit against the reference on the same inputs, so a
green run pins the oracle to the reference as it executes under the versions written to
tests/golden/MANIFEST.json.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import port  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
REWARD_CODE = {0: 0, 100: 1, -100 / 1000: 2}


def savez_lzma(path, arrays):
    """np.savez with LZMA members instead of deflate (np.load reads either): the N=10 tables stay well under 1 MB."""
    import zipfile

    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            with z.open(name + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


# ------------------------------------------------------------------ env + solver
def gen_env_tables(ref):
    out = {}
    max_steps = 200
    for n in (3, 4, 5, 7, 10):
        env = ref.TowersOfHanoi(N=n, max_steps=max_steps)
        n_states = 3 ** n
        variants = (0, 1) if n <= 7 else (0,)
        shape = (len(variants), n_states, 6)
        obs_idx = np.zeros(shape, np.uint32)
        stored_idx = np.zeros(shape, np.uint32)
        rcode = np.zeros(shape, np.uint8)
        done = np.zeros(shape, np.uint8)
        illegal = np.zeros(shape, np.uint8)
        ctr_after = np.zeros(shape, np.uint16)
        reset_check = np.zeros(shape, np.uint8)
        solver = np.zeros(n_states, np.uint16)
        legal = np.zeros(n_states, np.uint8)
        for vi, hit_max in enumerate(variants):
            for si in range(n_states):
                st = env.states[si]
                assert port.index_to_state(si, n) == st and port.state_to_index(st) == si
                for a in range(6):
                    env.c_state, env.reset_check = st, True
                    env.step_counter = max_steps - 1 if hit_max else 17
                    obs, r, d, ill = env.step(a)
                    obs_state = tuple(int(x) for x in obs.reshape(n, 3).argmax(1))
                    assert obs.dtype == np.float64 and np.array_equal(obs, port.one_hot(obs_state))
                    obs_idx[vi, si, a] = port.state_to_index(obs_state)
                    stored_idx[vi, si, a] = port.state_to_index(env.c_state)
                    rcode[vi, si, a] = REWARD_CODE[r]
                    done[vi, si, a], illegal[vi, si, a] = d, ill
                    ctr_after[vi, si, a], reset_check[vi, si, a] = env.step_counter, env.reset_check
                    # port == reference
                    moved, stored, c2, r2, d2, i2, rc2 = port.step_state(
                        st, max_steps - 1 if hit_max else 17, a, max_steps, env.goal)
                    assert (moved, stored, c2, d2, i2, rc2) == (obs_state, env.c_state, env.step_counter, d, ill, env.reset_check)
                    assert r2 == r and type(r2) is type(r)
                    if vi == 0:
                        env.c_state = st
                        if env._move_allowed(env.moves[a]):
                            legal[si] |= 1 << a
                if vi == 0:
                    solver[si] = ref.hanoi_solver(st)
                    assert port.hanoi_solver(st) == solver[si] and port.legal_mask(st) == legal[si]
        for k, v in dict(obs_idx=obs_idx, stored_idx=stored_idx, reward_code=rcode, done=done, illegal=illegal,
                         counter_after=ctr_after, reset_check=reset_check, solver=solver, legal=legal).items():
            out[f"n{n}_{k}"] = v
        print(f"env table N={n}: {n_states * 6 * len(variants)} transitions ok")
    out["max_steps"] = np.int64(max_steps)
    out["counter_before"] = np.array([17, max_steps - 1])
    savez_lzma(os.path.join(GOLDEN, "env_tables.npz"), out)
    # known-answer anchors quoted by the reference (acting_ablations.py:53-60, generate_all_figures.py:78)
    assert [ref.hanoi_solver(s) for s in ((2, 2, 0), (0, 0, 2), (1, 2, 2), (0, 0, 0))] == [7, 3, 1, 7]


# ------------------------------------------------------------------------ search
SEARCH_CONFIGS = {
    # name: N, S, alpha, temperature, deterministic, weight seed, lesion heads, n searches
    "n3_s50_noise_t1": dict(N=3, S=50, alpha=0.25, T=1.0, det=False, wseed=0, lesion=(), K=12),
    "n3_s25_nonoise_t0": dict(N=3, S=25, alpha=0.0, T=0.0, det=False, wseed=1, lesion=(), K=12),
    "n3_s25_det": dict(N=3, S=25, alpha=0.25, T=1.0, det=True, wseed=2, lesion=(), K=6),
    "n4_s200_lesion_t0": dict(N=4, S=200, alpha=0.0, T=0.0, det=False, wseed=3,
                              lesion=("policy_net", "value_net"), K=6),
    "n5_s100_noise_t05": dict(N=5, S=100, alpha=0.25, T=0.5, det=False, wseed=4, lesion=(), K=8),
    # the temperature of episodes >= 750 (utils.py:89-96): exponent 5, np.power(int64, 5.0) (MCTS/mcts.py:170-174)
    "n3_s50_noise_t01": dict(N=3, S=50, alpha=0.25, T=0.1, det=False, wseed=5, lesion=(), K=12),
    # a non-integer exponent (1 / 0.4 = 2.5): NumPy's pow() on the visit counts
    "n4_s60_noise_t04": dict(N=4, S=60, alpha=0.25, T=0.4, det=False, wseed=6, lesion=(), K=8),
}
DISCOUNT = 0.8


def gen_search(ref, name, cfg):
    import torch

    n, S, K = cfg["N"], cfg["S"], cfg["K"]
    sd = port.make_weights(n, cfg["wseed"])
    if cfg["lesion"]:
        sd = port.lesion_weights(sd, cfg["lesion"], seed=100 + cfg["wseed"])
    net = rh.TracingNet(rh.load_reference_net(ref, n, sd))
    pnet = port.PortNet(sd)
    rng = np.random.default_rng(1000 + cfg["wseed"])
    noises = rng.dirichlet(np.full(6, 0.25), size=K)  # f64[K,6]
    uniforms = rng.random(K)
    env = ref.TowersOfHanoi(N=n, max_steps=200)
    mcts = ref.MCTS(discount=DISCOUNT, root_dirichlet_alpha=cfg["alpha"], n_simulations=S, batch_s=1, device="cpu")
    pmm = port.MinMax()
    psearch = port.PortSearch(DISCOUNT, S, pmm)
    use_noise = (not cfg["det"]) and cfg["alpha"] > 0
    maxd = S + 1
    rec = dict(obs=[], state=[], p0=[], v0=[], h0=[], prior=[], depth=[], path=[], r=[], p=[], v=[],
               child_N=[], pi=[], root_q=[], action=[], mm_min=[], mm_max=[], env_reward=[], env_done=[])
    obs = env.reset()
    with rh.HookedSearch(ref, noises=[x for x in noises] if use_noise else [], uniforms=list(uniforms)) as hk:
        for k in range(K):
            state = tuple(env.current_state())
            u_used = None if cfg["det"] else uniforms[k] if not use_noise or True else None
            action, pi, root_q = mcts.run_mcts(obs, net, cfg["T"], cfg["det"])
            h0, _, p0, v0 = net.root
            prior = port.mix_dirichlet(p0, noises[k]) if use_noise else p0
            depth = np.zeros(S, np.uint16)
            path = np.full((S, maxd), 255, np.uint8)
            for s, (pth, _) in enumerate(net.calls):
                depth[s] = len(pth)
                path[s, : len(pth)] = pth
            r = np.array([c[1][1] for c in net.calls], np.float32)
            p = np.stack([c[1][2] for c in net.calls]).astype(np.float32)
            v = np.array([c[1][3] for c in net.calls], np.float32)
            assert all(float(np.float32(c[1][1])) == c[1][1] and float(np.float32(c[1][3])) == c[1][3] for c in net.calls)
            # --- port vs reference, full (own network) and injected
            tr = port.SearchTrace()
            mm_before = (pmm.minimum, pmm.maximum)
            a2, pi2, q2, visits2, prior2 = port.run_mcts_port(
                obs, pnet, psearch, cfg["T"], cfg["det"], alpha=cfg["alpha"], noise=noises[k],
                u=None if cfg["det"] else uniforms[k], trace=tr)
            assert np.array_equal(prior2, prior) and prior2.dtype == prior.dtype
            assert a2 == action and np.array_equal(pi2, pi) and q2 == root_q, (name, k)
            assert (pmm.minimum, pmm.maximum) == (mcts.min_max_stats.minimum, mcts.min_max_stats.maximum)
            assert [list(x) for x in tr.actions_path] == [c[0] for c in net.calls]
            assert np.array_equal(np.array(tr.r, np.float32), r) and np.array_equal(np.stack(tr.p), p)
            inj = port.PortSearch(DISCOUNT, S, port.MinMax(*mm_before))
            visits3, q3, _ = inj.run(prior, None, None, injected=(r, p, v))
            assert np.array_equal(visits3, visits2) and q3 == root_q
            rec["obs"].append(obs.copy()); rec["state"].append(port.state_to_packed(state))
            rec["p0"].append(p0); rec["v0"].append(np.float32(v0)); rec["h0"].append(h0); rec["prior"].append(np.asarray(prior, np.float64))
            rec["depth"].append(depth); rec["path"].append(path[:, : int(depth.max())].copy())
            rec["r"].append(r); rec["p"].append(p); rec["v"].append(v)
            rec["child_N"].append(visits2); rec["pi"].append(pi); rec["root_q"].append(root_q); rec["action"].append(action)
            rec["mm_min"].append(pmm.minimum); rec["mm_max"].append(pmm.maximum)
            obs, rwd, done, _ = env.step(action)
            rec["env_reward"].append(float(rwd)); rec["env_done"].append(done)
            if done:
                obs = env.reset()
    maxdepth = max(x.shape[1] for x in rec["path"])
    paths = np.full((K, S, maxdepth), 255, np.uint8)
    for k, x in enumerate(rec["path"]):
        paths[k, :, : x.shape[1]] = x
    out = dict(
        N=n, S=S, K=K, discount=DISCOUNT, alpha=cfg["alpha"], eps=0.25, temperature=cfg["T"],
        deterministic=cfg["det"], weight_seed=cfg["wseed"], lesion=np.array(cfg["lesion"], dtype="U16"),
        lesion_seed=100 + cfg["wseed"], prior_is_f64=use_noise,
        noise=noises, uniform=uniforms, obs=np.stack(rec["obs"]), state=np.array(rec["state"], np.uint32),
        p0=np.stack(rec["p0"]), v0=np.array(rec["v0"], np.float32), h0=np.stack(rec["h0"]),
        prior=np.stack(rec["prior"]), depth=np.stack(rec["depth"]), path=paths,
        r=np.stack(rec["r"]), p=np.stack(rec["p"]), v=np.stack(rec["v"]),
        child_N=np.stack(rec["child_N"]).astype(np.int32), pi=np.stack(rec["pi"]),
        root_q=np.array(rec["root_q"], np.float64), action=np.array(rec["action"], np.int32),
        mm_min=np.array(rec["mm_min"], np.float64), mm_max=np.array(rec["mm_max"], np.float64),
        env_reward=np.array(rec["env_reward"]), env_done=np.array(rec["env_done"]),
    )
    np.savez_compressed(os.path.join(GOLDEN, f"search_{name}.npz"), **out)
    print(f"search {name}: {K} searches x {S} sims ok; mean depth {np.mean([d.mean() for d in rec['depth']]):.2f}, "
          f"max {max(int(d.max()) for d in rec['depth'])}")


# ----------------------------------------------------------------------- network
def gen_net_io(ref):
    import torch

    out = {}
    for n, wseed in ((3, 0), (5, 4), (10, 7)):
        sd = port.make_weights(n, wseed)
        net = rh.load_reference_net(ref, n, sd)
        pnet = port.PortNet(sd)
        rng = np.random.default_rng(50 + n)
        M = 96
        h_in = rng.random((M, 64), dtype=np.float32)
        acts = rng.integers(0, 6, M)
        states = rng.integers(0, 3 ** n, M)
        rec = dict(h2=[], r=[], p=[], v=[], h0=[], p0=[], v0=[])
        for i in range(M):
            a1 = torch.zeros(6); a1[acts[i]] = 1.0
            h2, r, p, v = net.recurrent_inference(torch.from_numpy(h_in[i]), a1)
            q = pnet.recurrent_inference(torch.from_numpy(h_in[i]), a1)
            assert np.array_equal(q[0], h2) and q[1] == r and np.array_equal(q[2], p) and q[3] == v
            rec["h2"].append(h2); rec["r"].append(r); rec["p"].append(p); rec["v"].append(v)
            obs = port.one_hot(port.index_to_state(int(states[i]), n))
            x = torch.from_numpy(obs).to(dtype=torch.float32)
            h0, r0, p0, v0 = net.initial_inference(x)
            q = pnet.initial_inference(x)
            assert r0 == 0.0 and np.array_equal(q[0], h0) and np.array_equal(q[2], p0) and q[3] == v0
            rec["h0"].append(h0); rec["p0"].append(p0); rec["v0"].append(v0)
        out.update({f"n{n}_weight_seed": wseed, f"n{n}_h_in": h_in, f"n{n}_action": acts.astype(np.int32),
                    f"n{n}_state_idx": states.astype(np.int64),
                    f"n{n}_h_out": np.stack(rec["h2"]), f"n{n}_r": np.array(rec["r"], np.float32),
                    f"n{n}_p": np.stack(rec["p"]), f"n{n}_v": np.array(rec["v"], np.float32),
                    f"n{n}_h0": np.stack(rec["h0"]), f"n{n}_p0": np.stack(rec["p0"]),
                    f"n{n}_v0": np.array(rec["v0"], np.float32)})
        print(f"net io N={n}: {M} recurrent + {M} initial inferences ok")
    # scalar transform anchors (SURVEY §8a a22)
    net = rh.load_reference_net(ref, 3, port.make_weights(3, 0))
    xs = torch.tensor([[-16.0], [-1.0], [0.0], [0.5], [16.0]])
    out["signed_parabolic_in"] = xs.numpy()
    out["signed_parabolic_out"] = net._signed_parabolic(xs).numpy()
    np.savez_compressed(os.path.join(GOLDEN, "net_io.npz"), **out)


def gen_episode_post(ref):
    """Episode post-processing of Muzero._play_game (Muzero.py:189-205): n-step returns, priorities,
    organise_transitions — reference functions on random synthetic episodes."""
    import types

    sys.path.insert(0, rh.REFERENCE_ROOT)
    import Muzero as ref_muzero  # noqa: E402  (imports cleanly behind the plotting stubs)

    rng = np.random.default_rng(77)
    out, n_step, discount, unroll = {}, 10, 0.8, 5
    lengths = [1, 2, 5, 7, 11, 24, 60, 200]
    for k, T in enumerate(lengths):
        codes = rng.choice(3, size=T, p=[0.75, 0.0, 0.25])  # 0: legal (0), 2: illegal (-0.1)
        if k % 2 == 0:
            codes[-1] = 1  # solved episode: reward 100 on the last move
        rw = [{0: 0, 1: 100, 2: -100 / 1000}[int(c)] for c in codes]
        visits = rng.multinomial(100, rng.dirichlet(np.ones(6)), size=T)
        pis = [port.play_policy(v, 1.0) for v in visits]
        root_q = [float(x) for x in rng.normal(0, 20, T)]
        actions = [int(a) for a in rng.integers(0, 6, T)]
        states = [port.one_hot(port.index_to_state(int(i), 5)) for i in rng.integers(0, 242, T)]
        returns = ref.compute_n_step_returns(rw, root_q, n_step, discount)
        assert returns == port.n_step_returns(rw, root_q, n_step, discount), "port n-step returns != reference"
        prio = np.abs(np.array(returns, dtype=np.float32) - np.array(root_q, dtype=np.float32))
        assert np.array_equal(prio, port.priorities(returns, root_q))
        mc = ref.compute_MCreturns(rw, discount)  # the TD_return=False branch of Muzero._play_game (Muzero.py:193-194)
        assert [float(x) for x in mc] == port.mc_returns(rw, discount), "port MC returns != reference"
        mc_prio = np.abs(np.array(mc, dtype=np.float32) - np.array(root_q, dtype=np.float32))
        dummy = types.SimpleNamespace(unroll_n_steps=unroll, n_action=6)
        np.random.seed(100 + k)
        st, o_r, o_a, o_p, o_g = ref_muzero.Muzero.organise_transitions(dummy, list(states), list(rw), list(actions), list(pis),
                                                                      list(returns))
        np.random.seed(100 + k)
        absorbing = np.random.randint(0, 6)
        mine = port.organise_transitions(states, rw, actions, pis, returns, unroll, 6, absorbing)
        for a, b in zip((st, o_r, o_a, o_p, o_g), mine):
            assert a.dtype == b.dtype and np.array_equal(a, b), "port organise_transitions != reference"
        out.update({f"e{k}_reward_code": codes.astype(np.uint8), f"e{k}_visits": visits.astype(np.int32), f"e{k}_root_q": np.array(root_q),
                    f"e{k}_action": np.array(actions, np.int32), f"e{k}_returns": np.array(returns, np.float64), f"e{k}_priority": prio,
                    f"e{k}_absorbing": np.int64(absorbing), f"e{k}_mc_returns": np.array(mc, np.float64), f"e{k}_mc_priority": mc_prio, f"e{k}_o_r": o_r, f"e{k}_o_a": o_a, f"e{k}_o_p": o_p, f"e{k}_o_g": o_g})
    out.update(n_episodes=len(lengths), n_step=n_step, discount=discount, unroll=unroll)
    np.savez_compressed(os.path.join(GOLDEN, "episode_post.npz"), **out)
    print(f"episode post-processing: {len(lengths)} episodes ok (returns, priorities, transitions)")


def gen_learner(ref):
    """Two consecutive Muzero._update calls (Muzero.py:209-274, Adam of networks.py:69) of the unmodified reference on a
    synthetic batch: gradients after the first update and parameters after the second."""
    import torch

    sys.path.insert(0, rh.REFERENCE_ROOT)
    import Muzero as ref_muzero  # noqa: E402

    n, B, K = 3, 48, 5
    rng = np.random.default_rng(31)
    torch.manual_seed(0)
    m = ref_muzero.Muzero(env=None, s_space_size=3 * n, n_action=6, discount=0.8, dirichlet_alpha=0.25, n_mcts_simulations=5,
                          unroll_n_steps=K, batch_s=B, TD_return=True, n_TD_step=10, lr=0.002, buffer_size=64,
                          priority_replay=True, device="cpu")
    sd = port.make_weights(n, 17)
    m.networks.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    batches = []
    for _ in range(2):
        states = np.stack([port.one_hot(port.index_to_state(int(i), n)) for i in rng.integers(0, 27, B)]).astype(np.float32)
        rwds = rng.choice(np.array([0.0, 100.0, -0.1], np.float32), size=(B, K), p=[0.7, 0.1, 0.2]).astype(np.float32)
        actions = rng.integers(0, 6, (B, K)).astype(np.int64)
        pi = rng.dirichlet(np.ones(6), size=(B, K)).astype(np.float32)
        returns = (rng.normal(0, 20, (B, K))).astype(np.float32)
        w = rng.uniform(0.2, 1.0, B).astype(np.float32)
        batches.append((states, rwds, actions, pi, returns, w))
    out = dict(n=n, B=B, K=K, weight_seed=17, lr=0.002)
    for i, (states, rwds, actions, pi, returns, w) in enumerate(batches):
        new_p, v_loss, r_loss, p_loss = m._update(torch.from_numpy(states), torch.from_numpy(rwds), torch.from_numpy(actions),
                                                  torch.from_numpy(pi), torch.from_numpy(returns), torch.from_numpy(w))
        out.update({f"b{i}_states": states, f"b{i}_rwds": rwds, f"b{i}_actions": actions, f"b{i}_pi": pi, f"b{i}_returns": returns,
                    f"b{i}_w": w, f"b{i}_new_priorities": np.asarray(new_p, np.float32),
                    f"b{i}_losses": np.array([float(v_loss), float(r_loss), float(p_loss)], np.float32)})
        if i == 0:
            for k, prm in m.networks.named_parameters():
                out[f"grad0_{k}"] = prm.grad.detach().numpy().copy()
    for k, prm in m.networks.named_parameters():
        out[f"param2_{k}"] = prm.detach().numpy().copy()
    np.savez_compressed(os.path.join(GOLDEN, "learner.npz"), **out)
    print("learner: two reference updates recorded (losses %s)" % out["b1_losses"])


def check_choice_hook():
    """The uniform-as-input restatement of np.random.choice(p=...) equals numpy's legacy path."""
    rs = np.random.RandomState(7)
    rs2 = np.random.RandomState(7)
    for _ in range(2000):
        p = rs.dirichlet(np.ones(6))
        rs2.dirichlet(np.ones(6))
        a = rs.choice(np.arange(6), p=p)
        assert a == port.sample_action(p, rs2.random_sample())


def main():
    import torch

    os.makedirs(GOLDEN, exist_ok=True)
    ref = rh.import_reference()
    check_choice_hook()
    gen_env_tables(ref)
    for name, cfg in SEARCH_CONFIGS.items():
        gen_search(ref, name, cfg)
    gen_net_io(ref)
    gen_episode_post(ref)
    gen_learner(ref)
    manifest = dict(
        generated_by="python -m oracle.gen_golden",
        reference="A-Andrews/Muzero-Hanoi (unmodified, /root/reference)",
        numpy=np.__version__, torch=torch.__version__, python=sys.version.split()[0],
        hooks=["lowest-index tie-break (MCTS/node.py:86)", "dirichlet draw as input (MCTS/mcts.py:149)",
               "sampling uniform as input (MCTS/mcts.py:120)"],
        search_configs=SEARCH_CONFIGS,
    )
    with open(os.path.join(GOLDEN, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print("golden fixtures written to", GOLDEN)


if __name__ == "__main__":
    main()
