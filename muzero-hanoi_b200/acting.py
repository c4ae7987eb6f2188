"""Batched acting evaluation: ``acting_ablations.get_results`` / ``ablate_networks`` of the reference
(acting_experiments/acting_ablations.py:29-45, 72-128) with every episode of a setting run as one game
of a lock-step batch on the GPU (SURVEY.md §8f row 3).

Differences from the sequential reference, both forced by running the episodes in parallel: by default every
episode owns its MinMaxStats (the reference threads ONE stats object through all episodes of a run,
MCTS/mcts.py:23 and acting_ablations.py:343, so later episodes see the extrema of earlier ones), and the random
draws are inputs (``uniforms`` per move) or on-device Philox streams instead of the process-global NumPy state.
``shared_minmax=True`` reproduces the reference's experiment exactly in that respect: the episodes of a setting then
run ONE AFTER ANOTHER through a single search slot whose (min, max) persists from episode to episode — sequentially
consistent with the reference, and as serial as the reference is.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr
from .engine import BatchedMCTS, MultiMCTS, PackedWeights, VecHanoi, WeightSets, index_state, pack_state


def ablate_networks(reset_latent_policy, reset_latent_values, reset_latent_rwds, networks):
    """acting_ablations.py:29-45: re-initialise the chosen heads with ``networks.reset_param``."""
    if reset_latent_policy:
        networks.policy_net.apply(networks.reset_param)
    if reset_latent_values:
        networks.value_net.apply(networks.reset_param)
    if reset_latent_rwds:
        networks.rwd_net.apply(networks.reset_param)
    return networks


def get_results(weights: PackedWeights, N, max_steps, episode, n_mcts_simulations_range, temperature, *, start_idx=None,
                discount=0.8, root_dirichlet_alpha=0.0, seed=0, uniforms=None, start_indices=None, device="cuda",
                latent_dtype=None, return_details=False, shared_minmax=False):
    """``[[n_simulations, mean(steps - hanoi_solver(start))], ...]`` (acting_ablations.py:72-128) over
    ``episode`` parallel episodes per simulation budget.

    start_idx      index into env.states to reset to (``env.init_state_idx``); None = ``random_reset``
    start_indices  explicit start state index per episode (parity tests); overrides start_idx
    uniforms       float64 [moves, episode]: the ``np.random.choice`` draw of each move (MCTS/mcts.py:120);
                   drawn on device from Philox streams keyed by ``seed`` when omitted
    """
    _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(device)
    B = int(episode)
    ldt = (_lib.LATENT_BF16 if weights.mode == _lib.MODE_BF16 else _lib.LATENT_F32) if latent_dtype is None else latent_dtype
    data, details = [], []
    if shared_minmax:
        return _get_results_sequential(weights, N, max_steps, B, n_mcts_simulations_range, temperature, start_idx, discount,
                                       root_dirichlet_alpha, seed, uniforms, start_indices, dev, ldt, return_details)
    for n_sims in n_mcts_simulations_range:
        env = VecHanoi(N, max_steps, B, dev, init_state_idx=start_idx or 0)
        if start_indices is not None:
            env.set_state_indices(np.asarray(start_indices, dtype=np.int32))
        elif start_idx is not None:
            env.reset()
        else:
            env.random_reset(seed=seed, counter=int(n_sims))
        min_moves = env.solver_distance()  # hanoi_solver(tuple(env.current_state())), :96-98
        mcts = BatchedMCTS(discount, root_dirichlet_alpha, int(n_sims), B, dev, latent_dtype=ldt)
        steps = torch.zeros(B, dtype=torch.int32, device=dev)
        illegal = torch.zeros(B, dtype=torch.int32, device=dev)
        errors = torch.empty(B, dtype=torch.int32, device=dev)
        u_dev = torch.empty(B, dtype=torch.float64, device=dev)
        noise = torch.empty(B, 6, dtype=torch.float64, device=dev) if root_dirichlet_alpha > 0 else None
        for move in range(max_steps):  # every episode ends by max_steps (env/hanoi.py:77-80)
            if uniforms is not None:
                u_dev.copy_(torch.as_tensor(uniforms[move], dtype=torch.float64))
            else:
                check(lib.hmz_rng_uniform(ptr(u_dev), B, seed, (int(n_sims) << 20) | move, 0, current_stream()))
            if noise is not None:
                check(lib.hmz_rng_dirichlet(ptr(noise), B, float(root_dirichlet_alpha), seed, (int(n_sims) << 20) | move, 0,
                                            current_stream()))
            action, _, _, _ = mcts.run_mcts(weights, words=env.words, temperature=temperature, deterministic=False,
                                            noise=noise, uniforms=u_dev)
            _, _, flags = env.step(action, want_obs=False)
            check(lib.hmz_eval_track(ptr(flags), move, B, ptr(steps), ptr(illegal), current_stream()))
            if move % 8 == 7 and bool((steps > 0).all()):  # all first episodes over: stop early
                break
        check(lib.hmz_eval_errors(ptr(steps), ptr(min_moves), B, ptr(errors), current_stream()))
        err = errors.cpu().numpy()
        data.append([n_sims, float(err.sum()) / len(err)])  # sum(errors) / len(errors), :123
        details.append(dict(n_simulations=n_sims, steps=steps.cpu().numpy(), errors=err, illegal_moves=illegal.cpu().numpy(),
                            min_moves=min_moves.cpu().numpy()))
    return (data, details) if return_details else data


def _get_results_sequential(weights, N, max_steps, B, n_range, temperature, start_idx, discount, alpha, seed, uniforms,
                            start_indices, dev, ldt, return_details):
    """``shared_minmax=True``: acting_ablations.get_results exactly as the reference sequences it — one MCTS object per
    simulation budget (acting_ablations.py:76-79 mutates ``n_simulations`` on the SAME object, so the MinMaxStats even
    carries over from one budget to the next), episodes played one after another (:84-123)."""
    lib = _lib.load()
    data, details = [], []
    cap = max(int(n) for n in n_range)
    mcts = BatchedMCTS(discount, alpha, cap, 1, dev, latent_dtype=ldt)  # the one MinMaxStats of the run (MCTS/mcts.py:23)
    u_dev = torch.empty(1, dtype=torch.float64, device=dev)
    noise = torch.empty(1, 6, dtype=torch.float64, device=dev) if alpha > 0 else None
    for n_sims in n_range:
        mcts.n_simulations = int(n_sims)
        steps_all, err_all, ill_all, min_all = [], [], [], []
        for ep in range(B):
            env = VecHanoi(N, max_steps, 1, dev, init_state_idx=start_idx or 0, auto_reset=False)
            if start_indices is not None:
                env.set_state_indices(np.asarray([start_indices[ep]], dtype=np.int32))
            elif start_idx is not None:
                env.reset()
            else:
                env.random_reset(seed=seed, counter=(int(n_sims) << 20) | ep)  # (its own stream: the start states differ from the batched form's)
            min_moves = int(env.solver_distance().item())
            steps = illegal = 0
            done = False
            while not done:
                ctr = (int(n_sims) << 20) | steps  # item = the episode: the draws of the batched form's game `ep`
                if uniforms is not None:
                    u_dev.fill_(float(uniforms[steps][ep]))
                else:
                    check(lib.hmz_rng_uniform(ptr(u_dev), 1, seed, ctr, ep, current_stream()))
                if noise is not None:
                    check(lib.hmz_rng_dirichlet(ptr(noise), 1, float(alpha), seed, ctr, ep, current_stream()))
                action, _, _, _ = mcts.run_mcts(weights, words=env.words, temperature=temperature, deterministic=False, noise=noise,
                                                uniforms=u_dev)
                _, _, flags = env.step(action, want_obs=False)
                f = int(flags.item())
                illegal += int(bool(f & _lib.FLAG_ILLEGAL))
                steps += 1
                done = bool(f & _lib.FLAG_DONE)
            steps_all.append(steps), err_all.append(steps - min_moves), ill_all.append(illegal), min_all.append(min_moves)
        data.append([n_sims, float(sum(err_all)) / len(err_all)])
        details.append(dict(n_simulations=n_sims, steps=np.array(steps_all, np.int32), errors=np.array(err_all, np.int32),
                            illegal_moves=np.array(ill_all, np.int32), min_moves=np.array(min_all, np.int32)))
    return (data, details) if return_details else data


def get_results_grid(conditions, N, max_steps, temperature, *, discount=0.8, root_dirichlet_alpha=0.0, seed=0, device="cuda",
                     latent_dtype=None, return_details=False, stats=None):
    """A whole lesion-experiment grid (acting_ablations.get_results over networks x start states x budgets) as ONE batch of
    searches: per condition, exactly what ``get_results(weights, N, max_steps, episode, [n_simulations], temperature, ...)``
    returns for it with the same arguments — the same Philox draws, so the same games.

    conditions  list of dicts: ``weights`` (PackedWeights; one weight set per distinct object, all of one mode),
                ``n_simulations``, ``episode``, and at most one of ``start_idx`` / ``start_indices`` (neither = random_reset),
                optionally ``uniforms`` (float64 [moves, episode], as get_results)
    Returns a list with one entry per condition: its ``data`` (``[[n_simulations, mean error]]``), or ``(data, details)``.

    Layout: the games of each weight set are ordered by non-increasing budget and padded to whole 256-search blocks with
    extra episodes of the set's last condition (discarded); the blocks are then ordered by non-increasing budget, so each
    simulation of hmz_search_run_multi runs over a prefix of the batch.  Every 8 moves (where get_results checks for the
    end) the blocks whose games have all finished their first episode leave the batch and the others move up in order.
    (``shared_minmax`` is not available here: it serialises the episodes by design.)
    stats       optional dict, receives ``simulations`` (searched, padding included), ``moves`` and ``searches``."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(device)
    conds = list(conditions)
    if not conds:
        return []
    BLK = _lib.BLOCK
    nets, set_of = [], []
    for c in conds:
        k = next((i for i, w in enumerate(nets) if w is c["weights"]), None)
        if k is None:
            nets.append(c["weights"])
            k = len(nets) - 1
        set_of.append(k)
    sets = WeightSets(nets, N, nets[0].mode, dev)
    ldt = (_lib.LATENT_BF16 if sets.mode == _lib.MODE_BF16 else _lib.LATENT_F32) if latent_dtype is None else latent_dtype
    budgets = [int(c["n_simulations"]) for c in conds]
    if min(budgets) < 1 or max(budgets) > 32767:
        raise ValueError("n_simulations must lie in [1, 32767]")
    # layout L0: set by set, conditions by non-increasing budget, each condition's games contiguous (item = position - offset)
    off, cnt, first_of_block = [0] * len(conds), [0] * len(conds), []
    total = 0
    for k in range(len(nets)):
        members = sorted((i for i in range(len(conds)) if set_of[i] == k), key=lambda i: -budgets[i])
        start = total
        for i in members:
            off[i], cnt[i] = total, int(conds[i]["episode"])
            total += cnt[i]
        pad = -(total - start) % BLK
        cnt[members[-1]] += pad
        total += pad
        first_of_block += list(range(start, total, BLK))
    cond0 = np.empty(total, np.int64)
    item0 = np.empty(total, np.int64)
    for i in range(len(conds)):
        cond0[off[i]:off[i] + cnt[i]] = i
        item0[off[i]:off[i] + cnt[i]] = np.arange(cnt[i])
    budget0 = np.asarray(budgets, np.int64)[cond0]
    set0 = np.asarray(set_of, np.int64)[cond0]
    order = sorted(range(len(first_of_block)), key=lambda j: -budget0[first_of_block[j]])  # stable
    firsts = np.asarray([first_of_block[j] for j in order], np.int64)
    gid_h = (firsts[:, None] + np.arange(BLK)[None, :]).reshape(-1)  # slot -> L0 index
    B = len(gid_h)

    st = current_stream()
    words0 = torch.zeros(total, dtype=torch.int32, device=dev)
    for i, c in enumerate(conds):
        w = words0[off[i]:off[i] + cnt[i]]
        if c.get("start_indices") is not None:
            si = np.asarray(c["start_indices"], dtype=np.int32)
            idx = torch.as_tensor(si[np.arange(cnt[i]) % len(si)], device=dev)
            check(lib.hmz_env_from_index(ptr(idx), ptr(w), cnt[i], N, st))
        elif c.get("start_idx") is not None:
            check(lib.hmz_env_reset(ptr(w), cnt[i], pack_state(index_state(int(c["start_idx"]), N)), st))
        else:
            check(lib.hmz_env_random_reset(ptr(w), cnt[i], N, 2, seed, budgets[i], st))
    min_moves0 = torch.empty(total, dtype=torch.int32, device=dev)
    check(lib.hmz_env_solver_distance(ptr(words0), ptr(min_moves0), total, N, 2, st))
    steps0 = torch.zeros(total, dtype=torch.int32, device=dev)
    illegal0 = torch.zeros(total, dtype=torch.int32, device=dev)

    gid = torch.as_tensor(gid_h, device=dev)
    words = words0[gid].contiguous()
    budget = torch.as_tensor(budget0[gid_h], dtype=torch.int16, device=dev)
    ctr_hi = torch.as_tensor(budget0[gid_h] << 20, device=dev)
    item = torch.as_tensor(item0[gid_h], device=dev)
    block_set = torch.as_tensor(set0[firsts], dtype=torch.int16, device=dev)
    hbb = np.ascontiguousarray(budget0[firsts], dtype=np.int32)
    steps = torch.zeros(B, dtype=torch.int32, device=dev)
    illegal = torch.zeros(B, dtype=torch.int32, device=dev)
    rewards = torch.empty(B, dtype=torch.float32, device=dev)
    flags = torch.empty(B, dtype=torch.uint8, device=dev)
    u = torch.empty(B, dtype=torch.float64, device=dev)
    mcts = MultiMCTS(discount, root_dirichlet_alpha, max(budgets), B, dev, latent_dtype=ldt)
    noise = noise0 = None
    if root_dirichlet_alpha > 0:
        noise0 = torch.empty(total, 6, dtype=torch.float64, device=dev)
    given_u = {i: torch.as_tensor(np.asarray(c["uniforms"], np.float64), device=dev) for i, c in enumerate(conds)
               if c.get("uniforms") is not None}
    cond_slot = torch.as_tensor(cond0[gid_h], device=dev) if given_u else None
    n = B
    md = sets.desc(block_set, budget, hbb)
    budget_h = budget0[gid_h]
    sims_run = searches_run = moves_run = 0
    for move in range(max_steps):  # every episode ends by max_steps (env/hanoi.py:77-80)
        check(lib.hmz_rng_uniform_keyed(ptr(u), n, seed, ptr(ctr_hi), move, ptr(item), st))
        for i, ui in given_u.items():  # the condition's own draws for its real episodes
            sel = ((cond_slot[:n] == i) & (item[:n] < int(conds[i]["episode"]))).nonzero().flatten()
            u[sel] = ui[move][item[sel]]
        if noise0 is not None:
            for i in range(len(conds)):
                check(lib.hmz_rng_dirichlet(ptr(noise0[off[i]:]), cnt[i], float(root_dirichlet_alpha), seed,
                                            (budgets[i] << 20) | move, 0, st))
            noise = noise0[gid[:n]].contiguous()
        action, _, _, _ = mcts.run_mcts(sets, md, n, words=words, temperature=temperature, deterministic=False, noise=noise,
                                        uniforms=u)
        a8 = action.to(torch.uint8)
        check(lib.hmz_env_step(ptr(words), ptr(a8), ptr(rewards), ptr(flags), None, n, N, max_steps, 2, 1, 0, st))
        check(lib.hmz_eval_track(ptr(flags), move, n, ptr(steps), ptr(illegal), st))
        sims_run += int(budget_h[:n].sum())
        searches_run += n
        moves_run += 1
        if move % 8 != 7:
            continue
        alive = (steps[:n] == 0).view(-1, BLK).any(1).nonzero().flatten()
        if len(alive) == n // BLK:
            continue
        steps0[gid[:n]] = steps[:n]
        illegal0[gid[:n]] = illegal[:n]
        if len(alive) == 0:
            n = 0
            break
        # retire the finished blocks: the others move up, in order, with their per-game state
        slots = (alive[:, None] * BLK + torch.arange(BLK, device=dev)[None, :]).reshape(-1)
        m = len(slots)
        for t in (words, steps, illegal, gid, item, ctr_hi, budget, mcts.store.minmax) + ((cond_slot,) if given_u else ()):
            t[:m] = t[slots]
        block_set[:len(alive)] = block_set[alive]
        alive_h = alive.cpu().numpy()
        hbb = np.ascontiguousarray(hbb[alive_h])
        budget_h = budget_h.reshape(-1, BLK)[: n // BLK][alive_h].reshape(-1)
        n = m
        md = sets.desc(block_set, budget, hbb)
    if n:
        steps0[gid[:n]] = steps[:n]
        illegal0[gid[:n]] = illegal[:n]
    if stats is not None:
        stats.update(simulations=sims_run, searches=searches_run, moves=moves_run)
    errors0 = torch.empty(total, dtype=torch.int32, device=dev)
    check(lib.hmz_eval_errors(ptr(steps0), ptr(min_moves0), total, ptr(errors0), st))
    steps_h, err_h, ill_h, mm_h = (t.cpu().numpy() for t in (steps0, errors0, illegal0, min_moves0))
    out = []
    for i, c in enumerate(conds):
        sl = slice(off[i], off[i] + int(c["episode"]))
        err = err_h[sl]
        data = [[c["n_simulations"], float(err.sum()) / len(err)]]  # sum(errors) / len(errors), :123
        details = [dict(n_simulations=c["n_simulations"], steps=steps_h[sl].copy(), errors=err.copy(),
                        illegal_moves=ill_h[sl].copy(), min_moves=mm_h[sl].copy())]
        out.append((data, details) if return_details else data)
    return out
