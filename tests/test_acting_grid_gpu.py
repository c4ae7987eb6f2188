"""GPU: acting.get_results_grid — a whole lesion-experiment grid as one batch — returns for every condition exactly what
acting.get_results returns for it alone (data and every details array), including while finished blocks retire."""
import numpy as np
import pytest
import torch

from oracle import port

pytestmark = pytest.mark.gpu

N, MAX_STEPS = 3, 40
NEAR_GOAL = 17  # (1, 2, 2): one move, (1 -> 2) = action 3, from the goal


def _goal_seeker():
    """A network that always proposes action 3 with flat value and reward heads: from NEAR_GOAL its games end on the first
    or second move, so its blocks retire at the first check while the other conditions play on."""
    sd = dict(port.make_weights(N, 9))
    for head in ("value_net", "rwd_net", "policy_net"):
        sd[f"{head}.2.weight"] = np.zeros_like(sd[f"{head}.2.weight"])
        sd[f"{head}.2.bias"] = np.zeros_like(sd[f"{head}.2.bias"])
    sd["policy_net.2.bias"][3] = 20.0
    return sd


@pytest.mark.parametrize("mode", [0, 2, 1])
def test_grid_equals_get_results_per_condition(mode):
    from muzero_hanoi_b200 import acting
    from muzero_hanoi_b200.engine import PackedWeights

    base = port.make_weights(N, 31)
    nets = [PackedWeights(sd, N, mode) for sd in (base, port.lesion_weights(base, ["policy_net"], seed=1),
                                                  port.lesion_weights(base, ["value_net", "rwd_net"], seed=2))]
    rng = np.random.default_rng(4)
    conds, episodes = [], [37, 100, 61]
    for k, w in enumerate(nets):
        for j, b in enumerate((25, 7, 1)):
            e = episodes[(k + j) % 3]
            conds += [dict(weights=w, n_simulations=b, episode=e, start_idx=0),
                      dict(weights=w, n_simulations=b, episode=e, start_indices=rng.integers(0, 26, e)),
                      dict(weights=w, n_simulations=b, episode=e + 3)]
    conds[1]["uniforms"] = rng.random((MAX_STEPS, conds[1]["episode"]))
    seeker = PackedWeights(_goal_seeker(), N, mode)
    conds.append(dict(weights=seeker, n_simulations=50, episode=300, start_idx=NEAR_GOAL))
    stats = {}
    grid = acting.get_results_grid(conds, N, MAX_STEPS, 0.0, seed=11, return_details=True, stats=stats)
    torch.cuda.synchronize()
    longest = 0
    for i, c in enumerate(conds):
        kw = {key: c[key] for key in ("start_idx", "start_indices", "uniforms") if key in c}
        data, det = acting.get_results(c["weights"], N, MAX_STEPS, c["episode"], [c["n_simulations"]], 0.0, seed=11,
                                       return_details=True, **kw)
        gdata, gdet = grid[i]
        assert gdata == data, f"condition {i}"
        assert gdet[0]["n_simulations"] == det[0]["n_simulations"]
        for key in ("steps", "errors", "illegal_moves", "min_moves"):
            assert gdet[0][key].dtype == det[0][key].dtype and np.array_equal(gdet[0][key], det[0][key]), f"condition {i}: {key}"
        if i < len(conds) - 1:
            longest = max(longest, int(det[0]["steps"].max()) if (det[0]["steps"] > 0).all() else MAX_STEPS)
    # the goal seeker's two blocks (one condition of its own network) finished by the first check at move 8 while others
    # played on: they retired mid-run, and the grid searched fewer than (all blocks) x (moves played)
    assert (grid[-1][1][0]["steps"] <= 8).all() and longest > 8
    assert stats["searches"] < stats["moves"] * sum(-(-sum(c["episode"] for c in conds if c["weights"] is w) // 256) * 256
                                                    for w in nets + [seeker])
