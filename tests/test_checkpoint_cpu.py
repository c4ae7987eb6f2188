"""Checkpoint files on the host: the flat <-> torch.optim.Adam mapping of the learner's Adam state round-trips exactly and
agrees with what torch's own Adam holds, and malformed files (the reference's checkpoint format and BatchedMuzero.save's)
are rejected with ValueError before anything touches a device."""
import copy

import numpy as np
import pytest
import torch

from conftest import ROOT  # noqa: F401

N = 3


def _flat_moments(seed, n_disks=N):
    from muzero_hanoi_b200.learner import param_shapes

    n = sum(int(np.prod(s)) for _, s in param_shapes(n_disks))
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, generator=g), torch.rand(n, generator=g)


def test_param_shapes_are_muzeronet_parameters_in_order():
    from muzero_hanoi_b200.engine import STATE_DICT_ORDER
    from muzero_hanoi_b200.learner import param_shapes
    from muzero_hanoi_b200.networks import MuZeroNet

    for n in (1, 3, 5, 12):
        net = MuZeroNet(3 * n, 6, 0.002, "cpu", TD_return=True)
        assert [(k, tuple(p.shape)) for k, p in net.named_parameters()] == param_shapes(n)
        assert [k for k, _ in param_shapes(n)] == STATE_DICT_ORDER


@pytest.mark.parametrize("step_index", [0, 1, 37])
def test_adam_mapping_round_trips_through_torch_adam(step_index):
    from muzero_hanoi_b200.learner import adam_to_torch, torch_to_adam
    from muzero_hanoi_b200.networks import MuZeroNet

    m, v = _flat_moments(step_index)
    if step_index == 0:
        m, v = torch.zeros_like(m), torch.zeros_like(v)
    osd = adam_to_torch(m, v, step_index, N, 0.003)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    net.optimiser.load_state_dict(copy.deepcopy(osd))  # the reference's own optimiser takes it
    assert net.optimiser.param_groups[0]["lr"] == 0.003 and net.optimiser.param_groups[0]["weight_decay"] == 0
    back_m, back_v, step, lr, betas, eps = torch_to_adam(net.optimiser.state_dict(), N)
    assert torch.equal(back_m, m) and torch.equal(back_v, v) and step == step_index
    assert (lr, betas, eps) == (0.003, (0.9, 0.999), 1e-8)
    assert (len(osd["state"]) == 0) == (step_index == 0)


def test_torch_adam_state_maps_to_the_flat_layout():
    """After real torch Adam steps the flat moments are torch's exp_avg / exp_avg_sq concatenated in parameters() order."""
    from muzero_hanoi_b200.learner import torch_to_adam
    from muzero_hanoi_b200.networks import MuZeroNet

    torch.manual_seed(3)
    net = MuZeroNet(3 * N, 6, 0.002, "cpu", TD_return=True)
    for _ in range(2):
        for p in net.parameters():
            p.grad = torch.randn_like(p)
        net.optimiser.step()
    m, v, step, *_ = torch_to_adam(net.optimiser.state_dict(), N)
    state = [net.optimiser.state[p] for p in net.parameters()]
    assert step == 2
    assert torch.equal(m, torch.cat([s["exp_avg"].reshape(-1) for s in state]))
    assert torch.equal(v, torch.cat([s["exp_avg_sq"].reshape(-1) for s in state]))


def _reference_file(path, n_disks=N, mutate=None):
    from muzero_hanoi_b200.learner import adam_to_torch, split_flat

    m, v = _flat_moments(1, n_disks)
    ck = {"Muzero_net": split_flat(m.clone(), n_disks), "Net_optim": adam_to_torch(m, v, 4, n_disks, 0.002)}
    if mutate:
        mutate(ck)
    torch.save(ck, path)
    return path


def _drop_net_key(ck):
    del ck["Muzero_net"]["value_net.2.bias"]


def _extra_net_key(ck):
    ck["Muzero_net"]["extra.weight"] = torch.zeros(1)


def _drop_optim_key(ck):
    del ck["Net_optim"]["state"]


def _drop_moment(ck):
    del ck["Net_optim"]["state"][3]["exp_avg_sq"]


def _bad_net_shape(ck):
    ck["Muzero_net"]["dynamic_net.0.weight"] = torch.zeros(256, 71)


def _bad_moment_shape(ck):
    ck["Net_optim"]["state"][0]["exp_avg"] = torch.zeros(256, 3 * N + 1)


def _weight_decay(ck):
    ck["Net_optim"]["param_groups"][0]["weight_decay"] = 1e-4


def _amsgrad(ck):
    ck["Net_optim"]["param_groups"][0]["amsgrad"] = True


def _mixed_steps(ck):
    ck["Net_optim"]["state"][5]["step"] = torch.tensor(3.0)


def _betas(ck):
    ck["Net_optim"]["param_groups"][0]["betas"] = (0.8, 0.999)


def _extra_top_key(ck):
    ck["epoch"] = 3


@pytest.mark.parametrize("mutate, field", [
    (_drop_net_key, "Muzero_net"), (_extra_net_key, "Muzero_net"), (_drop_optim_key, "Net_optim"), (_drop_moment, "Net_optim.state[3]"),
    (_bad_net_shape, "dynamic_net.0.weight"), (_bad_moment_shape, "Net_optim.state[0].exp_avg"),
    (_weight_decay, "weight_decay"), (_amsgrad, "amsgrad"), (_mixed_steps, "step"), (_betas, "betas"),
    (_extra_top_key, "Muzero_net"),
])
def test_from_reference_rejects_malformed_files(tmp_path, mutate, field):
    from muzero_hanoi_b200.trainer import BatchedMuzero

    path = _reference_file(tmp_path / "muzero_model.pt", mutate=mutate)
    with pytest.raises(ValueError, match=field.replace("[", r"\[").replace("]", r"\]").replace(".", r"\.")):
        BatchedMuzero.from_reference(path, N, 40, 256)


def test_from_reference_rejects_another_n(tmp_path):
    from muzero_hanoi_b200.trainer import BatchedMuzero

    path = _reference_file(tmp_path / "muzero_model.pt", n_disks=4)
    with pytest.raises(ValueError, match=r"representation_net\.0\.weight.*N=3"):
        BatchedMuzero.from_reference(path, N, 40, 256)


# -- BatchedMuzero.save files ------------------------------------------------------------------------------
def _checkpoint(n_disks=N, games=8, max_steps=40, buffer_size=50, ptr=30, is_full=False):
    """A well-formed checkpoint of a run mid-way (synthetic contents)."""
    from muzero_hanoi_b200.learner import param_shapes
    from muzero_hanoi_b200.trainer import CHECKPOINT_VERSION

    K = 5
    P = sum(int(np.prod(s)) for _, s in param_shapes(n_disks))
    steps = torch.arange(games, dtype=torch.int32) % 4  # episodes in flight of 0..3 moves
    words = (steps << (2 * n_disks)) | 1
    L = int(steps.sum())
    rows = buffer_size if is_full else ptr
    config = dict(N=n_disks, max_steps=max_steps, n_games=games, discount=0.8, dirichlet_alpha=0.25, n_mcts_simulations=8,
                  unroll_n_steps=K, batch_s=64, n_TD_step=10, lr=0.002, buffer_size=buffer_size, priority_replay=True,
                  n_update_x_loop=2, moves_per_loop=8, acting_mode=0, seed=5)
    _, key, pos, has_gauss, cached = np.random.RandomState(0).get_state()
    return dict(
        version=CHECKPOINT_VERSION, config=config,
        trainer=dict(loops_done=7, episodes_done=40, weights_dirty=True, replay_status=0, temperature=1.0),
        learner=dict(params=torch.zeros(P), adam_m=torch.zeros(P), adam_v=torch.zeros(P), step_index=6),
        selfplay=dict(moves_done=56, words=words, minmax=torch.zeros(games, 2, dtype=torch.float64)),
        episodes=dict(state=torch.zeros(L, dtype=torch.int32), action=torch.zeros(L, dtype=torch.uint8),
                      flags=torch.zeros(L, dtype=torch.uint8), visits=torch.zeros(L, 6, dtype=torch.int16),
                      root_q=torch.zeros(L, dtype=torch.float64), exp=torch.ones(L, dtype=torch.uint8),
                      cur_slot=torch.zeros(games, dtype=torch.int32), ep_len=torch.zeros(games, dtype=torch.int32)),
        replay=dict(states=torch.zeros(rows, 3 * n_disks), rwds=torch.zeros(rows, K), actions=torch.zeros(rows, K, dtype=torch.int64),
                    pi_probs=torch.zeros(rows, K, 6), mc_returns=torch.zeros(rows, K), priorities=torch.zeros(rows), ptr=ptr,
                    is_full=is_full, status=0),
        rng=dict(numpy=dict(key=torch.from_numpy(key.astype(np.int64)), pos=int(pos), has_gauss=int(has_gauss),
                            cached_gaussian=float(cached)),
                 torch_cuda=torch.zeros(16, dtype=torch.uint8)))


def test_well_formed_checkpoint_passes_and_survives_weights_only_load(tmp_path):
    from muzero_hanoi_b200.trainer import check_checkpoint

    for ck in (_checkpoint(), _checkpoint(ptr=10, is_full=True)):
        check_checkpoint(ck)
        torch.save(ck, tmp_path / "ck.pt")
        check_checkpoint(torch.load(tmp_path / "ck.pt"))  # default weights_only=True


def _set(path, value):
    def mutate(ck):
        *parents, last = path.split(".")
        node = ck
        for p in parents:
            node = node[p]
        if value is KeyError:
            del node[last]
        else:
            node[last] = value(node[last]) if callable(value) else value
    return mutate


@pytest.mark.parametrize("mutate, field", [
    (_set("version", 2), "version"),
    (_set("config.N", 4), "learner.params"),                      # a file of another N
    (_set("config.n_games", 16), "selfplay.minmax"),
    (_set("config.seed", KeyError), "config"),
    (_set("learner.adam_v", lambda t: t[1:]), "learner.adam_v"),
    (_set("selfplay.words", lambda w: w + (1 << (2 * N))), "episodes.state"),   # one more live slot per game than stored
    (_set("episodes.visits", lambda t: t[:, :5]), "episodes.visits"),
    (_set("replay.states", lambda t: t[1:]), "replay.states"),
    (_set("replay.actions", lambda t: t.to(torch.int32)), "replay.actions"),
    (_set("replay.ptr", 50), "replay.ptr"),
    (_set("rng.numpy.key", lambda t: t[:10]), "rng.numpy.key"),
    (_set("trainer.loops_done", 7.0), "trainer.loops_done"),
])
def test_malformed_checkpoints_are_rejected(tmp_path, mutate, field):
    from muzero_hanoi_b200.trainer import BatchedMuzero, check_checkpoint

    ck = _checkpoint()
    mutate(ck)
    with pytest.raises(ValueError, match=f"'{field}'"):
        check_checkpoint(ck)
    torch.save(ck, tmp_path / "ck.pt")
    with pytest.raises(ValueError, match=f"'{field}'"):
        BatchedMuzero.load(tmp_path / "ck.pt")  # rejected before any device work
