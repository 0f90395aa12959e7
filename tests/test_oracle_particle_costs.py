"""CPU tests of the constraint-cost oracle over distinct particles (particle_cost_oracle.py), and of the argument checks
of mbpo_icem_penalize_particles / mbpo_ensemble_rollout_transitions, which run before anything touches a GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import jax_prng as jr
from oracle import mbpo_oracle as orc

import particle_cost_oracle as pco


def speed_cost(limit):
    """Batched AbstractCost: max_t |x_t[-1]| - limit (the last state coordinate is a velocity for every System here);
    a max and one subtraction, so every implementation rounds it the same way."""
    return lambda obs, acts: (np.abs(obs[..., -1]).max(axis=-1) - np.float32(limit)).astype(np.float32)


def _pendulum_states(rng, n):
    th, w = rng.uniform(-np.pi, np.pi, n), rng.uniform(-8, 8, n)
    return np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)


def _inputs(system, rng, m=9, h=7):
    x0 = (_pendulum_states(rng, 1)[0] if system.x_dim == 3 else rng.uniform(-1, 1, 4).astype(np.float32))
    acts = rng.uniform(-1.5, 1.5, (m, h, system.u_dim)).astype(np.float32)
    keys = rng.integers(0, 2 ** 32, (m, 2), dtype=np.uint64).astype(np.uint32)
    return x0, acts, keys


@pytest.mark.parametrize("partitionable", [False, True])
@pytest.mark.parametrize("use_optimism", [False, True])
@pytest.mark.parametrize("system,P", [(orc.NoisyPendulumOracle(0.3), 4), (orc.PointMassOracle(), 3),
                                      (orc.NoisyPendulumOracle(0.3), 1)])
def test_no_cost_equals_system_objective(system, P, use_optimism, partitionable):
    rng = np.random.default_rng(P)
    x0, acts, keys = _inputs(system, rng)
    params = orc.ICemParams(num_particles=P)
    values, obs, rew, nxt, cost = pco.system_objective_with_cost(system, x0, acts, keys, params, None, use_optimism,
                                                                 False, partitionable)
    want = orc.system_objective(system, x0, acts, keys, params, use_optimism, partitionable)
    assert cost is None and np.array_equal(values, want)
    m, h = acts.shape[:2]
    assert obs.shape == (m, P, h, system.x_dim) and rew.shape == (m, P, h) and nxt.shape == obs.shape
    assert np.array_equal(obs[:, :, 0], np.broadcast_to(x0, (m, P, system.x_dim)))
    assert np.array_equal(obs[:, :, 1:], nxt[:, :, :-1])
    # the buffers' own horizon means, summarised, are the values
    ret = np.stack([orc.particle_mean(rew[:, p], np.float32) for p in range(P)], axis=1)
    assert np.array_equal(pco.summarize(ret, use_optimism), values)


@pytest.mark.parametrize("use_optimism", [False, True])
def test_no_cost_equals_ensemble_rollout_returns(use_optimism):
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    rng = np.random.default_rng(1)
    x0 = _pendulum_states(rng, 2)
    acts = rng.uniform(-2, 2, (2, 3, 6)).astype(np.float32)
    values, obs, rew, cost = pco.ensemble_objective_with_cost(x0, acts, ens, None, use_optimism)
    assert cost is None
    assert np.array_equal(values, orc.ensemble_rollout_returns(x0, acts, ens, bf16=True, use_max=use_optimism))
    assert obs.shape == (2, 3, 5, 6, 3) and rew.shape == (2, 3, 5, 6)
    assert np.array_equal(obs[:, :, :, 0], np.broadcast_to(x0[:, None, None], (2, 3, 5, 3)))
    # rows of one member are independent of the member layout: member 2's rollout is member 2's steps
    x, r = orc.mlp_ensemble_step(obs[:, :, 2, 3].reshape(-1, 3), acts[:, :, 3].reshape(-1), np.full(6, 2, np.int32),
                                 ens, bf16=True)
    assert np.array_equal(x.reshape(2, 3, 3), obs[:, :, 2, 4]) and np.array_equal(r.reshape(2, 3), rew[:, :, 2, 3])


@pytest.mark.parametrize("use_optimism,use_pessimism", [(False, False), (True, False), (False, True), (True, True)])
@pytest.mark.parametrize("P", [1, 3])
def test_identical_pendulum_particles_equal_icem_objective(P, use_optimism, use_pessimism):
    rng = np.random.default_rng(7)
    x0, acts, keys = _inputs(orc.PendulumOracle(), rng, m=11, h=9)
    params = orc.ICemParams(num_particles=P, lambda_constraint=10.0)
    cost_fn = speed_cost(4.0)
    got = pco.system_objective_with_cost(orc.PendulumOracle(), x0, acts, keys, params, cost_fn, use_optimism,
                                         use_pessimism)[0]
    want = orc.icem_objective(x0, acts, params, orc.PendulumParams(), use_optimism, cost_fn=cost_fn,
                              use_pessimism=use_pessimism)
    assert np.array_equal(got, want)


def test_binding_cost_over_distinct_particles():
    """Pessimism summarises the cost by its max and optimism the reward by its max: row by row, both are at least the
    particle mean, and on distinct particles some rows differ."""
    system = orc.NoisyPendulumOracle(0.5)
    rng = np.random.default_rng(3)
    x0, acts, keys = _inputs(system, rng, m=32, h=10)
    params = orc.ICemParams(num_particles=6, lambda_constraint=1.0)
    cost_fn = speed_cost(float(np.abs(x0[2])) + 0.3)
    v = {}
    for opt in (False, True):
        for pes in (False, True):
            v[opt, pes], obs, rew, _, cost = pco.system_objective_with_cost(system, x0, acts, keys, params, cost_fn,
                                                                             opt, pes)
    ret = np.stack([orc.particle_mean(rew[:, p], np.float32) for p in range(6)], axis=1)
    assert np.all(ret.max(axis=1) >= orc.particle_mean(ret, np.float32))
    assert np.all(cost.max(axis=1) >= orc.particle_mean(cost, np.float32))
    assert np.all(v[False, True] <= v[False, False]) and np.any(v[False, True] < v[False, False])
    assert np.all(v[True, False] >= v[False, False]) and np.any(v[True, False] > v[False, False])
    assert np.any(cost.max(axis=1) > 0) and np.any(cost.min(axis=1) < 0)      # the cost binds on some particles only


def test_ensemble_binding_cost_pessimism():
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    rng = np.random.default_rng(4)
    x0 = _pendulum_states(rng, 1)
    acts = rng.uniform(-2, 2, (1, 16, 5)).astype(np.float32)
    cost_fn = speed_cost(float(np.abs(x0[0, 2])) + 0.05)
    mean = pco.ensemble_objective_with_cost(x0, acts, ens, cost_fn, False, False, 1.0)
    pes = pco.ensemble_objective_with_cost(x0, acts, ens, cost_fn, False, True, 1.0)
    assert np.array_equal(mean[1], pes[1]) and np.array_equal(mean[3], pes[3])
    assert np.all(pes[0] <= mean[0]) and np.any(pes[0] < mean[0])


def test_driver_without_cost_equals_system_icem_optimize():
    system = orc.NoisyPendulumOracle(0.1)
    params = orc.ICemParams(num_particles=3, num_samples=24, num_elites=5, num_steps=2)
    x0 = _pendulum_states(np.random.default_rng(5), 1)[0]
    st = orc.icem_init(jr.PRNGKey(11), 8)
    tr_a, tr_b = [], []
    a = pco.system_icem_optimize_with_cost(system, x0, st, params, 8, trace=tr_a)
    b = orc.system_icem_optimize(system, x0, st, params, 8, trace=tr_b)
    assert np.array_equal(a.best_sequence, b.best_sequence) and a.best_reward == b.best_reward
    assert np.array_equal(a.key, b.key)
    for x, y in zip(tr_a, tr_b):
        assert np.array_equal(x["values"], y["values"]) and np.array_equal(x["elite_idx"], y["elite_idx"])


def test_new_entry_points_check_arguments():
    import mbpo_b200
    L = mbpo_b200._lib
    buf = (C.c_float * 8)()
    assert L.lib.mbpo_icem_penalize_particles(None, None, 5, None, 0, 2, 0, 0, 1.0, None) == L.MBPO_OK   # n == 0
    assert L.lib.mbpo_icem_penalize_particles(None, buf, 5, None, 3, 2, 0, 0, 1.0, None) == L.MBPO_EINVAL
    assert L.lib.mbpo_icem_penalize_particles(buf, buf, 5, None, 3, 0, 0, 0, 1.0, None) == L.MBPO_EINVAL  # P == 0
    assert L.lib.mbpo_icem_penalize_particles(buf, buf, 0, None, 3, 2, 0, 0, 1.0, None) == L.MBPO_EINVAL  # H == 0
    assert L.lib.mbpo_icem_penalize_particles(buf, buf, 5, None, 3, 2, 2, 0, 1.0, None) == L.MBPO_EINVAL
    assert L.lib.mbpo_ensemble_rollout_transitions(None, 5, buf, buf, 1, 1, buf, buf, None) == L.MBPO_EINVAL
    ens = L.MlpEnsembleParamsC()
    assert L.lib.mbpo_ensemble_rollout_transitions(C.byref(ens), 5, buf, buf, 1, 1, buf, None, None) == L.MBPO_EINVAL
    assert L.lib.mbpo_ensemble_rollout_transitions(C.byref(ens), 5, buf, buf, 1, 1, buf, buf, None) == L.MBPO_EINVAL
