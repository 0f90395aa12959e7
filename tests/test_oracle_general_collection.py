"""CPU tests of the collection oracle over any System (general_collection_oracle.py: system_env_rollout /
system_actor_rollout): it restates env_rollout exactly for the pendulum, and for a keyed System it threads
system_params.key through action_repeat System steps per env step and across AutoReset, which resets obs but not
the key."""
import numpy as np
import pytest

from oracle import jax_prng as jr
from oracle import mbpo_oracle as orc

import general_collection_oracle as gco


def _pendulum_states(rng, e):
    th, w = rng.uniform(-np.pi, np.pi, e), rng.uniform(-8, 8, e)
    return np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)


def _keys(e, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2 ** 32, size=(e, 2), dtype=np.uint64).astype(np.uint32)


FIELDS = ("observation", "action", "reward", "discount", "next_observation", "truncation", "final_obs",
          "final_steps", "final_done")


@pytest.mark.parametrize("action_repeat", [1, 2])
def test_pendulum_system_env_rollout_equals_env_rollout(action_repeat):
    rng = np.random.default_rng(0)
    E, T, L = 9, 23, 7
    x0 = _pendulum_states(rng, E)
    acts = rng.uniform(-1.5, 1.5, (T, E)).astype(np.float32)
    steps0 = rng.integers(0, L, E).astype(np.float32)
    done0 = (rng.uniform(size=E) < 0.3).astype(np.float32)
    want = orc.env_rollout(x0, acts, L, action_repeat=action_repeat, steps0=steps0, done0=done0)
    got = gco.system_env_rollout(orc.PendulumOracle(), x0, acts[..., None], L, action_repeat, steps0=steps0, done0=done0)
    for f in FIELDS:
        assert np.array_equal(got[f], want[f]), f
        assert got[f].dtype == want[f].dtype
    assert got["final_keys"] is None


@pytest.mark.parametrize("partitionable", [False, True])
def test_noisy_pendulum_without_noise_is_the_pendulum(partitionable):
    rng = np.random.default_rng(1)
    E, T, L = 8, 30, 11
    x0 = _pendulum_states(rng, E)
    acts = rng.uniform(-1, 1, (T, E, 1)).astype(np.float32)
    keys = _keys(E, 2)
    want = gco.system_env_rollout(orc.PendulumOracle(), x0, acts, L)
    got = gco.system_env_rollout(orc.NoisyPendulumOracle(noise_std=0.0), x0, acts, L, keys=keys,
                                 partitionable=partitionable)
    for f in FIELDS:
        # equal as numbers: mean + 0 * z turns a -0 of the mean into +0 (-0 + 0 = +0), nothing else changes
        np.testing.assert_array_equal(got[f], want[f], err_msg=f)
    # ... and the key advanced once per step all the same
    k = keys
    for _ in range(T):
        k = orc.split_keys(k, 2, partitionable)[:, 0]
    assert np.array_equal(got["final_keys"], k)


def _step_by_step(system, x0, acts, L, action_repeat, keys, partitionable):
    """The wrapper stack written out per env with system.step on one row at a time."""
    T, E, A = acts.shape
    out = dict(reward=np.zeros((T, E), np.float32), next_observation=np.zeros((T, E, system.x_dim), np.float32),
               discount=np.zeros((T, E), np.float32), truncation=np.zeros((T, E), np.float32))
    final_keys = np.zeros_like(keys) if keys is not None else None
    for e in range(E):
        x, first = x0[e:e + 1].copy(), x0[e:e + 1].copy()
        k = None if keys is None else keys[e:e + 1].copy()
        steps, done = np.float32(0), np.float32(0)
        for t in range(T):
            if done:
                steps = np.float32(0)
            done = np.float32(0)
            rew = np.float32(0)
            for _ in range(action_repeat):
                x, r, k = system.step(x, acts[t, e:e + 1], k, partitionable)
                rew = np.float32(rew + r[0])
            steps = np.float32(steps + action_repeat)
            trunc = np.float32(0)
            if steps >= L:
                trunc, done, x = np.float32(1), np.float32(1), first.copy()
            out["reward"][t, e], out["next_observation"][t, e] = rew, x[0]
            out["discount"][t, e], out["truncation"][t, e] = 1 - done, trunc
        if keys is not None:
            final_keys[e] = k[0]
    return out, final_keys


@pytest.mark.parametrize("action_repeat", [1, 2])
@pytest.mark.parametrize("partitionable", [False, True])
@pytest.mark.parametrize("which", ["noisy_pendulum", "point_mass"])
def test_system_env_rollout_composes_system_step(which, partitionable, action_repeat):
    rng = np.random.default_rng(3)
    E, T, L = 5, 17, 6                           # several AutoResets inside T
    if which == "noisy_pendulum":
        system, x0, keys = orc.NoisyPendulumOracle(0.1), _pendulum_states(rng, E), _keys(E, 4)
    else:
        system, x0, keys = orc.PointMassOracle(), rng.uniform(-2, 2, (E, 4)).astype(np.float32), None
    acts = rng.uniform(-1.5, 1.5, (T, E, system.u_dim)).astype(np.float32)
    got = gco.system_env_rollout(system, x0, acts, L, action_repeat, keys=keys, partitionable=partitionable)
    want, want_keys = _step_by_step(system, x0, acts, L, action_repeat, keys, partitionable)
    for f in want:
        assert np.array_equal(got[f], want[f]), f
    assert got["truncation"].sum() >= E          # episodes did end inside T
    if keys is None:
        assert got["final_keys"] is None
    else:
        assert np.array_equal(got["final_keys"], want_keys)
        # AutoReset does not reset the key: it advanced action_repeat times per env step, T steps in all
        k = keys
        for _ in range(T * action_repeat):
            k = orc.split_keys(k, 2, partitionable)[:, 0]
        assert np.array_equal(got["final_keys"], k)


def test_system_actor_rollout_pendulum_equals_actor_rollout():
    rng = np.random.default_rng(5)
    E, T, L = 6, 9, 4
    x0 = _pendulum_states(rng, E)
    pol = orc.make_policy_params(seed=7, hidden=(64, 64))
    key = jr.PRNGKey(3)
    for conv in ("sac", "unroll", "as_is"):
        want, wk = orc.actor_rollout(pol, x0, key, T, L, key_convention=conv)
        got, gk = gco.system_actor_rollout(orc.PendulumOracle(), pol, x0, key, T, L, key_convention=conv)
        assert np.array_equal(gk, wk)
        for f in ("observation", "action", "reward", "discount", "next_observation", "truncation"):
            assert np.array_equal(got[f], want[f]), (conv, f)


def test_system_actor_rollout_point_mass_draws_per_action_dim():
    """A = 2: env e, dim a of step t reads element e * 2 + a of normal(k_t, (2 E,)); log_prob sums the two dims."""
    rng = np.random.default_rng(6)
    E, T = 5, 3
    x0 = rng.uniform(-1, 1, (E, 4)).astype(np.float32)
    pol = orc.make_policy_params(seed=9, obs_dim=4, action_dim=2, hidden=(64,))
    key = jr.PRNGKey(11)
    got, _ = gco.system_actor_rollout(orc.PointMassOracle(), pol, x0, key, T, 100, with_extras=True)
    k = key
    for t in range(T):
        k, k_t = jr.split(k, 2)
        logits = orc.policy_logits(pol, got["observation"][t])
        eps = jr.normal(k_t, 2 * E).reshape(E, 2)
        scale = (orc.softplus(logits[:, 2:]) + np.float32(pol.min_std)).astype(np.float32)
        raw = ((scale * eps).astype(np.float32) + logits[:, :2]).astype(np.float32)
        assert np.array_equal(got["raw_action"][t], raw)
        assert np.array_equal(got["action"][t], np.tanh(raw))
        _, _, lp = orc.policy_sample(pol, got["observation"][t], k_t, with_extras=True)
        assert np.array_equal(got["log_prob"][t], lp)
