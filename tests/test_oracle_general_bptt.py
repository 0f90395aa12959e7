"""CPU tests of the BPTT oracle over any oracle System (general_bptt_oracle.py): its pendulum instance against
orc.rollout_policy / orc.rollout_policy_vjp, system_step_vjp against float64 central differences of system.step, the
cotangent pass against torch autograd through a float64 torch restatement of the rollout, and the two forms of a
keyed System's key."""
import numpy as np
import pytest
import torch

from oracle import jax_prng as jr
from oracle import mbpo_oracle as orc
from oracle.mbpo_oracle import F32, U32

import general_bptt_oracle as gbo

SYSTEMS = {"pendulum": orc.PendulumOracle, "noisy_pendulum": lambda: orc.NoisyPendulumOracle(noise_std=0.05),
           "point_mass": orc.PointMassOracle}


def _actor(system, seed=31, hidden=(64, 64)):
    X, A = system.x_dim, system.u_dim
    return orc.BpttActorParams(mlp=orc.make_policy_params(seed=seed, obs_dim=X, action_dim=A, hidden=hidden),
                               init_stddev=0.5, obs_mean=np.linspace(-0.2, 0.3, X).astype(F32),
                               obs_std=np.linspace(0.7, 2.0, X).astype(F32))


def _states(system, n, seed, off_circle=False):
    """States away from the clip kinks: speeds stay well inside max_speed and the pendulum angle away from the wrap
    at +-pi.  off_circle: [cos, sin] pairs of norm 0.95..1.05, as NoisyPendulum's noisy observations are."""
    rng = np.random.default_rng(seed)
    if system.x_dim == 3:
        th = rng.uniform(-2.5, 2.5, n)
        r = rng.uniform(0.95, 1.05, n) if off_circle else np.ones(n)
        return np.stack([r * np.cos(th), r * np.sin(th), rng.uniform(-5, 5, n)], -1)
    return np.concatenate([rng.uniform(-2, 2, (n, 2)), rng.uniform(-1.5, 1.5, (n, 2))], -1)


def _keys(n, seed):
    return np.random.default_rng(seed).integers(0, 2 ** 32, size=(n, 2), dtype=np.uint64).astype(U32)


@pytest.mark.parametrize("evaluate", [False, True])
def test_pendulum_instance_equals_rollout_policy(evaluate):
    system = orc.PendulumOracle()
    actor = _actor(system)
    x0 = _states(system, 17, 1).astype(F32)
    key = jr.PRNGKey(5)
    want, wkey = orc.rollout_policy(actor, x0, key, 9, evaluate=evaluate)
    got, gkey, gsys = gbo.system_rollout_policy(system, actor, x0, key, 9, evaluate=evaluate)
    assert gsys is None and np.array_equal(gkey, wkey)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    rng = np.random.default_rng(2)
    cots = [rng.standard_normal(s).astype(F32) for s in ((17, 9), (17, 9, 3), (17, 9, 3), (17, 9, 1))]
    for use in [(1, 1, 1, 1), (1, 0, 0, 0), (0, 1, 0, 1)]:
        args = [c if u else None for c, u in zip(cots, use)]
        wa, wx = orc.rollout_policy_vjp(want["observation"], want["action"], *args)
        ga, gx = gbo.system_rollout_policy_vjp(system, want["observation"], want["action"], *args)
        assert np.array_equal(ga, wa) and np.array_equal(gx, wx)


@pytest.mark.parametrize("which", list(SYSTEMS))
def test_system_step_vjp_central_differences(which):
    system = SYSTEMS[which]()
    n = 256
    rng = np.random.default_rng(3)
    x = _states(system, n, 4, off_circle=True)
    u = rng.uniform(-0.9, 0.9, (n, system.u_dim))
    gn, gr = rng.standard_normal((n, system.x_dim)), rng.standard_normal(n)
    keys = _keys(n, 6) if system.keyed else None                       # fixed keys: the noise is a constant
    gx, gu = gbo.system_step_vjp(system, x, u, gn, gr, dtype=np.float64)

    def loss(x_, u_):
        nx, r, _ = system.step(x_, u_, keys, False, np.float64)
        return (nx * gn).sum(-1) + r * gr
    eps = 1e-6
    for i in range(system.x_dim):
        d = np.zeros_like(x)
        d[:, i] = eps
        np.testing.assert_allclose((loss(x + d, u) - loss(x - d, u)) / (2 * eps), gx[:, i], rtol=1e-5, atol=1e-6)
    for j in range(system.u_dim):
        d = np.zeros_like(u)
        d[:, j] = eps
        np.testing.assert_allclose((loss(x, u + d) - loss(x, u - d)) / (2 * eps), gu[:, j], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("which", list(SYSTEMS))
def test_rollout_vjp_matches_torch_autograd(which):
    """Actions as leaves (the stop_gradient structure of rollout_policy); NoisyPendulum's noise enters as constants
    drawn from the oracle's key chain."""
    system = SYSTEMS[which]()
    rng = np.random.default_rng(7)
    B, H, X, A = 8, 9, system.x_dim, system.u_dim
    x0 = _states(system, B, 8)
    acts = rng.uniform(-0.9, 0.9, (B, H, A))
    cots = [rng.standard_normal(s) for s in ((B, H), (B, H, X), (B, H, X), (B, H, A))]
    zs, k = [], _keys(B, 9)
    for _ in range(H):                                                 # NoisyPendulumOracle.step's draws
        ks = orc.split_keys(k, 2)
        zs.append(torch.tensor(jr.bits_to_normal(orc.random_bits_keys(ks[:, 1], 3)).astype(np.float64)))
        k = ks[:, 0]
    xt, at = torch.tensor(x0, requires_grad=True), torch.tensor(acts, requires_grad=True)
    x, obs, nxt, rew = xt, [], [], []
    for t in range(H):
        obs.append(x)
        x, r = gbo.torch_system_step(system, x, at[:, t], zs[t] if system.keyed else None)
        nxt.append(x)
        rew.append(r)
    obs, nxt, rew = torch.stack(obs, 1), torch.stack(nxt, 1), torch.stack(rew, 1)
    c = [torch.tensor(v) for v in cots]
    loss = (rew * c[0]).sum() + (nxt * c[1]).sum() + (obs * c[2]).sum() + (at * c[3]).sum()
    want_a, want_x0 = torch.autograd.grad(loss, [at, xt])
    got_a, got_x0 = gbo.system_rollout_policy_vjp(system, obs.detach().numpy(), acts, *cots, dtype=np.float64)
    np.testing.assert_allclose(got_a, want_a.numpy(), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(got_x0, want_x0.numpy(), rtol=1e-9, atol=1e-10)


def test_system_key_forms():
    """A [2] key is shared: identical x0 rows give identical trajectories (the same noise sequence).  [B, 2] keys:
    row b is the B = 1 rollout with key b."""
    system = orc.NoisyPendulumOracle(noise_std=0.05)
    actor = _actor(system, seed=41)
    x0 = np.repeat(_states(system, 1, 10).astype(F32), 5, axis=0)
    key, skey = jr.PRNGKey(3), jr.PRNGKey(8)
    tr, _, k_out = gbo.system_rollout_policy(system, actor, x0, key, 7, sys_keys=skey)
    assert k_out.shape == (2,)
    for f in ("observation", "action", "reward", "next_observation"):
        assert (tr[f] == tr[f][:1]).all(), f
    kk = skey
    for _ in range(7):
        kk = jr.split(kk, 2)[0]
    assert np.array_equal(k_out, kk)
    x1 = _states(system, 5, 11).astype(F32)
    keys = _keys(5, 12)
    tr, _, k_out = gbo.system_rollout_policy(system, actor, x1, key, 7, sys_keys=keys)
    assert k_out.shape == (5, 2)
    for b in range(5):
        one, _, kb = gbo.system_rollout_policy(system, actor, x1[b:b + 1], key, 7, sys_keys=keys[b:b + 1])
        assert np.array_equal(kb[0], k_out[b])
        for f in ("observation", "action", "reward", "next_observation"):
            assert np.array_equal(one[f][0], tr[f][b]), (b, f)
    # different trajectories of one batch see different noise with per-trajectory keys, the same with a shared key
    same = np.repeat(x1[:1], 2, axis=0)
    per, _, _ = gbo.system_rollout_policy(system, actor, same, key, 3, sys_keys=keys[:2])
    assert not np.array_equal(per["next_observation"][0], per["next_observation"][1])
