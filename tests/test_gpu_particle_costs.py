"""GPU parity of iCemTO's constraint cost over distinct particles: the particle-axis Transition buffers of
mbpo_system_objective, the per-member buffers of mbpo_ensemble_rollout_transitions, the tail
mbpo_icem_penalize_particles, and the planner routes that compose them (particle_cost_oracle.py)."""
import numpy as np
import pytest
import torch

from oracle import jax_prng as ojr
from oracle import mbpo_oracle as orc

import particle_cost_oracle as pco

pytestmark = pytest.mark.gpu

RTOL = 1e-5
E = 5


@pytest.fixture(scope="module")
def mb(cuda_device):
    import mbpo_b200
    return mbpo_b200


@pytest.fixture(scope="module")
def ens():
    return orc.make_mlp_ensemble(seed=3, members=E)


@pytest.fixture(params=[False, True], ids=["legacy", "partitionable"])
def prng_mode(request, mb):
    mb.config.threefry_partitionable = request.param
    yield request.param
    mb.config.threefry_partitionable = False


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _keys(n, seed):
    return np.random.default_rng(seed).integers(0, 2 ** 32, size=(n, 2), dtype=np.uint64).astype(np.uint32)


def _pendulum_states(n, seed):
    rng = np.random.default_rng(seed)
    th, w = rng.uniform(-np.pi, np.pi, n), rng.uniform(-8, 8, n)
    return np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)


def _general(mb, kind):
    from mbpo_b200.systems import NoisyPendulumSystem, PointMassSystem
    if kind == "noisy_pendulum":
        return NoisyPendulumSystem(0.05), orc.NoisyPendulumOracle(0.05)
    return PointMassSystem(), orc.PointMassOracle()


def _general_states(kind, n, seed):
    if kind == "noisy_pendulum":
        return _pendulum_states(n, seed)
    return np.random.default_rng(seed).uniform(-1.5, 1.5, (n, 4)).astype(np.float32)


def _ensemble_system(mb, dev, ens):
    from mbpo_b200.systems import MLPEnsembleSystem, MlpEnsembleDynamicsParams, PendulumRewardParams, SystemParams
    dyn = MlpEnsembleDynamicsParams(weights=[_dev(w, dev) for w in ens.weights],
                                    biases=[_dev(b, dev) for b in ens.biases])
    return MLPEnsembleSystem(dynamics_params=dyn), SystemParams(dynamics_params=dyn,
                                                                 reward_params=PendulumRewardParams())


class SpeedLimit:
    """AbstractCost: the largest |x_t[-1]| (a velocity for every System here) must stay below `limit`; a max and one
    subtraction, so the GPU and the oracle see bit-identical costs for bit-identical observations."""

    def __init__(self, limit):
        self.limit = limit

    def __call__(self, states, actions):                       # one trajectory: [H, X], [H, A] -> scalar
        return states[:, -1].abs().max() - self.limit

    def numpy(self, obs, acts):                                # batched: [R, H, X] -> [R]
        return (np.abs(obs[..., -1]).max(axis=-1) - np.float32(self.limit)).astype(np.float32)


# ---- 1. particle-axis buffers of the general Systems ------------------------------------------------------------
@pytest.mark.parametrize("P", [1, 4])
@pytest.mark.parametrize("kind", ["noisy_pendulum", "point_mass"])
def test_general_particle_buffers(mb, cuda_device, prng_mode, kind, P):
    system, osys = _general(mb, kind)
    B, M, H, A, X = 3, 37, 12, system.u_dim, system.x_dim
    x0 = _general_states(kind, B, 501)
    acts = np.clip(np.random.default_rng(502).normal(0, 0.5, (B, M, H, A)), -1, 1).astype(np.float32)
    keys = _keys(B * M, 503).reshape(B, M, 2)
    sp = system.init_params(mb.random.PRNGKey(0, cuda_device))
    d = lambda a: _dev(a, cuda_device)
    for use_max in (False, True):
        vals, obs, rew, nxt = system.objective(sp, d(x0), d(acts), d(keys), num_particles=P, use_optimism=use_max,
                                               full=True)
        assert torch.equal(vals, system.objective(sp, d(x0), d(acts), d(keys), num_particles=P, use_optimism=use_max))
    assert obs.shape == (B, M, P, H, X) and rew.shape == (B, M, P, H) and nxt.shape == obs.shape
    obs, rew, nxt = obs.cpu().numpy(), rew.cpu().numpy(), nxt.cpu().numpy()
    assert np.array_equal(obs[..., 0, :], np.broadcast_to(x0[:, None, None], (B, M, P, X)))
    assert np.array_equal(obs[..., 1:, :], nxt[..., :-1, :])
    # teacher-forced: every step from the kernel's own observation and the particle's key
    R = B * M * P
    k = orc.split_keys(keys.reshape(-1, 2), P, prng_mode).reshape(R, 2) if osys.keyed else None
    u = np.broadcast_to(acts[:, :, None], (B, M, P, H, A))
    for t in range(H):
        xn, r, k = osys.step(obs[..., t, :].reshape(R, X), u[..., t, :].reshape(R, A), k, prng_mode)
        if kind == "point_mass":
            assert np.array_equal(nxt[..., t, :].reshape(R, X), xn) and np.array_equal(rew[..., t].reshape(R), r)
        else:
            np.testing.assert_allclose(nxt[..., t, :].reshape(R, X), xn, rtol=RTOL, atol=2e-6)
            np.testing.assert_allclose(rew[..., t].reshape(R), r, rtol=RTOL, atol=3e-6)
    if not osys.keyed:                                  # P copies of the one rollout
        assert np.array_equal(obs, np.broadcast_to(obs[:, :, :1], obs.shape))


# ---- 2. per-member buffers of the tcgen05 ensemble kernels ------------------------------------------------------
@pytest.mark.parametrize("B,M,H", [(3, 100, 8), (1, 1039, 50), (36, 1039, 50)])   # one tile / one tile / two tiles
def test_ensemble_transitions(mb, cuda_device, ens, B, M, H):
    system, sp = _ensemble_system(mb, cuda_device, ens)
    x0 = _pendulum_states(B, 601)
    acts = np.random.default_rng(602).uniform(-2, 2, (B, M, H, 1)).astype(np.float32)
    x0_d, acts_d = _dev(x0, cuda_device), _dev(acts, cuda_device)
    obs, rew = system.ensemble_transitions(sp, x0_d, acts_d)
    assert obs.shape == (B, M, E, H, 3) and rew.shape == (B, M, E, H)
    # the horizon means of the kernel's own rewards, summarised, are mbpo_ensemble_rollout's returns, bit for bit
    L = mb._lib
    for use_max in (False, True):
        want = system.ensemble_returns(sp, x0_d, acts_d, use_optimism=use_max)
        got = torch.empty_like(want)
        L.check(L.lib.mbpo_icem_penalize_particles(L.ptr(got), L.ptr(rew), H, None, B * M, E, int(use_max), 0, 1.0,
                                                   L.stream_ptr(cuda_device)))
        assert torch.equal(got, want)
    obs, rew = obs.cpu().numpy(), rew.cpu().numpy()
    assert np.array_equal(obs[..., 0, :], np.broadcast_to(x0[:, None, None], (B, M, E, 3)))
    rows = np.random.default_rng(603).choice(B * M, size=min(B * M, 256), replace=False)
    o = obs.reshape(B * M, E, H, 3)[rows]
    r = rew.reshape(B * M, E, H)[rows]
    u = acts.reshape(B * M, H)[rows]
    n = len(rows)
    for t in range(H):
        for e in range(E):
            _, want_r = orc.pendulum_step(o[:, e, t], u[:, t], ens.reward)
            np.testing.assert_allclose(r[:, e, t], want_r, rtol=RTOL, atol=1e-6)
            if t + 1 < H:
                xn, _ = orc.mlp_ensemble_step(o[:, e, t], u[:, t], np.full(n, e, np.int32), ens, bf16=True)
                np.testing.assert_allclose(o[:, e, t + 1], xn, rtol=5e-3, atol=5e-3)


# ---- 3. the tail -------------------------------------------------------------------------------------------------
def _tail(mb, dev, reward, cost, H, P, s_rew, s_cost, lam):
    L = mb._lib
    n = reward.shape[0]
    out = torch.empty((n,), dtype=torch.float32, device=dev)
    L.check(L.lib.mbpo_icem_penalize_particles(L.ptr(out), L.ptr(reward), H, L.ptr(cost), n, P, s_rew, s_cost, lam,
                                               L.stream_ptr(dev)))
    return out


@pytest.mark.parametrize("kind", ["noisy_pendulum", "point_mass"])
def test_tail_reproduces_system_objective(mb, cuda_device, prng_mode, kind):
    system, _ = _general(mb, kind)
    B, M, H, P = 2, 45, 15, 3
    x0 = _general_states(kind, B, 701)
    acts = np.clip(np.random.default_rng(702).normal(0, 0.5, (B, M, H, system.u_dim)), -1, 1).astype(np.float32)
    keys = _keys(B * M, 703).reshape(B, M, 2)
    sp = system.init_params(mb.random.PRNGKey(0, cuda_device))
    d = lambda a: _dev(a, cuda_device)
    _, _, rew, _ = system.objective(sp, d(x0), d(acts), d(keys), num_particles=P, full=True)
    for use_max in (0, 1):
        want = system.objective(sp, d(x0), d(acts), d(keys), num_particles=P, use_optimism=bool(use_max))
        got = _tail(mb, cuda_device, rew.reshape(B * M, P, H), None, H, P, use_max, 0, 5.0)
        assert torch.equal(got.reshape(B, M), want)


def test_tail_with_cost_matches_numpy(mb, cuda_device):
    rng = np.random.default_rng(801)
    n, P, H, lam = 1000, 7, 13, 37.5
    reward = rng.normal(-3, 2, (n, P, H)).astype(np.float32)
    cost = rng.normal(0, 1, (n, P)).astype(np.float32)
    ret = np.zeros((n, P), np.float32)
    for t in range(H):
        ret = (ret + reward[:, :, t]).astype(np.float32)
    ret = (ret / np.float32(H)).astype(np.float32)
    for s_rew in (0, 1):
        for s_cost in (0, 1):
            want = pco.penalized(ret, cost, lam, bool(s_rew), bool(s_cost))
            got = _tail(mb, cuda_device, _dev(reward, cuda_device), _dev(cost, cuda_device), H, P, s_rew, s_cost, lam)
            assert np.array_equal(got.cpu().numpy(), want)


# ---- 4. a cost that never binds gives the plan without a cost ----------------------------------------------------
def _opt(mb, system, horizon, cost=None, use_optimism=False, use_pessimism=False, **params):
    from mbpo_b200.optimizers import iCemTO, iCemParams
    opt = iCemTO(horizon=horizon, action_dim=system.u_dim, opt_params=iCemParams(**params), cost_fn=cost,
                 use_optimism=use_optimism, use_pessimism=use_pessimism)
    opt.set_system(system)
    return opt


@pytest.mark.parametrize("kind,use_optimism", [("noisy_pendulum", False), ("noisy_pendulum", True),
                                               ("point_mass", False)])
def test_never_binding_cost_gives_the_fused_plan(mb, cuda_device, prng_mode, kind, use_optimism):
    system, _ = _general(mb, kind)
    horizon, B = 20, 4
    params = dict(num_samples=128, num_elites=12, num_particles=4, num_steps=3)
    x0 = _dev(_general_states(kind, B, 901), cuda_device)
    keys = _dev(_keys(B, 902), cuda_device)
    plain = _opt(mb, system, horizon, None, use_optimism, **params)
    costed = _opt(mb, system, horizon, SpeedLimit(1e6), use_optimism, **params)
    assert plain._fused(plain._cfg(), system.pack_params(system.init_params(keys[0])))
    st = plain.init(keys)
    a, b = plain.optimize(x0, st), costed.optimize(x0, st)
    assert torch.equal(a.best_sequence, b.best_sequence) and torch.equal(a.best_reward, b.best_reward)
    assert torch.equal(a.key, b.key)


def test_never_binding_cost_gives_the_ensemble_staged_plan(mb, cuda_device, ens):
    system, _ = _ensemble_system(mb, cuda_device, ens)
    horizon, B = 15, 3
    params = dict(num_samples=200, num_elites=20, num_particles=E, num_steps=3)
    x0 = _dev(_pendulum_states(B, 911), cuda_device)
    keys = _dev(_keys(B, 912), cuda_device)
    for use_optimism in (False, True):
        plain = _opt(mb, system, horizon, None, use_optimism, **params)
        costed = _opt(mb, system, horizon, SpeedLimit(1e6), use_optimism, use_pessimism=True, **params)
        st = plain.init(keys)
        a, b = plain.optimize(x0, st), costed.optimize(x0, st)
        assert torch.equal(a.best_sequence, b.best_sequence) and torch.equal(a.best_reward, b.best_reward)
        assert torch.equal(a.key, b.key)


# ---- 5. a binding cost against the oracle ------------------------------------------------------------------------
def _check_elites(values_oracle, g_idx, tol):
    """The GPU's elites are the oracle's best K up to candidates closer than tol."""
    mask = np.zeros(values_oracle.shape[0], bool)
    mask[g_idx] = True
    if mask.all():
        return
    assert values_oracle[mask].min() >= values_oracle[~mask].max() - tol


def _noisy_binding_plan(mb, cuda_device, prng_mode, use_pessimism):
    """A binding-cost plan over the noisy pendulum, teacher-forced against the oracle per iteration; returns the trace."""
    system, osys = _general(mb, "noisy_pendulum")
    horizon, B, lam = 20, 3, 1.0
    params = dict(num_samples=128, num_elites=12, num_particles=4, num_steps=3, lambda_constraint=lam)
    x0 = _pendulum_states(B, 1001)
    keys = _keys(B, 1002)
    cost = SpeedLimit(float(np.abs(x0[:, 2]).mean()))
    opt = _opt(mb, system, horizon, cost, use_pessimism=use_pessimism, **params)
    st = opt.init(_dev(keys, cuda_device))
    _, _, out_key, tr = opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params, trace=True)
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    p = orc.ICemParams(**params)
    M = p.num_samples + p.num_prev_elites
    for b in range(B):
        ks = ojr.split(st.key[b].cpu().numpy(), 2, prng_mode)
        carry = ks[0]
        assert np.array_equal(out_key[b].cpu().numpy(), ks[1])
        mean = np.zeros((horizon, 1), np.float32)
        std = np.full((horizon, 1), p.init_std, np.float32)
        for it in range(p.num_steps):
            carry, o_acts, pkeys = orc.icem_sample_actions(carry, mean, std, p, horizon, 1, prng_mode)
            g_acts = tr["actions"][it, b].reshape(M, horizon, 1)
            np.testing.assert_allclose(g_acts, o_acts, rtol=RTOL, atol=1e-5)
            vals = pco.system_objective_with_cost(osys, x0[b], g_acts, pkeys, p, cost.numpy, False, use_pessimism,
                                                  prng_mode)[0]
            np.testing.assert_allclose(tr["values"][it, b], vals, rtol=2e-5, atol=2e-5)
            _check_elites(vals, tr["elite_idx"][it, b], 4e-5 + 2e-5 * np.abs(vals).max())
            mean, std = tr["mean"][it, b].reshape(horizon, 1), tr["std"][it, b].reshape(horizon, 1)
    return tr


def test_noisy_pendulum_binding_cost_teacher_forced(mb, cuda_device, prng_mode):
    """Mean and pessimism against the oracle; on the same keys pessimism picks different elites."""
    elites = [_noisy_binding_plan(mb, cuda_device, prng_mode, pes)["elite_idx"] for pes in (False, True)]
    assert not np.array_equal(elites[0], elites[1])


@pytest.mark.parametrize("use_pessimism", [False, True])
def test_ensemble_binding_cost_teacher_forced(mb, cuda_device, ens, use_pessimism):
    system, sp = _ensemble_system(mb, cuda_device, ens)
    horizon, B, lam = 10, 2, 1.0
    params = dict(num_samples=64, num_elites=8, num_particles=E, num_steps=2, lambda_constraint=lam)
    x0 = _pendulum_states(B, 1101)
    keys = _keys(B, 1102)
    cost = SpeedLimit(float(np.abs(x0[:, 2]).mean()))
    opt = _opt(mb, system, horizon, cost, use_pessimism=use_pessimism, **params)
    st = opt.init(_dev(keys, cuda_device))
    x0_d = _dev(x0, cuda_device)
    seq, val, _, tr = opt._plan_raw(x0_d, st.key, st.best_sequence, st.system_params, trace=True)
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    p = orc.ICemParams(**params)
    M = p.num_samples + p.num_prev_elites
    for it in range(p.num_steps):
        g_acts = tr["actions"][it].reshape(B, M, horizon)
        vals = pco.ensemble_objective_with_cost(x0, g_acts, ens, cost.numpy, False, use_pessimism, lam)[0]
        np.testing.assert_allclose(tr["values"][it], vals, rtol=5e-3, atol=1e-2)
        for b in range(B):
            _check_elites(vals[b], tr["elite_idx"][it, b], 1e-2 + 5e-3 * np.abs(vals[b]).max())
    # best_reward is the penalised objective of best_sequence, recomputed from its own buffers
    obs, rew = system.ensemble_transitions(st.system_params, x0_d, seq.reshape(B, 1, horizon, 1))
    c = cost.numpy(obs.reshape(B * E, horizon, 3).cpu().numpy(), None).reshape(B, E)
    got = _tail(mb, cuda_device, rew.reshape(B, E, horizon), _dev(c, cuda_device), horizon, E, 0, int(use_pessimism),
                lam)
    assert torch.equal(got, val)


def test_ensemble_pessimism_changes_the_elites(mb, cuda_device, ens):
    system, _ = _ensemble_system(mb, cuda_device, ens)
    horizon, B = 10, 4
    params = dict(num_samples=64, num_elites=8, num_particles=E, num_steps=2, lambda_constraint=1.0)
    x0 = _pendulum_states(B, 1201)
    cost = SpeedLimit(float(np.abs(x0[:, 2]).mean()))
    keys = _dev(_keys(B, 1202), cuda_device)
    elites = []
    for pes in (False, True):
        opt = _opt(mb, system, horizon, cost, use_pessimism=pes, **params)
        st = opt.init(keys)
        elites.append(opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params,
                                    trace=True)[3]["elite_idx"].cpu().numpy())
    assert not np.array_equal(elites[0], elites[1])


def test_point_mass_best_reward_from_buffers(mb, cuda_device):
    system, _ = _general(mb, "point_mass")
    horizon, B, P, lam = 20, 3, 4, 2.0
    params = dict(num_samples=128, num_elites=12, num_particles=P, num_steps=3, lambda_constraint=lam)
    cost = SpeedLimit(0.5)
    x0 = _dev(_general_states("point_mass", B, 1301), cuda_device)
    for pes in (False, True):
        opt = _opt(mb, system, horizon, cost, use_pessimism=pes, **params)
        st = opt.init(_dev(_keys(B, 1302), cuda_device))
        new = opt.optimize(x0, st)
        _, obs, rew, _ = system.objective(st.system_params, x0, new.best_sequence.reshape(B, 1, horizon, 2),
                                          num_particles=P, full=True)
        c = cost.numpy(obs.reshape(B * P, horizon, 4).cpu().numpy(), None).reshape(B, P)
        got = _tail(mb, cuda_device, rew.reshape(B, P, horizon), _dev(c, cuda_device), horizon, P, 0, int(pes), lam)
        assert torch.equal(got, new.best_reward)


# ---- 6. closed loop and refusals ---------------------------------------------------------------------------------
def test_closed_loop_with_cost_equals_successive_acts(mb, cuda_device, prng_mode):
    system, _ = _general(mb, "noisy_pendulum")
    horizon, B, T = 15, 2, 3
    params = dict(num_samples=64, num_elites=8, num_particles=3, num_steps=2, lambda_constraint=1.0)
    opt = _opt(mb, system, horizon, SpeedLimit(3.0), use_pessimism=True, **params)
    x0 = _dev(_pendulum_states(B, 1401), cuda_device)
    st = opt.init(_dev(_keys(B, 1402), cuda_device))
    states, rewards, actions, end = opt.closed_loop(x0, st, T)
    x, s, sp = x0, st, st.system_params
    for t in range(T):
        u, s = opt.act(x, s)
        nxt = system.step(x, u, sp)
        sp, x = nxt.system_params, nxt.x_next
        assert torch.equal(actions[t], u) and torch.equal(states[t], x) and torch.equal(rewards[t], nxt.reward)
    assert torch.equal(end.best_sequence, s.best_sequence) and torch.equal(end.key, s.key)


def test_refusals(mb, cuda_device, ens):
    system, _ = _ensemble_system(mb, cuda_device, ens)
    x0 = _dev(_pendulum_states(2, 1501), cuda_device)
    keys = _dev(_keys(2, 1502), cuda_device)
    for cost, bounds in ((SpeedLimit(1.0), -1.0), (None, [[-1.0]] * 9 + [[-0.5]])):
        opt = _opt(mb, system, 10, cost, num_samples=32, num_elites=4, num_particles=3, num_steps=1, u_min=bounds)
        with pytest.raises(mb._lib.MbpoUnsupported, match="num_members"):
            opt.optimize(x0, opt.init(keys))
    wrong = lambda states, actions: states[:, 2].abs() - 1.0            # [H] per trajectory, not a scalar
    for sysm in (_general(mb, "noisy_pendulum")[0], _general(mb, "point_mass")[0], system):
        P = E if sysm is system else 2
        opt = _opt(mb, sysm, 10, wrong, num_samples=32, num_elites=4, num_particles=P, num_steps=1)
        xs = x0 if sysm.x_dim == 3 else _dev(_general_states("point_mass", 2, 1503), cuda_device)
        with pytest.raises(ValueError, match="one scalar per trajectory"):
            opt.optimize(xs, opt.init(keys))
