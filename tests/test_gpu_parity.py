"""GPU parity tests: the CUDA path (through the C ABI / the host mirror) against the CPU oracle.

Bars (BASELINE.json north_star): uint32 PRNG words and elite indices bit-exact; states,
returns and refit mean/std within rel 1e-5 (fp32).  Floats that depend on libm
(log1p/atan2/sin/cos) differ from the NumPy oracle by a few ulp, so tolerances are stated per
test.  Chaotic amplification over long open-loop rollouts is handled by teacher forcing
(SURVEY.md section 7).
"""
import numpy as np
import pytest
import torch

import f64_truth as ft
from oracle import jax_prng as ojr
from oracle import mbpo_oracle as orc

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _beyond(got, want, rtol=RTOL, atol=1e-6):
    """Rows outside the north star's tolerance (counted and explained, never excused by a quota)."""
    return np.abs(np.asarray(got, np.float64) - want) > rtol * np.abs(want) + atol


def _check_returns_against_truth(name, x0_rows, acts_rows, got, budget_report, oracle_vals=None, max_frac=1.0,
                                 particles=1):
    """Open-loop returns of float32 rollouts against the float64 truth of the same (x0, actions): EVERY row must
    lie inside the first-order amplification bound of its own rollout (tests/f64_truth.py).  The rows beyond rel
    1e-5 of the float32 oracle are counted and each of them must be one whose bound itself exceeds that tolerance
    (an f64-bounded amplification); the counts go to the budget report."""
    r64, bound = ft.rollout_return_budget(x0_rows, acts_rows)
    if particles > 1:                                     # float32 mean over P identical particles: P + 1 roundings
        bound = bound + (particles + 1) * ft.U * np.abs(r64)
    got = np.asarray(got, np.float64).reshape(-1)
    frac = np.abs(got - r64) / bound
    rec = dict(rows=int(got.size), max_frac=float(frac.max()), median_frac=float(np.median(frac)))
    assert frac.max() <= max_frac, "%s: a float32 return is %.2f x its float64 amplification bound" % (name, frac.max())
    if oracle_vals is not None:
        ov = np.asarray(oracle_vals, np.float64).reshape(-1)
        ofrac = np.abs(ov - r64) / bound
        assert ofrac.max() <= max_frac
        miss = _beyond(got, ov)
        rec.update(oracle_max_frac=float(ofrac.max()), rows_beyond_rel_1e5_of_oracle=int(miss.sum()))
        # a miss is explained only if both float32 values are inside a bound that is itself wider than the tolerance
        assert np.all(2 * bound[miss] > RTOL * np.abs(r64[miss])), "%s: unexplained miss" % name
    budget_report(name, **rec)
    return r64, bound


@pytest.fixture(scope="module")
def mb(cuda_device):
    import mbpo_b200
    return mbpo_b200


def _keys(n, seed=0):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2 ** 32, size=(n, 2), dtype=np.uint64).astype(np.uint32)


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


@pytest.fixture(params=[False, True], ids=["legacy", "partitionable"])
def prng_mode(request, mb):
    mb.config.threefry_partitionable = request.param
    yield request.param
    mb.config.threefry_partitionable = False


@pytest.fixture(params=["reference", "theta_carry"])
def math_mode(request, mb):
    mb.config.math_mode = request.param
    yield request.param
    mb.config.math_mode = "reference"


# ---------------------------------------------------------------------------------------------
# PRNG: bit-exact
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("num", [1, 2, 3, 7, 501])
def test_split_bit_exact(mb, cuda_device, prng_mode, num):
    keys = _keys(33, seed=num)
    got = mb.random.split(_dev(keys, cuda_device), num).cpu().numpy()
    want = orc.split_keys(keys, num, prng_mode)
    assert got.dtype == np.uint32 and np.array_equal(got, want)


@pytest.mark.parametrize("n", [1, 2, 11, 16, 26, 1000])
def test_random_bits_bit_exact(mb, cuda_device, prng_mode, n):
    keys = _keys(17, seed=n)
    got = mb.random.random_bits(_dev(keys, cuda_device), n).cpu().numpy()
    assert np.array_equal(got, orc.random_bits_keys(keys, n, prng_mode))


def test_prngkey_and_known_answers(mb, cuda_device):
    k0 = mb.random.PRNGKey(0, cuda_device)
    assert k0.cpu().numpy().tolist() == [0, 0]
    assert mb.random.split(k0).cpu().numpy().tolist() == [[4146024105, 967050713], [2718843009, 1272950319]]
    assert abs(float(mb.random.normal(k0, 1)[0]) - (-0.20584226)) < 1e-6
    assert abs(float(mb.random.uniform(k0, 1)[0]) - 0.41845703) < 1e-7
    assert abs(float(mb.random.normal(mb.random.PRNGKey(42, cuda_device), 1)[0]) - (-0.18471177)) < 1e-6


def test_uniform_normal_vs_oracle(mb, cuda_device, prng_mode):
    keys = _keys(64, seed=5)
    n = 257
    bits = orc.random_bits_keys(keys, n, prng_mode)
    u = mb.random.uniform(_dev(keys, cuda_device), n, -2.0, 3.0).cpu().numpy()
    assert np.array_equal(u, ojr.bits_to_uniform(bits, -2.0, 3.0))          # pure bit ops + one fma-free affine
    z = mb.random.normal(_dev(keys, cuda_device), n).cpu().numpy()
    np.testing.assert_allclose(z, ojr.bits_to_normal(bits), rtol=2e-6, atol=1e-7)   # log1pf/sqrtf: few ulp
    z64 = ft.normal_truth(bits)
    assert np.all(np.abs(z - z64) <= ft.NORMAL_REL * np.abs(z64) + ft.NORMAL_ABS)
    assert np.all(np.abs(ojr.bits_to_normal(bits) - z64) <= ft.NORMAL_REL * np.abs(z64) + ft.NORMAL_ABS)


# ---------------------------------------------------------------------------------------------
# stage 1: colored noise and action sampling
# ---------------------------------------------------------------------------------------------
def _cfg(mb, horizon, params, action_dim=1):
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    opt = iCemTO(horizon=horizon, action_dim=action_dim, opt_params=iCemParams(**params))
    opt.set_system(PendulumSystem())
    return opt, opt._cfg()


@pytest.mark.parametrize("horizon", [5, 8, 15, 20, 30, 50])
@pytest.mark.parametrize("exponent", [0.0, 2.0])
def test_powerlaw_noise(mb, cuda_device, prng_mode, horizon, exponent, budget_report):
    L = mb._lib
    _, cfg = _cfg(mb, horizon, dict(exponent=exponent))
    keys = _keys(300, seed=horizon)
    F = horizon // 2 + 1
    dkeys = _dev(keys, cuda_device)
    out = torch.empty((300, horizon), dtype=torch.float32, device=cuda_device)
    bits = torch.empty((300, 2, F), dtype=torch.uint32, device=cuda_device)
    L.check(L.lib.mbpo_powerlaw_noise(L.C.byref(cfg), L.ptr(dkeys), 300, L.ptr(out), L.ptr(bits),
                                      L.stream_ptr(cuda_device)))
    want, br, bi = orc.powerlaw_psd_gaussian_keys(exponent, horizon, keys, prng_mode, return_bits=True)
    got_bits = bits.cpu().numpy()
    assert np.array_equal(got_bits[:, 0], br) and np.array_equal(got_bits[:, 1], bi)      # bit-exact words
    # s_scale / sigma computed by the C host helper match the oracle's float32 tables
    s_scale, sigma = orc.powerlaw_tables(exponent, horizon)
    np.testing.assert_allclose(np.array(cfg.s_scale[:F]), s_scale, rtol=2e-7)
    np.testing.assert_allclose(cfg.sigma, sigma, rtol=3e-7)
    # direct f32 DFT vs the oracle's double-precision irfft: unit-variance rows, abs error ~1e-6
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=RTOL, atol=5e-6)
    # float64 truth of the same words (tests/f64_truth.py): kernel and float32 oracle inside one stated budget
    truth = ft.powerlaw_truth(exponent, horizon, br, bi)
    f_gpu = float(np.abs(out.cpu().numpy() - truth).max() / ft.noise_budget(horizon))
    f_orc = float(np.abs(want - truth).max() / ft.noise_budget(horizon))
    budget_report("gpu/noise_H%d_exp%g_%s" % (horizon, exponent, "part" if prng_mode else "legacy"),
                  noise_frac=f_gpu, oracle_noise_frac=f_orc)
    assert f_gpu <= 1.0 and f_orc <= 1.0, (f_gpu, f_orc)


@pytest.mark.parametrize("horizon,action_dim", [(20, 1), (30, 1), (8, 3)])
def test_sample_actions(mb, cuda_device, prng_mode, horizon, action_dim):
    L = mb._lib
    params = dict(num_samples=64, num_elites=10, exponent=1.0)
    _, cfg = _cfg(mb, horizon, params, action_dim)
    B, N, Np = 5, 64, cfg.num_prev_elites
    assert Np == 3
    rng = np.random.default_rng(1)
    keys = _keys(B, seed=9)
    mean = rng.uniform(-0.5, 0.5, (B, horizon, action_dim)).astype(np.float32)
    std = rng.uniform(0.1, 0.8, (B, horizon, action_dim)).astype(np.float32)
    acts = torch.empty((B, N + Np, horizon, action_dim), dtype=torch.float32, device=cuda_device)
    nk = torch.empty((B, 2), dtype=torch.uint32, device=cuda_device)
    pk = torch.empty((B, N + Np, 2), dtype=torch.uint32, device=cuda_device)
    dk, dm, ds = _dev(keys, cuda_device), _dev(mean, cuda_device), _dev(std, cuda_device)
    L.check(L.lib.mbpo_icem_sample_actions(L.C.byref(cfg), L.ptr(dk), L.ptr(dm), L.ptr(ds), B, L.ptr(acts), L.ptr(nk),
                                           L.ptr(pk), L.stream_ptr(cuda_device)))
    p = orc.ICemParams(**params)
    for b in range(B):
        want_key, want_acts, want_pk = orc.icem_sample_actions(keys[b], mean[b], std[b], p, horizon, action_dim,
                                                               prng_mode)
        assert np.array_equal(nk[b].cpu().numpy(), want_key)
        assert np.array_equal(pk[b].cpu().numpy(), want_pk)
        np.testing.assert_allclose(acts[b].cpu().numpy(), want_acts, rtol=RTOL, atol=5e-6)
        assert np.all(acts[b, N:].cpu().numpy() == 0.0)          # closure prev_elites quirk: zero rows


# ---------------------------------------------------------------------------------------------
# any horizon: iCemTO(horizon=h) is a free int in the reference (icem_optimizer.py:94-96)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("horizon", [2, 3, 4, 6, 7, 10, 11, 13, 21, 25, 33, 40, 47, 64, 77, 128])
def test_any_horizon_noise_vs_oracle(mb, cuda_device, prng_mode, horizon, budget_report):
    """Horizons without an unrolled instance run the rolled-loop kernel: words bit-exact, floats to tolerance and
    inside the float64 budget, for even / odd / prime / maximal sizes."""
    L = mb._lib
    exponent = 1.0 if horizon % 3 else 0.0
    _, cfg = _cfg(mb, horizon, dict(exponent=exponent))
    M = 200
    keys = _keys(M, seed=100 + horizon)
    F = horizon // 2 + 1
    dkeys = _dev(keys, cuda_device)
    out = torch.empty((M, horizon), dtype=torch.float32, device=cuda_device)
    bits = torch.empty((M, 2, F), dtype=torch.uint32, device=cuda_device)
    L.check(L.lib.mbpo_powerlaw_noise(L.C.byref(cfg), L.ptr(dkeys), M, L.ptr(out), L.ptr(bits),
                                      L.stream_ptr(cuda_device)))
    want, br, bi = orc.powerlaw_psd_gaussian_keys(exponent, horizon, keys, prng_mode, return_bits=True)
    got_bits = bits.cpu().numpy()
    assert np.array_equal(got_bits[:, 0], br) and np.array_equal(got_bits[:, 1], bi)
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=RTOL, atol=5e-6)
    truth = ft.powerlaw_truth(exponent, horizon, br, bi)
    f_gpu = float(np.abs(out.cpu().numpy() - truth).max() / ft.noise_budget(horizon))
    budget_report("gpu/noise_rolled_H%d_%s" % (horizon, "part" if prng_mode else "legacy"), noise_frac=f_gpu)
    assert f_gpu <= 1.0, f_gpu


@pytest.mark.parametrize("horizon", [5, 8, 15, 20, 30, 50])
@pytest.mark.parametrize("exponent", [0.0, 2.0])
def test_rolled_noise_kernel_bit_identical_to_unrolled(mb, cuda_device, prng_mode, horizon, exponent):
    """Same key tree, same words, same operation order: at the six unrolled horizons the any-horizon kernel gives
    the unrolled instances' bits (so a plan's results do not depend on which one sampled it)."""
    L = mb._lib
    _, cfg = _cfg(mb, horizon, dict(exponent=exponent))
    M = 1000
    dkeys = _dev(_keys(M, seed=7 * horizon), cuda_device)
    a, b = (torch.empty((M, horizon), dtype=torch.float32, device=cuda_device) for _ in range(2))
    ba, bb = (torch.empty((M, 2, horizon // 2 + 1), dtype=torch.uint32, device=cuda_device) for _ in range(2))
    L.check(L.lib.mbpo_powerlaw_noise(L.C.byref(cfg), L.ptr(dkeys), M, L.ptr(a), L.ptr(ba), L.stream_ptr(cuda_device)))
    L.check(L.lib.mbpo_powerlaw_noise_rolled(L.C.byref(cfg), L.ptr(dkeys), M, L.ptr(b), L.ptr(bb),
                                             L.stream_ptr(cuda_device)))
    assert torch.equal(ba.view(torch.int32), bb.view(torch.int32))
    assert torch.equal(a, b)


@pytest.mark.parametrize("horizon,action_dim", [(10, 1), (25, 1), (7, 2)])
def test_any_horizon_sample_actions(mb, cuda_device, prng_mode, horizon, action_dim):
    L = mb._lib
    params = dict(num_samples=64, num_elites=10, exponent=1.0)
    _, cfg = _cfg(mb, horizon, params, action_dim)
    B, N, Np = 4, 64, cfg.num_prev_elites
    rng = np.random.default_rng(1)
    keys = _keys(B, seed=9)
    mean = rng.uniform(-0.5, 0.5, (B, horizon, action_dim)).astype(np.float32)
    std = rng.uniform(0.1, 0.8, (B, horizon, action_dim)).astype(np.float32)
    acts = torch.empty((B, N + Np, horizon, action_dim), dtype=torch.float32, device=cuda_device)
    nk = torch.empty((B, 2), dtype=torch.uint32, device=cuda_device)
    pk = torch.empty((B, N + Np, 2), dtype=torch.uint32, device=cuda_device)
    dk, dm, ds = _dev(keys, cuda_device), _dev(mean, cuda_device), _dev(std, cuda_device)
    L.check(L.lib.mbpo_icem_sample_actions(L.C.byref(cfg), L.ptr(dk), L.ptr(dm), L.ptr(ds), B, L.ptr(acts), L.ptr(nk),
                                           L.ptr(pk), L.stream_ptr(cuda_device)))
    p = orc.ICemParams(**params)
    for b in range(B):
        want_key, want_acts, want_pk = orc.icem_sample_actions(keys[b], mean[b], std[b], p, horizon, action_dim,
                                                               prng_mode)
        assert np.array_equal(nk[b].cpu().numpy(), want_key) and np.array_equal(pk[b].cpu().numpy(), want_pk)
        np.testing.assert_allclose(acts[b].cpu().numpy(), want_acts, rtol=RTOL, atol=5e-6)
        assert np.all(acts[b, N:].cpu().numpy() == 0.0)


@pytest.mark.parametrize("horizon", [10, 25, 40])
def test_any_horizon_plan_vs_oracle(mb, cuda_device, horizon, budget_report):
    """iCemTO(horizon=h) for horizons without an unrolled instance: the any-horizon FUSED kernel (rolled sampling
    loops, one launch) against the oracle, free-running with the explanation walk; it gives the staged plan's bits
    (the same per-stage device functions); the closed loop runs in one launch too and equals plan -> System.step."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    B = 5
    params = dict(num_samples=150, num_elites=15, num_particles=1, num_steps=3)
    opt = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params))
    system = PendulumSystem()
    opt.set_system(system)
    assert mb._lib.lib.mbpo_icem_plan_is_fused(mb._lib.C.byref(opt._cfg())) == 1
    keys = _keys(B, seed=200 + horizon)
    x0 = _random_states(B, 201 + horizon)
    st, seq, val = _free_running_vs_oracle("any_horizon_H%d" % horizon, opt, mb, cuda_device, x0, keys, params,
                                           horizon, budget_report)
    action, new = opt.act(_dev(x0, cuda_device), st)
    assert torch.equal(new.best_sequence, seq) and torch.equal(new.best_reward, val)
    s_seq, s_val, s_key, _ = opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params, staged=True)
    assert torch.equal(s_seq, seq) and torch.equal(s_val, val) and torch.equal(s_key.view(torch.int32), new.key.view(torch.int32))
    states, rewards, actions, fin = opt.closed_loop(_dev(x0, cuda_device), st, 4)          # one launch
    assert states.shape == (4, B, 3) and rewards.shape == (4, B) and actions.shape == (4, B, 1)
    assert torch.equal(actions[0], action)
    one = system.step(_dev(x0, cuda_device), action, st.system_params)
    assert torch.equal(states[0], one.x_next) and torch.equal(rewards[0], one.reward)
    single, x0c, keyc, seqc = opt._canon(_dev(x0, cuda_device), st)
    s2, r2, a2, fin2 = opt._closed_loop_staged(single, x0c, keyc, seqc, st, 4)           # plan -> step launches
    assert torch.equal(states, s2) and torch.equal(rewards, r2) and torch.equal(actions, a2)
    assert torch.equal(fin.best_sequence, fin2.best_sequence)


@pytest.mark.parametrize("target", [0.0, 3.0, -6.0, 7.5, 40.0])
def test_plan_target_angle_inside_and_outside_the_fused_range(mb, cuda_device, target):
    """The fused kernel's reward wrap assumes |target_angle| <= 6 rad (no fmod slow path in its instruction stream);
    beyond that the same plan runs staged.  Either way the returns match the oracle's floored mod
    (pendulum_reward.py:34-35) and best_reward is the return of best_sequence."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem, PendulumRewardParams, SystemParams, PendulumDynamicsParams
    from mbpo_b200.utils import rollout_returns
    H, B = 20, 6
    opt = iCemTO(horizon=H, action_dim=1, opt_params=iCemParams(num_samples=128, num_elites=16, num_particles=1,
                                                                 num_steps=3))
    system = PendulumSystem()
    opt.set_system(system)
    sp = SystemParams(dynamics_params=PendulumDynamicsParams(), reward_params=PendulumRewardParams(target_angle=target))
    st = opt.init(_dev(_keys(B, seed=61), cuda_device)).replace(system_params=sp)
    x0 = _random_states(B, 62)
    assert opt._fused(opt._cfg(), system.pack_params(sp)) == (abs(target) <= 6.0)
    action, new = opt.act(_dev(x0, cuda_device), st)
    ret = rollout_returns(system, sp, _dev(x0, cuda_device), new.best_sequence.reshape(B, 1, H, 1))[:, 0]
    assert torch.equal(ret, new.best_reward)                      # fused and staged rollouts: the same bits
    p = orc.PendulumParams(target_angle=target)
    want = orc.rollout_actions(x0, new.best_sequence.cpu().numpy().reshape(B, H), p)
    r64 = orc.rollout_actions(x0.astype(np.float64), new.best_sequence.cpu().numpy().reshape(B, H).astype(np.float64),
                              p, dtype=np.float64)
    np.testing.assert_allclose(ret.cpu().numpy(), r64, rtol=RTOL, atol=2e-6)
    np.testing.assert_allclose(want, r64, rtol=RTOL, atol=2e-6)


def test_icemopt_reference_test_at_an_uncompiled_horizon(mb, cuda_device):
    """tests/test_icemopt.py with horizon=25 (no unrolled kernel): the closed loop still swings the pendulum up."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    jr = mb.random
    ks = jr.split(jr.PRNGKey(0, cuda_device), 3)
    system = PendulumSystem()
    system_state = system.reset(ks[2])
    cem = iCemTO(horizon=25, action_dim=1, system=None, opt_params=iCemParams(num_particles=1), key=ks[0])
    cem.set_system(system)
    states, rewards, actions, _ = cem.closed_loop(system_state.x_next, cem.init(ks[1]), 200)
    assert float(rewards.sum()) >= -400, float(rewards.sum())


# ---------------------------------------------------------------------------------------------
# stage 2: System.step and rollouts
# ---------------------------------------------------------------------------------------------
def _random_states(n, seed):
    rng = np.random.default_rng(seed)
    th = rng.uniform(-np.pi, np.pi, n)
    w = rng.uniform(-8, 8, n)
    return np.stack([np.cos(th), np.sin(th), w], axis=-1).astype(np.float32)


def test_system_step(mb, cuda_device, math_mode, budget_report):
    from mbpo_b200.systems import PendulumSystem
    sys_ = PendulumSystem()
    st = sys_.reset(mb.random.split(mb.random.PRNGKey(0, cuda_device), 20))      # tests/test_sys_pendulum.py
    assert st.x_next.shape == (20, 3)
    x = _random_states(4096, 0)
    u = np.random.default_rng(1).uniform(-1.5, 1.5, (4096, 1)).astype(np.float32)   # beyond the torque clip too
    out = sys_.step(_dev(x, cuda_device), _dev(u, cuda_device), st.system_params)
    assert out.x_next.shape == (4096, 3) and out.reward.shape == (4096,)
    assert out.system_params.key is None                                           # key dropped (:38)
    xn, r = orc.pendulum_step(x, u[:, 0])
    np.testing.assert_allclose(out.x_next.cpu().numpy(), xn, rtol=RTOL, atol=2e-6)
    np.testing.assert_allclose(out.reward.cpu().numpy(), r, rtol=RTOL, atol=2e-6)
    # float64 truth of the same float32 inputs: kernel and float32 oracle inside the stated per-step budget
    fx, fr = ft.step_errors(out.x_next.cpu().numpy(), out.reward.cpu().numpy(), x, u[:, 0])
    ox, orr = ft.step_errors(xn, r, x, u[:, 0])
    budget_report("gpu/system_step_%s" % math_mode, state_frac=fx, reward_frac=fr, oracle_state_frac=ox,
                  oracle_reward_frac=orr, n=4096)
    assert max(fx, fr, ox, orr) <= 1.0, (fx, fr, ox, orr)
    # the wrap of the reward's floored mod (theta near +-pi), saturated speed, tiny angles
    th = np.concatenate([np.pi - np.logspace(-7, -1, 500), -np.pi + np.logspace(-7, -1, 500), np.logspace(-8, -2, 500)])
    xe = np.stack([np.cos(th), np.sin(th), np.tile([8.0, -8.0, 0.0], 500)], -1).astype(np.float32)
    ue = np.tile([1.0, -1.0, 0.3], 500).astype(np.float32)[:, None]
    oe = sys_.step(_dev(xe, cuda_device), _dev(ue, cuda_device), st.system_params)
    fx, fr = ft.step_errors(oe.x_next.cpu().numpy(), oe.reward.cpu().numpy(), xe, ue[:, 0])
    budget_report("gpu/system_step_edges_%s" % math_mode, state_frac=fx, reward_frac=fr)
    assert max(fx, fr) <= 1.0, (fx, fr)


@pytest.mark.parametrize("horizon", [1, 7, 20, 30, 50])
def test_rollout_actions_vs_oracle(mb, cuda_device, math_mode, horizon, budget_report):
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils import rollout_actions, rollout_returns
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    B, M = 7, 45                                       # ragged: 315 rows, not a multiple of 32
    x0 = _random_states(B, 3)
    acts = np.clip(np.random.default_rng(4).normal(0, 0.5, (B, M, horizon, 1)), -1, 1).astype(np.float32)
    tr = rollout_actions(sys_, sp, _dev(x0, cuda_device), _dev(acts, cuda_device), horizon)
    ret = rollout_returns(sys_, sp, _dev(x0, cuda_device), _dev(acts, cuda_device)).cpu().numpy()
    want_ret, obs, rew, nxt = orc.rollout_actions(np.repeat(x0, M, axis=0), acts.reshape(B * M, horizon), full=True)
    # teacher-forced per-step parity: step the oracle from the GPU's own observations
    g_obs = tr.observation.cpu().numpy().reshape(-1, 3)
    g_nxt = tr.next_observation.cpu().numpy().reshape(-1, 3)
    g_rew = tr.reward.cpu().numpy().reshape(-1)
    xn, r = orc.pendulum_step(g_obs, acts.reshape(-1))
    np.testing.assert_allclose(g_nxt, xn, rtol=RTOL, atol=3e-6)
    np.testing.assert_allclose(g_rew, r, rtol=RTOL, atol=3e-6)
    # observation[t] is next_observation[t-1], observation[0] is the initial state (optimizer_utils.py:47-50)
    o = tr.observation.cpu().numpy()
    assert np.array_equal(o[:, :, 1:], tr.next_observation.cpu().numpy()[:, :, :-1])
    assert np.array_equal(o[:, :, 0], np.broadcast_to(x0[:, None], (B, M, 3)))
    assert bool((tr.discount == 1).all())
    # every teacher-forced step inside the float64 per-step budget as well
    fx, fr = ft.step_errors(g_nxt, g_rew, g_obs, acts.reshape(-1))
    assert max(fx, fr) <= 1.0, (fx, fr)
    # returns: mean reward.  Open loop, so float32 evaluations drift apart along the unstable directions: every
    # return must stay inside the float64 amplification bound of its own rollout, misses of rel 1e-5 are counted
    np.testing.assert_allclose(ret.reshape(-1), g_rew.reshape(B * M, horizon).astype(np.float64).mean(1), rtol=2e-6)
    _check_returns_against_truth("gpu/rollout_actions_H%d_%s" % (horizon, math_mode), np.repeat(x0, M, axis=0),
                                 acts.reshape(B * M, horizon), ret, budget_report, oracle_vals=want_ret)
    # single-sequence form
    tr1 = rollout_actions(sys_, sp, _dev(x0[0], cuda_device), _dev(acts[0, 0], cuda_device), horizon)
    assert tr1.observation.shape == (horizon, 3) and tr1.reward.shape == (horizon,)
    assert np.array_equal(tr1.reward.cpu().numpy(), tr.reward[0, 0].cpu().numpy())


# ---------------------------------------------------------------------------------------------
# stage 3: elite selection + refit (bit-exact given identical inputs)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [0.0, 0.1])
@pytest.mark.parametrize("ties", [False, True])
def test_elite_refit_bit_exact(mb, cuda_device, alpha, ties):
    L = mb._lib
    horizon, N, K = 20, 500, 50
    params = dict(num_samples=N, num_elites=K, alpha=alpha)
    _, cfg = _cfg(mb, horizon, params)
    M = N + cfg.num_prev_elites
    B = 6
    rng = np.random.default_rng(7)
    acts = rng.uniform(-1, 1, (B, M, horizon)).astype(np.float32)
    acts[:, N:] = 0
    vals = rng.normal(-5, 2, (B, M)).astype(np.float32)
    if ties:
        vals = np.round(vals)                      # many exact ties across the K-th boundary
        vals[0, :7] = np.nan                       # NaN sorts last (= best) under the total order
        vals[1, 3] = -0.0
        vals[1, 4] = 0.0
    mean = rng.uniform(-0.3, 0.3, (B, horizon)).astype(np.float32)
    std = rng.uniform(0.2, 0.6, (B, horizon)).astype(np.float32)
    bval = np.array([-np.inf, -1.0, 100.0, -np.inf, -3.0, 0.0], dtype=np.float32)
    bseq = rng.uniform(-1, 1, (B, horizon)).astype(np.float32)
    d = lambda a: _dev(a, cuda_device)
    o_mean, o_std, o_bseq = (torch.empty((B, horizon), dtype=torch.float32, device=cuda_device) for _ in range(3))
    o_bval = torch.empty((B,), dtype=torch.float32, device=cuda_device)
    o_idx = torch.empty((B, K), dtype=torch.int32, device=cuda_device)
    ta, tv, tm, ts, tb, tq = d(acts), d(vals), d(mean), d(std), d(bval), d(bseq)
    L.check(L.lib.mbpo_icem_elite_refit(L.C.byref(cfg), L.ptr(ta), L.ptr(tv), L.ptr(tm), L.ptr(ts), L.ptr(tb),
                                        L.ptr(tq), B, L.ptr(o_mean), L.ptr(o_std), L.ptr(o_bval), L.ptr(o_bseq),
                                        L.ptr(o_idx), L.stream_ptr(cuda_device)))
    p = orc.ICemParams(**params)
    for b in range(B):
        m, s, bv, bs, idx = orc.icem_refit(acts[b][..., None], vals[b], mean[b][:, None], std[b][:, None], bval[b],
                                           bseq[b][:, None], p)
        assert np.array_equal(o_idx[b].cpu().numpy(), idx), "elite indices differ (problem %d)" % b
        assert np.array_equal(o_mean[b].cpu().numpy(), m[:, 0])
        assert np.array_equal(o_std[b].cpu().numpy(), s[:, 0])
        got_bv = o_bval[b].cpu().numpy()
        assert (np.isnan(got_bv) and np.isnan(bv)) or got_bv == bv
        assert np.array_equal(o_bseq[b].cpu().numpy(), np.asarray(bs)[:, 0])


# ---------------------------------------------------------------------------------------------
# fused plan, teacher-forced against the oracle iteration by iteration
# ---------------------------------------------------------------------------------------------
def _check_plan_trace(mb, cuda_device, horizon, params, B, prng_mode, exact_refit=True, budget_report=None,
                      name="plan"):
    from mbpo_b200.systems import PendulumSystem
    opt, cfg = _cfg(mb, horizon, params)
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    x0 = _random_states(B, 11)
    keys = _keys(B, seed=12)
    seq = np.random.default_rng(13).uniform(-1, 1, (B, horizon, 1)).astype(np.float32)
    out_seq, out_val, out_key, tr = opt._plan_raw(_dev(x0, cuda_device), _dev(keys, cuda_device),
                                                  _dev(seq, cuda_device), sp, trace=True)
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    p = orc.ICemParams(**params)
    N, K = p.num_samples, p.num_elites
    assert mb._lib.lib.mbpo_icem_plan_is_fused(mb._lib.C.byref(cfg)) == 1
    for b in range(B):
        ks = ojr.split(keys[b], 2, prng_mode)
        assert np.array_equal(out_key[b].cpu().numpy(), ks[1])                    # new opt_state.key (:246-247)
        carry = ks[0]
        mean = np.zeros((horizon, 1), np.float32)
        if p.warm_start:
            mean[:-1] = seq[b, 1:]
            mean[-1] = seq[b, -1]
        std = np.full((horizon, 1), p.init_std, np.float32)
        bval, bseq = np.float32(-np.inf), mean.copy()
        for it in range(p.num_steps):
            carry, acts, _ = orc.icem_sample_actions(carry, mean, std, p, horizon, 1, prng_mode)
            g_acts = tr["actions"][it, b].reshape(N + p.num_prev_elites, horizon, 1)
            np.testing.assert_allclose(g_acts, acts, rtol=RTOL, atol=5e-6)        # sampling from the GPU's own mean/std
            vals = orc.icem_objective(x0[b], g_acts, p, orc.PendulumParams())      # oracle rollout of the GPU's actions
            g_vals = tr["values"][it, b]
            M_ = g_acts.shape[0]
            _check_returns_against_truth("gpu/%s_H%d_b%d_it%d" % (name, horizon, b, it),
                                         np.broadcast_to(x0[b], (M_, 3)), g_acts[:, :, 0], g_vals,
                                         budget_report or (lambda *a, **k: None), oracle_vals=vals,
                                         particles=p.num_particles)
            # selection + refit are exact functions of (actions, values): feed the GPU's own
            mean, std, bval, bseq, idx = orc.icem_refit(g_acts, g_vals, mean, std, bval, bseq, p)
            assert np.array_equal(tr["elite_idx"][it, b], idx)
            if exact_refit:
                assert np.array_equal(tr["mean"][it, b], mean[:, 0])
                assert np.array_equal(tr["std"][it, b], std[:, 0])
            assert tr["best_value"][it, b] == bval
            mean, std = tr["mean"][it, b][:, None].copy(), tr["std"][it, b][:, None].copy()
        assert np.array_equal(out_seq[b].cpu().numpy(), np.asarray(bseq))
        assert out_val[b].cpu().numpy() == bval


@pytest.mark.parametrize("horizon,params", [
    (20, dict()),                                                            # iCemParams() defaults = config 1
    (30, dict(num_samples=512, num_particles=1)),                            # config 2
    (30, dict(num_samples=512, num_particles=1, exponent=2.0, alpha=0.1)),   # spectral + momentum paths
    (8, dict(num_samples=40, num_elites=7, num_steps=3, warm_start=False)),
    (15, dict(num_samples=100, num_elites=20, num_steps=2, exponent=1.0)),   # odd horizon
    (50, dict(num_samples=1024, num_particles=1)),                           # config 4 population
])
def test_fused_plan_teacher_forced(mb, cuda_device, prng_mode, horizon, params, budget_report):
    _check_plan_trace(mb, cuda_device, horizon, params, B=3, prng_mode=prng_mode, budget_report=budget_report,
                      name="plan_%s_%d" % ("part" if prng_mode else "legacy", len(params)))


def test_fused_plan_theta_carry(mb, cuda_device):
    mb.config.math_mode = "theta_carry"
    try:
        _check_plan_trace(mb, cuda_device, 30, dict(num_samples=512, num_particles=1), B=3, prng_mode=False)
    finally:
        mb.config.math_mode = "reference"


def _free_running_vs_oracle(name, opt, mb, cuda_device, x0, keys, params, horizon, budget_report, cost=None,
                            use_pessimism=False, lam=0.0):
    """Free-running (NOT teacher-forced) plans against the oracle, without a quota: problem by problem the two
    traces are walked iteration by iteration.  While the elite selections coincide everything must agree to
    tolerance; the first iteration where they differ must be an elite flip (or a rank / best swap) between
    candidates whose oracle values are closer than tolerance + the float64 amplification bound of their own
    rollouts (tests/f64_truth.flip_explained) -- after such a flip the two runs legitimately refit to different
    distributions, so the comparison of that problem stops there.  Counts are reported."""
    B = x0.shape[0]
    st = opt.init(_dev(keys, cuda_device))
    out_seq, out_val, out_key, tr = opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params,
                                                  trace=True)
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    p = orc.ICemParams(**params)
    M = p.num_samples + p.num_prev_elites
    flips = 0
    for b in range(B):
        otr = []
        onew = orc.icem_optimize(x0[b], orc.icem_init(keys[b], horizon), p, horizon, trace=otr,
                                 cost_fn=cost.numpy if cost is not None else None, use_pessimism=use_pessimism)
        assert np.array_equal(out_key[b].cpu().numpy(), onew.key)
        flipped = False
        for it, o in enumerate(otr):
            o_acts = o["actions"].reshape(M, horizon)
            np.testing.assert_allclose(tr["actions"][it, b], o_acts, rtol=RTOL, atol=1e-5)
            g_idx = tr["elite_idx"][it, b]
            if np.array_equal(g_idx, o["elite_idx"]):
                continue
            r64, bound = ft.rollout_return_budget(np.broadcast_to(x0[b], (M, 3)), o_acts)
            gap = RTOL * np.abs(o["values"]) + 1e-6 + 2 * bound + (p.num_particles + 1) * ft.U * np.abs(r64)
            if cost is not None:                       # the penalty lambda * relu(max |thdot| - limit): forward bound
                _, e = ft.rollout_state_budget(np.broadcast_to(x0[b], (M, 3)), o_acts)
                gap = gap + 2 * lam * e[:, :, 2].max(axis=1)
            assert ft.flip_explained(o["values"], g_idx, o["elite_idx"], gap), \
                "%s: problem %d diverges at iteration %d without a sub-tolerance elite flip" % (name, b, it)
            flips += 1
            flipped = True
            break
        if not flipped:
            np.testing.assert_allclose(out_seq[b].cpu().numpy(), onew.best_sequence, rtol=RTOL, atol=1e-5)
            np.testing.assert_allclose(float(out_val[b]), float(onew.best_reward), rtol=1e-4 if cost is not None else 2e-5,
                                       atol=1e-4 if cost is not None else 2e-6)
    budget_report("gpu/free_running_%s" % name, problems=B, explained_elite_flips=flips, agree_end_to_end=B - flips)
    print("%s: %d of %d problems agree end to end, %d stop at an explained sub-tolerance elite flip" % (
        name, B - flips, B, flips))
    return st, out_seq, out_val


def test_plan_end_to_end_vs_oracle(mb, cuda_device, budget_report):
    """Free-running (not teacher-forced) comparison through the public API + the walk of _free_running_vs_oracle."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    horizon, B = 20, 8
    params = dict(num_samples=200, num_elites=20, num_particles=1, num_steps=3)
    opt = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params))
    opt.set_system(PendulumSystem())
    keys = _keys(B, seed=21)
    x0 = _random_states(B, 22)
    st, seq, val = _free_running_vs_oracle("fused_H20", opt, mb, cuda_device, x0, keys, params, horizon, budget_report)
    action, new = opt.act(_dev(x0, cuda_device), st)                     # the public call gives the traced call's bits
    assert action.shape == (B, 1) and new.best_sequence.shape == (B, horizon, 1)
    assert torch.equal(new.best_sequence, seq) and torch.equal(new.best_reward, val)


class _SpeedLimit:
    """AbstractCost: the largest |thdot| along the trajectory must stay below `limit` (max is exact in
    float32, so the GPU and the oracle see bit-identical costs for bit-identical observations)."""

    def __init__(self, limit):
        self.limit = limit

    def __call__(self, states, actions):                       # one trajectory: [H, 3], [H, 1] -> scalar
        return states[:, 2].abs().max() - self.limit

    def numpy(self, obs, acts):                                # vmapped: [M, H, 3] -> [M]
        return (np.abs(obs[:, :, 2]).max(axis=1) - np.float32(self.limit)).astype(np.float32)


@pytest.mark.parametrize("use_pessimism", [False, True])
def test_plan_with_cost_fn_vs_oracle(mb, cuda_device, use_pessimism, budget_report):
    """iCemTO with a constraint cost (icem_optimizer.py:161-166): staged CUDA plan against the oracle."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils import rollout_actions
    horizon, B = 20, 8
    params = dict(num_samples=200, num_elites=20, num_particles=3, num_steps=3, lambda_constraint=10.0)
    cost = _SpeedLimit(5.0)
    opt = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params), cost_fn=cost,
                 use_pessimism=use_pessimism)
    system = PendulumSystem()
    opt.set_system(system)
    keys = _keys(B, seed=23)
    x0 = _random_states(B, 24)
    st, seq, val = _free_running_vs_oracle("cost_fn_%s" % ("pess" if use_pessimism else "mean"), opt, mb, cuda_device,
                                           x0, keys, params, horizon, budget_report, cost=cost,
                                           use_pessimism=use_pessimism, lam=10.0)
    action, new = opt.act(_dev(x0, cuda_device), st)
    assert action.shape == (B, 1) and new.best_sequence.shape == (B, horizon, 1)
    assert torch.equal(new.best_sequence, seq) and torch.equal(new.best_reward, val)
    # best_reward is the penalised objective of best_sequence: recompute it from the Transition
    tr = rollout_actions(system, st.system_params, _dev(x0, cuda_device), new.best_sequence.reshape(B, 1, horizon, 1),
                         horizon)
    ret = tr.reward[:, 0].cpu().numpy()
    obs = tr.observation[:, 0].cpu().numpy()
    acc = np.zeros(B, np.float32)
    for t in range(horizon):
        acc = (acc + ret[:, t]).astype(np.float32)
    rew = (acc / np.float32(horizon)).astype(np.float32)
    c = cost.numpy(obs, None)
    p3 = lambda v: ((v + v + v) / np.float32(3)).astype(np.float32)                 # mean over 3 identical particles
    c_s = c if use_pessimism else p3(c)
    want = (p3(rew) - np.float32(10.0) * np.maximum(c_s, np.float32(0))).astype(np.float32)
    np.testing.assert_allclose(new.best_reward.cpu().numpy(), want, rtol=1e-6, atol=1e-6)
    # the constraint binds for fast initial states: penalised value below the plain return there
    assert np.all(new.best_reward.cpu().numpy() <= p3(rew) + 1e-6)
    # the closed loop of a configuration without a fused kernel: plan -> System.step launches, same bits as act()
    states, rewards, actions, _ = opt.closed_loop(_dev(x0, cuda_device), st, 2)
    assert torch.equal(actions[0], action)
    one = system.step(_dev(x0, cuda_device), action, st.system_params)
    assert torch.equal(states[0], one.x_next) and torch.equal(rewards[0], one.reward)
    a2, _ = opt.act(one.x_next, new)
    assert torch.equal(actions[1], a2)


def test_plan_with_array_bounds_vs_oracle(mb, cuda_device, budget_report):
    """u_min / u_max broadcastable to (H, A) (icem_optimizer.py:47-48,191)."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    horizon, B = 20, 6
    u_min = -np.linspace(0.2, 1.0, horizon, dtype=np.float32).reshape(horizon, 1)
    u_max = np.linspace(1.0, 0.3, horizon, dtype=np.float32).reshape(horizon, 1)
    params = dict(num_samples=200, num_elites=20, num_particles=1, num_steps=3, u_min=u_min, u_max=u_max)
    opt = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params))
    opt.set_system(PendulumSystem())
    keys = _keys(B, seed=25)
    st = opt.init(_dev(keys, cuda_device))
    x0 = _random_states(B, 26)
    st, seq_t, val_t = _free_running_vs_oracle("array_bounds", opt, mb, cuda_device, x0, keys, params, horizon,
                                               budget_report)
    action, new = opt.act(_dev(x0, cuda_device), st)
    assert torch.equal(new.best_sequence, seq_t) and torch.equal(new.best_reward, val_t)
    seq = new.best_sequence.cpu().numpy()
    assert np.all(seq >= u_min[None] - 1e-7) and np.all(seq <= u_max[None] + 1e-7)
    # scalar bounds given as arrays take the fused path and agree with plain scalars bit for bit
    o1 = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(num_samples=128, num_particles=1,
                                                                     u_min=np.full((horizon, 1), -0.5, np.float32),
                                                                     u_max=0.5))
    o2 = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(num_samples=128, num_particles=1, u_min=-0.5,
                                                                     u_max=0.5))
    o1.set_system(PendulumSystem()); o2.set_system(PendulumSystem())
    n1 = o1.optimize(_dev(x0, cuda_device), st)
    n2 = o2.optimize(_dev(x0, cuda_device), st)
    assert torch.equal(n1.best_sequence, n2.best_sequence) and torch.equal(n1.best_reward, n2.best_reward)


def test_general_staged_plan_matches_fused(mb, cuda_device):
    """The Python-composed staged plan (cost / array-bounds route) with a never-binding cost reproduces the
    fused kernel bit for bit: same kernels' arithmetic, x - lambda * relu(negative) = x."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    horizon, B = 20, 5
    params = dict(num_samples=128, num_elites=16, num_particles=10, num_steps=4, alpha=0.1)
    free = _SpeedLimit(1e6)
    for optimism in (False, True):
        fused = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params), use_optimism=optimism)
        staged = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params), cost_fn=free,
                        use_optimism=optimism)
        fused.set_system(PendulumSystem()); staged.set_system(PendulumSystem())
        keys = _dev(_keys(B, seed=27), cuda_device)
        st = fused.init(keys)
        st = st.replace(best_sequence=torch.rand_like(st.best_sequence) - 0.5)    # exercise the warm start
        x0 = _dev(_random_states(B, 28), cuda_device)
        a, b_ = fused.optimize(x0, st), staged.optimize(x0, st)
        assert torch.equal(a.key, b_.key)
        assert torch.equal(a.best_sequence, b_.best_sequence) and torch.equal(a.best_reward, b_.best_reward)


def test_staged_plan_matches_fused(mb, cuda_device):
    L = mb._lib
    from mbpo_b200.systems import PendulumSystem
    horizon, B = 20, 4
    params = dict(num_samples=128, num_elites=16, num_particles=10, num_steps=4, alpha=0.1)
    opt, cfg = _cfg(mb, horizon, params)
    sp = PendulumSystem().reset(device=cuda_device).system_params
    x0, keys = _dev(_random_states(B, 31), cuda_device), _dev(_keys(B, 32), cuda_device)
    seq = torch.zeros((B, horizon, 1), device=cuda_device)
    f_seq, f_val, f_key, _ = opt._plan_raw(x0, keys, seq, sp)
    nbytes = L.lib.mbpo_icem_workspace_bytes(L.C.byref(cfg), B)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=cuda_device)
    s_seq, s_val = torch.empty_like(f_seq), torch.empty_like(f_val)
    s_key = torch.empty_like(f_key)
    pp = PendulumSystem().pack_params(sp)
    L.check(L.lib.mbpo_icem_plan_staged(L.C.byref(cfg), L.C.addressof(pp), L.ptr(x0), L.ptr(keys), L.ptr(seq), B,
                                        L.ptr(s_seq), L.ptr(s_val), L.ptr(s_key), L.ptr(ws), nbytes,
                                        L.stream_ptr(cuda_device)))
    assert torch.equal(f_key, s_key)
    assert torch.equal(f_seq, s_seq) and torch.equal(f_val, s_val)     # same device math in both paths
    with pytest.raises(mb.MbpoError):
        L.check(L.lib.mbpo_icem_plan_staged(L.C.byref(cfg), L.C.addressof(pp), L.ptr(x0), L.ptr(keys), L.ptr(seq), B,
                                            L.ptr(s_seq), L.ptr(s_val), L.ptr(s_key), L.ptr(ws), 16,
                                            L.stream_ptr(cuda_device)))


# ---------------------------------------------------------------------------------------------
# config 1: the reference's own test (tests/test_icemopt.py), closed loop, threshold -400
# ---------------------------------------------------------------------------------------------
def _icemopt_setup(mb, cuda_device):
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    jr = mb.random
    key = jr.PRNGKey(0, cuda_device)
    ks = jr.split(key, 3)
    optimizer_key, init_key, key = ks[0], ks[1], ks[2]
    system = PendulumSystem()
    system_state = system.reset(key)
    cem = iCemTO(horizon=20, action_dim=1, system=None, opt_params=iCemParams(), key=optimizer_key)
    cem.set_system(system)
    return system, system_state, cem, cem.init(init_key)


def test_icemopt_reference_test_python_loop(mb, cuda_device):
    system, system_state, cem, st = _icemopt_setup(mb, cuda_device)
    rewards = []
    for _ in range(200):
        action, st = cem.act(obs=system_state.x_next, opt_state=st)
        system_state = system.step(x=system_state.x_next, u=action, system_params=system_state.system_params)
        st = st.replace(system_params=system_state.system_params)
        rewards.append(system_state.reward)
    total = float(torch.stack(rewards).sum())
    assert total >= -400, total                                            # tests/test_icemopt.py:37-38


def test_icemopt_closed_loop_kernel_matches_python_loop(mb, cuda_device, prng_mode):
    system, system_state, cem, st = _icemopt_setup(mb, cuda_device)
    states, rewards, actions, new = cem.closed_loop(system_state.x_next, st, 200)
    assert states.shape == (200, 3) and rewards.shape == (200,) and actions.shape == (200, 1)
    assert float(rewards.sum()) >= -400
    s2, st2 = system_state, st
    for t in range(25):                                                    # same kernels, same bits
        a, st2 = cem.act(obs=s2.x_next, opt_state=st2)
        s2 = system.step(x=s2.x_next, u=a, system_params=s2.system_params)
        assert torch.equal(a, actions[t]) and torch.equal(s2.x_next, states[t]) and torch.equal(s2.reward, rewards[t])


# ---------------------------------------------------------------------------------------------
# few problems: one problem per thread-block cluster (csrc/icem_cluster_kernels.cuh) -- same bits
# ---------------------------------------------------------------------------------------------
_SCRIBBLER = {}


def _scribble_shared_memory(mb, cuda_device):
    """Run an unrelated kernel that fills the shared memory of every SM (a fused plan over 444 problems).  A cluster
    kernel launched right after one of its own launches finds its previous contents at the same offsets, which hides
    a read of a stale or never-written location; after this call it does not."""
    from mbpo_b200.systems import PendulumSystem
    if "opt" not in _SCRIBBLER:
        opt, _ = _cfg(mb, 30, dict(num_samples=512, num_particles=1, num_steps=1))
        _SCRIBBLER["opt"] = opt
        _SCRIBBLER["sp"] = PendulumSystem().reset(device=cuda_device).system_params
        _SCRIBBLER["x0"] = _dev(_random_states(444, 77), cuda_device)
        _SCRIBBLER["keys"] = _dev(_keys(444, seed=78), cuda_device)
        _SCRIBBLER["seq"] = torch.zeros((444, 30, 1), device=cuda_device)
    k = _SCRIBBLER
    k["opt"]._plan_raw(k["x0"], k["keys"], k["seq"], k["sp"], cluster=1)


@pytest.mark.parametrize("horizon,params,B", [
    (20, dict(), 1),                                                             # tests/test_icemopt.py's shape
    (30, dict(num_samples=512, num_particles=1), 3),                             # config 2's problem
    (30, dict(num_samples=512, num_particles=1, exponent=2.0, alpha=0.1), 2),
    (8, dict(num_samples=40, num_elites=7, num_steps=3, warm_start=False), 5),   # 5 candidates per CTA of 8
    (15, dict(num_samples=100, num_elites=20, num_steps=2, exponent=1.0), 2),    # ragged split, odd horizon
    (50, dict(num_samples=1024, num_particles=1, num_steps=2), 1),               # 256 candidates per CTA at C = 4
    (20, dict(), 3),                 # config 1's problem: 500 + 15 candidates; at C = 4 the CTAs own 129 or 128 rows
    (20, dict(num_samples=250, num_elites=25, elite_set_fraction=0.5, num_steps=4), 2),   # 13 kept elites: ragged virtual rows
    (20, dict(num_samples=333, num_elites=40, num_particles=3, num_steps=3), 2),          # C * R > N at every C
])
def test_cluster_plan_bit_identical(mb, cuda_device, prng_mode, horizon, params, B):
    """A problem spread over a cluster of 2 / 4 / 8 / 16 CTAs (keys, elite rows and refit columns exchanged through
    distributed shared memory; few rows per CTA: the sampling of a row shared by several warps) gives the one-CTA
    kernel's bits: final state and every per-iteration dump (actions, values, elite indices, mean, std, best value)."""
    from mbpo_b200.systems import PendulumSystem
    opt, cfg = _cfg(mb, horizon, params)
    sp = PendulumSystem().reset(device=cuda_device).system_params
    x0 = _dev(_random_states(B, 301), cuda_device)
    keys = _dev(_keys(B, seed=302), cuda_device)
    seq = _dev(np.random.default_rng(303).uniform(-1, 1, (B, horizon, 1)).astype(np.float32), cuda_device)
    ref = opt._plan_raw(x0, keys, seq, sp, trace=True, cluster=1)
    N = cfg.num_samples
    for c in (2, 4, 8, 16):
        if (N + c - 1) // c > 256:
            with pytest.raises(mb.MbpoUnsupported):
                opt._plan_raw(x0, keys, seq, sp, cluster=c)
            continue
        _scribble_shared_memory(mb, cuda_device)
        got = opt._plan_raw(x0, keys, seq, sp, trace=True, cluster=c)
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), "cluster %d" % c
        assert torch.equal(got[2].view(torch.int32), ref[2].view(torch.int32))
        for name in ("actions", "values", "elite_idx", "mean", "std", "best_value"):
            assert torch.equal(got[3][name], ref[3][name]), "cluster %d: %s" % (c, name)
    _scribble_shared_memory(mb, cuda_device)
    auto = opt._plan_raw(x0, keys, seq, sp)                                       # the library's own choice
    assert torch.equal(auto[0], ref[0]) and torch.equal(auto[1], ref[1])


@pytest.mark.parametrize("seed", range(12))
def test_cluster_plan_random_shapes(mb, cuda_device, prng_mode, seed):
    """Random populations / elite counts / horizons / batch sizes: every cluster size the library accepts gives the
    one-CTA kernel's final state and per-iteration dumps (ragged row counts, partial warps, kept elites that do not
    divide by the cluster size, C x R > N)."""
    from mbpo_b200.systems import PendulumSystem
    rng = np.random.default_rng(9000 + seed)
    horizon = int(rng.choice([5, 8, 15, 20, 30, 50]))
    N = int(rng.integers(64, 900))
    K = int(rng.integers(4, max(5, N // 6)))
    params = dict(num_samples=N, num_elites=K, num_steps=int(rng.integers(1, 5)),
                  elite_set_fraction=float(rng.choice([0.0, 0.1, 0.3, 0.5])), alpha=float(rng.choice([0.0, 0.2])),
                  exponent=float(rng.choice([0.0, 1.0, 2.0])), num_particles=int(rng.choice([1, 4])),
                  warm_start=bool(rng.integers(0, 2)))
    B = int(rng.integers(1, 5))
    opt, cfg = _cfg(mb, horizon, params)
    sp = PendulumSystem().reset(device=cuda_device).system_params
    x0 = _dev(_random_states(B, 9100 + seed), cuda_device)
    keys = _dev(_keys(B, seed=9200 + seed), cuda_device)
    seq = _dev(rng.uniform(-1, 1, (B, horizon, 1)).astype(np.float32), cuda_device)
    ref = opt._plan_raw(x0, keys, seq, sp, trace=True, cluster=1)
    ran = 0
    for c in (2, 4, 8, 16):
        _scribble_shared_memory(mb, cuda_device)
        try:
            got = opt._plan_raw(x0, keys, seq, sp, trace=True, cluster=c)
        except mb.MbpoUnsupported:
            continue                                    # more than 256 candidates per CTA, or too few candidates
        ran += 1
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), "cluster %d %r" % (c, params)
        assert torch.equal(got[2].view(torch.int32), ref[2].view(torch.int32))
        for name in ("actions", "values", "elite_idx", "mean", "std", "best_value"):
            assert torch.equal(got[3][name], ref[3][name]), "cluster %d: %s %r" % (c, name, params)
    assert ran >= 2


@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_plan_with_all_equal_objectives(mb, cuda_device, prng_mode, bad):
    """An initial state that is NaN (or has an infinite speed: every reward is -inf) makes EVERY candidate's objective
    equal: jnp.argsort is stable, so the elites are the last K rows in index order (the kept-elite rows among them),
    `best_value <= elite_value` is False for NaN and True for -inf.  The one-CTA kernel, every cluster size (ranked
    selection: ties broken by index; redundant selection: every key in one histogram bin) and the staged plan agree
    with each other and with the oracle's refit of the kernel's own actions; a normal problem runs beside it."""
    from mbpo_b200.systems import PendulumSystem
    horizon, params = 20, dict(num_steps=3)
    opt, cfg = _cfg(mb, horizon, params)
    p = orc.ICemParams(**params)
    N, K, Np = p.num_samples, p.num_elites, cfg.num_prev_elites
    M = N + Np
    sp = PendulumSystem().reset(device=cuda_device).system_params
    x0 = _random_states(2, 71)
    x0[1] = [np.nan, np.nan, np.nan] if bad == "nan" else [1.0, 0.0, np.inf]
    keys = _keys(2, seed=72)
    seq = np.random.default_rng(73).uniform(-1, 1, (2, horizon, 1)).astype(np.float32)
    args = (_dev(x0, cuda_device), _dev(keys, cuda_device), _dev(seq, cuda_device), sp)
    ref = opt._plan_raw(*args, trace=True, cluster=1)
    tr = {k: v.cpu().numpy() for k, v in ref[3].items()}
    vals = tr["values"][:, 1]
    assert np.all(np.isnan(vals)) if bad == "nan" else np.all(np.isneginf(vals))
    for it in range(p.num_steps):
        assert np.array_equal(tr["elite_idx"][it, 1], np.arange(M - K, M)), "stable argsort of equal keys"
    # the oracle's refit of the kernel's own actions and values, iteration by iteration
    mean = np.zeros((horizon, 1), np.float32)
    mean[:-1] = seq[1, 1:]
    mean[-1] = seq[1, -1]
    std = np.full((horizon, 1), p.init_std, np.float32)
    bval, bseq = np.float32(-np.inf), mean.copy()
    for it in range(p.num_steps):
        acts = tr["actions"][it, 1].reshape(M, horizon, 1)
        mean, std, bval, bseq, idx = orc.icem_refit(acts, tr["values"][it, 1], mean, std, bval, bseq, p)
        assert np.array_equal(tr["elite_idx"][it, 1], idx)
        assert np.array_equal(tr["mean"][it, 1], mean[:, 0]) and np.array_equal(tr["std"][it, 1], std[:, 0])
    assert np.array_equal(ref[0][1].cpu().numpy(), bseq)
    got_val = ref[1][1].item()
    assert np.isneginf(got_val) and np.isneginf(bval)       # NaN never replaces -inf; -inf <= -inf takes the elite
    if bad == "inf":
        assert np.array_equal(bseq, tr["actions"][p.num_steps - 1, 1].reshape(M, horizon, 1)[M - 1])
    for c in (2, 4, 8, 16):
        _scribble_shared_memory(mb, cuda_device)
        got = opt._plan_raw(*args, trace=True, cluster=c)
        assert torch.equal(got[0], ref[0]), "cluster %d" % c
        assert torch.equal(got[1].view(torch.int32), ref[1].view(torch.int32))
        for name in ("actions", "values", "elite_idx", "mean", "std", "best_value"):
            a_, b_ = got[3][name], ref[3][name]
            if a_.dtype.is_floating_point:               # NaN == NaN here (the payload of a dumped NaN is not specified)
                assert torch.equal(torch.isnan(a_), torch.isnan(b_)), "cluster %d: %s" % (c, name)
                a_, b_ = torch.nan_to_num(a_, nan=0.0), torch.nan_to_num(b_, nan=0.0)
            assert torch.equal(a_, b_), "cluster %d: %s" % (c, name)
    staged = opt._plan_raw(*args, staged=True)
    assert torch.equal(staged[0], ref[0]) and torch.equal(staged[1].view(torch.int32), ref[1].view(torch.int32))


@pytest.mark.parametrize("seed", range(6))
def test_cluster_closed_loop_random_shapes(mb, cuda_device, prng_mode, seed):
    """The one-launch closed loop on clusters against the one-CTA closed loop for random populations, bounds,
    momentum, noise colours and batch sizes (states, rewards, actions, final sequence and key: bit-identical)."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    rng = np.random.default_rng(9500 + seed)
    horizon = int(rng.choice([8, 15, 20, 30]))
    N = int(rng.integers(64, 700))
    params = dict(num_samples=N, num_elites=int(rng.integers(4, max(5, N // 6))), num_steps=int(rng.integers(1, 4)),
                  elite_set_fraction=float(rng.choice([0.0, 0.3, 0.5])), alpha=float(rng.choice([0.0, 0.2])),
                  exponent=float(rng.choice([0.0, 2.0])), num_particles=int(rng.choice([1, 3])),
                  u_min=float(rng.choice([-1.0, -0.5])), u_max=float(rng.choice([1.0, 0.7])))
    B = int(rng.integers(1, 4))
    cem = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params))
    cem.set_system(PendulumSystem())
    x = _dev(_random_states(B, 9600 + seed), cuda_device)
    st = cem.init(_dev(_keys(B, seed=9700 + seed), cuda_device))
    one = cem.closed_loop(x, st, 6, cluster=1)
    ran = 0
    for c in (2, 4, 8, 16):
        _scribble_shared_memory(mb, cuda_device)
        try:
            got = cem.closed_loop(x, st, 6, cluster=c)
        except mb.MbpoUnsupported:
            continue
        ran += 1
        for a, b in zip(one[:3], got[:3]):
            assert torch.equal(a, b), "cluster %d %r" % (c, params)
        assert torch.equal(one[3].best_sequence, got[3].best_sequence)
        assert torch.equal(one[3].key.view(torch.int32), got[3].key.view(torch.int32))
    assert ran >= 2


@pytest.mark.parametrize("B", [1, 40, 600])
def test_plan_under_cuda_graph_capture(mb, cuda_device, B):
    """The plan is one launch on the caller's stream with no allocation or synchronisation of its own, so a caller can
    capture `iCemTO.optimize` in a CUDA graph (cluster launches included) and replay it: same bits as the eager call."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    cem = iCemTO(horizon=20, action_dim=1, opt_params=iCemParams(num_steps=3))
    cem.set_system(PendulumSystem())
    x = _dev(_random_states(B, 41), cuda_device)
    st = cem.init(_dev(_keys(B, seed=42), cuda_device))
    eager = cem.optimize(x, st)
    side = torch.cuda.Stream(device=cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        for _ in range(2):
            cem.optimize(x, st)                      # warm-up on the side stream (first-use attribute / occupancy calls)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = cem.optimize(x, st)
    captured.best_sequence.zero_()
    graph.replay()
    torch.cuda.synchronize(cuda_device)
    assert torch.equal(captured.best_sequence, eager.best_sequence)
    assert torch.equal(captured.key.view(torch.int32), eager.key.view(torch.int32))
    # new inputs through the captured buffers
    x.copy_(_dev(_random_states(B, 43), cuda_device))
    graph.replay()
    torch.cuda.synchronize(cuda_device)
    again = cem.optimize(x, st)
    assert torch.equal(captured.best_sequence, again.best_sequence)


def test_cluster_choice_and_closed_loop(mb, cuda_device, prng_mode):
    """The library spreads few problems over clusters by itself (B = 1 -> 16 CTAs, ...) and the closed loop
    (tests/test_icemopt.py:19-32) on a cluster reproduces the one-CTA closed loop bit for bit."""
    L = mb._lib
    system, system_state, cem, st = _icemopt_setup(mb, cuda_device)
    cfg = cem._cfg()
    # the choice: the largest cluster size whose clusters all run at once (the device's own occupancy answer: the GPCs
    # decide, not the SM count) with 32 .. 256 candidates per CTA
    cap = {c: L.lib.mbpo_icem_plan_cluster_capacity(L.C.byref(cfg), c) for c in (16, 8, 4, 2)}
    assert cap[16] >= 1 and cap[2] >= cap[4] >= cap[8] >= cap[16], cap
    N = cfg.num_samples
    for B in (1, 2, cap[16], cap[16] + 1, cap[8], cap[8] + 1, cap[4], cap[4] + 1, cap[2], cap[2] + 1, 148, 4096):
        want = 0
        for c in (16, 8, 4, 2):
            if 32 <= -(-N // c) <= 256 and B <= cap[c]:
                want = c
                break
        assert L.lib.mbpo_icem_plan_cluster_size(L.C.byref(cfg), B) == want, (B, want, cap)
    assert L.lib.mbpo_icem_plan_cluster_size(L.C.byref(cfg), 1) == 16
    assert L.lib.mbpo_icem_plan_cluster_size(L.C.byref(cfg), 4096) == 0
    one = cem.closed_loop(system_state.x_next, st, 40, cluster=1)
    for c in (2, 4, 8, 16, -1):
        _scribble_shared_memory(mb, cuda_device)
        got = cem.closed_loop(system_state.x_next, st, 40, cluster=c)
        for a, b in zip(one[:3], got[:3]):
            assert torch.equal(a, b), "cluster %d" % c
        assert torch.equal(one[3].best_sequence, got[3].best_sequence)
        assert torch.equal(one[3].key.view(torch.int32), got[3].key.view(torch.int32))
    # a batch of closed loops on clusters (B = 3 -> 8 CTAs each)
    x3 = _dev(_random_states(3, 311), cuda_device)
    st3 = cem.init(_dev(_keys(3, seed=312), cuda_device))
    a = cem.closed_loop(x3, st3, 5, cluster=1)
    for c in (2, 4, 8, 16):
        _scribble_shared_memory(mb, cuda_device)
        b = cem.closed_loop(x3, st3, 5, cluster=c)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]), "cluster %d" % c


# ---------------------------------------------------------------------------------------------
# config 3: vmapped env rollouts with Episode / AutoReset bookkeeping
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E,T,episode_length,action_repeat", [(1000, 57, 20, 1), (77, 40, 7, 2), (4096, 16, 200, 1)])
def test_env_rollout(mb, cuda_device, math_mode, E, T, episode_length, action_repeat):
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    env = wrap(sys_, sp, episode_length=episode_length, action_repeat=action_repeat)
    x0 = _random_states(E, 41)
    acts = np.random.default_rng(42).uniform(-1, 1, (T, E, 1)).astype(np.float32)
    st = env.reset(_dev(x0, cuda_device))
    new, tr = env.unroll(st, _dev(acts, cuda_device))
    want = orc.env_rollout(x0, acts[..., 0], episode_length, action_repeat=action_repeat)
    # bookkeeping is exact
    for name in ("discount", "truncation"):
        got = tr.discount if name == "discount" else tr.extras["state_extras"]["truncation"]
        assert np.array_equal(got.cpu().numpy(), want[name]), name
    assert np.array_equal(new.info["steps"].cpu().numpy(), want["final_steps"])
    assert np.array_equal(new.done.cpu().numpy(), want["final_done"])
    # teacher-forced float parity: step the oracle from the GPU's recorded observations
    o = tr.observation.cpu().numpy()
    x, rew = o.reshape(-1, 3), np.zeros(T * E, np.float32)
    for _ in range(action_repeat):
        x, r = orc.pendulum_step(x, acts.reshape(-1))
        rew = rew + r
    done = (1.0 - want["discount"]).reshape(-1, 1)
    nxt = np.where(done != 0, np.broadcast_to(x0[None], (T, E, 3)).reshape(-1, 3), x)
    tol = dict(rtol=RTOL * (4 if action_repeat > 1 else 1), atol=4e-6)
    np.testing.assert_allclose(tr.next_observation.cpu().numpy().reshape(-1, 3), nxt, **tol)
    np.testing.assert_allclose(tr.reward.cpu().numpy().reshape(-1), rew, **tol)
    assert np.array_equal(o[1:], tr.next_observation.cpu().numpy()[:-1])       # obs[t+1] = next_obs[t]
    assert np.array_equal(o[0], x0)
    # chunked unroll == one unroll (state carried in EnvState)
    mid = T // 3
    s1, t1 = env.unroll(st, _dev(acts[:mid], cuda_device))
    s2, t2 = env.unroll(s1, _dev(acts[mid:], cuda_device))
    cat = torch.cat([t1.next_observation, t2.next_observation])
    if math_mode == "reference":
        assert torch.equal(cat, tr.next_observation) and torch.equal(s2.obs, new.obs)
    else:   # theta is carried in a register within a launch and re-derived from [cos, sin] at its start
        assert torch.equal(cat[:mid], tr.next_observation[:mid])
        # the second chunk restarts from the rounded [cos, sin]: its trajectory leaves the single launch's, so it is
        # checked step by step from its own recorded observations (every step, no quota)
        o2 = t2.observation.cpu().numpy().reshape(-1, 3)
        x2, rew2 = o2, np.zeros(o2.shape[0], np.float32)
        for _ in range(action_repeat):
            x2, r2 = orc.pendulum_step(x2, acts[mid:].reshape(-1))
            rew2 = rew2 + r2
        nxt2 = np.where(done.reshape(T, E, 1)[mid:].reshape(-1, 1) != 0,
                        np.broadcast_to(x0[None], (T - mid, E, 3)).reshape(-1, 3), x2)
        np.testing.assert_allclose(t2.next_observation.cpu().numpy().reshape(-1, 3), nxt2, **tol)
        np.testing.assert_allclose(t2.reward.cpu().numpy().reshape(-1), rew2, **tol)
    assert torch.equal(s2.info["steps"], new.info["steps"])


def test_env_rollout_abi_variants(mb, cuda_device):
    """Separate observation buffer (OBS kernel), NULL outputs (env_unroll_general_kernel) and the aliased
    fast path, in both math modes.  In reference math all three produce identical bits.  Under theta-carry the
    NULL-output path re-derives theta every step where the segmented kernel carries it, so it is checked instead
    against a step-by-step loop of mbpo_system_step (the same atan2 -> step -> sincos) and the AutoReset
    bookkeeping."""
    try:
        for math_mode in ("reference", "theta_carry"):
            mb.config.math_mode = math_mode
            _check_env_rollout_abi_variants(mb, cuda_device, math_mode)
    finally:
        mb.config.math_mode = "reference"


def _check_env_rollout_abi_variants(mb, cuda_device, math_mode):
    L = mb._lib
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    E, T, ep_len = 333, 23, 9
    M = mb.config.math_mode_id
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    env = wrap(sys_, sp, episode_length=ep_len)
    x0 = _dev(_random_states(E, 61), cuda_device)
    acts = _dev(np.random.default_rng(62).uniform(-1, 1, (T, E, 1)).astype(np.float32), cuda_device)
    st = env.reset(x0)
    _, tr = env.unroll(st, acts)
    pp = sys_.pack_params(sp)

    def call(with_obs, with_rest):
        obs, steps, done = st.obs.clone(), st.info["steps"].clone(), st.done.clone()
        o = torch.zeros((T, E, 3), device=cuda_device) if with_obs else None
        n = torch.zeros((T, E, 3), device=cuda_device)
        r = torch.zeros((T, E), device=cuda_device)
        d = torch.zeros((T, E), device=cuda_device) if with_rest else None
        t_ = torch.zeros((T, E), device=cuda_device) if with_rest else None
        L.check(L.lib.mbpo_env_rollout(0, L.C.addressof(pp), M, 3, 1, ep_len, 1, L.ptr(obs), L.ptr(steps),
                                       L.ptr(done), L.ptr(st.info["first_obs"]), L.ptr(acts), E, T, L.ptr(o), L.ptr(r),
                                       L.ptr(d), L.ptr(n), L.ptr(t_), L.stream_ptr(cuda_device)))
        return o, n, r, d, t_, obs
    o, n, r, d, t_, obs = call(True, True)                     # OBS kernel
    assert torch.equal(o, tr.observation) and torch.equal(n, tr.next_observation) and torch.equal(r, tr.reward)
    assert torch.equal(d, tr.discount) and torch.equal(t_, tr.extras["state_extras"]["truncation"])
    o2, n2, r2, _, _, obs2 = call(True, False)                 # NULL discount / truncation
    if math_mode == "reference":
        assert torch.equal(o2, o) and torch.equal(n2, n) and torch.equal(r2, r) and torch.equal(obs2, obs)
        return
    x, steps, done = st.obs.clone(), st.info["steps"].clone(), st.done.clone()
    first = st.info["first_obs"]
    for t in range(T):
        steps = torch.where(done != 0, torch.zeros_like(steps), steps)
        assert torch.equal(o2[t], x)
        xn, rew = torch.empty_like(x), torch.empty((E,), device=cuda_device)
        L.check(L.lib.mbpo_system_step(0, L.C.addressof(pp), M, L.ptr(x), L.ptr(acts[t].contiguous()), E, L.ptr(xn),
                                       L.ptr(rew), L.stream_ptr(cuda_device)))
        steps = steps + 1.0
        over = steps >= ep_len
        done = over.to(torch.float32)
        x = torch.where(over[:, None], first, xn)
        assert torch.equal(r2[t], rew) and torch.equal(n2[t], x)
    assert torch.equal(obs2, x)


@pytest.mark.parametrize("E,T,episode_length,action_repeat", [(1000, 61, 13, 1), (95, 50, 11, 3), (64, 5, 200, 1)])
def test_env_unroll_ragged_episode_pieces(mb, cuda_device, math_mode, E, T, episode_length, action_repeat):
    """mbpo_env_unroll rolls the pieces between AutoReset points concurrently.  Envs whose step
    counters differ reset at different times inside one warp: the result must still equal the
    sequential scan (mbpo_env_rollout) bit for bit, and the oracle's bookkeeping exactly."""
    L = mb._lib
    from mbpo_b200.envs import wrap, EnvState
    from mbpo_b200.systems import PendulumSystem
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    env = wrap(sys_, sp, episode_length=episode_length, action_repeat=action_repeat)
    rng = np.random.default_rng(71)
    x0, first = _random_states(E, 72), _random_states(E, 73)
    steps0 = (rng.integers(0, episode_length, E) // action_repeat * action_repeat).astype(np.float32)
    done0 = (rng.uniform(size=E) < 0.2).astype(np.float32)
    acts = rng.uniform(-1, 1, (T, E, 1)).astype(np.float32)
    st = EnvState(obs=_dev(x0, cuda_device), reward=torch.zeros(E, device=cuda_device), done=_dev(done0, cuda_device),
                  system_params=sp, info=dict(steps=_dev(steps0, cuda_device), truncation=torch.zeros(E, device=cuda_device),
                                              first_obs=_dev(first, cuda_device)))
    new, tr = env.unroll(st, _dev(acts, cuda_device))
    assert torch.equal(st.obs, _dev(x0, cuda_device)) and torch.equal(st.info["steps"], _dev(steps0, cuda_device))
    want = orc.env_rollout(x0, acts[..., 0], episode_length, action_repeat=action_repeat, steps0=steps0, done0=done0,
                           first_obs=first)
    assert np.array_equal(tr.discount.cpu().numpy(), want["discount"])
    assert np.array_equal(tr.extras["state_extras"]["truncation"].cpu().numpy(), want["truncation"])
    assert np.array_equal(new.info["steps"].cpu().numpy(), want["final_steps"])
    assert np.array_equal(new.done.cpu().numpy(), want["final_done"])
    # the sequential kernel through the in-place entry point
    pp = sys_.pack_params(sp)
    obs, steps, done = st.obs.clone(), st.info["steps"].clone(), st.done.clone()
    n = torch.zeros((T, E, 3), device=cuda_device)
    r, d, t_ = (torch.zeros((T, E), device=cuda_device) for _ in range(3))
    L.check(L.lib.mbpo_env_rollout(0, L.C.addressof(pp), mb.config.math_mode_id, 3, 1, episode_length, action_repeat,
                                   L.ptr(obs), L.ptr(steps), L.ptr(done), L.ptr(st.info["first_obs"]),
                                   L.ptr(_dev(acts, cuda_device)), E, T, None, L.ptr(r), L.ptr(d), L.ptr(n), L.ptr(t_),
                                   L.stream_ptr(cuda_device)))
    assert torch.equal(n, tr.next_observation) and torch.equal(r, tr.reward) and torch.equal(d, tr.discount)
    assert torch.equal(t_, tr.extras["state_extras"]["truncation"])
    assert torch.equal(obs, new.obs) and torch.equal(steps, new.info["steps"]) and torch.equal(done, new.done)
    # aliasing the outgoing state with the incoming one is refused when pieces run concurrently
    if T > 1 and episode_length < T:
        with pytest.raises(mb.MbpoError):
            L.check(L.lib.mbpo_env_unroll(0, L.C.addressof(pp), 0, 3, 1, episode_length, action_repeat, L.ptr(obs),
                                          L.ptr(steps), L.ptr(done), L.ptr(obs), L.ptr(steps), L.ptr(done),
                                          L.ptr(st.info["first_obs"]), L.ptr(_dev(acts, cuda_device)), E, T, None,
                                          L.ptr(r), L.ptr(d), L.ptr(n), L.ptr(t_), L.stream_ptr(cuda_device)))


def test_env_unroll_random_shapes_match_sequential_scan(mb, cuda_device):
    """Thirty random (envs, steps, episode_length, action_repeat, step counters, done flags): the episode-piece
    launch equals the one-scan-per-env launch bit for bit, whichever loop (mask-free or general) each warp takes."""
    L = mb._lib
    from mbpo_b200.systems import PendulumSystem
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    pp = sys_.pack_params(sp)
    rng = np.random.default_rng(2024)
    for case in range(30):
        E = int(rng.choice([1, 7, 32, 33, 64, 100, 128, 255, 256, 1000, 4097]))
        T = int(rng.integers(1, 70))
        ep = int(rng.integers(1, 40))
        rep = int(rng.choice([1, 1, 1, 2, 3]))
        uniform = bool(rng.integers(0, 2))
        x0, first = _random_states(E, 500 + case), _random_states(E, 900 + case)
        steps0 = (np.zeros(E) if uniform else rng.integers(0, ep, E) // rep * rep).astype(np.float32)
        done0 = (np.zeros(E) if uniform else rng.uniform(size=E) < 0.3).astype(np.float32)
        acts = _dev(rng.uniform(-1.2, 1.2, (T, E)).astype(np.float32), cuda_device)
        outs = []
        for which in ("unroll", "rollout"):
            obs, steps, done = _dev(x0, cuda_device), _dev(steps0, cuda_device), _dev(done0, cuda_device)
            n = torch.full((T, E, 3), float("nan"), device=cuda_device)
            r, d, t_ = (torch.full((T, E), float("nan"), device=cuda_device) for _ in range(3))
            if which == "unroll":
                o2, s2, d2 = torch.empty_like(obs), torch.empty_like(steps), torch.empty_like(done)
                L.check(L.lib.mbpo_env_unroll(0, L.C.addressof(pp), 0, 3, 1, ep, rep, L.ptr(obs), L.ptr(steps), L.ptr(done),
                                              L.ptr(o2), L.ptr(s2), L.ptr(d2), L.ptr(_dev(first, cuda_device)), L.ptr(acts),
                                              E, T, None, L.ptr(r), L.ptr(d), L.ptr(n), L.ptr(t_), L.stream_ptr(cuda_device)))
                outs.append((n, r, d, t_, o2, s2, d2))
            else:
                L.check(L.lib.mbpo_env_rollout(0, L.C.addressof(pp), 0, 3, 1, ep, rep, L.ptr(obs), L.ptr(steps), L.ptr(done),
                                               L.ptr(_dev(first, cuda_device)), L.ptr(acts), E, T, None, L.ptr(r), L.ptr(d),
                                               L.ptr(n), L.ptr(t_), L.stream_ptr(cuda_device)))
                outs.append((n, r, d, t_, obs, steps, done))
        for a_, b_ in zip(*outs):
            assert torch.equal(a_, b_), (case, E, T, ep, rep, uniform)
        assert not bool(torch.isnan(outs[0][0]).any()) and not bool(torch.isnan(outs[0][1]).any())


# ---------------------------------------------------------------------------------------------
# policy in the env loop: actor_step / generate_unroll / get_experience (SURVEY 8f-2)
# ---------------------------------------------------------------------------------------------
def _policy_on_device(mb, cuda_device, pol, deterministic=False, kernel="auto"):
    from mbpo_b200.acting import Policy, PolicyParams
    return Policy(PolicyParams(weights=[_dev(w, cuda_device) for w in pol.weights],
                               biases=[_dev(b, cuda_device) for b in pol.biases], min_std=pol.min_std), deterministic,
                  kernel=kernel)


@pytest.mark.parametrize("convention", ["sac", "unroll"])
@pytest.mark.parametrize("hidden,kernel", [((64, 64, 64), "tcgen05"), ((64, 64, 64), "cuda_cores"), ((64, 64), "tcgen05"),
                                           ((64,), "auto"), ((64, 64, 64), "tcgen05_wide"), ((64, 64), "tcgen05_wide")])
def test_actor_rollout_vs_oracle(mb, cuda_device, prng_mode, math_mode, convention, hidden, kernel):
    """T steps of policy forward + NormalTanh sample + wrapped env step in one launch, per step against the
    oracle teacher-forced on the GPU's observations; the PRNG carry key is bit exact.  Both kernels: the
    float32 network on the CUDA cores, and the hidden -> hidden layers as TF32 x 3 split-precision tcgen05 MMAs."""
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    E, T, L = 333, 23, 7
    pol = orc.make_policy_params(seed=7, hidden=hidden)
    policy = _policy_on_device(mb, cuda_device, pol, kernel=kernel)
    system = PendulumSystem()
    env = wrap(system, system.reset(device=cuda_device).system_params, episode_length=L)
    x0 = _random_states(E, 91)
    key = ojr.PRNGKey(5)
    st = env.reset(_dev(x0, cuda_device))
    if convention == "sac":
        key_out, nst, tr = acting.get_experience(env, st, policy, _dev(key, cuda_device), T)
    else:
        nst, tr = acting.generate_unroll(env, st, policy, _dev(key, cuda_device), T, extra_fields=("truncation",))
        key_out = None
    g_obs = tr.observation.cpu().numpy()
    want, okey = orc.actor_rollout(pol, x0, key, T, L, key_convention=convention, partitionable=prng_mode,
                                   teacher_obs=g_obs)
    if key_out is not None:
        assert np.array_equal(key_out.cpu().numpy(), okey)
    np.testing.assert_allclose(tr.action.cpu().numpy(), want["action"], rtol=2e-5, atol=2e-6)
    # the env step is compared on the GPU's own actions (the policy was checked just above)
    g_act = tr.action.cpu().numpy()[..., 0]
    steps = np.zeros(E, np.float32); done = np.zeros(E, np.float32)
    for t in range(T):
        one = orc.env_rollout(g_obs[t], g_act[t][None], L, steps0=steps, done0=done, first_obs=x0)
        np.testing.assert_allclose(tr.reward[t].cpu().numpy(), one["reward"][0], rtol=1e-5, atol=3e-6)
        np.testing.assert_allclose(tr.next_observation[t].cpu().numpy(), one["next_observation"][0], rtol=1e-5, atol=2e-6)
        assert np.array_equal(tr.discount[t].cpu().numpy(), one["discount"][0])
        assert np.array_equal(tr.extras["state_extras"]["truncation"][t].cpu().numpy(), one["truncation"][0])
        steps, done = one["final_steps"], one["final_done"]
    assert np.array_equal(g_obs[1:], tr.next_observation[:-1].cpu().numpy())          # observation[t] = next_observation[t-1]
    assert np.array_equal(nst.obs.cpu().numpy(), tr.next_observation[-1].cpu().numpy())
    assert np.array_equal(nst.info["steps"].cpu().numpy(), steps) and np.array_equal(nst.done.cpu().numpy(), done)
    assert float(tr.action.abs().max()) <= 1.0


def test_actor_step_and_deterministic_policy(mb, cuda_device):
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    E = 1000
    pol = orc.make_policy_params(seed=8)
    system = PendulumSystem()
    env = wrap(system, system.reset(device=cuda_device).system_params, episode_length=50)
    x0 = _random_states(E, 92)
    key = ojr.PRNGKey(11)
    st = env.reset(_dev(x0, cuda_device))
    # actor_step: the key is the sample key itself (acting.py:35-55)
    nst, tr = acting.actor_step(env, st, _policy_on_device(mb, cuda_device, pol), _dev(key, cuda_device),
                                extra_fields=("truncation",))
    want = orc.policy_sample(pol, x0, key)
    np.testing.assert_allclose(tr.action.cpu().numpy(), want, rtol=2e-5, atol=2e-6)
    assert tr.observation.shape == (E, 3) and tr.action.shape == (E, 1) and tr.reward.shape == (E,)
    # the policy callable alone (make_inference_fn(...)(params)(obs, key))
    make_policy = acting.make_inference_fn()
    policy_fn = make_policy(acting.PolicyParams([_dev(w, cuda_device) for w in pol.weights],
                                                [_dev(b, cuda_device) for b in pol.biases]))
    a, extras = policy_fn(_dev(x0, cuda_device), _dev(key, cuda_device))
    assert torch.equal(a, tr.action) and extras == {}
    # deterministic: tanh(loc), no key dependence
    det = _policy_on_device(mb, cuda_device, pol, deterministic=True)
    _, t1 = acting.actor_step(env, st, det, _dev(key, cuda_device))
    _, t2 = acting.actor_step(env, st, det, _dev(ojr.PRNGKey(99), cuda_device))
    assert torch.equal(t1.action, t2.action)
    np.testing.assert_allclose(t1.action.cpu().numpy(), orc.policy_sample(pol, x0, key, deterministic=True),
                               rtol=2e-5, atol=2e-6)
    # unsupported network shapes fail loudly
    bad = orc.make_policy_params(seed=9, hidden=(32, 32))
    with pytest.raises(mb.MbpoUnsupported):
        acting.actor_step(env, st, _policy_on_device(mb, cuda_device, bad), _dev(key, cuda_device))


@pytest.mark.parametrize("E,T,chunk", [(1000, 37, 5), (256, 200, 64), (77, 10, 100)])
def test_env_unroll_streamed_equals_unroll(mb, cuda_device, E, T, chunk):
    """Actions in pinned host memory, copies and rollout overlapped on three streams: same bits as unroll, rewards
    delivered to the host buffer."""
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    system = PendulumSystem()
    env = wrap(system, system.reset(device=cuda_device).system_params, episode_length=23)
    x0 = _dev(_random_states(E, 3), cuda_device)
    acts_host = torch.from_numpy(np.random.default_rng(4).uniform(-1, 1, (T, E, 1)).astype(np.float32)).pin_memory()
    rew_host = torch.zeros((T, E), dtype=torch.float32).pin_memory()
    st = env.reset(x0)
    n1, t1 = env.unroll(st, acts_host.to(cuda_device))
    n2, t2 = env.unroll_streamed(st, acts_host, rew_host, chunk_steps=chunk)
    torch.cuda.synchronize()
    for a, b in ((t1.observation, t2.observation), (t1.action, t2.action), (t1.reward, t2.reward),
                 (t1.discount, t2.discount), (t1.next_observation, t2.next_observation),
                 (t1.extras["state_extras"]["truncation"], t2.extras["state_extras"]["truncation"]),
                 (n1.obs, n2.obs), (n1.done, n2.done), (n1.info["steps"], n2.info["steps"])):
        assert torch.equal(a, b)
    assert torch.equal(rew_host, t1.reward.cpu())
    with pytest.raises(mb.MbpoError):
        env.unroll_streamed(st, acts_host.to(cuda_device))


@pytest.mark.parametrize("hidden", [(64, 64, 64), (64, 64)])
@pytest.mark.parametrize("E,T", [(1, 3), (129, 17), (1000, 40), (4096, 5)])
def test_wide_and_four_tile_tcgen05_kernels_agree_bit_for_bit(mb, cuda_device, hidden, E, T):
    """The latency kernel (one tile per CTA, sixteen producer warps, PRNG warps) and the throughput kernel (four tiles
    per CTA, thread = env) are the same computation in the same order: every output and the carry key are equal, for
    SAC's head, PPO's extras and BPTT's actor."""
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    pol = orc.make_policy_params(seed=E + T, hidden=hidden)
    system = PendulumSystem()
    env = wrap(system, system.reset(device=cuda_device).system_params, episode_length=7)
    x0 = _dev(_random_states(E, 5), cuda_device)
    key = _dev(ojr.PRNGKey(E), cuda_device)
    params = acting.PolicyParams([_dev(w, cuda_device) for w in pol.weights], [_dev(b, cuda_device) for b in pol.biases])

    def run(kernel, which):
        if which == "ppo":
            policy = acting.Policy(params, False, [0.1, -0.2, 0.5], [0.7, 0.8, 3.0], emit_extras=True, kernel=kernel)
        elif which == "bptt":
            policy = acting.BpttActorPolicy(params, init_stddev=0.5, obs_mean=[0.1, -0.2, 0.5], obs_std=[0.7, 0.8, 3.0])
            policy.struct.kernel = {"tcgen05": mb._lib.ACTOR_TCGEN05, "tcgen05_wide": mb._lib.ACTOR_TCGEN05_WIDE}[kernel]
        else:
            policy = acting.Policy(params, which == "det", kernel=kernel)
        st = env.reset(x0)
        key_out, nst, tr = acting.get_experience(env, st, policy, key, T)
        outs = [key_out, nst.obs, nst.done, nst.info["steps"], tr.action, tr.reward, tr.discount, tr.next_observation,
                tr.extras["state_extras"]["truncation"]]
        outs += list(tr.extras["policy_extras"].values())
        return outs

    for which in ("sac", "det", "ppo", "bptt"):
        a, b = run("tcgen05", which), run("tcgen05_wide", which)
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert torch.equal(x, y), which


@pytest.mark.parametrize("kernel", ["tcgen05", "cuda_cores", "tcgen05_wide"])
def test_actor_rollout_env_sharding_is_bit_identical(mb, cuda_device, kernel):
    """Envs sharded over ranks: each shard draws its slice of normal(key, (num_envs, A)), so the shards together
    reproduce the unsharded launch bit for bit (the multi-GPU invariant of DESIGN.md section 4.3)."""
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    E, T = 700, 9
    pol = orc.make_policy_params(seed=5, hidden=(64, 64))
    policy = _policy_on_device(mb, cuda_device, pol, kernel=kernel)
    system = PendulumSystem()
    env = wrap(system, system.reset(device=cuda_device).system_params, episode_length=4)
    x0 = _dev(_random_states(E, 141), cuda_device)
    key = _dev(ojr.PRNGKey(8), cuda_device)
    k_all, s_all, tr_all = acting.get_experience(env, env.reset(x0), policy, key, T)
    cuts = [0, 256, 300, E]
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        k, s, tr = acting.get_experience(env, env.reset(x0[lo:hi].contiguous()), policy, key, T, env_offset=lo, total_envs=E)
        assert torch.equal(tr.action, tr_all.action[:, lo:hi]) and torch.equal(tr.reward, tr_all.reward[:, lo:hi])
        assert torch.equal(tr.next_observation, tr_all.next_observation[:, lo:hi]) and torch.equal(k, k_all)
        assert torch.equal(s.obs, s_all.obs[lo:hi])
    with pytest.raises(mb.MbpoError):
        acting.get_experience(env, env.reset(x0[:10].contiguous()), policy, key, T, env_offset=695, total_envs=E)


def test_ppo_policy_extras_and_normaliser(mb, cuda_device, prng_mode):
    """PPO's generate_unroll (ppo/ppo.py:194-213): the policy also returns raw_action and log_prob
    (ppo_network.py:66-80), and the policy network normalises observations with the running statistics."""
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    E, T, L = 257, 11, 6
    pol = orc.make_policy_params(seed=13, hidden=(64, 64))
    mean, std = np.array([0.05, -0.1, 0.4], np.float32), np.array([0.7, 0.75, 3.5], np.float32)
    make_policy = acting.make_ppo_inference_fn()
    policy = make_policy(acting.PolicyParams([_dev(w, cuda_device) for w in pol.weights],
                                             [_dev(b, cuda_device) for b in pol.biases]), obs_mean=mean, obs_std=std)
    system = PendulumSystem()
    env = wrap(system, system.reset(device=cuda_device).system_params, episode_length=L)
    x0 = _random_states(E, 131)
    key = ojr.PRNGKey(21)
    nst, tr = acting.generate_unroll(env, env.reset(_dev(x0, cuda_device)), policy, _dev(key, cuda_device), T,
                                     extra_fields=("truncation",))
    pe = tr.extras["policy_extras"]
    assert pe["raw_action"].shape == (T, E, 1) and pe["log_prob"].shape == (T, E)
    g_obs = tr.observation.cpu().numpy()
    k = key
    for t in range(T):
        ks = ojr.split(k, 2, prng_mode)
        k_actor, k = ks[0], ks[1]                                          # acting.py:68-73
        act, raw, logp = orc.policy_sample(pol, g_obs[t], k_actor, partitionable=prng_mode, obs_mean=mean, obs_std=std,
                                           with_extras=True)
        np.testing.assert_allclose(tr.action[t].cpu().numpy(), act, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(pe["raw_action"][t].cpu().numpy(), raw, rtol=2e-5, atol=3e-6)
        # log_prob divides by scale and takes its log: compare with a tolerance on the standardised residual
        np.testing.assert_allclose(pe["log_prob"][t].cpu().numpy(), logp, rtol=1e-4, atol=1e-4)
    assert torch.equal(torch.tanh(pe["raw_action"]), tr.action)
    # a deterministic policy returns no extras, like the reference's `{}`
    det = make_policy(acting.PolicyParams([_dev(w, cuda_device) for w in pol.weights],
                                          [_dev(b, cuda_device) for b in pol.biases]), deterministic=True,
                      obs_mean=mean, obs_std=std)
    _, trd = acting.generate_unroll(env, env.reset(_dev(x0, cuda_device)), det, _dev(key, cuda_device), 2)
    assert trd.extras["policy_extras"] == {}
    want = np.tanh(orc.policy_logits(pol, ((x0 - mean) / std).astype(np.float32))[:, :1])
    np.testing.assert_allclose(trd.action[0].cpu().numpy(), want, rtol=2e-5, atol=2e-6)


# ---------------------------------------------------------------------------------------------
# stage 4: learned MLP-ensemble dynamics forward
# ---------------------------------------------------------------------------------------------
def test_mlp_dynamics_forward(mb, cuda_device):
    L = mb._lib
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    R = 1000
    rng = np.random.default_rng(50)
    inp = rng.uniform(-1, 1, (R, 4)).astype(np.float32)
    member = rng.integers(0, 5, R).astype(np.int32)
    d = lambda a: _dev(a, cuda_device)
    w_in, b_in = d(ens.weights[0]), d(ens.biases[0])
    w_h = torch.stack([d(ens.weights[1]), d(ens.weights[2])], dim=1)              # [E, 2, in, out]
    w_h = w_h.transpose(-1, -2).contiguous().to(torch.bfloat16)                   # K-major [E, 2, out, in]
    b_h = torch.stack([d(ens.biases[1]), d(ens.biases[2])], dim=1).contiguous()
    w_out, b_out = d(ens.weights[3]), d(ens.biases[3])
    p = L.MlpEnsembleParamsC(5, 256, 3, 1, L.ptr(w_in), L.ptr(b_in), L.ptr(w_h), L.ptr(b_h), L.ptr(w_out),
                             L.ptr(b_out), L.PendulumParamsC(8, 2, .05, 9.81, 1, 1, .02, 1, 0))
    out = torch.empty((R, 3), dtype=torch.float32, device=cuda_device)
    ti, tm = d(inp), d(member)
    L.check(L.lib.mbpo_mlp_dynamics_forward(L.C.byref(p), L.ptr(ti), L.ptr(tm), R, L.ptr(out),
                                            L.stream_ptr(cuda_device)))
    want = orc.mlp_member_forward(ens, member, inp, bf16=True)
    # identical bf16 operand rounding, fp32 accumulate; swish via __expf: a flipped bf16 rounding of one
    # activation moves an output by ~1e-4 relative
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=2e-3, atol=2e-4)
    full = orc.mlp_member_forward(ens, member, inp, bf16=False)
    assert np.abs(out.cpu().numpy() - full).max() < 5e-2                            # bf16 vs fp32 network


def _ensemble_on_device(mb, cuda_device, ens):
    from mbpo_b200.systems import MLPEnsembleSystem, MlpEnsembleDynamicsParams, SystemParams, PendulumRewardParams
    d = lambda a: _dev(a, cuda_device)
    dyn = MlpEnsembleDynamicsParams(weights=[d(w) for w in ens.weights], biases=[d(b) for b in ens.biases])
    return MLPEnsembleSystem(), SystemParams(dynamics_params=dyn, reward_params=PendulumRewardParams())


# (1, 256, 5) .. (5, 300, 3): few rows -> the one-tile kernel; (20, 1039, 2) = 20,780 rows -> more than one round of CTA
# pairs -> the two-tile ping-pong kernel (ens::launch_ensemble_rollout_auto decides on the row count alone)
@pytest.mark.parametrize("B,M,H", [(1, 256, 5), (3, 139, 12), (2, 527, 8), (5, 300, 3), (20, 1039, 2), (37, 513, 3)])
def test_ensemble_rollout_fused_tcgen05(mb, cuda_device, B, M, H):
    """Fused cta_group::2 rollout kernels against the oracle (same bf16 operand rounding, fp32 accumulate)."""
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    sys_, sp = _ensemble_on_device(mb, cuda_device, ens)
    x0 = _random_states(B, 71)
    acts = np.clip(np.random.default_rng(72).normal(0, 0.5, (B, M, H, 1)), -1, 1).astype(np.float32)
    got = sys_.ensemble_returns(sp, _dev(x0, cuda_device), _dev(acts, cuda_device)).cpu().numpy()
    want = orc.ensemble_rollout_returns(x0, acts[..., 0], ens, bf16=True)
    # a flipped bf16 rounding of one activation moves a step's delta by ~1e-4 relative; errors accumulate over H
    np.testing.assert_allclose(got, want, rtol=5e-3, atol=5e-3)
    assert np.abs(got - want).mean() < 5e-4
    got_max = sys_.ensemble_returns(sp, _dev(x0, cuda_device), _dev(acts, cuda_device), use_optimism=True).cpu().numpy()
    want_max = orc.ensemble_rollout_returns(x0, acts[..., 0], ens, bf16=True, use_max=True)
    np.testing.assert_allclose(got_max, want_max, rtol=5e-3, atol=5e-3)
    assert np.all(got_max >= got - 1e-6)
    # the rollout_actions ABI routes the ensemble System to the same kernel
    from mbpo_b200.utils import rollout_returns
    again = rollout_returns(sys_, sp, _dev(x0, cuda_device), _dev(acts, cuda_device)).cpu().numpy()
    assert np.array_equal(again, got)


def test_ensemble_system_step_matches_forward_kernel(mb, cuda_device):
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    sys_, sp = _ensemble_on_device(mb, cuda_device, ens)
    R = 700
    x = _random_states(R, 73)
    u = np.random.default_rng(74).uniform(-1, 1, (R, 1)).astype(np.float32)
    member = (np.arange(R) // 128 % 5).astype(np.int32)                       # homogeneous tiles
    sp2 = sp.replace(dynamics_params=sp.dynamics_params.replace(member=_dev(member, cuda_device)))
    st = sys_.step(_dev(x, cuda_device), _dev(u, cuda_device), sp2)
    xn, r = orc.mlp_ensemble_step(x, u[:, 0], member, ens, bf16=True)
    np.testing.assert_allclose(st.x_next.cpu().numpy(), xn, rtol=2e-3, atol=2e-4)
    np.testing.assert_allclose(st.reward.cpu().numpy(), r, rtol=1e-5, atol=3e-6)


def test_icem_plan_with_ensemble_system(mb, cuda_device):
    """iCemTO over the learned-ensemble System through the unchanged API (staged plan)."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    sys_, sp = _ensemble_on_device(mb, cuda_device, ens)
    H, B = 20, 3
    params = dict(num_samples=200, num_elites=20, num_particles=5, num_steps=3)
    opt = iCemTO(horizon=H, action_dim=1, opt_params=iCemParams(**params))
    opt.set_system(sys_)
    keys = _keys(B, seed=81)
    st = opt.init(_dev(keys, cuda_device)).replace(system_params=sp)
    x0 = _random_states(B, 82)
    action, new = opt.act(_dev(x0, cuda_device), st)
    assert action.shape == (B, 1) and new.best_sequence.shape == (B, H, 1)
    for b in range(B):                                                            # integer path is exact
        assert np.array_equal(new.key[b].cpu().numpy(), ojr.split(ojr.split(keys[b], 3)[2], 2)[1])
    # best_reward is the ensemble objective of best_sequence (same kernel, same bits)
    again = sys_.ensemble_returns(sp, _dev(x0, cuda_device), new.best_sequence.reshape(B, 1, H, 1))[:, 0]
    assert torch.equal(again, new.best_reward)
    zero = sys_.ensemble_returns(sp, _dev(x0, cuda_device), torch.zeros((B, 1, H, 1), device=cuda_device))[:, 0]
    assert bool((new.best_reward >= zero).all())
    want = orc.ensemble_rollout_returns(x0, new.best_sequence.cpu().numpy().reshape(B, 1, H), ens)[:, 0]
    np.testing.assert_allclose(new.best_reward.cpu().numpy(), want, rtol=5e-3, atol=5e-3)
    with pytest.raises(mb.MbpoUnsupported):                                       # particles must be the members
        o2 = iCemTO(horizon=H, action_dim=1, opt_params=iCemParams(num_samples=64, num_particles=3))
        o2.set_system(sys_)
        o2.act(_dev(x0, cuda_device), st)


# ---------------------------------------------------------------------------------------------
# error behaviour: no fallback, loud failures
# ---------------------------------------------------------------------------------------------
def test_errors(mb, cuda_device):
    from mbpo_b200.optimizers import iCemTO, iCemParams, AbstractCost
    from mbpo_b200.systems import PendulumSystem, System
    oc = iCemTO(horizon=20, action_dim=1, opt_params=iCemParams(num_samples=64, num_particles=1),
                cost_fn=AbstractCost(20))                                             # the abstract cost has no body
    oc.set_system(PendulumSystem())
    with pytest.raises(NotImplementedError):
        oc.act(torch.tensor([-1.0, 0.0, 0.0], device=cuda_device), oc.init(mb.random.PRNGKey(0, cuda_device)))
    opt = iCemTO(horizon=200, action_dim=1, opt_params=iCemParams(num_particles=1))  # beyond MBPO_MAX_HORIZON = 128
    opt.set_system(PendulumSystem())
    st = opt.init(mb.random.PRNGKey(0, cuda_device))
    with pytest.raises(mb.MbpoError):
        opt.act(torch.tensor([-1.0, 0.0, 0.0], device=cuda_device), st)
    with pytest.raises(mb.MbpoError):                                                # CPU tensors are refused
        PendulumSystem().step(torch.zeros(3), torch.zeros(1), st.system_params)

    class Other(System):
        system_kind = 7
    o = iCemTO(horizon=20, action_dim=1)
    o.set_system(PendulumSystem())
    st20 = o.init(mb.random.PRNGKey(0, cuda_device))
    o.set_system(Other(x_dim=3, u_dim=1))
    with pytest.raises(mb.MbpoUnsupported):                                         # a System without a CUDA step
        o.optimize(torch.zeros(3, device=cuda_device), st20)


# ---------------------------------------------------------------------------------------------
# full-size properties (BASELINE config 2 / 3 sizes): size-independent invariants
# ---------------------------------------------------------------------------------------------
def test_full_size_config2_properties(mb, cuda_device, budget_report):
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    B, H = 4096, 30
    opt = iCemTO(horizon=H, action_dim=1, opt_params=iCemParams(num_samples=512, num_particles=1))
    sys_ = PendulumSystem()
    opt.set_system(sys_)
    keys = mb.random.split(mb.random.PRNGKey(0, cuda_device), B)
    st = opt.init(keys)
    x0 = _dev(_random_states(B, 0), cuda_device)
    a1, n1 = opt.act(x0, st)
    a2, n2 = opt.act(x0, st)
    assert torch.equal(a1, a2) and torch.equal(n1.best_sequence, n2.best_sequence)       # deterministic
    assert bool(((n1.best_sequence >= -1) & (n1.best_sequence <= 1)).all())               # clipped actions
    # best_reward is the return of best_sequence: re-roll it out through the staged kernel
    from mbpo_b200.utils import rollout_returns
    ret = rollout_returns(sys_, st.system_params, x0, n1.best_sequence.reshape(B, 1, H, 1))[:, 0]
    assert torch.equal(ret, n1.best_reward)
    # sharding invariance: planning a slice alone gives the same bits as inside the batch
    sl = slice(1000, 1100)
    st_sl = st.replace(key=st.key[sl].contiguous(), best_sequence=st.best_sequence[sl].contiguous(),
                       best_reward=st.best_reward[sl].contiguous())
    a3, n3 = opt.act(x0[sl].contiguous(), st_sl)
    assert torch.equal(a3, a1[sl]) and torch.equal(n3.key, n1.key[sl])
    # planning beats the zero sequence (which is always among the candidates)
    zero = rollout_returns(sys_, st.system_params, x0, torch.zeros((B, 1, H, 1), device=cuda_device))[:, 0]
    assert bool((n1.best_reward >= zero).all())
    # 32 problems of the full-size launch against the oracle: the traced plan of those problems alone reproduces
    # their slice of the 4,096-problem launch bit for bit (traces are [S, B, 527, 30]: too large to dump for all),
    # and its every iteration is checked -- PRNG keys and elite indices exact, sampled actions to tolerance, every
    # return inside its float64 amplification bound, refit bit-exact given the kernel's own actions and values.
    pick = np.sort(np.random.default_rng(5).choice(B, 32, replace=False))
    pk = torch.from_numpy(pick).to(cuda_device)
    # (torch has no CUDA index kernel for uint32: index the int32 view of the keys)
    xs, bs = x0[pk].contiguous(), st.best_sequence[pk].contiguous()
    ks = st.key.view(torch.int32)[pk].contiguous().view(torch.uint32)
    seq_s, val_s, key_s, tr = opt._plan_raw(xs, ks, bs, st.system_params, trace=True)
    assert torch.equal(seq_s, n1.best_sequence[pk]) and torch.equal(val_s, n1.best_reward[pk])
    assert torch.equal(key_s.view(torch.int32), n1.key.view(torch.int32)[pk])
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    p = orc.ICemParams(num_samples=512, num_particles=1)
    x0n, kn = xs.cpu().numpy(), ks.cpu().numpy()
    worst, misses = 0.0, 0
    for j in range(32):
        ksp = ojr.split(kn[j], 2)
        assert np.array_equal(key_s[j].cpu().numpy(), ksp[1])
        carry = ksp[0]
        mean, std = np.zeros((H, 1), np.float32), np.full((H, 1), p.init_std, np.float32)
        bval, bseq = np.float32(-np.inf), mean.copy()
        for it in range(p.num_steps):
            carry, acts, _ = orc.icem_sample_actions(carry, mean, std, p, H)
            g_acts = tr["actions"][it, j].reshape(-1, H, 1)
            np.testing.assert_allclose(g_acts, acts, rtol=RTOL, atol=5e-6)
            g_vals = tr["values"][it, j]
            vals = orc.icem_objective(x0n[j], g_acts, p, orc.PendulumParams())
            r64, bound = ft.rollout_return_budget(np.broadcast_to(x0n[j], (g_acts.shape[0], 3)), g_acts[:, :, 0])
            frac = np.abs(g_vals - r64) / bound
            assert frac.max() <= 1.0 and (np.abs(vals - r64) / bound).max() <= 1.0
            miss = _beyond(g_vals, vals.astype(np.float64))
            assert np.all(2 * bound[miss] > RTOL * np.abs(r64[miss]))
            worst, misses = max(worst, float(frac.max())), misses + int(miss.sum())
            mean, std, bval, bseq, idx = orc.icem_refit(g_acts, g_vals, mean, std, bval, bseq, p)
            assert np.array_equal(tr["elite_idx"][it, j], idx)
            assert np.array_equal(tr["mean"][it, j], mean[:, 0]) and np.array_equal(tr["std"][it, j], std[:, 0])
            assert tr["best_value"][it, j] == bval
        assert np.array_equal(seq_s[j].cpu().numpy(), np.asarray(bseq)) and float(val_s[j]) == float(bval)
    budget_report("gpu/full_size_config2_sample32", problems=32, rows=32 * 5 * 527, max_frac=worst,
                  rows_beyond_rel_1e5_of_oracle=misses)


def test_full_size_config3_properties(mb, cuda_device):
    """BASELINE config 3 at full size (65,536 envs x 1,000 steps, episode_length 200): the episode-piece kernel
    against the one-scan-per-env kernel bit for bit, the AutoReset bookkeeping in closed form, a random sample of
    transitions against the oracle, and shard invariance (an env range alone = its slice of the full launch)."""
    L = mb._lib
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    E, T, EP = 65536, 1000, 200
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    env = wrap(sys_, sp, episode_length=EP)
    x0 = _dev(_random_states(E, 1), cuda_device)
    acts = torch.rand((T, E, 1), device=cuda_device, generator=torch.Generator(cuda_device).manual_seed(2)) * 2 - 1
    st = env.reset(x0)
    new, tr = env.unroll(st, acts)
    # sequential kernel, in place
    pp = sys_.pack_params(sp)
    obs, steps, done = st.obs.clone(), st.info["steps"].clone(), st.done.clone()
    n = torch.empty((T, E, 3), device=cuda_device)
    r, d, t_ = (torch.empty((T, E), device=cuda_device) for _ in range(3))
    L.check(L.lib.mbpo_env_rollout(0, L.C.addressof(pp), 0, 3, 1, EP, 1, L.ptr(obs), L.ptr(steps), L.ptr(done),
                                   L.ptr(st.info["first_obs"]), L.ptr(acts), E, T, None, L.ptr(r), L.ptr(d), L.ptr(n),
                                   L.ptr(t_), L.stream_ptr(cuda_device)))
    assert torch.equal(n, tr.next_observation) and torch.equal(r, tr.reward)
    assert torch.equal(d, tr.discount) and torch.equal(t_, tr.extras["state_extras"]["truncation"])
    assert torch.equal(obs, new.obs) and torch.equal(steps, new.info["steps"]) and torch.equal(done, new.done)
    del n, r, d, t_
    # bookkeeping in closed form: an episode ends (discount 0, truncation 1, obs reset) exactly at t % 200 == 199
    ends = (torch.arange(T, device=cuda_device) % EP == EP - 1).float()[:, None].expand(T, E)
    assert torch.equal(tr.discount, 1 - ends) and torch.equal(tr.extras["state_extras"]["truncation"], ends)
    assert torch.equal(tr.next_observation[EP - 1::EP], x0[None].expand(T // EP, E, 3))
    assert bool((new.info["steps"] == EP).all()) and bool((new.done == 1).all())
    assert bool(torch.isfinite(tr.reward).all()) and float(tr.reward.max()) <= 0.0
    assert float((tr.next_observation[..., 0] ** 2 + tr.next_observation[..., 1] ** 2 - 1).abs().max()) < 1e-5
    # a random sample of transitions against the oracle (teacher-forced on the GPU's observations)
    g = torch.Generator().manual_seed(5)
    ti, ei = torch.randint(0, T, (20000,), generator=g), torch.randint(0, E, (20000,), generator=g)
    keep = (ti % EP) != EP - 1                                         # the step that resets returns first_obs instead
    ti, ei = ti[keep].to(cuda_device), ei[keep].to(cuda_device)
    xs, us = tr.observation[ti, ei].cpu().numpy(), acts[ti, ei, 0].cpu().numpy()
    nxt, rew = orc.pendulum_step(xs, us)
    np.testing.assert_allclose(tr.next_observation[ti, ei].cpu().numpy(), nxt, rtol=RTOL, atol=2e-6)
    np.testing.assert_allclose(tr.reward[ti, ei].cpu().numpy(), rew, rtol=RTOL, atol=3e-6)
    # shard invariance: envs [8192, 16384) alone (rank 1 of 8) = that slice of the full launch
    lo, hi = 8192, 16384
    st_sl = env.reset(x0[lo:hi].contiguous())
    new_sl, tr_sl = env.unroll(st_sl, acts[:, lo:hi].contiguous())
    assert torch.equal(tr_sl.next_observation, tr.next_observation[:, lo:hi]) and torch.equal(tr_sl.reward, tr.reward[:, lo:hi])
    assert torch.equal(new_sl.obs, new.obs[lo:hi])


@pytest.mark.parametrize("E,T", [(1, 1), (31, 3), (129, 5), (257, 2), (500, 4)])
def test_no_out_of_bounds_writes_for_ragged_sizes(mb, cuda_device, E, T):
    """Every output of the env and policy-rollout kernels is placed inside a larger NaN-filled buffer: partial
    warps, partial tiles and the row-transposing stores must leave the guard zones on both sides untouched, and
    the guarded call must equal the plain call bit for bit."""
    L = mb._lib
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.systems import PendulumSystem
    G = 256                                                    # guard floats before and after every array
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    env = wrap(sys_, sp, episode_length=2)
    pp = sys_.pack_params(sp)
    x0 = _dev(_random_states(E, 151), cuda_device)
    acts = _dev(np.random.default_rng(152).uniform(-1, 1, (T, E, 1)).astype(np.float32), cuda_device)
    st = env.reset(x0)

    def guarded(n, dtype=torch.float32):
        buf = torch.full((n + 2 * G,), float("nan"), device=cuda_device, dtype=torch.float32)
        if dtype != torch.float32:
            buf = torch.full((n + 2 * G,), 0x7FC00000, device=cuda_device, dtype=torch.int64).to(dtype)
        return buf, buf[G:G + n]

    def intact(buf, n):
        head, tail = buf[:G], buf[G + n:]
        if buf.dtype == torch.float32:
            return bool(torch.isnan(head).all()) and bool(torch.isnan(tail).all())
        return bool((head == 0x7FC00000).all()) and bool((tail == 0x7FC00000).all())
    # ---- env unroll -------------------------------------------------------------------------------------------
    _, tr = env.unroll(st, acts)
    bufs = {k: guarded(n) for k, n in dict(obs=3 * E, steps=E, done=E, nxt=3 * T * E, r=T * E, d=T * E, t=T * E).items()}
    L.check(L.lib.mbpo_env_unroll(0, L.C.addressof(pp), 0, 3, 1, 2, 1, L.ptr(st.obs), L.ptr(st.info["steps"]),
                                  L.ptr(st.done), bufs["obs"][1].data_ptr(), bufs["steps"][1].data_ptr(),
                                  bufs["done"][1].data_ptr(), L.ptr(st.info["first_obs"]), L.ptr(acts), E, T, None,
                                  bufs["r"][1].data_ptr(), bufs["d"][1].data_ptr(), bufs["nxt"][1].data_ptr(),
                                  bufs["t"][1].data_ptr(), L.stream_ptr(cuda_device)))
    for k, n in dict(obs=3 * E, steps=E, done=E, nxt=3 * T * E, r=T * E, d=T * E, t=T * E).items():
        assert intact(bufs[k][0], n), k
    assert torch.equal(bufs["nxt"][1].reshape(T, E, 3), tr.next_observation) and torch.equal(bufs["r"][1].reshape(T, E), tr.reward)
    # ---- policy in the loop, both kernels ---------------------------------------------------------------------------
    pol = orc.make_policy_params(seed=9, hidden=(64, 64))
    key = _dev(ojr.PRNGKey(2), cuda_device)
    for kernel in ("tcgen05", "cuda_cores"):
        policy = _policy_on_device(mb, cuda_device, pol, kernel=kernel)
        policy.emit_extras = True
        _, _, tra = acting.get_experience(env, st, policy, key, T)
        sizes = dict(obs=3 * E, steps=E, done=E, act=T * E, r=T * E, d=T * E, nxt=3 * T * E, t=T * E, raw=T * E, lp=T * E)
        b = {k: guarded(n) for k, n in sizes.items()}
        kb, kv = guarded(2, torch.uint32)
        b["obs"][1].copy_(st.obs.reshape(-1)); b["steps"][1].copy_(st.info["steps"]); b["done"][1].copy_(st.done)
        policy.struct.draw_total = 0
        L.check(L.lib.mbpo_actor_rollout_extras(
            0, L.C.addressof(pp), 0, mb.config.prng_mode, L.C.byref(policy.struct), 0, L.KEYS_SAC, L.ptr(key), 2, 1,
            b["obs"][1].data_ptr(), b["steps"][1].data_ptr(), b["done"][1].data_ptr(), L.ptr(st.info["first_obs"]), E, T,
            b["act"][1].data_ptr(), b["r"][1].data_ptr(), b["d"][1].data_ptr(), b["nxt"][1].data_ptr(),
            b["t"][1].data_ptr(), kv.data_ptr(), b["raw"][1].data_ptr(), b["lp"][1].data_ptr(), L.stream_ptr(cuda_device)))
        for k, n in sizes.items():
            assert intact(b[k][0], n), (kernel, k)
        assert intact(kb, 2), kernel
        assert torch.equal(b["act"][1].reshape(T, E, 1), tra.action) and torch.equal(b["nxt"][1].reshape(T, E, 3), tra.next_observation)
        assert torch.equal(b["lp"][1].reshape(T, E), tra.extras["policy_extras"]["log_prob"])
        assert not bool(torch.isnan(b["act"][1]).any()) and not bool(torch.isnan(b["nxt"][1]).any())


def test_empty_and_degenerate_inputs(mb, cuda_device):
    """Zero problems / envs / steps are valid calls that launch nothing; one env, one step and a one-step episode
    exercise the piece arithmetic at its corners."""
    from mbpo_b200.envs import wrap
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils import lambda_return, rollout_actions
    sys_ = PendulumSystem()
    sp = sys_.reset(device=cuda_device).system_params
    env = wrap(sys_, sp, episode_length=5)
    st0 = env.reset(torch.zeros((0, 3), device=cuda_device))
    new, tr = env.unroll(st0, torch.zeros((7, 0, 1), device=cuda_device))                 # no envs
    assert tr.reward.shape == (7, 0) and new.obs.shape == (0, 3)
    x0 = _dev(_random_states(3, 9), cuda_device)
    st = env.reset(x0)
    new, tr = env.unroll(st, torch.zeros((0, 3, 1), device=cuda_device))                  # no steps: state unchanged
    assert tr.reward.shape == (0, 3) and torch.equal(new.obs, x0) and torch.equal(new.info["steps"], st.info["steps"])
    env1 = wrap(sys_, sp, episode_length=1)                                               # every step ends an episode
    acts = torch.full((6, 3, 1), 0.3, device=cuda_device)
    new, tr = env1.unroll(env1.reset(x0), acts)
    want = orc.env_rollout(x0.cpu().numpy(), acts[..., 0].cpu().numpy(), 1)
    assert np.array_equal(tr.discount.cpu().numpy(), want["discount"]) and bool((tr.discount == 0).all())
    assert torch.equal(tr.next_observation, x0[None].expand(6, 3, 3))
    np.testing.assert_allclose(tr.reward.cpu().numpy(), want["reward"], rtol=RTOL, atol=3e-6)
    opt = iCemTO(horizon=20, action_dim=1, opt_params=iCemParams(num_samples=64, num_particles=1))
    opt.set_system(sys_)
    st_b0 = opt.init(torch.zeros((0, 2), dtype=torch.uint32, device=cuda_device))
    a, nst = opt.act(torch.zeros((0, 3), device=cuda_device), st_b0)                      # no problems
    assert a.shape == (0, 1) and nst.best_sequence.shape == (0, 20, 1)
    tr0 = rollout_actions(sys_, sp, torch.zeros((0, 3), device=cuda_device), torch.zeros((0, 4, 20, 1), device=cuda_device), 20)
    assert tr0.reward.shape == (0, 4, 20)
    assert lambda_return(torch.zeros((0, 9), device=cuda_device), torch.zeros((0, 9), device=cuda_device), 0.99, 0.9).shape == (0, 9)


# ---------------------------------------------------------------------------------------------
# rollout_policy, its cotangent pass and lambda_return (BPTT; SURVEY 8f-4)
# ---------------------------------------------------------------------------------------------
def _bptt_policy(mb, cuda_device, hidden=(64, 64), evaluate=False, normalize=True, seed=17):
    from mbpo_b200.acting import BpttActorPolicy, PolicyParams
    pol = orc.make_policy_params(seed=seed, hidden=hidden)
    mean = np.array([0.1, -0.2, 0.5], np.float32) if normalize else None
    std = np.array([0.7, 0.8, 3.0], np.float32) if normalize else None
    oparams = orc.BpttActorParams(mlp=pol, init_stddev=0.5, sig_min=1e-6, sig_max=1e2, obs_mean=mean, obs_std=std)
    policy = BpttActorPolicy(PolicyParams(weights=[_dev(w, cuda_device) for w in pol.weights],
                                          biases=[_dev(b, cuda_device) for b in pol.biases]),
                             init_stddev=0.5, sig_min=1e-6, sig_max=1e2, obs_mean=mean, obs_std=std, evaluate=evaluate)
    return policy, oparams


@pytest.mark.parametrize("evaluate", [False, True])
@pytest.mark.parametrize("hidden,normalize", [((64, 64), True), ((64, 64, 64), False)])
def test_rollout_policy_vs_oracle(mb, cuda_device, prng_mode, evaluate, hidden, normalize):
    """rollout_policy with BPTT's train_policy in one launch, per step against the oracle teacher-forced on the
    GPU's observations; the carried key is bit exact and every trajectory of the batch shares the draw."""
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils.optimizer_utils import rollout_policy
    B, H = 203, 15
    policy, oparams = _bptt_policy(mb, cuda_device, hidden, evaluate, normalize)
    system = PendulumSystem()
    sp = system.reset(device=cuda_device).system_params
    x0 = _random_states(B, 101)
    key = ojr.PRNGKey(9)
    tr = rollout_policy(system, sp, _dev(x0, cuda_device), policy, _dev(key, cuda_device), H)
    assert tr.observation.shape == (B, H, 3) and tr.action.shape == (B, H, 1) and tr.reward.shape == (B, H)
    g_obs = tr.observation.cpu().numpy()
    want, okey = orc.rollout_policy(oparams, x0, key, H, evaluate=evaluate, partitionable=prng_mode, teacher_obs=g_obs)
    key_out = tr.extras["policy_state_key"].cpu().numpy()
    if evaluate:
        assert np.array_equal(key_out, key)
    else:
        assert np.array_equal(key_out, okey)
    np.testing.assert_allclose(tr.action.cpu().numpy(), want["action"], rtol=3e-5, atol=3e-6)
    assert float(tr.action.abs().max()) <= 0.999 + 1e-7
    # the System step on the GPU's own actions
    nxt, rew = orc.pendulum_step(g_obs.reshape(-1, 3), tr.action.cpu().numpy().reshape(-1))
    np.testing.assert_allclose(tr.next_observation.cpu().numpy().reshape(-1, 3), nxt, rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(tr.reward.cpu().numpy().reshape(-1), rew, rtol=1e-5, atol=3e-6)
    assert np.array_equal(g_obs[:, 0], x0) and np.array_equal(g_obs[:, 1:], tr.next_observation.cpu().numpy()[:, :-1])
    assert bool((tr.discount == 1).all())
    # single init_state form: fields [H, ...], same bits as row 0 of the batch
    one = rollout_policy(system, sp, _dev(x0[0], cuda_device), policy, _dev(key, cuda_device), H)
    assert one.observation.shape == (H, 3) and torch.equal(one.action, tr.action[0]) and torch.equal(one.reward, tr.reward[0])
    with pytest.raises(mb.MbpoUnsupported):
        rollout_policy(system, sp, _dev(x0, cuda_device), policy, _dev(key, cuda_device), H, stop_grads=False)
    with pytest.raises(mb.MbpoUnsupported):
        rollout_policy(system, sp, _dev(x0, cuda_device), lambda o, s: (o, s), _dev(key, cuda_device), H)


def test_rollout_policy_vjp_vs_oracle(mb, cuda_device):
    """The reverse scan through System.step against the oracle's hand-derived cotangent pass evaluated in
    float64 on the same float32 trajectory, for both array layouts the kernel accepts."""
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils.optimizer_utils import Transition, rollout_policy, rollout_policy_vjp
    B, H = 300, 20
    policy, _ = _bptt_policy(mb, cuda_device)
    system = PendulumSystem()
    sp = system.reset(device=cuda_device).system_params
    x0 = _random_states(B, 111)
    tr = rollout_policy(system, sp, _dev(x0, cuda_device), policy, _dev(ojr.PRNGKey(3), cuda_device), H)
    rng = np.random.default_rng(112)
    g_r, g_n = rng.standard_normal((B, H)).astype(np.float32), rng.standard_normal((B, H, 3)).astype(np.float32)
    g_o, g_a = rng.standard_normal((B, H, 3)).astype(np.float32), rng.standard_normal((B, H, 1)).astype(np.float32)
    obs, act = tr.observation.cpu().numpy(), tr.action.cpu().numpy()
    for use in [(True, True, True, True), (True, False, False, False), (False, True, False, True)]:
        args = [a if u else None for a, u in zip((g_r, g_n, g_o, g_a), use)]
        want_a, want_x0 = orc.rollout_policy_vjp(obs, act, *args, dtype=np.float64)
        dargs = [None if a is None else _dev(a, cuda_device) for a in args]
        got_a, got_x0 = rollout_policy_vjp(system, sp, tr, *dargs)                       # time-major strided views
        dense = Transition(*(f.contiguous() for f in tr[:5]))
        got_a2, got_x02 = rollout_policy_vjp(system, sp, dense, *dargs)                  # the reference's [B, H, ...]
        assert torch.equal(got_a, got_a2) and torch.equal(got_x0, got_x02)
        scale = np.abs(want_a).max(axis=(1, 2), keepdims=True) + 1e-3                    # adjoints grow along the horizon
        assert float(np.abs((got_a.cpu().numpy() - want_a) / scale).max()) < 2e-4
        scale0 = np.abs(want_x0).max(axis=1, keepdims=True) + 1e-3
        assert float(np.abs((got_x0.cpu().numpy() - want_x0) / scale0).max()) < 2e-4


def test_bptt_actor_gradient_matches_autograd(mb, cuda_device):
    """End to end: forward kernel -> cotangents of a loss -> adjoint kernel -> one batched backward of the policy
    network equals torch autograd through the whole differentiable rollout (policy on detached observations,
    pendulum dynamics and reward written in torch, float64) -- the gradient jax.value_and_grad returns in
    BPTT._train_step (bptt_optimizer.py:361-376)."""
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils.optimizer_utils import lambda_return, lambda_return_vjp, rollout_policy, rollout_policy_vjp
    B, H, disc, lam = 64, 12, 0.99, 0.95
    policy, oparams = _bptt_policy(mb, cuda_device, hidden=(64, 64), seed=23)
    system = PendulumSystem()
    sp = system.reset(device=cuda_device).system_params
    x0 = _random_states(B, 121)
    key = ojr.PRNGKey(4)
    tr = rollout_policy(system, sp, _dev(x0, cuda_device), policy, _dev(key, cuda_device), H)
    rng = np.random.default_rng(122)
    wv = _dev(rng.standard_normal(3).astype(np.float32), cuda_device)                 # a linear "critic" v(x) = wv . x
    # loss = -mean(lambda_return(reward, v(next_obs)) * disc_t)
    pc = torch.cumprod(torch.tensor([1.0] + [disc] * (H - 1), device=cuda_device), 0)
    nv = tr.next_observation @ wv
    lv = lambda_return(tr.reward, nv, disc, lam)
    np.testing.assert_array_equal(lv.cpu().numpy(), orc.lambda_return(tr.reward.cpu().numpy(), nv.cpu().numpy(), disc, lam))
    g_lv = -(pc / (B * H)).expand(B, H).contiguous()
    g_rew, g_nv = lambda_return_vjp(g_lv, disc, lam)
    want_gr, want_gnv = orc.lambda_return_vjp(g_lv.cpu().numpy(), disc, lam)
    np.testing.assert_allclose(g_rew.cpu().numpy(), want_gr, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(g_nv.cpu().numpy(), want_gnv, rtol=1e-5, atol=1e-9)
    g_next = g_nv[..., None] * wv
    g_act, _ = rollout_policy_vjp(system, sp, tr, g_reward=g_rew, g_next_observation=g_next)

    # the policy network in torch (float64), used both for the batched backward and for the autograd reference
    ws = [_dev(w, cuda_device).double().requires_grad_(True) for w in oparams.mlp.weights]
    bs = [_dev(b, cuda_device).double().requires_grad_(True) for b in oparams.mlp.biases]
    mean, std = _dev(oparams.obs_mean, cuda_device).double(), _dev(oparams.obs_std, cuda_device).double()
    eps_t = []                                                                          # the draws the kernel used
    k = key
    for _ in range(H):
        ks = ojr.split(k, 2)
        eps_t.append(float(ojr.normal(ks[0], 1)[0]))
        k = ks[1]
    sig_bias = float(orc.inv_softplus(oparams.init_stddev))

    def actor(o, eps):
        h = (o - mean) / std
        for i in range(len(ws)):
            h = h @ ws[i] + bs[i]
            if i < len(ws) - 1:
                h = h * torch.sigmoid(h)
        mu, sg = h[..., :1], h[..., 1:]
        sg = torch.clamp(torch.nn.functional.softplus(sg + sig_bias), 1e-6, 1e2)
        return torch.clamp(torch.tanh(mu + eps * sg), -0.999, 0.999)
    # (1) our pipeline: one batched backward over all (obs_t, g_action_t) rows
    eps_all = torch.tensor(eps_t, device=cuda_device, dtype=torch.float64).reshape(1, H, 1)
    a_re = actor(tr.observation.double().detach(), eps_all)
    np.testing.assert_allclose(a_re.detach().cpu().numpy(), tr.action.cpu().numpy(), rtol=3e-5, atol=3e-6)
    grads_ours = torch.autograd.grad((a_re * g_act.double()).sum(), ws + bs)
    # (2) autograd through the whole rollout
    p = orc.PendulumParams()
    x = _dev(x0, cuda_device).double()
    rews, nvs = [], []
    for t in range(H):
        a = actor(x.detach(), eps_t[t])[:, 0]
        th = torch.atan2(x[:, 1], x[:, 0])
        d = torch.remainder(th - p.target_angle + np.pi, 2 * np.pi) - np.pi
        rews.append(-(p.angle_cost * d ** 2 + 0.1 * x[:, 2] ** 2) - p.control_cost * a ** 2)
        thdd = 3 * p.g / (2 * p.l) * torch.sin(th) + 3.0 / (p.m * p.l ** 2) * torch.clamp(a, -1, 1) * p.max_torque
        nw = torch.clamp(x[:, 2] + thdd * p.dt, -p.max_speed, p.max_speed)
        nth = th + nw * p.dt
        x = torch.stack([torch.cos(nth), torch.sin(nth), nw], -1)
        nvs.append(x @ wv.double())
    rews, nvs = torch.stack(rews, 1), torch.stack(nvs, 1)
    inputs = rews + disc * nvs * (1 - lam)
    agg, rets = nvs[:, -1], []
    for t in range(H - 1, -1, -1):
        agg = inputs[:, t] + disc * lam * agg
        rets.append(agg)
    rets = torch.stack(rets[::-1], 1)
    loss = -(rets * pc.double()).mean()
    grads_ref = torch.autograd.grad(loss, ws + bs)
    for go, gr in zip(grads_ours, grads_ref):
        denom = float(gr.abs().max()) + 1e-12
        assert float((go - gr).abs().max()) / denom < 2e-3, (float((go - gr).abs().max()), denom)


def test_bptt_golden_fixture(mb, cuda_device):
    """The committed vectors of tests/golden/bptt_golden.npz (frozen oracle outputs): rollout_policy teacher-free
    over 10 steps, the cotangent pass on the fixture's trajectory, lambda_return bit for bit."""
    import os
    from mbpo_b200.acting import BpttActorPolicy, PolicyParams
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils.optimizer_utils import Transition, lambda_return, lambda_return_vjp, rollout_policy, rollout_policy_vjp
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bptt_golden.npz"))
    pol = orc.make_policy_params(seed=33, hidden=(64, 64))
    policy = BpttActorPolicy(PolicyParams([_dev(w, cuda_device) for w in pol.weights], [_dev(b, cuda_device) for b in pol.biases]),
                             init_stddev=0.5, obs_mean=[0.1, -0.2, 0.5], obs_std=[0.7, 0.8, 3.0])
    system = PendulumSystem()
    sp = system.reset(device=cuda_device).system_params
    tr = rollout_policy(system, sp, _dev(G["x0"], cuda_device), policy, _dev(G["key"], cuda_device), 10)
    assert np.array_equal(tr.extras["policy_state_key"].cpu().numpy(), G["key_out"])
    # 10 closed-loop steps: 1-ulp differences grow a little along the horizon
    np.testing.assert_allclose(tr.action.cpu().numpy(), G["tr_action"], rtol=1e-3, atol=1e-4)
    np.testing.assert_allclose(tr.next_observation.cpu().numpy(), G["tr_next_observation"], rtol=1e-3, atol=1e-4)
    np.testing.assert_allclose(tr.reward.cpu().numpy(), G["tr_reward"], rtol=1e-3, atol=1e-4)
    fix = Transition(*(_dev(G["tr_" + k], cuda_device) for k in ("observation", "action", "reward", "discount", "next_observation")))
    ga, gx0 = rollout_policy_vjp(system, sp, fix, *(_dev(G[k], cuda_device) for k in ("g_reward", "g_next_obs", "g_obs", "g_action")))
    scale = np.abs(G["vjp_g_action"]).max(axis=(1, 2), keepdims=True) + 1e-3
    assert float(np.abs((ga.cpu().numpy() - G["vjp_g_action"]) / scale).max()) < 2e-4
    scale0 = np.abs(G["vjp_g_x0"]).max(axis=1, keepdims=True) + 1e-3
    assert float(np.abs((gx0.cpu().numpy() - G["vjp_g_x0"]) / scale0).max()) < 2e-4
    lv = lambda_return(_dev(G["tr_reward"], cuda_device), _dev(G["next_values"], cuda_device), 0.99, 0.95)
    assert np.array_equal(lv.cpu().numpy(), G["lambda_returns"])
    gr, gnv = lambda_return_vjp(_dev(G["g_reward"], cuda_device), 0.99, 0.95)
    np.testing.assert_allclose(gr.cpu().numpy(), G["lambda_g_reward"], rtol=1e-5, atol=1e-6)     # fused vs unfused mul-add
    np.testing.assert_allclose(gnv.cpu().numpy(), G["lambda_g_next_values"], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------
# iCEMOptimizer wrapper (icem_optimizer.py:260-319) and the dummy true buffer (base_optimizer.py:44-57)
# ---------------------------------------------------------------------------------------------
def test_icem_optimizer_wrapper_on_gpu(mb, cuda_device):
    """iCEMOptimizer.init with and without true_buffer_state, act reshaping obs (-1,) in and action (1, -1) out
    (icem_optimizer.py:287-312); its plan is iCemTO's plan bit for bit and matches the oracle's keys."""
    from mbpo_b200.optimizers import iCEMOptimizer, iCemTO, iCemParams
    from mbpo_b200.replay_buffers import ReplayBufferState
    from mbpo_b200.systems import PendulumSystem
    jr = mb.random
    params = iCemParams(num_samples=128, num_elites=16, num_particles=1, num_steps=3)
    system = PendulumSystem()
    key = jr.PRNGKey(0, cuda_device)
    opt = iCEMOptimizer(horizon=20, opt_params=params, system=system, key=key)
    assert opt.can_act_in_batches is False
    # without a true buffer: dummy_buffer_key, key = split(key, 2); agent.init(key) splits that again in 3
    st = opt.init(key)
    k_np = np.zeros(2, np.uint32)
    dummy_key, agent_key = ojr.split(k_np, 2)
    assert isinstance(st.true_buffer_state, ReplayBufferState)
    assert np.array_equal(st.true_buffer_state.key.cpu().numpy(), dummy_key)
    assert tuple(st.true_buffer_state.ring.shape) == (10, 3 + 1 + 1 + 1 + 3)           # base_optimizer.py:47-56
    assert st.true_buffer_state.insert_position == 0 and st.true_buffer_state.sample_position == 0
    assert np.array_equal(st.key.cpu().numpy(), ojr.split(agent_key, 3)[2])               # iCemTO.init (:123)
    assert st.best_sequence.shape == (20, 1) and float(st.best_reward) == 0.0
    # with a true buffer: the key is not split by the wrapper, the buffer is carried as given
    mine = object()
    st2 = opt.init(key, true_buffer_state=mine)
    assert st2.true_buffer_state is mine
    assert np.array_equal(st2.key.cpu().numpy(), ojr.split(k_np, 3)[2])
    # act: obs of any shape is flattened, the action comes back as (1, A)
    obs = torch.tensor([[-1.0, 0.0, 0.0]], device=cuda_device)
    action, new = opt.act(obs, st)
    assert action.shape == (1, 1) and new.best_sequence.shape == (20, 1)
    plain = iCemTO(horizon=20, action_dim=1, opt_params=params)
    plain.set_system(system)
    a2, n2 = plain.act(obs.reshape(-1), st)
    assert torch.equal(action.reshape(-1), a2) and torch.equal(new.best_sequence, n2.best_sequence)
    assert torch.equal(new.key, n2.key) and torch.equal(new.best_reward, n2.best_reward)
    onew = orc.icem_optimize(np.array([-1, 0, 0], np.float32),
                             orc.ICemState(key=st.key.cpu().numpy(), best_sequence=np.zeros((20, 1), np.float32),
                                           best_reward=np.float32(0)),
                             orc.ICemParams(num_samples=128, num_elites=16, num_particles=1, num_steps=3), 20)
    assert np.array_equal(new.key.cpu().numpy(), onew.key)
    out = opt.train(new)
    assert out.summary == [] and out.optimizer_state is new                               # :314-319
    # a second act warm-starts from the first plan
    action3, new3 = opt.act(obs, new)
    assert action3.shape == (1, 1) and not torch.equal(new3.key, new.key)


def test_dummy_true_buffer_state_feeds_brax_wrapper(mb, cuda_device, prng_mode):
    """The reference pattern BraxWrapper(system, params, sample_buffer_state=opt_state.true_buffer_state, ...)
    (brax_optimizers.py:86-91) works on the dummy buffer iCemTO.init builds: reset draws row 0 of the empty queue
    (randint over an empty range returns minval)."""
    from oracle import brax_replay as obr
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.replay_buffers import UniformSamplingQueue
    from mbpo_b200.systems import BraxWrapper, PendulumSystem
    from mbpo_b200.utils.optimizer_utils import Transition
    dev = cuda_device
    system = PendulumSystem()
    opt = iCemTO(horizon=20, action_dim=1, opt_params=iCemParams(num_particles=1))
    opt.set_system(system)
    st = opt.init(_dev(ojr.PRNGKey(3), dev))
    z = lambda n: torch.zeros((n,), device=dev)
    queue = UniformSamplingQueue(10, Transition(z(3), z(1), z(1), z(1), z(3)), 1)
    env = BraxWrapper(system, st.system_params, st.true_buffer_state, queue)
    rngs = ojr.split(ojr.PRNGKey(4), 50, prng_mode)
    state = env.reset(_dev(rngs, dev))
    oq = obr.UniformSamplingQueue(10, 9, 1, prng_mode)
    obs, reward, sys_keys, _ = obr.brax_wrapper_reset(rngs, oq, oq.init(st.true_buffer_state.key.cpu().numpy()), 3, 1)
    assert np.array_equal(state.obs.cpu().numpy(), obs) and np.all(obs == 0)
    assert np.array_equal(state.reward.cpu().numpy(), reward)
    assert np.array_equal(state.system_params.key.cpu().numpy(), sys_keys)
    # batched init (additive vmap): the vmapped pytree
    stb = opt.init(mb.random.split(_dev(ojr.PRNGKey(5), dev), 4))
    assert tuple(stb.true_buffer_state.ring.shape) == (4, 10, 9) and tuple(stb.true_buffer_state.key.shape) == (4, 2)


# ---------------------------------------------------------------------------------------------
# iCEM generality (SURVEY 8f-3): a System that consumes the per-particle key, and action_dim > 1
# ---------------------------------------------------------------------------------------------
def _general_systems(mb):
    from mbpo_b200.systems import NoisyPendulumSystem, PointMassSystem
    return {"noisy_pendulum": (NoisyPendulumSystem(0.05), orc.NoisyPendulumOracle(0.05)),
            "point_mass": (PointMassSystem(), orc.PointMassOracle())}


def _general_states(kind, n, seed):
    if kind == "noisy_pendulum":
        return _random_states(n, seed)
    return np.random.default_rng(seed).uniform(-1.5, 1.5, (n, 4)).astype(np.float32)


@pytest.mark.parametrize("kind", ["noisy_pendulum", "point_mass"])
def test_general_system_step(mb, cuda_device, prng_mode, kind):
    """System.step of the key-consuming pendulum (key, sub = split(key); x' = mean + std * normal(sub, (3,)); the key
    is carried on) and of the two-action point mass, against the oracle: keys bit-exact, the point mass bit-exact
    (single-rounded arithmetic in the oracle's order), the pendulum's floats to the north star's tolerance."""
    system, osys = _general_systems(mb)[kind]
    R = 1000
    x = _general_states(kind, R, 401)
    u = np.random.default_rng(402).uniform(-1.3, 1.3, (R, system.u_dim)).astype(np.float32)
    keys = _keys(R, seed=403)
    sp = system.init_params(mb.random.PRNGKey(0, cuda_device)).replace(key=_dev(keys, cuda_device))
    out = system.step(_dev(x, cuda_device), _dev(u, cuda_device), sp)
    xn, r, kn = osys.step(x, u, keys, prng_mode)
    if kind == "point_mass":
        assert np.array_equal(out.x_next.cpu().numpy(), xn) and np.array_equal(out.reward.cpu().numpy(), r)
        assert out.system_params.key is None
    else:
        assert np.array_equal(out.system_params.key.cpu().numpy(), kn)           # the key is carried on
        np.testing.assert_allclose(out.x_next.cpu().numpy(), xn, rtol=RTOL, atol=2e-6)
        np.testing.assert_allclose(out.reward.cpu().numpy(), r, rtol=RTOL, atol=2e-6)
        det = orc.pendulum_step(x, u[:, 0])[0]
        assert np.abs(out.x_next.cpu().numpy() - det).std() > 0.03                 # the draw is really there
        # a second step continues the stream: different noise
        out2 = system.step(out.x_next, _dev(u, cuda_device), out.system_params)
        xn2, _, kn2 = osys.step(out.x_next.cpu().numpy(), u, kn, prng_mode)
        assert np.array_equal(out2.system_params.key.cpu().numpy(), kn2)
        np.testing.assert_allclose(out2.x_next.cpu().numpy(), xn2, rtol=RTOL, atol=2e-6)


@pytest.mark.parametrize("kind", ["noisy_pendulum", "point_mass"])
def test_general_objective_vs_oracle(mb, cuda_device, prng_mode, kind):
    """vmap(vmap(objective)) (icem_optimizer.py:144-160): split(key, P), one rollout per particle key, horizon mean,
    mean / max over particles; and vmap(rollout_actions) with the key threaded through the scan, step by step."""
    system, osys = _general_systems(mb)[kind]
    B, M, H, P = 3, 37, 12, 4
    A = system.u_dim
    x0 = _general_states(kind, B, 411)
    acts = np.clip(np.random.default_rng(412).normal(0, 0.5, (B, M, H, A)), -1, 1).astype(np.float32)
    keys = _keys(B * M, seed=413).reshape(B, M, 2)
    sp = system.init_params(mb.random.PRNGKey(0, cuda_device))
    d = lambda a: _dev(a, cuda_device)
    p = orc.ICemParams(num_particles=P)
    for use_max in (False, True):
        got = system.objective(sp, d(x0), d(acts), d(keys), num_particles=P, use_optimism=use_max).cpu().numpy()
        for b in range(B):
            want = orc.system_objective(osys, x0[b], acts[b], keys[b], p, use_max, prng_mode)
            if kind == "point_mass":
                assert np.array_equal(got[b], want)
            else:
                np.testing.assert_allclose(got[b], want, rtol=2e-5, atol=2e-6)
    # single rollouts with the Transition buffers, teacher-forced: every step from the kernel's own observation and key
    vals, obs, rew, nxt = system.objective(sp, d(x0), d(acts), d(keys), num_particles=0, full=True)
    obs, rew, nxt = obs.cpu().numpy(), rew.cpu().numpy(), nxt.cpu().numpy()
    assert np.array_equal(obs[:, :, 1:], nxt[:, :, :-1])
    assert np.array_equal(obs[:, :, 0], np.broadcast_to(x0[:, None], (B, M, system.x_dim)))
    k = keys.reshape(-1, 2)
    for t in range(H):
        xn, r, k = osys.step(obs[:, :, t].reshape(B * M, -1), acts[:, :, t].reshape(B * M, A), k, prng_mode)
        np.testing.assert_allclose(nxt[:, :, t].reshape(B * M, -1), xn, rtol=RTOL, atol=2e-6)
        np.testing.assert_allclose(rew[:, :, t].reshape(-1), r, rtol=RTOL, atol=3e-6)
    np.testing.assert_allclose(vals.cpu().numpy(), rew.astype(np.float64).mean(-1), rtol=2e-6, atol=1e-6)


@pytest.mark.parametrize("horizon", [10, 20])        # 10: no unrolled instance -> the staged plan; 20: the fused kernel
@pytest.mark.parametrize("kind,use_optimism", [("noisy_pendulum", False), ("noisy_pendulum", True), ("point_mass", False)])
def test_icem_plan_over_general_systems(mb, cuda_device, prng_mode, kind, use_optimism, horizon):
    """iCemTO through its unchanged API over a key-consuming System (P distinct particles per candidate, mean and max
    summaries) and over a System with two action dimensions: teacher-forced against the oracle iteration by iteration
    (keys and elite indices exact, sampled actions and objectives to tolerance, the refit bit-exact given the
    kernel's own actions and values); act() -- the C staged plan -- gives the traced composition's bits."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    system, osys = _general_systems(mb)[kind]
    H, B, A = horizon, 4, system.u_dim
    params = dict(num_samples=96, num_elites=12, num_particles=3, num_steps=3, alpha=0.1, exponent=1.0)
    opt = iCemTO(horizon=H, action_dim=A, opt_params=iCemParams(**params), use_optimism=use_optimism)
    opt.set_system(system)
    keys = _keys(B, seed=421)
    st = opt.init(_dev(keys, cuda_device))
    assert st.best_sequence.shape == (B, H, A)
    x0 = _general_states(kind, B, 422)
    seq_t, val_t, key_t, tr = opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params, trace=True)
    action, new = opt.act(_dev(x0, cuda_device), st)
    assert action.shape == (B, A)
    assert torch.equal(new.best_sequence, seq_t) and torch.equal(new.best_reward, val_t)
    assert torch.equal(new.key.view(torch.int32), key_t.view(torch.int32))
    # act() ran the FUSED general kernel (one launch); the staged plan (one launch per stage) gives the same bits,
    # and so does its traced composition, dump by dump
    assert mb._lib.lib.mbpo_icem_plan_is_fused(mb._lib.C.byref(opt._cfg())) == (1 if horizon == 20 else 0)
    s_seq, s_val, s_key, _ = opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params, staged=True)
    assert torch.equal(s_seq, seq_t) and torch.equal(s_val, val_t)
    _, _, _, tr_s = opt._plan_raw(_dev(x0, cuda_device), st.key, st.best_sequence, st.system_params, trace=True,
                                  staged=True)
    for name in ("actions", "values", "elite_idx", "mean", "std", "best_value"):
        assert torch.equal(tr[name], tr_s[name]), name
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    p = orc.ICemParams(**params)
    M = p.num_samples + p.num_prev_elites
    k_np = st.key.cpu().numpy()
    for b in range(B):
        ks = ojr.split(k_np[b], 2, prng_mode)
        assert np.array_equal(new.key[b].cpu().numpy(), ks[1])
        carry = ks[0]
        mean, std = np.zeros((H, A), np.float32), np.full((H, A), p.init_std, np.float32)
        bval, bseq = np.float32(-np.inf), mean.copy()
        for it in range(p.num_steps):
            carry, acts, pkeys = orc.icem_sample_actions(carry, mean, std, p, H, A, prng_mode)
            g_acts = tr["actions"][it, b].reshape(M, H, A)
            np.testing.assert_allclose(g_acts, acts, rtol=RTOL, atol=5e-6)
            vals = orc.system_objective(osys, x0[b], g_acts, pkeys, p, use_optimism, prng_mode)
            g_vals = tr["values"][it, b]
            np.testing.assert_allclose(g_vals, vals, rtol=2e-5, atol=2e-6)
            if kind == "noisy_pendulum":                       # the kept-elite zero rows are distinct rollouts now
                assert len(np.unique(g_vals[p.num_samples:])) > 1
            mean, std, bval, bseq, idx = orc.icem_refit(g_acts, g_vals, mean, std, bval, bseq, p)
            assert np.array_equal(tr["elite_idx"][it, b], idx)
            assert np.array_equal(tr["mean"][it, b].reshape(H, A), mean)
            assert np.array_equal(tr["std"][it, b].reshape(H, A), std)
            assert tr["best_value"][it, b] == bval
        assert np.array_equal(seq_t[b].cpu().numpy(), np.asarray(bseq)) and float(val_t[b]) == float(bval)
    # closed loop through plan -> System.step launches (the key of the true System threads through as well)
    states, rewards, actions, _ = opt.closed_loop(_dev(x0, cuda_device), st, 3)
    assert states.shape == (3, B, system.x_dim) and actions.shape == (3, B, A)
    assert torch.equal(actions[0], action)
