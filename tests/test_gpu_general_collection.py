"""GPU parity of the SAC / PPO collection path for the general Systems (mbpo_env_unroll_general,
mbpo_actor_rollout_general) against system_env_rollout / system_actor_rollout (general_collection_oracle.py):
NoisyPendulumSystem (keyed, X = 3, A = 1) and PointMassSystem (X = 4, A = 2) in both PRNG layouts.  PRNG words are
bit-exact; floats are compared per step, teacher-forced on the GPU's observations, at rel 1e-5 (the bar of
test_gpu_parity.py)."""
import numpy as np
import pytest
import torch

from oracle import brax_replay as obr
from oracle import jax_prng as ojr
from oracle import mbpo_oracle as orc

import general_collection_oracle as gco

pytestmark = pytest.mark.gpu

RTOL = 1e-5


@pytest.fixture(scope="module")
def mb(cuda_device):
    import mbpo_b200
    return mbpo_b200


@pytest.fixture(params=[False, True], ids=["legacy", "partitionable"])
def prng_mode(request, mb):
    mb.config.threefry_partitionable = request.param
    yield request.param
    mb.config.threefry_partitionable = False


@pytest.fixture(params=["noisy_pendulum", "point_mass"])
def which(request):
    return request.param


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _keys(n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2 ** 32, size=(n, 2), dtype=np.uint64).astype(np.uint32)


def _pair(which, mb, dev, E, seed=0):
    """(GPU System, its SystemParams with one key per env, oracle System, first observations [E, X], keys [E, 2])."""
    from mbpo_b200.systems import NoisyPendulumSystem, PointMassSystem
    from mbpo_b200.systems.base_systems import SystemParams
    rng = np.random.default_rng(seed)
    if which == "noisy_pendulum":
        system, osys = NoisyPendulumSystem(noise_std=0.05), orc.NoisyPendulumOracle(noise_std=0.05)
        th, w = rng.uniform(-np.pi, np.pi, E), rng.uniform(-8, 8, E)
        x0 = np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)
        keys = _keys(E, seed + 1)
        params = system.init_params(_dev(ojr.PRNGKey(1), dev)).replace(key=_dev(keys, dev))
    else:
        system, osys = PointMassSystem(), orc.PointMassOracle()
        x0 = rng.uniform(-2, 2, (E, 4)).astype(np.float32)
        keys = None
        params = SystemParams(dynamics_params=None, reward_params=None, key=None)
    return system, params, osys, x0, keys


def _keys_of(state):
    k = state.system_params.key
    return None if k is None else k.cpu().numpy()


def _env_state(mb, env, x0, steps0, done0, dev, params):
    st = env.reset(_dev(x0, dev))
    st.info["steps"].copy_(_dev(steps0, dev))
    st.done.copy_(_dev(done0, dev))
    return st.replace(system_params=params)


def _check_teacher_forced_env(osys, tr, acts, x0, steps0, done0, keys, L, rep, partitionable):
    """Every step re-run by the oracle from the GPU's observation[t]; keys and bookkeeping carried by the oracle."""
    T = acts.shape[0]
    obs, steps, done, k = x0, steps0, done0, keys
    g_obs = tr.observation.cpu().numpy()
    assert np.array_equal(g_obs[0], x0)
    for t in range(T):
        one = gco.system_env_rollout(osys, g_obs[t], acts[t:t + 1], L, rep, steps0=steps, done0=done, first_obs=x0,
                                     keys=k, partitionable=partitionable)
        np.testing.assert_allclose(tr.reward[t].cpu().numpy(), one["reward"][0], rtol=RTOL, atol=3e-6)
        np.testing.assert_allclose(tr.next_observation[t].cpu().numpy(), one["next_observation"][0], rtol=RTOL,
                                   atol=2e-6)
        for f in ("discount", "truncation"):
            assert np.array_equal(getattr(tr, f)[t].cpu().numpy() if f == "discount"
                                  else tr.extras["state_extras"]["truncation"][t].cpu().numpy(), one[f][0]), (t, f)
        steps, done, k = one["final_steps"], one["final_done"], one["final_keys"]
    return steps, done, k


@pytest.mark.parametrize("rep", [1, 2])
def test_env_unroll_vs_oracle(mb, cuda_device, prng_mode, which, rep):
    """E not a multiple of the 64-thread block, episodes ending inside T (and carried-in done / step counters),
    action_repeat 1 and 2: keys bit-exact, floats per step."""
    from mbpo_b200 import envs
    dev = cuda_device
    E, T, L = 133, 41, 9
    system, params, osys, x0, keys = _pair(which, mb, dev, E)
    rng = np.random.default_rng(7)
    acts = rng.uniform(-1.5, 1.5, (T, E, system.u_dim)).astype(np.float32)
    steps0 = rng.integers(0, L, E).astype(np.float32)
    done0 = (rng.uniform(size=E) < 0.2).astype(np.float32)
    env = envs.wrap(system, params, episode_length=L, action_repeat=rep)
    st = _env_state(mb, env, x0, steps0, done0, dev, params)
    nst, tr = env.unroll(st, _dev(acts, dev))
    assert tr.observation.shape == (T, E, system.x_dim) and tr.action.shape == (T, E, system.u_dim)
    assert tr.extras["state_extras"]["truncation"].sum() > E          # episodes end inside T
    steps, done, k = _check_teacher_forced_env(osys, tr, acts, x0, steps0, done0, keys, L, rep, prng_mode)
    assert np.array_equal(nst.info["steps"].cpu().numpy(), steps)
    assert np.array_equal(nst.done.cpu().numpy(), done)
    assert np.array_equal(nst.obs.cpu().numpy(), tr.next_observation[-1].cpu().numpy())
    if keys is None:
        assert nst.system_params.key is None
    else:
        assert np.array_equal(_keys_of(nst), k)
        want = gco.system_env_rollout(osys, x0, acts, L, rep, steps0=steps0, done0=done0, keys=keys,
                                      partitionable=prng_mode)
        assert np.array_equal(_keys_of(nst), want["final_keys"])
        assert np.array_equal(_keys_of(st), keys)                     # the incoming state is left as it was


def test_env_step_and_streamed_equal_unroll(mb, cuda_device, which):
    from mbpo_b200 import envs
    dev = cuda_device
    E, T, L = 200, 70, 13
    system, params, _, x0, _ = _pair(which, mb, dev, E, seed=3)
    acts = np.random.default_rng(2).uniform(-1, 1, (T, E, system.u_dim)).astype(np.float32)
    env = envs.wrap(system, params, episode_length=L)
    st0 = env.reset(_dev(x0, dev)).replace(system_params=params)
    nst, tr = env.unroll(st0, _dev(acts, dev))
    s = st0
    for t in range(3):
        s = env.step(s, _dev(acts[t], dev))
    assert torch.equal(s.obs, tr.next_observation[2])
    host = torch.from_numpy(acts).pin_memory()
    rew = torch.empty((T, E), dtype=torch.float32).pin_memory()
    sst, str_ = env.unroll_streamed(st0, host, rew, chunk_steps=16)
    torch.cuda.synchronize(dev)
    assert torch.equal(str_.next_observation, tr.next_observation) and torch.equal(rew, tr.reward.cpu())
    assert torch.equal(sst.obs, nst.obs) and torch.equal(sst.info["steps"], nst.info["steps"])
    if system.keyed:
        assert torch.equal(sst.system_params.key, nst.system_params.key)


def test_env_unroll_equals_system_step_calls(mb, cuda_device, prng_mode, which):
    """Without an episode end the unroll is T calls of System.step (mbpo_system_step_general), bit for bit."""
    from mbpo_b200 import envs
    dev = cuda_device
    E, T = 96, 25
    system, params, _, x0, _ = _pair(which, mb, dev, E, seed=5)
    acts = _dev(np.random.default_rng(4).uniform(-1.5, 1.5, (T, E, system.u_dim)).astype(np.float32), dev)
    env = envs.wrap(system, params, episode_length=10 ** 6)
    nst, tr = env.unroll(env.reset(_dev(x0, dev)).replace(system_params=params), acts)
    x, p = _dev(x0, dev), params
    for t in range(T):
        out = system.step(x, acts[t], p)
        assert torch.equal(tr.next_observation[t], out.x_next) and torch.equal(tr.reward[t], out.reward), t
        x, p = out.x_next, out.system_params
    if system.keyed:
        assert torch.equal(nst.system_params.key, p.key)


def test_env_unroll_empty(mb, cuda_device, which):
    from mbpo_b200 import envs
    dev = cuda_device
    system, params, _, x0, keys = _pair(which, mb, dev, 7)
    env = envs.wrap(system, params, episode_length=5)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    nst, tr = env.unroll(st, torch.zeros((0, 7, system.u_dim), device=dev))
    assert tr.reward.shape == (0, 7) and torch.equal(nst.obs, st.obs)
    if keys is not None:
        assert np.array_equal(_keys_of(nst), keys)
    p0 = params.replace(key=torch.zeros((0, 2), dtype=torch.uint32, device=dev)) if keys is not None else params
    env0 = envs.wrap(system, p0, episode_length=5)
    nst0, tr0 = env0.unroll(env0.reset(torch.zeros((0, system.x_dim), device=dev)).replace(system_params=p0),
                            torch.zeros((4, 0, system.u_dim), device=dev))
    assert tr0.reward.shape == (4, 0) and nst0.obs.shape == (0, system.x_dim)


def _policy(mb, dev, system, seed, hidden=(64, 64), **kw):
    from mbpo_b200 import acting
    pol = orc.make_policy_params(seed=seed, obs_dim=system.x_dim, action_dim=system.u_dim, hidden=hidden)
    params = acting.PolicyParams([_dev(w, dev) for w in pol.weights], [_dev(b, dev) for b in pol.biases])
    return pol, acting.Policy(params, **kw)


def _check_teacher_forced_actor(osys, pol, tr, x0, key, keys, L, conv, prng, deterministic=False, extras=None,
                                rep=1):
    want, wk = gco.system_actor_rollout(osys, pol, x0, key, tr.reward.shape[0], L, key_convention=conv,
                                        deterministic=deterministic, action_repeat=rep, partitionable=prng,
                                        teacher_obs=tr.observation.cpu().numpy(), keys=keys,
                                        with_extras=extras is not None)
    np.testing.assert_allclose(tr.action.cpu().numpy(), want["action"], rtol=2e-5, atol=2e-6)
    # the env step of each row, from the GPU's own observation and action
    for t in range(tr.reward.shape[0]):
        np.testing.assert_allclose(tr.reward[t].cpu().numpy(), want["reward"][t], rtol=RTOL, atol=3e-5)
    assert np.array_equal(tr.discount.cpu().numpy(), want["discount"])
    if extras is not None:
        np.testing.assert_allclose(extras["raw_action"].cpu().numpy(), want["raw_action"], rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(extras["log_prob"].cpu().numpy(), want["log_prob"], rtol=2e-5, atol=2e-5)
    return want, wk


@pytest.mark.parametrize("conv", ["sac", "unroll", "as_is"])
def test_actor_rollout_vs_oracle(mb, cuda_device, prng_mode, which, conv):
    """All three key conventions; E not a multiple of the block; episodes end inside T.  The carry key and every env's
    system key are bit-exact."""
    from mbpo_b200 import acting, envs
    dev = cuda_device
    E, T, L = 150, 1 if conv == "as_is" else 23, 8
    system, params, osys, x0, keys = _pair(which, mb, dev, E, seed=11)
    pol, policy = _policy(mb, dev, system, 7)
    env = envs.wrap(system, params, episode_length=L)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = ojr.PRNGKey(3)
    kc = {"sac": mb._lib.KEYS_SAC, "unroll": mb._lib.KEYS_UNROLL, "as_is": mb._lib.KEYS_AS_IS}[conv]
    nst, tr, key_out = acting._rollout(env, st, policy, _dev(key, dev), T, kc, ("truncation",))
    want, wk = _check_teacher_forced_actor(osys, pol, tr, x0, key, keys, L, conv, prng_mode)
    assert np.array_equal(key_out.cpu().numpy(), wk)
    if keys is not None:
        assert np.array_equal(_keys_of(nst), want["final_keys"])
    assert np.array_equal(nst.info["steps"].cpu().numpy(), want["final_steps"])


def test_public_entry_points_route_general_systems(mb, cuda_device, which):
    """actor_step / generate_unroll / get_experience run for the general Systems and agree with _rollout."""
    from mbpo_b200 import acting, envs
    dev = cuda_device
    E, T, L = 64, 12, 5
    system, params, osys, x0, keys = _pair(which, mb, dev, E, seed=12)
    pol, policy = _policy(mb, dev, system, 8, hidden=(64,))
    env = envs.wrap(system, params, episode_length=L)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = ojr.PRNGKey(5)
    k, nst, tr = acting.get_experience(env, st, policy, _dev(key, dev), T)
    want, wk = _check_teacher_forced_actor(osys, pol, tr, x0, key, keys, L, "sac", False)
    assert np.array_equal(k.cpu().numpy(), wk)
    _, tru = acting.generate_unroll(env, st, policy, _dev(key, dev), T)
    _check_teacher_forced_actor(osys, pol, tru, x0, key, keys, L, "unroll", False)
    s1, t1 = acting.actor_step(env, st, policy, _dev(key, dev))
    assert t1.action.shape == (E, system.u_dim) and t1.reward.shape == (E,)
    if keys is not None:
        assert np.array_equal(_keys_of(nst), want["final_keys"])


def test_actor_deterministic_and_action_repeat(mb, cuda_device, prng_mode, which):
    from mbpo_b200 import acting, envs
    dev = cuda_device
    E, T, L = 70, 15, 9
    system, params, osys, x0, keys = _pair(which, mb, dev, E, seed=13)
    pol, policy = _policy(mb, dev, system, 9, hidden=(64, 64, 64), deterministic=True)
    env = envs.wrap(system, params, episode_length=L, action_repeat=2)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = ojr.PRNGKey(6)
    nst, tr = acting.generate_unroll(env, st, policy, _dev(key, dev), T)
    want, _ = _check_teacher_forced_actor(osys, pol, tr, x0, key, keys, L, "unroll", prng_mode, deterministic=True,
                                          rep=2)
    if keys is not None:                                   # two System steps per env step
        assert np.array_equal(_keys_of(nst), want["final_keys"])


def test_ppo_extras_point_mass(mb, cuda_device, prng_mode):
    """A = 2: raw_action [T, E, 2], log_prob summed over the two action dims."""
    from mbpo_b200 import acting, envs
    dev = cuda_device
    E, T, L = 97, 10, 6
    system, params, osys, x0, keys = _pair("point_mass", mb, dev, E, seed=14)
    pol, policy = _policy(mb, dev, system, 13, emit_extras=True)
    env = envs.wrap(system, params, episode_length=L)
    key = ojr.PRNGKey(8)
    _, tr = acting.generate_unroll(env, env.reset(_dev(x0, dev)).replace(system_params=params), policy,
                                   _dev(key, dev), T)
    ex = tr.extras["policy_extras"]
    assert ex["raw_action"].shape == (T, E, 2) and ex["log_prob"].shape == (T, E)
    _check_teacher_forced_actor(osys, pol, tr, x0, key, keys, L, "unroll", prng_mode, extras=ex)


def test_actor_env_sharding_is_bit_identical(mb, cuda_device, prng_mode, which):
    """Two launches owning envs [0, 77) and [77, 150) of 150 draw their slices of normal(key, (150, A))."""
    from mbpo_b200 import acting, envs
    dev = cuda_device
    E, T, L, cut = 150, 9, 4, 77
    system, params, _, x0, keys = _pair(which, mb, dev, E, seed=15)
    _, policy = _policy(mb, dev, system, 5)
    env = envs.wrap(system, params, episode_length=L)
    key = _dev(ojr.PRNGKey(4), dev)
    k, whole, tw = acting.get_experience(env, env.reset(_dev(x0, dev)).replace(system_params=params), policy, key, T)
    for lo, hi in ((0, cut), (cut, E)):
        p = params if keys is None else params.replace(key=params.key[lo:hi].contiguous())
        e = envs.wrap(system, p, episode_length=L)
        kk, part, tp = acting.get_experience(e, e.reset(_dev(x0[lo:hi], dev)).replace(system_params=p), policy, key, T,
                                             env_offset=lo, total_envs=E)
        assert torch.equal(kk, k)
        assert torch.equal(tp.action, tw.action[:, lo:hi]) and torch.equal(tp.reward, tw.reward[:, lo:hi])
        assert torch.equal(tp.next_observation, tw.next_observation[:, lo:hi])
        if keys is not None:
            assert torch.equal(part.system_params.key, whole.system_params.key[lo:hi])


def test_refusals(mb, cuda_device):
    from mbpo_b200 import acting, envs
    from mbpo_b200.systems import NoisyPendulumSystem
    L = mb._lib
    dev = cuda_device
    E = 8
    system, params, _, x0, _ = _pair("noisy_pendulum", mb, dev, E)
    env = envs.wrap(system, params, episode_length=5)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = _dev(ojr.PRNGKey(0), dev)
    # the pendulum keeps its own entry points
    g = system.pack_params(params)
    f = torch.zeros(E * 4, device=dev)
    rc = L.lib.mbpo_env_unroll_general(L.SYSTEM_PENDULUM, L.C.byref(g), 0, 5, 1, L.ptr(f), L.ptr(f), L.ptr(f), None,
                                       L.ptr(f), L.ptr(f), L.ptr(f), None, L.ptr(f), L.ptr(f), E, 1, None, None, None,
                                       None, None, None)
    assert rc == L.MBPO_EINVAL and b"mbpo_env_unroll" in L.lib.mbpo_last_error()
    _, policy = _policy(mb, dev, system, 3)
    rc = L.lib.mbpo_actor_rollout_general(L.SYSTEM_PENDULUM, L.C.byref(g), 0, L.C.byref(policy.struct), 0, 0,
                                          L.ptr(key), 5, 1, None, None, None, None, None, None, 0, 0, None, None, None,
                                          None, None, None, None, None, None)
    assert rc == L.MBPO_EINVAL and b"mbpo_actor_rollout" in L.lib.mbpo_last_error()
    # the BPTT head, an explicit tcgen05 kernel, a policy of the wrong shape
    bptt = acting.BpttActorPolicy(acting.PolicyParams(policy.weights, policy.biases))
    for bad in (bptt, _policy(mb, dev, system, 3, kernel="tcgen05")[1], _policy(mb, dev, system, 3,
                                                                                kernel="tcgen05_wide")[1],
                _policy(mb, dev, system, 3, hidden=(32, 32))[1]):
        with pytest.raises(mb._lib.MbpoUnsupported):
            acting.generate_unroll(env, st, bad, key, 3)
    # a keyed System whose params carry no key
    nokey = st.replace(system_params=params.replace(key=None))
    with pytest.raises(ValueError):
        env.unroll(nokey, torch.zeros((2, E, 1), device=dev))
    with pytest.raises(ValueError):
        acting.generate_unroll(env, nokey, policy, key, 2)
    assert isinstance(system, NoisyPendulumSystem)


def test_point_mass_collection_end_to_end(mb, cuda_device, prng_mode):
    """BraxWrapper reset from a PointMass true buffer (rows of 4 + 2 + 1 + 1 + 4 + 1 = 13 floats) -> get_experience ->
    replay insert -> running-statistics update, against the oracle."""
    from mbpo_b200 import acting, envs, running_statistics as rs
    from mbpo_b200.replay_buffers import UniformSamplingQueue
    from mbpo_b200.systems import BraxWrapper, PointMassSystem
    from mbpo_b200.systems.base_systems import SystemParams
    from mbpo_b200.utils.optimizer_utils import Transition
    dev = cuda_device
    z = lambda *s: torch.zeros(s, device=dev)
    system = PointMassSystem()
    dummy = Transition(z(4), z(2), z(), z(), z(4), {"state_extras": {"truncation": z()}, "policy_extras": {}})
    tq, otq = UniformSamplingQueue(64, dummy, 1), obr.UniformSamplingQueue(64, 13, 1, prng_mode)
    rng = np.random.default_rng(21)
    rows = rng.uniform(-1.5, 1.5, (40, 13)).astype(np.float32)
    r = _dev(rows, dev)
    tst = tq.insert(tq.init(_dev(ojr.PRNGKey(0), dev)),
                    Transition(r[:, :4], r[:, 4:6], r[:, 6], r[:, 7], r[:, 8:12],
                               {"state_extras": {"truncation": r[:, 12]}, "policy_extras": {}}))
    otst = otq.insert(otq.init(ojr.PRNGKey(0)), rows)
    assert np.array_equal(tst.data.cpu().numpy(), otst.data)
    E, T, L = 300, 16, 7
    params = SystemParams(dynamics_params=None, reward_params=None, key=None)
    env = envs.wrap(BraxWrapper(system, params, tst, tq), L, 1)
    rngs = ojr.split(ojr.PRNGKey(9), E, prng_mode)
    state = env.reset(_dev(rngs, dev))
    x0, _, _, _ = obr.brax_wrapper_reset(rngs, otq, otst, 4, 2)
    assert np.array_equal(state.obs.cpu().numpy(), x0)
    pol = orc.make_policy_params(seed=17, obs_dim=4, action_dim=2, hidden=(64, 64))
    pp = acting.PolicyParams([_dev(w, dev) for w in pol.weights], [_dev(b, dev) for b in pol.biases])
    q = UniformSamplingQueue(2 ** 13, dummy, 32)
    col = acting.ExperienceCollector(env, acting.make_normalized_inference_fn(), q, T)
    norm, buf = rs.init_state(4, dev), q.init(_dev(ojr.PRNGKey(2), dev))
    key = _dev(ojr.PRNGKey(4), dev)
    norm, nst, buf = col.get_experience(norm, pp, state, buf, key)
    live = buf.data[:T * E].cpu().numpy()
    assert buf.insert_position == T * E and live.shape == (T * E, 13)
    obs = live[:, :4].reshape(T, E, 4)
    # the first collection's statistics are the initial ones (mean 0, std 1): the policy saw the raw observations
    want, wk = gco.system_actor_rollout(orc.PointMassOracle(), pol, x0, ojr.PRNGKey(4), T, L, key_convention="sac",
                                        partitionable=prng_mode, teacher_obs=obs, obs_mean=np.zeros(4, np.float32),
                                        obs_std=np.ones(4, np.float32))
    np.testing.assert_allclose(live[:, 4:6].reshape(T, E, 2), want["action"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(live[:, 6].reshape(T, E), want["reward"], rtol=RTOL, atol=3e-5)
    assert np.array_equal(live[:, 7].reshape(T, E), want["discount"])
    assert np.array_equal(live[:, 12].reshape(T, E), want["truncation"])
    assert np.array_equal(col.last_key.cpu().numpy(), wk)
    onorm = obr.running_statistics_update(obr.running_statistics_init(4), obs, accumulate=np.float64)
    for k in ("count", "mean", "std"):
        np.testing.assert_allclose(getattr(norm, k).cpu().numpy(), onorm[k], rtol=1e-5, atol=1e-6)


def test_graphed_rollout_replays_eager_bits(mb, cuda_device, which):
    from mbpo_b200 import acting, envs
    dev = cuda_device
    E, T, L = 256, 8, 5
    system, params, _, x0, keys = _pair(which, mb, dev, E, seed=19)
    _, policy = _policy(mb, dev, system, 21)
    env = envs.wrap(system, params, episode_length=L)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = _dev(ojr.PRNGKey(12), dev)
    collect = acting.GraphedRollout(env, st, policy, key, T)
    k, s = key, st
    for _ in range(3):                                     # the graph hands env state, carry key and System keys on
        k, s, tr = acting.get_experience(env, s, policy, k, T)
        gk, gs, gtr = collect()
        assert torch.equal(gk, k) and torch.equal(gtr.action, tr.action) and torch.equal(gtr.reward, tr.reward)
        assert torch.equal(gtr.next_observation, tr.next_observation) and torch.equal(gs.obs, s.obs)
        if keys is not None:
            assert torch.equal(gs.system_params.key, s.system_params.key)
