"""GPU parity of the learned ensemble as a SAC / PPO env (mbpo_ensemble_env_rollout) against the collection oracle
(general_collection_oracle.py over ensemble_collection_oracle.EnsembleOracle): env e rolled through
dynamics_params.member[e].  Wrapper fields (steps, done, truncation, discount) and PRNG words are exact; the model's
next state is compared per step, teacher-forced on the GPU's own observations, at the single-step ensemble tolerance
(rtol 2e-3, atol 2e-4; at most one element in 200 beyond it, none beyond atol 2.5e-3)."""
import numpy as np
import pytest
import torch

from oracle import brax_replay as obr
from oracle import jax_prng as ojr
from oracle import mbpo_oracle as orc

import ensemble_collection_oracle as eco
import general_collection_oracle as gco

pytestmark = pytest.mark.gpu

M = 5


@pytest.fixture(scope="module")
def mb(cuda_device):
    import mbpo_b200
    return mbpo_b200


@pytest.fixture(scope="module")
def ens():
    return orc.make_mlp_ensemble(seed=3, members=M)


@pytest.fixture(params=[False, True], ids=["legacy", "partitionable"])
def prng_mode(request, mb):
    mb.config.threefry_partitionable = request.param
    yield request.param
    mb.config.threefry_partitionable = False


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _members(kind, E):
    if kind == "none":
        return None
    if kind == "contiguous":
        return (np.arange(E) * M // max(E, 1)).astype(np.int32)
    return (np.arange(E) % M).astype(np.int32)


def _system(mb, dev, ens, member):
    from mbpo_b200.systems import MLPEnsembleSystem, MlpEnsembleDynamicsParams, PendulumRewardParams, SystemParams
    dyn = MlpEnsembleDynamicsParams(weights=[_dev(w, dev) for w in ens.weights],
                                    biases=[_dev(b, dev) for b in ens.biases],
                                    member=None if member is None else _dev(member, dev))
    return MLPEnsembleSystem(), SystemParams(dynamics_params=dyn, reward_params=PendulumRewardParams())


def _states(rng, e):
    th, w = rng.uniform(-np.pi, np.pi, e), rng.uniform(-8, 8, e)
    return np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)


def _start(mb, env, x0, first, steps0, done0, dev, params):
    st = env.reset(_dev(first, dev))
    st = st.replace(obs=_dev(x0, dev), system_params=params)
    st.info["steps"].copy_(_dev(steps0, dev))
    st.done.copy_(_dev(done0, dev))
    return st


def _policy(mb, dev, seed, hidden=(64, 64), **kw):
    from mbpo_b200 import acting
    pol = orc.make_policy_params(seed=seed, obs_dim=3, action_dim=1, hidden=hidden)
    params = acting.PolicyParams([_dev(w, dev) for w in pol.weights], [_dev(b, dev) for b in pol.biases])
    return pol, acting.Policy(params, **kw)


def _check_env(osys, tr, acts, x0, first, steps0, done0, L, rep, rows=None):
    """Each step re-run by the oracle from the GPU's observation[t]; the bookkeeping carried by the oracle."""
    obs, nxt = tr.observation.cpu().numpy(), tr.next_observation.cpu().numpy()
    rew, disc, trunc = tr.reward.cpu().numpy(), tr.discount.cpu().numpy(), tr.extras["state_extras"]["truncation"]
    trunc = trunc.cpu().numpy()
    T, E = rew.shape
    assert np.array_equal(obs[0], x0)
    sel = np.arange(E) if rows is None else rows
    steps, done = steps0.copy(), done0.copy()
    beyond = checked = r_beyond = r_checked = 0
    for t in range(T):
        steps = np.where(done != 0, np.float32(0), steps).astype(np.float32)
        done = np.zeros(E, np.float32)
        x, r = obs[t][sel], np.zeros(len(sel), np.float32)
        for _ in range(rep):
            x, rr, _ = osys.step(x, acts[t][sel], None)
            r = (r + rr).astype(np.float32)
        steps = (steps + np.float32(rep)).astype(np.float32)
        over = steps >= np.float32(L)
        want_trunc = np.where(over, np.float32(1) - done, np.float32(0)).astype(np.float32)
        done = np.where(over, np.float32(1), done).astype(np.float32)
        assert np.array_equal(disc[t], 1 - done) and np.array_equal(trunc[t], want_trunc), t
        assert np.array_equal(nxt[t][over], first[over]), t                  # reset rows: first_obs, bit for bit
        live = ~over[sel]
        # the single-step bar.  The fused kernel's swish (tanh.approx, as the iCEM kernel's) can flip one activation's
        # bf16 rounding against the oracle, which moves that row's delta by up to ~1e-3 on the large states these
        # learned-model rollouts reach: at most 1 element in 200 may pass the bar, none by more than 2.5e-3.
        got, want = nxt[t][sel][live], x[live]
        np.testing.assert_allclose(got, want, rtol=2e-3, atol=2.5e-3)
        beyond += int(np.count_nonzero(np.abs(got - want) > 2e-4 + 2e-3 * np.abs(want)))
        checked += got.size
        if rep == 1:
            np.testing.assert_allclose(rew[t][sel], r, rtol=1e-5, atol=3e-6)
        else:                                   # the second model step starts from the oracle's own state
            np.testing.assert_allclose(rew[t][sel], r, rtol=2e-3, atol=1e-2)
            r_beyond += int(np.count_nonzero(np.abs(rew[t][sel] - r) > 2e-4 + 2e-3 * np.abs(r)))
            r_checked += r.size
    assert beyond <= max(1, checked // 200), (beyond, checked)
    assert r_beyond <= max(1, r_checked // 200), (r_beyond, r_checked)
    return steps, done


@pytest.mark.parametrize("E,T,rep,kind", [(1, 5, 1, "none"), (77, 200, 1, "interleaved"), (77, 40, 2, "contiguous"),
                                          (300, 30, 2, "interleaved"), (300, 24, 1, "none"),
                                          (1000, 12, 1, "contiguous"), (1000, 10, 2, "interleaved"),
                                          (20000, 6, 1, "interleaved"), (20000, 4, 2, "contiguous")])
def test_env_unroll_vs_oracle(mb, cuda_device, ens, E, T, rep, kind):
    """Teacher-forced unroll; episode_length 7 so that resets happen; E = 20,000 is more than one round of CTA pairs
    with partial tiles (its model step is checked on 2,000 rows, its wrapper fields on all)."""
    from mbpo_b200 import envs
    dev, L = cuda_device, 7
    rng = np.random.default_rng(E + T)
    member = _members(kind, E)
    system, params = _system(mb, dev, ens, member)
    x0, first = _states(rng, E), _states(rng, E)
    steps0 = rng.integers(0, L, E).astype(np.float32)
    done0 = (rng.uniform(size=E) < 0.2).astype(np.float32)
    acts = rng.uniform(-2, 2, (T, E, 1)).astype(np.float32)
    env = envs.wrap(system, params, episode_length=L, action_repeat=rep)
    st = _start(mb, env, x0, first, steps0, done0, dev, params)
    nst, tr = env.unroll(st, _dev(acts, dev))
    rows = None if E <= 1000 else np.sort(rng.choice(E, 2000, replace=False))
    osys = eco.EnsembleOracle(ens, member if member is None or rows is None else member[rows])   # the rows checked
    steps, done = _check_env(osys, tr, acts, x0, first, steps0, done0, L, rep, rows)
    assert np.array_equal(nst.info["steps"].cpu().numpy(), steps) and np.array_equal(nst.done.cpu().numpy(), done)
    assert torch.equal(nst.obs, tr.next_observation[-1])
    # one step at a time is the same launch per step
    if E <= 300 and T <= 40:
        s = st
        for t in range(3):
            s = env.step(s, _dev(acts[t], dev))
            assert torch.equal(s.obs, tr.next_observation[t])


def test_independence_from_other_envs(mb, cuda_device, ens):
    """Permuting the envs with their states and members permutes every output bit for bit; changing the other envs'
    members leaves an env's rows bit-identical."""
    from mbpo_b200 import envs
    dev, E, T, L = cuda_device, 700, 20, 7
    rng = np.random.default_rng(5)
    member = rng.integers(0, M, E).astype(np.int32)
    x0 = _states(rng, E)
    steps0 = rng.integers(0, L, E).astype(np.float32)
    acts = rng.uniform(-2, 2, (T, E, 1)).astype(np.float32)

    def run(mem, x, s, a):
        system, params = _system(mb, dev, ens, mem)
        env = envs.wrap(system, params, episode_length=L, action_repeat=2)
        return env.unroll(_start(mb, env, x, x, s, np.zeros(len(x), np.float32), dev, params), _dev(a, dev))

    nst, tr = run(member, x0, steps0, acts)
    perm = rng.permutation(E)
    pst, ptr = run(member[perm], x0[perm], steps0[perm], acts[:, perm])
    p = _dev(perm, dev)
    for f in ("observation", "next_observation", "reward", "discount"):
        assert torch.equal(getattr(ptr, f), getattr(tr, f)[:, p]), f
    assert torch.equal(ptr.extras["state_extras"]["truncation"], tr.extras["state_extras"]["truncation"][:, p])
    assert torch.equal(pst.obs, nst.obs[p]) and torch.equal(pst.info["steps"], nst.info["steps"][p])
    keep = rng.uniform(size=E) < 0.3
    other = np.where(keep, member, (member + 1 + rng.integers(0, M - 1, E)) % M).astype(np.int32)
    _, otr = run(other, x0, steps0, acts)
    k = _dev(np.nonzero(keep)[0], dev)
    for f in ("next_observation", "reward"):
        assert torch.equal(getattr(otr, f)[:, k], getattr(tr, f)[:, k]), f
    assert not torch.equal(otr.next_observation, tr.next_observation)


def _check_actor(osys, pol, tr, x0, key, L, conv, prng, deterministic=False, extras=None, rep=1, mean=None, std=None):
    want, wk = gco.system_actor_rollout(osys, pol, x0, key, tr.reward.shape[0], L, key_convention=conv,
                                        deterministic=deterministic, action_repeat=rep, partitionable=prng,
                                        teacher_obs=tr.observation.cpu().numpy(), obs_mean=mean, obs_std=std,
                                        with_extras=extras is not None)
    np.testing.assert_allclose(tr.action.cpu().numpy(), want["action"], rtol=2e-5, atol=2e-6)
    assert np.array_equal(tr.discount.cpu().numpy(), want["discount"])
    if "truncation" in tr.extras["state_extras"]:
        assert np.array_equal(tr.extras["state_extras"]["truncation"].cpu().numpy(), want["truncation"])
    if rep == 1:
        np.testing.assert_allclose(tr.reward.cpu().numpy(), want["reward"], rtol=1e-5, atol=3e-5)
    if extras is not None:
        np.testing.assert_allclose(extras["raw_action"].cpu().numpy(), want["raw_action"], rtol=2e-5, atol=3e-6)
        np.testing.assert_allclose(extras["log_prob"].cpu().numpy(), want["log_prob"], rtol=1e-4, atol=1e-4)
    return want, wk


@pytest.mark.parametrize("conv", ["sac", "unroll", "as_is"])
def test_policy_in_the_loop_vs_oracle(mb, cuda_device, ens, prng_mode, conv):
    """actor_step / generate_unroll / get_experience: actions against policy_sample on the kernel's own observations,
    the carry key bit-exact."""
    from mbpo_b200 import acting, envs
    dev, E, L = cuda_device, 300, 7
    T = 1 if conv == "as_is" else 20
    rng = np.random.default_rng(9)
    member = _members("interleaved", E)
    system, params = _system(mb, dev, ens, member)
    osys = eco.EnsembleOracle(ens, member)
    x0 = _states(rng, E)
    pol, policy = _policy(mb, dev, 7)
    env = envs.wrap(system, params, episode_length=L)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = ojr.PRNGKey(3)
    if conv == "sac":
        k, nst, tr = acting.get_experience(env, st, policy, _dev(key, dev), T)
    elif conv == "unroll":
        nst, tr = acting.generate_unroll(env, st, policy, _dev(key, dev), T, extra_fields=("truncation",))
        _, _, k = acting._rollout(env, st, policy, _dev(key, dev), T, mb._lib.KEYS_UNROLL, ())
    else:
        nst, t1 = acting.actor_step(env, st, policy, _dev(key, dev), extra_fields=("truncation",))
        tr = acting._rollout(env, st, policy, _dev(key, dev), 1, mb._lib.KEYS_AS_IS, ("truncation",))[1]
        assert torch.equal(t1.action, tr.action[0]) and torch.equal(t1.next_observation, tr.next_observation[0])
        k = None
    want, wk = _check_actor(osys, pol, tr, x0, key, L, conv, prng_mode)
    if k is not None:
        assert np.array_equal(k.cpu().numpy(), wk)
    assert np.array_equal(nst.info["steps"].cpu().numpy(), want["final_steps"])


def test_deterministic_extras_and_normaliser(mb, cuda_device, ens, prng_mode):
    """deterministic mode does not depend on the key; PPO's extras; the normaliser as floats and as device tensors
    gives the same bits; action_repeat 2; a 1-hidden-layer policy."""
    from mbpo_b200 import acting, envs
    dev, E, T, L = cuda_device, 257, 15, 9
    rng = np.random.default_rng(10)
    member = _members("contiguous", E)
    system, params = _system(mb, dev, ens, member)
    osys = eco.EnsembleOracle(ens, member)
    x0 = _states(rng, E)
    mean = np.array([0.1, -0.2, 0.5], np.float32)
    std = np.array([0.9, 1.1, 3.0], np.float32)
    env = envs.wrap(system, params, episode_length=L, action_repeat=2)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    pol, det = _policy(mb, dev, 9, hidden=(64,), deterministic=True, obs_mean=mean.tolist(), obs_std=std.tolist())
    _, tr1 = acting.generate_unroll(env, st, det, _dev(ojr.PRNGKey(1), dev), T)
    _, tr2 = acting.generate_unroll(env, st, det, _dev(ojr.PRNGKey(2), dev), T)
    assert torch.equal(tr1.action, tr2.action) and torch.equal(tr1.next_observation, tr2.next_observation)
    _check_actor(osys, pol, tr1, x0, ojr.PRNGKey(1), L, "unroll", prng_mode, deterministic=True, rep=2, mean=mean,
                 std=std)
    env1 = envs.wrap(system, params, episode_length=L)
    pol2, ppo = _policy(mb, dev, 13, emit_extras=True, obs_mean=mean.tolist(), obs_std=std.tolist())
    _, tr = acting.generate_unroll(env1, st, ppo, _dev(ojr.PRNGKey(8), dev), T)
    ex = tr.extras["policy_extras"]
    assert ex["raw_action"].shape == (T, E, 1) and ex["log_prob"].shape == (T, E)
    _check_actor(osys, pol2, tr, x0, ojr.PRNGKey(8), L, "unroll", prng_mode, extras=ex, mean=mean, std=std)
    _, ppo_dev = _policy(mb, dev, 13, emit_extras=True, obs_mean=_dev(mean, dev), obs_std=_dev(std, dev))
    _, trd = acting.generate_unroll(env1, st, ppo_dev, _dev(ojr.PRNGKey(8), dev), T)
    assert torch.equal(trd.action, tr.action) and torch.equal(trd.extras["policy_extras"]["log_prob"], ex["log_prob"])


def test_closure_policy_actions_through_unroll(mb, cuda_device, ens, prng_mode):
    """The policy run's actions fed back through unroll give bit-identical observations, rewards and wrapper fields."""
    from mbpo_b200 import acting, envs
    dev, E, T, L = cuda_device, 600, 25, 7
    rng = np.random.default_rng(11)
    system, params = _system(mb, dev, ens, _members("interleaved", E))
    x0 = _states(rng, E)
    _, policy = _policy(mb, dev, 5)
    env = envs.wrap(system, params, episode_length=L, action_repeat=2)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    _, nst, tr = acting.get_experience(env, st, policy, _dev(ojr.PRNGKey(4), dev), T)
    ust, utr = env.unroll(st, tr.action)
    for f in ("observation", "next_observation", "reward", "discount"):
        assert torch.equal(getattr(utr, f), getattr(tr, f)), f
    assert torch.equal(utr.extras["state_extras"]["truncation"], tr.extras["state_extras"]["truncation"])
    assert torch.equal(ust.obs, nst.obs) and torch.equal(ust.info["steps"], nst.info["steps"])
    assert torch.equal(ust.done, nst.done)


def test_sharding_is_bit_identical(mb, cuda_device, ens, prng_mode):
    """Launches owning envs [0, 301) and [301, 600) of 600 equal those slices of the whole launch."""
    from mbpo_b200 import acting, envs
    dev, E, T, L, cut = cuda_device, 600, 9, 4, 301
    rng = np.random.default_rng(12)
    member = _members("interleaved", E)
    x0 = _states(rng, E)
    _, policy = _policy(mb, dev, 5)
    key = _dev(ojr.PRNGKey(4), dev)
    system, params = _system(mb, dev, ens, member)
    env = envs.wrap(system, params, episode_length=L)
    k, whole, tw = acting.get_experience(env, env.reset(_dev(x0, dev)).replace(system_params=params), policy, key, T)
    for lo, hi in ((0, cut), (cut, E)):
        s, p = _system(mb, dev, ens, member[lo:hi])
        e = envs.wrap(s, p, episode_length=L)
        kk, part, tp = acting.get_experience(e, e.reset(_dev(x0[lo:hi], dev)).replace(system_params=p), policy, key, T,
                                             env_offset=lo, total_envs=E)
        assert torch.equal(kk, k)
        for f in ("action", "reward", "next_observation", "discount"):
            assert torch.equal(getattr(tp, f), getattr(tw, f)[:, lo:hi]), f
        assert torch.equal(part.obs, whole.obs[lo:hi])


def test_graphed_rollout_replays_eager_bits(mb, cuda_device, ens):
    from mbpo_b200 import acting, envs
    dev, E, T, L = cuda_device, 500, 8, 5
    rng = np.random.default_rng(13)
    system, params = _system(mb, dev, ens, _members("interleaved", E))
    x0 = _states(rng, E)
    _, policy = _policy(mb, dev, 21)
    env = envs.wrap(system, params, episode_length=L)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = _dev(ojr.PRNGKey(12), dev)
    collect = acting.GraphedRollout(env, st, policy, key, T)
    k, s = key, st
    for _ in range(3):
        k, s, tr = acting.get_experience(env, s, policy, k, T)
        gk, gs, gtr = collect()
        assert torch.equal(gk, k) and torch.equal(gtr.action, tr.action) and torch.equal(gtr.reward, tr.reward)
        assert torch.equal(gtr.next_observation, tr.next_observation) and torch.equal(gs.obs, s.obs)


def test_end_to_end_true_buffer_replay_and_evaluator(mb, cuda_device, ens, prng_mode):
    """BraxWrapper(ensemble) resets from a true buffer -> ExperienceCollector.get_experience into a
    UniformSamplingQueue -> one Evaluator.run_evaluation."""
    from mbpo_b200 import acting, envs, running_statistics as rs
    from mbpo_b200.replay_buffers import UniformSamplingQueue
    from mbpo_b200.systems import BraxWrapper
    from mbpo_b200.utils.optimizer_utils import Transition
    dev = cuda_device
    z = lambda *s: torch.zeros(s, device=dev)
    dummy = Transition(z(3), z(1), z(), z(), z(3), {"state_extras": {"truncation": z()}, "policy_extras": {}})
    tq, otq = UniformSamplingQueue(64, dummy, 1), obr.UniformSamplingQueue(64, 10, 1, prng_mode)
    rng = np.random.default_rng(21)
    rows = rng.uniform(-1.5, 1.5, (40, 10)).astype(np.float32)   # 3 + 1 + 1 + 1 + 3 + 1
    r = _dev(rows, dev)
    tst = tq.insert(tq.init(_dev(ojr.PRNGKey(0), dev)),
                    Transition(r[:, :3], r[:, 3:4], r[:, 4], r[:, 5], r[:, 6:9],
                               {"state_extras": {"truncation": r[:, 9]}, "policy_extras": {}}))
    otst = otq.insert(otq.init(ojr.PRNGKey(0)), rows)
    E, T, L = 300, 12, 7
    system, params = _system(mb, dev, ens, None)
    env = envs.wrap(BraxWrapper(system, params, tst, tq), L, 1)
    rngs = ojr.split(ojr.PRNGKey(9), E, prng_mode)
    state = env.reset(_dev(rngs, dev))
    x0, _, _, _ = obr.brax_wrapper_reset(rngs, otq, otst, 3, 1)
    assert np.array_equal(state.obs.cpu().numpy(), x0)
    pol = orc.make_policy_params(seed=17, obs_dim=3, action_dim=1, hidden=(64, 64))
    pp = acting.PolicyParams([_dev(w, dev) for w in pol.weights], [_dev(b, dev) for b in pol.biases])
    q = UniformSamplingQueue(2 ** 13, dummy, 32)
    col = acting.ExperienceCollector(env, acting.make_normalized_inference_fn(), q, T)
    norm, buf = rs.init_state(3, dev), q.init(_dev(ojr.PRNGKey(2), dev))
    norm, nst, buf = col.get_experience(norm, pp, state, buf, _dev(ojr.PRNGKey(4), dev))
    live = buf.data[:T * E].cpu().numpy()
    assert buf.insert_position == T * E and live.shape == (T * E, 10)
    obs = live[:, :3].reshape(T, E, 3)
    want, wk = gco.system_actor_rollout(eco.EnsembleOracle(ens), pol, x0, ojr.PRNGKey(4), T, L, key_convention="sac",
                                        partitionable=prng_mode, teacher_obs=obs, obs_mean=np.zeros(3, np.float32),
                                        obs_std=np.ones(3, np.float32))
    np.testing.assert_allclose(live[:, 3].reshape(T, E), want["action"][..., 0], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(live[:, 4].reshape(T, E), want["reward"], rtol=1e-5, atol=3e-5)
    assert np.array_equal(live[:, 5].reshape(T, E), want["discount"])
    assert np.array_equal(live[:, 9].reshape(T, E), want["truncation"])
    assert np.array_equal(col.last_key.cpu().numpy(), wk)
    ev = acting.Evaluator(env, acting.make_inference_fn(), 64, L, 1, _dev(ojr.PRNGKey(6), dev))
    metrics = ev.run_evaluation(pp, {})
    assert np.isfinite(metrics["eval/episode_reward"]) and metrics["eval/avg_episode_length"] > 0


def test_refusals(mb, cuda_device, ens):
    from mbpo_b200 import acting, envs
    dev, E = cuda_device, 16
    rng = np.random.default_rng(0)
    x0 = _states(rng, E)
    system, params = _system(mb, dev, ens, _members("interleaved", E))
    env = envs.wrap(system, params, episode_length=5)
    st = env.reset(_dev(x0, dev)).replace(system_params=params)
    key = _dev(ojr.PRNGKey(0), dev)
    _, policy = _policy(mb, dev, 3)
    bptt = acting.BpttActorPolicy(acting.PolicyParams(policy.weights, policy.biases))
    for bad in (bptt, _policy(mb, dev, 3, kernel="tcgen05")[1], _policy(mb, dev, 3, kernel="tcgen05_wide")[1],
                _policy(mb, dev, 3, hidden=(64, 64, 64))[1], _policy(mb, dev, 3, hidden=(32, 32))[1]):
        with pytest.raises(mb._lib.MbpoUnsupported):
            acting.generate_unroll(env, st, bad, key, 3)
    with pytest.raises(mb._lib.MbpoUnsupported, match="shared memory"):
        acting.generate_unroll(env, st, _policy(mb, dev, 3, hidden=(64, 64, 64, 64))[1], key, 3)
    # bad member tensors: ValueError before anything is launched
    for bad in (np.arange(E) % M + 1, -(np.arange(E) % 2), np.zeros(E + 1, np.int32), np.zeros((E, 2), np.int32)):
        s, p = _system(mb, dev, ens, bad.astype(np.int32))
        e = envs.wrap(s, p, episode_length=5)
        stb = e.reset(_dev(x0, dev)).replace(system_params=p)
        with pytest.raises(ValueError):
            e.unroll(stb, torch.zeros((2, E, 1), device=dev))
        with pytest.raises(ValueError):
            acting.generate_unroll(e, stb, policy, key, 2)
    # the existing entry points keep refusing the ensemble kind
    L = mb._lib
    assert L.lib.mbpo_env_unroll(L.SYSTEM_MLP_ENSEMBLE, None, 0, 3, 1, 5, 1, None, None, None, None, None, None, None,
                                 None, 1, 1, None, None, None, None, None, None) == L.MBPO_EUNSUPPORTED
    # E = 0 / T = 0
    nst, tr = env.unroll(st, torch.zeros((0, E, 1), device=dev))
    assert torch.equal(nst.obs, st.obs) and tr.reward.shape == (0, E)
    k, _, tr0 = acting.get_experience(env, st, policy, key, 0)
    assert torch.equal(k, key) and tr0.action.shape == (0, E, 1)
