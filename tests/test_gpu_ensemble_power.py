"""The learned-ensemble kernels against the oracle on the weight families of ensemble_power.py, at 1, 2, 3, 5 and 8
members: ensemble_transitions (one-tile and two-tile kernels on both sides of the dispatch switch, and config 4's
shape on a row subset) with its summary kernels, mbpo_ensemble_env_rollout with given actions under member layouts
that leave members empty, MLPEnsembleSystem.step (mlp_forward_tc_kernel) and a staged iCEM plan with one particle per
member.  Every next state is teacher-forced from the kernel's own state and compared with ensemble_power.check, whose
bars tests/test_oracle_ensemble_power.py shows every defect of ensemble_power.DEFECTS failing.  torch.profiler
confirms which kernel each case reached."""
import numpy as np
import pytest
import torch

from oracle import mbpo_oracle as orc

import ensemble_power as ep

pytestmark = pytest.mark.gpu

FAMILY = pytest.mark.parametrize("family", ep.FAMILIES)
MEMBERS = pytest.mark.parametrize("E", ep.MEMBER_COUNTS)


@pytest.fixture(scope="module")
def mb(cuda_device):
    import mbpo_b200
    return mbpo_b200


@pytest.fixture(scope="module")
def sms(cuda_device):
    return torch.cuda.get_device_properties(cuda_device).multi_processor_count


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _system(dev, family, E, member=None):
    """A fresh System and its params per call: MLPEnsembleSystem.packed caches the device weights by
    id(dynamics_params.weights), which a new list reused at a freed address would alias."""
    from mbpo_b200.systems import MLPEnsembleSystem, MlpEnsembleDynamicsParams, PendulumRewardParams, SystemParams
    ens = ep.ensemble(family, E)
    dyn = MlpEnsembleDynamicsParams(weights=[_dev(w, dev) for w in ens.weights],
                                    biases=[_dev(b, dev) for b in ens.biases],
                                    member=None if member is None else _dev(member, dev))
    return (MLPEnsembleSystem(num_members=E, dynamics_params=dyn),
            SystemParams(dynamics_params=dyn, reward_params=PendulumRewardParams()))


def _profiled(fn):
    """fn() under torch.profiler -> (its result, the names of the CUDA kernels it launched)."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return out, names


def _reached(names, kernel):
    """Whether `kernel` (an unqualified kernel name) is among the profiled names."""
    return any(n.split("(")[0].split("<")[0].split("::")[-1] == kernel for n in names)


def _rewards_ok(r, o, u):
    _, want = orc.pendulum_step(o.reshape(-1, 3), u.reshape(-1), orc.PendulumParams())
    np.testing.assert_allclose(r.reshape(-1), want, rtol=1e-5, atol=1e-6)


# ---- ensemble_transitions: both row-tile kernels, per step and per member ---------------------------------------
@pytest.mark.parametrize("case", [c[0] for c in ep.rollout_cases()])
@MEMBERS
@FAMILY
def test_transitions(mb, cuda_device, sms, family, E, case):
    idx = [c[0] for c in ep.rollout_cases(sms)].index(case)
    name, B, M, H, n = ep.rollout_cases(sms)[idx]
    x0, acts, rows = ep.rollout_inputs(name, B, M, H, n, seed=1000 + idx)
    system, sp = _system(cuda_device, family, E)
    x0_d, acts_d = _dev(x0, cuda_device), _dev(acts, cuda_device)
    (obs, rew), names = _profiled(lambda: system.ensemble_transitions(sp, x0_d, acts_d))
    assert _reached(names, ep.rollout_kernel(B, M, sms)), names
    assert obs.shape == (B, M, E, H, 3) and rew.shape == (B, M, E, H)

    # the summary kernels: bit for bit the member summary of the kernel's own rewards, through
    # mbpo_icem_penalize_particles and through the float32 restatement of it
    L = mb._lib
    rew_np = rew.reshape(B * M, E, H).cpu().numpy()
    summary_kernel = ep.rollout_kernel(B, M, sms).replace("transitions", "rollout")
    for use_max in (False, True):
        want, names = _profiled(lambda: system.ensemble_returns(sp, x0_d, acts_d, use_optimism=use_max))
        assert _reached(names, summary_kernel), names
        tail = torch.empty_like(want)
        L.check(L.lib.mbpo_icem_penalize_particles(L.ptr(tail), L.ptr(rew), H, None, B * M, E, int(use_max), 0, 1.0,
                                                   L.stream_ptr(cuda_device)))
        assert torch.equal(tail, want)
        assert np.array_equal(want.reshape(-1).cpu().numpy(), ep.summary(rew_np, use_max))

    o = obs.reshape(B * M, E, H, 3)[torch.from_numpy(rows).to(cuda_device)].cpu().numpy()
    r = rew_np[rows]
    u = acts.reshape(B * M, H)[rows]
    assert np.array_equal(o[:, :, 0], np.broadcast_to(x0[rows // M][:, None], (len(rows), E, 3)))
    _rewards_ok(r, o, np.broadcast_to(u[:, None], r.shape))
    if H == 1:
        return
    # teacher-forced: step t of member e from the kernel's own state o[:, e, t]; items are (row, member) pairs
    obs_t = o[:, :, :-1].transpose(2, 0, 1, 3).reshape(H - 1, -1, 3)
    acts_t = np.broadcast_to(u.T[:, :, None], (H, len(rows), E)).reshape(H, -1)
    member = np.broadcast_to(np.arange(E, dtype=np.int32), (len(rows), E)).reshape(-1)
    want, _ = ep.teacher_forced(family, E, obs_t, acts_t, member)
    got = o[:, :, 1:].transpose(2, 0, 1, 3).reshape(-1, 3)
    ep.check("fused", family, got, want, test="transitions", case=case, E=E)


# ---- mbpo_ensemble_env_rollout with given actions ---------------------------------------------------------------
@pytest.mark.parametrize("layout,n_envs,T", ep.ENV_CASES)
@MEMBERS
@FAMILY
def test_env_rollout(mb, cuda_device, family, E, layout, n_envs, T):
    from mbpo_b200 import envs
    x0, acts, member, rows = ep.env_inputs(layout, n_envs, T, E)
    system, params = _system(cuda_device, family, E, member)
    env = envs.wrap(system, params, episode_length=1000, action_repeat=1)
    st = env.reset(_dev(x0, cuda_device)).replace(system_params=params)
    (nst, tr), names = _profiled(lambda: env.unroll(st, _dev(acts, cuda_device)))
    assert _reached(names, "ensemble_env_kernel"), names
    obs, nxt = tr.observation.cpu().numpy(), tr.next_observation.cpu().numpy()
    assert np.array_equal(obs[0], x0) and np.array_equal(obs[1:], nxt[:-1])
    assert not tr.extras["state_extras"]["truncation"].any()
    _rewards_ok(tr.reward.cpu().numpy()[:, rows], obs[:, rows], acts[:, rows, 0])
    want, _ = ep.teacher_forced(family, E, obs[:, rows], acts[:, rows, 0], member[rows])
    ep.check("fused", family, nxt[:, rows].reshape(-1, 3), want, test="env", case="%s-%d" % (layout, n_envs), E=E)


# ---- MLPEnsembleSystem.step --------------------------------------------------------------------------------------
@MEMBERS
@FAMILY
def test_system_step(mb, cuda_device, family, E):
    x, u, member = ep.step_inputs(E)
    system, sp = _system(cuda_device, family, E, member)
    st, names = _profiled(lambda: system.step(_dev(x, cuda_device), _dev(u, cuda_device), sp))
    assert _reached(names, "mlp_forward_tc_kernel"), names
    want, _ = ep.teacher_forced(family, E, x[None], u.T, member)
    ep.check("forward", family, st.x_next.cpu().numpy(), want, test="step", case="mixed", E=E)


# ---- the staged iCEM plan with one particle per member -----------------------------------------------------------
@MEMBERS
@FAMILY
def test_staged_plan(mb, cuda_device, family, E):
    """The plan's values are mbpo_ensemble_rollout's returns of its own actions, bit for bit, and the oracle's refit
    of those values picks the plan's elites and gives its mean and std."""
    from mbpo_b200.optimizers import iCemTO, iCemParams
    system, _ = _system(cuda_device, family, E)
    H, B = 10, 2
    params = dict(num_samples=64, num_elites=8, num_particles=E, num_steps=2)
    opt = iCemTO(horizon=H, action_dim=1, opt_params=iCemParams(**params))
    opt.set_system(system)
    keys = np.random.default_rng(4000 + E).integers(0, 2 ** 32, (B, 2), dtype=np.uint64).astype(np.uint32)
    st = opt.init(_dev(keys, cuda_device))
    x0_d = _dev(ep.pendulum_states(B, 4001), cuda_device)
    seq, val, _, tr = opt._plan_raw(x0_d, st.key, st.best_sequence, st.system_params, trace=True)
    p = orc.ICemParams(**params)
    M = p.num_samples + p.num_prev_elites
    for it in range(p.num_steps):
        again = system.ensemble_returns(st.system_params, x0_d, tr["actions"][it].reshape(B, M, H, 1))
        assert torch.equal(again, tr["values"][it])
    tr = {k: v.cpu().numpy() for k, v in tr.items()}
    for b in range(B):
        mean, std = np.zeros((H, 1), np.float32), np.full((H, 1), p.init_std, np.float32)
        bval, bseq = np.float32(-np.inf), mean.copy()
        for it in range(p.num_steps):
            g_acts = tr["actions"][it, b].reshape(M, H, 1)
            mean, std, bval, bseq, idx = orc.icem_refit(g_acts, tr["values"][it, b], mean, std, bval, bseq, p)
            assert np.array_equal(tr["elite_idx"][it, b], idx)
            assert np.array_equal(tr["mean"][it, b].reshape(H, 1), mean)
            assert np.array_equal(tr["std"][it, b].reshape(H, 1), std)
        assert np.array_equal(seq[b].cpu().numpy(), bseq) and float(val[b]) == float(bval)
