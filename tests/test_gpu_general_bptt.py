"""GPU parity of BPTT's forward and cotangent pass for the general Systems (mbpo_rollout_policy_general,
mbpo_rollout_adjoint_general) against general_bptt_oracle.py: NoisyPendulumSystem (keyed, X = 3, A = 1) and
PointMassSystem (X = 4, A = 2) in both PRNG layouts.  PRNG words are bit-exact; actions are compared per step,
teacher-forced on the GPU's observations; the adjoint against the float64 oracle on the GPU's trajectory; the whole
gradient against torch autograd through a float64 rollout."""
import numpy as np
import pytest
import torch

from oracle import jax_prng as ojr
from oracle import mbpo_oracle as orc

import general_bptt_oracle as gbo
import general_collection_oracle as gco

pytestmark = pytest.mark.gpu


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
    return np.random.default_rng(seed).integers(0, 2 ** 32, size=(n, 2), dtype=np.uint64).astype(np.uint32)


def _system(which, dev, B, seed):
    """(GPU System, SystemParams without a key, oracle System, x0 [B, X])."""
    from mbpo_b200.systems import NoisyPendulumSystem, PointMassSystem
    from mbpo_b200.systems.base_systems import SystemParams
    rng = np.random.default_rng(seed)
    if which == "noisy_pendulum":
        system, osys = NoisyPendulumSystem(noise_std=0.05), orc.NoisyPendulumOracle(noise_std=0.05)
        th, w = rng.uniform(-np.pi, np.pi, B), rng.uniform(-6, 6, B)
        x0 = np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)
        params = system.init_params(_dev(ojr.PRNGKey(1), dev))
    else:
        system, osys = PointMassSystem(), orc.PointMassOracle()
        x0 = rng.uniform(-2, 2, (B, 4)).astype(np.float32)
        params = SystemParams(dynamics_params=None, reward_params=None, key=None)
    return system, params, osys, x0


def _key_forms(system, params, B, dev, seed):
    """(name, SystemParams, oracle sys_keys) for every System-key form: none for PointMass; [2] shared and [B, 2]
    per trajectory for NoisyPendulum."""
    if not system.keyed:
        return [("none", params, None)]
    shared, per = ojr.PRNGKey(seed), _keys(B, seed)
    return [("shared", params.replace(key=_dev(shared, dev)), shared),
            ("per_trajectory", params.replace(key=_dev(per, dev)), per)]


def _bptt_policy(dev, system, hidden, evaluate, normalize, seed=17, device_stats=False):
    from mbpo_b200.acting import BpttActorPolicy, PolicyParams
    X, A = system.x_dim, system.u_dim
    pol = orc.make_policy_params(seed=seed, obs_dim=X, action_dim=A, hidden=hidden)
    mean = np.linspace(-0.2, 0.4, X).astype(np.float32) if normalize else None
    std = np.linspace(0.7, 2.5, X).astype(np.float32) if normalize else None
    oparams = orc.BpttActorParams(mlp=pol, init_stddev=0.5, sig_min=1e-6, sig_max=1e2, obs_mean=mean, obs_std=std)
    m, s = (_dev(mean, dev), _dev(std, dev)) if (normalize and device_stats) else (mean, std)
    policy = BpttActorPolicy(PolicyParams(weights=[_dev(w, dev) for w in pol.weights],
                                          biases=[_dev(b, dev) for b in pol.biases]),
                             init_stddev=0.5, sig_min=1e-6, sig_max=1e2, obs_mean=m, obs_std=s, evaluate=evaluate)
    return policy, oparams


def _step_keys(k, shared, B):
    return None if k is None else (np.repeat(k.reshape(1, 2), B, axis=0) if shared else k)


@pytest.mark.parametrize("evaluate", [False, True])
@pytest.mark.parametrize("net", ["64x64_normalized", "64x4_raw", "64_device_stats"])
def test_rollout_policy_vs_oracle(mb, cuda_device, prng_mode, which, evaluate, net):
    """One launch per key form: actions per step against the oracle teacher-forced on the GPU's observations, policy
    key and System keys bit-exact, the System step from the GPU's own observations and actions, the single-state form
    and a launch over a slice of the rows."""
    from mbpo_b200.utils.optimizer_utils import rollout_policy
    dev = cuda_device
    B, H, lo, hi = 203, 15, 37, 170
    hidden, normalize, dstats = {"64x64_normalized": ((64, 64), True, False), "64x4_raw": ((64,) * 4, False, False),
                                 "64_device_stats": ((64,), True, True)}[net]
    system, params, osys, x0 = _system(which, dev, B, 101)
    policy, oparams = _bptt_policy(dev, system, hidden, evaluate, normalize, device_stats=dstats)
    X, A = system.x_dim, system.u_dim
    key = ojr.PRNGKey(9)
    for form, sp, okeys in _key_forms(system, params, B, dev, 31):
        tr = rollout_policy(system, sp, _dev(x0, dev), policy, _dev(key, dev), H)
        assert tr.observation.shape == (B, H, X) and tr.action.shape == (B, H, A) and tr.reward.shape == (B, H)
        g_obs, g_act = tr.observation.cpu().numpy(), tr.action.cpu().numpy()
        want, okey, osk = gbo.system_rollout_policy(osys, oparams, x0, key, H, evaluate, okeys, prng_mode,
                                                    teacher_obs=g_obs)
        assert np.array_equal(tr.extras["policy_state_key"].cpu().numpy(), key if evaluate else okey)
        if okeys is None:
            assert "system_params" not in tr.extras
        else:
            got_k = tr.extras["system_params"].key
            assert tuple(got_k.shape) == okeys.shape and np.array_equal(got_k.cpu().numpy(), osk), form
        np.testing.assert_allclose(g_act, want["action"], rtol=3e-5, atol=3e-6)
        assert float(tr.action.abs().max()) <= 0.999 + 1e-7
        # System.step from the GPU's own observations and actions
        k = None if okeys is None else np.asarray(okeys).reshape(-1, 2)
        for t in range(H):
            nxt, r, kk = osys.step(g_obs[:, t], g_act[:, t], _step_keys(k, form == "shared", B), prng_mode)
            k = None if kk is None else (kk[:1] if form == "shared" else kk)
            if system.keyed:
                np.testing.assert_allclose(tr.next_observation[:, t].cpu().numpy(), nxt, rtol=1e-5, atol=2e-6)
                np.testing.assert_allclose(tr.reward[:, t].cpu().numpy(), r, rtol=1e-5, atol=3e-6)
            else:
                assert np.array_equal(tr.next_observation[:, t].cpu().numpy(), nxt), t
                assert np.array_equal(tr.reward[:, t].cpu().numpy(), r), t
        assert np.array_equal(g_obs[:, 0], x0) and np.array_equal(g_obs[:, 1:], tr.next_observation.cpu().numpy()[:, :-1])
        assert bool((tr.discount == 1).all())
        # the single init_state form: fields [H, ...], the bits of row 0
        sp1 = sp if form != "per_trajectory" else sp.replace(key=sp.key[:1])
        one = rollout_policy(system, sp1, _dev(x0[0], dev), policy, _dev(key, dev), H)
        assert one.observation.shape == (H, X) and torch.equal(one.action, tr.action[0])
        assert torch.equal(one.reward, tr.reward[0]) and torch.equal(one.next_observation, tr.next_observation[0])
        # rows [lo, hi) alone
        spr = sp if form != "per_trajectory" else sp.replace(key=sp.key[lo:hi])
        part = rollout_policy(system, spr, _dev(x0[lo:hi], dev), policy, _dev(key, dev), H)
        for f in ("observation", "action", "reward", "next_observation"):
            assert torch.equal(getattr(part, f), getattr(tr, f)[lo:hi]), f
        if form == "per_trajectory":
            assert torch.equal(part.extras["system_params"].key, tr.extras["system_params"].key[lo:hi])


def test_shared_system_key_gives_every_trajectory_the_same_noise(mb, cuda_device):
    from mbpo_b200.utils.optimizer_utils import rollout_policy
    dev = cuda_device
    system, params, _, x0 = _system("noisy_pendulum", dev, 1, 5)
    policy, _ = _bptt_policy(dev, system, (64, 64), False, True)
    xs = _dev(np.repeat(x0, 64, axis=0), dev)
    key = _dev(ojr.PRNGKey(2), dev)
    shared = rollout_policy(system, params.replace(key=_dev(ojr.PRNGKey(7), dev)), xs, policy, key, 10)
    assert bool((shared.next_observation == shared.next_observation[:1]).all())
    per = rollout_policy(system, params.replace(key=_dev(_keys(64, 3), dev)), xs, policy, key, 10)
    assert not bool((per.next_observation == per.next_observation[:1]).all())


def test_normal_tanh_policy_is_accepted(mb, cuda_device, prng_mode, which):
    """A NormalTanh Policy draws per trajectory (element e * A + a of normal(key, (E, A))), as in collection."""
    from mbpo_b200 import acting
    from mbpo_b200.utils.optimizer_utils import rollout_policy
    dev = cuda_device
    B, H = 150, 9
    system, params, osys, x0 = _system(which, dev, B, 7)
    pol = orc.make_policy_params(seed=5, obs_dim=system.x_dim, action_dim=system.u_dim, hidden=(64, 64))
    policy = acting.Policy(acting.PolicyParams([_dev(w, dev) for w in pol.weights], [_dev(b, dev) for b in pol.biases]))
    keys = _keys(B, 8) if system.keyed else None
    sp = params if keys is None else params.replace(key=_dev(keys, dev))
    key = ojr.PRNGKey(4)
    tr = rollout_policy(system, sp, _dev(x0, dev), policy, _dev(key, dev), H)
    want, wk = gco.system_actor_rollout(osys, pol, x0, key, H, 1 << 30, key_convention="unroll",
                                        partitionable=prng_mode, teacher_obs=tr.observation.transpose(0, 1).cpu().numpy(),
                                        keys=keys)
    np.testing.assert_allclose(tr.action.transpose(0, 1).cpu().numpy(), want["action"], rtol=2e-5, atol=2e-6)
    assert np.array_equal(tr.extras["policy_state_key"].cpu().numpy(), wk)
    if keys is not None:
        assert np.array_equal(tr.extras["system_params"].key.cpu().numpy(), want["final_keys"])


def test_rollout_policy_vjp_vs_oracle(mb, cuda_device, which):
    """The reverse scan through the general System.step against the oracle's cotangent pass in float64 on the same
    float32 trajectory, for both layouts (which agree bit for bit) and several None-cotangent combinations."""
    from mbpo_b200.utils.optimizer_utils import Transition, rollout_policy, rollout_policy_vjp
    dev = cuda_device
    B, H = 300, 20
    system, params, osys, x0 = _system(which, dev, B, 111)
    sp = _key_forms(system, params, B, dev, 3)[-1][1]
    policy, _ = _bptt_policy(dev, system, (64, 64), False, True)
    tr = rollout_policy(system, sp, _dev(x0, dev), policy, _dev(ojr.PRNGKey(3), dev), H)
    X, A = system.x_dim, system.u_dim
    rng = np.random.default_rng(112)
    cots = [rng.standard_normal(s).astype(np.float32) for s in ((B, H), (B, H, X), (B, H, X), (B, H, A))]
    obs, act = tr.observation.cpu().numpy(), tr.action.cpu().numpy()
    for use in [(True, True, True, True), (True, False, False, False), (False, True, False, True),
                (False, False, True, False)]:
        args = [c if u else None for c, u in zip(cots, use)]
        want_a, want_x0 = gbo.system_rollout_policy_vjp(osys, obs, act, *args, dtype=np.float64)
        dargs = [None if c is None else _dev(c, dev) for c in args]
        got_a, got_x0 = rollout_policy_vjp(system, sp, tr, *dargs)                          # time-major strided views
        dense = Transition(*(f.contiguous() for f in tr[:5]))
        got_a2, got_x02 = rollout_policy_vjp(system, sp, dense, *dargs)                     # the reference's [B, H, ...]
        assert got_a.shape == (B, H, A) and got_x0.shape == (B, X)
        assert torch.equal(got_a, got_a2) and torch.equal(got_x0, got_x02)
        scale = np.abs(want_a).max(axis=(1, 2), keepdims=True) + 1e-3                       # adjoints grow along the horizon
        assert float(np.abs((got_a.cpu().numpy() - want_a) / scale).max()) < 2e-4
        scale0 = np.abs(want_x0).max(axis=1, keepdims=True) + 1e-3
        assert float(np.abs((got_x0.cpu().numpy() - want_x0) / scale0).max()) < 2e-4


def test_bptt_actor_gradient_matches_autograd(mb, cuda_device, which):
    """End to end: forward kernel -> lambda_return and its transpose -> adjoint kernel -> one batched backward of the
    actor equals torch autograd through the whole float64 rollout (policy on detached observations; NoisyPendulum's
    noise, with one System key shared by the batch, enters as constants from the oracle's key chain)."""
    from mbpo_b200.utils.optimizer_utils import lambda_return, lambda_return_vjp, rollout_policy, rollout_policy_vjp
    dev = cuda_device
    B, H, disc, lam = 64, 12, 0.99, 0.95
    system, params, osys, x0 = _system(which, dev, B, 121)
    X, A = system.x_dim, system.u_dim
    skey = ojr.PRNGKey(6)
    sp = params.replace(key=_dev(skey, dev)) if system.keyed else params
    policy, oparams = _bptt_policy(dev, system, (64, 64), False, True, seed=23)
    key = ojr.PRNGKey(4)
    tr = rollout_policy(system, sp, _dev(x0, dev), policy, _dev(key, dev), H)
    rng = np.random.default_rng(122)
    wv = _dev(rng.standard_normal(X).astype(np.float32), dev)                        # a linear "critic" v(x) = wv . x
    pc = torch.cumprod(torch.tensor([1.0] + [disc] * (H - 1), device=dev), 0)
    nv = tr.next_observation @ wv
    g_lv = -(pc / (B * H)).expand(B, H).contiguous()                                # loss = -mean(lambda_return * disc_t)
    lambda_return(tr.reward, nv, disc, lam)
    g_rew, g_nv = lambda_return_vjp(g_lv, disc, lam)
    g_act, _ = rollout_policy_vjp(system, sp, tr, g_reward=g_rew, g_next_observation=g_nv[..., None] * wv)

    ws = [_dev(w, dev).double().requires_grad_(True) for w in oparams.mlp.weights]
    bs = [_dev(b, dev).double().requires_grad_(True) for b in oparams.mlp.biases]
    mean, std = _dev(oparams.obs_mean, dev).double(), _dev(oparams.obs_std, dev).double()
    eps_t, zs, k, kz = [], [], key, skey                                             # the draws the kernels used
    for _ in range(H):
        ks = ojr.split(k, 2)
        eps_t.append(torch.tensor(ojr.normal(ks[0], A), dtype=torch.float64, device=dev))
        k = ks[1]
        kk = ojr.split(kz, 2)
        zs.append(torch.tensor(ojr.normal(kk[1], 3), dtype=torch.float64, device=dev).expand(B, 3))
        kz = kk[0]
    sig_bias = float(orc.inv_softplus(oparams.init_stddev))

    def actor(o, eps):
        h = (o - mean) / std
        for i in range(len(ws)):
            h = h @ ws[i] + bs[i]
            if i < len(ws) - 1:
                h = h * torch.sigmoid(h)
        mu, sg = h[..., :A], h[..., A:]
        sg = torch.clamp(torch.nn.functional.softplus(sg + sig_bias), 1e-6, 1e2)
        return torch.clamp(torch.tanh(mu + eps * sg), -0.999, 0.999)
    # (1) the kernels' gradient: one batched backward over all (obs_t, g_action_t) rows
    eps_all = torch.stack(eps_t).reshape(1, H, A)
    a_re = actor(tr.observation.double().detach(), eps_all)
    np.testing.assert_allclose(a_re.detach().cpu().numpy(), tr.action.cpu().numpy(), rtol=3e-5, atol=3e-6)
    grads_ours = torch.autograd.grad((a_re * g_act.double()).sum(), ws + bs)
    # (2) autograd through the whole rollout
    x = _dev(x0, dev).double()
    rews, nvs = [], []
    for t in range(H):
        a = actor(x.detach(), eps_t[t])
        x, r = gbo.torch_system_step(osys, x, a, zs[t] if system.keyed else None)
        rews.append(r)
        nvs.append(x @ wv.double())
    rews, nvs = torch.stack(rews, 1), torch.stack(nvs, 1)
    inputs = rews + disc * nvs * (1 - lam)
    agg, rets = nvs[:, -1], []
    for t in range(H - 1, -1, -1):
        agg = inputs[:, t] + disc * lam * agg
        rets.append(agg)
    loss = -(torch.stack(rets[::-1], 1) * pc.double()).mean()
    grads_ref = torch.autograd.grad(loss, ws + bs)
    for go, gr in zip(grads_ours, grads_ref):
        denom = float(gr.abs().max()) + 1e-12
        assert float((go - gr).abs().max()) / denom < 2e-3, (float((go - gr).abs().max()), denom)


def test_refusals_and_empty(mb, cuda_device):
    from mbpo_b200 import acting
    from mbpo_b200.utils.optimizer_utils import Transition, rollout_policy, rollout_policy_vjp
    L = mb._lib
    dev = cuda_device
    B, H = 8, 5
    system, params, _, x0 = _system("noisy_pendulum", dev, B, 1)
    sp = params.replace(key=_dev(_keys(B, 2), dev))
    policy, _ = _bptt_policy(dev, system, (64, 64), False, True)
    key = _dev(ojr.PRNGKey(0), dev)
    xs = _dev(x0, dev)
    with pytest.raises(L.MbpoUnsupported):
        rollout_policy(system, sp, xs, policy, key, H, stop_grads=False)
    with pytest.raises(L.MbpoUnsupported):
        rollout_policy(system, sp, xs, lambda o, s: (o, s), key, H)
    for kernel in ("tcgen05", "tcgen05_wide"):
        tc = acting.BpttActorPolicy(acting.PolicyParams(policy.weights, policy.biases))
        tc.struct.kernel = {"tcgen05": L.ACTOR_TCGEN05, "tcgen05_wide": L.ACTOR_TCGEN05_WIDE}[kernel]
        with pytest.raises(L.MbpoUnsupported):
            rollout_policy(system, sp, xs, tc, key, H)
    # a keyed System without a key, or with a key count that is neither 1 (shared) nor B
    for bad in (None, _dev(_keys(3, 4), dev)):
        with pytest.raises(ValueError):
            rollout_policy(system, params.replace(key=bad), xs, policy, key, H)
    # the pendulum keeps its own entry points
    g = system.pack_params(sp)
    f = torch.zeros(B * 4 * H, device=dev)
    rc = L.lib.mbpo_rollout_policy_general(L.SYSTEM_PENDULUM, L.C.byref(g), 0, L.C.byref(policy.struct), 0,
                                           L.KEYS_UNROLL, L.ptr(key), None, 0, L.ptr(f), B, H, L.ptr(f), L.ptr(f),
                                           L.ptr(f), None, None, None)
    assert rc == L.MBPO_EINVAL and b"mbpo_actor_rollout" in L.lib.mbpo_last_error()
    rc = L.lib.mbpo_rollout_adjoint_general(L.SYSTEM_PENDULUM, L.C.byref(g), B, H, 1, H, 3, 3 * H, 1, H, L.ptr(f),
                                            L.ptr(f), None, None, None, None, L.ptr(f), None, None)
    assert rc == L.MBPO_EINVAL and b"mbpo_rollout_adjoint" in L.lib.mbpo_last_error()
    # no trajectories, no steps: the keys pass through
    for xe, h in ((xs[:0], H), (xs, 0)):
        spe = sp.replace(key=sp.key[:xe.shape[0]])
        tr = rollout_policy(system, spe, xe, policy, key, h)
        assert tr.action.shape == (xe.shape[0], h, 1) and tr.reward.shape == (xe.shape[0], h)
        assert torch.equal(tr.extras["policy_state_key"], key)
        assert torch.equal(tr.extras["system_params"].key, spe.key)
        g_a, g_x0 = rollout_policy_vjp(system, spe, Transition(*(f.contiguous() for f in tr[:5])))
        assert g_a.shape == (xe.shape[0], h, 1) and g_x0.shape == (xe.shape[0], 3)
    shared = rollout_policy(system, params.replace(key=_dev(ojr.PRNGKey(5), dev)), xs, policy, key, 0)
    assert np.array_equal(shared.extras["system_params"].key.cpu().numpy(), ojr.PRNGKey(5))
