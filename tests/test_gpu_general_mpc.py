"""Thread-block-cluster plans and the one-launch closed loop over the general Systems (NoisyPendulumSystem, which
draws from its key, and the two-action PointMassSystem).

* A plan spread over a cluster of C CTAs gives the one-CTA kernel's bits: every trace array, best_seq, best_value and
  the key, for every C.
* iCemTO.closed_loop runs one launch (mbpo_icem_mpc_closed_loop_general) and gives the bits of the loop of staged
  plans and System.step launches, the final System key included.
* A short closed loop against the oracle composed from icem_sample_actions / system_objective / icem_refit and the
  oracle System's step."""
import numpy as np
import pytest
import torch

from oracle import jax_prng as ojr
from oracle import mbpo_oracle as orc

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


def _keys(n, seed=0):
    return np.random.default_rng(seed).integers(0, 2 ** 32, size=(n, 2), dtype=np.uint64).astype(np.uint32)


def _dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _systems(kind):
    from mbpo_b200.systems import NoisyPendulumSystem, PointMassSystem
    if kind == "noisy_pendulum":
        return NoisyPendulumSystem(0.05), orc.NoisyPendulumOracle(0.05)
    return PointMassSystem(), orc.PointMassOracle()


def _states(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "noisy_pendulum":
        th, w = rng.uniform(-np.pi, np.pi, n), rng.uniform(-8, 8, n)
        return np.stack([np.cos(th), np.sin(th), w], axis=-1).astype(np.float32)
    return rng.uniform(-1.5, 1.5, (n, 4)).astype(np.float32)


def _optimizer(kind, H, use_optimism=False, **params):
    from mbpo_b200.optimizers import iCemTO, iCemParams
    system, osys = _systems(kind)
    opt = iCemTO(horizon=H, action_dim=system.u_dim, opt_params=iCemParams(**params), use_optimism=use_optimism)
    opt.set_system(system)
    return opt, system, osys


def _rows_per_cta(opt, cluster):
    cfg = opt._cfg()
    return -(-(cfg.num_samples + cfg.num_prev_elites) // cluster)


PLAN_CASES = [
    # kind, H, N, P, optimism, B
    ("noisy_pendulum", 20, 100, 1, False, 1),
    ("noisy_pendulum", 30, 77, 3, True, 3),
    ("noisy_pendulum", 8, 200, 10, False, 17),
    ("noisy_pendulum", 30, 512, 10, True, 1),
    ("noisy_pendulum", 20, 150, 10, True, 3),
    ("point_mass", 20, 100, 3, False, 3),
    ("point_mass", 30, 150, 1, True, 17),
    ("point_mass", 15, 512, 3, False, 1),
]


@pytest.mark.parametrize("kind,H,N,P,optimism,B", PLAN_CASES)
def test_general_cluster_plan_bit_identical(mb, cuda_device, prng_mode, kind, H, N, P, optimism, B):
    """Cluster sizes 2, 4, 8, 16 and the library's choice against one CTA per problem: all six trace arrays,
    best_seq, best_value and the key, bit for bit; sizes beyond 256 rows per CTA raise MbpoUnsupported."""
    opt, system, _ = _optimizer(kind, H, optimism, num_samples=N, num_elites=max(N // 10, 4), num_particles=P,
                                num_steps=3, alpha=0.1, exponent=1.0)
    st = opt.init(_dev(_keys(B, 91 + B), cuda_device))
    x0 = _dev(_states(kind, B, 92 + N), cuda_device)
    seq0 = torch.randn(st.best_sequence.shape, generator=torch.Generator().manual_seed(3)).to(cuda_device)
    ref = opt._plan_raw(x0, st.key, seq0, st.system_params, trace=True, cluster=1)
    for cluster in (2, 4, 8, 16, -1):
        if cluster > 0 and _rows_per_cta(opt, cluster) > 256:
            with pytest.raises(mb.MbpoUnsupported):
                opt._plan_raw(x0, st.key, seq0, st.system_params, trace=True, cluster=cluster)
            continue
        got = opt._plan_raw(x0, st.key, seq0, st.system_params, trace=True, cluster=cluster)
        assert torch.equal(got[0], ref[0]), cluster
        assert torch.equal(got[1].view(torch.int32), ref[1].view(torch.int32)), cluster
        assert torch.equal(got[2].view(torch.int32), ref[2].view(torch.int32)), cluster
        for name in ("actions", "values", "elite_idx", "mean", "std", "best_value"):
            assert torch.equal(got[3][name], ref[3][name]), (cluster, name)
    # the library picks a cluster for few problems
    if B == 1 and N >= 100:
        chosen = mb._lib.lib.mbpo_icem_plan_cluster_size(mb._lib.C.byref(opt._cfg()), 1)
        assert chosen > 1
        assert mb._lib.lib.mbpo_icem_plan_cluster_capacity(mb._lib.C.byref(opt._cfg()), chosen) >= 1


def test_general_cluster_plan_small_population_unsupported(mb, cuda_device):
    opt, system, _ = _optimizer("point_mass", 20, num_samples=24, num_elites=4, num_particles=1, num_steps=2)
    st = opt.init(_dev(_keys(2, 5), cuda_device))
    x0 = _dev(_states("point_mass", 2, 6), cuda_device)
    with pytest.raises(mb.MbpoUnsupported):
        opt._plan_raw(x0, st.key, st.best_sequence, st.system_params, cluster=2)
    opt._plan_raw(x0, st.key, st.best_sequence, st.system_params, cluster=-1)   # the library's choice: one CTA


def _staged_loop(opt, x0, key, seq, sp, T):
    """plan (per-stage kernels) -> System.step -> warm start, T times; the System key threads through."""
    states, rewards, actions = [], [], []
    for _ in range(T):
        seq, _, key, _ = opt._plan_raw(x0, key, seq, sp, staged=True)
        u = seq[:, 0, :].contiguous()
        nxt = opt.system.step(x0, u, sp)
        if nxt.system_params.key is not None:
            sp = nxt.system_params
        x0 = nxt.x_next
        states.append(x0), rewards.append(nxt.reward), actions.append(u)
    return states, rewards, actions, seq, key, sp


def _raw_closed_loop(mb, opt, sp, x0, key, seq, sys_keys, T, cluster):
    L = mb._lib
    B, X = x0.shape
    H, A = opt.opt_dim
    dev = x0.device
    out = dict(states=torch.empty((T, B, X), dtype=torch.float32, device=dev),
               rewards=torch.empty((T, B), dtype=torch.float32, device=dev),
               actions=torch.empty((T, B, A), dtype=torch.float32, device=dev),
               seq=torch.empty((B, H, A), dtype=torch.float32, device=dev),
               key=torch.empty((B, 2), dtype=torch.uint32, device=dev),
               sys_key=torch.empty((B, 2), dtype=torch.uint32, device=dev) if sys_keys is not None else None)
    params = opt.system.pack_params(sp)
    L.check(L.lib.mbpo_icem_mpc_closed_loop_general(
        L.C.byref(opt._cfg()), L.C.byref(params), L.ptr(x0), L.ptr(key), L.ptr(seq), L.ptr(sys_keys), B, T,
        L.ptr(out["states"]), L.ptr(out["rewards"]), L.ptr(out["actions"]), L.ptr(out["seq"]), L.ptr(out["key"]),
        L.ptr(out["sys_key"]), cluster, L.stream_ptr(dev)))
    torch.cuda.synchronize()
    return out


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("kind", ["noisy_pendulum", "point_mass"])
@pytest.mark.parametrize("B", [1, 5])
@pytest.mark.parametrize("cluster", [1, 2, 4, 8, 16, -1])
def test_general_closed_loop_matches_staged(mb, cuda_device, prng_mode, kind, B, cluster):
    """closed_loop in one launch = the loop of staged plans and System.step launches, bit for bit: states, rewards,
    actions, the final best sequence and planner key, and the System key the last System.step returned."""
    H = 20
    opt, system, _ = _optimizer(kind, H, num_samples=100, num_elites=10, num_particles=3, num_steps=3, alpha=0.1)
    keys = _dev(_keys(B, 700 + B), cuda_device)
    st = opt.init(keys[0] if B == 1 else keys)                       # B = 1: a single problem, key [2]
    x0_np = _states(kind, B, 800 + B)
    x0 = _dev(x0_np[0] if B == 1 else x0_np, cuda_device)
    for T in ((0, 1, 6) if cluster in (1, -1) else (6,)):
        s, r, a, new = opt.closed_loop(x0, st, T, cluster=cluster)
        xs = x0.reshape(-1, system.x_dim)
        s_s, r_s, a_s, seq_s, key_s, sp_s = _staged_loop(opt, xs, st.key.reshape(-1, 2),
                                                       st.best_sequence.reshape(-1, H, system.u_dim),
                                                       st.system_params, T)
        lead = () if B == 1 else (B,)
        assert s.shape == (T,) + lead + (system.x_dim,) and a.shape == (T,) + lead + (system.u_dim,)
        if T:
            assert torch.equal(_bits(s.reshape(T, -1)), _bits(torch.stack(s_s).reshape(T, -1))), T
            assert torch.equal(_bits(r.reshape(T, -1)), _bits(torch.stack(r_s).reshape(T, -1))), T
            assert torch.equal(_bits(a.reshape(T, -1)), _bits(torch.stack(a_s).reshape(T, -1))), T
        assert new.best_sequence.shape == st.best_sequence.shape and new.key.shape == st.key.shape
        assert torch.equal(_bits(new.best_sequence.reshape(-1)), _bits(seq_s.reshape(-1))), T
        assert torch.equal(_bits(new.key.reshape(-1)), _bits(key_s.reshape(-1))), T
        # the library's own staged loop (iCemTO._closed_loop_staged) agrees as well
        single, xc, kc, sc = opt._canon(x0, st)
        s2, r2, a2, new2 = opt._closed_loop_staged(single, xc, kc, sc, st, T)
        assert torch.equal(_bits(s2), _bits(s)) and torch.equal(_bits(a2), _bits(a))
        assert torch.equal(_bits(new2.best_sequence), _bits(new.best_sequence))
        # the final System key, through the C entry
        sys_keys = st.system_params.key.reshape(-1, 2).contiguous() if system.keyed else None
        raw = _raw_closed_loop(mb, opt, st.system_params, xs.contiguous(), st.key.reshape(-1, 2).contiguous(),
                               st.best_sequence.reshape(-1, H, system.u_dim).contiguous(), sys_keys, T, cluster)
        assert torch.equal(_bits(raw["seq"]), _bits(seq_s)) and torch.equal(_bits(raw["key"]), _bits(key_s))
        if system.keyed:
            assert torch.equal(_bits(raw["sys_key"]), _bits(sp_s.key.reshape(-1, 2)))
            if T == 0:
                assert torch.equal(_bits(raw["sys_key"]), _bits(sys_keys))


def test_general_closed_loop_routing(mb, cuda_device, monkeypatch):
    """Without a cost and with scalar bounds closed_loop makes one library launch (never the staged loop); with a
    cost_fn or array-valued bounds it takes the staged loop."""
    from mbpo_b200.optimizers import iCemParams
    from mbpo_b200.optimizers.trajectory_optimizers.icem_optimizer import AbstractCost, iCemTO
    for kind in ("noisy_pendulum", "point_mass"):
        opt, system, _ = _optimizer(kind, 20, num_samples=64, num_elites=8, num_particles=2, num_steps=2)
        st = opt.init(_dev(_keys(3, 31), cuda_device))
        x0 = _dev(_states(kind, 3, 32), cuda_device)

        def boom(*args, **kw):
            raise AssertionError("staged loop")
        with monkeypatch.context() as m:
            m.setattr(iCemTO, "_closed_loop_staged", boom)
            opt.closed_loop(x0, st, 2)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                opt.closed_loop(x0, st, 3)
                torch.cuda.synchronize()
            names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                     and "mpc_general" in e.name]
            assert len(names) == 1, names

        class Cost(AbstractCost):
            def __call__(self, states, actions):
                return states[..., 0].sum() * 0.0

        calls = []
        real = iCemTO._closed_loop_staged

        def spy(self, *args, **kw):
            calls.append(1)
            return real(self, *args, **kw)
        with monkeypatch.context() as m:
            m.setattr(iCemTO, "_closed_loop_staged", spy)
            opt.cost_fn = Cost(20)
            opt.closed_loop(x0, st, 1)
            opt.cost_fn = None
            assert len(calls) == 1
            lo = -torch.ones((20, system.u_dim))
            lo[0] = -0.5
            opt.opt_params = iCemParams(num_samples=64, num_elites=8, num_particles=2, num_steps=2, u_min=lo)
            opt.closed_loop(x0, st, 1)
            assert len(calls) == 2


@pytest.mark.parametrize("kind", ["noisy_pendulum", "point_mass"])
def test_general_closed_loop_against_oracle(mb, cuda_device, prng_mode, kind):
    """A T = 3 closed loop against the oracle's composition (icem_sample_actions -> system_objective -> icem_refit,
    then the oracle System's step): planner and System keys exact, each step's elite indices exact (the plan traced
    on the oracle's own state), states / rewards / actions to the general plan test's tolerances."""
    H, B, T = 20, 2, 3
    params = dict(num_samples=48, num_elites=6, num_particles=3, num_steps=2, alpha=0.1, exponent=1.0)
    opt, system, osys = _optimizer(kind, H, **params)
    A = system.u_dim
    st = opt.init(_dev(_keys(B, 611), cuda_device))
    x0 = _states(kind, B, 612)
    s, r, a, new = opt.closed_loop(_dev(x0, cuda_device), st, T, cluster=2)
    raw = _raw_closed_loop(mb, opt, st.system_params, _dev(x0, cuda_device), st.key.contiguous(), st.best_sequence.contiguous(),
                           st.system_params.key.contiguous() if system.keyed else None, T, 2)
    p = orc.ICemParams(**params)
    pkey = st.key.cpu().numpy()
    skey = st.system_params.key.cpu().numpy().reshape(B, 2) if system.keyed else None
    for b in range(B):
        x = x0[b:b + 1]
        k = pkey[b]
        sk = skey[b:b + 1] if skey is not None else None
        prev = np.zeros((H, A), np.float32)
        for t in range(T):
            _, _, _, tr = opt._plan_raw(_dev(x, cuda_device), _dev(k[None], cuda_device), _dev(prev[None], cuda_device),
                                        st.system_params, trace=True, cluster=2)
            ks = ojr.split(k, 2, prng_mode)
            carry, k = ks[0], ks[1]
            mean = np.concatenate([prev[1:], prev[-1:]]).astype(np.float32)
            std = np.full((H, A), p.init_std, np.float32)
            bval, bseq = np.float32(-np.inf), mean.copy()
            for it in range(p.num_steps):
                carry, acts, pk = orc.icem_sample_actions(carry, mean, std, p, H, A, prng_mode)
                vals = orc.system_objective(osys, x[0], acts, pk, p, False, prng_mode)
                mean, std, bval, bseq, idx = orc.icem_refit(acts, vals, mean, std, bval, bseq, p)
                assert np.array_equal(tr["elite_idx"][it, 0].cpu().numpy(), idx), (b, t, it)
            u = np.asarray(bseq[0:1], np.float32)
            xn, rew, sk = osys.step(x, u, sk, prng_mode)
            np.testing.assert_allclose(a[t, b].cpu().numpy(), u[0], rtol=1e-5, atol=5e-6)
            np.testing.assert_allclose(s[t, b].cpu().numpy(), xn[0], rtol=2e-5, atol=2e-5)
            np.testing.assert_allclose(float(r[t, b]), rew[0], rtol=2e-5, atol=2e-5)
            # the next step starts from the oracle's own state and warm start (teacher-forced)
            x, prev = np.asarray(xn, np.float32), np.asarray(bseq, np.float32)
        assert np.array_equal(new.key[b].cpu().numpy(), k)
        np.testing.assert_allclose(new.best_sequence[b].cpu().numpy(), prev, rtol=1e-5, atol=5e-6)
        if system.keyed:
            assert np.array_equal(raw["sys_key"][b].cpu().numpy(), sk[0])
