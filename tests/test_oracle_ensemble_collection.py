"""CPU tests of the learned ensemble as a collection System (ensemble_collection_oracle.py) and of the argument checks
of mbpo_ensemble_env_rollout, which run before anything touches a GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import mbpo_oracle as orc

import ensemble_collection_oracle as eco
import general_collection_oracle as gco


def _states(rng, e):
    th, w = rng.uniform(-np.pi, np.pi, e), rng.uniform(-8, 8, e)
    return np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)


@pytest.fixture(scope="module")
def ens():
    return orc.make_mlp_ensemble(seed=3, members=5)


def test_adapter_equals_mlp_ensemble_step_row_for_row(ens):
    rng = np.random.default_rng(0)
    E = 23
    x = _states(rng, E)
    u = rng.uniform(-2, 2, (E, 1)).astype(np.float32)
    member = (np.arange(E) * 3 % 5).astype(np.int32)
    xn, r, k = eco.EnsembleOracle(ens, member).step(x, u, None)
    want_x, want_r = orc.mlp_ensemble_step(x, u[:, 0], member, ens, bf16=True)
    assert k is None
    assert np.array_equal(xn, want_x) and np.array_equal(r, want_r)
    for i in range(E):                           # each row is its own member's step
        one_x, one_r = orc.mlp_ensemble_step(x[i:i + 1], u[i:i + 1, 0], member[i:i + 1], ens, bf16=True)
        assert np.array_equal(xn[i], one_x[0]) and r[i] == one_r[0]
    xn0, _, _ = eco.EnsembleOracle(ens, None).step(x, u, None)
    assert np.array_equal(xn0, orc.mlp_ensemble_step(x, u[:, 0], np.zeros(E, np.int32), ens, bf16=True)[0])


@pytest.mark.parametrize("action_repeat", [1, 2])
def test_oracle_rollout_is_invariant_under_env_permutation(ens, action_repeat):
    rng = np.random.default_rng(1)
    E, T, L = 17, 9, 4
    x0 = _states(rng, E)
    acts = rng.uniform(-2, 2, (T, E, 1)).astype(np.float32)
    steps0 = rng.integers(0, L, E).astype(np.float32)
    member = (np.arange(E) % 5).astype(np.int32)
    perm = rng.permutation(E)
    a = gco.system_env_rollout(eco.EnsembleOracle(ens, member), x0, acts, L, action_repeat, steps0=steps0)
    b = gco.system_env_rollout(eco.EnsembleOracle(ens, member[perm]), x0[perm], acts[:, perm], L, action_repeat,
                               steps0=steps0[perm])
    for f in ("observation", "reward", "discount", "next_observation", "truncation"):
        assert np.array_equal(a[f][:, perm], b[f]), f
    for f in ("final_obs", "final_steps", "final_done"):
        assert np.array_equal(a[f][perm], b[f]), f


@pytest.fixture(scope="module")
def L():
    import mbpo_b200
    return mbpo_b200._lib


def _params(L, hidden=256, x_dim=3, u_dim=1, members=5):
    fake = 0x1000   # never dereferenced: every check below fails before a launch
    return L.MlpEnsembleParamsC(members, hidden, x_dim, u_dim, fake, fake, fake, fake, fake, fake, L.PendulumParamsC())


def _policy(L, num_hidden=2):
    s = L.PolicyParamsC()
    s.num_hidden, s.hidden, s.obs_dim, s.action_dim = num_hidden, 64, 3, 1
    for i in range(num_hidden + 1):
        s.w[i] = s.b[i] = 0x1000
    s.head = L.HEAD_NORMAL_TANH
    s.kernel = L.ACTOR_AUTO
    return s


def _call(L, p, policy=None, E=4, T=3, ep=5, rep=1, prng=0, key=0x1000, keyconv=0, obs=0x1000, acts=0x1000,
          order=0x1000, raw=None, logp=None):
    f = 0x1000
    return L.lib.mbpo_ensemble_env_rollout(None if p is None else C.byref(p), prng,
                                           None if policy is None else C.byref(policy), 0, keyconv, key, ep, rep,
                                           order, f, obs, f, f, f, E, T, acts, f, f, f, f, f, f, raw, logp, None)


def test_entry_point_refuses_bad_arguments_without_a_gpu(L):
    p = _params(L)
    assert _call(L, None) == L.MBPO_EINVAL                                # null params
    assert _call(L, p, E=-1) == L.MBPO_EINVAL                             # bad sizes
    assert _call(L, p, T=-1) == L.MBPO_EINVAL
    assert _call(L, p, ep=0) == L.MBPO_EINVAL
    assert _call(L, p, rep=0) == L.MBPO_EINVAL
    assert _call(L, p, prng=2) == L.MBPO_EINVAL
    assert _call(L, p, obs=None) == L.MBPO_EINVAL                         # null env state
    assert _call(L, p, order=None) == L.MBPO_EINVAL                       # null grouping
    assert _call(L, p, acts=None) == L.MBPO_EINVAL                        # actions given, but NULL
    pol = _policy(L)
    assert _call(L, p, pol, key=None) == L.MBPO_EINVAL                   # the policy's carry key
    assert _call(L, p, pol, keyconv=3) == L.MBPO_EINVAL
    assert _call(L, p, pol, raw=0x1000) == L.MBPO_EINVAL                 # raw_action without log_prob
    pol.draw_total, pol.draw_offset = 4, 2                                # envs [2, 6) outside draw_total 4
    assert _call(L, p, pol) == L.MBPO_EINVAL
    for bad in (_params(L, hidden=128), _params(L, x_dim=4), _params(L, u_dim=2), _params(L, members=0)):
        assert _call(L, bad) == L.MBPO_EUNSUPPORTED
    assert "hidden == 256" in L.lib.mbpo_last_error().decode()


def test_entry_point_refusals_name_their_reason(L):
    p = _params(L)
    for num_hidden in (3, 4):                                             # beside the ensemble's 211 KB
        assert _call(L, p, _policy(L, num_hidden)) == L.MBPO_EUNSUPPORTED
        assert "shared memory" in L.lib.mbpo_last_error().decode()
    bptt = _policy(L)
    bptt.head = L.HEAD_BPTT_ACTOR
    bptt.shared_noise = 1
    assert _call(L, p, bptt) == L.MBPO_EUNSUPPORTED
    for k in (L.ACTOR_TCGEN05, L.ACTOR_TCGEN05_WIDE):
        tc = _policy(L)
        tc.kernel = k
        assert _call(L, p, tc) == L.MBPO_EUNSUPPORTED
