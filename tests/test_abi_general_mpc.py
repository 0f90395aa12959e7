"""CPU tests of mbpo_icem_mpc_closed_loop_general's argument checks: every error below is reported before anything
touches a device, so these run without a GPU."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def mb():
    import mbpo_b200
    return mbpo_b200


def _cfg(L, kind, action_dim, x_dim, horizon=20):
    cfg = L.IcemCfgC()
    L.check(L.lib.mbpo_icem_cfg_init(C.byref(cfg), horizon, action_dim, x_dim, 3, 100, 10, 0.5, 0.0, 3, 0.0, 0.3,
                                     -1.0, 1.0, 1, 1e4))
    cfg.system_kind = kind
    return cfg


def _call(L, cfg, B, T=2, sys_keys_in=0x3000, sys_keys_out=0x3800, cluster=1, states=0x4000):
    p = L.GeneralSystemParamsC()
    return L.lib.mbpo_icem_mpc_closed_loop_general(C.byref(cfg), C.byref(p), 0x1000, 0x1100, 0x1200, sys_keys_in, B, T,
                                                   states, 0x5000, 0x6000, 0x7000, 0x7100, sys_keys_out, cluster, None)


def test_mpc_closed_loop_general_argument_errors(mb):
    L = mb._lib
    noisy = _cfg(L, L.SYSTEM_NOISY_PENDULUM, 1, 3)
    point = _cfg(L, L.SYSTEM_POINT_MASS, 2, 4)
    # a System that draws needs its keys
    assert _call(L, noisy, 4, sys_keys_in=None) == L.MBPO_EINVAL
    assert b"sys_keys_in" in L.lib.mbpo_last_error()
    # a System that does not draw takes none; keys out without keys in are refused
    assert _call(L, point, 4, sys_keys_in=None, sys_keys_out=0x3800) == L.MBPO_EINVAL
    # T > 0 needs the per-step outputs
    assert _call(L, point, 4, states=None) == L.MBPO_EINVAL
    # B = 0 is a no-op, whatever the pointers
    assert _call(L, noisy, 0, sys_keys_in=None) == L.MBPO_OK
    # cluster sizes other than -1, 1, 2, 4, 8, 16
    assert _call(L, noisy, 4, cluster=3) == L.MBPO_EINVAL
    assert b"cluster_size" in L.lib.mbpo_last_error()
    # more than 256 candidate rows per CTA (100 + 3 rows fit any size; 600 + 3 do not fit a 2-cluster)
    big = _cfg(L, L.SYSTEM_POINT_MASS, 2, 4)
    big.num_samples = 600
    assert _call(L, big, 4, sys_keys_in=None, sys_keys_out=None, cluster=2) == L.MBPO_EUNSUPPORTED
    # the pendulum keeps its own entry; a System kind without a fused plan is refused
    pend = _cfg(L, L.SYSTEM_PENDULUM, 1, 3)
    assert _call(L, pend, 4) == L.MBPO_EUNSUPPORTED
    mism = _cfg(L, L.SYSTEM_NOISY_PENDULUM, 2, 4)       # action_dim / x_dim do not match the System
    assert _call(L, mism, 4) == L.MBPO_EUNSUPPORTED
