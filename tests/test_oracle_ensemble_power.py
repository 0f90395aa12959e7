"""The checks of tests/test_gpu_ensemble_power.py can fail: for every case of that file, built from the same inputs
and with the oracle's own rollout standing in for the kernel's states, a kernel with any one defect of
ensemble_power.DEFECTS that can show in the case fails its check.  Also the claims the weight families make."""
import numpy as np
import pytest

from oracle import mbpo_oracle as orc

import ensemble_power as ep

FAMILY = pytest.mark.parametrize("family", ep.FAMILIES)
MEMBERS = pytest.mark.parametrize("E", ep.MEMBER_COUNTS)


def _fails_for_every_defect(kind, bar_kind, family, E, obs, acts, member, case=None):
    """Teacher-forced from obs [T, n, 3] with acts [T or T + 1, n]: the oracle passes its own check, and every defect
    that applies to the case fails it."""
    bar = ep.BARS[(bar_kind, family)]
    want, same = ep.teacher_forced(family, E, obs, acts, member)
    assert ep.passes(same, want, bar)[0]
    checked = 0
    for d in ep.STEP_DEFECTS:
        if not ep.applies(d, kind, E, family, case):
            continue
        _, got = ep.teacher_forced(family, E, obs, acts, member, d)
        ok, s = ep.passes(got, want, bar)
        assert not ok, (d, s, bar)
        checked += 1
    assert checked >= 2


def _free_run(family, E, x0, acts, member):
    """The oracle's rollout: x0 [n, 3], acts [T, n], member [n] -> states [T + 1, n, 3]."""
    xs = [x0]
    for t in range(acts.shape[0]):
        xs.append(ep.step(family, E, xs[-1], acts[t], member))
    return np.stack(xs)


def _rollout_items(name, B, M, H, n, seed, E):
    """The checked (row, member) items of a Transition case, ordered as the GPU test orders them."""
    x0, acts, rows = ep.rollout_inputs(name, B, M, H, n, seed)
    u = acts.reshape(B * M, H)[rows]
    x = np.repeat(x0[rows // M], E, axis=0)
    acts_t = np.repeat(u, E, axis=0).T.copy()                  # [H, n * E]
    member = np.tile(np.arange(E, dtype=np.int32), len(rows))
    return x, acts_t, member


@pytest.mark.parametrize("case", [c[0] for c in ep.rollout_cases()])
@MEMBERS
@FAMILY
def test_transition_checks_fail_on_defects(family, E, case):
    idx = [c[0] for c in ep.rollout_cases()].index(case)
    name, B, M, H, n = ep.rollout_cases()[idx]
    x, acts_t, member = _rollout_items(name, B, M, H, n, 1000 + idx, E)
    states = _free_run(family, E, x, acts_t[:H - 1], member)          # [H, items, 3]
    _fails_for_every_defect("rollout", "fused", family, E, states[:-1], acts_t, member, case)


@MEMBERS
def test_summary_check_fails_on_mean_over_5(E):
    """The summary is compared bit for bit; a member mean divided by 5 shows at every E but 5."""
    name, B, M, H, n = ep.rollout_cases()[0]
    x, acts_t, member = _rollout_items(name, B, M, H, n, 1000, E)
    states = _free_run("seed3", E, x, acts_t[:H - 1], member)
    _, r = orc.pendulum_step(states.reshape(-1, 3), acts_t.reshape(-1), orc.PendulumParams())
    reward = r.reshape(H, -1, E).transpose(1, 2, 0)                   # [rows, E, H]
    right = ep.summary(reward, False)
    assert np.array_equal(ep.summary(reward, False, divisor=E), right)
    assert ep.applies("mean_over_5", "summary", E) == (not np.array_equal(ep.summary(reward, False, 5), right))


@pytest.mark.parametrize("layout,n_envs,T", ep.ENV_CASES)
@MEMBERS
@FAMILY
def test_env_checks_fail_on_defects(family, E, layout, n_envs, T):
    x0, acts, member, rows = ep.env_inputs(layout, n_envs, T, E)
    states = _free_run(family, E, x0[rows], acts[:, rows, 0], member[rows])
    _fails_for_every_defect("env", "fused", family, E, states[:-1], acts[:, rows, 0], member[rows])


@MEMBERS
@FAMILY
def test_step_checks_fail_on_defects(family, E):
    x, u, member = ep.step_inputs(E)
    _fails_for_every_defect("forward", "forward", family, E, x[None], u.T, member)


def test_every_defect_is_seen_by_the_saturated_family():
    for d in ep.STEP_DEFECTS:
        for kind in ("rollout", "env", "forward"):
            assert ep.applies(d, kind, 8, "saturated", "config4") == (kind != "forward" or d != "action_shifted")


def test_env_layouts():
    for E in ep.MEMBER_COUNTS:
        assert np.array_equal(np.unique(ep.env_members("interleaved", 600, E)), np.arange(E))
        assert np.array_equal(np.unique(ep.env_members("last", 600, E)), [E - 1])
        gaps = np.unique(ep.env_members("gaps", 600, E))
        assert np.array_equal(gaps, np.arange(0, E, 2)) and (E == 1 or len(gaps) < E)


def test_rollout_cases_straddle_the_kernel_switch():
    for sms in (ep.B200_SMS, 132, 160):
        kernels = {name: ep.rollout_kernel(B, M, sms) for name, B, M, _, _ in ep.rollout_cases(sms)}
        assert kernels == {"one_tile": "ensemble_transitions_kernel", "one_tile_edge": "ensemble_transitions_kernel",
                           "two_tile_edge": "ensemble_transitions_pp_kernel",
                           "config4": "ensemble_transitions_pp_kernel"}


@MEMBERS
def test_saturated_family_is_saturated_on_its_inputs(E):
    """Every hidden pre-activation of the saturated family is beyond SATURATION_MIN on the pendulum's states and
    actions in [-2, 2], and the network is then exactly piecewise linear in the oracle: swish(v) = max(v, 0) to the
    last bit of float32 for the live units."""
    x, u, member = ep.step_inputs(E, R=4000)
    inp = np.concatenate([x, u], -1)
    ep.assert_saturated(ep.ensemble("saturated", E), inp, member)
    v = np.array([20.0, 26.5, 34.0, 1e3], np.float32)
    assert np.array_equal(orc.swish(v).astype(np.float32), v)
    assert np.all(np.abs(orc.swish(-v)) < 1e-7)
