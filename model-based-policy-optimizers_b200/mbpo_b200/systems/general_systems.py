"""Systems beyond the reference's deterministic pendulum, for the parts of iCemTO it leaves unexercised
(SURVEY 8f-3; csrc/systems.cuh):

* ``NoisyPendulumSystem(noise_std)`` -- a System that CONSUMES ``system_params.key``.  ``PendulumDynamics.next_state``
  already returns ``distrax.Normal(mean, std)`` (pendulum_dynamics.py:45-46) with ``std = 0``; here ``std = noise_std``
  and ``step`` samples it: ``key, sub = split(system_params.key)``; ``x_next = mean + noise_std * normal(sub, (3,))``;
  the returned ``SystemParams`` carries ``key`` on.  iCemTO hands every particle its own key
  (icem_optimizer.py:146-147,155-156), so the particles of one candidate are distinct rollouts.
* ``PointMassSystem`` -- two action dimensions (``split(x, action_dim)``, icem_optimizer.py:180): a planar double
  integrator, state ``[px, py, vx, vy]``, action ``[ax, ay]``.

Neither exists in the reference (which ships one System); both run the CUDA kernels behind ``mbpo_system_step_general``
/ ``mbpo_system_objective`` and are restated in the oracle (NoisyPendulumOracle, PointMassOracle).
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from .. import _lib
from ..config import config
from .base_systems import System, SystemParams, SystemState, _Replaceable
from .pendulum_system import PendulumDynamics, PendulumDynamicsParams, PendulumReward, PendulumRewardParams, pack_pendulum


class _GeneralSystem(System):
    """Shared host code: ``step`` and ``rollout`` through the general kernels."""
    keyed = False

    def _general(self, system_params: SystemParams) -> _lib.GeneralSystemParamsC:
        raise NotImplementedError

    def pack_params(self, system_params: SystemParams):
        return self._general(system_params)

    def step(self, x: torch.Tensor, u: torch.Tensor, system_params: SystemParams) -> SystemState:
        """x [..., X], u [..., A] (leading dims = jax.vmap); a keyed System needs system_params.key [..., 2]."""
        X, A = self.x_dim, self.u_dim
        if x.shape[-1] != X or u.shape[-1] != A or x.shape[:-1] != u.shape[:-1]:
            raise ValueError("%s.step expects x[..., %d] and u[..., %d] with equal batch dims" % (type(self).__name__, X, A))
        xc, uc = x.to(torch.float32).contiguous(), u.to(torch.float32).contiguous()
        rows = xc.numel() // X
        x_next = torch.empty_like(xc)
        reward = torch.empty(xc.shape[:-1], dtype=torch.float32, device=xc.device)
        keys = keys_out = None
        if self.keyed:
            if system_params.key is None:
                raise ValueError("%s draws from system_params.key: it must be set" % type(self).__name__)
            keys = system_params.key.contiguous()
            if keys.numel() // 2 != rows:
                raise ValueError("system_params.key holds %d keys for %d rows" % (keys.numel() // 2, rows))
            keys_out = torch.empty_like(keys)
        params = self._general(system_params)
        with _lib.cuda_guard(xc):
            _lib.check(_lib.lib.mbpo_system_step_general(self.system_kind, _lib.C.byref(params), config.prng_mode,
                                                         _lib.ptr(xc), _lib.ptr(uc), _lib.ptr(keys), rows,
                                                         _lib.ptr(x_next), _lib.ptr(reward), _lib.ptr(keys_out),
                                                         _lib.stream_ptr(xc.device)))
        return SystemState(x_next=x_next, reward=reward,
                           system_params=system_params.replace(key=keys_out if self.keyed else None))

    def objective(self, system_params: SystemParams, x0: torch.Tensor, actions: torch.Tensor, keys=None,
                  num_particles: int = 0, use_optimism: bool = False, full: bool = False):
        """vmap(vmap(objective)): x0 [B, X], actions [B, M, H, A], keys [B, M, 2] -> values [B, M]
        (num_particles = 0: one rollout per row with keys[b, m] as the System's key; ``full`` adds the Transition
        buffers observation / reward / next_observation, [B, M, H, X] / [B, M, H] / [B, M, H, X] -- with
        num_particles = P >= 1 they carry the particle axis, [B, M, P, H, X] / [B, M, P, H] / [B, M, P, H, X], particle
        p being the rollout with key split(keys[b, m], P)[p])."""
        B, M, H, A = actions.shape
        dev = x0.device
        values = torch.empty((B, M), dtype=torch.float32, device=dev)
        obs = rew = nxt = None
        if full:
            lead = (B, M, int(num_particles), H) if num_particles else (B, M, H)
            obs = torch.empty(lead + (self.x_dim,), dtype=torch.float32, device=dev)
            rew = torch.empty(lead, dtype=torch.float32, device=dev)
            nxt = torch.empty_like(obs)
        params = self._general(system_params)
        keys = keys.contiguous() if keys is not None else None
        with _lib.cuda_guard(x0):
            _lib.check(_lib.lib.mbpo_system_objective(
                self.system_kind, _lib.C.byref(params), config.prng_mode, H, _lib.ptr(x0.contiguous()),
                _lib.ptr(actions.contiguous()), _lib.ptr(keys), B, M, int(num_particles),
                _lib.SUMMARIZE_MAX if use_optimism else _lib.SUMMARIZE_MEAN, _lib.ptr(values), _lib.ptr(obs),
                _lib.ptr(rew), _lib.ptr(nxt), _lib.stream_ptr(dev)))
        return (values, obs, rew, nxt) if full else values


class NoisyPendulumSystem(_GeneralSystem):
    system_kind = _lib.SYSTEM_NOISY_PENDULUM
    keyed = True

    def __init__(self, noise_std: float = 0.05):
        super().__init__(dynamics=PendulumDynamics(), reward=PendulumReward())
        self.noise_std = float(noise_std)
        self.min_action, self.max_action = -1.0, 1.0

    def _general(self, system_params):
        g = _lib.GeneralSystemParamsC()
        g.pendulum = pack_pendulum(system_params.dynamics_params, system_params.reward_params)
        g.noise_std = self.noise_std
        return g


@dataclass
class PointMassParams(_Replaceable):
    dt: float = 0.1
    max_accel: float = 1.0
    max_speed: float = 2.0
    target_x: float = 1.0
    target_y: float = -0.5
    speed_cost: float = 0.1
    control_cost: float = 0.02


class _PointMassDynamics:
    x_dim, u_dim = 4, 2

    def init_params(self, key):
        return PointMassParams()


class _PointMassReward:
    x_dim, u_dim = 4, 2

    def init_params(self, key):
        return None


class PointMassSystem(_GeneralSystem):
    system_kind = _lib.SYSTEM_POINT_MASS

    def __init__(self):
        super().__init__(dynamics=_PointMassDynamics(), reward=_PointMassReward())
        self.min_action, self.max_action = -1.0, 1.0

    def _general(self, system_params):
        p = system_params.dynamics_params if system_params.dynamics_params is not None else PointMassParams()
        g = _lib.GeneralSystemParamsC()
        g.point_mass = _lib.PointMassParamsC(float(p.dt), float(p.max_accel), float(p.max_speed), float(p.target_x),
                                             float(p.target_y), float(p.speed_cost), float(p.control_cost))
        return g
