"""The oracle of BPTT's rollout over any oracle System (test infrastructure, beside oracle/mbpo_oracle.py, which it
reuses unchanged): ``rollout_policy`` with BPTT's actor (``orc.bptt_act``) and ``system.step(x, u, keys)``
(``PendulumOracle`` / ``NoisyPendulumOracle`` / ``PointMassOracle``) in place of ``pendulum_step``, and the cotangent
pass through it.  rollout_policy is the plain scan of optimizer_utils.py:62-116 -- no Episode / AutoReset wrapper --
and each System.step splits a keyed System's key once.  BPTT vmaps actor_loss over initial states only
(bptt_optimizer.py:366-368), so a System key of shape [2] is shared by every trajectory; [B, 2] gives each its own."""
from __future__ import annotations

from typing import Optional

import numpy as np

from oracle import mbpo_oracle as orc
from oracle.mbpo_oracle import F32, U32


def system_rollout_policy(system, actor: orc.BpttActorParams, x0: np.ndarray, key, H: int, evaluate: bool = False,
                          sys_keys: Optional[np.ndarray] = None, partitionable: bool = False,
                          teacher_obs: Optional[np.ndarray] = None):
    """x0 [B, X] -> (dict of [B, H, ...] fields: observation, action, reward, next_observation, discount; the carried
    policy key; the System key after H steps in the shape it was given: [2], [B, 2] or None).  teacher_obs [B, H, X]
    forces the observation the policy sees and the System steps from at step t."""
    b, X, A = x0.shape[0], system.x_dim, system.u_dim
    obs = np.asarray(x0, dtype=F32).copy()
    out = dict(observation=np.empty((b, H, X), F32), action=np.empty((b, H, A), F32), reward=np.empty((b, H), F32),
               next_observation=np.empty((b, H, X), F32), discount=np.ones((b, H), F32))
    key = np.asarray(key, dtype=U32)
    shared = sys_keys is not None and np.asarray(sys_keys).ndim == 1
    k = None if sys_keys is None else np.asarray(sys_keys, U32).reshape(-1, 2)
    for t in range(H):
        if teacher_obs is not None:
            obs = np.asarray(teacher_obs[:, t], dtype=F32)
        act, key = orc.bptt_act(actor, obs, key, evaluate, partitionable)
        kk = None if k is None else (np.repeat(k, b, axis=0) if shared else k)
        nxt, r, kk = system.step(obs, act, kk, partitionable)
        if k is not None:
            k = kk[:1] if shared else kk
        out["observation"][:, t] = obs
        out["action"][:, t] = act
        out["reward"][:, t] = r
        out["next_observation"][:, t] = nxt
        obs = nxt
    k_out = None if k is None else (k[0] if shared else k)
    return out, key, k_out


def point_mass_step_vjp(system: orc.PointMassOracle, x, u, g_next, g_reward, dtype=F32):
    """Cotangents of one PointMassOracle.step, per axis with pre = v + a dt, a = clip(u, +-1) max_accel:
    g_v' = g_next_v + dt g_next_p; g_pre = g_v' clip'(pre, +-max_speed); g_v = g_pre - g_r 2 speed_cost v;
    g_p = g_next_p - g_r 2 (p - target); g_u = g_pre dt max_accel clip'(u, +-1) - g_r 2 control_cost u."""
    d, p = dtype, system.p
    x, u = np.asarray(x, d), np.asarray(u, d)
    g_next, g_r = np.asarray(g_next, d), np.asarray(g_reward, d)[:, None]
    pos, vel = x[:, 0:2], x[:, 2:4]
    tgt = np.array([p.target_x, p.target_y], d)
    a = (np.clip(u, d(-1), d(1)) * d(p.max_accel)).astype(d)
    pre = (vel + (a * d(p.dt)).astype(d)).astype(d)                   # rounded as step rounds it: same clip ties
    g_pre = (g_next[:, 2:4] + d(p.dt) * g_next[:, 0:2]) * orc._clip_grad(pre, d(-p.max_speed), d(p.max_speed))
    g_p = g_next[:, 0:2] - g_r * d(2.0) * (pos - tgt)
    g_v = g_pre - g_r * d(2.0) * d(p.speed_cost) * vel
    g_u = (g_pre * d(p.dt) * d(p.max_accel) * orc._clip_grad(u, d(-1), d(1))
           - g_r * d(2.0) * d(p.control_cost) * u)
    return np.concatenate([g_p, g_v], axis=1).astype(d), g_u.astype(d)


def system_step_vjp(system, x, u, g_next, g_reward, dtype=F32):
    """Cotangents of one system.step: x [n,X], u [n,A], g_next [n,X], g_reward [n] -> (g_x [n,X], g_u [n,A]).
    NoisyPendulum adds noise that depends on neither x nor u: its Jacobians are the pendulum's at x."""
    if isinstance(system, orc.PointMassOracle):
        return point_mass_step_vjp(system, x, u, g_next, g_reward, dtype)
    g_x, g_u = orc.pendulum_step_vjp(x, np.asarray(u)[:, 0], g_next, g_reward, system.p, dtype)
    return g_x, g_u[:, None]


def system_rollout_policy_vjp(system, observation, action, g_reward=None, g_next_obs=None, g_obs=None,
                              g_action=None, dtype=F32):
    """orc.rollout_policy_vjp for any oracle System: observation [B,H,X], action [B,H,A] and the cotangents of the
    Transition fields (None = 0) -> (g_action_total [B,H,A], g_x0 [B,X])."""
    b, h, X = observation.shape
    A = action.shape[-1]
    z1, zx = np.zeros((b, h), dtype), np.zeros((b, h, X), dtype)
    g_reward = z1 if g_reward is None else np.asarray(g_reward, dtype)
    g_next_obs = zx if g_next_obs is None else np.asarray(g_next_obs, dtype)
    g_obs = zx if g_obs is None else np.asarray(g_obs, dtype)
    g_action = np.zeros((b, h, A), dtype) if g_action is None else np.asarray(g_action, dtype)
    lam = np.zeros((b, X), dtype)
    out = np.empty((b, h, A), dtype)
    for t in range(h - 1, -1, -1):
        g_next = lam + g_next_obs[:, t] + (g_obs[:, t + 1] if t + 1 < h else 0)
        lam, g_u = system_step_vjp(system, observation[:, t], action[:, t], g_next, g_reward[:, t], dtype)
        out[:, t] = g_u + g_action[:, t]
    return out, (lam + (g_obs[:, 0] if h > 0 else 0)).astype(dtype)


def torch_system_step(system, x, a, z=None):
    """system.step restated in float64 torch, for autograd references: x [B, X], a [B, A]; z [B, 3] is
    NoisyPendulum's noise draw, which enters as a constant."""
    import torch
    if isinstance(system, orc.PointMassOracle):
        p = system.p
        tgt = x.new_tensor([p.target_x, p.target_y])
        pos, vel = x[:, :2], x[:, 2:]
        r = -(((pos - tgt) ** 2).sum(-1) + p.speed_cost * (vel ** 2).sum(-1)) - p.control_cost * (a ** 2).sum(-1)
        nv = torch.clamp(vel + torch.clamp(a, -1, 1) * p.max_accel * p.dt, -p.max_speed, p.max_speed)
        return torch.cat([pos + nv * p.dt, nv], -1), r
    p, u = system.p, a[:, 0]
    th = torch.atan2(x[:, 1], x[:, 0])
    d = torch.remainder(th - p.target_angle + np.pi, 2 * np.pi) - np.pi
    r = -(p.angle_cost * d ** 2 + 0.1 * x[:, 2] ** 2) - p.control_cost * u ** 2
    thdd = 3 * p.g / (2 * p.l) * torch.sin(th) + 3.0 / (p.m * p.l ** 2) * torch.clamp(u, -1, 1) * p.max_torque
    nw = torch.clamp(x[:, 2] + thdd * p.dt, -p.max_speed, p.max_speed)
    nth = th + nw * p.dt
    xn = torch.stack([torch.cos(nth), torch.sin(nth), nw], -1)
    return (xn if z is None else xn + system.noise_std * z), r
