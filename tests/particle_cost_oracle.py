"""The oracle of iCemTO's constraint objective over distinct particles (test infrastructure, beside
oracle/mbpo_oracle.py, which it reuses unchanged).  icem_optimizer.py:144-166 for one candidate:

    transitions = vmap(rollout over particle p)                 # split(key, P)[p], or ensemble member p
    reward      = summarize(mean_t transitions.reward)          # mean over particles, or max if use_optimism
    cost        = summarize_cost(cost_fn(transitions.observation, actions))   # mean, or max if use_pessimism
    value       = reward - lambda_constraint * relu(cost)

Every sum is a left-to-right float32 chain (``particle_mean``), as the CUDA library rounds it.  ``cost_fn`` is the
already vmapped AbstractCost of ``icem_objective``: states [R, H, X], actions [R, H, A] -> [R]."""
from __future__ import annotations

from typing import Optional

import numpy as np

from oracle import jax_prng as jr
from oracle.mbpo_oracle import (F32, ICemParams, ICemState, icem_refit, icem_sample_actions, mlp_ensemble_step,
                                particle_mean, split_keys, system_rollout_actions)


def summarize(per_particle: np.ndarray, use_max: bool, dtype=F32) -> np.ndarray:
    """[..., P] -> [...]: the max, or the left-to-right mean over the particle axis."""
    return per_particle.max(axis=-1) if use_max else particle_mean(per_particle, dtype)


def penalized(ret, cost, lam: float, use_optimism: bool, use_pessimism: bool, dtype=F32) -> np.ndarray:
    """ret [..., P] horizon means, cost [..., P] or None -> summarize(ret) - lam * relu(summarize_cost(cost))."""
    v = summarize(ret, use_optimism, dtype)
    if cost is None:
        return v
    c = summarize(np.asarray(cost, dtype), use_pessimism, dtype)
    return (v - (dtype(lam) * np.maximum(c, dtype(0))).astype(dtype)).astype(dtype)


def _particle_cost(cost_fn, obs, acts, dtype=F32):
    """obs [M, P, H, X], acts [M, H, A] -> cost [M, P] (the actions are the same for every particle)."""
    m, p, h, x = obs.shape
    a = np.broadcast_to(acts[:, None], (m, p) + acts.shape[1:]).reshape(m * p, h, -1)
    return np.asarray(cost_fn(obs.reshape(m * p, h, x), a), dtype).reshape(m, p)


def system_objective_with_cost(system, x0, acts, particle_keys, params: ICemParams, cost_fn=None,
                               use_optimism: bool = False, use_pessimism: bool = False, partitionable: bool = False,
                               dtype=F32):
    """acts [M, H, A], particle_keys [M, 2] -> (values [M], obs [M, P, H, X], reward [M, P, H], next_obs [M, P, H, X],
    cost [M, P] or None).  Particle p is the rollout with key split(particle_keys, P)[p] (:155); a System that draws
    nothing has P copies of its one rollout."""
    acts = np.asarray(acts, dtype)
    m, P = acts.shape[0], params.num_particles
    if system.keyed:
        pk = split_keys(particle_keys, P, partitionable)                       # [M, P, 2]
        outs = [system_rollout_actions(system, x0, acts, pk[:, p], partitionable, dtype, full=True) for p in range(P)]
    else:
        outs = [system_rollout_actions(system, x0, acts, None, partitionable, dtype, full=True)] * P
    ret = np.stack([o[0] for o in outs], axis=1)
    obs, rew, nxt = (np.stack([o[i] for o in outs], axis=1) for i in (1, 2, 3))
    cost = None if cost_fn is None else _particle_cost(cost_fn, obs, acts, dtype)
    values = penalized(ret, cost, params.lambda_constraint, use_optimism, use_pessimism, dtype)
    return values, obs, rew, nxt, cost


def ensemble_objective_with_cost(x0, acts, ens, cost_fn=None, use_optimism: bool = False, use_pessimism: bool = False,
                                 lambda_constraint: float = ICemParams().lambda_constraint, dtype=F32):
    """x0 [B, 3], acts [B, M, H] or [B, M, H, 1] -> (values [B, M], obs [B, M, E, H, 3], reward [B, M, E, H],
    cost [B, M, E] or None).  Particle e is rolled through member e with the bf16 forward of the tensor-core kernel."""
    x0 = np.asarray(x0, dtype)
    acts = np.asarray(acts, dtype)
    b, m, h = acts.shape[:3]
    E, rows = ens.num_members, b * m
    a = acts.reshape(rows, h)
    obs = np.empty((rows, E, h, 3), dtype)
    rew = np.empty((rows, E, h), dtype)
    ret = np.empty((rows, E), dtype)
    for e in range(E):
        x = np.repeat(x0, m, axis=0).copy()
        member = np.full(rows, e, dtype=np.int32)
        acc = np.zeros(rows, dtype)
        for t in range(h):
            obs[:, e, t] = x
            x, r = mlp_ensemble_step(x, a[:, t], member, ens, bf16=True)
            rew[:, e, t] = r
            acc = (acc + r).astype(dtype)
        ret[:, e] = (acc / dtype(h)).astype(dtype)
    cost = None if cost_fn is None else _particle_cost(cost_fn, obs, a[:, :, None], dtype)
    values = penalized(ret, cost, lambda_constraint, use_optimism, use_pessimism, dtype)
    out_cost = None if cost is None else cost.reshape(b, m, E)
    return values.reshape(b, m), obs.reshape(b, m, E, h, 3), rew.reshape(b, m, E, h), out_cost


def system_icem_optimize_with_cost(system, x0, state: ICemState, params: ICemParams, horizon: int, cost_fn=None,
                                   use_optimism: bool = False, use_pessimism: bool = False,
                                   partitionable: bool = False, dtype=F32, trace: Optional[list] = None) -> ICemState:
    """iCemTO.optimize (icem_optimizer.py:134-252) for one problem of any oracle System, with the constraint cost."""
    A = system.u_dim
    mean = np.zeros((horizon, A), dtype)
    if params.warm_start:
        mean[:-1] = state.best_sequence[1:]
        mean[-1] = state.best_sequence[-1]
    std = np.full((horizon, A), params.init_std, dtype)
    best_seq, best_value = mean.copy(), dtype(-np.inf)
    ks = jr.split(state.key, 2, partitionable)
    carry_key, new_state_key = ks[0], ks[1]
    for _ in range(params.num_steps):
        carry_key, acts, pkeys = icem_sample_actions(carry_key, mean, std, params, horizon, A, partitionable, dtype)
        values = system_objective_with_cost(system, x0, acts, pkeys, params, cost_fn, use_optimism, use_pessimism,
                                            partitionable, dtype)[0]
        mean, std, best_value, best_seq, idx = icem_refit(acts, values, mean, std, best_value, best_seq, params, dtype)
        if trace is not None:
            trace.append(dict(actions=acts, values=values, elite_idx=idx, mean=mean, std=std, best_value=best_value,
                              particle_keys=pkeys))
    return ICemState(key=new_state_key, best_sequence=np.asarray(best_seq, F32), best_reward=F32(best_value))
