"""The oracle of SAC / PPO collection over any oracle System (test infrastructure, beside oracle/mbpo_oracle.py,
which it reuses unchanged): the wrapper stack of ``env_rollout`` and the policy of ``actor_rollout`` with
``system.step(x, u, keys)`` (``PendulumOracle`` / ``NoisyPendulumOracle`` / ``PointMassOracle``) in place of
``pendulum_step``.  What a keyed System adds (brax_wrapper.py:40-50, training.py:91-137): every System.step advances
system_params.key once (key, sub = split(key)), so it advances action_repeat times per env step, and AutoReset resets
obs but NOT system_params -- the key keeps advancing across episode boundaries."""
from __future__ import annotations

from typing import Optional

import numpy as np

from oracle import jax_prng as jr
from oracle.mbpo_oracle import F32, U32, PolicyParams, policy_sample


def system_env_rollout(system, x0: np.ndarray, actions: np.ndarray, episode_length: int, action_repeat: int = 1,
                       steps0: Optional[np.ndarray] = None, done0: Optional[np.ndarray] = None,
                       first_obs: Optional[np.ndarray] = None, keys: Optional[np.ndarray] = None,
                       partitionable: bool = False, dtype=F32):
    """x0 [E,X], actions [T,E,A], keys uint32 [E,2] (keyed Systems) -> dict of Transition fields, time-major, plus
    final_obs / final_steps / final_done / final_keys.  Steps (1)-(5) of env_rollout."""
    actions = np.asarray(actions, dtype=dtype)
    t_len, e, _ = actions.shape
    X = system.x_dim
    obs = np.asarray(x0, dtype=dtype).reshape(e, X).copy()
    first = obs.copy() if first_obs is None else np.asarray(first_obs, dtype=dtype)
    steps = np.zeros(e, dtype=dtype) if steps0 is None else np.asarray(steps0, dtype=dtype).copy()
    done = np.zeros(e, dtype=dtype) if done0 is None else np.asarray(done0, dtype=dtype).copy()
    k = None if keys is None else np.asarray(keys, U32).reshape(e, 2).copy()
    out = dict(observation=np.empty((t_len, e, X), dtype), action=actions.copy(),
               reward=np.empty((t_len, e), dtype), discount=np.empty((t_len, e), dtype),
               next_observation=np.empty((t_len, e, X), dtype), truncation=np.empty((t_len, e), dtype))
    for t in range(t_len):
        steps = np.where(done != 0, dtype(0), steps)
        done = np.zeros(e, dtype=dtype)                               # a System's own done is 0.0
        prev = obs
        rew = np.zeros(e, dtype=dtype)
        x = obs
        for _ in range(action_repeat):
            x, r, k = system.step(x, actions[t], k, partitionable, dtype)
            rew = (rew + r).astype(dtype)
        steps = (steps + dtype(action_repeat)).astype(dtype)
        over = steps >= dtype(episode_length)
        trunc = np.where(over, dtype(1) - done, dtype(0)).astype(dtype)
        done = np.where(over, dtype(1), done).astype(dtype)
        obs = np.where(done[:, None] != 0, first, x).astype(dtype)
        out["observation"][t] = prev
        out["reward"][t] = rew
        out["discount"][t] = dtype(1) - done
        out["next_observation"][t] = obs
        out["truncation"][t] = trunc
    out["final_obs"] = obs
    out["final_steps"] = steps
    out["final_done"] = done
    out["final_keys"] = k
    return out


def system_actor_rollout(system, params: PolicyParams, x0: np.ndarray, key, num_steps: int, episode_length: int,
                         key_convention: str = "sac", deterministic: bool = False, action_repeat: int = 1,
                         partitionable: bool = False, teacher_obs: Optional[np.ndarray] = None,
                         keys: Optional[np.ndarray] = None, obs_mean=None, obs_std=None, with_extras: bool = False,
                         steps0: Optional[np.ndarray] = None, done0: Optional[np.ndarray] = None,
                         first_obs: Optional[np.ndarray] = None):
    """actor_rollout over any oracle System: the policy sees obs [E,X] and acts in A = system.u_dim dims (its draw is
    normal(key, (E, A)): env e, dim a reads element e * A + a).  keys: the envs' system_params.key [E,2].
    with_extras adds PPO's raw_action [T,E,A] and log_prob [T,E].  Returns (Transition dict with final_obs /
    final_steps / final_done / final_keys, carry key)."""
    e, X, A = x0.shape[0], system.x_dim, system.u_dim
    obs = np.asarray(x0, dtype=F32).copy()
    first = obs.copy() if first_obs is None else np.asarray(first_obs, F32)
    steps = np.zeros(e, F32) if steps0 is None else np.asarray(steps0, F32).copy()
    done = np.zeros(e, F32) if done0 is None else np.asarray(done0, F32).copy()
    k = None if keys is None else np.asarray(keys, U32).copy()
    out = dict(observation=np.empty((num_steps, e, X), F32), action=np.empty((num_steps, e, A), F32),
               reward=np.empty((num_steps, e), F32), discount=np.empty((num_steps, e), F32),
               next_observation=np.empty((num_steps, e, X), F32), truncation=np.empty((num_steps, e), F32))
    with_extras = with_extras and not deterministic                   # the reference returns {} there
    if with_extras:
        out["raw_action"] = np.empty((num_steps, e, A), F32)
        out["log_prob"] = np.empty((num_steps, e), F32)
    key = np.asarray(key, dtype=U32)
    for t in range(num_steps):
        if key_convention == "as_is":
            k_actor = key
        else:
            ks = jr.split(key, 2, partitionable)
            if key_convention == "sac":
                key, k_actor = ks[0], ks[1]
            else:
                k_actor, key = ks[0], ks[1]
        if teacher_obs is not None:
            obs = np.asarray(teacher_obs[t], dtype=F32)
        if with_extras:
            act, raw, logp = policy_sample(params, obs, k_actor, deterministic, partitionable, obs_mean, obs_std, True)
            out["raw_action"][t], out["log_prob"][t] = raw, logp
        else:
            act = policy_sample(params, obs, k_actor, deterministic, partitionable, obs_mean, obs_std)
        one = system_env_rollout(system, obs, act[None], episode_length, action_repeat, steps0=steps, done0=done,
                                 first_obs=first, keys=k, partitionable=partitionable)
        out["observation"][t] = obs
        out["action"][t] = act
        for f in ("reward", "discount", "next_observation", "truncation"):
            out[f][t] = one[f][0]
        obs = one["next_observation"][0]
        steps, done, k = one["final_steps"], one["final_done"], one["final_keys"]
    out["final_obs"], out["final_steps"], out["final_done"], out["final_keys"] = obs, steps, done, k
    return out, key
