"""rollout_actions / rollout_policy / lambda_return behind the reference's signatures.

Mirrors mbpo/utils/optimizer_utils.py:11-59 and returns the same brax-style Transition
fields.  Batched forms replace ``jax.vmap(rollout_actions)``:
    init_state [X],   actions [H, A]        -> fields [H, ...]
    init_state [B,X], actions [B, M, H, A]  -> fields [B, M, H, ...]  (M sequences per state)

rollout_policy (optimizer_utils.py:62-116) runs the policy inside the horizon loop in one kernel launch
(mbpo_actor_rollout; mbpo_rollout_policy_general for NoisyPendulumSystem / PointMassSystem); ``rollout_policy_vjp``
is the cotangent pass jax.grad takes through it with stop_grads=True (mbpo_rollout_adjoint /
mbpo_rollout_adjoint_general), ``lambda_return`` / ``lambda_return_vjp`` the Dreamer lambda return (:119-131) and
its transpose.
"""
from __future__ import annotations

from typing import Any, NamedTuple, Optional, Tuple

import torch

from .. import _lib
from ..config import config
from ..systems.base_systems import System, SystemParams


class Transition(NamedTuple):
    """brax.training.types.Transition."""
    observation: torch.Tensor
    action: torch.Tensor
    reward: torch.Tensor
    discount: torch.Tensor
    next_observation: torch.Tensor
    extras: Any = ()


def rollout_actions(system: System, system_params: SystemParams, init_state: torch.Tensor, actions: torch.Tensor,
                    horizon: int) -> Transition:
    single = init_state.dim() == 1
    if single:
        if actions.dim() != 2:
            raise ValueError("rollout_actions: actions must be [H, A] for a single init_state")
        x0 = init_state.reshape(1, -1)
        acts = actions.reshape(1, 1, *actions.shape)
    else:
        if actions.dim() != 4 or actions.shape[0] != init_state.shape[0]:
            raise ValueError("rollout_actions: batched form needs init_state [B, X] and actions [B, M, H, A]")
        x0, acts = init_state, actions
    assert acts.shape[2] == horizon, "actions.shape[0] must equal horizon"   # optimizer_utils.py:26
    x0 = x0.to(torch.float32).contiguous()
    acts = acts.to(torch.float32).contiguous()
    B, M, H, A = acts.shape
    X = x0.shape[-1]
    dev = x0.device
    obs = torch.empty((B, M, H, X), dtype=torch.float32, device=dev)
    nxt = torch.empty((B, M, H, X), dtype=torch.float32, device=dev)
    rew = torch.empty((B, M, H), dtype=torch.float32, device=dev)
    params = system.pack_params(system_params)
    with _lib.cuda_guard(x0):
        _lib.check(_lib.lib.mbpo_rollout_actions(system.system_kind, _lib.C.addressof(params), config.math_mode_id, H, A,
                                                 X, _lib.ptr(x0), _lib.ptr(acts), B, M, None, _lib.ptr(obs),
                                                 _lib.ptr(rew), _lib.ptr(nxt), _lib.stream_ptr(dev)))
    tr = Transition(observation=obs, action=acts, reward=rew, discount=torch.ones_like(rew), next_observation=nxt)
    if single:
        tr = Transition(*(f[0, 0] for f in tr[:5]))
    return tr


def rollout_returns(system: System, system_params: SystemParams, init_state: torch.Tensor,
                    actions: torch.Tensor) -> torch.Tensor:
    """Horizon-mean reward of each action sequence (icem_optimizer.py:160 inner mean) without
    materialising the Transition: init_state [B,X], actions [B,M,H,A] -> [B,M]."""
    x0 = init_state.to(torch.float32).contiguous()
    acts = actions.to(torch.float32).contiguous()
    B, M, H, A = acts.shape
    out = torch.empty((B, M), dtype=torch.float32, device=x0.device)
    params = system.pack_params(system_params)
    with _lib.cuda_guard(x0):
        _lib.check(_lib.lib.mbpo_rollout_actions(system.system_kind, _lib.C.addressof(params), config.math_mode_id, H, A,
                                                 x0.shape[-1], _lib.ptr(x0), _lib.ptr(acts), B, M, _lib.ptr(out), None,
                                                 None, None, _lib.stream_ptr(x0.device)))
    return out


def rollout_policy(system: System, system_params: SystemParams, init_state: torch.Tensor, policy, policy_state,
                   horizon: int, stop_grads: bool = True) -> Transition:
    """optimizer_utils.py:62-116.  ``policy`` is a mbpo_b200.acting policy object (the kernel runs its network
    inside the horizon loop; an arbitrary Python callable has no CUDA path); ``policy_state`` carries the policy's
    PRNG key: a uint32[2] tensor or any object with a ``.key`` (BPTTState).  init_state [X] -> fields [H, ...];
    init_state [B, X] -> fields [B, H, ...] (vmap over init_state with the policy state shared, as
    bptt_optimizer.py:366-368).  The fields are strided views of time-major buffers.  The carried key is returned
    in ``extras['policy_state_key']``.  stop_grads=False (policy differentiated w.r.t. its observation) is not
    what BPTT uses (:337) and has no kernel.

    NoisyPendulumSystem / PointMassSystem run mbpo_rollout_policy_general.  A keyed System's ``system_params.key``
    is either [2], one key every trajectory steps with (BPTT vmaps over initial states only, so its system_params
    are unbatched and every trajectory sees the same noise), or [B, 2], one per trajectory; the advanced key comes
    back in the same shape in ``extras['system_params']``."""
    from .. import acting
    from ..envs import VmappedSystemEnv, is_general
    if not stop_grads:
        raise _lib.MbpoUnsupported(_lib.MBPO_EUNSUPPORTED, "rollout_policy: only stop_grads=True has a CUDA path")
    if not isinstance(policy, acting.Policy):
        raise _lib.MbpoUnsupported(_lib.MBPO_EUNSUPPORTED,
                                   "rollout_policy: policy must be a mbpo_b200.acting.Policy (no Python callables)")
    single = init_state.dim() == 1
    x0 = init_state.reshape(1, -1) if single else init_state
    key = policy_state.key if hasattr(policy_state, "key") else policy_state
    # act(evaluate=False) splits the key every step (sample_key, key = split(key, 2), :321-323); evaluate leaves it
    convention = _lib.KEYS_AS_IS if policy.deterministic else _lib.KEYS_UNROLL
    if is_general(system):
        fields, extras = _rollout_policy_general(system, system_params, x0, policy, key, int(horizon), convention)
    else:
        env = VmappedSystemEnv(system, system_params, episode_length=1 << 30)  # no Episode / AutoReset wrapper here
        _, tr, key_out = acting._rollout(env, env.reset(x0), policy, key, int(horizon), convention, ())
        fields = (tr.observation, tr.action, tr.reward, tr.discount, tr.next_observation)
        extras = {"policy_state_key": key_out}
    fields = [f.transpose(0, 1) for f in fields]
    if single:
        fields = [f[0] for f in fields]
    return Transition(*fields, extras=extras)


def _rollout_policy_general(system: System, system_params: SystemParams, x0: torch.Tensor, policy, key: torch.Tensor,
                            T: int, convention: int):
    """rollout_policy's launch for a general System: time-major fields [T, E, ...] and the extras."""
    from ..envs import system_keys
    X, A = system.x_dim, system.u_dim
    x0 = x0.to(torch.float32)
    E = x0.shape[0]
    dev = x0.device
    sys_key = None if system_params is None else system_params.key
    shared = bool(system.keyed) and sys_key is not None and sys_key.dim() == 1
    sys_keys = system_keys(system, system_params, 1 if shared else E)
    sys_keys_out = torch.empty_like(sys_keys) if sys_keys is not None else None
    key = key.reshape(2).contiguous()
    key_out = torch.empty_like(key)
    buf = torch.empty((T + 1, E, X), dtype=torch.float32, device=dev)       # observation / next_observation views
    buf[0].copy_(x0)
    act = torch.empty((T, E, A), dtype=torch.float32, device=dev)
    rew = torch.empty((T, E), dtype=torch.float32, device=dev)
    params = system.pack_params(system_params)
    policy.struct.draw_total = policy.struct.draw_offset = 0                 # the launch owns every trajectory
    with _lib.cuda_guard(x0):
        _lib.check(_lib.lib.mbpo_rollout_policy_general(
            system.system_kind, _lib.C.byref(params), config.prng_mode, _lib.C.byref(policy.struct),
            int(policy.deterministic), convention, _lib.ptr(key), _lib.ptr(sys_keys), int(shared), _lib.ptr(buf[0]),
            E, T, _lib.ptr(act), _lib.ptr(rew), _lib.ptr(buf[1:]), _lib.ptr(key_out), _lib.ptr(sys_keys_out),
            _lib.stream_ptr(dev)))
    extras = {"policy_state_key": key_out}
    if sys_keys_out is not None:
        extras["system_params"] = system_params.replace(key=sys_keys_out.reshape(sys_key.shape))
    return (buf[:T], act, rew, torch.ones_like(rew), buf[1:]), extras


def _strides(t: torch.Tensor, per_step_dims: int) -> Tuple[int, int]:
    """(stride_t, stride_e) in elements of a [B, H, ...] tensor whose trailing dims are dense."""
    if t.dim() != 2 + per_step_dims or (per_step_dims and t.stride(-1) != 1):
        raise _lib.MbpoError(_lib.MBPO_EINVAL, "expected a [B, H%s] tensor with a dense last axis" %
                             (", X" if per_step_dims else ""))
    return t.stride(1), t.stride(0)


def rollout_policy_vjp(system: System, system_params: SystemParams, trajectory: Transition,
                       g_reward: Optional[torch.Tensor] = None, g_next_observation: Optional[torch.Tensor] = None,
                       g_observation: Optional[torch.Tensor] = None, g_action: Optional[torch.Tensor] = None):
    """The cotangent pass jax.value_and_grad takes through rollout_policy(..., stop_grads=True)
    (bptt_optimizer.py:361-376).  trajectory: the [B, H, ...] Transition ``rollout_policy`` returned; g_*: the
    cotangents of its fields (None = zero), same shapes.  Returns (g_action_total [B, H, A], g_init_state [B, X]).
    g_action_total[b, t] is what reaches a_t = policy(stop_gradient(obs_t)); the parameter gradient is one
    batched backward of the policy network over all (obs_t, g_action_total_t) rows.  For NoisyPendulumSystem /
    PointMassSystem (mbpo_rollout_adjoint_general) the [B, H, A] arrays have their own stride pair."""
    from ..envs import is_general
    obs, act = trajectory.observation, trajectory.action
    B, H, X = obs.shape
    A = act.shape[-1]
    dev = obs.device

    def like(ref, t):
        """Cotangents are given the layout of the array they belong to (the kernel takes one stride pair)."""
        if t is None:
            return None
        t = t.to(torch.float32)
        if t.stride() != ref.stride():
            buf = torch.empty_strided(ref.shape, ref.stride(), dtype=torch.float32, device=dev)
            buf.copy_(t)
            t = buf
        return t

    def p(t):
        return None if t is None else t.data_ptr()
    params = system.pack_params(system_params)
    if is_general(system):
        act = act.to(torch.float32)
        if act.stride(-1) != 1:
            act = act.contiguous()
        g_act_out = torch.empty_strided(act.shape, act.stride(), dtype=torch.float32, device=dev)
        g_x0 = torch.empty((B, X), dtype=torch.float32, device=dev)
        g_r = like(trajectory.reward, g_reward)
        g_n, g_o = like(obs, g_next_observation), like(obs, g_observation)
        g_a = like(act, g_action)
        st_t, st_e = _strides(trajectory.reward, 0)
        sx_t, sx_e = _strides(obs, 1)
        sa_t, sa_e = _strides(act, 1)
        with _lib.cuda_guard(obs):
            _lib.check(_lib.lib.mbpo_rollout_adjoint_general(
                system.system_kind, _lib.C.byref(params), B, H, st_t, st_e, sx_t, sx_e, sa_t, sa_e, p(obs), p(act),
                p(g_r), p(g_n), p(g_o), p(g_a), p(g_act_out), p(g_x0), _lib.stream_ptr(dev)))
        return g_act_out, g_x0
    rew_like = trajectory.reward
    if act.reshape(B, H).stride() != rew_like.stride():
        rew_like = act.reshape(B, H)
    act2 = like(rew_like, act.reshape(B, H))
    g_r = like(rew_like, g_reward)
    g_a = like(rew_like, None if g_action is None else g_action.reshape(B, H))
    g_n = like(obs, g_next_observation)
    g_o = like(obs, g_observation)
    g_act_out = torch.empty_strided(rew_like.shape, rew_like.stride(), dtype=torch.float32, device=dev)
    g_x0 = torch.empty((B, X), dtype=torch.float32, device=dev)
    st_t, st_e = _strides(rew_like, 0)
    sx_t, sx_e = _strides(obs, 1)
    with _lib.cuda_guard(obs):
        _lib.check(_lib.lib.mbpo_rollout_adjoint(system.system_kind, _lib.C.addressof(params), X, A, B, H, st_t, st_e,
                                                 sx_t, sx_e, p(obs), p(act2), p(g_r), p(g_n), p(g_o), p(g_a),
                                                 p(g_act_out), p(g_x0), _lib.stream_ptr(dev)))
    return g_act_out.reshape(B, H, A), g_x0


def lambda_return(reward: torch.Tensor, next_values: torch.Tensor, discount: float, lambda_: float) -> torch.Tensor:
    """optimizer_utils.py:119-131 (Dreamer's lambda return) along the last axis: [H] or [B, H] (vmapped)."""
    assert reward.dim() == next_values.dim(), (reward.shape, next_values.shape)
    r = reward.to(torch.float32).reshape(-1, reward.shape[-1])
    nv = next_values.to(torch.float32).reshape(-1, reward.shape[-1])
    if nv.stride() != r.stride():
        buf = torch.empty_strided(r.shape, r.stride(), dtype=torch.float32, device=r.device)
        nv = buf.copy_(nv)
    out = torch.empty_strided(r.shape, r.stride(), dtype=torch.float32, device=r.device)
    st_t, st_e = _strides(r, 0)
    with _lib.cuda_guard(r):
        _lib.check(_lib.lib.mbpo_lambda_return(r.data_ptr(), nv.data_ptr(), r.shape[0], r.shape[1], st_t, st_e,
                                               float(discount), float(lambda_), out.data_ptr(),
                                               _lib.stream_ptr(r.device)))
    return out.reshape(reward.shape)


def lambda_return_vjp(g_returns: torch.Tensor, discount: float, lambda_: float):
    """Transpose of ``lambda_return``: cotangents (g_reward, g_next_values) of a cotangent of the returns."""
    g = g_returns.to(torch.float32).reshape(-1, g_returns.shape[-1])
    g_r = torch.empty_strided(g.shape, g.stride(), dtype=torch.float32, device=g.device)
    g_nv = torch.empty_strided(g.shape, g.stride(), dtype=torch.float32, device=g.device)
    st_t, st_e = _strides(g, 0)
    with _lib.cuda_guard(g):
        _lib.check(_lib.lib.mbpo_lambda_return_vjp(g.data_ptr(), g.shape[0], g.shape[1], st_t, st_e, float(discount),
                                                   float(lambda_), g_r.data_ptr(), g_nv.data_ptr(),
                                                   _lib.stream_ptr(g.device)))
    return g_r.reshape(g_returns.shape), g_nv.reshape(g_returns.shape)


def compute_gae(truncation: torch.Tensor, termination: torch.Tensor, rewards: torch.Tensor, values: torch.Tensor,
                bootstrap_value: torch.Tensor, lambda_: float = 1.0, discount: float = 0.99):
    """PPO's generalised advantage estimation (ppo/losses.py:128-184 ``compute_gae``; brax's argument order with
    ``self.gae_lambda`` / ``self.discounting`` as keywords): [T, B] inputs (time-major, as the loss makes them at
    :78) and ``bootstrap_value`` [B] -> (vs [T, B], advantages [T, B]), both stop-gradient.  One reverse pass per
    env in one launch; every product and sum is rounded once in the order the reference writes them."""
    tr = truncation.to(torch.float32)
    T, B = tr.shape
    tr = tr.contiguous()
    te, r, v = (x.to(torch.float32).contiguous() for x in (termination, rewards, values))
    bv = bootstrap_value.to(torch.float32).contiguous()
    vs, adv = torch.empty_like(tr), torch.empty_like(tr)
    with _lib.cuda_guard(tr):
        _lib.check(_lib.lib.mbpo_compute_gae(_lib.ptr(tr), _lib.ptr(te), _lib.ptr(r), _lib.ptr(v), _lib.ptr(bv), B, T, B, 1,
                                             float(discount), float(lambda_), _lib.ptr(vs), _lib.ptr(adv),
                                             _lib.stream_ptr(tr.device)))
    return vs, adv
