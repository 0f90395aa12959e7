"""Vmapped env rollouts for SAC/PPO data collection (BASELINE config 3).

One object stands for the reference's wrapper stack AutoResetWrapper(VmapWrapper(
EpisodeWrapper(BraxWrapper(system)))) (mbpo/systems/brax_wrapper.py:40-50;
mbpo/optimizers/policy_optimizers/brax_utils/training.py:29-47,50-137) and ``unroll`` emits
the Transition that sac/acting.py:35-55 ``actor_step`` builds, for T steps in one launch.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict

import torch

from . import _lib
from .config import config
from .systems.base_systems import System, SystemParams, _Replaceable
from .utils.optimizer_utils import Transition


def is_general(system: System) -> bool:
    """NoisyPendulumSystem / PointMassSystem: their collection runs mbpo_env_unroll_general /
    mbpo_actor_rollout_general; the pendulum keeps its own tuned entry points."""
    return getattr(system, "system_kind", None) in (_lib.SYSTEM_NOISY_PENDULUM, _lib.SYSTEM_POINT_MASS)


def is_ensemble(system: System) -> bool:
    """MLPEnsembleSystem: its collection runs mbpo_ensemble_env_rollout (env e rolled through
    dynamics_params.member[e])."""
    return getattr(system, "system_kind", None) == _lib.SYSTEM_MLP_ENSEMBLE


def system_keys(system: System, system_params: SystemParams, E: int):
    """The envs' system_params.key [E, 2] a keyed general System steps with (None for one that draws nothing)."""
    if not getattr(system, "keyed", False):
        return None
    key = None if system_params is None else system_params.key
    if key is None:
        raise ValueError("%s draws from system_params.key: it must be set" % type(system).__name__)
    key = key.reshape(-1, 2).contiguous()
    if key.shape[0] != E:
        raise ValueError("system_params.key holds %d keys for %d envs" % (key.shape[0], E))
    return key


@dataclass
class EnvState(_Replaceable):
    """brax_utils/base.py:12-23 State, restricted to what the System path uses.  info holds
    'steps', 'truncation' and 'first_obs' like the Episode/AutoReset wrappers' info dict."""
    obs: torch.Tensor = None          # [E, X]
    reward: torch.Tensor = None       # [E]
    done: torch.Tensor = None         # [E] float, as brax
    system_params: SystemParams = None
    info: Dict[str, torch.Tensor] = None


class VmappedSystemEnv:
    def __init__(self, system: System, system_params: SystemParams, episode_length: int = 1000,
                 action_repeat: int = 1, brax_env=None):
        self.system = system
        self.init_system_params = system_params
        self.brax_env = brax_env      # a systems.BraxWrapper: resets draw from its true buffer
        self.episode_length = int(episode_length)
        self.action_repeat = int(action_repeat)

    @property
    def action_size(self) -> int:
        return self.system.u_dim

    @property
    def observation_size(self) -> int:
        return self.system.x_dim

    def reset(self, rng_or_first_obs: torch.Tensor) -> EnvState:
        """uint32 keys [E, 2] (``env.reset(jr.split(env_key, num_envs))``, sac.py:411-412): every env draws its first
        observation and reward from the true replay buffer and gets its own system_params key
        (brax_wrapper.py:25-38; needs ``wrap(BraxWrapper(...))``).  float32 [E, X]: the caller supplies the first
        observations.  Either way the Episode / AutoReset wrappers' info starts as training.py:87-89,115-116."""
        if rng_or_first_obs.dtype in (torch.uint32, torch.int32):
            if self.brax_env is None:
                raise _lib.MbpoError(_lib.MBPO_EINVAL, "reset(keys) needs the env built by wrap(BraxWrapper(...)): "
                                     "first observations come from its true buffer")
            st = self.brax_env.reset(rng_or_first_obs.reshape(-1, 2))
            obs, reward, params = st.obs, st.reward, st.system_params
        else:
            obs = rng_or_first_obs.to(torch.float32).contiguous().clone()
            reward, params = None, self.init_system_params
        e = obs.shape[0]
        zeros = torch.zeros(e, dtype=torch.float32, device=obs.device)
        return EnvState(obs=obs, reward=zeros.clone() if reward is None else reward, done=zeros.clone(),
                        system_params=params,
                        info=dict(steps=zeros.clone(), truncation=zeros.clone(), first_obs=obs.clone()))

    def unroll(self, state: EnvState, actions: torch.Tensor):
        """actions [T, E, A] -> (final EnvState, Transition with fields [T, E, ...]); extras
        carries state_extras.truncation like actor_step (acting.py:46-55).  observation and
        next_observation are overlapping views of one buffer (treat them as read-only)."""
        acts = actions.to(torch.float32).contiguous()
        T, E, A = acts.shape
        X = self.system.x_dim
        dev = acts.device
        obs_in = state.obs.contiguous()
        steps_in = state.info["steps"].contiguous()
        done_in = state.done.contiguous()
        first = state.info["first_obs"].contiguous()
        obs, steps, done = torch.empty_like(obs_in), torch.empty_like(steps_in), torch.empty_like(done_in)
        # observation[t] = next_observation[t-1]: both are views of one [T+1, E, X] buffer
        buf = torch.empty((T + 1, E, X), dtype=torch.float32, device=dev)
        buf[0].copy_(obs_in)
        o, n = buf[:T], buf[1:]
        r = torch.empty((T, E), dtype=torch.float32, device=dev)
        d = torch.empty((T, E), dtype=torch.float32, device=dev)
        tr = torch.empty((T, E), dtype=torch.float32, device=dev)
        params = self.system.pack_params(state.system_params)
        self._grouping = self.system.env_grouping(state.system_params, E, dev) if is_ensemble(self.system) else None
        keys_in = system_keys(self.system, state.system_params, E) if is_general(self.system) else None
        keys_out = torch.empty_like(keys_in) if keys_in is not None else None
        if T == 0:
            obs, steps, done = obs_in.clone(), steps_in.clone(), done_in.clone()
        with _lib.cuda_guard(acts):
            self._launch(params, obs_in, steps_in, done_in, keys_in, obs, steps, done, keys_out, first, _lib.ptr(acts),
                         E, T, _lib.ptr(r), _lib.ptr(d), _lib.ptr(n), _lib.ptr(tr), _lib.stream_ptr(dev))
        new_state = EnvState(obs=obs, reward=r[-1] if T else state.reward, done=done,
                             system_params=self._params_after(state.system_params, keys_out),
                             info=dict(steps=steps, truncation=tr[-1] if T else state.info["truncation"],
                                       first_obs=first))
        transition = Transition(observation=o, action=acts, reward=r, discount=d, next_observation=n,
                                extras={"state_extras": {"truncation": tr}})
        return new_state, transition

    def unroll_streamed(self, state: EnvState, actions_host: torch.Tensor, reward_host: torch.Tensor = None,
                        chunk_steps: int = 64):
        """``unroll`` for actions that live in pinned host memory: the T steps are cut into chunks and the host ->
        device copy of chunk k + 1, the rollout of chunk k and the device -> host copy of chunk k - 1's rewards run
        concurrently on three streams (PCIe is full duplex; the rollout itself is a few percent of either copy).
        Same bits as ``unroll`` (chunked == whole, see DESIGN 4.7).  ``reward_host`` [T, E] (pinned) receives the
        rewards; the caller's stream is ordered after everything, so one synchronize covers the copies too."""
        if actions_host.is_cuda or not actions_host.is_pinned():
            raise _lib.MbpoError(_lib.MBPO_EINVAL, "unroll_streamed: actions_host must be a pinned host tensor")
        T, E, A = actions_host.shape
        X = self.system.x_dim
        dev = state.obs.device
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_streams"):
            self._streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        s_in, s_out = self._streams
        acts = torch.empty((T, E, A), dtype=torch.float32, device=dev)
        buf = torch.empty((T + 1, E, X), dtype=torch.float32, device=dev)
        buf[0].copy_(state.obs)
        r = torch.empty((T, E), dtype=torch.float32, device=dev)
        d = torch.empty((T, E), dtype=torch.float32, device=dev)
        tr = torch.empty((T, E), dtype=torch.float32, device=dev)
        first = state.info["first_obs"].contiguous()
        cur = [state.obs.contiguous(), state.info["steps"].contiguous(), state.done.contiguous()]
        keys = system_keys(self.system, state.system_params, E) if is_general(self.system) else None
        if keys is not None:
            cur.append(keys)
        nxt = [torch.empty_like(t) for t in cur]
        spare = [torch.empty_like(t) for t in cur]
        params = self.system.pack_params(state.system_params)
        self._grouping = self.system.env_grouping(state.system_params, E, dev) if is_ensemble(self.system) else None
        s_in.wait_stream(main)              # acts / buf exist before the copies start
        s_out.wait_stream(main)
        bounds = [(t0, min(t0 + chunk_steps, T)) for t0 in range(0, T, max(int(chunk_steps), 1))]
        ev_in = []
        with torch.cuda.stream(s_in):
            for t0, t1 in bounds:
                acts[t0:t1].copy_(actions_host[t0:t1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(s_in)
                ev_in.append(ev)
        with _lib.cuda_guard(acts):
            for k, (t0, t1) in enumerate(bounds):
                main.wait_event(ev_in[k])
                self._launch(params, cur[0], cur[1], cur[2], cur[3] if keys is not None else None, nxt[0], nxt[1],
                             nxt[2], nxt[3] if keys is not None else None, first, acts[t0:t1].data_ptr(), E, t1 - t0,
                             r[t0:t1].data_ptr(), d[t0:t1].data_ptr(), buf[1 + t0:1 + t1].data_ptr(),
                             tr[t0:t1].data_ptr(), main.cuda_stream)
                cur, nxt, spare = nxt, spare, cur
                if reward_host is not None:
                    ev = torch.cuda.Event()
                    ev.record(main)
                    s_out.wait_event(ev)
                    with torch.cuda.stream(s_out):
                        reward_host[t0:t1].copy_(r[t0:t1], non_blocking=True)
        # the caller's stream is ordered after both side streams: buffers allocated on it may be reused in its order
        # (no record_stream: that would keep the caching allocator from recycling the big blocks call after call)
        main.wait_stream(s_in)
        main.wait_stream(s_out)
        new_state = EnvState(obs=cur[0], reward=r[-1] if T else state.reward, done=cur[2],
                             system_params=self._params_after(state.system_params,
                                                              cur[3] if keys is not None else None),
                             info=dict(steps=cur[1], truncation=tr[-1] if T else state.info["truncation"],
                                       first_obs=first))
        transition = Transition(observation=buf[:T], action=acts, reward=r, discount=d, next_observation=buf[1:],
                                extras={"state_extras": {"truncation": tr}})
        return new_state, transition

    def _launch(self, params, obs_in, steps_in, done_in, keys_in, obs_out, steps_out, done_out, keys_out, first,
                acts_ptr, E, T, r_ptr, d_ptr, n_ptr, tr_ptr, stream):
        """One launch of T wrapped env steps (observation_out = NULL: observation[t] is next_observation[t-1])."""
        X, A = self.system.x_dim, self.system.u_dim
        if is_ensemble(self.system):
            # the ensemble's kernel steps the env state in place
            for src, dst in ((obs_in, obs_out), (steps_in, steps_out), (done_in, done_out)):
                if dst.data_ptr() != src.data_ptr():
                    dst.copy_(src)
            order, offsets = self._grouping
            _lib.check(_lib.lib.mbpo_ensemble_env_rollout(
                _lib.C.byref(params), config.prng_mode, None, 0, 0, None, self.episode_length, self.action_repeat,
                _lib.ptr(order), _lib.ptr(offsets), _lib.ptr(obs_out), _lib.ptr(steps_out), _lib.ptr(done_out),
                _lib.ptr(first), E, T, acts_ptr, None, r_ptr, d_ptr, n_ptr, tr_ptr, None, None, None, stream))
            return
        if is_general(self.system):
            _lib.check(_lib.lib.mbpo_env_unroll_general(
                self.system.system_kind, _lib.C.byref(params), config.prng_mode, self.episode_length,
                self.action_repeat, _lib.ptr(obs_in), _lib.ptr(steps_in), _lib.ptr(done_in), _lib.ptr(keys_in),
                _lib.ptr(obs_out), _lib.ptr(steps_out), _lib.ptr(done_out), _lib.ptr(keys_out), _lib.ptr(first),
                acts_ptr, E, T, None, r_ptr, d_ptr, n_ptr, tr_ptr, stream))
            return
        _lib.check(_lib.lib.mbpo_env_unroll(
            self.system.system_kind, _lib.C.addressof(params), config.math_mode_id, X, A, self.episode_length,
            self.action_repeat, _lib.ptr(obs_in), _lib.ptr(steps_in), _lib.ptr(done_in), _lib.ptr(obs_out),
            _lib.ptr(steps_out), _lib.ptr(done_out), _lib.ptr(first), acts_ptr, E, T, None, r_ptr, d_ptr, n_ptr,
            tr_ptr, stream))

    @staticmethod
    def _params_after(system_params: SystemParams, keys_out):
        """system_params after the unroll: a keyed System carries its advanced keys on."""
        return system_params if keys_out is None else system_params.replace(key=keys_out)

    def step(self, state: EnvState, action: torch.Tensor) -> EnvState:
        """One wrapped env step: action [E, A]."""
        new_state, _ = self.unroll(state, action.reshape(1, *action.shape))
        return new_state


def wrap(env_or_system, *args, **kwargs) -> VmappedSystemEnv:
    """training.py:29-47 ``wrap(env, episode_length=1000, action_repeat=1)`` with ``env`` a systems.BraxWrapper; also
    accepts ``wrap(system, system_params, episode_length, action_repeat)`` (resets then take the first observations
    from the caller)."""
    if isinstance(env_or_system, System):
        return VmappedSystemEnv(env_or_system, *args, **kwargs)

    def _lengths(episode_length: int = 1000, action_repeat: int = 1):
        return int(episode_length), int(action_repeat)

    episode_length, action_repeat = _lengths(*args, **kwargs)
    env = env_or_system
    return VmappedSystemEnv(env.system, env.init_system_params, episode_length, action_repeat, brax_env=env)
