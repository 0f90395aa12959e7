"""Policy-in-the-loop data collection for SAC / PPO behind the reference's acting API.

Mirrors mbpo/optimizers/policy_optimizers/sac/acting.py:35-78 (``actor_step``, ``generate_unroll``),
sac/sac_networks.py:58-73 (``make_inference_fn``) and the experience scan of sac/sac.py:283-292
(``get_experience``): the policy MLP forward, the NormalTanh sample (JAX's threefry draw, bit for bit),
the wrapped env step and the Transition for T steps of E envs are ONE kernel launch
(mbpo_actor_rollout); nothing is computed on the host.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence, Tuple

import torch

from . import _lib
from .config import config
from .envs import EnvState, VmappedSystemEnv, is_ensemble, is_general, system_keys
from .utils.optimizer_utils import Transition


@dataclass
class PolicyParams:
    """flax Dense kernels [in, out] and biases of the policy network: obs -> 64 x num_hidden -> 2 * A."""
    weights: List[torch.Tensor]
    biases: List[torch.Tensor]
    min_std: float = 0.001          # NormalTanhDistribution(min_std=0.001), parametric_distribution.py:100


class Policy:
    """What ``make_policy(params, deterministic)`` returns (sac_networks.py:61-70).  Calling it samples
    actions for a batch of observations; actor_step / generate_unroll run it inside the env loop."""

    def __init__(self, params: PolicyParams, deterministic: bool = False, obs_mean: Sequence[float] = None,
                 obs_std: Sequence[float] = None, emit_extras: bool = False, kernel: str = "auto"):
        """obs_mean / obs_std: the running-statistics normaliser the reference passes as ``normalizer_params``
        (``policy_network.apply(normalizer_params, policy_params, obs)``: (obs - mean) / std); emit_extras: PPO's
        policy also returns {'log_prob', 'raw_action'} (ppo_network.py:72-80); kernel: "auto" (tcgen05 for 2..3
        hidden layers -- the wide latency kernel when the envs do not fill the GPU --, CUDA cores otherwise; the
        CUDA-core kernel of mbpo_actor_rollout_general for NoisyPendulumSystem / PointMassSystem; for
        MLPEnsembleSystem the policy runs on the CUDA cores inside the ensemble's tcgen05 env kernel,
        mbpo_ensemble_env_rollout, with 1..2 hidden layers), "cuda_cores", "tcgen05" (throughput kernel) or
        "tcgen05_wide" (latency kernel); the tcgen05 kernels hold the pendulum only."""
        w = [t.to(torch.float32).contiguous() for t in params.weights]
        b = [t.to(torch.float32).contiguous() for t in params.biases]
        if len(w) < 2 or len(w) != len(b) or len(w) > 5:
            raise _lib.MbpoUnsupported(_lib.MBPO_EUNSUPPORTED, "policy needs 1..4 hidden layers")
        self.weights, self.biases = w, b
        self.deterministic = bool(deterministic)
        self.min_std = float(params.min_std)
        s = _lib.PolicyParamsC()
        s.num_hidden = len(w) - 1
        s.hidden = w[0].shape[1]
        s.obs_dim = w[0].shape[0]
        s.action_dim = w[-1].shape[1] // 2
        for i, (wi, bi) in enumerate(zip(w, b)):
            s.w[i] = _lib.ptr(wi)
            s.b[i] = _lib.ptr(bi)
        s.min_std = self.min_std
        s.head = _lib.HEAD_NORMAL_TANH
        s.kernel = {"auto": _lib.ACTOR_AUTO, "cuda_cores": _lib.ACTOR_CUDA_CORES, "tcgen05": _lib.ACTOR_TCGEN05,
                    "tcgen05_wide": _lib.ACTOR_TCGEN05_WIDE}[kernel]
        self.struct = s
        self.emit_extras = bool(emit_extras) and not self.deterministic
        self._set_normalizer(obs_mean, obs_std)

    def _set_normalizer(self, obs_mean, obs_std):
        """Sequences of floats go into the struct by value; CUDA tensors stay on the device (the kernels read them
        through obs_mean_dev / obs_std_dev: no read-back of the running statistics in a collection loop)."""
        s = self.struct
        s.normalize = int(obs_mean is not None)
        s.obs_mean_dev = s.obs_std_dev = None
        if torch.is_tensor(obs_mean) and obs_mean.is_cuda:
            self._norm = (obs_mean.to(torch.float32).contiguous(), obs_std.to(torch.float32).contiguous())
            s.obs_mean_dev, s.obs_std_dev = _lib.ptr(self._norm[0]), _lib.ptr(self._norm[1])
        elif obs_mean is not None:
            mean = [float(v) for v in (obs_mean.tolist() if hasattr(obs_mean, "tolist") else obs_mean)]
            std = [float(v) for v in (obs_std.tolist() if hasattr(obs_std, "tolist") else obs_std)]
            for i in range(len(mean)):
                s.obs_mean[i], s.obs_std[i] = mean[i], std[i]

    def __call__(self, observations: torch.Tensor, key_sample: torch.Tensor):
        """policy(observations [E, X], key) -> (actions [E, A], {}).  Runs one actor step on a scratch env
        state and returns its actions (the env outputs are discarded)."""
        from .systems.pendulum_system import PendulumSystem
        system = PendulumSystem()
        env = VmappedSystemEnv(system, system.reset(device=observations.device).system_params, episode_length=1 << 30)
        _, tr = actor_step(env, env.reset(observations), self, key_sample)
        return tr.action, {}


class BpttActorPolicy(Policy):
    """BPTT's actor as a policy for ``rollout_policy`` (bptt_optimizer.py:123-142 ``Actor``; :306-326 ``act``;
    :246 ``train_policy = lambda obs, opt_state: self.act(obs, opt_state, evaluate=False)``):
    mu, sig = split(MLP(normalize(obs)), 2); sig = clip(softplus(sig + inv_softplus(init_stddev)), sig_min, sig_max);
    action = clip(tanh(mu + normal(sample_key, mu.shape) * sig), +-0.999) with sample_key, key = split(key, 2), or
    clip(tanh(mu)) when evaluate.  obs_mean / obs_std are the state normaliser's (:70-72).  One key serves every
    trajectory of a batch: the reference vmaps actor_loss over initial states only (:366-368)."""

    def __init__(self, params: PolicyParams, init_stddev: float = 1.0, sig_min: float = 1e-6, sig_max: float = 1e2,
                 obs_mean: Sequence[float] = None, obs_std: Sequence[float] = None, evaluate: bool = False):
        super().__init__(params, deterministic=evaluate, obs_mean=obs_mean, obs_std=obs_std)
        import numpy as np
        s = self.struct
        s.head = _lib.HEAD_BPTT_ACTOR
        s.shared_noise = 1
        x = np.float32(init_stddev)                                      # inv_softplus on a weak-typed python float
        s.sig_bias = float(np.log(np.exp(x) - np.float32(1.0))) if init_stddev < 20.0 else float(x)
        s.sig_min, s.sig_max, s.action_clip = float(sig_min), float(sig_max), 0.999


def make_inference_fn():
    """sac_networks.make_inference_fn: returns make_policy(params, deterministic=False) -> Policy."""
    def make_policy(params: PolicyParams, deterministic: bool = False, obs_mean=None, obs_std=None) -> Policy:
        return Policy(params, deterministic, obs_mean, obs_std)
    return make_policy


def make_ppo_inference_fn():
    """ppo/ppo_network.py:59-84 make_inference_fn: the same NormalTanh policy, whose sample also returns
    {'log_prob', 'raw_action'}; they arrive in Transition.extras['policy_extras'] ([T, E] / [T, E, A])."""
    def make_policy(params: PolicyParams, deterministic: bool = False, obs_mean=None, obs_std=None) -> Policy:
        return Policy(params, deterministic, obs_mean, obs_std, emit_extras=True)
    return make_policy


def _rollout(env: VmappedSystemEnv, env_state: EnvState, policy: Policy, key: torch.Tensor, T: int,
             key_convention: int, extra_fields: Sequence[str], env_offset: int = 0, total_envs: int = None):
    for f in extra_fields:
        if f != "truncation":
            raise _lib.MbpoUnsupported(_lib.MBPO_EUNSUPPORTED, "extra field %r is not produced by the env kernel" % f)
    system = env.system
    X, A = system.x_dim, system.u_dim
    obs = env_state.obs.to(torch.float32).contiguous().clone()
    E = obs.shape[0]
    dev = obs.device
    steps = env_state.info["steps"].clone()
    done = env_state.done.clone()
    first = env_state.info["first_obs"].contiguous()
    key = key.reshape(2).contiguous()
    key_out = torch.empty_like(key)
    buf = torch.empty((T + 1, E, X), dtype=torch.float32, device=dev)       # observation / next_observation views
    buf[0].copy_(obs)
    act = torch.empty((T, E, A), dtype=torch.float32, device=dev)
    r = torch.empty((T, E), dtype=torch.float32, device=dev)
    d = torch.empty((T, E), dtype=torch.float32, device=dev)
    tr = torch.empty((T, E), dtype=torch.float32, device=dev)
    params = system.pack_params(env_state.system_params)
    # a shard of the envs draws its slice of normal(key, (total_envs, A)): same bits as the unsharded launch
    policy.struct.draw_total = int(total_envs) if total_envs is not None else 0
    policy.struct.draw_offset = int(env_offset) if total_envs is not None else 0
    raw = torch.empty((T, E, A), dtype=torch.float32, device=dev) if policy.emit_extras else None
    logp = torch.empty((T, E), dtype=torch.float32, device=dev) if policy.emit_extras else None
    system_params = env_state.system_params
    with _lib.cuda_guard(obs):
        if is_ensemble(system):
            order, offsets = system.env_grouping(system_params, E, dev)
            _lib.check(_lib.lib.mbpo_ensemble_env_rollout(
                _lib.C.byref(params), config.prng_mode, _lib.C.byref(policy.struct), int(policy.deterministic),
                key_convention, _lib.ptr(key), env.episode_length, env.action_repeat, _lib.ptr(order),
                _lib.ptr(offsets), _lib.ptr(obs), _lib.ptr(steps), _lib.ptr(done), _lib.ptr(first), E, T, None,
                _lib.ptr(act), _lib.ptr(r), _lib.ptr(d), _lib.ptr(buf[1:]), _lib.ptr(tr), _lib.ptr(key_out),
                _lib.ptr(raw), _lib.ptr(logp), _lib.stream_ptr(dev)))
        elif is_general(system):
            sys_keys = system_keys(system, system_params, E)
            sys_keys_out = torch.empty_like(sys_keys) if sys_keys is not None else None
            _lib.check(_lib.lib.mbpo_actor_rollout_general(
                system.system_kind, _lib.C.byref(params), config.prng_mode, _lib.C.byref(policy.struct),
                int(policy.deterministic), key_convention, _lib.ptr(key), env.episode_length, env.action_repeat,
                _lib.ptr(obs), _lib.ptr(steps), _lib.ptr(done), _lib.ptr(sys_keys), _lib.ptr(sys_keys_out),
                _lib.ptr(first), E, T, _lib.ptr(act), _lib.ptr(r), _lib.ptr(d), _lib.ptr(buf[1:]), _lib.ptr(tr),
                _lib.ptr(key_out), _lib.ptr(raw), _lib.ptr(logp), _lib.stream_ptr(dev)))
            if sys_keys_out is not None:
                system_params = system_params.replace(key=sys_keys_out)
        else:
            _lib.check(_lib.lib.mbpo_actor_rollout_extras(
                system.system_kind, _lib.C.addressof(params), config.math_mode_id, config.prng_mode,
                _lib.C.byref(policy.struct), int(policy.deterministic), key_convention, _lib.ptr(key),
                env.episode_length, env.action_repeat, _lib.ptr(obs), _lib.ptr(steps), _lib.ptr(done), _lib.ptr(first),
                E, T, _lib.ptr(act), _lib.ptr(r), _lib.ptr(d), _lib.ptr(buf[1:]), _lib.ptr(tr), _lib.ptr(key_out),
                _lib.ptr(raw), _lib.ptr(logp), _lib.stream_ptr(dev)))
    nstate = EnvState(obs=obs, reward=r[-1] if T else env_state.reward, done=done,
                      system_params=system_params,
                      info=dict(steps=steps, truncation=tr[-1] if T else env_state.info["truncation"], first_obs=first))
    policy_extras = {"log_prob": logp, "raw_action": raw} if policy.emit_extras else {}
    extras = {"policy_extras": policy_extras, "state_extras": {f: tr for f in extra_fields}}
    transition = Transition(observation=buf[:T], action=act, reward=r, discount=d, next_observation=buf[1:],
                            extras=extras)
    return nstate, transition, key_out


def actor_step(env: VmappedSystemEnv, env_state: EnvState, policy: Policy, key: torch.Tensor,
               extra_fields: Sequence[str] = ()) -> Tuple[EnvState, Transition]:
    """sac/acting.py:35-55: one step, the key is the policy's sample key.  Fields are [E, ...]."""
    nstate, tr, _ = _rollout(env, env_state, policy, key, 1, _lib.KEYS_AS_IS, extra_fields)
    ex = {"policy_extras": {k: v[0] for k, v in tr.extras["policy_extras"].items()},
          "state_extras": {k: v[0] for k, v in tr.extras["state_extras"].items()}}
    return nstate, Transition(tr.observation[0], tr.action[0], tr.reward[0], tr.discount[0], tr.next_observation[0], ex)


def generate_unroll(env: VmappedSystemEnv, env_state: EnvState, policy: Policy, key: torch.Tensor, unroll_length: int,
                    extra_fields: Sequence[str] = (), env_offset: int = 0,
                    total_envs: int = None) -> Tuple[EnvState, Transition]:
    """sac/acting.py:58-78: lax.scan of actor_step; per step current_key, next_key = split(current_key), the
    policy samples with current_key.  Fields are time-major [T, E, ...]."""
    nstate, tr, _ = _rollout(env, env_state, policy, key, unroll_length, _lib.KEYS_UNROLL, extra_fields, env_offset,
                             total_envs)
    return nstate, tr


def get_experience(env: VmappedSystemEnv, env_state: EnvState, policy: Policy, key: torch.Tensor,
                   num_env_steps: int, env_offset: int = 0,
                   total_envs: int = None) -> Tuple[torch.Tensor, EnvState, Transition]:
    """The scan of SAC.get_experience (sac/sac.py:288-294): per step k, k_t = split(k), actor_step with k_t and
    extra_fields=('truncation',).  env_offset / total_envs (additive): this call owns envs [env_offset, env_offset + E)
    of total_envs sharded over ranks, and draws its slice of the unsharded noise.
    Returns (carry key, env_state, transitions [T, E, ...]); the replay-buffer
    insert and the normaliser update stay with the caller (SURVEY 8f-2 boundary)."""
    nstate, tr, key_out = _rollout(env, env_state, policy, key, num_env_steps, _lib.KEYS_SAC, ("truncation",),
                                   env_offset, total_envs)
    return key_out, nstate, tr


def eval_metrics(env_state: EnvState, transitions: Transition, action_repeat: int = 1, carry=None):
    """EvalWrapper (brax_utils/training.py:156-199) folded over the Transition of an unroll that started from
    ``env_state``: -> (episode_reward [E], episode_steps [E], active_episodes [E]).  ``carry`` = the triple of an
    earlier chunk of the same evaluation (default: EvalWrapper.reset's zeros, zeros, ones)."""
    r, d = transitions.reward, transitions.discount
    T, E = r.shape
    dev = r.device
    if carry is None:
        carry = (torch.zeros(E, device=dev), torch.zeros(E, device=dev), torch.ones(E, device=dev))
    ep_reward, ep_steps, active = [c.to(torch.float32).contiguous().clone() for c in carry]
    if r.stride() != d.stride():
        d = d.contiguous()
        r = r.contiguous()
    steps_in, done_in = env_state.info["steps"].contiguous(), env_state.done.contiguous()
    with _lib.cuda_guard(r):
        _lib.check(_lib.lib.mbpo_eval_metrics(r.data_ptr(), d.data_ptr(), _lib.ptr(steps_in), _lib.ptr(done_in),
                                              int(action_repeat), E, T, r.stride(0) if T else 0, r.stride(1) if T else 1,
                                              _lib.ptr(ep_reward), _lib.ptr(ep_steps), _lib.ptr(active),
                                              _lib.stream_ptr(dev)))
    return ep_reward, ep_steps, active


class Evaluator:
    """sac/acting.py:82-151.  ``eval_env`` is the wrapped env (``envs.wrap(BraxWrapper(...), episode_length,
    action_repeat)``); every evaluation resets ``num_eval_envs`` envs from the true buffer, unrolls one episode with
    ``eval_policy_fn(policy_params)`` in one launch and folds EvalWrapper's episode metrics over the Transition."""

    def __init__(self, eval_env: VmappedSystemEnv, eval_policy_fn, num_eval_envs: int, episode_length: int,
                 action_repeat: int, key: torch.Tensor):
        self._key = key
        self._eval_walltime = 0.
        self._env = eval_env
        self._policy_fn = eval_policy_fn
        self._num_eval_envs = int(num_eval_envs)
        self._unroll_length = int(episode_length) // int(action_repeat)
        self._action_repeat = int(action_repeat)
        self._steps_per_unroll = int(episode_length) * int(num_eval_envs)

    def _generate_eval_unroll(self, policy_params, key: torch.Tensor):
        from . import random as jr
        reset_keys = jr.split(key, self._num_eval_envs)
        first = self._env.reset(reset_keys)
        nstate, tr = generate_unroll(self._env, first, self._policy_fn(policy_params), key, self._unroll_length)
        ep_reward, ep_steps, active = eval_metrics(first, tr, self._action_repeat)
        nstate.info["eval_metrics"] = dict(episode_metrics={"reward": ep_reward}, active_episodes=active,
                                           episode_steps=ep_steps)
        return nstate

    def run_evaluation(self, policy_params, training_metrics, unroll_key: torch.Tensor = None,
                       aggregate_episodes: bool = True):
        import time
        import numpy as np
        from . import random as jr
        if unroll_key is None:
            keys = jr.split(self._key, 2)
            self._key, unroll_key = keys[0], keys[1]
        t = time.time()
        eval_state = self._generate_eval_unroll(policy_params, unroll_key)
        em = eval_state.info["eval_metrics"]
        values = {name: v.cpu().numpy() for name, v in em["episode_metrics"].items()}     # synchronises
        epoch_eval_time = time.time() - t
        metrics = {"eval/episode_%s" % name: (np.mean(v) if aggregate_episodes else v) for name, v in values.items()}
        metrics["eval/avg_episode_length"] = np.mean(em["episode_steps"].cpu().numpy())
        metrics["eval/epoch_eval_time"] = epoch_eval_time
        metrics["eval/sps"] = self._steps_per_unroll / epoch_eval_time
        self._eval_walltime = self._eval_walltime + epoch_eval_time
        return {"eval/walltime": self._eval_walltime, **training_metrics, **metrics}


class ExperienceCollector:
    """SAC.get_experience in full (sac/sac.py:283-304): the scan of actor steps (one launch), the observation
    normaliser update (running_statistics.update, with the psum over ranks when ``pmap_axis_name`` is given) and the
    replay-buffer insert.  Same argument order and return value as the reference method (the carry key of the scan,
    which the reference drops, is kept in ``last_key``)."""

    def __init__(self, env: VmappedSystemEnv, make_policy, replay_buffer, num_env_steps_between_updates: int,
                 pmap_axis_name: str = None, env_offset: int = 0, total_envs: int = None):
        self.env = env
        self.make_policy = make_policy                 # make_policy((normalizer_params, policy_params)) -> Policy
        self.replay_buffer = replay_buffer
        self.num_env_steps_between_updates = int(num_env_steps_between_updates)
        self._PMAP_AXIS_NAME = pmap_axis_name
        self._env_offset, self._total_envs = env_offset, total_envs
        self.last_key = None

    def get_experience(self, normalizer_params, policy_params, env_state: EnvState, buffer_state, key: torch.Tensor):
        from . import running_statistics
        policy = self.make_policy((normalizer_params, policy_params))
        key, env_state, transitions = get_experience(self.env, env_state, policy, key,
                                                     self.num_env_steps_between_updates, self._env_offset,
                                                     self._total_envs)
        normalizer_params = running_statistics.update(normalizer_params, transitions.observation,
                                                      pmap_axis_name=self._PMAP_AXIS_NAME)
        buffer_state = self.replay_buffer.insert(buffer_state, transitions)
        self.last_key = key            # the scan's carry key (the reference discards it: sac.py:294,304)
        return normalizer_params, env_state, buffer_state


def make_normalized_inference_fn(emit_extras: bool = False, kernel: str = "auto"):
    """sac_networks.make_inference_fn with ``normalize_observations=True`` (sac_networks.py:58-73):
    make_policy((normalizer_params, policy_params), deterministic) -> Policy that reads (obs - mean) / std."""
    def make_policy(params, deterministic: bool = False) -> Policy:
        normalizer_params, policy_params = params
        return Policy(policy_params, deterministic, normalizer_params.mean, normalizer_params.std,
                      emit_extras=emit_extras, kernel=kernel)
    return make_policy


class GraphedRollout:
    """``get_experience`` / ``generate_unroll`` captured in a CUDA graph for the launch-bound regime (the reference's own
    configurations: tests/test_sac.py collects 20 steps of 32 envs per call, ~0.1 ms of GPU time -- as much as the host
    spends allocating outputs and crossing ctypes).  The C ABI neither allocates nor synchronises, so the whole call --
    state copies, the rollout launch, the hand-over of the env state and the carry key to the next call -- replays from
    one ``cudaGraphLaunch``.  Buffers are static: the returned Transition is overwritten by the next call.

        collect = GraphedRollout(env, env_state, policy, key, num_env_steps)      # captures
        key, env_state, transitions = collect()                                   # replays; same bits as get_experience
    """

    def __init__(self, env: VmappedSystemEnv, env_state: EnvState, policy: Policy, key: torch.Tensor, num_env_steps: int,
                 key_convention: int = _lib.KEYS_SAC, extra_fields: Sequence[str] = ("truncation",)):
        dev = env_state.obs.device
        params = env_state.system_params
        keys = system_keys(env.system, params, env_state.obs.shape[0])   # a keyed System's keys are replay state too
        if keys is not None:
            params = params.replace(key=keys.clone())
        self._state = EnvState(obs=env_state.obs.clone(), reward=env_state.reward.clone(), done=env_state.done.clone(),
                               system_params=params, info={k: v.clone() for k, v in env_state.info.items()})
        self._key = key.reshape(2).clone()
        self._policy = policy                      # keeps the weight tensors (and the struct's pointers) alive
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):              # warm-up outside the capture (lazy initialisation, allocator)
            for _ in range(2):
                _rollout(env, self._state, policy, self._key, num_env_steps, key_convention, extra_fields)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            nstate, tr, key_out = _rollout(env, self._state, policy, self._key, num_env_steps, key_convention,
                                           extra_fields)
            # hand the env state and the carry key over to the next replay
            self._state.obs.copy_(nstate.obs)
            self._state.done.copy_(nstate.done)
            self._state.info["steps"].copy_(nstate.info["steps"])
            self._key.copy_(key_out)
            if keys is not None:
                self._state.system_params.key.copy_(nstate.system_params.key)
        self._out = (key_out, nstate, tr)

    def __call__(self) -> Tuple[torch.Tensor, EnvState, Transition]:
        self._graph.replay()
        return self._out
