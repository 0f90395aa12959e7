"""iCEM trajectory optimizer behind the reference's call signatures.

Mirrors mbpo/optimizers/trajectory_optimizers/icem_optimizer.py: iCemParams :25-50,
iCemOptimizerState :62-69, AbstractCost :78-90, iCemTO :93-257, iCEMOptimizer :260-319.
``optimize`` is one launch of the fused CUDA plan kernel (mbpo_icem_plan): sampling, rollouts,
elite selection and refit for all num_steps iterations run on the GPU; nothing is computed on
the host.

Additive to the reference: every method also accepts a leading problem axis -- initial_state
[B, X] with an opt_state whose key is [B, 2] and best_sequence [B, H, A] -- which is
``jax.vmap(optimize)`` with per-problem keys, and ``closed_loop`` runs the plan -> true
System.step -> warm start loop of tests/test_icemopt.py:19-32 in a single launch.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, List, NamedTuple, Optional, Tuple

import torch

from ... import _lib
from ... import random as jr
from ...config import config
from ...envs import is_general
from ...systems.base_systems import System
from ...utils.type_aliases import OptimizerState, OptimizerTrainingOutPut
from ..base_optimizer import BaseOptimizer


class iCemParams(NamedTuple):
    """icem_optimizer.py:25-50."""
    num_particles: int = 10
    num_samples: int = 500
    num_elites: int = 50
    init_std: float = 0.5
    alpha: float = 0.0
    num_steps: int = 5
    exponent: float = 0.0
    elite_set_fraction: float = 0.3
    u_min: Any = -1.0
    u_max: Any = 1.0
    warm_start: bool = True
    lambda_constraint: float = 1e4


@dataclass
class iCemOptimizerState(OptimizerState):
    """icem_optimizer.py:62-69."""
    best_sequence: torch.Tensor = None
    best_reward: torch.Tensor = None

    @property
    def action(self):
        # best_sequence[0]; with a leading problem axis: the first action of every problem
        return self.best_sequence[..., 0, :]


@dataclass
class iCemTrainingOutput(OptimizerTrainingOutPut):
    summary: List = None


class AbstractCost:
    """icem_optimizer.py:78-90: ``cost(states [H, X], actions [H, A]) -> scalar`` with the constraint
    E[sum_t c(x_t, u_t)] <= 0.  Here the cost is a torch function of CUDA tensors; like the reference
    (``vmap(self.cost_fn)``, :162) it is written for ONE trajectory and vmapped over problems and
    candidates by the optimizer (torch.vmap).  The rollouts that feed it, the particle summaries and the
    penalty ``reward - lambda * relu(cost)`` (:166) run in the CUDA library (staged plan)."""

    def __init__(self, horizon: int):
        self.horizon = horizon

    def __call__(self, states, actions):
        raise NotImplementedError


def _scalar_bound(v):
    """float(v) if the bound is a scalar (or an array of one repeated value), else None."""
    if isinstance(v, torch.Tensor):
        if v.numel() == 1 or bool((v == v.reshape(-1)[0]).all()):
            return float(v.reshape(-1)[0])
        return None
    try:
        return float(v)
    except TypeError:
        import numpy as np
        a = np.asarray(v, dtype=np.float32)
        if (a == a.reshape(-1)[0]).all():
            return float(a.reshape(-1)[0])
        return None


def _array_bound(v, opt_dim, device) -> torch.Tensor:
    """A bound broadcastable to (H, A) (icem_optimizer.py:47-48) as a contiguous float32 [H*A] device tensor."""
    t = torch.as_tensor(v, dtype=torch.float32, device=device)
    return torch.broadcast_to(t, opt_dim).reshape(-1).contiguous()


class iCemTO(BaseOptimizer):
    def __init__(self, horizon: int, action_dim: int, key: Optional[torch.Tensor] = None,
                 opt_params: iCemParams = iCemParams(), cost_fn: AbstractCost | None = None,
                 use_optimism: bool = False, use_pessimism: bool = False, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.horizon = horizon
        self.opt_params = opt_params
        self.key = key
        self.opt_dim = (horizon,) + (action_dim,)
        self.action_dim = action_dim
        self.cost_fn = cost_fn
        self.use_optimism = use_optimism
        self.use_pessimism = use_pessimism

    # ---- C-ABI configuration -----------------------------------------------------------------
    def _array_bounds(self) -> bool:
        p = self.opt_params
        return _scalar_bound(p.u_min) is None or _scalar_bound(p.u_max) is None

    def _cfg(self) -> _lib.IcemCfgC:
        assert self.system is not None, "iCem optimizer requires system to be defined."
        p = self.opt_params
        # the struct depends on nothing but these; a plan at B = 1 is ~50 us on the device, so the ~12 us of
        # mbpo_icem_cfg_init per call are worth a memo (callers get their own copy)
        memo_key = (self.horizon, self.action_dim, self.system.x_dim, self.system.system_kind, config.prng_mode,
                    config.math_mode_id, bool(self.use_optimism))
        memo = getattr(self, "_cfg_memo", None)
        if memo is not None and memo[3] is p and memo[0] == memo_key:     # (opt_params is an immutable NamedTuple)
            return _lib.IcemCfgC.from_buffer_copy(memo[1])
        cfg = _lib.IcemCfgC()
        # array-valued bounds: the sampling kernel runs unclipped and mbpo_icem_clip_actions applies them
        lo, hi = (float("-inf"), float("inf")) if self._array_bounds() else (_scalar_bound(p.u_min),
                                                                           _scalar_bound(p.u_max))
        _lib.check(_lib.lib.mbpo_icem_cfg_init(
            _lib.C.byref(cfg), self.horizon, self.action_dim, self.system.x_dim, p.num_particles, p.num_samples,
            p.num_elites, p.init_std, p.alpha, p.num_steps, p.exponent, p.elite_set_fraction,
            lo, hi, int(bool(p.warm_start)), p.lambda_constraint))
        cfg.prng_mode = config.prng_mode
        cfg.summarize = _lib.SUMMARIZE_MAX if self.use_optimism else _lib.SUMMARIZE_MEAN   # :112-115
        cfg.system_kind = self.system.system_kind
        cfg.math_mode = config.math_mode_id
        self._cfg_memo = (memo_key, _lib.IcemCfgC.from_buffer_copy(cfg), {}, p)
        return cfg

    def _fused(self, cfg, packed_params) -> bool:
        """Whether mbpo_icem_plan / mbpo_icem_mpc_closed_loop (one launch) take this configuration; otherwise the
        staged plan (the same per-stage kernels, one launch per stage and iteration) runs it."""
        target = float(getattr(packed_params, "target_angle", 0.0))  # the fused reward wrap assumes |target| <= 6 rad
        memo = getattr(self, "_cfg_memo", None)
        same = memo is not None and bytes(memo[1]) == bytes(cfg)
        if same and "fused" in memo[2]:
            return memo[2]["fused"] and abs(target) <= 6.0
        fused = bool(_lib.lib.mbpo_icem_plan_is_fused(_lib.C.byref(cfg)))
        if same:
            memo[2]["fused"] = fused
        return fused and abs(target) <= 6.0

    # ---- reference API -------------------------------------------------------------------------
    def init(self, key: torch.Tensor, true_buffer_state=None) -> iCemOptimizerState:
        """icem_optimizer.py:121-132.  key [2] -> single-problem state; key [B, 2] -> B problems."""
        assert self.system is not None, "iCem optimizer requires system to be defined."
        ks = jr.split(key, 3)                                   # init_key, dummy_buffer_key, key
        init_key, dummy_buffer_key, new_key = ks[..., 0, :], ks[..., 1, :], ks[..., 2, :]
        system_params = self.system.init_params(init_key)
        batch = tuple(key.shape[:-1])
        return iCemOptimizerState(
            true_buffer_state=self.dummy_true_buffer_state(dummy_buffer_key),
            system_params=system_params,
            best_sequence=torch.zeros(batch + self.opt_dim, dtype=torch.float32, device=key.device),
            best_reward=torch.zeros(batch, dtype=torch.float32, device=key.device),
            key=new_key.contiguous(),
        )

    def _plan_raw(self, x0: torch.Tensor, key: torch.Tensor, best_seq: torch.Tensor, system_params,
                  trace: bool = False, cluster: int = -1, staged: bool = False):
        """x0 [B,X], key [B,2], best_seq [B,H,A] -> (best_seq', best_value, key', trace dict|None).
        cluster: thread-block-cluster size of the fused plan (-1: the library's choice for B; 1, 2, 4, 8: forced --
        every choice gives the same bits)."""
        if self.cost_fn is not None or self._array_bounds():
            return self._plan_general(x0, key, best_seq, system_params, trace=trace)
        cfg = self._cfg()
        B = x0.shape[0]
        dev = x0.device
        H, A = self.opt_dim
        # one allocation for the three outputs (best_seq', best_value, key'): the call is launch-latency sized
        out = torch.empty((B * (H * A + 3),), dtype=torch.float32, device=dev)
        out_seq = out[:B * H * A].view(B, H, A)
        out_val = out[B * H * A:B * H * A + B]
        out_key = out[B * H * A + B:].view(torch.uint32).view(B, 2)
        params = self.system.pack_params(system_params)
        tr_c, tr = None, None
        fused = self._fused(cfg, params) and not staged     # staged=True: the per-stage kernels even where a fused one exists
        with _lib.cuda_guard(x0):
            if fused:
                if trace:
                    S, M, K = cfg.num_steps, cfg.num_samples + cfg.num_prev_elites, cfg.num_elites
                    tr = dict(actions=torch.empty((S, B, M, H * A), dtype=torch.float32, device=dev),
                              values=torch.empty((S, B, M), dtype=torch.float32, device=dev),
                              elite_idx=torch.empty((S, B, K), dtype=torch.int32, device=dev),
                              mean=torch.empty((S, B, H * A), dtype=torch.float32, device=dev),
                              std=torch.empty((S, B, H * A), dtype=torch.float32, device=dev),
                              best_value=torch.empty((S, B), dtype=torch.float32, device=dev))
                    tr_c = _lib.IcemTraceC(*(_lib.ptr(tr[n]) for n in ("actions", "values", "elite_idx", "mean",
                                                                        "std", "best_value")))
                _lib.check(_lib.lib.mbpo_icem_plan_clustered(
                    _lib.C.byref(cfg), _lib.C.addressof(params), _lib.ptr(x0), _lib.ptr(key), _lib.ptr(best_seq), B,
                    _lib.ptr(out_seq), _lib.ptr(out_val), _lib.ptr(out_key),
                    _lib.C.byref(tr_c) if tr_c is not None else None, int(cluster), _lib.stream_ptr(dev)))
            elif trace:
                # the per-stage kernels composed from Python dump the same per-iteration arrays (and give the
                # same bits as mbpo_icem_plan_staged: the same kernels in the same order)
                return self._plan_general(x0, key, best_seq, system_params, trace=True)
            else:
                nbytes = _lib.lib.mbpo_icem_workspace_bytes(_lib.C.byref(cfg), B)
                ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
                _lib.check(_lib.lib.mbpo_icem_plan_staged(_lib.C.byref(cfg), _lib.C.addressof(params), _lib.ptr(x0),
                                                          _lib.ptr(key), _lib.ptr(best_seq), B, _lib.ptr(out_seq),
                                                          _lib.ptr(out_val), _lib.ptr(out_key), _lib.ptr(ws), nbytes,
                                                          _lib.stream_ptr(dev)))
        return out_seq, out_val, out_key, tr

    def _plan_general(self, x0: torch.Tensor, key: torch.Tensor, best_seq: torch.Tensor, system_params,
                      trace: bool = False):
        """iCemTO.optimize with a constraint cost (:161-166) and / or array-valued bounds (:47-48): the
        per-stage C-ABI kernels composed on the caller's stream.  Every number is produced by the CUDA
        library except the user's own cost function, which is vmapped torch code on the same device.

        With a cost, each iteration rolls out with Transition buffers, evaluates the cost on their observations and
        penalises the objective; one route per System kind:

        * PendulumSystem / PointMassSystem (deterministic, P identical particles): one rollout per candidate
          (mbpo_rollout_actions / mbpo_system_objective with P = 0), cost on [B, M, H, X], mbpo_icem_penalize.
        * NoisyPendulumSystem (draws from its key): mbpo_system_objective with P particles, cost on [B, M, P, H, X],
          mbpo_icem_penalize_particles.
        * MLPEnsembleSystem (particle p = member p): mbpo_ensemble_rollout_transitions, cost on [B, M, E, H, X],
          mbpo_icem_penalize_particles.

        The buffers of the particle routes take 4 * B * M * P * H * (X + 1) bytes per iteration (e.g. ~150 MB for
        the ensemble at B = 36, M = 1,039, P = 5, H = 50)."""
        cfg = self._cfg()
        L = _lib
        dev = x0.device
        B, X = x0.shape
        H, A = self.opt_dim
        N, Np, S = cfg.num_samples, cfg.num_prev_elites, cfg.num_steps
        M, D, P = N + Np, H * A, cfg.num_particles
        p = self.opt_params
        kind = self.system.system_kind
        general, ensemble = is_general(self.system), kind == L.SYSTEM_MLP_ENSEMBLE
        params = self.system.pack_params(system_params)
        if ensemble and P != params.num_members:
            raise L.MbpoUnsupported(L.MBPO_EUNSUPPORTED, "the ensemble System rolls particle p through member p; "
                                    "num_particles (%d) must equal num_members (%d)" % (P, params.num_members))
        lo = hi = None
        if self._array_bounds():
            lo, hi = _array_bound(p.u_min, self.opt_dim, dev), _array_bound(p.u_max, self.opt_dim, dev)
        cost_on = self.cost_fn is not None
        # a particle axis where the particles differ: a System that draws from its key, or the ensemble's members
        per_particle = cost_on and (ensemble or (general and self.system.keyed))
        st = L.stream_ptr(dev)
        ks = jr.split(key, 2)                                             # optimizer_key, key  (:246)
        carry, out_key = ks[:, 0].contiguous(), ks[:, 1].contiguous()
        mean = torch.zeros((B, H, A), dtype=torch.float32, device=dev)
        if p.warm_start:                                                  # :239-241
            mean[:, :-1] = best_seq[:, 1:]
            mean[:, -1] = best_seq[:, -1]
        std = torch.full((B, H, A), float(p.init_std), dtype=torch.float32, device=dev)       # :243
        bseq, bval = mean.clone(), torch.full((B,), float("-inf"), dtype=torch.float32, device=dev)   # :244,:235
        actions = torch.empty((B, M, H, A), dtype=torch.float32, device=dev)
        values = torch.empty((B, M), dtype=torch.float32, device=dev)
        lead = (B, M, P, H) if per_particle else (B, M, H)
        obs = torch.empty(lead + (X,), dtype=torch.float32, device=dev) if cost_on else None
        rew = torch.empty(lead, dtype=torch.float32, device=dev) if per_particle else None
        s_rew = L.SUMMARIZE_MAX if self.use_optimism else L.SUMMARIZE_MEAN    # :112-115
        s_cost = L.SUMMARIZE_MAX if self.use_pessimism else L.SUMMARIZE_MEAN  # :116-119
        lam = float(p.lambda_constraint)
        tr = {n: [] for n in ("actions", "values", "elite_idx", "mean", "std", "best_value")} if trace else None
        with L.cuda_guard(x0):
            for _ in range(S):
                nxt_carry = torch.empty_like(carry)
                pkeys = torch.empty((B, M, 2), dtype=torch.uint32, device=dev) if general else None
                L.check(L.lib.mbpo_icem_sample_actions(L.C.byref(cfg), L.ptr(carry), L.ptr(mean), L.ptr(std), B,
                                                       L.ptr(actions), L.ptr(nxt_carry), L.ptr(pkeys), st))
                if lo is not None:
                    L.check(L.lib.mbpo_icem_clip_actions(L.ptr(actions), L.ptr(lo), L.ptr(hi), B, M, N, D, st))
                if per_particle:
                    if ensemble:
                        L.check(L.lib.mbpo_ensemble_rollout_transitions(L.C.byref(params), H, L.ptr(x0),
                                                                        L.ptr(actions), B, M, L.ptr(obs), L.ptr(rew),
                                                                        st))
                    else:
                        L.check(L.lib.mbpo_system_objective(kind, L.C.byref(params), config.prng_mode, H, L.ptr(x0),
                                                            L.ptr(actions), L.ptr(pkeys), B, M, P, s_rew, None,
                                                            L.ptr(obs), L.ptr(rew), None, st))
                    cost = self._cost(obs, actions, (B, M, P))
                    L.check(L.lib.mbpo_icem_penalize_particles(L.ptr(values), L.ptr(rew), H, L.ptr(cost), B * M, P,
                                                               s_rew, s_cost, lam, st))
                elif general:
                    # one rollout per particle key, horizon mean, mean / max over the particles (:144-160); with a
                    # cost, the one rollout of a deterministic System and the tail over its P identical particles
                    L.check(L.lib.mbpo_system_objective(kind, L.C.byref(params), config.prng_mode, H, L.ptr(x0),
                                                        L.ptr(actions), L.ptr(pkeys), B, M, 0 if cost_on else P,
                                                        s_rew, L.ptr(values), L.ptr(obs), None, None, st))
                    if cost_on:
                        L.check(L.lib.mbpo_icem_penalize(L.ptr(values), L.ptr(self._cost(obs, actions, (B, M))),
                                                         B * M, P, s_rew, s_cost, lam, st))
                elif ensemble:
                    # particles = members; the rollout kernel summarises over them itself (:160)
                    L.check(L.lib.mbpo_ensemble_rollout(L.C.byref(params), H, L.ptr(x0), L.ptr(actions), B, M,
                                                        s_rew, L.ptr(values), st))
                else:
                    L.check(L.lib.mbpo_rollout_actions(kind, L.C.addressof(params), config.math_mode_id, H, A, X,
                                                       L.ptr(x0), L.ptr(actions), B, M, L.ptr(values), L.ptr(obs),
                                                       None, None, st))
                    cost = self._cost(obs, actions, (B, M)) if cost_on else None
                    L.check(L.lib.mbpo_icem_penalize(L.ptr(values), L.ptr(cost), B * M, P, s_rew, s_cost, lam, st))
                n_mean, n_std = torch.empty_like(mean), torch.empty_like(std)
                n_bval, n_bseq = torch.empty_like(bval), torch.empty_like(bseq)
                eidx = torch.empty((B, cfg.num_elites), dtype=torch.int32, device=dev) if trace else None
                L.check(L.lib.mbpo_icem_elite_refit(L.C.byref(cfg), L.ptr(actions), L.ptr(values), L.ptr(mean),
                                                    L.ptr(std), L.ptr(bval), L.ptr(bseq), B, L.ptr(n_mean),
                                                    L.ptr(n_std), L.ptr(n_bval), L.ptr(n_bseq), L.ptr(eidx), st))
                carry, mean, std, bval, bseq = nxt_carry, n_mean, n_std, n_bval, n_bseq
                if trace:                                 # the per-iteration dumps of the fused kernel, same layout
                    for n, v in (("actions", actions.reshape(B, M, D)), ("values", values), ("elite_idx", eidx),
                                 ("mean", mean.reshape(B, D)), ("std", std.reshape(B, D)), ("best_value", bval)):
                        tr[n].append(v.clone())
        if trace:
            tr = {n: torch.stack(v) for n, v in tr.items()}
        return bseq, bval, out_key, tr

    def _cost(self, obs: torch.Tensor, actions: torch.Tensor, lead) -> torch.Tensor:
        """The user's one-trajectory cost (:162) vmapped over the leading axes `lead` of obs [*lead, H, X]: problems,
        candidates and, where they differ, particles (whose actions are the candidate's, an expanded view) ->
        contiguous float32 [*lead]."""
        fn = self.cost_fn
        for _ in lead:
            fn = torch.vmap(fn)
        acts = actions if len(lead) == 2 else actions.unsqueeze(2).expand(lead + tuple(actions.shape[2:]))
        cost = fn(obs, acts)
        if not isinstance(cost, torch.Tensor) or cost.numel() != obs.shape[:len(lead)].numel():
            raise ValueError("cost_fn must return one scalar per trajectory (states [H, X], actions [H, A]); got %s "
                             "for %s trajectories" % (tuple(cost.shape) if isinstance(cost, torch.Tensor)
                                                      else type(cost).__name__, tuple(lead)))
        return cost.to(torch.float32).reshape(lead).contiguous()

    def _canon(self, initial_state: torch.Tensor, opt_state: iCemOptimizerState):
        single = initial_state.dim() == 1
        x0 = initial_state.reshape(1, -1) if single else initial_state
        x0 = x0.to(torch.float32).contiguous()
        B = x0.shape[0]
        H, A = self.opt_dim
        key = opt_state.key.reshape(-1, 2).contiguous()
        seq = opt_state.best_sequence.reshape(-1, H, A).to(torch.float32).contiguous()
        if key.shape[0] != B or seq.shape[0] != B:
            raise ValueError("optimize: %d initial states but opt_state holds %d keys / %d sequences" % (
                B, key.shape[0], seq.shape[0]))
        return single, x0, key, seq

    def optimize(self, initial_state: torch.Tensor, opt_state: iCemOptimizerState) -> iCemOptimizerState:
        """icem_optimizer.py:134-252."""
        assert self.system is not None, "iCem optimizer requires system to be defined."
        single, x0, key, seq = self._canon(initial_state, opt_state)
        out_seq, out_val, out_key, _ = self._plan_raw(x0, key, seq, opt_state.system_params)
        if single:
            out_seq, out_val, out_key = out_seq[0], out_val[0], out_key[0]
        return opt_state.replace(key=out_key, best_sequence=out_seq, best_reward=out_val)

    def act(self, obs: torch.Tensor, opt_state: iCemOptimizerState, evaluate: bool = True):
        """icem_optimizer.py:254-257."""
        new_opt_state = self.optimize(initial_state=obs, opt_state=opt_state)
        return new_opt_state.action, new_opt_state

    # ---- additive: closed loop in one launch (tests/test_icemopt.py:19-32) ---------------------
    def closed_loop(self, initial_state: torch.Tensor, opt_state: iCemOptimizerState, num_steps: int,
                    cluster: int = -1):
        """Returns (states [T, (B,) X], rewards [T, (B)], actions [T, (B,) A], new opt_state).  cluster: as in
        ``_plan_raw`` (a single problem is spread over 8 SMs by default).  The pendulum and the general Systems
        (NoisyPendulumSystem, PointMassSystem) run the whole loop in one launch; a System that draws steps with
        opt_state.system_params.key ([B, 2], or [2] for a single problem) as ``system.step`` does."""
        assert self.system is not None, "iCem optimizer requires system to be defined."
        single, x0, key, seq = self._canon(initial_state, opt_state)
        cfg = self._cfg()
        params = self.system.pack_params(opt_state.system_params)
        kind = self.system.system_kind
        general = kind in (_lib.SYSTEM_NOISY_PENDULUM, _lib.SYSTEM_POINT_MASS)
        sys_key = opt_state.system_params.key if general and self.system.keyed else None
        if (self.cost_fn is not None or self._array_bounds() or not self._fused(cfg, params)
                or not (kind == _lib.SYSTEM_PENDULUM or general)
                or (general and self.system.keyed and sys_key is None)):   # (system.step raises for the missing key)
            return self._closed_loop_staged(single, x0, key, seq, opt_state, num_steps)
        B, dev = x0.shape[0], x0.device
        H, A = self.opt_dim
        states = torch.empty((num_steps, B, x0.shape[1]), dtype=torch.float32, device=dev)
        rewards = torch.empty((num_steps, B), dtype=torch.float32, device=dev)
        actions = torch.empty((num_steps, B, A), dtype=torch.float32, device=dev)
        out_seq = torch.empty((B, H, A), dtype=torch.float32, device=dev)
        out_key = torch.empty((B, 2), dtype=torch.uint32, device=dev)
        with _lib.cuda_guard(x0):
            if general:
                sys_keys = sys_key_out = None
                if sys_key is not None:
                    sys_keys = sys_key.reshape(-1, 2).contiguous()
                    if sys_keys.shape[0] != B:
                        raise ValueError("system_params.key holds %d keys for %d problems" % (sys_keys.shape[0], B))
                    sys_key_out = torch.empty_like(sys_keys)
                _lib.check(_lib.lib.mbpo_icem_mpc_closed_loop_general(
                    _lib.C.byref(cfg), _lib.C.byref(params), _lib.ptr(x0), _lib.ptr(key), _lib.ptr(seq),
                    _lib.ptr(sys_keys), B, num_steps, _lib.ptr(states), _lib.ptr(rewards), _lib.ptr(actions),
                    _lib.ptr(out_seq), _lib.ptr(out_key), _lib.ptr(sys_key_out), int(cluster), _lib.stream_ptr(dev)))
            else:
                _lib.check(_lib.lib.mbpo_icem_mpc_closed_loop_clustered(
                    _lib.C.byref(cfg), _lib.C.addressof(params), _lib.ptr(x0), _lib.ptr(key), _lib.ptr(seq), B,
                    num_steps, _lib.ptr(states), _lib.ptr(rewards), _lib.ptr(actions), _lib.ptr(out_seq),
                    _lib.ptr(out_key), int(cluster), _lib.stream_ptr(dev)))
        if single:
            states, rewards, actions, out_seq, out_key = states[:, 0], rewards[:, 0], actions[:, 0], out_seq[0], out_key[0]
        return states, rewards, actions, opt_state.replace(key=out_key, best_sequence=out_seq)


    def _closed_loop_staged(self, single, x0, key, seq, opt_state, num_steps):
        """The same loop for configurations without a fused kernel (cost_fn, array-valued bounds, a horizon without an
        unrolled instance, a population beyond shared memory, a learned System): plan -> System.step -> warm start,
        one plan call and one step launch per MPC step, all on the device."""
        states, rewards, actions = [], [], []
        sp = opt_state.system_params
        x = x0
        for _ in range(num_steps):
            seq, _, key, _ = self._plan_raw(x, key, seq, sp)
            u = seq[:, 0, :].contiguous()
            nxt = self.system.step(x, u, sp)
            if nxt.system_params is not None and nxt.system_params.key is not None:
                sp = nxt.system_params                      # a System that draws carries its key on (tests/test_icemopt.py:24)
            x = nxt.x_next
            states.append(x); rewards.append(nxt.reward); actions.append(u)
        B, dev = x0.shape[0], x0.device
        if num_steps:
            states, rewards, actions = torch.stack(states), torch.stack(rewards), torch.stack(actions)
        else:
            states = torch.empty((0, B, x0.shape[1]), dtype=torch.float32, device=dev)
            rewards = torch.empty((0, B), dtype=torch.float32, device=dev)
            actions = torch.empty((0, B, self.action_dim), dtype=torch.float32, device=dev)
        if single:
            states, rewards, actions, seq, key = states[:, 0], rewards[:, 0], actions[:, 0], seq[0], key[0]
        return states, rewards, actions, opt_state.replace(key=key, best_sequence=seq)


class iCEMOptimizer(BaseOptimizer):
    """icem_optimizer.py:260-319: wrapper for consistency with the SAC / PPO optimizers."""

    def __init__(self, horizon: int, opt_params: iCemParams = iCemParams(), system: System | None = None,
                 key: Optional[torch.Tensor] = None, **agent_kwargs):
        super().__init__(system, key)
        self.horizon = horizon
        self.key = key
        self.opt_params = opt_params
        self.agent_class = iCemTO
        self.agent_kwargs = agent_kwargs
        if system is not None:
            self.set_system(system)

    @property
    def can_act_in_batches(self):
        return False

    def init(self, key: torch.Tensor, true_buffer_state=None) -> iCemOptimizerState:
        assert self.system is not None, "iCEM optimizer requires system to be defined."
        self.agent = self.agent_class(horizon=self.horizon, action_dim=self.system.u_dim, key=self.key,
                                      opt_params=self.opt_params, **self.agent_kwargs)
        self.agent.set_system(self.system)
        if true_buffer_state is None:
            ks = jr.split(key, 2)
            dummy_buffer_key, key = ks[0], ks[1]
            true_buffer_state = self.dummy_true_buffer_state(dummy_buffer_key)
        agent_state = self.agent.init(key)
        agent_state.true_buffer_state = true_buffer_state
        return agent_state

    def act(self, obs: torch.Tensor, opt_state: iCemOptimizerState, evaluate: bool = True) -> Tuple[torch.Tensor, iCemOptimizerState]:
        assert self.system is not None, "iCEM optimizer requires system to be defined."
        action, opt_state = self.agent.act(obs.reshape(-1), opt_state, evaluate)
        return action.reshape(1, -1), opt_state

    def train(self, opt_state: iCemOptimizerState) -> iCemTrainingOutput:
        training_output = super().train(opt_state)
        return iCemTrainingOutput(optimizer_state=training_output.optimizer_state, summary=[])
