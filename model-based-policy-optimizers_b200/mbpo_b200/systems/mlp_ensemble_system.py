"""Learned MLP-ensemble System (BASELINE config 4).

The reference has no learned-dynamics System; it only ships the flax ``MLP`` template
(mbpo/utils/network_utils.py:5-17: Dense -> swish ... -> Dense) that such a System would wrap.
This class is that System: E ensemble members of [x_dim + u_dim -> 256 -> 256 -> 256 -> x_dim]
predicting the state increment, x_next = x + MLP_e([x, u]); the reward is the pendulum reward
(rewards/pendulum_reward.py:27-42).  In iCEM, particle p is rolled through member p.
The forward runs on the tcgen05 tensor cores (mbpo_mlp_dynamics_forward / mbpo_ensemble_rollout).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional

import torch

from .. import _lib
from .base_systems import System, SystemParams, SystemState, _Replaceable
from .pendulum_system import PendulumRewardParams, pack_pendulum


@dataclass
class MlpEnsembleDynamicsParams(_Replaceable):
    """Weights in flax Dense layout: weights[i] float32 [E, in, out], biases[i] float32 [E, out]
    for the four layers; `member` optionally selects the ensemble member per row in System.step."""
    weights: List[torch.Tensor] = None
    biases: List[torch.Tensor] = None
    member: Optional[torch.Tensor] = None

    @property
    def num_members(self) -> int:
        return self.weights[0].shape[0]


class _Packed:
    """Device buffers in the C-ABI layout + the ctypes struct pointing at them (kept alive together)."""

    def __init__(self, dyn: MlpEnsembleDynamicsParams, reward: PendulumRewardParams):
        w, b = dyn.weights, dyn.biases
        if len(w) != 4 or w[1].shape[-1] != w[1].shape[-2] or w[1].shape != w[2].shape:
            raise _lib.MbpoUnsupported(_lib.MBPO_EUNSUPPORTED, "MLP ensemble must be [in -> h -> h -> h -> out]")
        self.w_in = w[0].to(torch.float32).contiguous()
        self.b_in = b[0].to(torch.float32).contiguous()
        # hidden layers: bf16, K-major = [E, 2, out, in]
        self.w_h = torch.stack([w[1], w[2]], dim=1).transpose(-1, -2).contiguous().to(torch.bfloat16)
        self.b_h = torch.stack([b[1], b[2]], dim=1).to(torch.float32).contiguous()
        self.w_out = w[3].to(torch.float32).contiguous()
        self.b_out = b[3].to(torch.float32).contiguous()
        e, in_dim, hidden = self.w_in.shape
        x_dim = self.w_out.shape[-1]
        self.struct = _lib.MlpEnsembleParamsC(e, hidden, x_dim, in_dim - x_dim, _lib.ptr(self.w_in), _lib.ptr(self.b_in),
                                              _lib.ptr(self.w_h), _lib.ptr(self.b_h), _lib.ptr(self.w_out),
                                              _lib.ptr(self.b_out), pack_pendulum(None, reward))


class MLPEnsembleSystem(System):
    system_kind = _lib.SYSTEM_MLP_ENSEMBLE

    def __init__(self, x_dim: int = 3, u_dim: int = 1, num_members: int = 5, hidden: int = 256,
                 dynamics_params: Optional[MlpEnsembleDynamicsParams] = None,
                 reward_params: Optional[PendulumRewardParams] = None):
        super().__init__(x_dim=x_dim, u_dim=u_dim)
        self.num_members = num_members
        self.hidden = hidden
        self.dynamics_params = dynamics_params
        self.reward_params = reward_params or PendulumRewardParams()
        self._cache = None

    def init_params(self, key: torch.Tensor) -> SystemParams:
        """System.init_params (base_systems.py:54-60): keys = split(key, 3).  The dynamics parameters are
        the ones given to the constructor, or a random initialisation (N(0, 1/fan_in)) drawn from keys[0]."""
        from .. import random as jr
        keys = jr.split(key, 3)
        k_dyn = keys[..., 0, :].reshape(-1, 2)[0]
        dyn = self.dynamics_params
        if dyn is None:
            dims = (self.x_dim + self.u_dim, self.hidden, self.hidden, self.hidden, self.x_dim)
            lk = jr.split(k_dyn, 4)
            ws, bs = [], []
            for i in range(4):
                n = self.num_members * dims[i] * dims[i + 1]
                w = jr.normal(lk[i], n).reshape(self.num_members, dims[i], dims[i + 1]) / (dims[i] ** 0.5)
                ws.append(w * (0.1 if i == 3 else 1.0))
                bs.append(torch.zeros((self.num_members, dims[i + 1]), dtype=torch.float32, device=key.device))
            dyn = MlpEnsembleDynamicsParams(weights=ws, biases=bs)
        return SystemParams(dynamics_params=dyn, reward_params=self.reward_params, key=keys[..., 2, :].contiguous())

    def packed(self, system_params: SystemParams) -> _Packed:
        dyn = system_params.dynamics_params
        key = (id(dyn.weights), id(system_params.reward_params))
        if self._cache is None or self._cache[0] != key:
            self._cache = (key, _Packed(dyn, system_params.reward_params or PendulumRewardParams()))
        return self._cache[1]

    def pack_params(self, system_params: SystemParams):
        return self.packed(system_params).struct

    def _checked_member(self, member: torch.Tensor, E: int, num_members: int) -> torch.Tensor:
        """dynamics_params.member as int32 [E], checked on the host once per tensor: one read-back at its first use,
        cached by identity (as ``packed`` caches the weights).  A wrong shape or a member outside [0, num_members)
        raises ValueError before anything is launched."""
        cached = getattr(self, "_member_cache", None)
        if cached is not None and cached[0] is member and cached[1] == (E, num_members):
            return cached[2]
        if torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
            raise ValueError("dynamics_params.member is checked on the host at its first use, which cannot happen "
                             "inside a CUDA graph capture: run the call once before capturing it")
        if member.dtype.is_floating_point or member.dtype == torch.bool or member.numel() != E or \
                (member.dim() > 1 and tuple(member.shape) != (E, 1)):
            raise ValueError("dynamics_params.member must be an integer tensor [E] = [%d] (got %s %s)"
                             % (E, member.dtype, tuple(member.shape)))
        m = member.to(torch.int32).reshape(E).contiguous()
        if E:
            lo, hi = (int(v) for v in torch.stack([m.min(), m.max()]).cpu())
            if lo < 0 or hi >= num_members:
                raise ValueError("dynamics_params.member holds members in [%d, %d]; the ensemble has %d"
                                 % (lo, hi, num_members))
        self._member_cache = (member, (E, num_members), m)
        return m

    def env_grouping(self, system_params: SystemParams, E: int, device):
        """The envs grouped by ensemble member for mbpo_ensemble_env_rollout: (env_order int32 [E], the env indices
        stably sorted by member; member_offsets int32 [num_members + 1], where member k's envs start in env_order).
        Env e is rolled through dynamics_params.member[e], or member 0 when member is None.  Computed on the device
        without a synchronisation (a CUDA graph captures it); the members are checked once per tensor."""
        dyn = system_params.dynamics_params
        num_members = dyn.num_members
        if dyn.member is None:
            order = torch.arange(E, dtype=torch.int32, device=device)
            offsets = torch.full((num_members + 1,), E, dtype=torch.int32, device=device)
            offsets[0] = 0
            return order, offsets
        m = self._checked_member(dyn.member, E, num_members).to(device)
        sorted_m, order = torch.sort(m, stable=True)
        # searchsorted takes any value: no index reaches the device unchecked
        bounds = torch.arange(num_members + 1, dtype=torch.int32, device=device)
        offsets = torch.searchsorted(sorted_m, bounds).to(torch.int32)
        return order.to(torch.int32), offsets

    def step(self, x: torch.Tensor, u: torch.Tensor, system_params: SystemParams) -> SystemState:
        """x[..., X], u[..., A] -> SystemState.  Rows use dynamics_params.member (int32 [...]) or member 0."""
        pk = self.packed(system_params)
        xc = x.to(torch.float32).reshape(-1, self.x_dim).contiguous()
        uc = u.to(torch.float32).reshape(-1, self.u_dim).contiguous()
        rows = xc.shape[0]
        member = system_params.dynamics_params.member
        member = (torch.zeros(rows, dtype=torch.int32, device=xc.device) if member is None
                  else member.to(torch.int32).reshape(-1).contiguous())
        inp = torch.cat([xc, uc], dim=-1).contiguous()
        delta = torch.empty((rows, self.x_dim), dtype=torch.float32, device=xc.device)
        with _lib.cuda_guard(xc):
            _lib.check(_lib.lib.mbpo_mlp_dynamics_forward(_lib.C.byref(pk.struct), _lib.ptr(inp), _lib.ptr(member), rows,
                                                          _lib.ptr(delta), _lib.stream_ptr(xc.device)))
        from .pendulum_system import PendulumSystem
        rew = PendulumSystem().step(xc, uc, SystemParams(reward_params=system_params.reward_params)).reward
        return SystemState(x_next=(xc + delta).reshape(x.shape), reward=rew.reshape(x.shape[:-1]),
                           system_params=system_params)

    def ensemble_returns(self, system_params: SystemParams, init_state: torch.Tensor, actions: torch.Tensor,
                         use_optimism: bool = False) -> torch.Tensor:
        """init_state [B, X], actions [B, M, H, A] -> objective [B, M] (mean or max over members)."""
        pk = self.packed(system_params)
        x0 = init_state.to(torch.float32).contiguous()
        acts = actions.to(torch.float32).contiguous()
        B, M, H, _ = acts.shape
        out = torch.empty((B, M), dtype=torch.float32, device=x0.device)
        with _lib.cuda_guard(x0):
            _lib.check(_lib.lib.mbpo_ensemble_rollout(_lib.C.byref(pk.struct), H, _lib.ptr(x0), _lib.ptr(acts), B, M,
                                                      _lib.SUMMARIZE_MAX if use_optimism else _lib.SUMMARIZE_MEAN,
                                                      _lib.ptr(out), _lib.stream_ptr(x0.device)))
        return out

    def ensemble_transitions(self, system_params: SystemParams, init_state: torch.Tensor, actions: torch.Tensor):
        """init_state [B, X], actions [B, M, H, A] -> (obs [B, M, E, H, X], reward [B, M, E, H]): the Transition
        fields of every member's rollout (obs[..., e, t, :] is the state before step t, obs[..., 0, :] = init_state)."""
        pk = self.packed(system_params)
        x0 = init_state.to(torch.float32).contiguous()
        acts = actions.to(torch.float32).contiguous()
        B, M, H, _ = acts.shape
        E = system_params.dynamics_params.num_members
        obs = torch.empty((B, M, E, H, self.x_dim), dtype=torch.float32, device=x0.device)
        rew = torch.empty((B, M, E, H), dtype=torch.float32, device=x0.device)
        with _lib.cuda_guard(x0):
            _lib.check(_lib.lib.mbpo_ensemble_rollout_transitions(_lib.C.byref(pk.struct), H, _lib.ptr(x0),
                                                                  _lib.ptr(acts), B, M, _lib.ptr(obs), _lib.ptr(rew),
                                                                  _lib.stream_ptr(x0.device)))
        return obs, rew
