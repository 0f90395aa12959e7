"""The learned MLP ensemble behind the interface of general_collection_oracle.py (test infrastructure, beside
oracle/mbpo_oracle.py, which it reuses unchanged): ``EnsembleOracle(params, member).step(x, u, keys)`` is
``mlp_ensemble_step(x, u, member, params, bf16=True)`` -- x_next = x + MLP_m([x, u]) with the tensor-core operand
rounding, the reward the pendulum reward on (x, u) -- with env e rolled through member[e] (member 0 when member is
None).  The System draws nothing, so keys pass through; system_env_rollout / system_actor_rollout step it as any
other System."""
from __future__ import annotations

from typing import Optional

import numpy as np

from oracle.mbpo_oracle import F32, MlpEnsembleParams, mlp_ensemble_step


class EnsembleOracle:
    x_dim, u_dim, keyed = 3, 1, False

    def __init__(self, params: MlpEnsembleParams, member: Optional[np.ndarray] = None, bf16: bool = True):
        self.params, self.bf16 = params, bf16
        self.member = None if member is None else np.asarray(member, dtype=np.int32).reshape(-1)

    def members(self, rows: int) -> np.ndarray:
        if self.member is None:
            return np.zeros(rows, dtype=np.int32)
        if self.member.shape[0] != rows:
            raise ValueError("%d members for %d rows" % (self.member.shape[0], rows))
        return self.member

    def step(self, x, u, keys=None, partitionable=False, dtype=F32):
        """x [R,3], u [R,1] -> (x_next [R,3], reward [R], keys): row r through member[r]."""
        x = np.asarray(x, dtype=F32)
        u = np.asarray(u, dtype=F32).reshape(x.shape[0], -1)
        xn, r = mlp_ensemble_step(x, u[:, 0], self.members(x.shape[0]), self.params, self.bf16)
        return xn.astype(dtype), r.astype(dtype), keys
