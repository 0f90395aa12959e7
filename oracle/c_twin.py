"""ORACLE (test infrastructure, NOT product code) -- ctypes loader for the plain-C twin
(oracle/c/mbpo_oracle.c).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c")
LIB = os.path.join(_DIR, "libmbpo_oracle.so")


class OrcIcemCfg(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("horizon", "num_samples", "num_elites", "num_prev_elites", "num_particles",
                                       "num_steps", "warm_start", "partitionable", "summarize_max")] + \
               [(n, C.c_float) for n in ("init_std", "alpha", "exponent", "u_min", "u_max")]


def build(native: bool = False, out: str | None = None) -> str:
    """Compiles the twin.  native=True adds -march=native (for timing on the machine it runs on)."""
    if not native:
        subprocess.run(["make", "-s", "-C", _DIR], check=True)
        return LIB
    out = out or os.path.join(_DIR, "libmbpo_oracle_native.so")
    subprocess.run(["/usr/bin/gcc", "-O3", "-march=native", "-ffp-contract=off", "-fno-math-errno", "-fopenmp", "-fPIC",
                    "-shared", "-o", out, os.path.join(_DIR, "mbpo_oracle.c"), "-lm"], check=True)
    return out


def load(native: bool = False) -> C.CDLL:
    if native:
        # built in a temporary directory, so that the tree stays untouched (it may be read-only); the loaded
        # library outlives its deleted file
        with tempfile.TemporaryDirectory(prefix="mbpo_oracle_") as tmp:
            try:
                return _declare(C.CDLL(build(native=True, out=os.path.join(tmp, "libmbpo_oracle_native.so"))))
            except Exception:
                pass
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(os.path.join(_DIR, "mbpo_oracle.c")):
        build()
    return _declare(C.CDLL(LIB))


def _declare(lib: C.CDLL) -> C.CDLL:
    lib.orc_icem_optimize_batch.restype = C.c_int
    lib.orc_env_rollout.restype = C.c_int
    lib.orc_max_threads.restype = C.c_int
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def make_cfg(params, horizon: int, partitionable: bool = False, use_optimism: bool = False) -> OrcIcemCfg:
    return OrcIcemCfg(horizon, params.num_samples, params.num_elites, params.num_prev_elites, params.num_particles,
                      params.num_steps, int(params.warm_start), int(partitionable), int(use_optimism),
                      params.init_std, params.alpha, params.exponent, params.u_min, params.u_max)


def optimize_batch(lib, cfg: OrcIcemCfg, params9, x0, keys, best_seq, num_threads: int = 0):
    B = x0.shape[0]
    x0 = np.ascontiguousarray(x0, np.float32)
    keys = np.ascontiguousarray(keys, np.uint32)
    best_seq = np.ascontiguousarray(best_seq, np.float32).reshape(B, cfg.horizon)
    o_seq = np.empty((B, cfg.horizon), np.float32)
    o_val = np.empty(B, np.float32)
    o_key = np.empty((B, 2), np.uint32)
    p9 = np.ascontiguousarray(params9, np.float32)
    used = lib.orc_icem_optimize_batch(C.byref(cfg), _p(p9), _p(x0), _p(keys), _p(best_seq), B, _p(o_seq), _p(o_val),
                                       _p(o_key), num_threads)
    return o_seq, o_val, o_key, used


def closed_loop(lib, cfg: OrcIcemCfg, params9, x0, key, best_seq, T: int):
    states = np.empty((T, 3), np.float32)
    rewards = np.empty(T, np.float32)
    actions = np.empty(T, np.float32)
    o_seq = np.empty(cfg.horizon, np.float32)
    o_key = np.empty(2, np.uint32)
    p9 = np.ascontiguousarray(params9, np.float32)
    x0 = np.ascontiguousarray(x0, np.float32)
    key = np.ascontiguousarray(key, np.uint32)
    best_seq = np.ascontiguousarray(best_seq, np.float32).reshape(-1)
    lib.orc_icem_closed_loop(C.byref(cfg), _p(p9), _p(x0), _p(key), _p(best_seq), T, _p(states), _p(rewards),
                             _p(actions), _p(o_seq), _p(o_key))
    return states, rewards, actions, o_seq, o_key


def env_rollout(lib, params9, x0, actions, episode_length: int, action_repeat: int = 1, num_threads: int = 0,
                outputs: bool = True):
    T, E = actions.shape
    obs = np.ascontiguousarray(x0, np.float32).copy()
    first = obs.copy()
    steps = np.zeros(E, np.float32)
    done = np.zeros(E, np.float32)
    actions = np.ascontiguousarray(actions, np.float32)
    p9 = np.ascontiguousarray(params9, np.float32)
    out = {}
    if outputs:
        out = dict(observation=np.empty((T, E, 3), np.float32), reward=np.empty((T, E), np.float32),
                   discount=np.empty((T, E), np.float32), next_observation=np.empty((T, E, 3), np.float32),
                   truncation=np.empty((T, E), np.float32))
    g = lambda n: _p(out[n]) if outputs else None
    used = lib.orc_env_rollout(_p(p9), episode_length, action_repeat, _p(obs), _p(steps), _p(done), _p(first),
                               _p(actions), E, T, g("observation"), g("reward"), g("discount"),
                               g("next_observation"), g("truncation"), num_threads)
    out.update(final_obs=obs, final_steps=steps, final_done=done, threads=used)
    return out
