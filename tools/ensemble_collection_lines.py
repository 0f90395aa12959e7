"""One JSON line per case: the learned MLP ensemble as a SAC / PPO env (mbpo_ensemble_env_rollout).

  per case     E envs x T wrapped steps (action_repeat 1) of a 5-member ensemble, members contiguous (e * 5 // E) or
               interleaved (e % 5), timed three ways in one process:
    policy         get_experience with the SAC policy (2 x 64 hidden) in the loop;
    actions_given  env.unroll with the actions that policy run produced (the same model steps, no policy);
    ensemble_returns  MLPEnsembleSystem.ensemble_returns over E // 5 rows x 5 members x H = T: the iCEM kernel at
                   (nearly) the same rows x steps, as the nearest measured reference.
  cases        E = 18,944 (74 CTA pairs x 256 rows: one round of the one-tile schedule when the tiles fill) and
               E = 65,536 at T = 200 with episode_length 200; an MBPO-style branch: 262,144 envs reset from a true
               buffer by BraxWrapper, T = 5.
Model FLOP per model step and row: 2 x (4 x 256 + 256 x 256 x 2 + 256 x 3) = 265,728 (multiply-adds x 2).

Timing: CUDA events around one call, warm-ups first, the L2 flushed (256 MiB memset) before every timed pass; the card
name, power limit and SM clocks are read in the same process.
Usage:  python tools/ensemble_collection_lines.py [--passes 10] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "model-based-policy-optimizers_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import mbpo_b200  # noqa: E402
from mbpo_b200 import acting, envs  # noqa: E402
from mbpo_b200.systems import (BraxWrapper, MLPEnsembleSystem, MlpEnsembleDynamicsParams,  # noqa: E402
                               PendulumRewardParams, SystemParams)
from oracle import jax_prng as ojr  # noqa: E402
from oracle import mbpo_oracle as orc  # noqa: E402

FLOP_PER_MODEL_STEP = 2 * (4 * 256 + 256 * 256 * 2 + 256 * 3)
MEMBERS = 5


def card(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0),
                        "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_sm_clock_max_sm_clock":
            q.stdout.strip() or None}


def timed(fn, passes, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(passes):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ms.append(s.elapsed_time(e))
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def ensemble(dev, member):
    ens = orc.make_mlp_ensemble(seed=3, members=MEMBERS)
    d = lambda a: torch.from_numpy(a).to(dev)
    dyn = MlpEnsembleDynamicsParams(weights=[d(w) for w in ens.weights], biases=[d(b) for b in ens.biases],
                                    member=member)
    return MLPEnsembleSystem(), SystemParams(dynamics_params=dyn, reward_params=PendulumRewardParams())


def policy(dev):
    pol = orc.make_policy_params(seed=7, obs_dim=3, action_dim=1, hidden=(64, 64))
    d = lambda a: torch.from_numpy(a).to(dev)
    return acting.Policy(acting.PolicyParams([d(w) for w in pol.weights], [d(b) for b in pol.biases]))


def true_buffer_env(system, params, dev, episode_length):
    from mbpo_b200.replay_buffers import UniformSamplingQueue
    from mbpo_b200.utils.optimizer_utils import Transition
    z = lambda *s: torch.zeros(s, device=dev)
    dummy = Transition(z(3), z(1), z(), z(), z(3), {"state_extras": {"truncation": z()}, "policy_extras": {}})
    q = UniformSamplingQueue(4096, dummy, 1)
    rng = np.random.default_rng(4)
    th, w = rng.uniform(-np.pi, np.pi, 4096), rng.uniform(-8, 8, 4096)
    obs = torch.from_numpy(np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)).to(dev)
    st = q.insert(q.init(torch.from_numpy(ojr.PRNGKey(0)).to(dev)),
                  Transition(obs, z(4096, 1), z(4096), z(4096) + 1, obs, {"state_extras": {"truncation": z(4096)},
                                                                           "policy_extras": {}}))
    return envs.wrap(BraxWrapper(system, params, st, q), episode_length, 1)


def run_case(dev, E, T, episode_length, layout, from_buffer, passes, warmup, flush):
    idx = torch.arange(E, dtype=torch.int32, device=dev)
    member = idx * MEMBERS // E if layout == "contiguous" else idx % MEMBERS
    system, params = ensemble(dev, member.to(torch.int32).contiguous())
    pol = policy(dev)
    key = torch.from_numpy(ojr.PRNGKey(4)).to(dev)
    if from_buffer:
        env = true_buffer_env(system, params, dev, episode_length)
        from mbpo_b200 import random as jr
        st = env.reset(jr.split(torch.from_numpy(ojr.PRNGKey(9)).to(dev), E))
    else:
        env = envs.wrap(system, params, episode_length=episode_length)
        rng = np.random.default_rng(1)
        th, w = rng.uniform(-np.pi, np.pi, E), rng.uniform(-8, 8, E)
        st = env.reset(torch.from_numpy(np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)).to(dev))
    st = st.replace(system_params=params)
    _, _, tr = acting.get_experience(env, st, pol, key, T)
    actions = tr.action.clone()
    t_pol = timed(lambda: acting.get_experience(env, st, pol, key, T), passes, warmup, flush)
    t_act = timed(lambda: env.unroll(st, actions), passes, warmup, flush)
    R = E // MEMBERS                                 # rows, each through all 5 members: R x 5 x T model steps
    x0 = st.obs[:R].contiguous()
    acts = actions[:, :R, 0].t().reshape(R, 1, T, 1).contiguous()
    t_ref = timed(lambda: system.ensemble_returns(params, x0, acts), passes, warmup, flush)
    model_steps = E * T
    ref_steps = R * MEMBERS * T
    line = {"case": "mbpo_branch_true_buffer" if from_buffer else "env_rollouts", "envs": E, "steps": T,
            "episode_length": episode_length, "action_repeat": 1, "members": MEMBERS, "member_layout": layout,
            "policy": "NormalTanh, 2 x 64 hidden, SAC keys (get_experience)",
            "policy_ms_median": t_pol[0], "policy_ms_min": t_pol[1], "policy_ms_max": t_pol[2],
            "policy_env_steps_per_s": model_steps / (t_pol[0] * 1e-3),
            "policy_model_tflops": model_steps * FLOP_PER_MODEL_STEP / (t_pol[0] * 1e-3) / 1e12,
            "actions_given_ms_median": t_act[0], "actions_given_ms_min": t_act[1], "actions_given_ms_max": t_act[2],
            "actions_given_env_steps_per_s": model_steps / (t_act[0] * 1e-3),
            "actions_given_model_tflops": model_steps * FLOP_PER_MODEL_STEP / (t_act[0] * 1e-3) / 1e12,
            "policy_share_of_step": 1.0 - t_act[0] / t_pol[0],
            "ensemble_returns_rows_x_members_x_H": [R, MEMBERS, T],
            "ensemble_returns_ms_median": t_ref[0],
            "ensemble_returns_model_tflops": ref_steps * FLOP_PER_MODEL_STEP / (t_ref[0] * 1e-3) / 1e12,
            "tiles": int(sum(-(-int(c) // 256) for c in np.bincount(member.cpu().numpy(), minlength=MEMBERS))),
            "cta_pairs": min(torch.cuda.get_device_properties(dev).multi_processor_count // 2,
                             (E + 255) // 256 + MEMBERS - 1),
            "flop_per_model_step": FLOP_PER_MODEL_STEP, "passes": passes, "warmup": warmup,
            "l2": "flushed (256 MiB memset) before every timed pass", "timing": "CUDA events around one call"}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_collection_lines: no CUDA device (a time needs the GPU)")
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    info = card(dev)
    cases = [(18944, 200, 200, "contiguous", False), (18944, 200, 200, "interleaved", False),
             (65536, 200, 200, "contiguous", False), (65536, 200, 200, "interleaved", False),
             (262144, 5, 1000, "interleaved", True)]
    out = open(args.out, "w") if args.out else None
    for E, T, L, layout, buf in cases:
        line = run_case(dev, E, T, L, layout, buf, args.passes, args.warmup, flush)
        line["card"] = info
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
