"""One JSON line per case: SAC / PPO collection for the general Systems beside the pendulum, in one process.

  env rollouts     65,536 envs x 1,000 wrapped steps (episode_length 200, as bench.py config 3), actions from
                   default_rng(2), one launch per pass into preallocated Transition buffers (observation and
                   next_observation as overlapping views of one [T+1, E, X] buffer), for each System;
  get_experience   200 steps at 65,536 envs, the SAC policy (3 x 64 hidden) in the loop, for each System.

Timing: CUDA events around each pass, warm-ups first, the L2 flushed (256 MiB memset) before every timed pass.
Bytes per transition come from shapes: actions read (4 A) + next_observation (4 X), reward, discount and truncation
(12) written.  The bound of an env rollout: "hbm" when it moves at least 60% of the device-to-device copy bandwidth
measured in the same process, otherwise "issue" (the SM instruction stream, not memory, sets its time).
Usage:  python tools/general_collection_lines.py [--passes 10] [--warmup 3] [--out FILE]
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
from mbpo_b200.systems import NoisyPendulumSystem, PendulumSystem, PointMassSystem  # noqa: E402
from mbpo_b200.systems.base_systems import SystemParams  # noqa: E402
from oracle import mbpo_oracle as orc  # noqa: E402

E, T, EPISODE, EXP_T = 65536, 1000, 200, 200


def card(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip() or None}


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


def systems(dev):
    rng = np.random.default_rng(1)
    th, w = rng.uniform(-np.pi, np.pi, E), rng.uniform(-8, 8, E)
    x_pend = np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)
    keys = torch.from_numpy(rng.integers(0, 2 ** 32, (E, 2), dtype=np.uint64).astype(np.uint32)).to(dev)
    pend = PendulumSystem()
    noisy = NoisyPendulumSystem(noise_std=0.05)
    pm = PointMassSystem()
    return [("pendulum", pend, pend.reset(device=dev).system_params, x_pend),
            ("noisy_pendulum", noisy, noisy.init_params(mbpo_b200.random.PRNGKey(1, dev)).replace(key=keys), x_pend),
            ("point_mass", pm, SystemParams(), rng.uniform(-2, 2, (E, 4)).astype(np.float32))]


def env_line(name, system, params, x0, dev, args, flush, copy_bw, info):
    X, A = system.x_dim, system.u_dim
    env = envs.wrap(system, params, episode_length=EPISODE)
    st = env.reset(torch.from_numpy(x0).to(dev)).replace(system_params=params)
    acts = torch.from_numpy(np.random.default_rng(2).uniform(-1, 1, (T, E, A)).astype(np.float32)).to(dev)
    buf = torch.empty((T + 1, E, X), device=dev)
    r, d, tr = (torch.empty((T, E), device=dev) for _ in range(3))
    pk = system.pack_params(params)
    keyed = envs.is_general(system) and system.keyed
    # the env state ping-pongs between two buffer sets (the unroll reads one and writes the other)
    state = [[st.obs.clone(), st.info["steps"].clone(), st.done.clone(), params.key.clone() if keyed else None]
             for _ in range(2)]
    flip = [0]
    L = mbpo_b200._lib

    def launch():
        src, dst = state[flip[0]], state[flip[0] ^ 1]
        flip[0] ^= 1
        env._launch(pk, src[0], src[1], src[2], src[3], dst[0], dst[1], dst[2], dst[3], st.info["first_obs"],
                    L.ptr(acts), E, T, L.ptr(r), L.ptr(d), L.ptr(buf[1:]), L.ptr(tr), L.stream_ptr(dev))
    med, lo, hi = timed(launch, args.passes, args.warmup, flush)
    rate = E * T / (med * 1e-3)
    bpt = 4 * A + 4 * X + 12
    bw = rate * bpt
    return {"case": "env_rollouts", "system": name, "envs": E, "steps": T, "episode_length": EPISODE,
            "x_dim": X, "action_dim": A, "keyed": bool(keyed), "ms_per_launch_median": med, "ms_min": lo, "ms_max": hi,
            "env_steps_per_s": rate, "bytes_per_transition": bpt, "achieved_bytes_per_s": bw,
            "frac_of_copy_bw": bw / copy_bw, "frac_of_hbm_datasheet_7p7TBs": bw / 7.7e12,
            "bound": "hbm" if bw >= 0.6 * copy_bw else "issue",
            "kernel": "env_unroll_general_kernel" if envs.is_general(system) else "env_rollout_pendulum_kernel (pieces)",
            "passes": args.passes, "warmup": args.warmup, "l2": "flushed (256 MiB memset) before every timed pass",
            "timing": "CUDA events around one launch", **info}


def experience_line(name, system, params, x0, dev, args, flush, info):
    X, A = system.x_dim, system.u_dim
    pol = orc.make_policy_params(seed=7, obs_dim=X, action_dim=A, hidden=(64, 64, 64))
    policy = acting.Policy(acting.PolicyParams([torch.from_numpy(w).to(dev) for w in pol.weights],
                                               [torch.from_numpy(b).to(dev) for b in pol.biases]))
    env = envs.wrap(system, params, episode_length=EPISODE)
    st = env.reset(torch.from_numpy(x0).to(dev)).replace(system_params=params)
    key = mbpo_b200.random.PRNGKey(0, dev)
    med, lo, hi = timed(lambda: acting.get_experience(env, st, policy, key, EXP_T), args.passes, args.warmup, flush)
    return {"case": "get_experience", "system": name, "envs": E, "steps": EXP_T, "policy_hidden": [64, 64, 64],
            "ms_per_call_median": med, "ms_min": lo, "ms_max": hi, "env_steps_per_s": E * EXP_T / (med * 1e-3),
            "kernel": "actor_rollout_general_kernel (CUDA cores)" if envs.is_general(system)
            else "tcgen05 policy kernel (MBPO_ACTOR_AUTO)",
            "passes": args.passes, "warmup": args.warmup, "l2": "flushed (256 MiB memset) before every timed pass",
            "timing": "CUDA events around one get_experience call (allocations from the caching allocator included)",
            **info}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("general_collection_lines: no CUDA device (these are GPU measurements)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    # device-to-device copy bandwidth of a 1 GiB buffer: the reference for "HBM-bound"
    src, dst = torch.empty(1 << 28, device=dev), torch.empty(1 << 28, device=dev)
    cmed, _, _ = timed(lambda: dst.copy_(src), 10, 3, flush)
    copy_bw = 2 * src.numel() * 4 / (cmed * 1e-3)
    del src, dst
    info = {"card": card(dev), "copy_bw_bytes_per_s": copy_bw}
    lines = []
    for name, system, params, x0 in systems(dev):
        lines.append(env_line(name, system, params, x0, dev, args, flush, copy_bw, info))
        print(json.dumps(lines[-1]), flush=True)
        torch.cuda.empty_cache()
    for name, system, params, x0 in systems(dev):
        lines.append(experience_line(name, system, params, x0, dev, args, flush, info))
        print(json.dumps(lines[-1]), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
