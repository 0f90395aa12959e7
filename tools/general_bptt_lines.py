"""One JSON line per System: BPTT's rollout and its cotangent pass for the general Systems beside the pendulum, in one
process.

  shape     65,536 initial states x H = 20 (the shape of bench.py --workload bptt_rollout_grad), BPTT's actor
            X-64-64-2A (swish, normalised observations), NoisyPendulum with one System key shared by the batch;
  stages    rollout_policy (forward), lambda_return, lambda_return_vjp (its transpose), rollout_policy_vjp (adjoint),
            each timed on its own, and the four in sequence.

Timing: CUDA events around each stage, warm-ups first, the L2 flushed (256 MiB memset) before every timed pass; the
median over the passes.  Transitions/s = 65,536 x 20 over the time of the four stages in sequence.
Usage:  python tools/general_bptt_lines.py [--passes 20] [--warmup 3] [--out FILE]
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
from mbpo_b200 import acting  # noqa: E402
from mbpo_b200.systems import NoisyPendulumSystem, PendulumSystem, PointMassSystem  # noqa: E402
from mbpo_b200.systems.base_systems import SystemParams  # noqa: E402
from mbpo_b200.utils.optimizer_utils import (lambda_return, lambda_return_vjp, rollout_policy,  # noqa: E402
                                             rollout_policy_vjp)
from oracle import mbpo_oracle as orc  # noqa: E402

B, H, DISCOUNT, LAMBDA = 65536, 20, 0.99, 0.95


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
    th, w = rng.uniform(-np.pi, np.pi, B), rng.uniform(-8, 8, B)
    x_pend = np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)
    pend, noisy, pm = PendulumSystem(), NoisyPendulumSystem(noise_std=0.05), PointMassSystem()
    return [("pendulum", pend, pend.reset(device=dev).system_params, x_pend),
            ("noisy_pendulum", noisy, noisy.init_params(mbpo_b200.random.PRNGKey(1, dev)), x_pend),
            ("point_mass", pm, SystemParams(), rng.uniform(-2, 2, (B, 4)).astype(np.float32))]


def line(name, system, params, x0, dev, args, flush, info):
    X, A = system.x_dim, system.u_dim
    pol = orc.make_policy_params(seed=7, obs_dim=X, action_dim=A, hidden=(64, 64))
    policy = acting.BpttActorPolicy(acting.PolicyParams([torch.from_numpy(w).to(dev) for w in pol.weights],
                                                        [torch.from_numpy(b).to(dev) for b in pol.biases]),
                                    init_stddev=2.0, obs_mean=[0.0] * X, obs_std=[1.0] * X)
    xs = torch.from_numpy(x0).to(dev)
    key = mbpo_b200.random.PRNGKey(0, dev)
    wv = torch.from_numpy(np.linspace(-0.3, 0.3, X).astype(np.float32)).to(dev)
    g_lv = torch.from_numpy(np.random.default_rng(3).standard_normal((B, H)).astype(np.float32)).to(dev)
    tr = rollout_policy(system, params, xs, policy, key, H)
    nv = (tr.next_observation @ wv).contiguous()
    g_r, g_nv = lambda_return_vjp(g_lv, DISCOUNT, LAMBDA)
    g_next = (g_nv[..., None] * wv).contiguous()
    t_fwd = timed(lambda: rollout_policy(system, params, xs, policy, key, H), args.passes, args.warmup, flush)
    t_lam = timed(lambda: lambda_return(tr.reward, nv, DISCOUNT, LAMBDA), args.passes, args.warmup, flush)
    t_lamT = timed(lambda: lambda_return_vjp(g_lv, DISCOUNT, LAMBDA), args.passes, args.warmup, flush)
    t_adj = timed(lambda: rollout_policy_vjp(system, params, tr, g_reward=g_r, g_next_observation=g_next),
                  args.passes, args.warmup, flush)

    def pipeline():
        t = rollout_policy(system, params, xs, policy, key, H)
        lambda_return(t.reward, (t.next_observation @ wv), DISCOUNT, LAMBDA)
        gr, gn = lambda_return_vjp(g_lv, DISCOUNT, LAMBDA)
        rollout_policy_vjp(system, params, t, g_reward=gr, g_next_observation=gn[..., None] * wv)
    t_all = timed(pipeline, args.passes, args.warmup, flush)
    general = system.system_kind in (mbpo_b200._lib.SYSTEM_NOISY_PENDULUM, mbpo_b200._lib.SYSTEM_POINT_MASS)
    ms = lambda t: {"median": t[0], "min": t[1], "max": t[2]}                  # noqa: E731
    return {"case": "bptt_rollout_grad", "system": name, "initial_states": B, "horizon": H, "x_dim": X,
            "action_dim": A, "policy": "BPTT actor %d-64-64-%d swish" % (X, 2 * A),
            "system_key": "one [2] key shared by the batch" if getattr(system, "keyed", False) else None,
            "forward_ms": ms(t_fwd), "lambda_return_ms": ms(t_lam), "lambda_return_vjp_ms": ms(t_lamT),
            "adjoint_ms": ms(t_adj), "pipeline_ms": ms(t_all),
            "transitions_per_s": B * H / (t_all[0] * 1e-3),
            "forward_kernel": "rollout_policy_general_kernel (CUDA cores)" if general
            else "tcgen05 policy kernel (MBPO_ACTOR_AUTO)",
            "adjoint_kernel": "rollout_adjoint_general_kernel" if general else "rollout_adjoint_pendulum_kernel",
            "passes": args.passes, "warmup": args.warmup, "l2": "flushed (256 MiB memset) before every timed pass",
            "timing": "CUDA events around each stage; pipeline = the four stages in sequence, with the small "
                      "elementwise ops between them (the critic v(x) = w . x)", **info}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("general_bptt_lines: no CUDA device (these are GPU measurements)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    info = {"card": card(dev)}
    lines = []
    for name, system, params, x0 in systems(dev):
        lines.append(line(name, system, params, x0, dev, args, flush, info))
        print(json.dumps(lines[-1]), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
