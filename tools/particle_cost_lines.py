"""One JSON line per case: iCemTO with a constraint cost over distinct particles (mbpo_ensemble_rollout_transitions /
mbpo_system_objective with particle buffers -> the torch cost -> mbpo_icem_penalize_particles).

  plan cases   iCemTO.optimize per call, the same plan without a cost beside it, and with a speed-limit cost
               (max_t |x_t[-1]| - limit) summarised by the mean and by the max (use_pessimism):
    ensemble       BASELINE config 4: 36 problems, 5 members (particles), num_samples 1,024, H 50, 5 iterations
                   (the plan without a cost is the library's staged plan);
    noisy pendulum B = 64 and 4,096, P = 10, num_samples 512, H 30, 5 iterations (without a cost: the fused plan).
  kernel cases mbpo_ensemble_rollout_transitions against mbpo_ensemble_rollout on 37,404 rows (config 4: the two-tile
               kernel) and 18,944 rows (the one-tile kernel), H 50, with the bytes the buffers add.
  split        a separate torch.profiler run of one plan per cost case: CUDA time of the library's kernels (mbpo::)
               and of everything else (the torch cost).

Timing: CUDA events around one call, warm-ups first, the L2 flushed (256 MiB memset) before every timed pass, as
bench.py does; the card name, power limit and SM clocks are read in the same process.
Usage:  python tools/particle_cost_lines.py OUT_DIR [--passes 10] [--warmup 2]
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
from mbpo_b200 import _lib as L  # noqa: E402
from mbpo_b200.optimizers import iCemParams, iCemTO  # noqa: E402
from mbpo_b200.systems import (MLPEnsembleSystem, MlpEnsembleDynamicsParams, NoisyPendulumSystem,  # noqa: E402
                               PendulumRewardParams, SystemParams)
from oracle import mbpo_oracle as orc  # noqa: E402


class SpeedLimit:
    def __init__(self, limit):
        self.limit = limit

    def __call__(self, states, actions):
        return states[:, -1].abs().max() - self.limit


def card(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0),
                        "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(dev),
            "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": q.stdout.strip() or None}


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
    return {"median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms))}


def split(fn):
    """CUDA time of one call under torch.profiler: the library's kernels vs everything else."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    lib = other = 0.0
    names = {}
    for ev in prof.key_averages():
        us = ev.self_device_time_total if hasattr(ev, "self_device_time_total") else ev.self_cuda_time_total
        if us <= 0:
            continue
        if "mbpo" in ev.key:
            lib += us
            names[ev.key.split("(")[0][-80:]] = round(us / 1e3, 3)
        else:
            other += us
    return {"library_kernels_ms": lib / 1e3, "torch_cost_and_other_ms": other / 1e3, "library_kernels": names}


def ensemble_system(dev):
    ens = orc.make_mlp_ensemble(seed=3, members=5)
    d = lambda a: torch.from_numpy(a).to(dev)
    dyn = MlpEnsembleDynamicsParams(weights=[d(w) for w in ens.weights], biases=[d(b) for b in ens.biases])
    return MLPEnsembleSystem(dynamics_params=dyn), SystemParams(dynamics_params=dyn, reward_params=PendulumRewardParams())


def states(n, seed, dev):
    rng = np.random.default_rng(seed)
    th, w = rng.uniform(-np.pi, np.pi, n), rng.uniform(-8, 8, n)
    return torch.from_numpy(np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)).to(dev)


def plan_lines(name, system, B, params, horizon, dev, args, flush, meta):
    x0 = states(B, 1, dev)
    keys = mbpo_b200.random.split(mbpo_b200.random.PRNGKey(0, dev), B)
    out = []
    cost = SpeedLimit(4.0)
    for label, c, pes in (("no_cost", None, False), ("cost_mean", cost, False), ("cost_pessimism", cost, True)):
        opt = iCemTO(horizon=horizon, action_dim=1, opt_params=iCemParams(**params), cost_fn=c, use_pessimism=pes)
        opt.set_system(system)
        st = opt.init(keys)
        fn = lambda: opt.optimize(x0, st)
        t = timed(fn, args.passes, args.warmup, flush)
        M = params["num_samples"] + max(int(0.3 * params.get("num_elites", 50)), 1)
        line = dict(meta, case=name, variant=label, B=B, horizon=horizon, params=params, ms_per_plan=t,
                    buffer_bytes_per_iteration=(4 * B * M * params["num_particles"] * horizon * 4) if c else 0)
        if c is not None:
            line["profile_split_one_plan"] = split(fn)
        out.append(line)
    return out


def kernel_lines(dev, args, flush, meta):
    system, sp = ensemble_system(dev)
    pk = system.packed(sp)
    out = []
    H, E = 50, 5
    for B, M in ((36, 1039), (1, 18944)):
        R = B * M
        x0 = states(B, 2, dev)
        acts = torch.rand((B, M, H, 1), device=dev) * 2 - 1
        ret = torch.empty((B, M), device=dev)
        obs = torch.empty((B, M, E, H, 3), device=dev)
        rew = torch.empty((B, M, E, H), device=dev)
        st = L.stream_ptr(dev)
        f_ret = lambda: L.check(L.lib.mbpo_ensemble_rollout(L.C.byref(pk.struct), H, L.ptr(x0), L.ptr(acts), B, M, 0,
                                                            L.ptr(ret), st))
        f_tr = lambda: L.check(L.lib.mbpo_ensemble_rollout_transitions(L.C.byref(pk.struct), H, L.ptr(x0), L.ptr(acts),
                                                                       B, M, L.ptr(obs), L.ptr(rew), st))
        t = {}
        for rep in range(3):                      # alternate the two kernels
            for label, fn in (("ensemble_rollout", f_ret), ("ensemble_rollout_transitions", f_tr)):
                t.setdefault(label, []).append(timed(fn, args.passes, args.warmup, flush)["median_ms"])
        a, b = float(np.median(t["ensemble_rollout"])), float(np.median(t["ensemble_rollout_transitions"]))
        out.append(dict(meta, case="ensemble_kernel", rows=R, horizon=H, members=E,
                        ms_ensemble_rollout=a, ms_ensemble_rollout_transitions=b, added_fraction=(b - a) / a,
                        alternations_ms=t, buffer_bytes_written=4 * R * E * H * 4,
                        kernel=("one-tile" if R <= 18944 else "two-tile")))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("particle_cost_lines: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(args.out_dir, exist_ok=True)
    meta = {"card": card(dev), "l2": "flushed (256 MiB memset) before every timed pass"}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    lines = kernel_lines(dev, args, flush, meta)
    ens_sys, _ = ensemble_system(dev)
    lines += plan_lines("ensemble_config4", ens_sys, 36, dict(num_samples=1024, num_particles=5, num_steps=5), 50,
                        dev, args, flush, meta)
    for B in (64, 4096):
        lines += plan_lines("noisy_pendulum_B%d" % B, NoisyPendulumSystem(0.05), B,
                            dict(num_samples=512, num_particles=10, num_steps=5), 30, dev, args, flush, meta)
    with open(os.path.join(args.out_dir, "particle_cost_lines.jsonl"), "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps(ln), flush=True)


if __name__ == "__main__":
    main()
