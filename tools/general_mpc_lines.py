"""One JSON line per case: thread-block-cluster plans and the one-launch closed loop over the general Systems.

  plan cases    one fused plan (mbpo_icem_plan_clustered) for B = 1, 8, 64 at every cluster size (1 = one CTA per
                problem, 2, 4, 8, 16, and the library's choice -1), for NoisyPendulumSystem (P = 10 particles) and
                PointMassSystem, num_samples 512, H 30, 5 iterations (iCemParams defaults otherwise).
  closed loop   200 MPC steps at iCemParams() defaults, H 20, B = 1: iCemTO.closed_loop (one launch) against
                iCemTO._closed_loop_staged (a plan call and a System.step launch per step), for both Systems.

Timing: CUDA events around one call, warm-ups first, the L2 flushed (256 MiB memset) before every timed plan pass;
the card name, power limit and SM clocks are read in the same process and written on every line.
Usage:  python tools/general_mpc_lines.py OUT_FILE [--passes 10] [--warmup 2]
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

from mbpo_b200 import _lib as L  # noqa: E402
from mbpo_b200.optimizers import iCemParams, iCemTO  # noqa: E402
from mbpo_b200.systems import NoisyPendulumSystem, PointMassSystem  # noqa: E402


def card(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0),
                        "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(dev),
            "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": q.stdout.strip() or None}


def timed(fn, passes, warmup, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(passes):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}


def make(kind, H, params):
    system = NoisyPendulumSystem(0.05) if kind == "noisy_pendulum" else PointMassSystem()
    opt = iCemTO(horizon=H, action_dim=system.u_dim, opt_params=params)
    opt.set_system(system)
    return opt, system


def states(kind, B, dev, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "noisy_pendulum":
        th, w = rng.uniform(-np.pi, np.pi, B), rng.uniform(-8, 8, B)
        x = np.stack([np.cos(th), np.sin(th), w], axis=-1)
    else:
        x = rng.uniform(-1.5, 1.5, (B, 4))
    return torch.from_numpy(x.astype(np.float32)).to(dev)


def keys(B, dev, seed=1):
    k = np.random.default_rng(seed).integers(0, 2 ** 32, size=(B, 2), dtype=np.uint64).astype(np.uint32)
    return torch.from_numpy(k).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("general_mpc_lines: no CUDA device; nothing is measured without one")
    dev = torch.device("cuda", 0)
    info = card(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        def emit(rec):
            rec = {"card": info, **rec}
            f.write(json.dumps(rec) + "\n")
            f.flush()
            print(json.dumps(rec), flush=True)

        for kind, P in (("noisy_pendulum", 10), ("point_mass", 1)):
            params = iCemParams(num_samples=512, num_particles=P, num_steps=5)
            opt, system = make(kind, 30, params)
            for B in (1, 8, 64):
                st = opt.init(keys(B, dev))
                x0 = states(kind, B, dev)
                chosen = L.lib.mbpo_icem_plan_cluster_size(L.C.byref(opt._cfg()), B)
                ref = None
                for cluster in (1, 2, 4, 8, 16, -1):
                    def run():
                        return opt._plan_raw(x0, st.key, st.best_sequence, st.system_params, cluster=cluster)
                    try:
                        out = run()
                    except L.MbpoUnsupported as e:
                        emit({"case": "plan", "system": kind, "B": B, "cluster": cluster, "num_samples": 512,
                              "num_particles": P, "horizon": 30, "num_steps": 5, "supported": False, "why": str(e)})
                        continue
                    if ref is None:
                        ref = out
                    same = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(out[:3], ref[:3]))
                    emit({"case": "plan", "system": kind, "B": B, "cluster": cluster,
                          "library_choice": chosen if cluster == -1 else None, "num_samples": 512,
                          "num_particles": P, "horizon": 30, "num_steps": 5, "supported": True,
                          "bits_equal_to_one_cta": same, "l2": "flushed (256 MiB memset) before every timed pass",
                          "ms_per_plan": timed(run, args.passes, args.warmup, flush)})

        T = 200
        for kind in ("noisy_pendulum", "point_mass"):
            opt, system = make(kind, 20, iCemParams())
            st = opt.init(keys(1, dev)[0])
            x0 = states(kind, 1, dev)[0]

            def one_launch():
                return opt.closed_loop(x0, st, T)

            def staged():
                single, xc, kc, sc = opt._canon(x0, st)
                return opt._closed_loop_staged(single, xc, kc, sc, st, T)
            a, b = one_launch(), staged()
            same = all(torch.equal(u.contiguous().view(torch.int32), v.contiguous().view(torch.int32))
                       for u, v in zip(a[:3], b[:3]))
            rec = {"case": "closed_loop", "system": kind, "B": 1, "mpc_steps": T, "horizon": 20,
                   "params": "iCemParams() defaults", "bits_equal": same,
                   "library_choice": L.lib.mbpo_icem_plan_cluster_size(L.C.byref(opt._cfg()), 1),
                   "l2": "not flushed (one call is 200 plans)"}
            # alternate the two paths; the staged loop is long, so fewer passes
            rec["ms_one_launch"] = timed(one_launch, max(3, args.passes // 2), 1)
            rec["ms_staged"] = timed(staged, 3, 1)
            rec["ms_one_launch_again"] = timed(one_launch, max(3, args.passes // 2), 1)
            rec["speedup_median"] = rec["ms_staged"]["median_ms"] / rec["ms_one_launch"]["median_ms"]
            emit(rec)


if __name__ == "__main__":
    main()
