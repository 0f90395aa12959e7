#!/usr/bin/env python
"""bench.py -- iCEM model-rollout transitions/sec on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU restatement of the reference

A "step" is one batched plan call (iCemTO.optimize over B independent problems): S CEM
iterations of sample -> rollout -> score -> elite-select -> refit.  Workload (default) is
BASELINE.json configs[1]: 4,096 initial states, pop=512 (+15 kept rows), horizon=30,
5 iterations, analytic pendulum, num_particles=1.  With N GPUs every rank plans its own 4,096
problems (weak scaling; problems are independent, no data-path collective; the first actions
are all-gathered over NCCL only in the end-to-end leg).

transitions per step = B * S * (N_samples + Np) * P * H = 4096*5*527*1*30 = 323,788,800 per GPU.

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True        # the bench writes nothing into the tree it runs from (which may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "model-based-policy-optimizers_b200"))

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (B per GPU, horizon, iCemParams overrides)
    "config2_batched_icem": dict(B=4096, horizon=30, params=dict(num_samples=512, num_particles=1)),
    "config1_single_state": dict(B=1, horizon=20, params=dict(num_particles=1)),
    "config2_colored": dict(B=4096, horizon=30, params=dict(num_samples=512, num_particles=1, exponent=2.0, alpha=0.1)),
    "config4_population": dict(B=1024, horizon=50, params=dict(num_samples=1024, num_particles=1)),
}
GUARD = None
METRIC = "iCEM model-rollout transitions/sec (pop x horizon x problems x CEM iterations)"
UNIT = "transitions/s"

# Roofline inputs measured with ncu live in a tracked file (profiles/roofline_inputs.json): per workload the
# executed lane-instructions per transition (smsp__inst_executed.sum x 32 / transitions) and the DRAM traffic per
# launch of the dominant kernel, each stamped with the commit of the kernel it was captured from.
ALGORITHMIC_LANE_INSTR_PER_TRANSITION = 220.0      # SURVEY.md section 8(d): ~110 rollout + ~110 sampling, fused plan


def roofline_inputs():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "roofline_inputs.json")))
    except Exception:
        return {}


def ncu_traffic(workload):
    return (roofline_inputs().get(workload) or {}).get("dram_bytes_per_launch")


def transitions_per_step(B, horizon, p):
    npe = max(int(p.elite_set_fraction * p.num_elites), 1)
    return B * p.num_steps * (p.num_samples + npe) * p.num_particles * horizon


def random_states(n, seed):
    rng = np.random.default_rng(seed)
    th, w = rng.uniform(-np.pi, np.pi, n), rng.uniform(-8, 8, n)
    return np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy.  Floats keep their dtype; integer words (PRNG keys) are stored as
    float64, which holds every uint32 exactly.  The plan workloads return at most ~0.6 MB per GPU, so everything is
    written."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


class ClockSampler:
    """Streams nvidia-smi clocks / throttle reasons (one sample every 20 ms) while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.out = ""

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)        # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.out.splitlines():
            r = [c.strip() for c in line.split(",")]
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def host_info():
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return os.cpu_count() or 1, model


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle's plain-C twin (OpenMP over problems) on a bounded sample of the workload
# ------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Host threads the CPU arm may use.  torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm runs
    on rank 0 alone and asks OpenMP for the whole host explicitly."""
    try:
        return max(len(os.sched_getaffinity(0)), 1)
    except AttributeError:
        return max(os.cpu_count() or 1, 1)


def cpu_reference_step(wl, steps: int, warmup: int, sample_B: int | None = None):
    """Times `steps` plan calls of the CPU restatement on a bounded sample; returns dict."""
    from oracle import c_twin, jax_prng as jr, mbpo_oracle as orc
    lib = c_twin.load(native=True)
    p = orc.ICemParams(**wl["params"])
    cores = host_threads()
    B = sample_B or max(cores * 32, 64)
    B = min(B, wl["B"]) if wl["B"] > 1 else 1
    cfg = c_twin.make_cfg(p, wl["horizon"])
    p9 = orc.PendulumParams().packed()
    x0 = random_states(wl["B"], 0)[:B]
    # the GPU arm's keys: opt.init(split(PRNGKey(0), B)).key = split(k, 3)[2] per problem (icem_optimizer.py:123)
    keys = orc.split_keys(orc.split_keys(jr.PRNGKey(0).reshape(1, 2), wl["B"])[0], 3)[:B, 2].copy()
    seq = np.zeros((B, wl["horizon"]), np.float32)
    used = cores
    for _ in range(max(warmup, 1)):
        c_twin.optimize_batch(lib, cfg, p9, x0[: max(B // 8, 1)], keys[: max(B // 8, 1)], seq[: max(B // 8, 1)], cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        _, _, _, used = c_twin.optimize_batch(lib, cfg, p9, x0, keys, seq, cores)
    dt = (time.perf_counter() - t0) / steps
    tr = transitions_per_step(B, wl["horizon"], p)
    return dict(value=tr / dt, ms_per_step=dt * 1e3, cores=used, sample_B=B,
                sample="%d of %d problems per step (same keys/states as the GPU arm), C restatement + OpenMP" % (
                    B, wl["B"]))


def run_reference(args, wl_name, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores, model = host_info()
    r = cpu_reference_step(wl, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl_name, wl, args.gpus),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                         "sample": r["sample"], "host_cpu": model, "host_logical_cpus": ncores,
                         "note": "CPU restatement of the reference semantics (oracle/c) -- the reference's JAX "
                                 "stack is not installable in this image, so this is not XLA"},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_json(line, GUARD)


def workload_config(name, wl, gpus):
    p = dict(num_particles=10, num_samples=500, num_elites=50, num_steps=5, exponent=0.0, alpha=0.0)
    p.update(wl["params"])
    return {"workload": name, "problems_per_gpu": wl["B"], "problems_total": wl["B"] * gpus, "horizon": wl["horizon"],
            "num_samples": p["num_samples"], "num_elites": p["num_elites"], "num_prev_elites": 15,
            "num_particles": p["num_particles"], "cem_iterations": p["num_steps"], "exponent": p["exponent"],
            "alpha": p["alpha"], "system": "analytic pendulum", "parallelism": "problems sharded x%d" % gpus,
            # one text for both arms, so that their configs compare equal
            "l2": "GPU arm: flushed (256 MiB memset) before every timed step; CPU arm: n/a"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, wl_name, wl):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU restatement)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import mbpo_b200
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.parallel import all_gather_blocks, shard_bounds

    mbpo_b200.config.math_mode = args.math
    p = iCemParams(**wl["params"])
    B, H = wl["B"], wl["horizon"]
    total_B = B * world
    opt = iCemTO(horizon=H, action_dim=1, opt_params=p)
    system = PendulumSystem()
    opt.set_system(system)
    lo, hi = shard_bounds(total_B, rank, world)
    keys_all = mbpo_b200.random.split(mbpo_b200.random.PRNGKey(0, dev), total_B)
    state = opt.init(keys_all[lo:hi].contiguous())
    x0_host = torch.from_numpy(random_states(total_B, 0)[lo:hi].copy()).pin_memory()
    x0 = x0_host.to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    tr_step = transitions_per_step(B, H, p)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing ---------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        opt.optimize(x0, state)
    barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(args.steps):
            flush.zero_()                     # evict L2 between timed iterations (untimed)
            starts[k].record()
            new_state = opt.optimize(x0, state)
            ends[k].record()
        barrier()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = tr_step * world / (ms_per_step * 1e-3)
    clocks = clk.summary()
    if args.dump_outputs:
        # the last timed step's result, every rank's problems in global order
        outs = {"best_sequence": new_state.best_sequence, "best_reward": new_state.best_reward,
                "key": new_state.key.view(torch.int32)}
        outs = {k: all_gather_blocks(v.contiguous(), total_B).cpu().numpy() for k, v in outs.items()}
        outs["key"] = outs["key"].view(np.uint32)
        if rank == 0:
            dump_outputs(args.dump_outputs, outs)

    # ---- end to end through the public API with host buffers ------------------------------------
    act_host = torch.empty((B, 1), dtype=torch.float32).pin_memory()
    gathered = None
    for _ in range(3):
        a, _ = opt.act(x0_host.to(dev, non_blocking=True), state)
        act_host.copy_(a, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        xd = x0_host.to(dev, non_blocking=True)            # h2d: this step's initial states
        a, st2 = opt.act(xd, state)
        if world > 1:
            gathered = all_gather_blocks(a.contiguous(), total_B)   # NCCL gather of the chosen first actions
        act_host.copy_(a, non_blocking=True)               # d2h: the step's result
        torch.cuda.synchronize(dev)
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = tr_step * world / e2e_s

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        sm_max = float(peaks.get("sm_max_mhz", 1965.0))
        issue_peak = 148 * 4 * 32 * sm_max * 1e6 / 1e12          # T lane-instr/s
        ri = (roofline_inputs().get(wl_name + ("" if args.math == "reference" else "_" + args.math)) or {})
        executed = ri.get("executed_lane_instr_per_transition")
        kernel_ms = ms_per_step                                   # one fused kernel per step: event time = launch time
        tps = tr_step / (kernel_ms * 1e-3)
        algorithmic = tps * ALGORITHMIC_LANE_INSTR_PER_TRANSITION / 1e12
        roofline = {
            "bound": "issue", "kernel": "icem_plan_pendulum_kernel",
            "achieved": algorithmic, "peak": issue_peak, "unit": "T lane-instr/s",
            "frac": algorithmic / issue_peak,
            "frac_algorithmic": algorithmic / issue_peak,
            "algorithmic_lane_instr_per_transition": ALGORITHMIC_LANE_INSTR_PER_TRANSITION,
            "issue_util": (tps * executed / 1e12 / issue_peak) if executed else None,
            "executed_lane_instr_per_transition": executed,
            "inputs_from": ri.get("source"), "inputs_commit": ri.get("kernel_commit"),
            "traffic": ncu_traffic(wl_name) if (world == 1 and args.math == "reference") else None,
            "peak_source": "148 SMs x 4 SMSPs x 32 lanes x sm_max_mhz (MEASURED_PEAKS.json)",
            "note": "the fused plan keeps actions in shared memory: HBM traffic is ~0 B/transition, so the limiting "
                    "roofline is the SM issue rate.  frac = frac_algorithmic counts SURVEY 8(d)'s 220 lane-instructions "
                    "per transition as the useful work; issue_util counts what the kernel executes (ncu)",
        }
        others = None
        if world == 1 and wl_name == "config2_batched_icem" and not args.no_others:
            others = measure_others(args)
        cpu = None
        if not args.no_cpu_baseline:
            r = cpu_reference_step(wl, steps=1, warmup=1)
            ncores, model = host_info()
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                   "host_cpu": model, "host_logical_cpus": ncores}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(wl_name, wl, world),
            "math_mode": args.math,
            "ms_per_plan_call": ms_per_step,
            "pop_x_horizon_x_problems_per_s": B * world * p.num_samples * H / (ms_per_step * 1e-3),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(x0_host.numel() * 4), "d2h_bytes_per_step": int(act_host.numel() * 4),
                    "api": "iCemTO.act(obs[B,3] from pinned host) -> first actions[B,1] to pinned host"
                           + ("; NCCL all_gather of first actions" if world > 1 else "")},
            "gpu_launches": 2 * args.steps,   # zero_row_value_kernel + icem_plan_pendulum_kernel per step
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if others is not None:
            line["others"] = others
        emit_json(line, GUARD)
    if world > 1:
        dist.destroy_process_group()


def measure_others(args):
    """BASELINE.json's other single-GPU configurations, measured in this same process right after the headline so
    that they sit under the same driver clock and loaded-library record: config 1 (the reference's own closed-loop
    test), config 3 (vmapped env rollouts; the same with the policy in the loop) and config 4 (learned-ensemble
    iCEM), each with its own CPU leg on a bounded sample.  Compact entries; `python bench.py --workload <name>`
    prints the full line of any of them."""
    global _CAPTURE
    from types import SimpleNamespace
    out = {}
    table = (("config1_closed_loop", run_closed_loop), ("config3_env_rollouts", run_env),
             ("config3_actor_rollouts", run_actor), ("config4_ensemble_icem", run_ensemble))
    for name, fn in table:
        entry = {}
        for impl in ("ours", "reference"):
            if impl == "reference" and args.no_cpu_baseline:
                continue
            a = SimpleNamespace(**vars(args))
            a.impl, a.workload = impl, name
            a.steps = args.steps if impl == "ours" else 1
            a.warmup = 3 if impl == "ours" else 1
            _CAPTURE = []
            try:
                fn(a)
                got = _CAPTURE[-1] if _CAPTURE else {"error": "no line"}
            except Exception as e:                       # one broken leg must not take the headline line down
                got = {"error": "%s: %s" % (type(e).__name__, e)}
            finally:
                _CAPTURE = None
            if impl == "ours":
                roof = got.get("roofline") or {}
                entry.update({k: got.get(k) for k in ("metric", "value", "unit", "ms_per_step", "clocks", "gpu_launches",
                                                      "error") if k in got})
                entry["roofline"] = {k: roof.get(k) for k in ("bound", "kernel", "achieved", "peak", "unit", "frac",
                                                               "traffic") if k in roof}
                e2e = got.get("e2e") or {}
                entry["e2e"] = {k: e2e.get(k) for k in ("value", "unit", "ms_per_step", "h2d_bytes_per_step",
                                                         "d2h_bytes_per_step") if k in e2e}
                for k in ("ms_per_plan_call", "sum_rewards"):
                    if k in got:
                        entry[k] = got[k]
            else:
                entry["cpu_baseline"] = got.get("cpu_baseline") or got
        out[name] = entry
    return out


# ------------------------------------------------------------------------------------------------
# config 3: vmapped System.step rollouts for SAC/PPO data collection (HBM-bound stream)
# ------------------------------------------------------------------------------------------------
ENV_E, ENV_T, ENV_EPISODE = 65536, 1000, 200
ENV_BYTES_PER_TRANSITION = 4 + 24    # action read; next_obs 12 (observation aliases it) + reward/discount/truncation 12 written


def run_env(args):
    """65,536 envs x 1,000 wrapped env steps per call, envs sharded over the ranks (strong scaling)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import c_twin, mbpo_oracle as orc
        lib = c_twin.load(native=True)
        E, T = 4096, 250                       # bounded sample of the same workload
        x0 = random_states(ENV_E, 1)[:E]
        acts = np.random.default_rng(2).uniform(-1, 1, (T, E)).astype(np.float32)
        p9 = orc.PendulumParams().packed()
        c_twin.env_rollout(lib, p9, x0[:256], acts[:, :256].copy(), ENV_EPISODE, num_threads=host_threads())
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = c_twin.env_rollout(lib, p9, x0, acts, ENV_EPISODE, num_threads=host_threads())
        dt = (time.perf_counter() - t0) / args.steps
        ncores, model = host_info()
        v = E * T / dt
        emit_json({"impl": "reference", "metric": "vmapped System.step env-steps/sec", "value": v,
                          "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                          "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "config3_env_rollouts", "envs": ENV_E, "steps_per_call": ENV_T},
                          "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": out["threads"], "kind": "port",
                                           "sample": "%d envs x %d steps of 65536 x 1000" % (E, T), "host_cpu": model},
                          "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
                  GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200.envs import wrap
    from mbpo_b200.parallel import shard_bounds
    from mbpo_b200.systems import PendulumSystem
    mbpo_b200.config.math_mode = args.math
    weak = args.scaling == "weak"
    total_E = ENV_E * world if weak else ENV_E
    lo, hi = shard_bounds(total_E, rank, world)
    E, T = hi - lo, ENV_T
    system = PendulumSystem()
    sp = system.reset(device=dev).system_params
    env = wrap(system, sp, episode_length=ENV_EPISODE)
    x0 = torch.from_numpy(random_states(total_E, 1)[lo:hi].copy()).to(dev)
    acts_host = torch.from_numpy(np.random.default_rng(2 + (rank if weak else 0)).uniform(-1, 1, (T, ENV_E if not weak else E, 1))
                                 .astype(np.float32)[:, (lo if not weak else 0):(hi if not weak else E)].copy())
    acts_host = acts_host.pin_memory()
    acts = acts_host.to(dev)
    st = env.reset(x0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # raw C-ABI launches into preallocated Transition buffers (no allocator traffic in the timed region)
    L = mbpo_b200._lib
    buf = torch.empty((T + 1, E, 3), device=dev)      # observation = buf[:T], next_observation = buf[1:]
    n = buf[1:]
    r = torch.empty((T, E), device=dev); d = torch.empty((T, E), device=dev); tr = torch.empty((T, E), device=dev)
    params = system.pack_params(sp)
    first = st.info["first_obs"]
    # env state ping-pongs between two buffer sets: mbpo_env_unroll reads one and writes the other
    state = [[st.obs.clone(), st.info["steps"].clone(), st.done.clone()],
             [st.obs.clone(), st.info["steps"].clone(), st.done.clone()]]
    flip = [0]

    def launch():
        src, dst = state[flip[0]], state[flip[0] ^ 1]
        flip[0] ^= 1
        if args.env_sequential:      # the one-thread-per-env scan, for comparison
            L.check(L.lib.mbpo_env_rollout(system.system_kind, L.C.addressof(params), mbpo_b200.config.math_mode_id,
                                           3, 1, ENV_EPISODE, 1, L.ptr(src[0]), L.ptr(src[1]), L.ptr(src[2]),
                                           L.ptr(first), L.ptr(acts), E, T, None, L.ptr(r), L.ptr(d), L.ptr(n),
                                           L.ptr(tr), L.stream_ptr(dev)))
            flip[0] ^= 1
            return
        L.check(L.lib.mbpo_env_unroll(system.system_kind, L.C.addressof(params), mbpo_b200.config.math_mode_id, 3, 1,
                                      ENV_EPISODE, 1, L.ptr(src[0]), L.ptr(src[1]), L.ptr(src[2]), L.ptr(dst[0]),
                                      L.ptr(dst[1]), L.ptr(dst[2]), L.ptr(first), L.ptr(acts), E, T, None, L.ptr(r),
                                      L.ptr(d), L.ptr(n), L.ptr(tr), L.stream_ptr(dev)))
    for _ in range(max(args.warmup, 3)):
        launch()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(args.steps):
            starts[k].record()
            launch()
            ends[k].record()
        barrier()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total_E * T / (ms * 1e-3)
    # end to end: actions from pinned host memory, rewards back to the host
    rew_host = torch.empty((T, E), dtype=torch.float32).pin_memory()
    for _ in range(3):                                               # untimed: the allocator's first blocks, the streams
        st2, trn = env.unroll_streamed(st, acts_host, rew_host)
        torch.cuda.synchronize(dev)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        st2, trn = env.unroll_streamed(st, acts_host, rew_host)      # copies and rollout overlapped, 64-step chunks
        torch.cuda.synchronize(dev)
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = E * T * ENV_BYTES_PER_TRANSITION / (ms * 1e-3) / 1e9     # this rank's kernel
        emit_json({
            "metric": "vmapped System.step env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "config3_env_rollouts", "envs": total_E, "envs_per_gpu": E, "steps_per_call": T,
                       "episode_length": ENV_EPISODE, "action_repeat": 1, "parallelism": "envs sharded x%d" % world,
                       "kernel": "sequential scan per env" if args.env_sequential else "episode pieces rolled concurrently",
                       "l2": "inputs+outputs %.2f GB per call >> 126 MB L2" % (E * T * ENV_BYTES_PER_TRANSITION / 1e9)},
            "math_mode": args.math, "clocks": clk.summary(),
            "e2e": {"value": total_E * T / e2e_s, "unit": "env-steps/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(acts_host.numel() * 4), "d2h_bytes_per_step": int(rew_host.numel() * 4),
                    "api": "VmappedSystemEnv.unroll_streamed(actions[T,E,1] in pinned host memory, rewards to pinned host): "
                           "H2D, rollout and D2H of 64-step chunks overlapped on three streams"},
            "gpu_launches": args.steps,
            "roofline": {"bound": "hbm", "kernel": "env_rollout_pendulum_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic("config3_env_rollouts") if world == 1 else None,
                         "algorithmic_bytes_per_launch": E * T * ENV_BYTES_PER_TRANSITION,
                         "algorithmic_bytes_per_transition": ENV_BYTES_PER_TRANSITION,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            "cpu_baseline": None}, GUARD)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# config 4: iCEM with learned MLP-ensemble dynamics (tcgen05 forward)
# ------------------------------------------------------------------------------------------------
ENS_B, ENS_N, ENS_H, ENS_E, ENS_S = 36, 1024, 50, 5, 5
ENS_FLOP_PER_FORWARD = 2 * (4 * 256 + 256 * 256 + 256 * 256 + 256 * 3)     # 265,728


def make_ensemble_numpy(seed=3, members=5):
    """Same construction as oracle.make_mlp_ensemble (random-init weights of the config-4 architecture)."""
    rng = np.random.default_rng(seed)
    dims = (4, 256, 256, 256, 3)
    ws, bs = [], []
    for i in range(4):
        ws.append((rng.standard_normal((members, dims[i], dims[i + 1])) / np.sqrt(dims[i])).astype(np.float32))
        bs.append((0.01 * rng.standard_normal((members, dims[i + 1]))).astype(np.float32))
    ws[-1] = (ws[-1] * np.float32(0.1)).astype(np.float32)
    return ws, bs


def run_ensemble(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import mbpo_oracle as orc                                     # CPU arm only
        ens = orc.make_mlp_ensemble(seed=3, members=ENS_E)
        rows, Hs = 1039, 5                                  # one problem's candidates, 5 of the 50 steps
        x0 = random_states(1, 0)
        acts = np.random.default_rng(1).uniform(-1, 1, (1, rows, Hs)).astype(np.float32)
        orc.ensemble_rollout_returns(x0, acts[:, :64], ens, bf16=True)
        t0 = time.perf_counter()
        for _ in range(max(args.steps, 1)):
            orc.ensemble_rollout_returns(x0, acts, ens, bf16=True)
        dt = (time.perf_counter() - t0) / max(args.steps, 1)
        ncores, model = host_info()
        v = rows * ENS_E * Hs / dt                           # member-transitions per second = the metric's unit
        emit_json({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
                   "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
                   "scaling": "weak", "vs_baseline": None, "dtype": "bf16-rounded operands, f32 accumulate (NumPy)",
                   "data": "synthetic (random-init ensemble weights)",
                   "config": {"workload": "config4_ensemble_icem", "problems_per_gpu": ENS_B, "num_samples": ENS_N,
                              "horizon": ENS_H, "members": ENS_E},
                   "cpu_baseline": {"value": v, "unit": UNIT, "cores": ncores, "kind": "port",
                                    "sample": "rollouts only: %d candidates x %d members x %d of %d steps, NumPy oracle "
                                              "(BLAS threads); the reference ships no learned-dynamics System" % (
                                                  rows, ENS_E, Hs, ENS_H), "host_cpu": model},
                   "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}, GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import MLPEnsembleSystem, MlpEnsembleDynamicsParams, PendulumRewardParams, SystemParams
    ws, bs = make_ensemble_numpy()
    dyn = MlpEnsembleDynamicsParams(weights=[torch.from_numpy(w).to(dev) for w in ws],
                                    biases=[torch.from_numpy(b).to(dev) for b in bs])
    system = MLPEnsembleSystem()
    sp = SystemParams(dynamics_params=dyn, reward_params=PendulumRewardParams())
    p = iCemParams(num_samples=ENS_N, num_particles=ENS_E, num_steps=ENS_S)
    opt = iCemTO(horizon=ENS_H, action_dim=1, opt_params=p)
    opt.set_system(system)
    B = ENS_B
    keys = mbpo_b200.random.split(mbpo_b200.random.PRNGKey(rank, dev), B)
    state = opt.init(keys).replace(system_params=sp)
    x0_host = torch.from_numpy(random_states(B * world, 0)[rank * B:(rank + 1) * B].copy()).pin_memory()
    x0 = x0_host.to(dev)
    tr_step = transitions_per_step(B, ENS_H, p)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    for _ in range(max(args.warmup, 3)):
        opt.optimize(x0, state)
    steps = args.steps
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(steps):
            starts[k].record()
            opt.optimize(x0, state)
            ends[k].record()
        barrier()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # kernel-only time of the ensemble rollout (the dominant kernel), for the tensor roofline
    acts = torch.zeros((B, ENS_N + 15, ENS_H, 1), device=dev).uniform_(-1, 1)
    system.ensemble_returns(sp, x0, acts)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        system.ensemble_returns(sp, x0, acts)
    e1.record()
    torch.cuda.synchronize(dev)
    k_ms = e0.elapsed_time(e1) / steps
    act_host = torch.empty((B, 1), dtype=torch.float32).pin_memory()
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        a, _ = opt.act(x0_host.to(dev, non_blocking=True), state)
        act_host.copy_(a, non_blocking=True)
        torch.cuda.synchronize(dev)
    barrier()
    e2e_s = (time.perf_counter() - t0) / steps
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        rows = B * (ENS_N + 15)
        flops = rows * ENS_E * ENS_H * ENS_FLOP_PER_FORWARD
        achieved = flops / (k_ms * 1e-3) / 1e12
        emit_json({
            "metric": METRIC, "value": tr_step * world / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 operands, f32 accumulate (hidden layers); f32 elsewhere",
            "data": "synthetic (random-init ensemble weights)",
            "config": {"workload": "config4_ensemble_icem", "problems_per_gpu": B, "num_samples": ENS_N,
                       "num_prev_elites": 15, "horizon": ENS_H, "cem_iterations": ENS_S, "members": ENS_E,
                       "mlp": "4-256-256-256-3 swish", "parallelism": "problems sharded x%d" % world,
                       "l2": "per-step working set (actions 7.5 MB + weights 1.3 MB) is L2-resident by design; "
                             "the kernel is tensor/issue bound"},
            "clocks": clk.summary(),
            "e2e": {"value": tr_step * world / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(x0_host.numel() * 4), "d2h_bytes_per_step": int(act_host.numel() * 4),
                    "api": "iCemTO.act with MLPEnsembleSystem (staged plan: sample -> ensemble rollout -> refit)"},
            "gpu_launches": steps * (1 + 3 * ENS_S + 1),
            "roofline": {"bound": "tensor",
                         "kernel": "ensemble_rollout_pp_kernel" if rows > 18944 else "ensemble_rollout_kernel",
                         "achieved": achieved, "peak": peak,
                         "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": ncu_traffic("config4_ensemble_icem") if world == 1 else None,
                         "kernel_ms": k_ms, "flops_per_launch": flops,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"},
            "cpu_baseline": None}, GUARD)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# config 1: the reference's own test loop (tests/test_icemopt.py:19-32) as one launch
# ------------------------------------------------------------------------------------------------
MPC_T, MPC_H = 200, 20


def run_closed_loop(args):
    """A "step" is one 200-step closed-loop MPC episode from x0 = [-1, 0, 0] with iCemParams() defaults
    (P = 10, N = 500, H = 20): plan -> true System.step -> warm start, 200 times, in ONE kernel launch (one
    8-CTA cluster)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                   # a single problem does not shard: "replicas only"
    from types import SimpleNamespace
    defaults = SimpleNamespace(num_particles=10, num_samples=500, num_elites=50, num_steps=5,
                               elite_set_fraction=0.3)                           # iCemParams() (icem_optimizer.py:39-50)
    tr_plan_written = transitions_per_step(1, MPC_H, defaults)                   # 515,000 (P = 10 as written)
    if args.impl == "reference":
        from oracle import c_twin, jax_prng as jr, mbpo_oracle as orc            # CPU arm only
        p_or = orc.ICemParams()
        lib = c_twin.load(native=True)
        cfg = c_twin.make_cfg(p_or, MPC_H)
        p9 = orc.PendulumParams().packed()
        ks = jr.split(jr.PRNGKey(0), 3)
        st = orc.icem_init(ks[1], MPC_H)
        T = 20                                                                   # bounded sample of the 200 steps
        x0 = np.array([-1, 0, 0], np.float32)
        c_twin.closed_loop(lib, cfg, p9, x0, st.key, st.best_sequence, 2)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            c_twin.closed_loop(lib, cfg, p9, x0, st.key, st.best_sequence, T)
        dt = (time.perf_counter() - t0) / args.steps
        ncores, model = host_info()
        v = T * tr_plan_written / dt
        emit_json({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
                   "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "ms_per_plan_call": dt * 1e3 / T,
                   "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "config1_closed_loop", "mpc_steps": MPC_T, "horizon": MPC_H,
                              "num_samples": 500, "num_particles": 10},
                   "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": "%d of %d closed-loop steps, C restatement, one problem = one thread" % (T, MPC_T),
                                    "host_cpu": model},
                   "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}, GUARD)
        return
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import mbpo_b200
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    mbpo_b200.config.math_mode = args.math
    jrr = mbpo_b200.random
    ks = jrr.split(jrr.PRNGKey(0, dev), 3)
    system = PendulumSystem()
    system_state = system.reset(ks[2])
    cem = iCemTO(horizon=MPC_H, action_dim=1, system=None, opt_params=iCemParams(), key=ks[0])
    cem.set_system(system)
    st = cem.init(ks[1])
    x0_host = system_state.x_next.cpu().pin_memory()
    x0 = x0_host.to(dev)
    for _ in range(max(args.warmup, 3)):
        cem.closed_loop(x0, st, MPC_T)
    torch.cuda.synchronize(dev)
    steps = args.steps
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    with ClockSampler(local_rank) as clk:
        for k in range(steps):
            flush.zero_()
            starts[k].record()
            states, rewards, actions, _ = cem.closed_loop(x0, st, MPC_T)
            ends[k].record()
        torch.cuda.synchronize(dev)
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps
    total_reward = float(rewards.sum())
    rew_host = torch.empty((MPC_T,), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(steps):
        _, r, _, _ = cem.closed_loop(x0_host.to(dev, non_blocking=True), st, MPC_T)
        rew_host.copy_(r, non_blocking=True)
        torch.cuda.synchronize(dev)
    e2e_s = (time.perf_counter() - t0) / steps
    sm_max = 1965.0
    try:
        sm_max = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("sm_max_mhz", 1965.0))
    except Exception:
        pass
    emit_json({
        "metric": METRIC, "value": MPC_T * tr_plan_written / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "ms_per_plan_call": ms / MPC_T, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config1_closed_loop", "mpc_steps": MPC_T, "horizon": MPC_H, "num_samples": 500,
                   "num_elites": 50, "num_prev_elites": 15, "num_particles": 10, "cem_iterations": 5,
                   "transitions_counted": "as written in the reference (x10 identical particles); distinct = value / 10",
                   "l2": "flushed (256 MiB memset) before every timed step"},
        "math_mode": args.math, "sum_rewards": total_reward, "reference_test_threshold": -400.0,
        "clocks": clk.summary(),
        "e2e": {"value": MPC_T * tr_plan_written / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                "h2d_bytes_per_step": 12, "d2h_bytes_per_step": 4 * MPC_T,
                "api": "iCemTO.closed_loop(x0 from pinned host, 200 steps) -> rewards[200] to pinned host"},
        "gpu_launches": steps,
        "roofline": {"bound": "issue", "kernel": "icem_mpc_cluster_kernel",
                     "achieved": MPC_T * tr_plan_written / 10.0 / (ms * 1e-3) * ALGORITHMIC_LANE_INSTR_PER_TRANSITION / 1e12,
                     "peak": 148 * 4 * 32 * sm_max * 1e6 / 1e12, "unit": "T lane-instr/s",
                     "frac": MPC_T * tr_plan_written / 10.0 / (ms * 1e-3) * ALGORITHMIC_LANE_INSTR_PER_TRANSITION / 1e12
                             / (148 * 4 * 32 * sm_max * 1e6 / 1e12),
                     "traffic": None,
                     "note": "one problem = one 16-CTA thread-block cluster (16 of 148 SMs) and a chain of 200 x 5 "
                             "dependent iterations: the episode is latency-bound by construction (distinct "
                             "transitions counted: the 10 particles of the deterministic pendulum are one rollout); "
                             "throughput configurations are config 2 / config 5"},
        "cpu_baseline": None}, GUARD)


# ------------------------------------------------------------------------------------------------
# config 5: throughput sweep over the number of independent planning problems
# ------------------------------------------------------------------------------------------------
SWEEP_B = (1, 8, 64, 512, 4096, 32768, 262144, 1048576)


def run_sweep(args):
    """Config-2 parameters with B in SWEEP_B TOTAL problems sharded over the ranks (strong scaling per B)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = WORKLOADS["config2_batched_icem"]
    H = wl["horizon"]
    if args.impl == "reference":
        if rank != 0:
            return
        rows = []
        for B in (1, 8, 64, 512):
            w = dict(wl, B=B)
            r = cpu_reference_step(w, steps=args.steps, warmup=args.warmup, sample_B=B)
            rows.append({"problems": B, "ms": r["ms_per_step"], "transitions_per_s": r["value"], "cores": r["cores"]})
        ncores, model = host_info()
        best = max(rows, key=lambda r: r["transitions_per_s"])
        emit_json({"impl": "reference", "metric": METRIC, "value": best["transitions_per_s"], "unit": UNIT,
                   "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": best["ms"], "higher_is_better": True,
                   "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "config5_sweep", "horizon": H, "num_samples": 512},
                   "sweep": rows,
                   "cpu_baseline": {"value": best["transitions_per_s"], "unit": UNIT, "cores": best["cores"], "kind": "port",
                                    "sample": "B in {1, 8, 64, 512} (larger B scale linearly on the CPU)", "host_cpu": model},
                   "e2e": {"value": best["transitions_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}}, GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.parallel import shard_bounds
    from mbpo_b200.systems import PendulumSystem
    mbpo_b200.config.math_mode = args.math
    p = iCemParams(**wl["params"])
    opt = iCemTO(horizon=H, action_dim=1, opt_params=p)
    opt.set_system(PendulumSystem())
    Bmax = max(SWEEP_B)
    lo_m, hi_m = shard_bounds(Bmax, rank, world)
    # keys / states of the largest sweep point; smaller points use a prefix (same problems at every world size)
    base_key = mbpo_b200.random.PRNGKey(0, dev)
    rows = []
    clocks = None
    for B in SWEEP_B:
        lo, hi = shard_bounds(B, rank, world)
        n = hi - lo
        keys = mbpo_b200.random.split(base_key, B)[lo:hi].contiguous() if n > 0 else None
        if n > 0:
            state = opt.init(keys)
            x0 = torch.from_numpy(random_states(B, 0)[lo:hi].copy()).to(dev)
        for _ in range(3):
            if n > 0:
                opt.optimize(x0, state)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local_rank) as clk:
            e0.record()
            for _ in range(args.steps):
                if n > 0:
                    opt.optimize(x0, state)
            e1.record()
            torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / args.steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        row = {"problems": B, "ms_per_plan_call": ms, "transitions_per_s": transitions_per_step(B, H, p) / (ms * 1e-3)}
        # end to end through iCemTO.act with host buffers (states from pinned memory, first actions back) at this B
        e2e_steps = args.steps
        if n > 0:
            xh = x0.cpu().pin_memory()
            ah = torch.empty((n, 1), dtype=torch.float32).pin_memory()
            opt.act(xh.to(dev, non_blocking=True), state)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            if n > 0:
                a_, _ = opt.act(xh.to(dev, non_blocking=True), state)
                ah.copy_(a_, non_blocking=True)
            torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        te = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        row["e2e_ms_per_plan_call"] = float(te.item()) * 1e3
        row["e2e_transitions_per_s"] = transitions_per_step(B, H, p) / float(te.item())
        rows.append(row)
        clocks = clk.summary()
        if n > 0:
            del state, x0, keys
    if rank == 0:
        top = rows[-1]
        # CPU column: the C restatement + OpenMP on this host, measured up to 512 problems; beyond that one plan call
        # is B independent problems over a fixed number of cores, so the rate of the largest measured point stands
        cpu = None
        if not args.no_cpu_baseline:
            cpu_rows = {}
            for Bc in (1, 8, 64, 512):
                r = cpu_reference_step(dict(wl, B=Bc), steps=1, warmup=1, sample_B=Bc)
                cpu_rows[Bc] = r
            last = cpu_rows[512]
            for row in rows:
                Bc = row["problems"]
                if Bc in cpu_rows:
                    row["cpu_transitions_per_s"] = cpu_rows[Bc]["value"]
                    row["cpu_ms_per_plan_call"] = cpu_rows[Bc]["ms_per_step"]
                    row["cpu_measured"] = True
                else:
                    row["cpu_transitions_per_s"] = last["value"]
                    row["cpu_ms_per_plan_call"] = last["ms_per_step"] * Bc / 512.0
                    row["cpu_measured"] = False
                row["gpu_over_cpu"] = row["transitions_per_s"] / row["cpu_transitions_per_s"]
            ncores, model = host_info()
            cpu = {"value": last["value"], "unit": UNIT, "cores": last["cores"], "kind": "port",
                   "sample": "B in {1, 8, 64, 512} measured per point (C restatement + OpenMP); larger B carry the "
                             "512-problem rate (independent problems over a fixed number of cores)",
                   "host_cpu": model, "host_logical_cpus": ncores}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        issue_peak = 148 * 4 * 32 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6 / 1e12 * world
        best = max(rows, key=lambda r: r["transitions_per_s"])
        for row in rows:
            row["frac_algorithmic"] = row["transitions_per_s"] * ALGORITHMIC_LANE_INSTR_PER_TRANSITION / 1e12 / issue_peak
        emit_json({"metric": METRIC, "value": top["transitions_per_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                   "warmup": 3, "ms_per_step": top["ms_per_plan_call"], "higher_is_better": True, "scaling": "strong",
                   "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "config5_sweep", "problems_total": [r["problems"] for r in rows], "horizon": H,
                              "num_samples": 512, "num_particles": 1, "cem_iterations": 5,
                              "parallelism": "problems sharded x%d" % world,
                              "l2": "back-to-back launches; per-problem state is ~0.4 KB and the kernel works out of shared memory"},
                   "math_mode": args.math, "sweep": rows, "clocks": clocks,
                   "gpu_launches": 2 * args.steps * len(rows),
                   "roofline": {"bound": "issue", "kernel": "icem_plan_pendulum_kernel (clusters below 148 problems)",
                                "achieved": best["transitions_per_s"] * ALGORITHMIC_LANE_INSTR_PER_TRANSITION / 1e12,
                                "peak": issue_peak, "unit": "T lane-instr/s", "frac": best["frac_algorithmic"],
                                "at_problems": best["problems"], "traffic": None,
                                "note": "per-point frac_algorithmic in `sweep`; the left end is latency-bound (one "
                                        "problem = one 8-CTA cluster of 148 SMs)"},
                   "cpu_baseline": cpu,
                   "e2e": {"value": top["e2e_transitions_per_s"], "unit": UNIT,
                           "ms_per_step": top["e2e_ms_per_plan_call"],
                           "h2d_bytes_per_step": int(top["problems"] // world * 12),
                           "d2h_bytes_per_step": int(top["problems"] // world * 4),
                           "api": "iCemTO.act(obs[B,3] from pinned host) -> first actions[B,1] to pinned host, per sweep "
                                  "point in `sweep`"}}, GUARD)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# config 3 with the policy in the loop: SAC get_experience (policy forward + sample + env step)
# ------------------------------------------------------------------------------------------------
ACT_INSTR_NOTE = ("float32 policy MLP 3-64-64-64-2 on the CUDA cores: 2 x 4096 + 192 + 128 = 8,512 FMA per env-step "
                  "are the algorithmic work; roofline = FP32 FMA issue rate (148 SMs x 128 lanes x sm_max_mhz)")
ACT_FMA_PER_STEP = 2 * 64 * 64 + 3 * 64 + 64 * 2


def make_policy_numpy(seed=7, hidden=(64, 64, 64), obs_dim=3, action_dim=1):
    """Random-init policy MLP (flax Dense kernels [in, out] + biases); same construction as
    oracle.make_policy_params so both arms of the bench run the same network."""
    rng = np.random.default_rng(seed)
    dims = (obs_dim,) + tuple(hidden) + (2 * action_dim,)
    ws = [(rng.standard_normal((dims[i], dims[i + 1])) / np.sqrt(dims[i])).astype(np.float32) for i in range(len(dims) - 1)]
    bs = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(dims) - 1)]
    return ws, bs
ACT_MUFU_PER_STEP = 2 * 3 * 64        # swish = x * rcp(1 + ex2(.)): two MUFU per hidden activation, 192 activations
ACT_TC_NOTE = ("hidden->hidden policy layers as TF32 x 3 split-precision tcgen05 MMAs (fp32-accurate, accumulate in TMEM); "
               "the tensor pipe is ~25% busy and the epilogues bound the kernel: the nearest hard limit is the MUFU pipe "
               "(16 results/clk/SM, 2 per float32 swish activation x 192 activations per env-step); roofline = that rate")


def run_actor(args):
    """65,536 envs x T wrapped env steps with the SAC policy in the loop, envs sharded over the ranks."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    pol_w, pol_b = make_policy_numpy(seed=7)
    T = 200
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import jax_prng as jr, mbpo_oracle as orc                    # CPU arm only
        pol = orc.PolicyParams(pol_w, pol_b)
        E, Ts = 4096, 4                                  # bounded sample; NumPy restatement (BLAS matmuls)
        x0 = random_states(ENV_E, 1)[:E]
        orc.actor_rollout(pol, x0[:256], jr.PRNGKey(0), 1, ENV_EPISODE)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            orc.actor_rollout(pol, x0, jr.PRNGKey(0), Ts, ENV_EPISODE)
        dt = (time.perf_counter() - t0) / args.steps
        ncores, model = host_info()
        v = E * Ts / dt
        emit_json({"impl": "reference", "metric": "policy-in-the-loop env-steps/sec", "value": v, "unit": "env-steps/s",
                   "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                   "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "config3_actor_rollouts", "envs": ENV_E, "steps_per_call": T},
                   "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": ncores, "kind": "port",
                                    "sample": "%d envs x %d steps of 65536 x %d, NumPy oracle (BLAS threads)" % (E, Ts, T),
                                    "host_cpu": model},
                   "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}, GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200 import acting
    from mbpo_b200.envs import wrap
    from mbpo_b200.parallel import shard_bounds
    from mbpo_b200.systems import PendulumSystem
    mbpo_b200.config.math_mode = args.math
    weak = args.scaling == "weak"
    total_E = ENV_E * world if weak else ENV_E
    lo, hi = shard_bounds(total_E, rank, world)
    E = hi - lo
    system = PendulumSystem()
    env = wrap(system, system.reset(device=dev).system_params, episode_length=ENV_EPISODE)
    policy = acting.Policy(acting.PolicyParams([torch.from_numpy(w).to(dev) for w in pol_w],
                                               [torch.from_numpy(b).to(dev) for b in pol_b]),
                           kernel=args.actor_kernel)
    x0_host = torch.from_numpy(random_states(total_E, 1)[lo:hi].copy()).pin_memory()
    key = mbpo_b200.random.PRNGKey(0, dev)              # one key for all ranks: a shard draws its slice of the stream
    st = env.reset(x0_host.to(dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    for _ in range(max(args.warmup, 3)):
        acting.get_experience(env, st, policy, key, T, env_offset=lo, total_envs=total_E)
    steps = args.steps
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(steps):
            starts[k].record()
            acting.get_experience(env, st, policy, key, T, env_offset=lo, total_envs=total_E)
            ends[k].record()
        barrier()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    rew_host = torch.empty((T, E), dtype=torch.float32).pin_memory()

    def e2e_step():
        st_k = env.reset(x0_host.to(dev, non_blocking=True))
        _, _, trn = acting.get_experience(env, st_k, policy, key, T, env_offset=lo, total_envs=total_E)
        rew_host.copy_(trn.reward, non_blocking=True)
        torch.cuda.synchronize(dev)
        return trn
    for _ in range(3):                 # untimed: the allocator's second set of output blocks
        trn = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        trn = e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / steps
    if rank == 0:
        sm_max = 1965.0
        try:
            sm_max = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("sm_max_mhz", 1965.0))
        except Exception:
            pass
        tc = args.actor_kernel != "cuda_cores"
        if tc:
            peak = 148 * 16 * sm_max * 1e6 / 1e12         # T MUFU results/s
            achieved = E * T * ACT_MUFU_PER_STEP / (ms * 1e-3) / 1e12
            roof = {"bound": "xu", "kernel": "actor_rollout_tc_kernel", "achieved": achieved, "peak": peak,
                    "unit": "T MUFU/s", "frac": achieved / peak,
                    "traffic": ncu_traffic("config3_actor_rollouts_tcgen05") if world == 1 else None,
                    "note": ACT_TC_NOTE,
                    "tensor_tflops_issued": E * T * 3 * 2 * 2 * 64 * 64 / (ms * 1e-3) / 1e12}
        else:
            peak = 148 * 128 * sm_max * 1e6 / 1e12        # T FMA/s
            achieved = E * T * ACT_FMA_PER_STEP / (ms * 1e-3) / 1e12
            roof = {"bound": "fma", "kernel": "actor_rollout_pendulum_kernel", "achieved": achieved, "peak": peak,
                    "unit": "T FMA/s", "frac": achieved / peak, "traffic": None, "note": ACT_INSTR_NOTE}
        emit_json({
            "metric": "policy-in-the-loop env-steps/sec", "value": total_E * T / (ms * 1e-3), "unit": "env-steps/s",
            "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (random-init policy)",
            "config": {"workload": "config3_actor_rollouts", "envs": total_E, "envs_per_gpu": E, "steps_per_call": T,
                       "policy": "3-64-64-64-2 swish, NormalTanh", "episode_length": ENV_EPISODE,
                       "policy_kernel": "tcgen05 (TF32 x 3 split precision)" if tc else "CUDA cores (float32 FFMA2)",
                       "parallelism": "envs sharded x%d" % world,
                       "l2": "per-call outputs %.0f MB > 126 MB L2; the kernel is compute bound" % (E * T * 28 / 1e6)},
            "math_mode": args.math, "clocks": clk.summary(),
            "e2e": {"value": total_E * T / e2e_s, "unit": "env-steps/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(x0_host.numel() * 4), "d2h_bytes_per_step": int(rew_host.numel() * 4),
                    "api": "acting.get_experience(env, reset(x0 from pinned host), policy, key, T) -> rewards to host"},
            "gpu_launches": steps,
            "roofline": roof,
            "cpu_baseline": None}, GUARD)
    if world > 1:
        dist.destroy_process_group()


def run_collect(args):
    """SAC.get_experience in full (sac/sac.py:283-304) per step: 65,536 envs x 200 actor steps (policy in the loop,
    one launch) -> running_statistics.update of the observation normaliser (the psum over ranks is an NCCL all-reduce
    of 7 doubles) -> replay insert of the 13.1 M transitions into a queue of 2**24 rows.  Envs sharded over ranks; each
    rank owns the queue of its envs (the reference's pmap keeps one replay buffer per device)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    pol_w, pol_b = make_policy_numpy(seed=7)
    T = 200
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import brax_replay as obr, jax_prng as jr, mbpo_oracle as orc          # CPU arm only
        pol = orc.PolicyParams(pol_w, pol_b)
        E, Ts, R = 4096, 4, 1 << 16                      # bounded sample of the same pipeline
        x0 = random_states(ENV_E, 1)[:E]
        q = obr.UniformSamplingQueue(R, 10, 1)
        qs = q.insert(q.init(jr.PRNGKey(0)), np.zeros((R, 10), np.float32))
        norm = obr.running_statistics_init(3)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            tr, _ = orc.actor_rollout(pol, (x0 - norm["mean"]) / norm["std"], jr.PRNGKey(0), Ts, ENV_EPISODE)
            norm = obr.running_statistics_update(norm, tr["observation"])
            n = Ts * E
            qs = q.insert(qs, np.concatenate([tr["observation"].reshape(n, 3), tr["action"].reshape(n, 1),
                                              tr["reward"].reshape(n, 1), tr["discount"].reshape(n, 1),
                                              tr["next_observation"].reshape(n, 3), tr["truncation"].reshape(n, 1)], 1))
        dt = (time.perf_counter() - t0) / args.steps
        ncores, model = host_info()
        v = E * Ts / dt
        emit_json({"impl": "reference", "metric": "SAC get_experience env-steps/sec", "value": v, "unit": "env-steps/s",
                   "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                   "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "config3_collect_experience", "envs": ENV_E, "steps_per_call": T},
                   "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": ncores, "kind": "port",
                                    "sample": "%d envs x %d steps of 65536 x %d into a full queue of %d rows, NumPy "
                                              "oracle (BLAS threads)" % (E, Ts, T, R), "host_cpu": model},
                   "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}, GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200 import acting, running_statistics as rs
    from mbpo_b200.envs import wrap
    from mbpo_b200.parallel import shard_bounds
    from mbpo_b200.replay_buffers import UniformSamplingQueue
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils.optimizer_utils import Transition
    mbpo_b200.config.math_mode = args.math
    lo, hi = shard_bounds(ENV_E, rank, world)
    E = hi - lo
    system = PendulumSystem()
    env = wrap(system, system.reset(device=dev).system_params, episode_length=ENV_EPISODE)
    w_host = [torch.from_numpy(w).pin_memory() for w in pol_w]
    b_host = [torch.from_numpy(b).pin_memory() for b in pol_b]
    params = acting.PolicyParams([w.to(dev) for w in w_host], [b.to(dev) for b in b_host])
    z = lambda *sh: torch.zeros(sh, device=dev)
    dummy = Transition(z(3), z(1), z(), z(), z(3), {"state_extras": {"truncation": z()}, "policy_extras": {}})
    queue = UniformSamplingQueue(REPLAY_ROWS // world, dummy, 256)
    col = acting.ExperienceCollector(env, acting.make_normalized_inference_fn(kernel=args.actor_kernel), queue, T,
                                     pmap_axis_name="i" if world > 1 else None, env_offset=lo, total_envs=ENV_E)
    state = env.reset(torch.from_numpy(random_states(ENV_E, 1)[lo:hi].copy()).to(dev))
    norm, buf = rs.init_state(3, dev), queue.init(mbpo_b200.random.PRNGKey(1, dev))
    key = mbpo_b200.random.PRNGKey(0, dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        norm, state, buf = col.get_experience(norm, params, state, buf, key); key = col.last_key
    steps = args.steps
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(steps):
            starts[k].record()
            norm, state, buf = col.get_experience(norm, params, state, buf, key); key = col.last_key
            ends[k].record()
        barrier()
    ms = sum(a.elapsed_time(b) for a, b in zip(starts, ends)) / steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # end to end: the learner's new policy parameters arrive from pinned host memory before every collection, the
    # normaliser statistics (what the learner logs / checkpoints) go back to the host after it
    stats_host = torch.empty(7, dtype=torch.float32).pin_memory()
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        params = acting.PolicyParams([w.to(dev, non_blocking=True) for w in w_host],
                                     [b.to(dev, non_blocking=True) for b in b_host])
        norm, state, buf = col.get_experience(norm, params, state, buf, key); key = col.last_key
        stats_host[:3].copy_(norm.mean, non_blocking=True)
        stats_host[3:6].copy_(norm.std, non_blocking=True)
        stats_host[6:].copy_(norm.count.reshape(1), non_blocking=True)
        torch.cuda.synchronize(dev)
    barrier()
    e2e_s = (time.perf_counter() - t0) / steps
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    if rank == 0:
        sm_max = 1965.0
        try:
            sm_max = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("sm_max_mhz", 1965.0))
        except Exception:
            pass
        peak = 148 * 16 * sm_max * 1e6 / 1e12
        achieved = E * T * ACT_MUFU_PER_STEP / (ms * 1e-3) / 1e12
        h2d = sum(int(w.numel()) for w in w_host + b_host) * 4
        emit_json({
            "metric": "SAC get_experience env-steps/sec", "value": ENV_E * T / (ms * 1e-3), "unit": "env-steps/s",
            "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init policy)",
            "config": {"workload": "config3_collect_experience", "envs": ENV_E, "steps_per_call": T,
                       "policy": "3-64-64-64-2 swish, NormalTanh, normalised observations",
                       "episode_length": ENV_EPISODE, "queue_rows": REPLAY_ROWS, "parallelism": "envs sharded x%d" % world,
                       "stages": "actor rollout (tcgen05) -> running_statistics.update (+ all-reduce) -> replay insert",
                       "l2": "per-call Transition buffers %.0f MB > 126 MB L2" % (E * T * 40 / 1e6)},
            "math_mode": args.math, "clocks": clk.summary(),
            "e2e": {"value": ENV_E * T / e2e_s, "unit": "env-steps/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 28,
                    "api": "ExperienceCollector.get_experience(normalizer, policy params from pinned host, env_state, "
                           "buffer_state, key) -> normaliser statistics to the host"},
            "gpu_launches": steps * 5,
            "roofline": {"bound": "xu", "kernel": "actor_rollout_tc_kernel (dominant: the whole step is timed)",
                         "achieved": achieved, "peak": peak, "unit": "T MUFU/s", "frac": achieved / peak, "traffic": None,
                         "note": ACT_TC_NOTE},
            "cpu_baseline": None}, GUARD)
    if world > 1:
        dist.destroy_process_group()


BPTT_B, BPTT_H, BPTT_DISCOUNT, BPTT_LAMBDA = 65536, 20, 0.99, 0.97      # horizon / lambda_ of tests/test_bptt.py:51-57
BPTT_ADJ_BYTES = 12 + 4 + 4 + 12 + 4         # observation, action, g_reward, g_next_obs read; g_action written


def run_bptt(args):
    """BPTT's differentiated rollout (SURVEY 8f-4): rollout_policy forward (policy in the loop), lambda_return,
    its transpose and the reverse scan through System.step, for 65,536 initial states x horizon 20."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    pol_w, pol_b = make_policy_numpy(seed=7, hidden=(64, 64))
    metric = "BPTT rollout + cotangent pass, transitions/sec"
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import jax_prng as jr, mbpo_oracle as orc                    # CPU arm only
        B = 4096
        actor = orc.BpttActorParams(mlp=orc.PolicyParams(pol_w, pol_b), init_stddev=2.0)
        x0 = random_states(BPTT_B, 1)[:B]
        g = np.random.default_rng(3).standard_normal((B, BPTT_H)).astype(np.float32)

        def once():
            tr, _ = orc.rollout_policy(actor, x0, jr.PRNGKey(0), BPTT_H)
            nv = tr["next_observation"][..., 2]
            orc.lambda_return(tr["reward"], nv, BPTT_DISCOUNT, BPTT_LAMBDA)
            gr, gnv = orc.lambda_return_vjp(g, BPTT_DISCOUNT, BPTT_LAMBDA)
            gn = np.zeros((B, BPTT_H, 3), np.float32)
            gn[..., 2] = gnv
            orc.rollout_policy_vjp(tr["observation"], tr["action"], gr, gn)
        once()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            once()
        dt = (time.perf_counter() - t0) / args.steps
        ncores, model = host_info()
        v = B * BPTT_H / dt
        emit_json({"impl": "reference", "metric": metric, "value": v, "unit": "transitions/s", "n_gpus": args.gpus,
                   "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
                   "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "bptt_rollout_grad", "initial_states": BPTT_B, "horizon": BPTT_H},
                   "cpu_baseline": {"value": v, "unit": "transitions/s", "cores": ncores, "kind": "port",
                                    "sample": "%d of %d initial states, NumPy oracle (BLAS threads)" % (B, BPTT_B),
                                    "host_cpu": model},
                   "e2e": {"value": v, "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}, GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200 import acting
    from mbpo_b200.parallel import shard_bounds
    from mbpo_b200.systems import PendulumSystem
    from mbpo_b200.utils.optimizer_utils import lambda_return, lambda_return_vjp, rollout_policy, rollout_policy_vjp
    lo, hi = shard_bounds(BPTT_B, rank, world)
    B, H = hi - lo, BPTT_H
    system = PendulumSystem()
    sp = system.reset(device=dev).system_params
    policy = acting.BpttActorPolicy(acting.PolicyParams([torch.from_numpy(w).to(dev) for w in pol_w],
                                                        [torch.from_numpy(b).to(dev) for b in pol_b]), init_stddev=2.0)
    x0_host = torch.from_numpy(random_states(BPTT_B, 1)[lo:hi].copy()).pin_memory()
    x0 = x0_host.to(dev)
    key = mbpo_b200.random.PRNGKey(0, dev)
    g_lv = torch.from_numpy(np.random.default_rng(3).standard_normal((H, BPTT_B)).astype(np.float32)[:, lo:hi].copy()).to(dev).t()
    wv = torch.tensor([0.3, -0.2, 0.1], device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    adj_ms = []

    def step(x0_dev, timed=False):
        tr = rollout_policy(system, sp, x0_dev, policy, key, H)
        nv = tr.next_observation @ wv                                  # stand-in for the critic (the caller's network)
        lv = lambda_return(tr.reward, nv, BPTT_DISCOUNT, BPTT_LAMBDA)
        g_r, g_nv = lambda_return_vjp(g_lv, BPTT_DISCOUNT, BPTT_LAMBDA)
        g_n = g_nv[..., None] * wv
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        g_a, g_x0 = rollout_policy_vjp(system, sp, tr, g_reward=g_r, g_next_observation=g_n)
        if timed:
            e1.record()
            adj_ms.append((e0, e1))
        return lv, g_a
    for _ in range(max(args.warmup, 3)):
        step(x0)
    steps = args.steps
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(steps):
            flush.zero_()
            starts[k].record()
            step(x0, timed=True)
            ends[k].record()
        barrier()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps
    a_ms = sum(s.elapsed_time(e) for s, e in adj_ms) / len(adj_ms)
    t = torch.tensor([ms, a_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, a_ms = float(t[0]), float(t[1])
    ga_host = torch.empty((B, H, 1), dtype=torch.float32).pin_memory()
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        _, g_a = step(x0_host.to(dev, non_blocking=True))
        ga_host.copy_(g_a, non_blocking=True)
        torch.cuda.synchronize(dev)
    barrier()
    e2e_s = (time.perf_counter() - t0) / steps
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = B * H * BPTT_ADJ_BYTES / (a_ms * 1e-3) / 1e9
        emit_json({
            "metric": metric, "value": BPTT_B * H / (ms * 1e-3), "unit": "transitions/s", "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init policy)",
            "config": {"workload": "bptt_rollout_grad", "initial_states": BPTT_B, "horizon": H,
                       "policy": "BPTT actor 3-64-64-2 swish", "discount": BPTT_DISCOUNT, "lambda": BPTT_LAMBDA,
                       "parallelism": "initial states sharded x%d" % world,
                       "l2": "flushed (256 MiB memset) before every timed step"},
            "clocks": clk.summary(),
            "adjoint_kernel_ms": a_ms,
            "e2e": {"value": BPTT_B * H / e2e_s, "unit": "transitions/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(x0_host.numel() * 4), "d2h_bytes_per_step": int(ga_host.numel() * 4),
                    "api": "rollout_policy -> lambda_return -> lambda_return_vjp -> rollout_policy_vjp; x0 from pinned host, g_action to host"},
            "gpu_launches": 4 * steps,
            "roofline": {"bound": "hbm", "kernel": "rollout_adjoint_pendulum_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "algorithmic_bytes_per_transition": BPTT_ADJ_BYTES,
                         "note": "the step is dominated by the float32 policy MLP of the forward rollout (FMA-issue bound, see "
                                 "config3_actor_rollouts); the roofline object describes the reverse scan",
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            "cpu_baseline": None}, GUARD)
    if world > 1:
        dist.destroy_process_group()


class _StdoutGuard:
    """Everything the libraries print (e.g. the NCCL version banner) goes to stderr; only the final
    JSON line reaches the real stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


_real_print = print


_CAPTURE = None        # a list while run_ours collects the other configurations' lines instead of printing them


def emit_json(obj, guard):
    if _CAPTURE is not None:
        _CAPTURE.append(obj)
        return
    sys.stdout.flush()
    os.write(guard.saved, (json.dumps(obj) + "\n").encode())


# ------------------------------------------------------------------------------------------------
# replay insert: the Transition buffers of a config-3 unroll appended to SAC's UniformSamplingQueue
# ------------------------------------------------------------------------------------------------
REPLAY_E, REPLAY_T, REPLAY_D, REPLAY_ROWS = 65536, 200, 10, 1 << 24


def run_replay(args):
    """One step = UniformSamplingQueue.insert of 65,536 envs x 200 steps (13.1 M rows of 10 floats, sac.py:296-303)
    into a queue of 2**24 rows; the queue is full after the second step, so the timed inserts are the ones on which
    brax rolls the whole buffer.  Algorithmic bytes: 40 B read + 40 B written per row."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    E, T, D = REPLAY_E, REPLAY_T, REPLAY_D
    def cpu_arm(steps):
        from oracle import brax_replay as obr, jax_prng as jr
        Es, Ts, R = 4096, 50, 1 << 18          # bounded sample: 204,800 rows into a full queue of 262,144
        rng = np.random.default_rng(0)
        f = [rng.standard_normal((Ts * Es, w)).astype(np.float32) for w in (3, 1, 1, 1, 3, 1)]
        q = obr.UniformSamplingQueue(R, D, 1)
        st = q.insert(q.init(jr.PRNGKey(0)), np.zeros((R, D), np.float32))
        t0 = time.perf_counter()
        for _ in range(steps):
            st = q.insert(st, np.concatenate(f, axis=1))
        dt = (time.perf_counter() - t0) / steps
        _, model = host_info()
        return dt, {"value": Es * Ts / dt, "unit": "rows/s", "cores": 1, "kind": "port",
                    "sample": "%d rows per step into a full queue of %d rows (NumPy restatement of brax "
                              "insert_internal: ravel + roll + slice update)" % (Es * Ts, R), "host_cpu": model}

    if args.impl == "reference":
        if rank != 0:
            return
        dt, cpu = cpu_arm(args.steps)
        v = cpu["value"]
        emit_json({"impl": "reference", "metric": "replay rows inserted/sec", "value": v, "unit": "rows/s",
                   "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                   "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                   "config": {"workload": "config3_replay_insert", "envs": E, "steps_per_call": T, "row_floats": D},
                   "cpu_baseline": cpu,
                   "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}, GUARD)
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mbpo_b200
    from mbpo_b200.replay_buffers import UniformSamplingQueue
    from mbpo_b200.utils.optimizer_utils import Transition
    z = lambda *sh: torch.zeros(sh, device=dev)
    dummy = Transition(z(3), z(1), z(), z(), z(3), {"state_extras": {"truncation": z()}, "policy_extras": {}})
    q = UniformSamplingQueue(REPLAY_ROWS, dummy, 256)
    st = q.init(mbpo_b200.random.PRNGKey(0, dev))
    g = lambda *sh: torch.randn(sh, device=dev)
    buf = g(T + 1, E, 3)
    tr = Transition(buf[:T], g(T, E, 1), g(T, E), g(T, E), buf[1:], {"state_extras": {"truncation": g(T, E)},
                                                                      "policy_extras": {}})

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        st = q.insert(st, tr)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clk:
        barrier()
        for k in range(args.steps):
            starts[k].record()
            st = q.insert(st, tr)
            ends[k].record()
        barrier()
    ms = sum(a.elapsed_time(b) for a, b in zip(starts, ends)) / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    rows = E * T
    # end to end: a sampled batch (the learner's input) read back to the host after every insert
    batch_host = torch.empty((256, D), dtype=torch.float32).pin_memory()
    rew_host_in = torch.randn((T, E), dtype=torch.float32).pin_memory()
    def e2e_step(st):
        rew = rew_host_in.to(dev, non_blocking=True)
        st = q.insert(st, tr._replace(reward=rew))
        st, batch = q.sample(st)
        batch_host[:, 4].copy_(batch.reward, non_blocking=True)
        torch.cuda.synchronize(dev)
        return st
    for _ in range(3):
        st = e2e_step(st)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        st = e2e_step(st)
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = rows * 8 * D / (ms * 1e-3) / 1e9
        cpu = None if (args.no_cpu_baseline or world > 1) else cpu_arm(10)[1]
        emit_json({
            "metric": "replay rows inserted/sec", "value": world * rows / (ms * 1e-3), "unit": "rows/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "config3_replay_insert", "envs": E, "steps_per_call": T, "row_floats": D,
                       "queue_rows": REPLAY_ROWS, "parallelism": "one queue per GPU x%d" % world,
                       "l2": "%.2f GB moved per insert >> 126 MB L2" % (rows * 8 * D / 1e9)},
            "clocks": clk.summary(),
            "e2e": {"value": world * rows / e2e_s, "unit": "rows/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(rew_host_in.numel() * 4), "d2h_bytes_per_step": 256 * 4,
                    "api": "UniformSamplingQueue.insert(Transition with rewards from pinned host) + sample() -> "
                           "rewards of the batch to the host"},
            "gpu_launches": args.steps,
            "roofline": {"bound": "hbm", "kernel": "replay_pack_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic("config3_replay_insert") if world == 1 else None,
                         "algorithmic_bytes_per_launch": rows * 8 * D, "algorithmic_bytes_per_row": 8 * D,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            "cpu_baseline": cpu}, GUARD)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed steps: every timed loop of the workload (and of the `others` entries of the default "
                         "line; of every sweep point) runs exactly this many.  The `cpu_baseline` leg of a GPU line "
                         "times one step on a bounded sample; --impl reference times --steps steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS) + ["config1_closed_loop", "config3_env_rollouts", "config3_actor_rollouts",
                                                               "config4_ensemble_icem", "config5_sweep", "bptt_rollout_grad",
                                                               "config3_replay_insert", "config3_collect_experience"],
                    default="config2_batched_icem")
    ap.add_argument("--math", choices=["reference", "theta_carry"], default="reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", choices=["weak", "strong"], default=None,
                    help="config3_* workloads: strong = 65,536 envs split over the ranks (default, BASELINE.json's "
                         "wording); weak = 65,536 envs PER GPU")
    ap.add_argument("--no-others", action="store_true",
                    help="default workload: skip the compact measurements of configs 1, 3 and 4 (the `others` key)")
    ap.add_argument("--actor-kernel", choices=["auto", "cuda_cores", "tcgen05", "tcgen05_wide"], default="auto",
                    help="config3_actor_rollouts: which kernel runs the policy network")
    ap.add_argument("--env-sequential", action="store_true",
                    help="config3_env_rollouts: time the one-thread-per-env scan instead of the episode-piece kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed plan call returned (best_sequence, best_reward, key) as "
                         "DIR/<name>.npy; inputs are seeded, so runs with the same arguments compare output for output "
                         "(the iCEM plan workloads of the CUDA path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs is implemented for the CUDA path of %s" % ", ".join(sorted(WORKLOADS)))
    global GUARD
    with _StdoutGuard() as GUARD:
        if args.workload == "config3_env_rollouts":
            return run_env(args)
        if args.workload == "config4_ensemble_icem":
            return run_ensemble(args)
        if args.workload == "config3_actor_rollouts":
            return run_actor(args)
        if args.workload == "config1_closed_loop":
            return run_closed_loop(args)
        if args.workload == "bptt_rollout_grad":
            return run_bptt(args)
        if args.workload == "config5_sweep":
            return run_sweep(args)
        if args.workload == "config3_replay_insert":
            return run_replay(args)
        if args.workload == "config3_collect_experience":
            return run_collect(args)
        wl = WORKLOADS[args.workload]
        if args.impl == "reference":
            run_reference(args, args.workload, wl)
        else:
            run_ours(args, args.workload, wl)


if __name__ == "__main__":
    main()
