"""CPU tests of bench.py's contract: the reference arm (`--impl reference`) of the workloads that finish in seconds
prints ONE JSON line with the keys the driver reads, runs no GPU code, and under a multi-rank launch only rank 0
prints."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e")


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=600, env=e, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.strip()]


@pytest.mark.parametrize("workload", ["config3_replay_insert", "config3_collect_experience", "config5_sweep"])
def test_reference_arm_prints_one_contract_line(workload):
    lines = _run(["--impl", "reference", "--workload", workload, "--steps", "2", "--warmup", "1"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["config"]["workload"] == workload and d["value"] > 0
    assert d["steps"] == 2                                        # --steps sets the number of timed steps
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None and d["higher_is_better"] is True


def test_reference_arm_is_silent_on_other_ranks():
    lines = _run(["--impl", "reference", "--workload", "config3_replay_insert", "--steps", "1", "--warmup", "1",
                  "--gpus", "2"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert lines == []


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"],
                                  ["--workload", "config5_sweep", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused_before_any_work(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 2 and out.stdout == "" and "error:" in out.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("workload,steps", [("config1_closed_loop", 21), ("config3_actor_rollouts", 11)])
def test_gpu_arm_times_the_requested_steps(workload, steps, cuda_device):
    """Workloads with long steps time every step --steps asks for, also past 20 (closed loop) and 10 (policy in the
    loop)."""
    lines = _run(["--workload", workload, "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline"])
    d = json.loads(lines[-1])
    assert d["steps"] == steps and d["gpu_launches"] == steps


@pytest.mark.gpu
def test_dump_outputs_are_what_the_last_timed_plan_call_returned(tmp_path, cuda_device):
    """--dump-outputs of the default workload against iCemTO.optimize called here on the bench's seeded inputs
    (keys split from PRNGKey(0), states from default_rng(0)): equal bit for bit, so two runs compare exactly."""
    import numpy as np
    import torch
    import mbpo_b200
    from mbpo_b200.optimizers import iCemTO, iCemParams
    from mbpo_b200.systems import PendulumSystem
    lines = _run(["--steps", "2", "--warmup", "1", "--no-others", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)])
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    got = {n: np.load(os.path.join(str(tmp_path), n + ".npy")) for n in ("best_sequence", "best_reward", "key")}
    assert sorted(os.listdir(str(tmp_path))) == ["best_reward.npy", "best_sequence.npy", "key.npy"]
    B, H = 4096, 30
    opt = iCemTO(horizon=H, action_dim=1, opt_params=iCemParams(num_samples=512, num_particles=1))
    opt.set_system(PendulumSystem())
    state = opt.init(mbpo_b200.random.split(mbpo_b200.random.PRNGKey(0, cuda_device), B))
    rng = np.random.default_rng(0)
    th, w = rng.uniform(-np.pi, np.pi, B), rng.uniform(-8, 8, B)
    x0 = np.stack([np.cos(th), np.sin(th), w], -1).astype(np.float32)
    new = opt.optimize(torch.from_numpy(x0).to(cuda_device), state)
    assert got["best_sequence"].dtype == np.float32 and got["best_sequence"].shape == (B, H, 1)
    assert np.array_equal(got["best_sequence"], new.best_sequence.cpu().numpy())
    assert np.array_equal(got["best_reward"], new.best_reward.cpu().numpy())
    assert got["key"].dtype == np.float64
    assert np.array_equal(got["key"], new.key.view(torch.int32).cpu().numpy().view(np.uint32).astype(np.float64))
