"""Host-side multi-GPU logic on CPU: contiguous sharding and the world_size-2 gloo gather."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def test_shard_bounds_partition():
    from mbpo_b200.parallel import shard_bounds
    for total in (0, 1, 7, 4096, 65536, 1000003):
        for ws in (1, 2, 3, 4, 8):
            blocks = [shard_bounds(total, r, ws) for r in range(ws)]
            assert blocks[0][0] == 0 and blocks[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
            sizes = [hi - lo for lo, hi in blocks]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_bounds(10, 2, 2)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


class _FakeOptimizer:
    """Stands in for iCemTO.act on CPU: the 'plan' is a deterministic per-problem function of
    (state, key), so any sharding must reproduce the unsharded result exactly."""

    def act(self, obs, opt_state):
        action = (obs[:, :1] * 2.0 + opt_state.key[:, :1].to(torch.float32) * 0.5)
        return action, opt_state.replace(best_reward=action[:, 0].clone())


def _worker(rank, world, port, total, out_dir):
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(os.path.dirname(here), "model-based-policy-optimizers_b200"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from mbpo_b200.optimizers.trajectory_optimizers.icem_optimizer import iCemOptimizerState
    from mbpo_b200.parallel import all_gather_blocks, plan_sharded, shard_bounds
    g = torch.Generator().manual_seed(0)
    x = torch.rand((total, 3), generator=g)
    keys = torch.randint(0, 1000, (total, 2), generator=g, dtype=torch.int32)
    st = iCemOptimizerState(key=keys, best_sequence=torch.zeros((total, 4, 1)), best_reward=torch.zeros(total))
    actions, new_state, (lo, hi) = plan_sharded(_FakeOptimizer(), x, st)
    want, _ = _FakeOptimizer().act(x, st)
    # gather == unsharded result (plan_sharded plans on the GPU when there is one)
    assert actions.shape == (total, 1) and torch.equal(actions.cpu(), want)
    assert (lo, hi) == shard_bounds(total, rank, world)
    assert new_state.best_reward.shape[0] == hi - lo                           # state stays sharded
    blk = torch.arange(lo, hi, dtype=torch.float32).reshape(-1, 1)
    full = all_gather_blocks(blk, total)
    assert torch.equal(full[:, 0], torch.arange(total, dtype=torch.float32))
    torch.save(actions, os.path.join(out_dir, "a%d.pt" % rank))
    dist.destroy_process_group()


@pytest.mark.parametrize("total", [7, 64])
def test_world_size_2_gloo_gather(tmp_path, total):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, total, str(tmp_path)), nprocs=2, join=True)
    a0 = torch.load(os.path.join(str(tmp_path), "a0.pt"))
    a1 = torch.load(os.path.join(str(tmp_path), "a1.pt"))
    assert torch.equal(a0, a1) and a0.shape == (total, 1)


def _stats_worker(rank, world, port, out_dir):
    """The one exchange step of the data-collection path: running_statistics' psum as an all-reduce of the float64
    sums.  The per-rank sums come from the oracle here (no GPU); the product's all_reduce_sums carries them."""
    import sys
    import numpy as np
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "model-based-policy-optimizers_b200"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from mbpo_b200.parallel import shard_bounds
    from mbpo_b200.running_statistics import all_reduce_sums
    from oracle import brax_replay as obr
    rng = np.random.default_rng(0)
    obs = (rng.standard_normal((20, 101, 3)) * [1.0, 0.3, 8.0] + [0.5, -1.0, 0.0]).astype(np.float32)   # [T, E, X]
    state = obr.running_statistics_update(obr.running_statistics_init(3), obs[:2])      # a non-trivial old mean
    lo, hi = shard_bounds(obs.shape[1], rank, world)                                    # unequal env shards: 51 / 50
    mine = obs[:, lo:hi]
    sums = np.concatenate([obr.running_statistics_sums(mine, state["mean"]), [mine.shape[0] * mine.shape[1]]])
    total = all_reduce_sums(torch.from_numpy(sums)).numpy()
    got = obr.running_statistics_finalize(state, total[:6], total[6])
    want = obr.running_statistics_update(state, obs, accumulate=np.float64)
    assert total[6] == 20 * 101
    for k in ("count", "mean", "summed_variance", "std"):
        np.testing.assert_allclose(got[k], want[k], rtol=1e-5, atol=1e-6)
    torch.save(torch.from_numpy(np.concatenate([got["mean"], got["std"]])), os.path.join(out_dir, "s%d.pt" % rank))
    dist.destroy_process_group()


def test_world_size_2_gloo_running_statistics(tmp_path):
    port = _free_port()
    mp.spawn(_stats_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    s0 = torch.load(os.path.join(str(tmp_path), "s0.pt"))
    s1 = torch.load(os.path.join(str(tmp_path), "s1.pt"))
    assert torch.equal(s0, s1)                      # every rank ends with the same statistics
