"""Multi-GPU parity: a filter sharded over 2 GPUs (NCCL) must produce the SAME particle set, weight sum and
estimate as the single-GPU filter with the same total particle count, step after step -- both with
the NCCL all-to-all redistribution and with the fused kernel that stores over NVLink peer memory, with
recovery injection (random_intersperse) and with multinomial sampling (every rank filters the global
slots by its span of the CDF)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


MODES = ["nccl", "p2p", "nccl-recovery", "p2p-recovery", "p2p-multinomial", "p2p-kld"]


@pytest.mark.parametrize("mode", MODES)
def test_two_gpu_shards_match_single_gpu(mode):
    import beluga_b200 as bb
    from beluga_b200 import build as bb_build

    bb_build.build()
    if bb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(29711 + 2 * MODES.index(mode)), os.path.join(ROOT, "tests", "_shard_gpu_worker.py"), "40000", "6", mode]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "SHARD_GPU_WORKER_OK" in out.stdout


@pytest.mark.parametrize("mode", ["systematic", "multinomial", "selective"])
def test_one_process_two_devices_match_single_gpu(mode):
    """bb200_sharded_amcl over two DEVICES driven by one host thread (the shape of beluga_ros's node): peer access instead of
    IPC, the same mail-block exchanges; bit-identical to the single-GPU filter."""
    import numpy as np

    import beluga_b200 as bb
    from beluga_b200 import build as bb_build
    from beluga_b200 import synthetic

    bb_build.build()
    if bb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sc = synthetic.make_scenario(grid_size=200, n_beams=181, steps=8)
    n = 60_000
    kw = dict(systematic=dict(resample_scheme=1), multinomial=dict(resample_scheme=0, recovery_probability_override=0.02),
              selective=dict(resample_scheme=1, selective_resampling=True, resample_interval=2))[mode]
    motion = bb.DifferentialDriveModelParam(0.1, 0.05, 0.1, 0.05)
    single = bb.Amcl(motion, bb.AmclParams(min_particles=n, max_particles=n, seed=8, **kw))
    group = bb.ShardedAmcl(motion, bb.AmclParams(min_particles=n, max_particles=n, seed=8, **kw), devices=[0, 1])
    lfm = bb.LikelihoodFieldModelParam(max_obstacle_distance=2.0, max_laser_distance=100.0)
    for f in (single, group):
        f.update_map(0, lfm, bb.OccupancyGrid(sc.cells, sc.resolution))
        f.initialize(sc.initial_mean, sc.initial_cov)
    for k in range(6):
        pose = bb.se2(*sc.poses[k])
        rs, rg = single.update(pose, sc.scans[k]), group.update(pose, sc.scans[k])
        assert rs.resampled == rg.resampled and rs.weight_sum == rg.weight_sum
        assert np.array_equal(single.particles()[0], group.particles()[0])
        assert np.abs(np.array(rs.estimate.mean) - np.array(rg.estimate.mean)).max() < 1e-12
