"""Both beam loops of the fixed-point reweight kernels in one launch: warps whose particles' scans all stay on the map take the
unclamped lookup (fixed_lookup_in_map), warps with any particle near or off an edge take the clamped one.  The cloud below
straddles the map's right edge, arranged so that whole warps are on each side and some warps are mixed; the weights must be
bit-identical to the oracle's for the constant-bank kernel (scan of at most 1920 points) and the shared-memory one (longer)."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LFM = dict(max_obstacle_distance=2.0, max_laser_distance=100.0, z_hit=0.5, z_random=0.5, sigma_hit=0.2)


@pytest.fixture(scope="module")
def bb():
    import beluga_b200 as bb
    from beluga_b200 import build as bb_build

    bb_build.build()
    if bb.device_count() == 0:
        pytest.fail("no CUDA device: -m gpu tests must run on the GPU box")
    return bb


def box_map(width, height, seed):
    rng = np.random.default_rng(seed)
    cells = np.zeros((height, width), dtype=np.int8)
    for _ in range(120):
        x0, y0 = int(rng.integers(0, width - 8)), int(rng.integers(0, height - 8))
        cells[y0:y0 + int(rng.integers(2, 8)), x0:x0 + int(rng.integers(2, 8))] = 100
    return cells


def in_map(x, y, th, radius, width, height, res):
    """fixed_particle_setup's predicate (identity map origin)."""
    inv = 1.0 / res
    r = radius * np.maximum(np.abs(np.cos(th) * inv), np.abs(np.sin(th) * inv)) + 0.5
    gx, gy = x * inv + 1.0, y * inv + 1.0
    return (gx - r >= 0.0) & (gx + r <= width + 2) & (gy - r >= 0.0) & (gy + r <= height + 2)


@pytest.mark.parametrize("n_beams", [360, 2400])
def test_warps_on_and_off_the_map_in_one_launch(bb, orc, n_beams):
    width, height, res = 400, 300, 0.05  # 20 m x 15 m
    cells = box_map(width, height, seed=n_beams)
    rng = np.random.default_rng(n_beams + 1)
    reach = 3.0
    a = np.linspace(-math.pi, math.pi, n_beams, endpoint=False)
    rr = rng.uniform(0.2, reach, n_beams)
    rr[:4] = reach  # the scan's full reach
    pts = np.stack([rr * np.cos(a), rr * np.sin(a)], axis=1)
    radius = float(np.max(np.abs(pts[:, 0]) + np.abs(pts[:, 1])))
    warps = 600
    n = warps * 32
    # per warp: centre x from well inside (5 m) to past the right edge (23 m); mixed warps get one far particle
    cx = np.repeat(rng.uniform(5.0, 23.0, warps), 32)
    x = cx + rng.normal(0.0, 0.3, n)
    mixed = np.zeros(n, dtype=bool)
    mixed[np.arange(0, n, 32)[rng.random(warps) < 0.25]] = True
    x[mixed] = 19.5
    y = rng.uniform(6.0, 9.0, n)
    th = rng.uniform(-math.pi, math.pi, n)
    states = np.array([orc.se2(*p) for p in zip(x, y, th)])
    on = in_map(x, y, th, radius, width, height, res).reshape(warps, 32).all(axis=1)
    assert 0.2 < on.mean() < 0.8  # both loops run, warp by warp

    f = bb.Filter(capacity=n)
    f.set_likelihood_field_map(bb.LikelihoodFieldModelParam(**LFM), bb.OccupancyGrid(cells, res))
    f.set_particles(states)
    f.reweight(pts)
    got = f.particles()[1]
    exp = orc.sensor_weights(orc.LFM, orc.LfmParam(**LFM), orc.Grid(cells, res), pts, states)
    assert np.array_equal(got, exp)
    assert len(np.unique(got)) > n // 4
