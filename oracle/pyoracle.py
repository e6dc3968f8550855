"""TEST INFRASTRUCTURE ONLY -- ctypes binding over the CPU parity oracle (liboracle.so).

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs only.  The product package (beluga_b200/) never imports this module.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liboracle.so")


_SOURCES = ("oracle_capi.cpp", "amcl_oracle.hpp", "beluga_oracle.hpp", "cluster_oracle.hpp", "se2.hpp", "Makefile")


def build(force: bool = False) -> str:
    """Compile the oracle with the recipe committed in oracle/Makefile."""
    srcs = [os.path.join(_HERE, f) for f in _SOURCES]
    stale = force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return _LIB_PATH


def use_native_build() -> bool:
    """Timing legs only (bench.py): switch to a -march=native build of the same sources, compiled on this machine
    (make native) into a temporary directory that is removed at exit, so that a timing run writes nothing into the
    source tree.  Must run before the first oracle call.  Returns False (and keeps the portable build) if the
    library is already loaded or the build fails."""
    global _LIB_PATH
    if _lib is not None:
        return False
    out_dir = tempfile.mkdtemp(prefix="beluga_b200_oracle_")
    atexit.register(shutil.rmtree, out_dir, ignore_errors=True)
    native = os.path.join(out_dir, "liboracle.so")
    if subprocess.run(["make", "-C", _HERE, "-s", "-B", "native", f"NATIVE_OUT={native}"]).returncode != 0:
        return False
    _LIB_PATH = native
    globals()["build"] = lambda force=False: native  # lib() must not fall back to rebuilding the portable library
    return True


class LfmParam(C.Structure):
    """oracle::LikelihoodFieldParam (reference: sensor/likelihood_field_model_base.hpp:42-64)."""

    _fields_ = [
        ("max_obstacle_distance", C.c_double),
        ("max_laser_distance", C.c_double),
        ("z_hit", C.c_double),
        ("z_random", C.c_double),
        ("sigma_hit", C.c_double),
        ("model_unknown_space", C.c_int),
        ("only_obstacle_boundaries", C.c_int),
    ]

    def __init__(self, max_obstacle_distance=100.0, max_laser_distance=2.0, z_hit=0.5, z_random=0.5, sigma_hit=0.2,
                 model_unknown_space=False, only_obstacle_boundaries=False):
        super().__init__(max_obstacle_distance, max_laser_distance, z_hit, z_random, sigma_hit,
                         int(model_unknown_space), int(only_obstacle_boundaries))


class BeamParam(C.Structure):
    """oracle::BeamModelParam (reference: sensor/beam_model.hpp:43-58)."""

    _fields_ = [(n, C.c_double) for n in ("z_hit", "z_short", "z_max", "z_rand", "sigma_hit", "lambda_short", "beam_max_range")]

    def __init__(self, z_hit=0.5, z_short=0.5, z_max=0.05, z_rand=0.05, sigma_hit=0.2, lambda_short=0.1, beam_max_range=60.0):
        super().__init__(z_hit, z_short, z_max, z_rand, sigma_hit, lambda_short, beam_max_range)


class MotionParam(C.Structure):
    """oracle::DifferentialDriveParam (reference: motion/differential_drive_model.hpp:40-68)."""

    _fields_ = [(n, C.c_double) for n in ("alpha1", "alpha2", "alpha3", "alpha4", "distance_threshold")]

    def __init__(self, alpha1=0.0, alpha2=0.0, alpha3=0.0, alpha4=0.0, distance_threshold=0.01):
        super().__init__(alpha1, alpha2, alpha3, alpha4, distance_threshold)


class OmniParam(C.Structure):
    """oracle::OmnidirectionalDriveParam (reference: motion/omnidirectional_drive_model.hpp:36-68); also carries
    the differential-drive alphas (alpha5 unused) and nothing for the stationary model."""

    _fields_ = [(n, C.c_double) for n in ("alpha1", "alpha2", "alpha3", "alpha4", "alpha5", "distance_threshold")]

    def __init__(self, alpha1=0.0, alpha2=0.0, alpha3=0.0, alpha4=0.0, alpha5=0.0, distance_threshold=0.01):
        super().__init__(alpha1, alpha2, alpha3, alpha4, alpha5, distance_threshold)


DIFFERENTIAL, OMNIDIRECTIONAL, STATIONARY = 0, 1, 2


class AmclParam(C.Structure):
    """oracle::AmclParams (reference: algorithm/amcl_core.hpp:34-55 + backend knobs)."""

    _fields_ = [
        ("update_min_d", C.c_double),
        ("update_min_a", C.c_double),
        ("resample_interval", C.c_uint64),
        ("selective_resampling", C.c_int),
        ("min_particles", C.c_uint64),
        ("max_particles", C.c_uint64),
        ("alpha_slow", C.c_double),
        ("alpha_fast", C.c_double),
        ("kld_epsilon", C.c_double),
        ("kld_z", C.c_double),
        ("spatial_resolution_x", C.c_double),
        ("spatial_resolution_y", C.c_double),
        ("spatial_resolution_theta", C.c_double),
        ("rng_mode", C.c_int),
        ("scheme", C.c_int),
        ("seed", C.c_uint64),
        ("threads", C.c_int),
    ]

    def __init__(self, update_min_d=0.25, update_min_a=0.2, resample_interval=1, selective_resampling=False,
                 min_particles=500, max_particles=2000, alpha_slow=0.001, alpha_fast=0.1, kld_epsilon=0.05, kld_z=3.0,
                 spatial_resolution_x=0.5, spatial_resolution_y=0.5, spatial_resolution_theta=np.deg2rad(10.0),
                 rng_mode=1, scheme=0, seed=0, threads=1):
        super().__init__(update_min_d, update_min_a, resample_interval, int(selective_resampling), min_particles,
                         max_particles, alpha_slow, alpha_fast, kld_epsilon, kld_z, spatial_resolution_x,
                         spatial_resolution_y, spatial_resolution_theta, rng_mode, scheme, seed, threads)


class UpdateResult(C.Structure):
    _fields_ = [
        ("updated", C.c_int),
        ("resampled", C.c_int),
        ("n_particles", C.c_uint64),
        ("mean", C.c_double * 4),
        ("cov", C.c_double * 9),
        ("random_state_probability", C.c_double),
        ("weight_sum", C.c_double),
        ("cells_visited", C.c_uint64),
    ]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_last_error.restype = C.c_char_p
        _lib.orc_normalize.restype = C.c_double
        _lib.orc_effective_sample_size.restype = C.c_double
        _lib.orc_spatial_hash.restype = C.c_uint64
        _lib.orc_kld_target_size.restype = C.c_uint64
        _lib.orc_kld_take_count.restype = C.c_uint64
        _lib.orc_bresenham.restype = C.c_uint64
        _lib.orc_amcl_create.restype = C.c_void_p
        _lib.orc_amcl_create_motion.restype = C.c_void_p
        _lib.orc_amcl_size.restype = C.c_uint64
        _lib.orc_amcl_last_indices.restype = C.c_uint64
    return _lib


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


IDENTITY = np.array([1.0, 0.0, 0.0, 0.0])


def se2(x: float, y: float, theta: float) -> np.ndarray:
    """Sophus SE2d{theta, (x, y)} as data() order (cos, sin, x, y)."""
    out = np.zeros(4)
    lib().orc_se2_from_xytheta(C.c_double(x), C.c_double(y), C.c_double(theta), _p(out, C.c_double))
    return out


def se2_compose(a, b) -> np.ndarray:
    out = np.zeros(4)
    lib().orc_se2_compose(_p(_f64(a), C.c_double), _p(_f64(b), C.c_double), _p(out, C.c_double))
    return out


def se2_inverse(a) -> np.ndarray:
    out = np.zeros(4)
    lib().orc_se2_inverse(_p(_f64(a), C.c_double), _p(out, C.c_double))
    return out


def philox4x32_10(ctr, key) -> np.ndarray:
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().orc_philox4x32_10(_p(c, C.c_uint32), _p(k, C.c_uint32), _p(out, C.c_uint32))
    return out


@dataclass
class Grid:
    """Occupancy grid: int8 cells (0 free / 100 occupied / -1 unknown), row-major [height, width]."""

    cells: np.ndarray
    resolution: float = 1.0
    origin: np.ndarray = field(default_factory=lambda: IDENTITY.copy())

    def __post_init__(self):
        c = np.asarray(self.cells)
        if c.dtype == np.bool_:
            c = np.where(c, 100, 0)
        self.cells = np.ascontiguousarray(c, dtype=np.int8)
        self.origin = _f64(self.origin)

    @property
    def width(self) -> int:
        return int(self.cells.shape[1])

    @property
    def height(self) -> int:
        return int(self.cells.shape[0])

    def args(self):
        return (_p(self.cells, C.c_int8), C.c_int(self.width), C.c_int(self.height), C.c_double(self.resolution), _p(self.origin, C.c_double))


def distance_map(obstacles, max_distance: float, squared_euclidean: bool = False) -> np.ndarray:
    ob = np.ascontiguousarray(np.atleast_2d(np.asarray(obstacles)), dtype=np.uint8)
    out = np.zeros(ob.shape, dtype=np.float32)
    if ob.size:
        lib().orc_distance_map(_p(ob, C.c_uint8), C.c_int(ob.shape[1]), C.c_int(ob.shape[0]), C.c_float(max_distance), C.c_int(int(squared_euclidean)), _p(out, C.c_float))
    return out


def likelihood_field(param: LfmParam, grid: Grid) -> np.ndarray:
    out = np.zeros(grid.cells.shape, dtype=np.float32)
    rc = lib().orc_likelihood_field(C.byref(param), *grid.args(), _p(out, C.c_float))
    if rc != 0:
        raise RuntimeError(lib().orc_last_error().decode())
    return out


LFM, LFM_PROB, BEAM = 0, 1, 2


def sensor_weights(kind: int, param, grid: Grid, points, states, return_visited: bool = False):
    pts = _f64(points).reshape(-1, 2)
    st = _f64(states).reshape(-1, 4)
    out = np.zeros(len(st))
    visited = C.c_uint64(0)
    rc = lib().orc_sensor_weights(C.c_int(kind), C.byref(param), *grid.args(), _p(pts, C.c_double), C.c_uint64(len(pts)),
                                  _p(st, C.c_double), C.c_uint64(len(st)), _p(out, C.c_double), C.byref(visited))
    if rc != 0:
        raise RuntimeError(lib().orc_last_error().decode())
    return (out, visited.value) if return_visited else out


def bresenham(p0, p1, modified: bool = False) -> np.ndarray:
    cap = 2 * (abs(p1[0] - p0[0]) + abs(p1[1] - p0[1])) + 4
    out = np.zeros((cap, 2), dtype=np.int32)
    n = lib().orc_bresenham(C.c_int(p0[0]), C.c_int(p0[1]), C.c_int(p1[0]), C.c_int(p1[1]), C.c_int(int(modified)), _p(out, C.c_int), C.c_uint64(cap))
    return out[:n]


def raycast(grid: Grid, pose, max_range: float, bearing: float):
    d = C.c_double(0.0)
    hit = lib().orc_raycast(*grid.args(), _p(_f64(pose), C.c_double), C.c_double(max_range), C.c_double(bearing), C.byref(d))
    return d.value if hit else None


def diff_drive_sampling(param: MotionParam, pose, previous_pose) -> np.ndarray:
    out = np.zeros(6)
    lib().orc_diff_drive_sampling(C.byref(param), _p(_f64(pose), C.c_double), _p(_f64(previous_pose), C.c_double), _p(out, C.c_double))
    return out


def diff_drive_propagate(sampling6, states, mode: int, seed: int, step: int = 1, first_index: int = 0) -> np.ndarray:
    st = _f64(states).reshape(-1, 4).copy()
    lib().orc_diff_drive_propagate(_p(_f64(sampling6), C.c_double), C.c_int(mode), C.c_uint64(seed), C.c_uint32(step),
                                   C.c_uint64(first_index), _p(st, C.c_double), C.c_uint64(len(st)))
    return st


def motion_sampling(model: int, param: OmniParam, pose, previous_pose) -> np.ndarray:
    """{mean[3], stddev[3], first_rotation cos, sin, model, 0} of any motion model."""
    out = np.zeros(10)
    lib().orc_motion_sampling(C.c_int(model), C.byref(param), _p(_f64(pose), C.c_double), _p(_f64(previous_pose), C.c_double), _p(out, C.c_double))
    return out


def motion_propagate(sampling10, states, mode: int, seed: int, step: int = 1, first_index: int = 0) -> np.ndarray:
    st = _f64(states).reshape(-1, 4).copy()
    lib().orc_motion_propagate(_p(_f64(sampling10), C.c_double), C.c_int(mode), C.c_uint64(seed), C.c_uint32(step), C.c_uint64(first_index),
                               _p(st, C.c_double), C.c_uint64(len(st)))
    return st


def normalize(weights):
    w = _f64(weights).copy()
    f = lib().orc_normalize(_p(w, C.c_double), C.c_uint64(len(w)))
    return w, f


def effective_sample_size(weights) -> float:
    w = _f64(weights)
    return lib().orc_effective_sample_size(_p(w, C.c_double), C.c_uint64(len(w)))


def thrun(alpha_slow: float, alpha_fast: float, total_weights, sizes) -> np.ndarray:
    tw = _f64(total_weights)
    sz = np.ascontiguousarray(sizes, dtype=np.uint64)
    out = np.zeros(len(tw))
    lib().orc_thrun(C.c_double(alpha_slow), C.c_double(alpha_fast), _p(tw, C.c_double), _p(sz, C.c_uint64), C.c_uint64(len(tw)), _p(out, C.c_double))
    return out


def spatial_hash(state, rx: float, ry: float, rtheta: float) -> int:
    return lib().orc_spatial_hash(_p(_f64(state), C.c_double), C.c_double(rx), C.c_double(ry), C.c_double(rtheta))


def kld_target_size(k: int, epsilon: float, z: float) -> int:
    return lib().orc_kld_target_size(C.c_uint64(k), C.c_double(epsilon), C.c_double(z))


def kld_take_count(hashes, min_: int, max_: int, epsilon: float, z: float = 3.0) -> int:
    h = np.ascontiguousarray(hashes, dtype=np.uint64)
    return lib().orc_kld_take_count(_p(h, C.c_uint64), C.c_uint64(len(h)), C.c_uint64(min_), C.c_uint64(max_), C.c_double(epsilon), C.c_double(z))


def estimate(states, weights):
    st = _f64(states).reshape(-1, 4)
    w = _f64(weights)
    mean = np.zeros(4)
    cov = np.zeros(9)
    lib().orc_estimate(_p(st, C.c_double), _p(w, C.c_double), C.c_uint64(len(st)), _p(mean, C.c_double), _p(cov, C.c_double))
    return mean, cov.reshape(3, 3)


def inject_flags(seed: int, step: int, probability: float, m: int) -> np.ndarray:
    out = np.zeros(m, dtype=np.uint8)
    lib().orc_inject_flags(C.c_uint64(seed), C.c_uint32(step), C.c_double(probability), C.c_uint64(m), _p(out, C.c_uint8))
    return out


def exponential_filter(alpha: float, values, reset_before: int = -1) -> np.ndarray:
    v = _f64(values)
    out = np.zeros(len(v))
    lib().orc_exponential_filter(C.c_double(alpha), _p(v, C.c_double), C.c_uint64(len(v)), C.c_int64(reset_before), _p(out, C.c_double))
    return out


# ---- cluster-based estimate ---------------------------------------------------------------------

def percentile_threshold(values, percentile: float) -> float:
    v = _f64(values)
    fn = lib().orc_percentile_threshold
    fn.restype = C.c_double
    return fn(_p(v, C.c_double), C.c_uint64(len(v)), C.c_double(percentile))


def cluster_ids(states, weights, linear=0.2, angular=0.524, percentile=0.9) -> np.ndarray:
    st = _f64(states).reshape(-1, 4)
    w = _f64(weights)
    out = np.zeros(len(st), dtype=np.uint64)
    lib().orc_cluster_ids(_p(st, C.c_double), _p(w, C.c_double), C.c_uint64(len(st)), C.c_double(linear), C.c_double(angular),
                          C.c_double(percentile), _p(out, C.c_uint64))
    return out


def assign_clusters(cell_states, cell_weights, linear: float, angular: float, n_neighbors: int = 6) -> np.ndarray:
    st = _f64(cell_states).reshape(-1, 4)
    w = _f64(cell_weights)
    out = np.zeros(len(st), dtype=np.uint64)
    lib().orc_assign_clusters(_p(st, C.c_double), _p(w, C.c_double), C.c_uint64(len(st)), C.c_double(linear), C.c_double(angular),
                              C.c_int(n_neighbors), _p(out, C.c_uint64))
    return out


def estimate_clusters(states, weights, clusters):
    """-> list of (cluster id, total weight, mean[4], cov[3,3]) for clusters with more than one particle."""
    st = _f64(states).reshape(-1, 4)
    w = _f64(weights)
    c = np.ascontiguousarray(clusters, dtype=np.uint64)
    cap = len(st)
    wt, mean, cov, ids = np.zeros(cap), np.zeros((cap, 4)), np.zeros((cap, 9)), np.zeros(cap, dtype=np.uint64)
    fn = lib().orc_estimate_clusters
    fn.restype = C.c_uint64
    k = fn(_p(st, C.c_double), _p(w, C.c_double), _p(c, C.c_uint64), C.c_uint64(len(st)), C.c_uint64(cap), _p(wt, C.c_double),
           _p(mean, C.c_double), _p(cov, C.c_double), _p(ids, C.c_uint64))
    return [(int(ids[i]), float(wt[i]), mean[i].copy(), cov[i].reshape(3, 3).copy()) for i in range(k)]


def cluster_based_estimate(states, weights, linear=0.2, angular=0.524, percentile=0.9):
    st = _f64(states).reshape(-1, 4)
    w = _f64(weights)
    mean = np.zeros(4)
    cov = np.zeros(9)
    lib().orc_cluster_based_estimate(_p(st, C.c_double), _p(w, C.c_double), C.c_uint64(len(st)), C.c_double(linear), C.c_double(angular),
                                     C.c_double(percentile), _p(mean, C.c_double), _p(cov, C.c_double))
    return mean, cov.reshape(3, 3)


def normal_transform(cov) -> np.ndarray:
    c = _f64(cov).reshape(9)
    out = np.zeros(9)
    if lib().orc_normal_transform(_p(c, C.c_double), _p(out, C.c_double)) != 0:
        raise RuntimeError(lib().orc_last_error().decode())
    return out.reshape(3, 3)


MULTINOMIAL, SYSTEMATIC = 0, 1


def resample_indices(weights, scheme: int, seed: int, step: int, m: int | None = None, n_total: int = 0):
    """Mode-B indices plus the fixed-point CDF and exponent."""
    w = _f64(weights)
    m = len(w) if m is None else m
    idx = np.zeros(m, dtype=np.int64)
    cdf = np.zeros(len(w), dtype=np.uint64)
    ex = C.c_int(0)
    rc = lib().orc_resample_indices(_p(w, C.c_double), C.c_uint64(len(w)), C.c_uint64(n_total), C.c_int(scheme), C.c_uint64(seed),
                                    C.c_uint32(step), C.c_uint64(m), _p(idx, C.c_int64), _p(cdf, C.c_uint64), C.byref(ex))
    if rc != 0:
        raise RuntimeError(lib().orc_last_error().decode())
    return idx, cdf, ex.value


def resample_indices_std(weights, seed: int, m: int) -> np.ndarray:
    w = _f64(weights)
    idx = np.zeros(m, dtype=np.int64)
    lib().orc_resample_indices_std(_p(w, C.c_double), C.c_uint64(len(w)), C.c_uint64(seed), C.c_uint64(m), _p(idx, C.c_int64))
    return idx


class Amcl:
    """oracle::Amcl -- the CPU restatement of beluga::Amcl (algorithm/amcl_core.hpp:81-233)."""

    def __init__(self, param: AmclParam, motion, motion_model: int = DIFFERENTIAL):
        if isinstance(motion, MotionParam):
            motion = OmniParam(motion.alpha1, motion.alpha2, motion.alpha3, motion.alpha4, 0.0, motion.distance_threshold)
        self._h = C.c_void_p(lib().orc_amcl_create_motion(C.byref(param), C.c_int(motion_model), C.byref(motion)))
        self._grid = None

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_amcl_destroy(self._h)
            self._h = None

    def set_map(self, kind: int, param, grid: Grid):
        self._grid = grid
        if lib().orc_amcl_set_map(self._h, C.c_int(kind), C.byref(param), *grid.args()) != 0:
            raise RuntimeError(lib().orc_last_error().decode())

    def likelihood_field(self) -> np.ndarray:
        out = np.zeros(self._grid.cells.shape, dtype=np.float32)
        if lib().orc_amcl_get_likelihood_field(self._h, _p(out, C.c_float)) != 0:
            raise RuntimeError("no likelihood field model set")
        return out

    def initialize_normal(self, mean_xyt, cov):
        if lib().orc_amcl_initialize_normal(self._h, _p(_f64(mean_xyt), C.c_double), _p(_f64(cov).reshape(9), C.c_double)) != 0:
            raise RuntimeError(lib().orc_last_error().decode())

    def initialize_from_map(self):
        if lib().orc_amcl_initialize_from_map(self._h) != 0:
            raise RuntimeError(lib().orc_last_error().decode())

    def set_particles(self, states, weights):
        st = _f64(states).reshape(-1, 4)
        w = _f64(weights)
        lib().orc_amcl_set_particles(self._h, _p(st, C.c_double), _p(w, C.c_double), C.c_uint64(len(st)))

    def particles(self):
        n = lib().orc_amcl_size(self._h)
        st = np.zeros((n, 4))
        w = np.zeros(n)
        lib().orc_amcl_get_particles(self._h, _p(st, C.c_double), _p(w, C.c_double))
        return st, w

    def last_indices(self) -> np.ndarray:
        n = lib().orc_amcl_last_indices(self._h, None, C.c_uint64(0))
        out = np.zeros(n, dtype=np.int64)
        lib().orc_amcl_last_indices(self._h, _p(out, C.c_int64), C.c_uint64(n))
        return out

    def force_update(self):
        lib().orc_amcl_force_update(self._h)

    def update(self, control_pose, points) -> UpdateResult:
        pts = _f64(points).reshape(-1, 2)
        res = UpdateResult()
        if lib().orc_amcl_update(self._h, _p(_f64(control_pose), C.c_double), _p(pts, C.c_double), C.c_uint64(len(pts)), C.byref(res)) != 0:
            raise RuntimeError(lib().orc_last_error().decode())
        return res
