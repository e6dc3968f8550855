"""The unclamped lookup of reweight_lfm_fixed_*_kernel (csrc/kernels.cu: fixed_lookup_in_map), replayed on the CPU.

A warp whose particles' scans all stay on the bordered map skips the clamp and feeds the raw high words of the fixed-point
sums, biases included, to the index arithmetic; the table base it adds them to is moved back by fixed_index_bias(kx)
elements (FieldView::bordered_biased, set up in filter.cu).  Three claims make that exact:

  * the biased index is the bordered index plus fixed_index_bias(kx), for every padded cell and both fraction bits;
  * the in-map predicate of fixed_particle_setup is conservative: an end point of a particle on the predicate's boundary,
    at any heading, still lands in the bordered map (cells -1 .. side);
  * no supported map side lets bias + table size reach 2^32, so the host never has to turn the unclamped loop off.

CPU only; it models the arithmetic, it does not run the kernel."""
import math
import struct
from fractions import Fraction

import numpy as np
import pytest

MAGIC_X, MAGIC_Y = 393216.0, 1572864.0  # kFixedMagicX / kFixedMagicY
GUARD_X, GUARD_Y = 2.0 ** -33, 2.0 ** -31  # kFixedGuardX / kFixedGuardY
BIAS_X, BIAS_Y = 0x41180000, 0x41380000  # kFixedBiasX / kFixedBiasY (kernels.cuh)
MAX_SIDE = 8000  # kFixedMaxSide: largest padded side of the fixed-point kernel


def fixed_index_bias(kx: int) -> int:
    """kernels.cuh: fixed_index_bias -- (kFixedBiasY * 4 * 2^kx + kFixedBiasX) mod 2^32."""
    return (BIAS_Y * (4 << kx) + BIAS_X) & 0xFFFFFFFF


def border_kx(width: int) -> int:
    """filter.cu: the smallest kx with 2^kx tiles of four padded cells per row."""
    kx = 0
    while (1 << kx) < (width + 2 + 3) // 4:
        kx += 1
    return kx


def table_size(width: int, height: int) -> int:
    return ((height + 2 + 3) // 4) << (border_kx(width) + 4)


def bordered_index(px: int, py: int, kx: int) -> int:
    return ((py >> 2) << (kx + 4)) | ((px >> 2) << 4) | ((px & 3) << 2) | (py & 3)


def index_tail(hx: int, hy: int, kx: int) -> int:
    """The lookup's integer tail on 32-bit words: bit-select (lop3 0xB8, immediate 3), mask, multiply-add by 4 * 2^kx."""
    low = (hx & ~3 & 0xFFFFFFFF) | (hy & 3)
    return ((hy & ~3 & 0xFFFFFFFF) * (4 << kx) + low) & 0xFFFFFFFF


def fma(a: float, b: float, c: float) -> float:
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def hi_word(t: float) -> int:
    return struct.unpack("<Q", struct.pack("<d", t))[0] >> 32


@pytest.mark.parametrize("width,height", [(5, 7), (64, 33), (200, 200), (2000, 9)])
def test_biased_index_is_the_bordered_index_plus_the_folded_bias(width, height):
    kx = border_kx(width)
    bias = fixed_index_bias(kx)
    size = table_size(width, height)
    assert bias + size <= 1 << 32  # the host check passes for these maps
    for py in range(height + 2):
        for px in range(width + 2):
            want = bordered_index(px, py, kx)
            for frac in range(4):
                hx, hy = BIAS_X + 4 * px + frac, BIAS_Y + py  # raw high words: the biases' low 19 bits are clear
                got = index_tail(hx, hy, kx)
                # as the 32-bit index the kernel adds to bordered_biased = bordered - bias: no wrap in between
                assert got - bias == want


def particle(tx, ty, c, s, inv, radius, width, height):
    """fixed_particle_setup's per-particle values: (cx, sx, ox, oy, in_map)."""
    cx, sx = c * inv, s * inv
    ox = (tx * inv + 1.0) + (MAGIC_X + GUARD_X)
    oy = (ty * inv + 1.0) + (MAGIC_Y + GUARD_Y)
    r = radius * max(abs(cx), abs(sx)) + 0.5
    gx, gy = tx * inv + 1.0, ty * inv + 1.0
    in_map = gx - r >= 0.0 and gx + r <= float(width + 2) and gy - r >= 0.0 and gy + r <= float(height + 2)
    return cx, sx, ox, oy, in_map


def padded_cells(px, py, cx, sx, ox, oy):
    """The cells fixed_lookup_in_map reads, from the high words without any clamp: (4 * padded x + fraction, padded y)."""
    gx = fma(px, cx, fma(-py, sx, ox))
    gy = fma(px, sx, fma(py, cx, oy))
    return hi_word(gx) - BIAS_X, hi_word(gy) - BIAS_Y


def test_end_points_of_particles_on_the_in_map_boundary_stay_in_the_border():
    """Particles placed on (and a few ulps either side of) each of the four edges of the in-map predicate, at random headings,
    with the scan's extreme points (the corners of the L1 ball that points_radius bounds): wherever the predicate holds, every
    end point's cell is within -1 .. side, i.e. padded 0 .. side + 1, and the unclamped index is the clamped one."""
    rng = np.random.default_rng(7)
    checked = 0
    for width, height, res in ((400, 300, 0.05), (2000, 2000, 0.05), (37, 90, 1.0 / 3.0)):
        inv = 1.0 / res
        for _ in range(150):
            theta = float(rng.uniform(-math.pi, math.pi))
            c, s = math.cos(theta), math.sin(theta)
            radius = float(rng.uniform(0.0, 0.4)) * min(width, height) * res
            pts = [(radius, 0.0), (-radius, 0.0), (0.0, radius), (0.0, -radius)]
            pts += [tuple(v) for v in rng.uniform(-1.0, 1.0, (4, 2)) * radius / 2.0]
            r_cells = radius * inv * max(abs(c), abs(s)) + 0.5
            inner_x = float(rng.uniform(r_cells, width + 2 - r_cells) - 1.0) * res
            inner_y = float(rng.uniform(r_cells, height + 2 - r_cells) - 1.0) * res
            # the four boundary positions, solved in exact arithmetic and rounded once
            edges = [(0, (r_cells - 1.0) * res, inner_y), (0, (width + 1 - r_cells) * res, inner_y),
                     (1, inner_x, (r_cells - 1.0) * res), (1, inner_x, (height + 1 - r_cells) * res)]
            for axis, ex, ey in edges:
                for k in range(-3, 4):
                    tx = ex + k * 64 * math.ulp(ex) if axis == 0 else ex
                    ty = ey + k * 64 * math.ulp(ey) if axis == 1 else ey
                    cx, sx, ox, oy, in_map = particle(tx, ty, c, s, inv, radius, width, height)
                    if not in_map:
                        continue
                    kx = border_kx(width)
                    for px, py in pts:
                        ux4, uy = padded_cells(px, py, cx, sx, ox, oy)
                        assert 0 <= ux4 <= 4 * (width + 1) + 3 and 0 <= uy <= height + 1, (width, height, theta, tx, ty, px, py)
                        # the clamped lookup (min against x_max, y_max) would have read the same element
                        clamped = index_tail(min(ux4, 4 * (width + 1) + 3), min(uy, height + 1), kx)
                        assert index_tail(ux4 + BIAS_X, uy + BIAS_Y, kx) - fixed_index_bias(kx) == clamped
                        checked += 1
    assert checked > 5000


def test_in_map_predicate_rejects_particles_that_reach_off_the_map_and_nan():
    inv, width, height = 20.0, 400, 300
    assert particle(10.0, 7.5, 1.0, 0.0, inv, 4.0, width, height)[4]
    assert not particle(17.0, 7.5, 1.0, 0.0, inv, 4.0, width, height)[4]  # 17 m + 4 m > 20.05 m
    assert not particle(10.0, 12.0, 0.0, 1.0, inv, 4.0, width, height)[4]  # 12 m + 4 m > 15.05 m
    assert not particle(float("nan"), 7.5, 1.0, 0.0, inv, 4.0, width, height)[4]
    assert not particle(10.0, 7.5, 1.0, 0.0, inv, float("nan"), width, height)[4]


def test_host_wrap_check_keeps_the_in_map_loop_for_every_supported_map_side():
    """filter.cu turns the unclamped loop off when fixed_index_bias(kx) + table size exceeds 2^32.  Every width the fixed-point
    kernel accepts (padded side up to kFixedMaxSide) gives a row pitch 4 * 2^kx with kx in 0 .. 11; at the tallest supported map
    none of them wraps, so the unclamped loop is available on every map the fixed-point kernel runs on."""
    tallest = MAX_SIDE - 2
    kxs = sorted({border_kx(w) for w in range(1, MAX_SIDE - 1)})
    assert kxs == list(range(12))
    for kx in kxs:
        width = next(w for w in range(1, MAX_SIDE - 1) if border_kx(w) == kx)
        assert fixed_index_bias(kx) + table_size(width, tallest) <= 1 << 32, kx
