// Hand-written sm_100a kernels of the MCL particle-filter update.
//
// One filter step on the device (fixed particle count, resample every step):
//
//   begin_step            zero the per-filter scalars
//   propagate             a2 + a6 of SURVEY.md section 8(a): Philox normals, SE2 compose; cloud moments
//   schedule_*            counting sort of the particles over pose bins (execution order only)
//   reweight_lfm / _beam  a3 / a4 + a5: B likelihood-field lookups (or ray casts) per particle in
//                         schedule order, w *= L written to the particle's own slot, block max of w
//   prepare_cdf           exponent of the fixed-point grid from the largest weight
//   quantize_scan         q = floor(w * 2^e), single-pass decoupled look-back inclusive scan (u64)
//   resample              a10 + a11 + a13: one thread per output slot; counter draw, CDF search,
//                         32-byte state gather, w = 1, per-block raw moments for a14
//   reduce_partials       fixed-order sum of the per-block moments
//
// All floating-point arithmetic that decides a likelihood-field cell or a weight follows the
// reference's operation order without FMA contraction (the file is compiled with -fmad=false).
#include "kernels.cuh"

#include <cstdlib>
#include <cstring>

// Tuning knobs of the reweight kernel (overridable with -D from beluga_b200/build.py).
#ifndef BB200_RW_THREADS
#define BB200_RW_THREADS 256
#endif
#ifndef BB200_RW_UNROLL
#define BB200_RW_UNROLL 4
#endif
#ifndef BB200_RW_BLOCKS
#define BB200_RW_BLOCKS 4
#endif
#ifndef BB200_RW_CHUNK
#define BB200_RW_CHUNK 0  // > 0: experiment -- chunks of adjacent tasks per CTA instead of one global ticket per warp
#endif
#ifndef BB200_RS_UNROLL
#define BB200_RS_UNROLL 2  // particles per thread and round in resample_scatter_kernel
#endif
#ifndef BB200_RS_BLOCKS
#define BB200_RS_BLOCKS 3  // resident CTAs per SM the kernel is compiled for (register cap); measured at 1M (blocks, unroll):
                          // (2, 4) 34.9 us, (3, 4) 45.7 (spills), (4, 2) 39.0, (3, 2) 31.2
#endif

#include <algorithm>
#include <cfloat>

namespace bb200 {

namespace {

constexpr int kWarp = 32;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- fixed-order block reductions --------------------------------------------------------------

template <int kThreads>
__device__ __forceinline__ double block_sum(double v, double* scratch /* kThreads/32 doubles */) {
#pragma unroll
  for (int off = kWarp / 2; off > 0; off >>= 1) v = v + __shfl_down_sync(0xffffffffu, v, off);
  const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
  __syncthreads();  // scratch may still be read by a previous call
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  double total = 0.0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < kThreads / kWarp; ++w) total = total + scratch[w];
  }
  return total;  // valid in thread 0
}

/// Fixed-order block sums of K values at once: warp tree per value, one shared-memory round for all
/// of them, then thread 0 adds the per-warp partials in warp order.  Two barriers instead of 2K.
template <int kThreads, int K>
__device__ __forceinline__ void block_sum_many(double* v /* K values, in/out: totals valid in thread 0 */, double* scratch /* K * kThreads/32 */) {
  constexpr int kWarps = kThreads / kWarp;
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int off = kWarp / 2; off > 0; off >>= 1) v[k] = v[k] + __shfl_down_sync(0xffffffffu, v[k], off);
  }
  const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) scratch[k * kWarps + warp] = v[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double total = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) total = total + scratch[k * kWarps + w];
      v[k] = total;
    }
  }
}

template <int kThreads>
__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* scratch) {
#pragma unroll
  for (int off = kWarp / 2; off > 0; off >>= 1) {
    const unsigned long long o = __shfl_down_sync(0xffffffffu, v, off);
    v = o > v ? o : v;
  }
  const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  unsigned long long m = 0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < kThreads / kWarp; ++w) m = scratch[w] > m ? scratch[w] : m;
  }
  return m;
}

/// Positive finite weights order like their bit patterns; anything else counts as 0.
__device__ __forceinline__ unsigned long long weight_order_bits(double w) {
  return (w > 0.0 && w <= DBL_MAX) ? static_cast<unsigned long long>(__double_as_longlong(w)) : 0ull;
}

// ---- TMA 1-D bulk copy of the scan points into shared memory ------------------------------------

__device__ __forceinline__ void mbarrier_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarrier_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbarrier_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_global, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst_smem)),
               "l"(src_global), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void mbarrier_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "BB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra BB_DONE;\n"
      "bra BB_WAIT;\n"
      "BB_DONE:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}

__device__ __forceinline__ Pose2 load_pose(const Pose2* p) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *(reinterpret_cast<const double2*>(p) + 1);
  return Pose2{a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ void store_pose(Pose2* p, const Pose2& v) {
  *reinterpret_cast<double2*>(p) = make_double2(v.c, v.s);
  *(reinterpret_cast<double2*>(p) + 1) = make_double2(v.x, v.y);
}

// ---- begin_step ----------------------------------------------------------------------------------

__global__ void begin_step_kernel(Scalars* s) {
  s->wmax_bits = 0;
  s->tile_ticket = 0;
  s->total = 0;
  s->exponent = 0;
  s->valid = 0;
  s->kld_cutoff = ~0ull;
  s->work_ticket = 0;  // normally rewound by the persistent reweight kernel itself; a step starts clean regardless
  s->work_done = 0;
  s->blocks_done = 0;
}

/// The fused step's reset: the scalars above plus the scan state of the CDF build and -- when the execution schedule
/// is rebuilt this step -- the bin counters, the schedule's scan state and its moment sums.  One launch instead of a
/// scalar kernel, two memsets and a reset kernel.
struct StepReset {
  Scalars* scalars;
  unsigned long long* tile_state;
  uint32_t n_tiles;
  Schedule* sched;             // nullable
  uint32_t* counters;          // nullable
  uint32_t n_counters;
  unsigned long long* sched_tiles;
  uint32_t n_sched_tiles;
  const char* prefetch;        // nullable: a table the step is about to gather from (pulled into L2 while propagate runs)
  uint64_t prefetch_lines;     // its size in 128-byte lines
};

__global__ void __launch_bounds__(256) begin_fused_step_kernel(StepReset r) {
  const uint32_t t = blockIdx.x * 256 + threadIdx.x, stride = gridDim.x * 256;
  if (t == 0) {
    Scalars* s = r.scalars;
    s->wmax_bits = 0;
    s->tile_ticket = 0;
    s->total = 0;
    s->exponent = 0;
    s->valid = 0;
    s->kld_cutoff = ~0ull;
    s->work_ticket = 0;
    s->work_done = 0;
    s->blocks_done = 0;
    if (r.sched != nullptr) {
      for (int k = 0; k < 6; ++k) r.sched->sums[k] = 0.0;
      r.sched->tile_ticket = 0;
    }
  }
  for (uint32_t k = t; k < r.n_tiles; k += stride) r.tile_state[k] = 0;
  if (r.counters != nullptr) {
    uint4* c4 = reinterpret_cast<uint4*>(r.counters);  // cudaMalloc alignment; n_counters is a multiple of 4
    for (uint32_t k = t; k < r.n_counters / 4; k += stride) c4[k] = make_uint4(0u, 0u, 0u, 0u);
    for (uint32_t k = t; k < r.n_sched_tiles; k += stride) r.sched_tiles[k] = 0;
  }
  // The likelihood table is gathered from at random by the reweight kernel; after an L2 flush (or a map-sized
  // working set) its first touches would be demand misses to HBM, paid at full latency by warps that have nothing
  // else to do when a shard is small.  Streaming it into L2 now costs a few microseconds of HBM bandwidth that the
  // FP64-bound propagate kernel does not use.
  for (uint64_t k = t; k < r.prefetch_lines; k += stride) asm volatile("prefetch.global.L2 [%0];" ::"l"(r.prefetch + k * 128));
}

// ---- initialize_normal (a16) ---------------------------------------------------------------------
// MultivariateNormalDistribution<SE2d>: (x, y, theta) = mean + T * delta, SE2(exp(theta), (x, y))
// (random/multivariate_normal_distribution.hpp:96-103, multivariate_distribution_traits.hpp:110-112).

struct NormalInit {
  double mean[3];
  double t[9];
};

__global__ void __launch_bounds__(256) initialize_normal_kernel(Pose2* states, double* weights, uint64_t n, NormalInit p, uint64_t seed,
                                                                uint64_t first_index) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double d0, d1, d2, unused;
  box_muller(counter_draw(seed, first_index + i, 0, kStreamInit0), d0, d1);
  box_muller(counter_draw(seed, first_index + i, 0, kStreamInit1), d2, unused);
  double v[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) v[r] = p.mean[r] + (p.t[3 * r + 0] * d0 + p.t[3 * r + 1] * d1 + p.t[3 * r + 2] * d2);
  const Rot2 r = rot_exp(v[2]);
  states[i] = Pose2{r.c, r.s, v[0], v[1]};
  weights[i] = 1.0;
}

/// MultivariateUniformDistribution<SE2d, OccupancyGrid> (random/multivariate_uniform_distribution.hpp:143-160): a free
/// cell drawn uniformly, its centroid in the global frame (occupancy_grid.hpp:150-156,166-172), yaw ~ U[-pi, pi).
struct FreeSpace {
  const uint32_t* cells;  // row-major indices of the free cells
  uint64_t n;
  int grid_width;
  double resolution;
  Pose2 origin;
};

__device__ __forceinline__ Pose2 random_free_state(const FreeSpace& fs, const Draw& r) {
  const uint32_t cell = fs.cells[mulhi64(r.a, fs.n)];
  const double pi = 3.14159265358979323846;
  const double yaw = uniform01(r.b) * (pi - (-pi)) + (-pi);
  const double lx = (static_cast<double>(static_cast<int>(cell % static_cast<uint32_t>(fs.grid_width))) + 0.5) * fs.resolution;
  const double ly = (static_cast<double>(static_cast<int>(cell / static_cast<uint32_t>(fs.grid_width))) + 0.5) * fs.resolution;
  const Rot2 rot = rot_exp(yaw);
  return Pose2{rot.c, rot.s, (fs.origin.c * lx - fs.origin.s * ly) + fs.origin.x, (fs.origin.s * lx + fs.origin.c * ly) + fs.origin.y};
}

// initialize_from_map (a16; beluga_ros/include/beluga_ros/amcl.hpp:192-209): max_particles samples of the map
// distribution, weights 1.  Counter stream 6 at step 0, keyed by the global particle index.
__global__ void __launch_bounds__(256) initialize_uniform_kernel(Pose2* states, double* weights, uint64_t n, FreeSpace fs, uint64_t seed,
                                                                 uint64_t first_index) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  store_pose(states + i, random_free_state(fs, counter_draw(seed, first_index + i, 0, kStreamRandomState)));
  weights[i] = 1.0;
}

// ---- propagate (a2 + a6) --------------------------------------------------------------------------
// One thread per particle, original order.  Also accumulates the first and second moments of the
// propagated cloud (block reduction + double atomics); they only feed the execution schedule below,
// never a result, so their summation order does not matter.

constexpr int kPrThreads = 256;

__device__ __forceinline__ Pose2 propagate_one(const Pose2& st, const MotionSampling& p, uint64_t seed, uint64_t index, uint32_t step) {
  double z0, z1;
  box_muller_fast(counter_draw(seed, index, step, kStreamMotion0), z0, z1);
  const double z2 = box_muller_first(counter_draw(seed, index, step, kStreamMotion1));
  // std::normal_distribution: ret * stddev + mean (libstdc++ bits/random.tcc:1843)
  const double d0 = z0 * p.stddev[0] + p.mean[0];
  const double d1 = z1 * p.stddev[1] + p.mean[1];
  const double d2 = z2 * p.stddev[2] + p.mean[2];
  return motion_apply_fast(p.model, st, d0, d1, d2, Rot2{p.first_c, p.first_s});
}

__global__ void __launch_bounds__(kPrThreads) propagate_kernel(Pose2* __restrict__ states, uint64_t n, int do_propagate, MotionSampling sampling,
                                                               uint64_t seed, uint32_t step, uint64_t first_index, Schedule* __restrict__ sched) {
  __shared__ double s_red[6 * kPrThreads / kWarp];
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kPrThreads + threadIdx.x;
  double m[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (i < n) {
    Pose2 st = load_pose(states + i);
    if (do_propagate) {
      st = propagate_one(st, sampling, seed, first_index + i, step);
      store_pose(states + i, st);
    }
    m[0] = st.c, m[1] = st.s, m[2] = st.x, m[3] = st.y, m[4] = st.x * st.x, m[5] = st.y * st.y;
  }
  if (sched != nullptr) {
    block_sum_many<kPrThreads, 6>(m, s_red);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < 6; ++k) atomicAdd(&sched->sums[k], m[k]);
    }
  }
}

// ---- execution schedule ---------------------------------------------------------------------------
// The likelihood-field lookup of beam k lands, for two particles, in nearby cells only if their poses
// are close (x, y, and theta scaled by the beam range).  The posterior is wide, so in index order the
// 32 lanes of a warp gather from ~31 distinct 32-byte sectors and the kernel is bound by L2 sector
// bandwidth (profiles/r01_lfm_v1_*).  The reweight kernels therefore walk the particles in the order
// of a counting sort over a 3-D grid of pose bins.  This only permutes WHICH THREAD handles a
// particle: weights are written back to the particle's own slot, so every result is independent of it.

constexpr uint32_t kMaxBins = kScheduleMaxBins;

__global__ void schedule_reset_kernel(Schedule* sched) {
  for (int k = 0; k < 6; ++k) sched->sums[k] = 0.0;
  sched->tile_ticket = 0;
}

__global__ void schedule_params_kernel(Schedule* sched, uint64_t n, double mean_range, double min_bin, double per_bin, double x_split,
                                       bool equal_mass) {
  const double inv_n = 1.0 / static_cast<double>(n);
  const double mx = sched->sums[2] * inv_n, my = sched->sums[3] * inv_n;
  schedule_from_moments(*sched, sched->sums[0] * inv_n, sched->sums[1] * inv_n, mx, my, sched->sums[4] * inv_n - mx * mx,
                        sched->sums[5] * inv_n - my * my, static_cast<double>(n), mean_range, min_bin, per_bin, x_split, equal_mass);
}

__device__ __forceinline__ uint32_t schedule_bin(const Schedule& g, const Pose2& st) {
  // heading relative to the mean as u = 2 tan(dtheta / 2): monotone in dtheta, one division instead of an atan2
  const double cr = st.c * g.c0 + st.s * g.s0, sr = st.s * g.c0 - st.c * g.s0;
  const double u = cr > -0.4 ? 2.0 * sr / (1.0 + cr) : (sr >= 0.0 ? 1e6 : -1e6);
  int bt, bx, by;
  if (g.equal_mass != 0u) {
    // CDF value of each coordinate (single precision: the bin only decides which thread handles the particle)
    const float zt = static_cast<float>(u) * g.kt, zx = static_cast<float>(st.x - g.mx) * g.kx, zy = static_cast<float>(st.y - g.my) * g.ky;
    const float ft = __fdividef(static_cast<float>(g.nt), 1.0f + __expf(-zt));  // exp overflow -> 0, underflow -> count: the edge bins
    const float fx = __fdividef(static_cast<float>(g.nx), 1.0f + __expf(-zx));
    const float fy = __fdividef(static_cast<float>(g.ny), 1.0f + __expf(-zy));
    bt = min(max(__float2int_rz(ft), 0), static_cast<int>(g.nt) - 1);  // NaN converts to 0
    bx = min(max(__float2int_rz(fx), 0), static_cast<int>(g.nx) - 1);
    by = min(max(__float2int_rz(fy), 0), static_cast<int>(g.ny) - 1);
  } else {
    bt = min(max(static_cast<int>(fmin(fmax((u + g.half_u) * g.scale_t, 0.0), 1e6)), 0), static_cast<int>(g.nt) - 1);
    bx = min(max(static_cast<int>(fmin(fmax((st.x - g.x0) * g.scale_x, 0.0), 1e6)), 0), static_cast<int>(g.nx) - 1);
    by = min(max(static_cast<int>(fmin(fmax((st.y - g.y0) * g.scale_y, 0.0), 1e6)), 0), static_cast<int>(g.ny) - 1);
  }
  // Boustrophedon order: every other row runs backwards in x and every other plane backwards in y, so that consecutive
  // bins are always neighbours (a warp crossing a row end would otherwise span the whole cloud).
  if (bt & 1) by = static_cast<int>(g.ny) - 1 - by;
  const uint32_t row = static_cast<uint32_t>(bt) * g.ny + static_cast<uint32_t>(by);
  if (row & 1u) bx = static_cast<int>(g.nx) - 1 - bx;
  return row * g.nx + static_cast<uint32_t>(bx);
}

/// propagate with the histogram of the execution schedule fused in (the bin grid comes from the host's prediction).
__global__ void __launch_bounds__(kPrThreads) propagate_binned_kernel(Pose2* __restrict__ states, uint64_t n, MotionSampling sampling, uint64_t seed,
                                                                      uint32_t step, uint64_t first_index, Schedule grid,
                                                                      uint2* __restrict__ bin_rank, uint32_t* __restrict__ counters) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kPrThreads + threadIdx.x;
  if (i < n) {
    const Pose2 st = propagate_one(load_pose(states + i), sampling, seed, first_index + i, step);
    store_pose(states + i, st);
    const uint32_t b = schedule_bin(grid, st);
    // The particle's arrival rank inside its bin: the scatter pass then needs no second round of atomics.  (Which
    // particle gets which rank varies from run to run; it only permutes the execution order inside a bin.)
    const uint32_t rank = atomicAdd(counters + b, 1u);
    bin_rank[i] = make_uint2(b, rank);
  }
}

constexpr int kPlaceItems = 4;  // particles per thread: the bin-offset gathers of one thread are independent
__global__ void __launch_bounds__(256) schedule_place_kernel(const uint2* __restrict__ bin_rank, uint64_t n, const uint32_t* __restrict__ offsets,
                                                             uint32_t* __restrict__ perm) {
  const uint64_t first = static_cast<uint64_t>(blockIdx.x) * (256 * kPlaceItems) + threadIdx.x;
  uint2 br[kPlaceItems];
  uint32_t off[kPlaceItems];
#pragma unroll
  for (int k = 0; k < kPlaceItems; ++k) {
    const uint64_t i = first + static_cast<uint64_t>(k) * 256;
    br[k] = i < n ? __ldcs(bin_rank + i) : make_uint2(0u, 0u);
  }
#pragma unroll
  for (int k = 0; k < kPlaceItems; ++k) off[k] = __ldg(offsets + br[k].x);
#pragma unroll
  for (int k = 0; k < kPlaceItems; ++k) {
    const uint64_t i = first + static_cast<uint64_t>(k) * 256;
    if (i < n) perm[off[k] + br[k].y] = static_cast<uint32_t>(i);
  }
}

__global__ void __launch_bounds__(256) schedule_histogram_kernel(const Pose2* __restrict__ states, uint64_t n, const Schedule* __restrict__ sched,
                                                                 uint32_t* __restrict__ bins, uint32_t* __restrict__ counters) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= n) return;
  const uint32_t b = schedule_bin(*sched, load_pose(states + i));
  bins[i] = b;
  atomicAdd(counters + b, 1u);
}

__global__ void __launch_bounds__(256) schedule_scatter_kernel(const uint32_t* __restrict__ bins, uint64_t n, uint32_t* __restrict__ offsets,
                                                               uint32_t* __restrict__ perm) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= n) return;
  perm[atomicAdd(offsets + bins[i], 1u)] = static_cast<uint32_t>(i);
}

// ---- reweight (likelihood field; a3 + a5) --------------------------------------------------------

constexpr int kRwThreads = BB200_RW_THREADS;  // x kRwBlocksPerSm CTAs per SM
constexpr int kRwBlocksPerSm = BB200_RW_BLOCKS;
constexpr int kRwUnroll = BB200_RW_UNROLL;  // groups of four beams per trip of the beam loop
constexpr uint32_t kChunkBeams = 2048; // beams staged per shared-memory chunk (32 KB), multiple of 4

/// floor(g) as int32 for |g| < 2^31: one F2I.F64.FLOOR (saturating).
__device__ __forceinline__ int floor_to_int_fast(double g) { return __double2int_rd(g); }

template <bool kFast, bool kTiled>
__device__ __forceinline__ double field_lookup(const FieldView& f, double px, double py, double c, double s, double tx, double ty) {
  // likelihood_field_model.hpp:82-83 -- two products, one difference/sum, one offset; each rounded.
  const double x = (px * c - py * s) + tx;
  const double y = (px * s + py * c) + ty;
  // regular_grid.hpp:75-78 -- floor(p * inv_resolution) cast to int.
  const double gx = x * f.inv_resolution;
  const double gy = y * f.inv_resolution;
  int xi, yi;
  if (kFast) {
    xi = floor_to_int_fast(gx);
    yi = floor_to_int_fast(gy);
  } else {
    // General path: saturating conversion; non-finite coordinates fall outside the grid.
    const double fx = floor(gx), fy = floor(gy);
    xi = (fx >= 0.0 && fx < 2147483647.0) ? static_cast<int>(fx) : -1;
    yi = (fy >= 0.0 && fy < 2147483647.0) ? static_cast<int>(fy) : -1;
  }
  // dense_grid.hpp:92-96 contains().  Out-of-grid end points read the spare cell that holds
  // f(unknown_space_occupancy_prob), so the load is unconditional (no divergent branch).
  const bool inside = static_cast<unsigned>(xi) < static_cast<unsigned>(f.width) && static_cast<unsigned>(yi) < static_cast<unsigned>(f.height);
  uint32_t idx;
  if (kTiled) {
    const uint32_t ux = static_cast<uint32_t>(xi), uy = static_cast<uint32_t>(yi);
    idx = (((uy >> 2) * static_cast<uint32_t>(f.tiles_x) + (ux >> 2)) << 4) | ((uy & 3u) << 2) | (ux & 3u);
  } else {
    idx = static_cast<uint32_t>(yi) * static_cast<uint32_t>(f.width) + static_cast<uint32_t>(xi);  // linear_grid.hpp:73-75
  }
  idx = inside ? idx : f.spare_index;
  return __ldg((kTiled ? f.tiled : f.table) + idx);
}

template <bool kFast, bool kTiled>
__device__ __forceinline__ double accumulate_chunk(const FieldView& f, const double2* pts, uint32_t count, double acc, double c, double s,
                                                   double tx, double ty) {
  // libstdc++ std::transform_reduce (numeric:439-462): groups of four, init += ((f0+f1)+(f2+f3)).
  uint32_t b = 0;
#pragma unroll kRwUnroll
  for (; b + 4 <= count; b += 4) {
    const double2 p0 = pts[b], p1 = pts[b + 1], p2 = pts[b + 2], p3 = pts[b + 3];
    const double f0 = field_lookup<kFast, kTiled>(f, p0.x, p0.y, c, s, tx, ty);
    const double f1 = field_lookup<kFast, kTiled>(f, p1.x, p1.y, c, s, tx, ty);
    const double f2 = field_lookup<kFast, kTiled>(f, p2.x, p2.y, c, s, tx, ty);
    const double f3 = field_lookup<kFast, kTiled>(f, p3.x, p3.y, c, s, tx, ty);
    acc = acc + ((f0 + f1) + (f2 + f3));
  }
  for (; b < count; ++b) acc = acc + field_lookup<kFast, kTiled>(f, pts[b].x, pts[b].y, c, s, tx, ty);
  return acc;
}

/// Block-wide max of the weight bit patterns without a closing barrier: every warp folds its max
/// into a shared word and the last warp to arrive publishes the block's value.  Warps that finish
/// their beams early retire instead of idling at a __syncthreads.
__device__ __forceinline__ void publish_weight_max(unsigned long long bits, unsigned long long* s_max, unsigned int* s_arrived,
                                                   unsigned int n_warps, Scalars* scalars) {
#pragma unroll
  for (int off = kWarp / 2; off > 0; off >>= 1) {
    const unsigned long long o = __shfl_down_sync(0xffffffffu, bits, off);
    bits = o > bits ? o : bits;
  }
  if (threadIdx.x % kWarp == 0) {
    atomicMax(s_max, bits);
    __threadfence_block();
    if (atomicAdd(s_arrived, 1u) + 1u == n_warps) {
      const unsigned long long m = atomicMax(s_max, 0ull);  // read the final value
      if (m != 0) atomicMax(&scalars->wmax_bits, m);
    }
  }
}

template <bool kTiled>
__global__ void __launch_bounds__(kRwThreads, kRwBlocksPerSm)
    reweight_lfm_kernel(const Pose2* __restrict__ states, double* __restrict__ weights, uint64_t n, const uint32_t* __restrict__ perm,
                        FieldView field, const double2* __restrict__ points, uint32_t n_points, double points_radius,
                        Scalars* __restrict__ scalars) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* s_pts = reinterpret_cast<double2*>(smem_raw);
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ unsigned long long s_max;
  __shared__ unsigned int s_arrived;

  const uint64_t slot = static_cast<uint64_t>(blockIdx.x) * kRwThreads + threadIdx.x;
  const bool active = slot < n;
  const uint64_t i = active ? (perm != nullptr ? perm[slot] : slot) : 0;

  if (threadIdx.x == 0) {
    s_max = 0ull;
    s_arrived = 0u;
    mbarrier_init(&s_bar, 1);
    mbarrier_init_fence();
  }
  Pose2 st{1.0, 0.0, 0.0, 0.0};
  double w = 0.0;
  if (active) {
    st = load_pose(states + i);
    w = weights[i];
  }
  // transform = world_to_likelihood_field * state (likelihood_field_model.hpp:70-74)
  const Pose2 t = pose_mul(field.world_to_field, st);
  // Fast floor is exact while every |coordinate * inv_resolution| stays below 2^30.
  const double reach = (points_radius + fmax(fabs(t.x), fabs(t.y))) * field.inv_resolution;
  const bool fast = reach < 1073741824.0;  // false for NaN
  double acc = field.init;
  uint32_t phase = 0;
  __syncthreads();  // barrier and s_max initialised
  for (uint32_t base = 0; base < n_points; base += kChunkBeams) {
    const uint32_t count = min(kChunkBeams, n_points - base);
    if (threadIdx.x == 0) {
      // TMA bulk copy of the scan points into shared memory (UBLKCP), completion on the mbarrier.
      const uint32_t bytes = count * static_cast<uint32_t>(sizeof(double2));
      mbarrier_expect_tx(&s_bar, bytes);
      bulk_copy_g2s(s_pts, points + base, bytes, &s_bar);
    }
    mbarrier_wait(&s_bar, phase);
    phase ^= 1u;
    if (active) {
      acc = fast ? accumulate_chunk<true, kTiled>(field, s_pts, count, acc, t.c, t.s, t.x, t.y)
                 : accumulate_chunk<false, kTiled>(field, s_pts, count, acc, t.c, t.s, t.x, t.y);
    }
    if (base + kChunkBeams < n_points) __syncthreads();  // s_pts is about to be overwritten by the next chunk
  }
  if (active) {
    const double likelihood = field.exp_epilogue ? exp(acc) : acc;
    w = w * likelihood;  // actions/reweight.hpp:54-60
    weights[i] = w;
  }
  publish_weight_max(active ? weight_order_bits(w) : 0ull, &s_max, &s_arrived, kRwThreads / kWarp, scalars);
}

// ---- reweight, fixed-point cell lookup ----------------------------------------------------------------
// Same result as reweight_lfm_kernel, two thirds of the instructions per beam.  The reference rounds
// after every operation of   x = (px*c - py*s) + tx;  cell = floor(x * inv_resolution)   (4 mul, 4 add,
// 2 mul and 2 floor conversions per beam, all on the FP64 pipe).  The CELL is all that matters, so the
// kernel evaluates   g = fma(px, c*inv, fma(-py, s*inv, tx*inv + 1))   (2 fma per coordinate; the +1 is
// the border cell), which differs from the reference's value by d <= 11 * 2^13 * 2^-53 < 2^-36 cells
// while every term stays below 2^13 cells, and adds 1.5*2^20 (y): in the sum's bit pattern the low word is
// the fraction of g in units of 2^-32 (round to nearest) and the low 20 bits of the high word are
// 2^19 + floor(g).  If the fraction word is not zero, g is at least 2^-33 > d away from an integer and
// floor(reference value) = floor(g) exactly.  x adds 1.5*2^18 instead, so its high word carries
// floor(4g) -- x already shifted into the place the 4x4-tile index wants it -- and a non-zero fraction
// word puts g at least 2^-35 > d from an integer.  A thread that ever sees a zero fraction word (2^-32 per
// coordinate, about once every two steps among a million particles) or a particle out of the 2^13 range
// redoes its beams with the reference's own operation sequence; nothing else in the loop branches.
// Out-of-grid end points clamp (one DPX add-min per coordinate, which also strips the bias) to the
// one-cell border holding the unknown-space value, so the load is unconditional.  A warp whose particles'
// scans all stay on the bordered map skips the clamp and indexes with the biased words (fixed_lookup_in_map).

constexpr double kFixedMagicX = 393216.0;   // 1.5 * 2^18: ulp 2^-34; high word = kFixedBiasX + floor(4 g)    for |g| < 2^17
constexpr double kFixedMagicY = 1572864.0;  // 1.5 * 2^20: ulp 2^-32; high word = kFixedBiasY + floor(g)      for |g| < 2^19
// The magic constants ride in the FMAs' addend (per-particle offsets ox, oy below), which saves the two additions per beam
// but lets THREE roundings at the magic's ulp into the word instead of one (the offset sum and both FMAs): the computed
// fixed-point value is within 3 half-ulps + 2^-36 cells of the reference's.  Two ulps of guard are added to the offset so
// that the reference's value lies in (computed - 4.07 ulp, computed + 0.07 ulp): the high word is the reference's cell
// whenever the fraction word is at least 5.  tests/test_fixed_point_lookup_model.py replays this with exact rationals,
// including end points a hair (2^-36 .. 2^-30 cells) either side of a cell edge at arbitrary headings.
constexpr double kFixedGuardX = 1.16415321826934814453125e-10; // 2^-33 = 2 ulp of kFixedMagicX
constexpr double kFixedGuardY = 4.656612873077392578125e-10;   // 2^-31 = 2 ulp of kFixedMagicY
constexpr uint32_t kFixedAmbiguous = 4u;  // fraction words 0..4: the cell is not decided (5 * 2^-32 per coordinate)

struct FixedParticle {
  double cx, sx;         // cos, sin of the field-frame heading, times 1/resolution
  double ox, oy;         // field-frame position in cells, plus the border cell, plus magic constant and guard
  uint32_t x_max, y_max; // 4 (width + 1) + 3, height + 1: largest 4 * padded x (+ 2 fraction bits) and padded y
  uint32_t row_pitch;    // 4 * 2^kx: elements per row of cells (four rows of tiles' worth per tile row)
  bool in_map;           // every end point of the scan lands in the bordered map: fixed_lookup_in_map applies
};

/// `margin` collects the smallest fraction word seen (<= kFixedAmbiguous: a coordinate too close to a cell edge to call).
/// x arrives as 4 * padded x with two fraction bits below it, y as padded y: the element index
///   (y >> 2) * 16 * tiles_per_row  +  (x >> 2) * 16 + (x & 3) * 4 + (y & 3)
/// is then one bit-select (y's low two bits replace x's fraction bits), one mask and one multiply-add.
__device__ __forceinline__ double fixed_lookup(const double* __restrict__ bordered, const FixedParticle& q, double px, double py, uint32_t& margin) {
  const double gx = fma(px, q.cx, fma(-py, q.sx, q.ox));  // gx + 1 + magic + guard
  const double gy = fma(px, q.sx, fma(py, q.cx, q.oy));   // gy + 1 + magic + guard
  margin = __vimin3_u32(margin, static_cast<uint32_t>(__double2loint(gx)), static_cast<uint32_t>(__double2loint(gy)));
  // min(word - bias, max): a negative coordinate wraps to a huge unsigned and clamps to the far border,
  // which holds the same unknown-space value as the near one.
  const uint32_t ux = __viaddmin_u32(static_cast<uint32_t>(__double2hiint(gx)), 0u - kFixedBiasX, q.x_max);  // 4 * padded x + 2 fraction bits
  const uint32_t uy = __viaddmin_u32(static_cast<uint32_t>(__double2hiint(gy)), 0u - kFixedBiasY, q.y_max);  // padded y
  uint32_t low;  // (ux & ~3) | (uy & 3) as ONE bit-select (the compiler splits it into two operations)
  asm("lop3.b32 %0, %1, 3, %2, 0xB8;" : "=r"(low) : "r"(ux), "r"(uy));
  const uint32_t idx = (uy & ~3u) * q.row_pitch + low;
  return __ldg(bordered + idx);
}

/// fixed_lookup for a particle whose end points all land in the bordered map (q.in_map): no clamp, and no bias stripped.
/// The biases' low 19 bits are clear, so the bit-select and the mask act on the cell bits as before, and the index is the
/// bordered index plus fixed_index_bias(kx) (mod 2^32), which `biased` (FieldView::bordered_biased) takes back off.
__device__ __forceinline__ double fixed_lookup_in_map(const double* __restrict__ biased, const FixedParticle& q, double px, double py,
                                                      uint32_t& margin) {
  const double gx = fma(px, q.cx, fma(-py, q.sx, q.ox));
  const double gy = fma(px, q.sx, fma(py, q.cx, q.oy));
  margin = __vimin3_u32(margin, static_cast<uint32_t>(__double2loint(gx)), static_cast<uint32_t>(__double2loint(gy)));
  const uint32_t hx = static_cast<uint32_t>(__double2hiint(gx)), hy = static_cast<uint32_t>(__double2hiint(gy));
  uint32_t low;
  asm("lop3.b32 %0, %1, 3, %2, 0xB8;" : "=r"(low) : "r"(hx), "r"(hy));
  const uint32_t idx = (hy & ~3u) * q.row_pitch + low;
  return __ldg(biased + idx);
}

/// The reference's operation sequence (field_lookup) against the bordered layout.
__device__ __forceinline__ double bordered_lookup_exact(const FieldView& f, double px, double py, double c, double s, double tx, double ty) {
  const double x = (px * c - py * s) + tx;
  const double y = (px * s + py * c) + ty;
  const double fx = floor(x * f.inv_resolution), fy = floor(y * f.inv_resolution);
  // saturating: anything outside [-1, side] (NaN included) lands on the border
  const int xi = (fx >= 0.0 && fx < static_cast<double>(f.width)) ? static_cast<int>(fx) : -1;
  const int yi = (fy >= 0.0 && fy < static_cast<double>(f.height)) ? static_cast<int>(fy) : -1;
  return __ldg(f.bordered + bordered_index(static_cast<uint32_t>(xi + 1), static_cast<uint32_t>(yi + 1), f.border_kx));
}

/// transform = world_to_likelihood_field * state (likelihood_field_model.hpp:70-74); idle threads use the identity.
__device__ __forceinline__ Pose2 field_frame_pose(const FieldView& f, const Pose2* __restrict__ states, uint64_t i, bool active) {
  return pose_mul(f.world_to_field, active ? load_pose(states + i) : Pose2{1.0, 0.0, 0.0, 0.0});
}

/// Scan points as a kernel parameter: they sit in the constant bank and reach the FP64 instructions
/// through uniform registers -- no shared-memory load per beam and no L1 data-pipe traffic.  30 KB of
/// the 32 KB parameter space; longer scans take the shared-memory (TMA) variant.
constexpr uint32_t kParamBeams = 1920;
struct ScanParam {
  double2 p[kParamBeams];
};

// One group of four beams of the pipeline below: look up beams B..B+3, then add the previous group to acc.
#define BB200_FIXED_STEP(POINT, B, LOOKUP, TABLE)                                                             \
  {                                                                                                           \
    const double2 p0 = POINT(B), p1 = POINT((B) + 1), p2 = POINT((B) + 2), p3 = POINT((B) + 3);               \
    const double g0 = LOOKUP(TABLE, q, p0.x, p0.y, margin);                                                   \
    const double g1 = LOOKUP(TABLE, q, p1.x, p1.y, margin);                                                   \
    const double g2 = LOOKUP(TABLE, q, p2.x, p2.y, margin);                                                   \
    const double g3 = LOOKUP(TABLE, q, p3.x, p3.y, margin);                                                   \
    acc = acc + ((f0 + f1) + (f2 + f3));                                                                      \
    f0 = g0, f1 = g1, f2 = g2, f3 = g3;                                                                       \
  }
// libstdc++ transform_reduce (numeric:439-462): groups of four, init += ((f0+f1)+(f2+f3)), then one by one.
#define BB200_FIXED_PIPELINE(POINT, COUNT, LOOKUP, TABLE)                                                     \
  if (4 <= (COUNT)) {                                                                                         \
    /* Software pipeline: the loads of the next four beams are issued before the previous four are summed */  \
    /* (a warp issues in order: summing first would leave it with four loads in flight, then none).       */  \
    double f0, f1, f2, f3;                                                                                    \
    {                                                                                                         \
      const double2 p0 = POINT(0), p1 = POINT(1), p2 = POINT(2), p3 = POINT(3);                               \
      f0 = LOOKUP(TABLE, q, p0.x, p0.y, margin);                                                              \
      f1 = LOOKUP(TABLE, q, p1.x, p1.y, margin);                                                              \
      f2 = LOOKUP(TABLE, q, p2.x, p2.y, margin);                                                              \
      f3 = LOOKUP(TABLE, q, p3.x, p3.y, margin);                                                              \
    }                                                                                                         \
    b = 4;                                                                                                    \
    /* kRwUnroll groups per trip and a single exit test: the loop bookkeeping is one compare and branch per trip */\
    for (; b + 4 * kRwUnroll <= (COUNT); b += 4 * kRwUnroll) {                                                \
      _Pragma("unroll") for (uint32_t u = 0; u < 4 * kRwUnroll; u += 4) BB200_FIXED_STEP(POINT, uint64_t{b} + u, LOOKUP, TABLE)\
    }                                                                                                         \
    _Pragma("unroll 1") for (; b + 4 <= (COUNT); b += 4) BB200_FIXED_STEP(POINT, b, LOOKUP, TABLE)            \
    acc = acc + ((f0 + f1) + (f2 + f3));                                                                      \
  }                                                                                                           \
  for (; b < (COUNT); ++b) {                                                                                  \
    const double2 p0 = POINT(b);                                                                              \
    acc = acc + LOOKUP(TABLE, q, p0.x, p0.y, margin);                                                         \
  }
#define BB200_FIXED_SUM(POINT, COUNT)                                                                         \
  do {                                                                                                        \
    const double acc_before = acc;                                                                            \
    uint32_t margin = margin_start;                                                                           \
    uint32_t b = 0;                                                                                           \
    /* One loop per warp: a divergent beam loop loses the uniform datapath for the scan points (take_chunk_ticket). */\
    if (__all_sync(0xffffffffu, q.in_map)) {                                                                  \
      BB200_FIXED_PIPELINE(POINT, COUNT, fixed_lookup_in_map, field.bordered_biased);                         \
    } else {                                                                                                  \
      BB200_FIXED_PIPELINE(POINT, COUNT, fixed_lookup, field.bordered);                                       \
    }                                                                                                         \
    if (margin <= kFixedAmbiguous) { /* a coordinate within ~2^-30 cells of a cell edge, or a particle out of range */\
      const Pose2 te = field_frame_pose(field, states, i, active);                                            \
      acc = acc_before;                                                                                       \
      b = 0;                                                                                                  \
      for (; b + 4 <= (COUNT); b += 4) {                                                                      \
        const double2 p0 = POINT(b), p1 = POINT(b + 1), p2 = POINT(b + 2), p3 = POINT(b + 3);                 \
        const double f0 = bordered_lookup_exact(field, p0.x, p0.y, te.c, te.s, te.x, te.y);                   \
        const double f1 = bordered_lookup_exact(field, p1.x, p1.y, te.c, te.s, te.x, te.y);                   \
        const double f2 = bordered_lookup_exact(field, p2.x, p2.y, te.c, te.s, te.x, te.y);                   \
        const double f3 = bordered_lookup_exact(field, p3.x, p3.y, te.c, te.s, te.x, te.y);                   \
        acc = acc + ((f0 + f1) + (f2 + f3));                                                                  \
      }                                                                                                       \
      for (; b < (COUNT); ++b) {                                                                              \
        const double2 p0 = POINT(b);                                                                          \
        acc = acc + bordered_lookup_exact(field, p0.x, p0.y, te.c, te.s, te.x, te.y);                         \
      }                                                                                                       \
    }                                                                                                         \
  } while (0)

/// Per-particle constants of the fixed-point evaluation.
__device__ __forceinline__ void fixed_particle_setup(const FieldView& field, const Pose2* __restrict__ states, uint64_t i, bool active,
                                                     double points_radius, FixedParticle& q, uint32_t& margin_start) {
  const Pose2 t = field_frame_pose(field, states, i, active);
  const double inv = field.inv_resolution;
  // The error bound above needs every term of g below 2^13 cells.
  const double reach = (points_radius + fmax(fabs(t.x), fabs(t.y))) * inv + 2.0;
  margin_start = reach < 8100.0 ? 0xFFFFFFFFu : 0u;  // 0 also for NaN: straight to the exact sequence
  q.cx = t.c * inv, q.sx = t.s * inv;
  q.ox = (t.x * inv + 1.0) + (kFixedMagicX + kFixedGuardX);
  q.oy = (t.y * inv + 1.0) + (kFixedMagicY + kFixedGuardY);
  q.x_max = field.border_x_max;
  q.y_max = field.border_y_max;
  q.row_pitch = 4u * field.border_pitch;
  // In-map test in padded cells: |px*c - py*s| <= (|px| + |py|) max(|c|, |s|) <= points_radius max(|c|, |s|), and the
  // fixed-point sums are within 2^-30 cells of that, so half a cell of margin keeps every floor in 0 .. side + 1.
  // False for NaN and for maps whose biased indices would wrap.
  const double r = points_radius * fmax(fabs(q.cx), fabs(q.sx)) + 0.5;
  const double gx = t.x * inv + 1.0, gy = t.y * inv + 1.0;
  q.in_map = field.bordered_biased != nullptr && gx - r >= 0.0 && gx + r <= static_cast<double>(field.width + 2) && gy - r >= 0.0 &&
             gy + r <= static_cast<double>(field.height + 2);
}

#if BB200_RW_CHUNK > 0
/// Next task of the CTA's current chunk (see the experiment note in reweight_lfm_fixed_param_kernel).  Every branch is on a
/// value broadcast from lane 0, so that the warp provably stays converged: a spin loop inside `if (lane == 0)` makes ptxas
/// give up the uniform datapath (LDCU) for the scan points in the beam loop that follows (LDC through the ADU pipe instead,
/// which alone costs 20 %).
__device__ __forceinline__ unsigned long long take_chunk_ticket(unsigned long long* s_chunk, unsigned long long* ticket_counter, int lane) {
  for (;;) {
    unsigned long long old = 0;
    if (lane == 0) old = atomicAdd(s_chunk, 1ull);
    old = __shfl_sync(0xffffffffu, old, 0);
    const unsigned long long idx = old & 0xFFull, chunk = old >> 8;
    if (idx < BB200_RW_CHUNK) return chunk * BB200_RW_CHUNK + idx;
    if (idx == BB200_RW_CHUNK) {  // this warp refills: the new chunk's task 0 is its own
      unsigned long long fresh = 0;
      if (lane == 0) fresh = atomicAdd(ticket_counter, 1ull);
      fresh = __shfl_sync(0xffffffffu, fresh, 0);
      if (lane == 0) atomicExch(s_chunk, (fresh << 8) | 1ull);
      return fresh * BB200_RW_CHUNK;
    }
    for (;;) {  // another warp is fetching the next chunk
      unsigned long long cur = 0;
      if (lane == 0) cur = *reinterpret_cast<volatile unsigned long long*>(s_chunk);
      cur = __shfl_sync(0xffffffffu, cur, 0);
      if ((cur >> 8) != chunk) break;
    }
  }
}
#endif

/// Scan in the constant bank: nothing is shared between the warps of a CTA, so the grid is persistent
/// (CTAs/SM x SM count) and every WARP draws the next 32 particles of the schedule from a global
/// ticket counter.  A CTA-per-256-particles grid loses 10-13 % to its slowest warp (each CTA holds its
/// SM slot until the last of its warps is through 1080 beams) and to the partial last wave.
__global__ void __launch_bounds__(kRwThreads, kRwBlocksPerSm)
    reweight_lfm_fixed_param_kernel(const Pose2* __restrict__ states, double* __restrict__ weights, uint64_t n, const uint32_t* __restrict__ perm,
                                    FieldView field, uint32_t n_points, double points_radius, Scalars* __restrict__ scalars,
                                    const __grid_constant__ ScanParam scan) {
  const int lane = threadIdx.x % kWarp;
  const unsigned long long n_tasks = (n + kWarp - 1) / kWarp;  // a task = the next 32 particles of the schedule
  unsigned long long* ticket_counter = &scalars->work_ticket;
#if BB200_RW_CHUNK > 0
  // Experiment (profiles/r02_lfm_chunk_tickets.txt): the CTA draws CHUNKS of BB200_RW_CHUNK adjacent tasks from the global
  // counter and its warps take tasks from the current chunk through a shared-memory word (chunk id << 8 | next index), so that
  // the warps of a CTA work on neighbouring particles without waiting for each other; the warp that finds the chunk
  // exhausted fetches the next one, the others spin on the word for that round trip.
  __shared__ unsigned long long s_chunk;
  if (threadIdx.x == 0) s_chunk = atomicAdd(ticket_counter, 1ull) << 8;
  __syncthreads();
  unsigned long long ticket = take_chunk_ticket(&s_chunk, ticket_counter, lane);
#else
  unsigned long long ticket = __shfl_sync(0xffffffffu, lane == 0 ? atomicAdd(ticket_counter, 1ull) : 0ull, 0);
#endif
  unsigned long long best = 0ull;
  while (ticket < n_tasks) {
#if BB200_RW_CHUNK == 0
    // Draw the next ticket now; its round trip to L2 hides behind this task's beams.
    const unsigned long long next = lane == 0 ? atomicAdd(ticket_counter, 1ull) : 0ull;
#endif
    const uint64_t slot = ticket * kWarp + lane;
    const bool active = slot < n;  // idle lanes of the last task walk the beams with a dummy pose
    const uint64_t i = active ? (perm != nullptr ? perm[slot] : slot) : 0;
    uint32_t margin_start;
    FixedParticle q;
    fixed_particle_setup(field, states, i, active, points_radius, q, margin_start);
    double acc = field.init;
#define BB200_POINT(k) scan.p[(k)]
    BB200_FIXED_SUM(BB200_POINT, n_points);
#undef BB200_POINT
    if (active) {
      const double likelihood = field.exp_epilogue ? exp(acc) : acc;
      const double w = weights[i] * likelihood;  // actions/reweight.hpp:54-60
      weights[i] = w;
      const unsigned long long bits = weight_order_bits(w);
      best = bits > best ? bits : best;
    }
#if BB200_RW_CHUNK > 0
    ticket = take_chunk_ticket(&s_chunk, ticket_counter, lane);
#else
    ticket = __shfl_sync(0xffffffffu, next, 0);
#endif
  }
#pragma unroll
  for (int off = kWarp / 2; off > 0; off >>= 1) {
    const unsigned long long o = __shfl_down_sync(0xffffffffu, best, off);
    best = o > best ? o : best;
  }
  if (lane == 0) {
    if (best != 0ull) atomicMax(&scalars->wmax_bits, best);
    // The last warp out rewinds the ticket counter for the next launch.
    const unsigned long long warps = static_cast<unsigned long long>(gridDim.x) * (kRwThreads / kWarp);
    if (atomicAdd(&scalars->work_done, 1ull) + 1ull == warps) {
      scalars->work_done = 0ull;
      *ticket_counter = 0ull;
    }
  }
}

/// Scan staged in shared memory by TMA (scans longer than kParamBeams points): one CTA per kRwThreads particles.
__global__ void __launch_bounds__(kRwThreads, kRwBlocksPerSm)
    reweight_lfm_fixed_kernel(const Pose2* __restrict__ states, double* __restrict__ weights, uint64_t n, const uint32_t* __restrict__ perm,
                              FieldView field, const double2* __restrict__ points, uint32_t n_points, double points_radius,
                              Scalars* __restrict__ scalars) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* s_pts = reinterpret_cast<double2*>(smem_raw);
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ unsigned long long s_max;
  __shared__ unsigned int s_arrived;

  const uint64_t slot = static_cast<uint64_t>(blockIdx.x) * kRwThreads + threadIdx.x;
  const bool active = slot < n;
  const uint64_t i = active ? (perm != nullptr ? perm[slot] : slot) : 0;
  if (threadIdx.x == 0) {
    s_max = 0ull;
    s_arrived = 0u;
    mbarrier_init(&s_bar, 1);
    mbarrier_init_fence();
  }
  uint32_t margin_start;
  FixedParticle q;
  fixed_particle_setup(field, states, i, active, points_radius, q, margin_start);

  double acc = field.init;
  __syncthreads();  // s_max and the barrier initialised
  uint32_t phase = 0;
  for (uint32_t base = 0; base < n_points; base += kChunkBeams) {
    const uint32_t count = min(kChunkBeams, n_points - base);
    if (threadIdx.x == 0) {
      const uint32_t bytes = count * static_cast<uint32_t>(sizeof(double2));
      mbarrier_expect_tx(&s_bar, bytes);
      bulk_copy_g2s(s_pts, points + base, bytes, &s_bar);
    }
    mbarrier_wait(&s_bar, phase);
    phase ^= 1u;
#define BB200_POINT(k) s_pts[(k)]
    BB200_FIXED_SUM(BB200_POINT, count);
#undef BB200_POINT
    if (base + kChunkBeams < n_points) __syncthreads();
  }
  double w = 0.0;
  if (active) {
    const double likelihood = field.exp_epilogue ? exp(acc) : acc;
    w = weights[i] * likelihood;  // actions/reweight.hpp:54-60
    weights[i] = w;
  }
  publish_weight_max(active ? weight_order_bits(w) : 0ull, &s_max, &s_arrived, kRwThreads / kWarp, scalars);
}
#undef BB200_FIXED_SUM
#undef BB200_FIXED_PIPELINE
#undef BB200_FIXED_STEP

// ---- reweight (beam model; a4 + a5) -----------------------------------------------------------
// BeamSensorModel (sensor/beam_model.hpp:104-150): one thread per particle, beams in the inner
// loop, so the lanes of a warp (neighbouring particles, same beam) walk rays of similar length.
// Ray casting is Ray2d::cast (algorithm/raycasting.hpp:79-107) over the standard Bresenham2i
// iterator (algorithm/raycasting/bresenham.hpp:84-160) on the int8 occupancy grid.

struct BeamRay {
  double far_x, far_y;  // bearing.unit_complex() * max_range  (raycasting.hpp:83)
  double z;             // measured range (beam_model.hpp:116)
  double short_decay;   // exp(-lambda_short * z) of the short-reading term (:137-141)
};

/// regular_grid.hpp:75-78.  Clamped to +-2^28 cells so that spans of far-away end points cannot
/// overflow 32-bit integers (the reference's cast<int>() is undefined out there).
__device__ __forceinline__ int cell_near(double p, double inv_resolution) {
  return max(-(1 << 28), min(1 << 28, __double2int_rd(p * inv_resolution)));
}

/// One ray of Ray2d::cast (raycasting.hpp:79-107) over the standard Bresenham2i iterator (bresenham.hpp:84-160) as a
/// state machine, so that a thread can keep several rays in flight (ray_step is one dependent load of the
/// free-distance map plus a closed-form advance of the iterator; the walk is bound by that load's latency).
struct RayWalk {
  int x, y;            // iterator position: x along the longer axis (swapped when `reversed`)
  int xstep, ystep;
  int xspan, dxspan, dyspan;
  int error, step;
  uint32_t recip;      // floor((2^32 - 1) / dxspan): quotients below 2^8 come out exact or one low
  bool reversed, small_span, active;
  int hit_x, hit_y;    // cell of the first non-free cell (valid when hit)
  bool hit;
};

__device__ __forceinline__ void ray_begin(RayWalk& w, int sx, int sy, int fx, int fy) {
  int xspan = fx - sx, xstep = 1;
  if (xspan < 0) {
    xspan = -xspan;
    xstep = -1;
  }
  int yspan = fy - sy, ystep = 1;
  if (yspan < 0) {
    yspan = -yspan;
    ystep = -1;
  }
  w.x = sx, w.y = sy;
  w.reversed = false;
  if (xspan < yspan) {  // iterate along the longer axis (bresenham.hpp:99-105)
    int t = w.x; w.x = w.y; w.y = t;
    t = xspan; xspan = yspan; yspan = t;
    t = xstep; xstep = ystep; ystep = t;
    w.reversed = true;
  }
  w.xstep = xstep, w.ystep = ystep;
  w.xspan = xspan, w.dxspan = 2 * xspan, w.dyspan = 2 * yspan;
  w.small_span = xspan < (1 << 22);  // then error + 255 * dyspan stays below 2^32
  w.recip = xspan > 0 ? 0xFFFFFFFFu / static_cast<uint32_t>(w.dxspan) : 0u;
  w.error = xspan;
  w.step = 0;
  w.active = true;
  w.hit = false;
  w.hit_x = w.hit_y = 0;
}

/// One iteration: inspect the current cell, then jump as far as the free-distance map allows.
__device__ __forceinline__ void ray_step(RayWalk& w, const OccupancyView& g) {
  const int cx = w.reversed ? w.y : w.x, cy = w.reversed ? w.x : w.y;
  if (!(static_cast<unsigned>(cx) < static_cast<unsigned>(g.width) && static_cast<unsigned>(cy) < static_cast<unsigned>(g.height))) {
    w.active = false;  // take_while(cell_is_valid), raycasting.hpp:86-87: a miss
    return;
  }
  const int d = __ldg(g.free_distance + (static_cast<size_t>(cy) * static_cast<size_t>(g.width) + static_cast<size_t>(cx)));
  if (d == 0) {  // !free_at: first non-free cell on the line
    w.hit = true;
    w.hit_x = cx, w.hit_y = cy;
    w.active = false;
    return;
  }
  // Every cell within Chebyshev distance d - 1 is free and the line moves at most one cell per step in each axis,
  // so the next d - 1 cells cannot stop the ray: advance d steps of the iterator (bresenham.hpp:122-160, standard
  // variant) in closed form.  error stays in (0, dxspan].
  const int k = min(d, w.xspan - w.step);
  if (k == 0) {  // the far end cell was free too: sentinel reached (bresenham.hpp:179)
    w.active = false;
    return;
  }
  w.step += k;
  w.x += k * w.xstep;
  int m;  // floor((t - 1) / dxspan) with t = error + k * dyspan
  if (w.small_span) {
    // 32-bit: t - 1 < 2^32 and the quotient is at most k <= 255, so the high word of (t - 1) * floor((2^32 - 1) / dxspan)
    // is the quotient or one below it; one remainder check makes it exact.  (A 64-bit division costs more than the
    // rest of the loop; an FP64 reciprocal needs two conversions on the quarter-rate pipe.)
    const uint32_t tm1 = static_cast<uint32_t>(w.error) + static_cast<uint32_t>(k) * static_cast<uint32_t>(w.dyspan) - 1u;
    uint32_t q = __umulhi(tm1, w.recip);
    uint32_t r = tm1 - q * static_cast<uint32_t>(w.dxspan);
    if (r >= static_cast<uint32_t>(w.dxspan)) {
      ++q;
      r -= static_cast<uint32_t>(w.dxspan);
    }
    m = static_cast<int>(q);
    w.error = static_cast<int>(r) + 1;  // t - m * dxspan
  } else {
    const long long t = static_cast<long long>(w.error) + static_cast<long long>(k) * w.dyspan;
    m = static_cast<int>((t - 1) / w.dxspan);
    w.error = static_cast<int>(t - static_cast<long long>(m) * w.dxspan);
  }
  w.y += m * w.ystep;
}

/// Distance in metres from the source cell centroid to the ray's hit cell (clamped to max_range), or -1 on a miss;
/// d2 = squared cell distance of that cell (only meaningful on a hit).
__device__ __forceinline__ double ray_result(const RayWalk& w, const OccupancyView& g, int sx, int sy, double max_range, unsigned long long& d2) {
  if (!w.hit) return -1.0;
  const double dxm = (static_cast<double>(w.hit_x) + 0.5) * g.resolution - (static_cast<double>(sx) + 0.5) * g.resolution;
  const double dym = (static_cast<double>(w.hit_y) + 0.5) * g.resolution - (static_cast<double>(sy) + 0.5) * g.resolution;
  const long long ix = static_cast<long long>(w.hit_x) - sx, iy = static_cast<long long>(w.hit_y) - sy;
  d2 = static_cast<unsigned long long>(ix * ix + iy * iy);
  return fmin(sqrt(dxm * dxm + dym * dym), max_range);
}

/// beam_model.hpp:128-135: the two normalisers as functions of z_mean.
__device__ __forceinline__ double2 beam_normalisers(const BeamParams& p, double z_mean) {
  const double sqrt2 = sqrt(2.);
  const double eta_hit = 2. / (erf((p.beam_max_range - z_mean) / (sqrt2 * p.sigma_hit)) - erf(-z_mean / (sqrt2 * p.sigma_hit)));
  const double eta_short = 1. / (1. - exp(-p.lambda_short * z_mean));
  return make_double2(eta_hit, eta_short);
}

/// The four-term mixture cubed (beam_model.hpp:125-147); short_decay = exp(-lambda_short * z), a per-beam constant.
__device__ __forceinline__ double beam_pz3(const BeamParams& p, double z, double short_decay, double z_mean, double n, double eta_hit, double eta_short) {
  const double d = (z - z_mean) / p.sigma_hit;
  double pz = p.z_hit * eta_hit * n * exp(-(d * d) / 2.);
  if (z < z_mean) pz += p.z_short * p.lambda_short * eta_short * short_decay;
  if (z < p.beam_max_range) {
    pz += p.z_rand / p.beam_max_range;
  } else {
    pz += p.z_max;
  }
  return pz * pz * pz;
}

__global__ void __launch_bounds__(256) beam_eta_table_kernel(BeamParams p, double resolution, double2* __restrict__ table, uint32_t entries) {
  const uint32_t k = blockIdx.x * 256 + threadIdx.x;
  if (k >= entries) return;
  const double z_mean = k + 1 == entries ? p.beam_max_range : fmin(sqrt(static_cast<double>(k)) * resolution, p.beam_max_range);
  table[k] = beam_normalisers(p, z_mean);
}

#ifndef BB200_BEAM_BLOCKS
#define BB200_BEAM_BLOCKS 3
#endif
#ifndef BB200_BEAM_RAYS
#define BB200_BEAM_RAYS 1  // rays a thread walks together (1, 2 or 4); measured at C3: 1 -> 29.5 ms, 2 -> 31.4 ms, 4 (2 CTAs/SM) -> 40.0 ms
#endif
constexpr int kBeamRays = BB200_BEAM_RAYS;
constexpr int kBeamThreads = 256;
constexpr int kBeamBlocksPerSm = BB200_BEAM_BLOCKS;
constexpr uint32_t kBeamChunk = 1024;  // rays staged per shared-memory chunk (32 KB), multiple of 4

__global__ void __launch_bounds__(kBeamThreads, kBeamBlocksPerSm)
    reweight_beam_kernel(const Pose2* __restrict__ states, double* __restrict__ weights, uint64_t n, const uint32_t* __restrict__ perm,
                         OccupancyView grid, BeamParams params, const double2* __restrict__ points, uint32_t n_points,
                         Scalars* __restrict__ scalars) {
  __shared__ BeamRay s_rays[kBeamChunk];
  __shared__ unsigned long long s_red[kBeamThreads / kWarp];
  const uint64_t slot = static_cast<uint64_t>(blockIdx.x) * kBeamThreads + threadIdx.x;
  const bool active = slot < n;
  const uint64_t i = active ? (perm != nullptr ? perm[slot] : slot) : 0;

  Pose2 st{1.0, 0.0, 0.0, 0.0};
  double w = 0.0;
  if (active) {
    st = load_pose(states + i);
    w = weights[i];
  }
  // Ray2d: source pose in the grid frame and its cell (raycasting.hpp:67-70).
  const Pose2 src = pose_mul(grid.world_to_grid, st);
  const int sx = cell_near(src.x, grid.inv_resolution), sy = cell_near(src.y, grid.inv_resolution);
  const double n_norm = 1. / (sqrt(2. * 3.14159265358979323846) * params.sigma_hit);  // beam_model.hpp:107

  // The mixture value of one beam given its ray walk (beam_model.hpp:116-147).
  auto beam_value = [&](const BeamRay& ray, const RayWalk& walk) {
    unsigned long long d2 = 0;
    const double hit = ray_result(walk, grid, sx, sy, params.beam_max_range, d2);
    const double z_mean = hit >= 0.0 ? hit : params.beam_max_range;  // value_or(beam_max_range)
    double2 eta;
    if (params.eta != nullptr) {
      // hit within range: the entry of its cell distance; miss or clamped to the range: the last entry
      const bool in_table = hit >= 0.0 && hit < params.beam_max_range && d2 + 1 < params.eta_entries;
      eta = __ldg(params.eta + (in_table ? static_cast<uint32_t>(d2) : params.eta_entries - 1u));
    } else {
      eta = beam_normalisers(params, z_mean);
    }
    return beam_pz3(params, ray.z, ray.short_decay, z_mean, n_norm, eta.x, eta.y);
  };
  auto begin_walk = [&](RayWalk& walk, const BeamRay& ray) {
    // far end = r1 * t2 + t1 (raycasting.hpp:81-85)
    const double ex = (src.c * ray.far_x - src.s * ray.far_y) + src.x;
    const double ey = (src.s * ray.far_x + src.c * ray.far_y) + src.y;
    ray_begin(walk, sx, sy, cell_near(ex, grid.inv_resolution), cell_near(ey, grid.inv_resolution));
  };

  double acc = 0.0;
  for (uint32_t base = 0; base < n_points; base += kBeamChunk) {
    const uint32_t count = min(kBeamChunk, n_points - base);
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < count; b += kBeamThreads) {
      const double2 p = points[base + b];
      const double z = sqrt(p.x * p.x + p.y * p.y);                      // beam_model.hpp:116
      const double bx = p.x / z, by = p.y / z;                            // :120-123
      s_rays[b] = BeamRay{bx * params.beam_max_range, by * params.beam_max_range, z, exp(-params.lambda_short * z)};
    }
    __syncthreads();
    if (active) {
      uint32_t b = 0;
      for (; b + 4 <= count; b += 4) {  // transform_reduce grouping (numeric:439-462)
        // The four rays of a group are walked together: their free-distance loads are independent, so the thread
        // keeps kBeamRays of them in flight instead of waiting out one dependent chain after the other.
        double f[4];
#pragma unroll
        for (int g0 = 0; g0 < 4; g0 += kBeamRays) {
          RayWalk walk[kBeamRays];
#pragma unroll
          for (int r = 0; r < kBeamRays; ++r) begin_walk(walk[r], s_rays[b + g0 + r]);
          bool any = true;
          while (any) {
            any = false;
#pragma unroll
            for (int r = 0; r < kBeamRays; ++r) {
              if (walk[r].active) ray_step(walk[r], grid);
              any |= walk[r].active;
            }
          }
#pragma unroll
          for (int r = 0; r < kBeamRays; ++r) f[g0 + r] = beam_value(s_rays[b + g0 + r], walk[r]);
        }
        acc = acc + ((f[0] + f[1]) + (f[2] + f[3]));
      }
      for (; b < count; ++b) {
        RayWalk walk;
        begin_walk(walk, s_rays[b]);
        while (walk.active) ray_step(walk, grid);
        acc = acc + beam_value(s_rays[b], walk);
      }
    }
  }
  if (active) {
    w = w * acc;
    weights[i] = w;
  }
  const unsigned long long m = block_max_u64<kBeamThreads>(active ? weight_order_bits(w) : 0ull, s_red);
  if (threadIdx.x == 0 && m != 0) atomicMax(&scalars->wmax_bits, m);
}

// ---- beam model in two passes ----------------------------------------------------------------------
// The fused kernel above carries the ray walk (integer, one dependent load per iteration) and the mixture (FP64:
// sqrt, exp, three dozen constants) in one register allocation: 78 registers, 36 % occupancy, 800 issued instructions
// per beam.  Split: the WALK writes the hit cell of every (particle, beam) as one 32-bit word -- beam-major, so a
// warp's 32 particles store and later load consecutive words -- and the MIXTURE reads it back.  4 bytes per ray each
// way (2.9 GB at 1M x 720: under a millisecond of HBM time) buy a 40-register walk kernel at twice the occupancy
// and a branch-free mixture loop.  Hit words: 0xFFFFFFFF = miss, else cy << 16 | cx (grids up to 65535 cells a side).

constexpr uint32_t kHitMiss = 0xFFFFFFFFu;
#ifndef BB200_WALK_BLOCKS
#define BB200_WALK_BLOCKS 8  // resident CTAs per SM the walk is compiled for (register cap; the loop is latency-bound, so warps beat
                            // registers even with a few spills); measured at C3: 4 -> 17.8 ms, 5 -> 16.7, 6 -> 16.1, 7 -> 15.6, 8 -> 15.5
#endif
constexpr int kWalkThreads = 256;
constexpr uint32_t kWalkChunk = 1024;  // far ends staged per shared-memory chunk (16 KB)

/// The walk against the PADDED free-distance map (one border cell of zeros all round, 2^pad_shift bytes per row): a
/// jump of k <= d cells can at most land on the border, so the loop needs no bounds test -- a zero either is the first
/// non-free cell or the border (= the ray left the grid: a miss, raycasting.hpp:86-87), told apart after the loop.  The
/// iterator state is the linear cell index, advanced by k * (major stride) + m * (minor stride), so the x/y swap of the
/// steep case (bresenham.hpp:99-105) costs nothing per iteration.  Spans stay below 2^22 (checked by the launcher), so
/// the 32-bit reciprocal quotient of ray_step is the only path.  16 instructions per iteration instead of 45.
/// (Walking 2 or 4 rays per thread together was measured on this kernel as well: 21.9 / 25.6 ms against 18.5 ms at C3 --
/// the per-ray state machine and its activity flags cost more than the second load chain hides.)
__global__ void __launch_bounds__(kWalkThreads, BB200_WALK_BLOCKS)
    beam_walk_kernel(const Pose2* __restrict__ states, uint64_t n, uint64_t slot_base, uint64_t slot_count, const uint32_t* __restrict__ perm,
                     OccupancyView grid, double beam_max_range, const double2* __restrict__ points, uint32_t n_points,
                     uint32_t* __restrict__ hits, uint64_t hit_stride) {
  __shared__ double2 s_far[kWalkChunk];
  const uint64_t local = static_cast<uint64_t>(blockIdx.x) * kWalkThreads + threadIdx.x;
  const uint64_t slot = slot_base + local;
  const bool active = local < slot_count && slot < n;
  const uint64_t i = active ? (perm != nullptr ? perm[slot] : slot) : 0;
  // Ray2d: source pose in the grid frame and its cell (raycasting.hpp:67-70).
  const Pose2 src = pose_mul(grid.world_to_grid, active ? load_pose(states + i) : Pose2{1.0, 0.0, 0.0, 0.0});
  const int sx = cell_near(src.x, grid.inv_resolution), sy = cell_near(src.y, grid.inv_resolution);
  const bool source_inside = static_cast<unsigned>(sx) < static_cast<unsigned>(grid.width) && static_cast<unsigned>(sy) < static_cast<unsigned>(grid.height);
  const int shift = grid.pad_shift;
  const int pitch = 1 << shift;
  const uint8_t* __restrict__ map = grid.free_padded;
  const int source_index = ((sy + 1) << shift) + (sx + 1);
  for (uint32_t base = 0; base < n_points; base += kWalkChunk) {
    const uint32_t count = min(kWalkChunk, n_points - base);
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < count; b += kWalkThreads) {
      const double2 p = points[base + b];
      const double z = sqrt(p.x * p.x + p.y * p.y);                                    // beam_model.hpp:116
      s_far[b] = make_double2((p.x / z) * beam_max_range, (p.y / z) * beam_max_range);  // :120-123, raycasting.hpp:83
    }
    __syncthreads();
    if (!active) continue;
    for (uint32_t b = 0; b < count; ++b) {
      uint32_t word = kHitMiss;
      if (source_inside) {  // a source outside the grid sees nothing: the first cell already fails cell_is_valid
        // far end = r1 * t2 + t1 (raycasting.hpp:81-85)
        const double2 f = s_far[b];
        const double ex = (src.c * f.x - src.s * f.y) + src.x;
        const double ey = (src.s * f.x + src.c * f.y) + src.y;
        int span = cell_near(ex, grid.inv_resolution) - sx, minor = cell_near(ey, grid.inv_resolution) - sy;
        int stride_major = 1, stride_minor = pitch;
        if (span < 0) {
          span = -span;
          stride_major = -1;
        }
        if (minor < 0) {
          minor = -minor;
          stride_minor = -pitch;
        }
        if (span < minor) {  // iterate along the longer axis (bresenham.hpp:99-105)
          int t = span; span = minor; minor = t;
          t = stride_major; stride_major = stride_minor; stride_minor = t;
        }
        const uint32_t dxspan = 2u * static_cast<uint32_t>(span), dyspan = 2u * static_cast<uint32_t>(minor);
        const uint32_t recip = span > 0 ? 0xFFFFFFFFu / dxspan : 0u;
        int index = source_index;
        uint32_t err1 = static_cast<uint32_t>(span) - 1u;  // error - 1, error in (0, dxspan] (span == 0: never used)
        int remaining = span;
        for (;;) {
          const int d = __ldg(map + index);
          if (d == 0) {  // first non-free cell on the line, or the border
            const int cx = (index & (pitch - 1)) - 1, cy = (index >> shift) - 1;
            if (static_cast<unsigned>(cx) < static_cast<unsigned>(grid.width) && static_cast<unsigned>(cy) < static_cast<unsigned>(grid.height))
              word = (static_cast<uint32_t>(cy) << 16) | static_cast<uint32_t>(cx);
            break;
          }
          // Every cell within Chebyshev distance d - 1 is free and the line moves at most one cell per step in each axis:
          // advance d steps of the iterator (bresenham.hpp:122-160, standard variant) in closed form.
          const int k = min(d, remaining);
          if (k == 0) break;  // the far end cell was free too: sentinel reached (bresenham.hpp:179)
          remaining -= k;
          const uint32_t tm1 = err1 + static_cast<uint32_t>(k) * dyspan;  // t - 1, t = error + k * dyspan < 2^32
          uint32_t q = __umulhi(tm1, recip);                              // floor((t - 1) / dxspan) or one below
          uint32_t r = tm1 - q * dxspan;
          if (r >= dxspan) {
            ++q;
            r -= dxspan;
          }
          err1 = r;  // new error - 1
          index += k * stride_major + static_cast<int>(q) * stride_minor;
        }
      }
      __stcs(hits + static_cast<uint64_t>(base + b) * hit_stride + local, word);  // written once, read once: streaming
    }
  }
}

constexpr int kMixThreads = 256;
constexpr uint32_t kMixChunk = 2048;

__global__ void __launch_bounds__(kMixThreads)
    beam_mixture_kernel(const Pose2* __restrict__ states, double* __restrict__ weights, uint64_t n, uint64_t slot_base, uint64_t slot_count,
                        const uint32_t* __restrict__ perm, OccupancyView grid, BeamParams params, const double2* __restrict__ points,
                        uint32_t n_points, const uint32_t* __restrict__ hits, uint64_t hit_stride, Scalars* __restrict__ scalars) {
  __shared__ double2 s_beam[kMixChunk];  // {z, exp(-lambda_short * z)}
  __shared__ unsigned long long s_red[kMixThreads / kWarp];
  const uint64_t local = static_cast<uint64_t>(blockIdx.x) * kMixThreads + threadIdx.x;
  const uint64_t slot = slot_base + local;
  const bool active = local < slot_count && slot < n;
  const uint64_t i = active ? (perm != nullptr ? perm[slot] : slot) : 0;
  const Pose2 src = pose_mul(grid.world_to_grid, active ? load_pose(states + i) : Pose2{1.0, 0.0, 0.0, 0.0});
  const int sx = cell_near(src.x, grid.inv_resolution), sy = cell_near(src.y, grid.inv_resolution);
  const double source_x = (static_cast<double>(sx) + 0.5) * grid.resolution, source_y = (static_cast<double>(sy) + 0.5) * grid.resolution;
  const double n_norm = 1. / (sqrt(2. * 3.14159265358979323846) * params.sigma_hit);  // beam_model.hpp:107

  auto value = [&](uint32_t word, const double2& beam) {
    const bool hit_cell = word != kHitMiss;
    const int cx = static_cast<int>(word & 0xFFFFu), cy = static_cast<int>(word >> 16);
    // distance between the centroids of the source cell and the hit cell (raycasting.hpp:91-104), clamped to the range
    const double dxm = (static_cast<double>(cx) + 0.5) * grid.resolution - source_x;
    const double dym = (static_cast<double>(cy) + 0.5) * grid.resolution - source_y;
    const double hit = fmin(sqrt(dxm * dxm + dym * dym), params.beam_max_range);
    const double z_mean = hit_cell ? hit : params.beam_max_range;  // value_or(beam_max_range)
    double2 eta;
    if (params.eta != nullptr) {
      const long long ix = static_cast<long long>(cx) - sx, iy = static_cast<long long>(cy) - sy;
      const unsigned long long d2 = static_cast<unsigned long long>(ix * ix + iy * iy);
      const bool in_table = hit_cell && hit < params.beam_max_range && d2 + 1 < params.eta_entries;
      eta = __ldg(params.eta + (in_table ? static_cast<uint32_t>(d2) : params.eta_entries - 1u));
    } else {
      eta = beam_normalisers(params, z_mean);
    }
    return beam_pz3(params, beam.x, beam.y, z_mean, n_norm, eta.x, eta.y);
  };

  double acc = 0.0;
  for (uint32_t base = 0; base < n_points; base += kMixChunk) {
    const uint32_t count = min(kMixChunk, n_points - base);
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < count; b += kMixThreads) {
      const double2 p = points[base + b];
      const double z = sqrt(p.x * p.x + p.y * p.y);  // beam_model.hpp:116
      s_beam[b] = make_double2(z, exp(-params.lambda_short * z));
    }
    __syncthreads();
    if (!active) continue;
    const uint32_t* h = hits + static_cast<uint64_t>(base) * hit_stride + local;
    uint32_t b = 0;
    for (; b + 4 <= count; b += 4) {  // transform_reduce grouping (numeric:439-462)
      const uint32_t w0 = __ldcs(h + static_cast<uint64_t>(b) * hit_stride), w1 = __ldcs(h + static_cast<uint64_t>(b + 1) * hit_stride);
      const uint32_t w2 = __ldcs(h + static_cast<uint64_t>(b + 2) * hit_stride), w3 = __ldcs(h + static_cast<uint64_t>(b + 3) * hit_stride);
      const double f0 = value(w0, s_beam[b]), f1 = value(w1, s_beam[b + 1]), f2 = value(w2, s_beam[b + 2]), f3 = value(w3, s_beam[b + 3]);
      acc = acc + ((f0 + f1) + (f2 + f3));
    }
    for (; b < count; ++b) acc = acc + value(__ldcs(h + static_cast<uint64_t>(b) * hit_stride), s_beam[b]);
  }
  double w = 0.0;
  if (active) {
    w = weights[i] * acc;  // actions/reweight.hpp:54-60
    weights[i] = w;
  }
  const unsigned long long m = block_max_u64<kMixThreads>(active ? weight_order_bits(w) : 0ull, s_red);
  if (threadIdx.x == 0 && m != 0) atomicMax(&scalars->wmax_bits, m);
}

__global__ void __launch_bounds__(512) max_weight_kernel(const double* __restrict__ weights, uint64_t n, Scalars* scalars) {
  __shared__ unsigned long long s_red[512 / kWarp];
  unsigned long long m = 0;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * 512 + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * 512) {
    const unsigned long long b = weight_order_bits(weights[i]);
    m = b > m ? b : m;
  }
  m = block_max_u64<512>(m, s_red);
  if (threadIdx.x == 0 && m != 0) atomicMax(&scalars->wmax_bits, m);
}

// ---- fixed-point CDF ------------------------------------------------------------------------------
// q_i = floor(w_i * 2^e) with e chosen so that the largest weight lands in [2^(P-1), 2^P),
// P = min(52, 62 - ceil(log2(N_global))): the total stays below 2^62 and integer addition is
// associative, so the CDF is identical for any scan order, tile size or number of ranks.

constexpr int kScanThreads = 512;
constexpr int kScanItems = 8;
constexpr uint32_t kScanTile = kScanThreads * kScanItems;
// tile_state word: [63:62] flag (0 empty, 1 aggregate, 2 inclusive prefix), [61:0] value
constexpr unsigned long long kFlagAggregate = 1ull << 62, kFlagPrefix = 2ull << 62, kValueMask = (1ull << 62) - 1;

__device__ __forceinline__ void prepare_cdf_scalars(Scalars* s, double wmax, int ceil_log2_count) {
  int ex = 0;
  const bool ok = wmax > 0.0 && wmax <= DBL_MAX;
  if (ok) (void)frexp(wmax, &ex);
  const int p = min(52, 62 - ceil_log2_count);
  s->exponent = p - ex;
  s->valid = ok ? 1 : 0;
  s->tile_ticket = 0;
  s->total = 0;
}

__global__ void prepare_cdf_kernel(Scalars* s, double host_wmax, int ceil_log2_count, unsigned long long* tile_state, uint32_t n_tiles) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n_tiles; t += gridDim.x * blockDim.x) tile_state[t] = 0;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const double wmax = host_wmax >= 0.0 ? host_wmax : __longlong_as_double(static_cast<long long>(s->wmax_bits));
    prepare_cdf_scalars(s, wmax, ceil_log2_count);
  }
}

/// Inclusive scan of per-thread totals across the block (warp shuffles + one smem hop).
template <int kThreads>
__device__ __forceinline__ unsigned long long block_inclusive_scan_u64_n(unsigned long long v, unsigned long long* warp_sums,
                                                                          unsigned long long& block_total) {
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
#pragma unroll
  for (int off = 1; off < kWarp; off <<= 1) {
    const unsigned long long o = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= off) v += o;
  }
  if (lane == kWarp - 1) warp_sums[warp] = v;
  __syncthreads();
  if (warp == 0) {
    unsigned long long ws = lane < kThreads / kWarp ? warp_sums[lane] : 0ull;
#pragma unroll
    for (int off = 1; off < kWarp; off <<= 1) {
      const unsigned long long o = __shfl_up_sync(0xffffffffu, ws, off);
      if (lane >= off) ws += o;
    }
    if (lane < kThreads / kWarp) warp_sums[lane] = ws;
  }
  __syncthreads();
  block_total = warp_sums[kThreads / kWarp - 1];
  return v + (warp > 0 ? warp_sums[warp - 1] : 0ull);
}

__device__ __forceinline__ unsigned long long block_inclusive_scan_u64(unsigned long long v, unsigned long long* warp_sums,
                                                                        unsigned long long& block_total) {
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
#pragma unroll
  for (int off = 1; off < kWarp; off <<= 1) {
    const unsigned long long o = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= off) v += o;
  }
  if (lane == kWarp - 1) warp_sums[warp] = v;
  __syncthreads();
  if (warp == 0) {
    unsigned long long ws = lane < kScanThreads / kWarp ? warp_sums[lane] : 0ull;
#pragma unroll
    for (int off = 1; off < kWarp; off <<= 1) {
      const unsigned long long o = __shfl_up_sync(0xffffffffu, ws, off);
      if (lane >= off) ws += o;
    }
    if (lane < kScanThreads / kWarp) warp_sums[lane] = ws;
  }
  __syncthreads();
  block_total = warp_sums[kScanThreads / kWarp - 1];
  return v + (warp > 0 ? warp_sums[warp - 1] : 0ull);
}

/// Decoupled look-back: returns the exclusive prefix of this tile and publishes its inclusive one.
/// Warp 0 inspects 32 predecessors per round (one coalesced read of the tile words) instead of walking
/// them one L2 round trip at a time.
__device__ __forceinline__ unsigned long long lookback_exclusive_prefix(unsigned long long* tile_state, uint32_t tile,
                                                                         unsigned long long tile_total, unsigned long long* s_prefix) {
  if (threadIdx.x < kWarp) {
    const int lane = threadIdx.x;
    unsigned long long exclusive = 0;
    if (tile == 0) {
      if (lane == 0) atomicExch(&tile_state[0], kFlagPrefix | tile_total);
    } else {
      if (lane == 0) atomicExch(&tile_state[tile], kFlagAggregate | tile_total);
      int32_t window = static_cast<int32_t>(tile) - 1;  // newest predecessor of this round
      for (;;) {
        const int32_t look = window - lane;
        unsigned long long word;
        do {  // tiles before tile 0 count as a published prefix of zero
          word = look >= 0 ? *reinterpret_cast<volatile unsigned long long*>(&tile_state[look]) : (2ull << 62);
        } while (__any_sync(0xffffffffu, (word >> 62) == 0));
        const unsigned prefixes = __ballot_sync(0xffffffffu, (word >> 62) == 2);
        const int last = prefixes != 0 ? __ffs(prefixes) - 1 : kWarp - 1;  // nearest tile that already knows its prefix
        unsigned long long v = lane <= last ? (word & kValueMask) : 0ull;
#pragma unroll
        for (int off = kWarp / 2; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        exclusive += v;
        if (prefixes != 0) break;
        window -= kWarp;
      }
      if (lane == 0) atomicExch(&tile_state[tile], kFlagPrefix | (exclusive + tile_total));
    }
    if (lane == 0) *s_prefix = exclusive;
  }
  __syncthreads();
  return *s_prefix;
}

// Tile of the CDF build: 256 threads x 8 consecutive weights (two 32-byte sectors per thread, read and written with
// 16-byte accesses).  The quantisation is a multiplication by 2^e (exact, like scalbn, wherever the result is >= 1),
// split into two power-of-two factors so that each stays a normal double for any exponent.
constexpr int kQsThreads = 256;
constexpr int kQsItemsSmall = 8;   // up to a few million weights: more tiles than SM slots, shortest chain
#ifndef BB200_QS_LARGE_ITEMS
#define BB200_QS_LARGE_ITEMS 8  // 16 halves the tiles per byte but measured slower at 12.5M (83 us against 67)
#endif
constexpr int kQsItemsLarge = BB200_QS_LARGE_ITEMS;
constexpr uint32_t kQsTile = kQsThreads * kQsItemsSmall;  // the smaller tile sizes the look-back state

__device__ __forceinline__ double pow2_double(int e) {  // |e| <= 1000
  return __longlong_as_double(static_cast<long long>(e + 1023) << 52);
}
__device__ __forceinline__ unsigned long long quantize_mul(double w, double f1, double f2) {
  const double scaled = (w * f1) * f2;
  return scaled > 0.0 ? __double2ull_rd(scaled) : 0ull;  // zero / negative / NaN weights are never selected
}

/// derive_exponent: the fused step -- the exponent comes from scalars->wmax_bits here (no prepare_cdf launch; the
/// tile holding element 0 publishes exponent / valid for the host); otherwise scalars->exponent / valid are given.
template <int kQsItems>
__global__ void __launch_bounds__(kQsThreads) quantize_scan_kernel(const double* __restrict__ weights, uint64_t n,
                                                                   unsigned long long* __restrict__ cdf, Scalars* scalars,
                                                                   unsigned long long* tile_state, int derive_exponent, int ceil_log2_count) {
  __shared__ unsigned long long s_warp[kQsThreads / kWarp];
  __shared__ unsigned long long s_prefix;
  // Tiles are taken in blockIdx order (CTAs are dispatched in that order, which is what the look-back's forward progress
  // needs -- the same assumption CUB's decoupled look-back makes): no ticket atomic and no barrier before the loads.
  const uint32_t tile = blockIdx.x;
  int exponent, valid_flag;
  if (derive_exponent) {  // every thread derives the exponent itself: a broadcast load and a few integer operations
    const double wmax = __longlong_as_double(static_cast<long long>(scalars->wmax_bits));
    int ex = 0;
    const bool ok = wmax > 0.0 && wmax <= DBL_MAX;
    if (ok) (void)frexp(wmax, &ex);
    exponent = min(52, 62 - ceil_log2_count) - ex;
    valid_flag = ok ? 1 : 0;
    if (tile == 0 && threadIdx.x == 0) {
      scalars->exponent = exponent;
      scalars->valid = valid_flag;
    }
  } else {
    exponent = scalars->exponent;
    valid_flag = scalars->valid;
  }
  const int e1 = exponent / 2;
  const double f1 = pow2_double(e1), f2 = pow2_double(exponent - e1);
  const bool valid = valid_flag != 0;

  const uint64_t base = static_cast<uint64_t>(tile) * (kQsThreads * kQsItems) + static_cast<uint64_t>(threadIdx.x) * kQsItems;
  unsigned long long q[kQsItems];
  unsigned long long local = 0;
  if (base + kQsItems <= n) {
    const double2* src = reinterpret_cast<const double2*>(weights + base);
#pragma unroll
    for (int k = 0; k < kQsItems / 2; ++k) {
      const double2 w = __ldcs(src + k);  // read once: streaming
      // Degenerate weight set (no positive finite weight): fall back to a uniform CDF.
      q[2 * k] = valid ? quantize_mul(w.x, f1, f2) : (1ull << 20);
      q[2 * k + 1] = valid ? quantize_mul(w.y, f1, f2) : (1ull << 20);
      local += q[2 * k] + q[2 * k + 1];
    }
  } else {
#pragma unroll
    for (int k = 0; k < kQsItems; ++k) {
      const uint64_t idx = base + k;
      q[k] = idx < n ? (valid ? quantize_mul(weights[idx], f1, f2) : (1ull << 20)) : 0ull;
      local += q[k];
    }
  }
  unsigned long long tile_total;
  const unsigned long long inclusive = block_inclusive_scan_u64_n<kQsThreads>(local, s_warp, tile_total);
  const unsigned long long prefix = lookback_exclusive_prefix(tile_state, tile, tile_total, &s_prefix);
  unsigned long long running = prefix + inclusive - local;
  if (base + kQsItems <= n) {
    ulonglong2* dst = reinterpret_cast<ulonglong2*>(cdf + base);
#pragma unroll
    for (int k = 0; k < kQsItems / 2; ++k) {
      ulonglong2 v;
      running += q[2 * k];
      v.x = running;
      running += q[2 * k + 1];
      v.y = running;
      dst[k] = v;
    }
  } else {
#pragma unroll
    for (int k = 0; k < kQsItems; ++k) {
      const uint64_t idx = base + k;
      running += q[k];
      if (idx < n) cdf[idx] = running;
    }
  }
  if (base <= n - 1 && n - 1 < base + kQsItems) scalars->total = prefix + inclusive;  // thread holding the last element
}

/// Exclusive prefix sum of u32 values (bin counters, KLD first-occurrence flags) with the same
/// decoupled look-back machinery; `in` and `out` may alias.
__global__ void __launch_bounds__(kScanThreads) scan_u32_kernel(const uint32_t* in, uint32_t* out, uint32_t n, unsigned long long* ticket,
                                                                unsigned long long* tile_state, unsigned long long* total_out) {
  __shared__ unsigned long long s_warp[kScanThreads / kWarp];
  __shared__ unsigned long long s_prefix;
  (void)ticket;  // tiles in blockIdx order (see quantize_scan_kernel)
  const uint32_t tile = blockIdx.x;
  const uint32_t base = tile * kScanTile + threadIdx.x * kScanItems;
  unsigned long long q[kScanItems];
  unsigned long long local = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    q[k] = base + k < n ? in[base + k] : 0u;
    local += q[k];
  }
  unsigned long long tile_total;
  const unsigned long long inclusive = block_inclusive_scan_u64(local, s_warp, tile_total);
  const unsigned long long prefix = lookback_exclusive_prefix(tile_state, tile, tile_total, &s_prefix);
  unsigned long long running = prefix + inclusive - local;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    if (base + k < n) out[base + k] = static_cast<uint32_t>(running);
    running += q[k];
  }
  if (total_out != nullptr && base <= n - 1 && n - 1 < base + kScanItems) *total_out = prefix + inclusive;
}

// ---- KLD-adaptive sample size (a12) -----------------------------------------------------------------
// views::take_while_kld (views/take_while_kld.hpp:72-137) keeps drawing while
//   count <= min  ||  count <= target(k),   k = number of distinct spatial-hash buckets so far,
// a sequential early exit over an unordered_set.  Here candidate slots are generated in chunks;
// a device hash set keeps, per bucket, the SMALLEST slot index that produced it, so "slot j is the
// first occurrence of its bucket" is an order-independent fact; a prefix sum of those flags gives
// k after every slot and the first failing count is a min-reduction.

constexpr unsigned long long kEmptyKey = ~0ull;

__device__ __forceinline__ uint64_t kld_probe_start(unsigned long long key, uint64_t mask) {
  unsigned long long h = key * 0x9E3779B97F4A7C15ull;
  return (h ^ (h >> 29)) & mask;
}

__global__ void __launch_bounds__(256) kld_insert_kernel(const unsigned long long* __restrict__ hashes, uint64_t n, uint64_t slot_base,
                                                         unsigned long long* keys, unsigned int* vals, uint64_t mask) {
  const uint64_t j = static_cast<uint64_t>(blockIdx.x) * 256 + threadIdx.x;
  if (j >= n) return;
  unsigned long long key = hashes[j];
  if (key == kEmptyKey) key = kEmptyKey - 1;  // the sentinel itself cannot be stored (2^-64 event)
  uint64_t pos = kld_probe_start(key, mask);
  for (;;) {
    const unsigned long long prev = atomicCAS(keys + pos, kEmptyKey, key);
    if (prev == kEmptyKey || prev == key) {
      atomicMin(vals + pos, static_cast<unsigned int>(slot_base + j));
      return;
    }
    pos = (pos + 1) & mask;
  }
}

__global__ void __launch_bounds__(256) kld_flag_kernel(const unsigned long long* __restrict__ hashes, uint64_t n, uint64_t slot_base,
                                                       const unsigned long long* __restrict__ keys, const unsigned int* __restrict__ vals,
                                                       uint64_t mask, uint32_t* __restrict__ flags) {
  const uint64_t j = static_cast<uint64_t>(blockIdx.x) * 256 + threadIdx.x;
  if (j >= n) return;
  unsigned long long key = hashes[j];
  if (key == kEmptyKey) key = kEmptyKey - 1;
  uint64_t pos = kld_probe_start(key, mask);
  while (keys[pos] != key) pos = (pos + 1) & mask;
  flags[j] = vals[pos] == static_cast<unsigned int>(slot_base + j) ? 1u : 0u;
}

/// kld_condition target size (views/take_while_kld.hpp:73-80), same operation order as the reference.
__device__ __forceinline__ bool kld_count_allowed(unsigned long long count, unsigned long long k, unsigned long long min_count, double two_epsilon, double z) {
  if (count <= min_count || k <= 2ull) return true;
  const double common = 2. / static_cast<double>(9 * (k - 1));
  const double base = 1. - common + sqrt(common) * z;
  const double result = (static_cast<double>(k - 1) / two_epsilon) * base * base * base;
  const double target = ceil(result);
  return target >= 18446744073709551615.0 || count <= static_cast<unsigned long long>(target);
}

__global__ void __launch_bounds__(256) kld_check_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ exclusive, uint64_t n,
                                                        uint64_t slot_base, unsigned long long k_before, unsigned long long min_count,
                                                        double two_epsilon, double z, Scalars* scalars) {
  const uint64_t j = static_cast<uint64_t>(blockIdx.x) * 256 + threadIdx.x;
  unsigned long long failing = ~0ull;
  if (j < n) {
    const unsigned long long count = slot_base + j + 1;
    const unsigned long long k = k_before + exclusive[j] + flags[j];
    if (!kld_count_allowed(count, k, min_count, two_epsilon, z)) failing = count;
  }
  // Past the cutoff nearly every slot fails: one atomic per warp instead of one per thread on the same word.
#pragma unroll
  for (int off = kWarp / 2; off > 0; off >>= 1) {
    const unsigned long long o = __shfl_down_sync(0xffffffffu, failing, off);
    failing = o < failing ? o : failing;
  }
  if (threadIdx.x % kWarp == 0 && failing != ~0ull && failing < *reinterpret_cast<volatile unsigned long long*>(&scalars->kld_cutoff))
    atomicMin(&scalars->kld_cutoff, failing);
}

__global__ void kld_reset_kernel(Scalars* scalars) {
  scalars->kld_cutoff = ~0ull;
  scalars->pad[0] = 0;  // tile ticket of the flag scan
  scalars->pad[1] = 0;  // distinct buckets in the chunk
}

// ---- normalize -------------------------------------------------------------------------------------

constexpr int kStreamThreads = 256;

__global__ void __launch_bounds__(kStreamThreads) normalize_kernel(double* __restrict__ weights, uint64_t n, const Scalars* scalars,
                                                                   unsigned long long global_total, double* __restrict__ partials) {
  __shared__ double s_red[kStreamThreads / kWarp];
  // S = T * 2^-e: the normalisation factor derived from the exact integer total.
  // 0: single GPU, the total is on the device; ~0: sharded, the sum of the ranks' totals is on the device
  const unsigned long long t = global_total == ~0ull ? scalars->global_total : (global_total != 0 ? global_total : scalars->total);
  const double factor = scalbn(static_cast<double>(t), -scalars->exponent);
  const bool valid = scalars->valid != 0 && factor > 0.0;
  double sq = 0.0;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * kStreamThreads + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * kStreamThreads) {
    double w = weights[i];
    if (valid) {
      w = w / factor;  // actions/normalize.hpp:82
      weights[i] = w;
    }
    sq = sq + w * w;
  }
  const double total = block_sum<kStreamThreads>(sq, s_red);
  if (threadIdx.x == 0) partials[blockIdx.x] = total;
}

// ---- resample -------------------------------------------------------------------------------------

constexpr int kRsThreads = 256;

/// Smallest i in [0, n) with cdf[i] > t.
__device__ __forceinline__ uint64_t cdf_upper_bound(const unsigned long long* __restrict__ cdf, uint64_t n, unsigned long long t) {
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    const uint64_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(cdf + mid) > t) {
      hi = mid;
    } else {
      lo = mid + 1;
    }
  }
  return lo < n ? lo : n - 1;  // unreachable clamp (t < total by construction)
}

__device__ __forceinline__ void accumulate_moments(double* m, const Pose2& st, double w, double px, double py) {
  const double dx = st.x - px, dy = st.y - py;
  m[0] += w;
  m[1] += w * w;
  m[2] += w * st.c;
  m[3] += w * st.s;
  m[4] += w * dx;
  m[5] += w * dy;
  m[6] += w * dx * dx;
  m[7] += w * dx * dy;
  m[8] += w * dy * dy;
}

template <int kThreads>
__device__ __forceinline__ void store_block_moments(double* m, double* scratch /* kMomentCount * kThreads/32 */, double* __restrict__ partials_row) {
  block_sum_many<kThreads, kMomentCount>(m, scratch);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < kMomentCount; ++k) partials_row[k] = m[k];
  }
}

/// Stores the block's raw moments and, when the launch carries a StepTail, lets the LAST block to arrive add the
/// per-block rows up in a fixed order (thread-strided over the rows, then the block tree: the same sum for any
/// arrival order) -- the reduce_partials launch and the read-back copies of the fused step folded into the resample.
/// With tail.summary set (single GPU: pinned host memory, written straight over PCIe) the host finds the step's
/// results after its one stream synchronisation.
template <int kThreads>
__device__ __forceinline__ void finish_block_moments(double* m, double* scratch, double* __restrict__ moment_partials, Scalars* scalars,
                                                     const StepTail& tail) {
  store_block_moments<kThreads>(m, scratch, moment_partials + static_cast<size_t>(blockIdx.x) * kMomentCount);
  if (!tail.enabled) return;
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    __threadfence();  // the row above before the arrival count
    s_last = atomicAdd(&scalars->blocks_done, 1u) + 1u == gridDim.x ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double v[kMomentCount];
#pragma unroll
  for (int k = 0; k < kMomentCount; ++k) v[k] = 0.0;
  for (uint32_t r = threadIdx.x; r < gridDim.x; r += kThreads) {
    const double* row = moment_partials + static_cast<size_t>(r) * kMomentCount;
#pragma unroll
    for (int k = 0; k < kMomentCount; ++k) v[k] = v[k] + __ldcg(row + k);  // nine independent loads per row
  }
  block_sum_many<kThreads, kMomentCount>(v, scratch);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < kMomentCount; ++k) {
      tail.results[k] = v[k];
      if (tail.summary != nullptr) tail.summary->moments[k] = v[k];
    }
  }
  if (threadIdx.x == 0) {
    scalars->blocks_done = 0;
    if (tail.summary != nullptr) {
      tail.summary->total = scalars->total;
      tail.summary->exponent = scalars->exponent;
      tail.summary->valid = scalars->valid;
      tail.summary->error = 0;
      __threadfence_system();
      if (tail.seq != 0) {  // the host polls this word instead of synchronising with the stream
        *reinterpret_cast<volatile int*>(&tail.summary->seq) = tail.seq;
        __threadfence_system();
      }
    }
  }
}

__global__ void __launch_bounds__(kRsThreads) resample_kernel(ResampleArgs a, Scalars* __restrict__ scalars, double* __restrict__ moment_partials) {
  __shared__ double s_red[kMomentCount * kRsThreads / kWarp];
  unsigned long long total = a.global_total != 0 ? a.global_total : scalars->total;
  unsigned long long cdf_offset = a.cdf_offset, span_end = 0;
  uint64_t slot_first = a.slot_first, slot_count = a.slot_count;
  if (a.rank_totals != nullptr) {  // offsets = exclusive prefix of the ranks' totals (distributed.py: cdf_offsets)
    total = 0;
    cdf_offset = 0;
    for (int r = 0; r < a.world; ++r) {
      const unsigned long long t = a.rank_totals[r];
      if (r < a.rank) cdf_offset += t;
      total += t;
    }
    span_end = cdf_offset + a.rank_totals[a.rank];
  }
  unsigned long long stride = 0, offset = 0;
  if (a.scheme == 1) {
    // Systematic comb: stride = T / M, offset uniform in [0, stride).
    stride = total / a.total_slots;
    offset = mulhi64(counter_draw(a.seed, 0, a.step, kStreamSystematic).a, stride);
    if (a.rank_totals != nullptr) {
      // The slots whose comb position offset + j*stride lies in [cdf_offset, span_end) (distributed.py: slot_ranges).
      auto first_slot_at_or_after = [&](unsigned long long position) -> uint64_t {
        if (position <= offset) return 0;
        const unsigned long long j = (position - offset + stride - 1) / stride;
        return j < a.total_slots ? j : a.total_slots;
      };
      slot_first = first_slot_at_or_after(cdf_offset);
      uint64_t slot_end = a.rank + 1 == a.world ? a.total_slots : first_slot_at_or_after(span_end);
      // KLD on shards: only the slots of the current window [window_begin, window_end) -- the chunk being counted, or
      // [0, accepted count) for the final pass -- are produced.
      if (a.window_end > a.window_begin) {
        slot_first = slot_first < a.window_begin ? a.window_begin : slot_first;
        slot_end = slot_end > a.window_end ? a.window_end : slot_end;
      }
      slot_count = slot_end > slot_first ? slot_end - slot_first : 0;
    }
  }
  double m[kMomentCount];
#pragma unroll
  for (int k = 0; k < kMomentCount; ++k) m[k] = 0.0;

  for (uint64_t local = static_cast<uint64_t>(blockIdx.x) * kRsThreads + threadIdx.x; local < slot_count;
       local += static_cast<uint64_t>(gridDim.x) * kRsThreads) {
    const uint64_t j = slot_first + local;
    Pose2 st;
    long long ancestor = -1;
    bool inject = false;
    Draw d{0, 0};
    if (a.random_state_probability > 0.0 || a.scheme == 0) d = counter_draw(a.seed, j, a.step, kStreamResample);
    // random_intersperse.hpp:93-100: one coin per ADVANCE of the view -- slot 0, the element begin() yields, is never injected
    if (a.random_state_probability > 0.0) inject = j > 0 && uniform01(d.a) < a.random_state_probability;
    unsigned long long t = 0;
    if (!inject) t = a.scheme == 1 ? offset + j * stride : mulhi64(d.b, total);
    if (a.span_filter != 0) {
      // an injected state belongs to the slot's owner; with a particle count that is still being decided (KLD on shards)
      // slots are dealt round robin instead
      const bool my_slot = a.inject_mod > 0 ? (j % static_cast<uint64_t>(a.inject_mod) == static_cast<uint64_t>(a.rank))
                                            : (j >= a.owner_first && j - a.owner_first < a.owner_count);
      const bool mine = inject ? my_slot : (t >= cdf_offset && t - cdf_offset < scalars->total);
      if (!mine) continue;
    }
    if (inject) {
      st = random_free_state(FreeSpace{a.free_cells, a.n_free, a.grid_width, a.grid_resolution, a.grid_origin},
                             counter_draw(a.seed, j, a.step, kStreamRandomState));
    } else {
      const uint64_t idx = cdf_upper_bound(a.cdf, a.n_in, t - cdf_offset);  // the caller guarantees t lies in this shard's span
      ancestor = static_cast<long long>(idx);
      st = load_pose(a.states_in + idx);
    }
    if (a.peer_hash_count > 0) {
      // KLD on shards, counting pass: only the candidate's spatial hash is needed, and every rank needs it -- the
      // ranks then count distinct buckets over the same globally ordered hash stream and reach the same cutoff.
      const unsigned long long h = spatial_hash(st, a.hash_resolution[0], a.hash_resolution[1], a.hash_resolution[2]);
      for (int r = 0; r < a.peer_hash_count; ++r) a.peer_hashes[r][j] = h;
      continue;
    }
    if (a.peer_count > 0) {
      const uint64_t owner = j / a.peer_shard;  // P2P store over NVLink (or a local store when owner == this rank)
      store_pose(a.peer_out[owner] + (j - owner * a.peer_shard), st);
    } else {
      store_pose(a.states_out + local, st);
    }
    if (a.weights_out != nullptr) a.weights_out[local] = 1.0;  // make_from_state (particle_traits.hpp:105)
    if (a.ancestors != nullptr) a.ancestors[local] = ancestor;
    if (a.hashes != nullptr) a.hashes[local] = spatial_hash(st, a.hash_resolution[0], a.hash_resolution[1], a.hash_resolution[2]);
    accumulate_moments(m, st, 1.0, a.pivot_x, a.pivot_y);
  }
  finish_block_moments<kRsThreads>(m, s_red, moment_partials, scalars, a.tail);
}

// ---- resample, scatter form (systematic comb on one GPU) ----------------------------------------------
// With the comb t_j = offset + j * stride the slots that pick particle i are exactly those with
// cdf[i-1] <= t_j < cdf[i]: a contiguous slot range [ja, jb) that follows from two integer divisions.
// So instead of a binary search per SLOT (20 dependent probes of the CDF) every PARTICLE reads its two
// CDF entries and stores its state jb - ja times.  Same ancestors as resample_kernel by construction
// (the parity tests compare them with the oracle's lower_bound search); the raw moments are summed per
// particle (count * term) instead of per slot, which moves the estimate at rounding level only.

__device__ __forceinline__ uint64_t comb_slots_before(unsigned long long position, unsigned long long offset, unsigned long long stride,
                                                     uint64_t total_slots) {
  if (position <= offset) return 0;  // number of slots j with offset + j * stride < position
  const unsigned long long j = (position - offset + stride - 1) / stride;
  return j < total_slots ? j : total_slots;
}

/// The same with the division replaced by a multiplication with magic = floor((2^64 - 1) / stride): the high word of
/// x * magic is the quotient or one below it (x < 2^64, so the error of the reciprocal costs less than 1); one
/// remainder check makes it exact.  A 64-bit division is ~150 instructions; this is 8.
__device__ __forceinline__ uint64_t comb_slots_before_magic(unsigned long long position, unsigned long long offset, unsigned long long stride,
                                                           unsigned long long magic, uint64_t total_slots) {
  if (position <= offset) return 0;
  const unsigned long long x = position - offset + stride - 1;
  unsigned long long j = __umul64hi(x, magic);
  if (x - j * stride >= stride) ++j;
  return j < total_slots ? j : total_slots;
}

__global__ void __launch_bounds__(kRsThreads, BB200_RS_BLOCKS) resample_scatter_kernel(ResampleArgs a, Scalars* __restrict__ scalars,
                                                                     double* __restrict__ moment_partials) {
  __shared__ double s_red[kMomentCount * kRsThreads / kWarp];
  __shared__ unsigned long long s_comb[3];
  // One GPU: the local CDF is the global one.  Sharded (rank_totals set): positions shift by the totals of
  // the lower ranks and every copy goes to the rank that owns its slot, over NVLink peer memory.
  unsigned long long total = scalars->total, cdf_offset = 0;
  if (a.rank_totals != nullptr) {
    total = 0;
    for (int r = 0; r < a.world; ++r) {
      const unsigned long long t = a.rank_totals[r];
      if (r < a.rank) cdf_offset += t;
      total += t;
    }
  }
  if (threadIdx.x == 0) {  // the two 64-bit divisions of the comb, once per block
    const unsigned long long st = total / a.total_slots;
    s_comb[0] = st;
    s_comb[1] = mulhi64(counter_draw(a.seed, 0, a.step, kStreamSystematic).a, st);
    s_comb[2] = ~0ull / (st != 0 ? st : 1ull);
  }
  __syncthreads();
  const unsigned long long stride = s_comb[0], offset = s_comb[1], magic = s_comb[2];
  // the comb spans total_slots; only the slots below window_end (KLD: the accepted count) are produced
  const uint64_t slot_limit = a.window_end > 0 ? a.window_end : a.total_slots;
  const int lane = threadIdx.x % kWarp;
  double m[kMomentCount];
#pragma unroll
  for (int k = 0; k < kMomentCount; ++k) m[k] = 0.0;

  auto store_copy = [&](uint64_t j, const Pose2& st, uint64_t ancestor) {
    if (a.peer_count > 0) {
      const uint64_t owner = j / a.peer_shard;
      store_pose(a.peer_out[owner] + (j - owner * a.peer_shard), st);
    } else {
      store_pose(a.states_out + j, st);
      if (a.weights_out != nullptr) a.weights_out[j] = 1.0;  // make_from_state (particle_traits.hpp:105)
      if (a.ancestors != nullptr) a.ancestors[j] = static_cast<long long>(ancestor);
    }
  };

  // kRsUnroll particles per thread and round: their CDF reads, divisions and state loads are independent, so one thread keeps
  // several 32-byte gathers in flight (the kernel is bound by the latency of cdf -> state -> store, not by bandwidth).
  // Every thread runs the same number of rounds: whole warps stay together for the cooperative stores.
  constexpr int kRsUnroll = BB200_RS_UNROLL;
  constexpr uint64_t kOwnCopies = 4;  // up to this many copies a thread stores itself
  const uint64_t per_round = static_cast<uint64_t>(gridDim.x) * kRsThreads * kRsUnroll;
  const uint64_t rounds = (a.n_in + per_round - 1) / per_round;
  for (uint64_t round = 0; round < rounds; ++round) {
    const uint64_t first = round * per_round + static_cast<uint64_t>(blockIdx.x) * kRsThreads * kRsUnroll + threadIdx.x;
    uint64_t ja[kRsUnroll], copies[kRsUnroll];
#pragma unroll
    for (int u = 0; u < kRsUnroll; ++u) {
      const uint64_t i = first + static_cast<uint64_t>(u) * kRsThreads;
      ja[u] = 0;
      copies[u] = 0;
      if (i < a.n_in) {
        ja[u] = comb_slots_before_magic(cdf_offset + (i > 0 ? __ldg(a.cdf + i - 1) : 0ull), offset, stride, magic, slot_limit);
        copies[u] = comb_slots_before_magic(cdf_offset + __ldg(a.cdf + i), offset, stride, magic, slot_limit) - ja[u];
      }
    }
    Pose2 st[kRsUnroll];
#pragma unroll
    for (int u = 0; u < kRsUnroll; ++u) {
      st[u] = Pose2{1.0, 0.0, 0.0, 0.0};
      if (copies[u] > 0) st[u] = load_pose(a.states_in + first + static_cast<uint64_t>(u) * kRsThreads);
    }
#pragma unroll
    for (int u = 0; u < kRsUnroll; ++u) {
      const uint64_t i = first + static_cast<uint64_t>(u) * kRsThreads;
      if (copies[u] > 0) {
        const double c = static_cast<double>(copies[u]), dx = st[u].x - a.pivot_x, dy = st[u].y - a.pivot_y;
        m[0] += c;  // every copy has weight 1: sum w = sum w^2 = copies
        m[1] += c;
        m[2] += c * st[u].c;
        m[3] += c * st[u].s;
        m[4] += c * dx;
        m[5] += c * dy;
        m[6] += c * (dx * dx);
        m[7] += c * (dx * dy);
        m[8] += c * (dy * dy);
      }
      if (copies[u] <= kOwnCopies) {
        for (uint64_t j = ja[u]; j < ja[u] + copies[u]; ++j) store_copy(j, st[u], i);
      }
    }
    // Heavy particles: the warp stores their copies together, 32 slots per round.
#pragma unroll
    for (int u = 0; u < kRsUnroll; ++u) {
      unsigned heavy = __ballot_sync(0xffffffffu, copies[u] > kOwnCopies);
      while (heavy != 0u) {
        const int src = __ffs(heavy) - 1;
        heavy &= heavy - 1u;
        const uint64_t hja = __shfl_sync(0xffffffffu, ja[u], src), hcopies = __shfl_sync(0xffffffffu, copies[u], src);
        const uint64_t hi = __shfl_sync(0xffffffffu, first + static_cast<uint64_t>(u) * kRsThreads, src);
        Pose2 hs;
        hs.c = __shfl_sync(0xffffffffu, st[u].c, src);
        hs.s = __shfl_sync(0xffffffffu, st[u].s, src);
        hs.x = __shfl_sync(0xffffffffu, st[u].x, src);
        hs.y = __shfl_sync(0xffffffffu, st[u].y, src);
        for (uint64_t j = hja + lane; j < hja + hcopies; j += kWarp) store_copy(j, hs, hi);
      }
    }
  }
  finish_block_moments<kRsThreads>(m, s_red, moment_partials, scalars, a.tail);
}

// ---- moments / reductions -------------------------------------------------------------------------

__global__ void __launch_bounds__(kStreamThreads) moments_kernel(const Pose2* __restrict__ states, const double* __restrict__ weights, uint64_t n,
                                                                 double px, double py, double* __restrict__ moment_partials) {
  __shared__ double s_red[kMomentCount * kStreamThreads / kWarp];
  double m[kMomentCount];
#pragma unroll
  for (int k = 0; k < kMomentCount; ++k) m[k] = 0.0;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * kStreamThreads + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * kStreamThreads) {
    accumulate_moments(m, load_pose(states + i), weights[i], px, py);
  }
  store_block_moments<kStreamThreads>(m, s_red, moment_partials + static_cast<size_t>(blockIdx.x) * kMomentCount);
}

__global__ void __launch_bounds__(256) reduce_partials_kernel(const double* __restrict__ partials, uint32_t n_partials, int width, double* __restrict__ out) {
  // One block per column; fixed summation order (thread-strided, then the block tree).
  __shared__ double s_red[256 / kWarp];
  const int k = blockIdx.x;
  double v = 0.0;
  for (uint32_t r = threadIdx.x; r < n_partials; r += 256) v = v + partials[static_cast<size_t>(r) * width + k];
  const double total = block_sum<256>(v, s_red);
  if (threadIdx.x == 0) out[k] = total;
}

__global__ void __launch_bounds__(256) fill_kernel(double* __restrict__ out, uint64_t n, double value) {
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * 256) out[i] = value;
}

// ---- shard exchange ------------------------------------------------------------------------------------

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

constexpr unsigned long long kExchangeTimeoutNs = 4000000000ull;  // 4 s: a peer that has not posted by then never will

__global__ void __launch_bounds__(256) shard_exchange_kernel(ShardExchangeArgs a) {
  __shared__ unsigned long long s_u[kMaxShards];
  __shared__ double s_d[kMaxShards][kMomentCount];
  __shared__ int s_timeout;
  const int t = threadIdx.x;
  if (t == 0) s_timeout = 0;
  __syncthreads();
  if (a.post && t < a.world) {
    // my value -> entry [kind][my rank] of rank t's block
    volatile ShardMailEntry* dst = &a.peers[t]->e[a.kind][a.rank];
    if (a.kind == kExchangeWmax) {
      dst->u[0] = a.scalars->wmax_bits;
    } else if (a.kind == kExchangeTotal) {
      dst->u[0] = a.scalars->total;
    } else if (a.kind == kExchangeMoments) {
#pragma unroll
      for (int k = 0; k < kMomentCount; ++k) dst->d[k] = a.results[k];
    }
    __threadfence_system();  // the payload -- and every earlier store of this stream, e.g. the states pushed to the peers -- before the flag
    dst->seq = a.epoch;
  }
  if (a.wait) {
    if (t < a.world) {
      const volatile ShardMailEntry* src = &a.peers[a.rank]->e[a.kind][t];
      const unsigned long long t0 = global_timer_ns();
      bool ok = true;
      while (src->seq != a.epoch) {
        if (global_timer_ns() - t0 > kExchangeTimeoutNs) {
          ok = false;
          break;
        }
        __nanosleep(64);
      }
      __threadfence_system();
      if (!ok) atomicExch(&s_timeout, 1);
      s_u[t] = src->u[0];
      if (a.kind == kExchangeMoments) {
#pragma unroll
        for (int k = 0; k < kMomentCount; ++k) s_d[t][k] = src->d[k];
      }
    }
    __syncthreads();
    if (t == 0) {
      if (s_timeout) {
        a.scalars->exchange_error = 1;
        a.summary->error = 1;
      }
      if (a.kind == kExchangeWmax) {
        unsigned long long m = 0;
        for (int r = 0; r < a.world; ++r) m = s_u[r] > m ? s_u[r] : m;  // positive doubles order like their bit patterns
        a.scalars->wmax_bits = m;
        prepare_cdf_scalars(a.scalars, __longlong_as_double(static_cast<long long>(m)), a.ceil_log2_count);
        a.summary->exponent = a.scalars->exponent;
        a.summary->valid = a.scalars->valid;
      } else if (a.kind == kExchangeTotal) {
        unsigned long long total = 0;
        for (int r = 0; r < a.world; ++r) {
          a.rank_totals[r] = s_u[r];
          a.summary->rank_totals[r] = s_u[r];
          total += s_u[r];
        }
        a.summary->total = total;
        a.scalars->global_total = total;
      } else if (a.kind == kExchangeMoments) {
        for (int k = 0; k < kMomentCount; ++k) {  // rank order: the same sum on every rank
          double v = 0.0;
          for (int r = 0; r < a.world; ++r) v = v + s_d[r][k];
          a.results[k] = v;
          a.summary->moments[k] = v;
        }
      }
    }
    if (a.kind == kExchangeWmax && a.tile_state != nullptr) {
      for (uint32_t k = t; k < a.n_tiles; k += blockDim.x) a.tile_state[k] = 0;
    }
  }
}

__global__ void write_summary_kernel(const double* __restrict__ results, const Scalars* __restrict__ scalars, StepSummary* summary) {
  if (threadIdx.x < kMomentCount) summary->moments[threadIdx.x] = results[threadIdx.x];
  if (threadIdx.x == 0) {
    summary->total = scalars->total;
    summary->exponent = scalars->exponent;
    summary->valid = scalars->valid;
    summary->error = 0;
  }
  __threadfence_system();
}

int ceil_log2_u64(uint64_t n) {
  int b = 0;
  while ((uint64_t{1} << b) < n) ++b;
  return b;
}

constexpr uint32_t kStreamMaxBlocks = 148 * 8;

}  // namespace

// ---- launchers -------------------------------------------------------------------------------------

void launch_begin_step(Scalars* scalars, cudaStream_t stream) { begin_step_kernel<<<1, 1, 0, stream>>>(scalars); }

void launch_write_summary(const double* results, const Scalars* scalars, StepSummary* summary, cudaStream_t stream) {
  write_summary_kernel<<<1, 32, 0, stream>>>(results, scalars, summary);
}
void launch_shard_exchange(const ShardExchangeArgs& args, cudaStream_t stream) { shard_exchange_kernel<<<1, 256, 0, stream>>>(args); }
int ceil_log2_count(uint64_t n) { return ceil_log2_u64(n); }

void launch_initialize_normal(Pose2* states, double* weights, uint64_t n, const double mean[3], const double transform[9], uint64_t seed,
                              uint64_t first_index, cudaStream_t stream) {
  if (n == 0) return;
  NormalInit p;
  for (int i = 0; i < 3; ++i) p.mean[i] = mean[i];
  for (int i = 0; i < 9; ++i) p.t[i] = transform[i];
  initialize_normal_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(states, weights, n, p, seed, first_index);
}

void launch_initialize_uniform(Pose2* states, double* weights, uint64_t n, const uint32_t* free_cells, uint64_t n_free, int grid_width,
                               double grid_resolution, const Pose2& grid_origin, uint64_t seed, uint64_t first_index, cudaStream_t stream) {
  if (n == 0) return;
  const FreeSpace fs{free_cells, n_free, grid_width, grid_resolution, grid_origin};
  initialize_uniform_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(states, weights, n, fs, seed, first_index);
}

void launch_propagate(Pose2* states, uint64_t n, bool do_propagate, const MotionSampling& sampling, uint64_t seed, uint32_t step,
                      uint64_t first_index, Schedule* sched, cudaStream_t stream) {
  if (n == 0) return;
  if (sched != nullptr) schedule_reset_kernel<<<1, 1, 0, stream>>>(sched);
  propagate_kernel<<<static_cast<unsigned>((n + kPrThreads - 1) / kPrThreads), kPrThreads, 0, stream>>>(states, n, do_propagate ? 1 : 0, sampling,
                                                                                                      seed, step, first_index, sched);
}

void launch_propagate_binned(Pose2* states, uint64_t n, const MotionSampling& sampling, uint64_t seed, uint32_t step, uint64_t first_index,
                             const Schedule& grid, uint2* bin_rank, uint32_t* counters, Schedule* /*sched*/, cudaStream_t stream) {
  if (n == 0) return;
  propagate_binned_kernel<<<static_cast<unsigned>((n + kPrThreads - 1) / kPrThreads), kPrThreads, 0, stream>>>(
      states, n, sampling, seed, step, first_index, grid, bin_rank, counters);
}

void launch_begin_fused_step(Scalars* scalars, unsigned long long* tile_state, uint32_t n_tiles, Schedule* sched, uint32_t* counters,
                             uint32_t n_counters, unsigned long long* sched_tiles, uint32_t n_sched_tiles, const void* prefetch,
                             uint64_t prefetch_bytes, cudaStream_t stream) {
  const StepReset r{scalars, tile_state, n_tiles, sched, counters, (n_counters + 3u) & ~3u, sched_tiles, n_sched_tiles,
                    static_cast<const char*>(prefetch), prefetch != nullptr ? prefetch_bytes / 128 : 0};
  const uint64_t work = std::max<uint64_t>(std::max(n_tiles, counters != nullptr ? r.n_counters / 4 : 0u), r.prefetch_lines / 8);
  const unsigned blocks = static_cast<unsigned>(std::max<uint64_t>(1, std::min<uint64_t>((work + 255u) / 256u, 148u * 4u)));
  begin_fused_step_kernel<<<blocks, 256, 0, stream>>>(r);
}

uint32_t schedule_max_bins() { return kMaxBins; }
uint32_t schedule_tile_count() { return (kMaxBins + kScanTile - 1) / kScanTile; }

void launch_build_schedule(const Pose2* states, uint64_t n, Schedule* sched, uint32_t* bins, uint32_t* counters, uint32_t* perm,
                           unsigned long long* tile_state, double mean_range, double min_bin, double per_bin, double x_split, bool equal_mass,
                           cudaStream_t stream) {
  if (n == 0) return;
  const unsigned blocks = static_cast<unsigned>((n + 255) / 256);
  cudaMemsetAsync(counters, 0, kMaxBins * sizeof(uint32_t), stream);
  cudaMemsetAsync(tile_state, 0, schedule_tile_count() * sizeof(unsigned long long), stream);
  schedule_params_kernel<<<1, 1, 0, stream>>>(sched, n, mean_range, min_bin, per_bin, x_split, equal_mass);
  schedule_histogram_kernel<<<blocks, 256, 0, stream>>>(states, n, sched, bins, counters);
  scan_u32_kernel<<<schedule_tile_count(), kScanThreads, 0, stream>>>(counters, counters, kMaxBins, &sched->tile_ticket, tile_state, nullptr);
  schedule_scatter_kernel<<<blocks, 256, 0, stream>>>(bins, n, counters, perm);
}

void launch_finish_schedule(const uint2* bin_rank, uint64_t n, uint32_t n_bins, Schedule* sched, uint32_t* counters, uint32_t* perm,
                            unsigned long long* tile_state, cudaStream_t stream) {
  if (n == 0) return;
  // (Scanning the counters in the tail of propagate_binned_kernel -- its last block -- was tried: one SM reading 250 KB
  // in dependent 16-byte steps takes 40 us; sixteen look-back tiles take 8.)
  const unsigned blocks = static_cast<unsigned>((n + 256 * kPlaceItems - 1) / (256 * kPlaceItems));
  const uint32_t tiles = (n_bins + kScanTile - 1) / kScanTile;
  scan_u32_kernel<<<tiles, kScanThreads, 0, stream>>>(counters, counters, n_bins, &sched->tile_ticket, tile_state, nullptr);
  schedule_place_kernel<<<blocks, 256, 0, stream>>>(bin_rank, n, counters, perm);
}

bool scatter_resample_enabled() {
  static const bool enabled = [] {
    const char* v = std::getenv("BB200_SCATTER_RESAMPLE");  // development knob
    return v == nullptr || std::atoi(v) != 0;
  }();
  return enabled;
}

int sm_count() {
  static thread_local int cached_device = -1, cached = 0;
  int device = 0;
  cudaGetDevice(&device);
  if (device != cached_device) {
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, device);
    cached_device = device;
  }
  return cached > 0 ? cached : 148;
}

void launch_reweight_lfm(const Pose2* states, double* weights, uint64_t n, const uint32_t* perm, const FieldView& field,
                         const double* points_xy_device, const double* points_xy_host, uint32_t n_points, double points_radius, Scalars* scalars,
                         cudaStream_t stream) {
  if (n == 0) return;
  const unsigned blocks = static_cast<unsigned>((n + kRwThreads - 1) / kRwThreads);
  const size_t smem = static_cast<size_t>(n_points < kChunkBeams ? n_points : kChunkBeams) * sizeof(double2);
  const double2* points = reinterpret_cast<const double2*>(points_xy_device);
  if (field.use_fixed) {
    static thread_local ScanParam scan;  // launch parameters are copied at launch time
    if (points_xy_host != nullptr && n_points <= kParamBeams) {
      std::memcpy(scan.p, points_xy_host, static_cast<size_t>(n_points) * sizeof(double2));
      const unsigned ctas_needed = static_cast<unsigned>((n + kRwThreads - 1) / kRwThreads);
      const unsigned persistent = std::min<unsigned>(static_cast<unsigned>(sm_count()) * kRwBlocksPerSm, ctas_needed);
      reweight_lfm_fixed_param_kernel<<<persistent, kRwThreads, 0, stream>>>(states, weights, n, perm, field, n_points, points_radius, scalars, scan);
    } else {
      reweight_lfm_fixed_kernel<<<blocks, kRwThreads, smem, stream>>>(states, weights, n, perm, field, points, n_points, points_radius, scalars);
    }
  } else if (field.use_tiled) {
    reweight_lfm_kernel<true><<<blocks, kRwThreads, smem, stream>>>(states, weights, n, perm, field, points, n_points, points_radius, scalars);
  } else {
    reweight_lfm_kernel<false><<<blocks, kRwThreads, smem, stream>>>(states, weights, n, perm, field, points, n_points, points_radius, scalars);
  }
}

uint32_t beam_eta_entries(double beam_max_range, double resolution) {
  const double cells = beam_max_range / resolution + 2.0;
  const double entries = cells * cells + 2.0;
  return (entries > 0.0 && entries < 8.0e6) ? static_cast<uint32_t>(entries) : 0u;  // <= 128 MB; beyond that: per-beam evaluation
}

void launch_beam_eta_table(const BeamParams& params, double resolution, double2* table, uint32_t entries, cudaStream_t stream) {
  if (entries == 0) return;
  beam_eta_table_kernel<<<(entries + 255) / 256, 256, 0, stream>>>(params, resolution, table, entries);
}

uint64_t beam_hit_words(uint64_t particles, uint32_t n_points) {
  const uint64_t stride = (particles + 31) / 32 * 32;
  return stride * n_points;
}

void launch_reweight_beam_two_pass(const Pose2* states, double* weights, uint64_t n, const uint32_t* perm, const OccupancyView& grid,
                                   const BeamParams& params, const double* points_xy_device, uint32_t n_points, uint32_t* hits,
                                   uint64_t pass_particles, Scalars* scalars, cudaStream_t stream) {
  if (n == 0 || n_points == 0 || pass_particles == 0) return;
  const double2* points = reinterpret_cast<const double2*>(points_xy_device);
  const uint64_t stride = (pass_particles + 31) / 32 * 32;
  for (uint64_t base = 0; base < n; base += pass_particles) {
    const uint64_t count = std::min<uint64_t>(pass_particles, n - base);
    const unsigned blocks = static_cast<unsigned>((count + kWalkThreads - 1) / kWalkThreads);
    beam_walk_kernel<<<blocks, kWalkThreads, 0, stream>>>(states, n, base, count, perm, grid, params.beam_max_range, points, n_points, hits, stride);
    beam_mixture_kernel<<<blocks, kMixThreads, 0, stream>>>(states, weights, n, base, count, perm, grid, params, points, n_points, hits, stride, scalars);
  }
}

void launch_reweight_beam(const Pose2* states, double* weights, uint64_t n, const uint32_t* perm, const OccupancyView& grid,
                          const BeamParams& params, const double* points_xy_device, uint32_t n_points, Scalars* scalars, cudaStream_t stream) {
  if (n == 0) return;
  const unsigned blocks = static_cast<unsigned>((n + kBeamThreads - 1) / kBeamThreads);
  reweight_beam_kernel<<<blocks, kBeamThreads, 0, stream>>>(states, weights, n, perm, grid, params,
                                                            reinterpret_cast<const double2*>(points_xy_device), n_points, scalars);
}

void launch_max_weight(const double* weights, uint64_t n, Scalars* scalars, cudaStream_t stream) {
  if (n == 0) return;
  const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((n + 511) / 512, kStreamMaxBlocks));
  max_weight_kernel<<<blocks, 512, 0, stream>>>(weights, n, scalars);
}

uint32_t scan_tile_count(uint64_t n) { return static_cast<uint32_t>((n + kQsTile - 1) / kQsTile); }  // the smaller of the two tile sizes

void launch_prepare_cdf(Scalars* scalars, double host_wmax, uint64_t global_count, unsigned long long* tile_state, uint32_t n_tiles,
                        cudaStream_t stream) {
  const unsigned blocks = std::max(1u, std::min((n_tiles + 255u) / 256u, 64u));
  prepare_cdf_kernel<<<blocks, 256, 0, stream>>>(scalars, host_wmax, ceil_log2_u64(global_count), tile_state, n_tiles);
}

void launch_quantize_scan(const double* weights, uint64_t n, unsigned long long* cdf, Scalars* scalars, unsigned long long* tile_state,
                          cudaStream_t stream, bool derive_exponent, uint64_t global_count) {
  if (n == 0) return;
  if (n > (4u << 20)) {
    constexpr uint32_t tile = kQsThreads * kQsItemsLarge;
    quantize_scan_kernel<kQsItemsLarge><<<static_cast<unsigned>((n + tile - 1) / tile), kQsThreads, 0, stream>>>(
        weights, n, cdf, scalars, tile_state, derive_exponent ? 1 : 0, ceil_log2_u64(global_count));
  } else {
    quantize_scan_kernel<kQsItemsSmall><<<static_cast<unsigned>((n + kQsTile - 1) / kQsTile), kQsThreads, 0, stream>>>(
        weights, n, cdf, scalars, tile_state, derive_exponent ? 1 : 0, ceil_log2_u64(global_count));
  }
}

void launch_normalize(double* weights, uint64_t n, const Scalars* scalars, unsigned long long global_total, double* partials,
                      uint32_t* n_partials, cudaStream_t stream) {
  const unsigned blocks = static_cast<unsigned>(std::max<uint64_t>(1, std::min<uint64_t>((n + kStreamThreads - 1) / kStreamThreads, kStreamMaxBlocks)));
  *n_partials = blocks;
  normalize_kernel<<<blocks, kStreamThreads, 0, stream>>>(weights, n, scalars, global_total, partials);
}

void launch_kld_clear(unsigned long long* keys, unsigned int* vals, uint64_t table_size, cudaStream_t stream) {
  cudaMemsetAsync(keys, 0xFF, table_size * sizeof(unsigned long long), stream);
  cudaMemsetAsync(vals, 0xFF, table_size * sizeof(unsigned int), stream);
}

void launch_kld_chunk(const KldArgs& a, unsigned long long* keys, unsigned int* vals, uint64_t table_size, uint32_t* flags, uint32_t* exclusive,
                      Scalars* scalars, unsigned long long* tile_state, cudaStream_t stream) {
  if (a.n == 0) return;
  const unsigned blocks = static_cast<unsigned>((a.n + 255) / 256);
  const uint32_t tiles = static_cast<uint32_t>((a.n + kScanTile - 1) / kScanTile);
  kld_reset_kernel<<<1, 1, 0, stream>>>(scalars);
  cudaMemsetAsync(tile_state, 0, static_cast<size_t>(tiles) * sizeof(unsigned long long), stream);
  kld_insert_kernel<<<blocks, 256, 0, stream>>>(a.hashes, a.n, a.slot_base, keys, vals, table_size - 1);
  kld_flag_kernel<<<blocks, 256, 0, stream>>>(a.hashes, a.n, a.slot_base, keys, vals, table_size - 1, flags);
  scan_u32_kernel<<<tiles, kScanThreads, 0, stream>>>(flags, exclusive, static_cast<uint32_t>(a.n), &scalars->pad[0], tile_state, &scalars->pad[1]);
  kld_check_kernel<<<blocks, 256, 0, stream>>>(flags, exclusive, a.n, a.slot_base, a.k_before, a.min_particles, 2 * a.epsilon, a.z, scalars);
}

void launch_scan_u32(const uint32_t* in, uint32_t* out, uint32_t n, unsigned long long* ticket, unsigned long long* tile_state,
                     unsigned long long* total_out, cudaStream_t stream) {
  if (n == 0) return;
  const uint32_t tiles = (n + kScanTile - 1) / kScanTile;
  cudaMemsetAsync(ticket, 0, sizeof(unsigned long long), stream);
  cudaMemsetAsync(tile_state, 0, static_cast<size_t>(tiles) * sizeof(unsigned long long), stream);
  scan_u32_kernel<<<tiles, kScanThreads, 0, stream>>>(in, out, n, ticket, tile_state, total_out);
}

uint32_t resample_block_count(uint64_t slots) {
  return static_cast<uint32_t>(std::max<uint64_t>(1, std::min<uint64_t>((slots + kRsThreads - 1) / kRsThreads, 148 * 16)));
}

uint32_t launch_resample(const ResampleArgs& args, Scalars* scalars, double* moment_partials, cudaStream_t stream) {
  // The whole set on one GPU with the systematic comb and nothing per slot to draw: scatter form.
  // (Sharded with peer memory and device-side totals: the same, every copy stored into its owner's buffer.)
  const bool plain = args.scheme == 1 && args.random_state_probability <= 0.0 && args.hashes == nullptr && args.span_filter == 0 &&
                     args.peer_hash_count == 0 && args.window_begin == 0 &&
                     args.global_total == 0 && args.cdf_offset == 0 && args.slot_first == 0 && scatter_resample_enabled();
  const bool scatter = plain && ((args.peer_count == 0 && args.rank_totals == nullptr && args.slot_count == args.total_slots) ||
                                 (args.peer_count > 0 && args.rank_totals != nullptr));
  if (scatter) {
    // one pass over the input particles; a few particles per thread amortise the block reduction of the moments
    const uint32_t per_sm = BB200_RS_BLOCKS;  // resident CTAs at the kernel's register count
    const uint32_t blocks = static_cast<uint32_t>(std::max<uint64_t>(1, std::min<uint64_t>((args.n_in + kRsThreads - 1) / kRsThreads, 148 * per_sm)));
    resample_scatter_kernel<<<blocks, kRsThreads, 0, stream>>>(args, scalars, moment_partials);
    return blocks;
  }
  const uint32_t blocks = resample_block_count(args.slot_count);
  resample_kernel<<<blocks, kRsThreads, 0, stream>>>(args, scalars, moment_partials);
  return blocks;
}

uint32_t moments_block_count(uint64_t n) {
  return static_cast<uint32_t>(std::max<uint64_t>(1, std::min<uint64_t>((n + kStreamThreads - 1) / kStreamThreads, kStreamMaxBlocks)));
}

void launch_moments(const Pose2* states, const double* weights, uint64_t n, double pivot_x, double pivot_y, double* moment_partials,
                    cudaStream_t stream) {
  moments_kernel<<<moments_block_count(n), kStreamThreads, 0, stream>>>(states, weights, n, pivot_x, pivot_y, moment_partials);
}

void launch_fill(double* out, uint64_t n, double value, cudaStream_t stream) {
  if (n == 0) return;
  fill_kernel<<<static_cast<unsigned>(std::min<uint64_t>((n + 255) / 256, kStreamMaxBlocks)), 256, 0, stream>>>(out, n, value);
}

void launch_reduce_partials(const double* partials, uint32_t n_partials, int width, double* out, cudaStream_t stream) {
  reduce_partials_kernel<<<width, 256, 0, stream>>>(partials, n_partials, width, out);
}

}  // namespace bb200
