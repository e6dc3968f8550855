// Kernel launch interface of the B200 MCL backend (see kernels.cu for the kernels themselves).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "se2_math.cuh"

namespace bb200 {

/// Device view of the likelihood-field lookup table (LFM / LFM-prob).
struct FieldView {
  // f(pz) per cell (f = pz^3 or log pz), row-major, followed by one spare cell holding
  // unknown_value (index width*height) that out-of-grid end points read.
  const double* table;
  // The same values in 4x4-cell tiles (one 128-byte line per tile, row-major inside), padded to whole
  // tiles with unknown_value, plus the spare cell at tiles_x*tiles_y*16.  Index: tiled_index().
  const double* tiled;
  int tiles_x;
  int use_tiled;          // which of the two layouts the kernel gathers from
  uint32_t spare_index;   // index of the spare cell in the selected layout
  int width, height;
  double inv_resolution;  // 1. / resolution  (regular_grid.hpp:76)
  double unknown_value;   // f(float(1/max_laser_distance)) for out-of-grid end points
  double init;            // transform_reduce init: 1.0 (LFM) or 0.0 (prob)
  int exp_epilogue;       // prob model: weight = exp(sum)
  Pose2 world_to_field;   // grid.origin().inverse()
  // Bordered 4x4-tile layout for the fixed-point lookup kernel (reweight_lfm_fixed_kernel): the grid
  // with a one-cell border of unknown_value, cell (xi, yi) stored at padded coordinates
  // (px, py) = (xi + 1, yi + 1), index bordered_index(px, py, border_kx); 2^border_kx tiles per row.
  const double* bordered;
  int border_kx;
  uint32_t border_pitch;  // 2^border_kx
  uint32_t border_x_max;  // 4 (width + 1) + 3: largest 4 * padded x with its two fraction bits
  uint32_t border_y_max;  // height + 1: largest padded y
  // `bordered` minus fixed_index_bias(border_kx) elements: what the fixed-point kernel indexes with the unclamped, still
  // biased words of end points that are known to land on the map.  Null when the biased indices of this map would wrap
  // around 2^32 (every such end point then takes the clamped lookup).
  const double* bordered_biased;
  int use_fixed;          // launch the fixed-point kernel (map small enough for 16.16 cell coordinates)
};

/// Offset of padded cell (px, py) in the bordered tile layout.
BB_HD uint32_t bordered_index(uint32_t px, uint32_t py, int kx) {
  return (((py >> 2) << (kx + 4)) | ((px >> 2) << 4)) | ((px & 3u) << 2) | (py & 3u);  // 4 x 4 tiles, y fastest inside a tile
}
/// Largest padded grid side the fixed-point kernel accepts (cell coordinates below 2^13).
constexpr int kFixedMaxSide = 8000;
/// High words of the fixed-point x and y sums with the cell bits zero (see kernels.cu); their low 19 bits are clear.
constexpr uint32_t kFixedBiasX = 0x41180000u, kFixedBiasY = 0x41380000u;
/// What the bordered index gains, modulo 2^32, when the fixed-point kernel feeds the raw high words to its index arithmetic
/// instead of the words minus the biases: (kFixedBiasY * row pitch + kFixedBiasX) mod 2^32, row pitch 4 * 2^kx.
BB_HD uint32_t fixed_index_bias(int kx) { return kFixedBiasY * (4u << kx) + kFixedBiasX; }

/// Device view of the occupancy grid (beam model).
struct OccupancyView {
  const int8_t* cells;
  const uint8_t* free_distance;  // Chebyshev distance to the nearest non-free / outside cell (map_host.hpp)
  const uint8_t* free_padded;    // the same with one border cell of zeros all round, 2^pad_shift bytes per row (two-pass walk)
  int pad_shift;
  int width, height;
  double resolution, inv_resolution;
  Pose2 world_to_grid;  // grid.origin().inverse()
};

struct BeamParams {
  double z_hit, z_short, z_max, z_rand, sigma_hit, lambda_short, beam_max_range;
  // Normalisers of the hit and short terms (beam_model.hpp:128-141) tabulated over the squared cell
  // distance d2 = dx^2 + dy^2 of the ray's end cell: eta[d2] = {eta_hit, eta_short} at z_mean =
  // sqrt(d2) * resolution; the last entry is z_mean = beam_max_range (miss, or a hit beyond the range).
  // Null: evaluate them per beam (two erf and one exp more).
  const double2* eta;
  uint32_t eta_entries;
};
/// Entries of the normaliser table, 0 when the range/resolution ratio makes it too large to be worth it.
uint32_t beam_eta_entries(double beam_max_range, double resolution);
void launch_beam_eta_table(const BeamParams& params, double resolution, double2* table, uint32_t entries, cudaStream_t stream);

/// Mirrors bb200_motion_sampling (include/beluga_b200.h).
struct MotionSampling {
  int model;
  double mean[3];
  double stddev[3];
  double first_c, first_s;
};

/// Per-filter device scalars (zeroed at creation; the per-step fields are reset by launch_begin_step).
struct Scalars {
  unsigned long long wmax_bits;   // bit pattern of the largest weight (positive doubles order like integers)
  unsigned long long tile_ticket; // decoupled look-back: next tile id
  unsigned long long total;       // fixed-point total of the local CDF
  int exponent;                   // q = floor(w * 2^exponent)
  int valid;                      // 0 when no positive finite weight exists
  unsigned long long kld_cutoff;  // first slot (1-based count) at which the KLD condition fails
  unsigned long long pad[3];
  unsigned long long work_ticket;  // persistent reweight kernel: next 32-particle task (rewound by the last warp out)
  unsigned long long work_done;    // warps that have left that kernel
  int exchange_error;              // sticky: a shard exchange timed out
  unsigned int blocks_done;        // resample kernels: blocks that have stored their moment partials (the last one reduces them)
  unsigned long long global_total; // sharded filters: sum of the ranks' totals (set by the totals exchange)
};

// ---- sharded filters: exchange of step scalars through peer memory ---------------------------------------
// One filter split over several GPUs needs three tiny exchanges per step (largest weight -> common fixed-point
// exponent; fixed-point totals -> CDF offsets; raw moments -> estimate, which is also the barrier after which the
// peers' state stores are visible).  Every rank owns a ShardMail block in its device memory; rank r writes its value
// into entry [kind][r] of EVERY rank's block (peer stores over NVLink, or plain stores when the shards share a
// device) followed by a system-scope fence and the step's sequence number; a reader spins on the sequence numbers
// of its own block.  No NCCL, no host round trip: a post/wait costs one single-CTA kernel.
constexpr int kMaxShards = 8;
enum ShardExchangeKind : int { kExchangeWmax = 0, kExchangeTotal = 1, kExchangeMoments = 2, kExchangeKld = 3, kExchangeKinds = 4 };
struct alignas(128) ShardMailEntry {
  unsigned long long seq;   // written last, after a system-scope fence
  unsigned long long u[3];
  double d[12];
};
struct ShardMail {
  ShardMailEntry e[kExchangeKinds][kMaxShards];
};
/// What the host reads back at the end of a fused step (one copy).
struct StepSummary {
  double moments[9];              // raw moments of the new particle set (all ranks)
  unsigned long long total;       // global fixed-point total of the CDF
  unsigned long long rank_totals[kMaxShards];
  int exponent;
  int valid;                      // 0: no positive finite weight anywhere
  int error;                      // 1: a peer never posted (bounded spin ran out)
  int seq;                        // completion ticket of the step that wrote this block (written last; the host may poll it)
};
struct ShardExchangeArgs {
  int kind, post, wait;
  int rank, world;
  unsigned long long epoch;
  ShardMail* peers[kMaxShards];  // every rank's mail block (peers[rank] is this rank's own)
  struct Scalars* scalars;
  double* results;               // kMomentCount local sums in, global sums out (kExchangeMoments)
  StepSummary* summary;          // device copy, filled as the exchanges complete
  unsigned long long* rank_totals;  // device array of kMaxShards totals (kExchangeTotal)
  // kExchangeWmax also prepares the CDF build (what prepare_cdf does on one GPU)
  int ceil_log2_count;
  unsigned long long* tile_state;
  uint32_t n_tiles;
};
void launch_shard_exchange(const ShardExchangeArgs& args, cudaStream_t stream);
/// results (9 moments) + the CDF scalars -> the host's StepSummary block (pinned memory).
void launch_write_summary(const double* results, const struct Scalars* scalars, StepSummary* summary, cudaStream_t stream);
int ceil_log2_count(uint64_t n);

constexpr int kMomentCount = 9;  // sum w, sum w^2, sum w c, sum w s, sum w dx, sum w dy, sum w dx^2, sum w dx dy, sum w dy^2

// ---- launchers (all asynchronous on `stream`) ---------------------------------------------------

void launch_begin_step(Scalars* scalars, cudaStream_t stream);

void launch_initialize_normal(Pose2* states, double* weights, uint64_t n, const double mean[3], const double transform[9],
                              uint64_t seed, uint64_t first_index, cudaStream_t stream);

/// initialize_from_map: n states uniform over the free cells (centroids, global frame), yaw uniform, weights 1.
void launch_initialize_uniform(Pose2* states, double* weights, uint64_t n, const uint32_t* free_cells, uint64_t n_free, int grid_width,
                               double grid_resolution, const Pose2& grid_origin, uint64_t seed, uint64_t first_index, cudaStream_t stream);

/// Offset of cell (xi, yi) in the tiled table.
BB_HD size_t tiled_index(int xi, int yi, int tiles_x) {
  const unsigned x = static_cast<unsigned>(xi), y = static_cast<unsigned>(yi);
  const size_t tile = static_cast<size_t>(y >> 2) * static_cast<size_t>(tiles_x) + (x >> 2);
  return tile * 16 + (((y & 3u) << 2) | (x & 3u));
}

/// Execution schedule state: cloud moments and the pose-bin grid derived from them.
struct Schedule {
  double sums[6];  // sum cos, sin, x, y, x^2, y^2 of the propagated cloud (device-built schedules only)
  unsigned long long tile_ticket;
  double c0, s0;            // mean heading (unit complex)
  double x0, y0, half_u;    // lower corner of the box; half extent of the heading coordinate u = 2 tan(dtheta / 2)
  double scale_t, scale_x, scale_y;
  double mx, my;            // cloud mean (equal-mass bins)
  float kt, kx, ky;         // equal-mass bins: 1.702 / sigma of u, x, y (logistic stand-in for the normal CDF)
  uint32_t equal_mass;      // bins of equal expected particle count instead of equal size
  uint32_t nt, nx, ny;
  uint32_t n_bins;
};
constexpr uint32_t kScheduleMaxBins = 1u << 19;  // 4 particles per bin up to 2M particles per shard, coarser bins beyond

/// The pose-bin grid for a cloud with mean resultant (cbar, sbar), mean position (mx, my) and position variances
/// (vx, vy), about `per_bin` particles per bin.  Runs on the device (moments of the propagated cloud) or on the host
/// (moments predicted from the last estimate and the motion means).  The schedule only decides WHICH THREAD handles a
/// particle, never a result.
///
/// equal_mass = false: bins of equal physical edge in (range * heading, x, y) covering +-3 sigma.
/// equal_mass = true:  every coordinate goes through a sigmoid CDF (logistic with the normal's spread) first, so that bins
///   hold the same EXPECTED number of particles: small where the cloud is dense, large in the tails.  A uniform grid over
///   a normal cloud puts most particles into bins 13x over-full, and 32 schedule neighbours then span a whole bin.
/// x_split: bins are x_split times thinner in x than in the other two coordinates; x is the fastest index of the bin
///   order, so a warp (32 neighbours of the schedule) covers x_split bins of a row: a cube, whatever the bin boundaries.
BB_HD void schedule_from_moments(Schedule& g, double cbar, double sbar, double mx, double my, double vx, double vy, double n,
                                 double mean_range, double min_bin, double per_bin, double x_split = 1.0, bool equal_mass = false) {
  const double r = sqrt(cbar * cbar + sbar * sbar);
  const double pi = 3.14159265358979323846;
  double c0 = 1.0, s0 = 0.0, sigma_theta = pi;
  if (r > 1e-9) {
    c0 = cbar / r;
    s0 = sbar / r;
    sigma_theta = r < 1.0 ? sqrt(-2.0 * log(r)) : 0.0;
  }
  const double half_theta = fmin(2.0, fmax(3.0 * sigma_theta, 1e-4));  // beyond +-2 rad: the edge bins
  const double half_u = 2.0 * tan(0.5 * half_theta);
  const double half_x = fmax(3.0 * sqrt(fmax(vx, 0.0)), min_bin), half_y = fmax(3.0 * sqrt(fmax(vy, 0.0)), min_bin);
  const double lever = fmax(mean_range, 1.0);
  x_split = fmin(fmax(x_split, 1.0), 32.0);
  // Extents in physical units.  Equal-size bins tile the +-3 sigma box; equal-mass bins tile the unit cube of CDF values,
  // where a bin at the centre of the cloud is sigma / (density of the sigmoid at 0 = 1.702 / 4) / count wide.
  const double centre = equal_mass ? 1.0 / (3.0 * 0.4255) : 2.0;
  const double ext_t = centre * half_u * lever, ext_x = centre * half_x, ext_y = centre * half_y;
  double q = cbrt(x_split * ext_t * ext_x * ext_y / fmax(n / per_bin, 1.0));  // edge of x_split bins side by side
  q = fmax(q, min_bin);
  uint32_t nt, nx, ny;
  for (;;) {
    nt = static_cast<uint32_t>(fmin(fmax(ceil(ext_t / q), 1.0), 65536.0));
    nx = static_cast<uint32_t>(fmin(fmax(ceil(x_split * ext_x / q), 1.0), 65536.0));
    ny = static_cast<uint32_t>(fmin(fmax(ceil(ext_y / q), 1.0), 65536.0));
    if (static_cast<uint64_t>(nt) * nx * ny <= kScheduleMaxBins) break;
    q = q * 1.3;
  }
  g.c0 = c0, g.s0 = s0;
  g.x0 = mx - half_x, g.y0 = my - half_y, g.half_u = half_u;
  g.scale_t = static_cast<double>(nt) / (2.0 * half_u);
  g.scale_x = static_cast<double>(nx) / (2.0 * half_x);
  g.scale_y = static_cast<double>(ny) / (2.0 * half_y);
  g.mx = mx, g.my = my;
  g.kt = static_cast<float>(1.702 * 3.0 / half_u), g.kx = static_cast<float>(1.702 * 3.0 / half_x), g.ky = static_cast<float>(1.702 * 3.0 / half_y);
  g.equal_mass = equal_mass ? 1u : 0u;
  g.nt = nt, g.nx = nx, g.ny = ny;
  g.n_bins = nt * nx * ny;
}

/// propagate (or only accumulate the cloud moments when do_propagate is false).  sched may be null.
void launch_propagate(Pose2* states, uint64_t n, bool do_propagate, const MotionSampling& sampling, uint64_t seed, uint32_t step,
                      uint64_t first_index, Schedule* sched, cudaStream_t stream);
/// propagate with the pose-bin histogram fused in: `grid` was predicted on the host, every particle's bin goes to
/// bin_rank[] = {bin, arrival rank inside the bin} and into the counters (zeroed by launch_begin_fused_step).  launch_finish_schedule turns them into perm.
void launch_propagate_binned(Pose2* states, uint64_t n, const MotionSampling& sampling, uint64_t seed, uint32_t step, uint64_t first_index,
                             const Schedule& grid, uint2* bin_rank, uint32_t* counters, Schedule* sched, cudaStream_t stream);
void launch_finish_schedule(const uint2* bin_rank, uint64_t n, uint32_t n_bins, Schedule* sched, uint32_t* counters, uint32_t* perm,
                            unsigned long long* tile_state, cudaStream_t stream);
/// One launch resetting the per-step scalars, the CDF scan state and (counters != nullptr) the schedule's counters / scan state;
/// `prefetch` (nullable) is streamed into L2 (the table the reweight kernel gathers from).
void launch_begin_fused_step(Scalars* scalars, unsigned long long* tile_state, uint32_t n_tiles, Schedule* sched, uint32_t* counters,
                             uint32_t n_counters, unsigned long long* sched_tiles, uint32_t n_sched_tiles, const void* prefetch,
                             uint64_t prefetch_bytes, cudaStream_t stream);
uint32_t schedule_max_bins();
uint32_t schedule_tile_count();
/// Counting sort of the particle indices over pose bins -> perm (needs launch_propagate's moments).
void launch_build_schedule(const Pose2* states, uint64_t n, Schedule* sched, uint32_t* bins, uint32_t* counters, uint32_t* perm,
                           unsigned long long* tile_state, double mean_range, double min_bin, double per_bin, double x_split, bool equal_mass,
                           cudaStream_t stream);
/// reweight with the likelihood-field table in schedule order (perm may be null) | block max.
/// points_xy_host (optional): the same points in host memory; scans of up to 1920 points then travel as
/// kernel parameters (constant bank) instead of being staged through shared memory.
void launch_reweight_lfm(const Pose2* states, double* weights, uint64_t n, const uint32_t* perm, const FieldView& field,
                         const double* points_xy_device, const double* points_xy_host, uint32_t n_points, double points_radius, Scalars* scalars,
                         cudaStream_t stream);
/// reweight with the beam model (Bresenham ray casting) in schedule order | block max.
void launch_reweight_beam(const Pose2* states, double* weights, uint64_t n, const uint32_t* perm, const OccupancyView& grid,
                          const BeamParams& params, const double* points_xy_device, uint32_t n_points, Scalars* scalars, cudaStream_t stream);

/// The same in two passes over `pass_particles` particles at a time: ray walk -> one 32-bit hit word per (beam, particle)
/// in `hits` (beam_hit_words(pass_particles, n_points) words), then the mixture.  Grids up to 65535 cells a side.
uint64_t beam_hit_words(uint64_t particles, uint32_t n_points);
void launch_reweight_beam_two_pass(const Pose2* states, double* weights, uint64_t n, const uint32_t* perm, const OccupancyView& grid,
                                   const BeamParams& params, const double* points_xy_device, uint32_t n_points, uint32_t* hits,
                                   uint64_t pass_particles, Scalars* scalars, cudaStream_t stream);

/// Largest weight only (when propagate/reweight ran separately or particles were set by hand).
void launch_max_weight(const double* weights, uint64_t n, Scalars* scalars, cudaStream_t stream);

/// Sets scalars->exponent from wmax (device value when host_wmax < 0) and resets the scan state.
void launch_prepare_cdf(Scalars* scalars, double host_wmax, uint64_t global_count, unsigned long long* tile_state, uint32_t n_tiles,
                        cudaStream_t stream);
/// Exclusive prefix sum of n u32 values (in and out may alias); *total_out (optional) receives the sum.
/// `ticket` is one device word, `tile_state` holds scan_tile_count(n) words; both are reset here.
void launch_scan_u32(const uint32_t* in, uint32_t* out, uint32_t n, unsigned long long* ticket, unsigned long long* tile_state,
                     unsigned long long* total_out, cudaStream_t stream);
uint32_t scan_tile_count(uint64_t n);
/// Fixed-point quantisation + single-pass inclusive scan (decoupled look-back).
/// derive_exponent: take the exponent from scalars->wmax_bits inside the kernel (needs the scan state already reset,
/// launch_begin_fused_step or the shard exchange) instead of scalars->exponent set by launch_prepare_cdf.
void launch_quantize_scan(const double* weights, uint64_t n, unsigned long long* cdf, Scalars* scalars, unsigned long long* tile_state,
                          cudaStream_t stream, bool derive_exponent = false, uint64_t global_count = 1);

/// w /= S (S = global_total * 2^-exponent) and per-block partial sums of (w/S)^2.
/// global_total == ~0: the sharded filter's total on the device (scalars->global_total).
void launch_normalize(double* weights, uint64_t n, const Scalars* scalars, unsigned long long global_total, double* partials,
                      uint32_t* n_partials, cudaStream_t stream);

/// Optional tail of a resample launch: the last block sums the per-block moment rows into `results` (device) and,
/// when `summary` is set, writes the step's StepSummary there (pinned host memory on a single GPU).
struct StepTail {
  int enabled;
  double* results;
  StepSummary* summary;
  int seq;  // != 0: stored to summary->seq after everything else (system-scope fence in between)
};

struct ResampleArgs {
  const Pose2* states_in;
  const unsigned long long* cdf;
  uint64_t n_in;
  Pose2* states_out;
  double* weights_out;
  long long* ancestors;  // nullable
  unsigned long long* hashes;  // nullable (KLD)
  uint64_t slot_first;    // global index of local output slot 0
  uint64_t slot_count;    // local output slots
  uint64_t total_slots;   // M: the comb of systematic resampling spans all global slots
  unsigned long long global_total;  // fixed-point total over all ranks (0: scalars->total, single shard)
  unsigned long long cdf_offset;    // sum of the totals of the lower ranks: local position = t - cdf_offset
  // Fused redistribution over NVLink peer memory: when peer_count > 0 the state of global slot j is
  // stored straight into the staging buffer of the rank that owns the slot (peer_out[j / peer_shard]
  // at j % peer_shard) instead of states_out[local].
  int peer_count;
  uint64_t peer_shard;
  Pose2* peer_out[8];
  // Sharded multinomial sampling: the launch walks ALL global slots and keeps those whose draw lands in
  // this rank's span of the global CDF [cdf_offset, cdf_offset + local total); an injected random state
  // is produced by the rank that owns the slot ([owner_first, owner_first + owner_count)).
  int span_filter;
  uint64_t owner_first, owner_count;
  // Device-side bookkeeping of a sharded resample: when rank_totals is set (the all-gathered fixed-point
  // totals of the ranks, in device memory) the kernel derives the global total, this rank's CDF offset and --
  // for the systematic comb -- its slot range itself, so the host does not have to read the totals back first.
  const unsigned long long* rank_totals;
  int rank, world;
  // KLD on shards.  window: produce only the slots in [window_begin, window_end) (0, 0: all).  peer_hashes: counting
  // pass -- write the candidate's spatial hash to entry [slot] of every rank's hash array instead of storing the state.
  // inject_mod: recovery injection of slot j is handled by rank j % inject_mod (0: by the slot's owner).
  uint64_t window_begin, window_end;
  int peer_hash_count;
  unsigned long long* peer_hashes[8];
  int inject_mod;
  int scheme;
  uint64_t seed;
  uint32_t step;
  double random_state_probability;
  const uint32_t* free_cells;
  uint64_t n_free;
  int grid_width;
  double grid_resolution;
  Pose2 grid_origin;
  double hash_resolution[3];
  double pivot_x, pivot_y;
  StepTail tail;
};
uint32_t resample_block_count(uint64_t slots);
/// sample | random_intersperse | (hash) | assign, plus per-block raw moments of the new set.  Returns the number of
/// blocks launched (= rows of moment_partials written).
uint32_t launch_resample(const ResampleArgs& args, Scalars* scalars, double* moment_partials, cudaStream_t stream);

/// Per-block raw weighted moments of (states, weights).
uint32_t moments_block_count(uint64_t n);
void launch_moments(const Pose2* states, const double* weights, uint64_t n, double pivot_x, double pivot_y, double* moment_partials,
                    cudaStream_t stream);
void launch_fill(double* out, uint64_t n, double value, cudaStream_t stream);
/// Sums `n_partials` rows of kMomentCount doubles in a fixed order into out[kMomentCount].
void launch_reduce_partials(const double* partials, uint32_t n_partials, int width, double* out, cudaStream_t stream);

/// KLD (views/take_while_kld.hpp:72-137) over one chunk of candidate slots [slot_base, slot_base + n):
/// device hash set of buckets -> first-occurrence flags -> prefix count -> first failing count in
/// scalars->kld_cutoff (1-based; ~0 when every count in the chunk passes); scalars->pad[1] receives
/// the number of new buckets of the chunk.
struct KldArgs {
  const unsigned long long* hashes;  // spatial hash of each candidate of the chunk
  uint64_t n;
  uint64_t slot_base;     // slots accepted before this chunk
  uint64_t k_before;      // distinct buckets before this chunk
  uint64_t min_particles;
  double epsilon, z;
};
void launch_kld_clear(unsigned long long* keys, unsigned int* vals, uint64_t table_size, cudaStream_t stream);
void launch_kld_chunk(const KldArgs& args, unsigned long long* keys, unsigned int* vals, uint64_t table_size, uint32_t* flags,
                      uint32_t* exclusive, Scalars* scalars, unsigned long long* tile_state, cudaStream_t stream);

}  // namespace bb200
