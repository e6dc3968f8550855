#include "filter.hpp"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>

#include "cluster_host.hpp"
#include "map_host.hpp"

namespace bb200 {

namespace {

template <class T>
cudaError_t dev_alloc(T** p, size_t count) {
  return cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(T));
}

Pose2 pose_from_array(const double* d) { return Pose2{d[0], d[1], d[2], d[3]}; }

MotionSampling to_kernel_sampling(const bb200_motion_sampling& s) {
  MotionSampling m{};
  m.model = s.model;
  for (int k = 0; k < 3; ++k) {
    m.mean[k] = s.mean[k];
    m.stddev[k] = s.stddev[k];
  }
  m.first_c = s.first_rotation[0];
  m.first_s = s.first_rotation[1];
  return m;
}

}  // namespace

bool normal_transform(const double cov[9], double transform[9], std::string* error) {
  // isApprox(transpose) of Eigen: ||C - C^T||_F^2 <= 1e-24 * ||C||_F^2
  double diff2 = 0.0, norm2 = 0.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      const double d = cov[3 * i + j] - cov[3 * j + i];
      diff2 += d * d;
      norm2 += cov[3 * i + j] * cov[3 * i + j];
    }
  if (!(diff2 <= 1e-24 * norm2)) {
    if (error) *error = "Invalid covariance matrix, it is not symmetric.";
    return false;
  }
  // Cyclic Jacobi on the symmetric 3x3; eigenvalues ascending like SelfAdjointEigenSolver.
  double a[3][3], v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) a[i][j] = cov[3 * i + j];
  for (int sweep = 0; sweep < 64; ++sweep) {
    if (a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2] == 0.0) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) {
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq;
          a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk;
          a[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = c * vkp - s * vkq;
          v[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int order[3] = {0, 1, 2};
  std::sort(order, order + 3, [&](int i, int j) { return a[i][i] < a[j][j]; });
  for (int j = 0; j < 3; ++j) {
    const double lambda = a[order[j]][order[j]];
    if (lambda < 0.0) {
      if (error) *error = "Invalid covariance matrix, it has negative eigenvalues.";
      return false;
    }
    for (int i = 0; i < 3; ++i) transform[3 * i + j] = v[i][order[j]] * std::sqrt(lambda);
  }
  return true;
}

// ---------------------------------------------------------------------------------------------------

Filter::Filter(const bb200_filter_config& config) : config_(config) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    create_status_ = fail(BB200_ERR_NO_DEVICE, "no CUDA device available (this backend has no CPU fallback)");
    return;
  }
  if (config.device < 0 || config.device >= count) {
    create_status_ = fail(BB200_ERR_INVALID_ARGUMENT, "device ordinal out of range");
    return;
  }
  if (config.capacity == 0) {
    create_status_ = fail(BB200_ERR_INVALID_ARGUMENT, "capacity must be positive");
    return;
  }
  if (config_.global_count == 0) config_.global_count = config_.capacity;
  if (const char* v = std::getenv("BB200_SCHEDULE")) schedule_enabled_ = std::atoi(v) != 0;  // development knob: 0 disables the pose-sorted schedule
  if (const char* v = std::getenv("BB200_TILED")) tiled_layout_ = std::atoi(v) != 0;         // development knob: table layout
  if (const char* v = std::getenv("BB200_PARAM_POINTS")) param_points_ = std::atoi(v) != 0;  // development knob: scan as kernel parameters
  if (const char* v = std::getenv("BB200_BEAM_ETA_TABLE")) beam_eta_table_ = std::atoi(v) != 0;  // development knob: tabulated beam normalisers
  if (const char* v = std::getenv("BB200_FIXED")) fixed_lookup_ = std::atoi(v) != 0;         // development knob: fixed-point lookup kernel
  if (const char* v = std::getenv("BB200_POLL_COMPLETION")) poll_completion_ = std::atoi(v) != 0;  // development knob: 0 = cudaStreamSynchronize
  if (const char* v = std::getenv("BB200_PREDICT_SCHEDULE")) predict_schedule_ = std::atoi(v) != 0;  // development knob: host-predicted pose bins
  if (const char* v = std::getenv("BB200_PREFETCH_TABLE")) prefetch_table_ = std::atoi(v) != 0;  // development knob: L2 prefetch of the likelihood table
  if (const char* v = std::getenv("BB200_BEAM_TWO_PASS")) beam_two_pass_ = std::atoi(v) != 0;  // development knob: walk + mixture kernels
  if (const char* v = std::getenv("BB200_PER_BIN")) schedule_per_bin_ = std::atof(v);        // development knob: particles per pose bin
  if (const char* v = std::getenv("BB200_X_SPLIT")) schedule_x_split_ = std::atof(v);        // development knob: bins per warp along x
  if (const char* v = std::getenv("BB200_EQUAL_MASS")) schedule_equal_mass_ = std::atoi(v) != 0;  // development knob: 0 = equal-size bins
  if (const char* v = std::getenv("BB200_LEVER")) schedule_lever_ = std::atof(v);            // development knob: heading lever arm / mean range
  capacity_ = config.capacity;
  first_index_ = config.first_index;
#define BB_TRY(expr)                                \
  do {                                              \
    const int st = check((expr), #expr);            \
    if (st != BB200_OK) {                           \
      create_status_ = st;                          \
      return;                                       \
    }                                               \
  } while (0)
  BB_TRY(cudaSetDevice(config.device));
  BB_TRY(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  BB_TRY(dev_alloc(&states_[0], capacity_));
  BB_TRY(dev_alloc(&states_[1], capacity_));
  BB_TRY(dev_alloc(&weights_, capacity_));
  BB_TRY(dev_alloc(&cdf_, capacity_));
  if (config.record_ancestors) BB_TRY(dev_alloc(&ancestors_, capacity_));
  BB_TRY(dev_alloc(&scalars_, 1));
  BB_TRY(cudaMallocHost(reinterpret_cast<void**>(&scalars_host_), sizeof(Scalars)));
  tile_capacity_ = scan_tile_count(capacity_) + 1;
  BB_TRY(dev_alloc(&tile_state_, tile_capacity_));
  partials_rows_ = std::max(std::max(resample_block_count(capacity_), moments_block_count(capacity_)), 148u * 8u);
  BB_TRY(dev_alloc(&partials_, static_cast<size_t>(partials_rows_) * kMomentCount));
  BB_TRY(dev_alloc(&results_, 16));
  BB_TRY(cudaMallocHost(reinterpret_cast<void**>(&results_host_), 16 * sizeof(double)));
  BB_TRY(dev_alloc(&sched_, 1));
  BB_TRY(dev_alloc(&bins_, capacity_));
  BB_TRY(dev_alloc(&bin_rank_, capacity_));
  BB_TRY(dev_alloc(&perm_, capacity_));
  BB_TRY(dev_alloc(&counters_, schedule_max_bins()));
  BB_TRY(dev_alloc(&sched_tiles_, schedule_tile_count()));
  BB_TRY(dev_alloc(&mail_, 1));  // its own allocation: exported to peer processes through CUDA IPC
  BB_TRY(dev_alloc(&shard_totals_, kMaxShards));
  BB_TRY(dev_alloc(&summary_, 1));
  BB_TRY(cudaMallocHost(reinterpret_cast<void**>(&summary_host_), sizeof(StepSummary)));
  std::memset(summary_host_, 0, sizeof(StepSummary));  // pinned allocations are recycled with their old contents (a stale completion ticket)
  BB_TRY(cudaMemsetAsync(mail_, 0, sizeof(ShardMail), stream_));
  BB_TRY(cudaMemsetAsync(summary_, 0, sizeof(StepSummary), stream_));
  BB_TRY(cudaMemsetAsync(scalars_, 0, sizeof(Scalars), stream_));
  BB_TRY(cudaStreamSynchronize(stream_));
#undef BB_TRY
  global_size_ = config_.global_count;
  created_ = true;
}

Filter::~Filter() {
  if (stream_ != nullptr) cudaStreamSynchronize(stream_);
  release_peers();
  for (auto& e : event_pool_) cudaEventDestroy(e);
  cudaFree(mail_);
  cudaFree(shard_totals_);
  cudaFree(summary_);
  cudaFreeHost(summary_host_);
  cudaFree(states_[0]);
  cudaFree(states_[1]);
  cudaFree(weights_);
  cudaFree(cdf_);
  cudaFree(ancestors_);
  cudaFree(hashes_);
  cudaFree(scalars_);
  cudaFree(sched_);
  cudaFree(bins_);
  cudaFree(bin_rank_);
  cudaFree(perm_);
  cudaFree(counters_);
  cudaFree(sched_tiles_);
  cudaFreeHost(scalars_host_);
  cudaFree(tile_state_);
  cudaFree(partials_);
  cudaFree(results_);
  cudaFreeHost(results_host_);
  cudaFree(cluster_.hashes);
  cudaFree(cluster_.keys);
  cudaFree(cluster_.first);
  cudaFree(cluster_.slot_of);
  cudaFree(cluster_.flags);
  cudaFree(cluster_.cell_of);
  cudaFree(cluster_.starts);
  cudaFree(cluster_.keys_a);
  cudaFree(cluster_.keys_b);
  cudaFree(cluster_.idx_a);
  cudaFree(cluster_.idx_b);
  cudaFree(cluster_.histogram);
  cudaFree(cluster_.tile_state);
  cudaFree(cluster_.words);
  cudaFree(cluster_.records);
  cudaFree(kld_keys_);
  cudaFree(kld_vals_);
  cudaFree(kld_flags_);
  cudaFree(kld_scan_);
  cudaFree(kld_tile_state_);
  cudaFree(kld_hashes_global_);
  cudaFree(points_);
  cudaFreeHost(points_host_);
  cudaFree(table_);
  cudaFree(tiled_);
  cudaFree(bordered_);
  cudaFree(beam_eta_);
  cudaFree(beam_hits_);
  cudaFree(free_padded_);
  cudaFree(occupancy_);
  cudaFree(free_distance_);
  cudaFree(free_cells_);
  if (stream_ != nullptr && owns_stream_) cudaStreamDestroy(stream_);
}

int Filter::fail(int status, const std::string& message) {
  error_ = message;
  return status;
}

int Filter::check(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return BB200_OK;
  return fail(BB200_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define BB_CHECK(expr)                          \
  do {                                          \
    const int st_ = check((expr), #expr);       \
    if (st_ != BB200_OK) return st_;            \
  } while (0)
#define BB_LAUNCHED_N(name, count)                          \
  do {                                                      \
    launches_ += (count);                                   \
    const int st_ = check(cudaGetLastError(), name);        \
    if (st_ != BB200_OK) return st_;                        \
  } while (0)
#define BB_LAUNCHED(name) BB_LAUNCHED_N(name, 1)

void Filter::mark(const char* name) {
  if (!timing_) return;
  if (events_used_ == event_pool_.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    event_pool_.push_back(e);
  }
  cudaEvent_t e = event_pool_[events_used_++];
  cudaEventRecord(e, stream_);
  marks_.push_back(Mark{name, e});
}

void Filter::finish_marks() {
  if (!timing_ || marks_.empty()) {
    marks_.clear();
    events_used_ = 0;
    return;
  }
  if (std::string(marks_.back().name) != "end") mark("end");
  cudaEventSynchronize(marks_.back().event);
  for (size_t i = 0; i + 1 < marks_.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, marks_[i].event, marks_[i + 1].event);
    timings_.emplace_back(marks_[i].name, ms);
  }
  marks_.clear();
  events_used_ = 0;
}

int Filter::last_timings(const char** names, float* ms, int capacity) const {
  const int n = std::min<int>(capacity, static_cast<int>(timings_.size()));
  for (int i = 0; i < n; ++i) {
    names[i] = timings_[i].first;
    ms[i] = timings_[i].second;
  }
  return static_cast<int>(timings_.size());
}

int Filter::set_stream(void* stream) {
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  if (owns_stream_ && stream_ != nullptr) cudaStreamDestroy(stream_);
  stream_ = static_cast<cudaStream_t>(stream);
  owns_stream_ = false;
  return BB200_OK;
}

int Filter::enqueue_propagate_reweight(const bb200_motion_sampling* sampling, uint32_t step, const double* points_xy, uint64_t n_points) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  if (points_xy == nullptr || sensor_ < 0) return fail(BB200_ERR_STATE, "no sensor model map set / no points");
  if (n_points > 0xffffffffull) return fail(BB200_ERR_INVALID_ARGUMENT, "too many points");
  BB_CHECK(cudaSetDevice(config_.device));
  int st = upload_points(points_xy, n_points);  // the caller synchronised at the end of the previous step
  if (st != BB200_OK) return st;
  MotionSampling s{};
  if (sampling != nullptr) s = to_kernel_sampling(*sampling);
  mark("begin_step");
  launch_begin_step(scalars_, stream_);
  BB_LAUNCHED("begin_step");
  st = enqueue_propagate_reweight(sampling != nullptr ? &s : nullptr, step, true, n_points, false);
  cdf_valid_ = false;
  cloud_known_ = false;
  return st;
}

int Filter::enqueue_build_cdf() {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  BB_CHECK(cudaSetDevice(config_.device));
  mark("prepare_cdf");
  launch_prepare_cdf(scalars_, -1.0, config_.global_count, tile_state_, scan_tile_count(n_), stream_);
  BB_LAUNCHED("prepare_cdf");
  mark("quantize_scan");
  launch_quantize_scan(weights_, n_, cdf_, scalars_, tile_state_, stream_);
  BB_LAUNCHED("quantize_scan");
  cdf_valid_ = true;
  return BB200_OK;
}

int Filter::enqueue_resample_range(const bb200_resample_opts& o, uint64_t global_total, uint64_t cdf_offset, uint64_t slot_begin, uint64_t slot_end) {
  if (!cdf_valid_) return fail(BB200_ERR_STATE, "build_cdf must run before resample_range");
  if (o.scheme != BB200_RESAMPLE_SYSTEMATIC || o.min_particles < o.max_particles)
    return fail(BB200_ERR_STATE, "range resampling supports the systematic comb without KLD (multinomial: bb200_filter_enqueue_resample_push)");
  if (o.random_state_probability > 0.0 && n_free_ == 0) return fail(BB200_ERR_STATE, "recovery injection needs a map with free cells");
  if (slot_end < slot_begin || slot_end - slot_begin > capacity_) return fail(BB200_ERR_CAPACITY, "slot range exceeds the staging buffer");
  BB_CHECK(cudaSetDevice(config_.device));
  if (slot_end > slot_begin) {
    ResampleArgs a = make_resample_args(o, 0, slot_end - slot_begin, false);
    a.slot_first = slot_begin;
    a.global_total = global_total;
    a.cdf_offset = cdf_offset;
    a.weights_out = nullptr;
    mark("resample_range");
    launch_resample(a, scalars_, partials_, stream_);
    BB_LAUNCHED("resample_range");
  }
  return BB200_OK;
}

int Filter::ipc_handles(void* out128) {
  BB_CHECK(cudaSetDevice(config_.device));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "two IPC handles are exported as 128 bytes");
  cudaIpcMemHandle_t h[2];
  BB_CHECK(cudaIpcGetMemHandle(&h[0], states_[0]));
  BB_CHECK(cudaIpcGetMemHandle(&h[1], states_[1]));
  std::memcpy(out128, h, sizeof(h));
  return BB200_OK;
}

int Filter::open_peers(int world, int rank, const void* handles) {
  if (world < 1 || world > 8 || rank < 0 || rank >= world) return fail(BB200_ERR_INVALID_ARGUMENT, "peer groups hold 1..8 ranks");
  BB_CHECK(cudaSetDevice(config_.device));
  if (peer_world_ != 0) return fail(BB200_ERR_STATE, "the peers' buffers are already mapped");
  const auto* all = static_cast<const cudaIpcMemHandle_t*>(handles);
  for (int r = 0; r < world; ++r) {
    for (int b = 0; b < 2; ++b) {
      if (r == rank) {
        peer_states_[b][r] = states_[b];
      } else {
        void* p = nullptr;
        BB_CHECK(cudaIpcOpenMemHandle(&p, all[2 * r + b], cudaIpcMemLazyEnablePeerAccess));
        peer_states_[b][r] = static_cast<Pose2*>(p);
      }
    }
  }
  peer_world_ = world;
  peer_rank_ = rank;
  peers_ipc_ = true;
  return BB200_OK;
}

void Filter::release_peers() {
  if (peers_ipc_) {  // unmap what cudaIpcOpenMemHandle mapped; local peers are plain pointers owned by their filters
    for (int r = 0; r < peer_world_; ++r) {
      if (r == peer_rank_) continue;
      for (int b = 0; b < 2; ++b)
        if (peer_states_[b][r] != nullptr) cudaIpcCloseMemHandle(peer_states_[b][r]);
      if (peer_mail_[r] != nullptr) cudaIpcCloseMemHandle(peer_mail_[r]);
      if (peer_kld_hashes_[r] != nullptr) cudaIpcCloseMemHandle(peer_kld_hashes_[r]);
    }
  }
  for (int r = 0; r < kMaxShards; ++r) {
    peer_states_[0][r] = peer_states_[1][r] = nullptr;
    peer_mail_[r] = nullptr;
    peer_kld_hashes_[r] = nullptr;
  }
  peer_world_ = 0;
  peers_ipc_ = false;
}

int Filter::leave_shards() {
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  release_peers();
  return BB200_OK;
}

int Filter::enable_shard_kld() {
  if (kld_hashes_global_ != nullptr) return BB200_OK;
  if (peer_world_ != 0) return fail(BB200_ERR_STATE, "KLD on shards must be enabled before the shards are joined");
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(dev_alloc(&kld_hashes_global_, config_.global_count));  // one spatial hash per candidate slot of the WHOLE filter
  return BB200_OK;
}

int Filter::export_shard(void* out256) {
  BB_CHECK(cudaSetDevice(config_.device));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "four IPC handles are exported as 256 bytes");
  cudaIpcMemHandle_t h[4];
  std::memset(h, 0, sizeof(h));
  BB_CHECK(cudaIpcGetMemHandle(&h[0], states_[0]));
  BB_CHECK(cudaIpcGetMemHandle(&h[1], states_[1]));
  BB_CHECK(cudaIpcGetMemHandle(&h[2], mail_));
  if (kld_hashes_global_ != nullptr) BB_CHECK(cudaIpcGetMemHandle(&h[3], kld_hashes_global_));
  std::memcpy(out256, h, sizeof(h));
  return BB200_OK;
}

int Filter::join_shards_ipc(int world, int rank, const void* handles) {
  if (world < 1 || world > kMaxShards || rank < 0 || rank >= world) return fail(BB200_ERR_INVALID_ARGUMENT, "shard groups hold 1..8 ranks");
  if (peer_world_ != 0) return fail(BB200_ERR_STATE, "the peers' buffers are already mapped");
  if (config_.first_index != static_cast<uint64_t>(rank) * capacity_ || config_.global_count != static_cast<uint64_t>(world) * capacity_)
    return fail(BB200_ERR_INVALID_ARGUMENT, "shard r of R holds the global indices [r * capacity, (r + 1) * capacity) of R * capacity particles");
  BB_CHECK(cudaSetDevice(config_.device));
  const auto* all = static_cast<const cudaIpcMemHandle_t*>(handles);
  peers_ipc_ = true;
  peer_world_ = world;
  peer_rank_ = rank;
  for (int r = 0; r < world; ++r) {
    if (r == rank) {
      peer_states_[0][r] = states_[0];
      peer_states_[1][r] = states_[1];
      peer_mail_[r] = mail_;
      peer_kld_hashes_[r] = kld_hashes_global_;
      continue;
    }
    static const cudaIpcMemHandle_t kNoHandle{};
    void* p[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int b = 0; b < 4; ++b) {
      if (b == 3 && (kld_hashes_global_ == nullptr || std::memcmp(&all[4 * r + 3], &kNoHandle, sizeof(kNoHandle)) == 0)) continue;  // no KLD on this filter
      const int st = check(cudaIpcOpenMemHandle(&p[b], all[4 * r + b], cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
      if (st != BB200_OK) {
        peer_states_[0][r] = static_cast<Pose2*>(p[0]);
        peer_states_[1][r] = static_cast<Pose2*>(p[1]);
        peer_mail_[r] = static_cast<ShardMail*>(p[2]);
        release_peers();
        return st;
      }
    }
    peer_states_[0][r] = static_cast<Pose2*>(p[0]);
    peer_states_[1][r] = static_cast<Pose2*>(p[1]);
    peer_mail_[r] = static_cast<ShardMail*>(p[2]);
    peer_kld_hashes_[r] = static_cast<unsigned long long*>(p[3]);
  }
  shard_kld_ = kld_hashes_global_ != nullptr;
  for (int r = 0; r < world; ++r) shard_kld_ = shard_kld_ && peer_kld_hashes_[r] != nullptr;
  split_posts_ = false;  // every rank has its own host thread: post and wait travel in one launch
  return BB200_OK;
}

int Filter::join_shards_local(Filter* const* filters, int world) {
  if (filters == nullptr || world < 1 || world > kMaxShards) return BB200_ERR_INVALID_ARGUMENT;
  for (int r = 0; r < world; ++r) {
    Filter* f = filters[r];
    if (f == nullptr || !f->ok()) return BB200_ERR_INVALID_ARGUMENT;
    if (f->peer_world_ != 0) return f->fail(BB200_ERR_STATE, "the peers' buffers are already mapped");
    if (f->capacity_ != filters[0]->capacity_ || f->config_.first_index != static_cast<uint64_t>(r) * f->capacity_ ||
        f->config_.global_count != static_cast<uint64_t>(world) * f->capacity_ || f->config_.seed != filters[0]->config_.seed)
      return f->fail(BB200_ERR_INVALID_ARGUMENT, "shard r of R holds the global indices [r * capacity, (r + 1) * capacity) of R * capacity particles, same seed");
  }
  for (int a = 0; a < world; ++a) {
    Filter* fa = filters[a];
    for (int b = 0; b < world; ++b) {
      const Filter* fb = filters[b];
      if (fa->config_.device != fb->config_.device) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, fa->config_.device, fb->config_.device) != cudaSuccess || !can)
          return fa->fail(BB200_ERR_CUDA, "no peer access between the devices of two shards");
        if (fa->check(cudaSetDevice(fa->config_.device), "cudaSetDevice") != BB200_OK) return BB200_ERR_CUDA;
        const cudaError_t e = cudaDeviceEnablePeerAccess(fb->config_.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fa->check(e, "cudaDeviceEnablePeerAccess");
        (void)cudaGetLastError();
      }
      fa->peer_states_[0][b] = fb->states_[0];
      fa->peer_states_[1][b] = fb->states_[1];
      fa->peer_mail_[b] = fb->mail_;
      fa->peer_kld_hashes_[b] = fb->kld_hashes_global_;
    }
    fa->shard_kld_ = true;
    for (int b = 0; b < world; ++b) fa->shard_kld_ = fa->shard_kld_ && filters[b]->kld_hashes_global_ != nullptr;
    fa->peer_world_ = world;
    fa->peer_rank_ = a;
    fa->peers_ipc_ = false;
    fa->split_posts_ = true;  // one thread enqueues all shards: every post must be enqueued before any wait that needs it
  }
  return BB200_OK;
}

int Filter::enqueue_exchange(int kind, bool post, bool wait) {
  ShardExchangeArgs a{};
  a.kind = kind;
  a.post = post ? 1 : 0;
  a.wait = wait ? 1 : 0;
  a.rank = peer_rank_;
  a.world = peer_world_;
  a.epoch = epoch_;
  for (int r = 0; r < peer_world_; ++r) a.peers[r] = peer_mail_[r];
  a.scalars = scalars_;
  a.results = results_;
  a.summary = summary_host_;  // pinned host memory: the step's results need no copy
  a.rank_totals = shard_totals_;
  a.ceil_log2_count = ceil_log2_count(config_.global_count);
  a.tile_state = tile_state_;
  a.n_tiles = scan_tile_count(n_);
  launch_shard_exchange(a, stream_);
  BB_LAUNCHED("shard_exchange");
  return BB200_OK;
}

int Filter::step_begin(const bb200_motion_sampling& sampling, uint32_t step, const double* points_xy, uint64_t n_points, const bb200_resample_opts& o,
                       bool resample_planned) {
  const uint64_t world = peer_world_ > 1 ? static_cast<uint64_t>(peer_world_) : 1;
  const bool kld = o.min_particles < o.max_particles;
  if (n_ == 0 && !(world > 1 && shard_kld_)) return fail(BB200_ERR_STATE, "no particles");  // a KLD-sized filter may leave a shard empty
  if (sensor_ < 0) return fail(BB200_ERR_STATE, "no sensor model map set");
  if (kld && !(world > 1 && shard_kld_)) return fail(BB200_ERR_STATE, "the fused step does not run KLD on one GPU; use resample()");
  if (n_points > 0xffffffffull) return fail(BB200_ERR_INVALID_ARGUMENT, "too many points");
  if (o.random_state_probability > 0.0 && n_free_ == 0) return fail(BB200_ERR_STATE, "recovery injection needs a map with free cells");
  if (world > 1) {
    if ((!shard_kld_ && n_ != capacity_) || n_ > capacity_ || o.max_particles != world * capacity_)
      return fail(BB200_ERR_STATE, "a sharded filter keeps `capacity` particles on every rank (fewer only under KLD)");
  } else if (o.max_particles == 0 || o.max_particles > capacity_) {
    return fail(BB200_ERR_CAPACITY, "max_particles exceeds the filter capacity");
  }
  BB_CHECK(cudaSetDevice(config_.device));
  const int st = upload_points(points_xy, n_points);
  if (st != BB200_OK) return st;
  if (world > 1 && peer_mail_[0] == nullptr) return fail(BB200_ERR_STATE, "shards joined without mail blocks (legacy open_peers): use join_shards");
  step_ = StepContext{};
  summary_host_->error = 0;
  step_.active = true;
  step_.sampling = to_kernel_sampling(sampling);
  step_.step = step;
  step_.n_points = n_points;
  step_.opts = o;
  step_.resample_planned = resample_planned;
  return BB200_OK;
}

void Filter::step_abort() { step_.active = false; }

int Filter::step_phase(int phase) {
  if (!step_.active) return fail(BB200_ERR_STATE, "step_begin must run first");
  BB_CHECK(cudaSetDevice(config_.device));
  const bool sharded = peer_world_ > 1;
  const bb200_resample_opts& o = step_.opts;
  int st = BB200_OK;
  switch (phase) {
    case kPhaseReweight: {
      mark("begin_step");
      {
        const bool scheduled = schedule_enabled_ && n_ >= kScheduleMinParticles;
        const bool warm = prefetch_table_ && sensor_ != BB200_SENSOR_BEAM && field_.use_fixed && bordered_bytes_ <= (96ull << 20);
        launch_begin_fused_step(scalars_, tile_state_, scan_tile_count(n_), sched_, scheduled ? counters_ : nullptr, schedule_max_bins(), sched_tiles_,
                                schedule_tile_count(), warm ? bordered_ : nullptr, bordered_bytes_, stream_);
        BB_LAUNCHED("begin_step");
        st = enqueue_propagate_reweight(&step_.sampling, step_.step, true, step_.n_points, scheduled);
      }
      if (st != BB200_OK) return st;
      if (sharded) {
        ++epoch_;  // one sequence number per batch of exchanges
        if (split_posts_) {
          mark("exchange");
          st = enqueue_exchange(kExchangeWmax, true, false);
        }
      }
      return st;
    }
    case kPhaseCdf: {
      if (sharded) {
        mark("exchange_wmax");
        st = enqueue_exchange(kExchangeWmax, !split_posts_, true);  // global largest weight -> exponent; resets the scan state
        if (st != BB200_OK) return st;
      }
      mark("quantize_scan");
      // one GPU: the exponent comes from the shard's own largest weight inside the kernel (scan state reset by begin_step);
      // sharded: the exchange above has set the common exponent and reset the scan state
      launch_quantize_scan(weights_, n_, cdf_, scalars_, tile_state_, stream_, !sharded, config_.global_count);
      BB_LAUNCHED("quantize_scan");
      if (sharded) {
        if (step_.resample_planned) {  // the CDF holds what sampling needs; every new particle weighs 1 (overlaps the wait for the peers' totals)
          mark("fill_weights");
          launch_fill(weights_, capacity_, 1.0, stream_);
          BB_LAUNCHED("fill_weights");
          step_.weights_filled = true;
        }
        if (split_posts_) {
          mark("exchange");
          st = enqueue_exchange(kExchangeTotal, true, false);
        }
      }
      return st;
    }
    case kPhaseResample: {
      if (step_.resampled) return fail(BB200_ERR_STATE, "this step has already resampled");
      ResampleArgs a;
      if (sharded) {
        if (!step_.totals_exchanged) {
          mark("exchange_total");
          st = enqueue_exchange(kExchangeTotal, !split_posts_, true);  // every rank's fixed-point total -> CDF offsets
          if (st != BB200_OK) return st;
          step_.totals_exchanged = true;
        }
        const bool systematic = o.scheme == BB200_RESAMPLE_SYSTEMATIC;
        const uint64_t accepted = step_.kld_accepted;  // KLD on shards: the count take_while_kld settled on (0: fixed size)
        const uint64_t slots = accepted != 0 ? accepted : o.max_particles;
        a = make_resample_args(o, 0, systematic ? capacity_ : slots, false);
        a.slot_first = 0;
        a.weights_out = nullptr;
        a.ancestors = nullptr;
        a.peer_count = peer_world_;
        a.peer_shard = accepted != 0 ? (accepted + static_cast<uint64_t>(peer_world_) - 1) / static_cast<uint64_t>(peer_world_) : capacity_;
        a.rank_totals = shard_totals_;
        a.rank = peer_rank_;
        a.world = peer_world_;
        if (accepted != 0) {  // the comb still spans max_particles slots; only [0, accepted) are kept
          a.window_begin = 0;
          a.window_end = accepted;
          a.inject_mod = peer_world_;
        }
        if (!systematic) {  // draws are independent: walk all global slots, keep those landing in this rank's CDF span
          a.span_filter = 1;
          a.owner_first = first_index_;
          a.owner_count = capacity_;
        }
        for (int r = 0; r < peer_world_; ++r) a.peer_out[r] = peer_states_[cur_ ^ 1][r];
        if (!step_.weights_filled) {
          mark("fill_weights");
          launch_fill(weights_, capacity_, 1.0, stream_);  // the CDF holds what sampling needs; every new particle weighs 1
          BB_LAUNCHED("fill_weights");
          step_.weights_filled = true;
        }
        mark("resample_push");
      } else {
        a = make_resample_args(o, 0, o.max_particles, false);
        mark("resample");
      }
      // the last block sums the moments (one GPU: straight into pinned host memory, with the step's completion ticket)
      step_.poll_seq = 0;
      if (!sharded && poll_completion_ && !timing_) {
        step_seq_ = step_seq_ == 0x7fffffff ? 1 : step_seq_ + 1;
        step_.poll_seq = step_seq_;
        summary_host_->seq = 0;  // nothing of this filter is in flight: the previous step was seen to end
      }
      a.tail = StepTail{1, results_, sharded ? nullptr : summary_host_, step_.poll_seq};
      step_.partial_rows = launch_resample(a, scalars_, partials_, stream_);
      BB_LAUNCHED("resample");
      step_.resampled = true;
      if (sharded && split_posts_) {
        mark("exchange");
        st = enqueue_exchange(kExchangeMoments, true, false);
      }
      return st;
    }
    case kPhaseFinish: {
      if (sharded) {
        mark("exchange_moments");
        st = enqueue_exchange(kExchangeMoments, !split_posts_, true);  // also the barrier: the peers' stores into this rank's buffer are complete
        if (st != BB200_OK) return st;
      } else if (!step_.resampled) {  // kPhaseNormalize left the moments in results_: hand them to the host block
        mark("readback");
        launch_write_summary(results_, scalars_, summary_host_, stream_);
        BB_LAUNCHED("write_summary");
      }
      mark("end");
      return BB200_OK;
    }
    case kPhaseNormalize: {
      if (step_.normalized) return fail(BB200_ERR_STATE, "the weights of this step are already normalised");
      if (sharded) {
        mark("exchange");
        st = enqueue_exchange(kExchangeTotal, !split_posts_, true);
        if (st != BB200_OK) return st;
        step_.totals_exchanged = true;
      }
      uint32_t rows = 0;
      mark("normalize");
      launch_normalize(weights_, n_, scalars_, sharded ? ~0ull : 0ull, partials_, &rows, stream_);  // actions/normalize.hpp:82
      BB_LAUNCHED("normalize");
      mark("moments");
      launch_moments(states_[cur_], weights_, n_, pivot_[0], pivot_[1], partials_, stream_);
      BB_LAUNCHED("moments");
      launch_reduce_partials(partials_, moments_block_count(n_), kMomentCount, results_, stream_);
      BB_LAUNCHED("reduce_partials");
      step_.normalized = true;
      if (sharded && split_posts_) {
        mark("exchange");
        st = enqueue_exchange(kExchangeMoments, true, false);
      }
      return st;
    }
    default:
      return fail(BB200_ERR_INVALID_ARGUMENT, "unknown step phase");
  }
}

int Filter::kld_sharded_candidates(uint64_t begin, uint64_t end) {
  if (!step_.active || !shard_kld_ || peer_world_ < 2) return fail(BB200_ERR_STATE, "KLD on shards: no step in progress on a KLD-enabled shard group");
  if (!step_.totals_exchanged) return fail(BB200_ERR_STATE, "KLD on shards: the totals exchange must run first");
  if (end <= begin || end > config_.global_count) return fail(BB200_ERR_INVALID_ARGUMENT, "KLD on shards: bad slot window");
  BB_CHECK(cudaSetDevice(config_.device));
  const bb200_resample_opts& o = step_.opts;
  if (kld_keys_ == nullptr) {  // the counting pass runs over ALL slots on every rank: tables sized for the whole filter
    const uint64_t n = config_.global_count;
    BB_CHECK(dev_alloc(&kld_flags_, n));
    BB_CHECK(dev_alloc(&kld_scan_, n));
    kld_table_size_ = 2;
    while (kld_table_size_ < 2 * n) kld_table_size_ <<= 1;
    BB_CHECK(dev_alloc(&kld_keys_, kld_table_size_));
    BB_CHECK(dev_alloc(&kld_vals_, kld_table_size_));
    BB_CHECK(dev_alloc(&kld_tile_state_, static_cast<size_t>(scan_tile_count(n)) + 1));
  }
  if (begin == 0) {
    mark("kld");
    launch_kld_clear(kld_keys_, kld_vals_, kld_table_size_, stream_);
  }
  const bool systematic = o.scheme == BB200_RESAMPLE_SYSTEMATIC;
  ResampleArgs a = make_resample_args(o, 0, std::min<uint64_t>(end - begin, capacity_), false);
  a.states_out = nullptr;
  a.weights_out = nullptr;
  a.ancestors = nullptr;
  a.rank_totals = shard_totals_;
  a.rank = peer_rank_;
  a.world = peer_world_;
  a.window_begin = begin;
  a.window_end = end;
  a.peer_hash_count = peer_world_;
  for (int r = 0; r < peer_world_; ++r) a.peer_hashes[r] = peer_kld_hashes_[r];
  a.inject_mod = peer_world_;
  a.slot_first = 0;
  if (!systematic) {
    a.span_filter = 1;
    a.slot_first = begin;
    a.slot_count = end - begin;
  }
  mark("kld_candidates");
  launch_resample(a, scalars_, partials_, stream_);
  BB_LAUNCHED("kld_candidates");
  ++epoch_;
  if (split_posts_) return enqueue_exchange(kExchangeKld, true, false);
  return BB200_OK;
}

int Filter::kld_sharded_count(uint64_t begin, uint64_t end, uint64_t k_before) {
  if (!step_.active || !shard_kld_) return fail(BB200_ERR_STATE, "KLD on shards: no step in progress");
  BB_CHECK(cudaSetDevice(config_.device));
  const bb200_resample_opts& o = step_.opts;
  mark("exchange_kld");
  const int st = enqueue_exchange(kExchangeKld, !split_posts_, true);  // every rank's hashes of this window have arrived
  if (st != BB200_OK) return st;
  mark("kld");
  KldArgs k{kld_hashes_global_ + begin, end - begin, begin, k_before, o.min_particles, o.kld_epsilon, o.kld_z};
  launch_kld_chunk(k, kld_keys_, kld_vals_, kld_table_size_, kld_flags_, kld_scan_, scalars_, kld_tile_state_, stream_);
  BB_LAUNCHED_N("kld", 5);
  BB_CHECK(cudaMemcpyAsync(scalars_host_, scalars_, sizeof(Scalars), cudaMemcpyDeviceToHost, stream_));
  return BB200_OK;
}

int Filter::kld_sharded_read(uint64_t* cutoff, uint64_t* new_buckets) {
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  if (scalars_host_->exchange_error != 0) return fail(BB200_ERR_STATE, "shard exchange timed out during the KLD count");
  *cutoff = scalars_host_->kld_cutoff;
  *new_buckets = scalars_host_->pad[1];
  return BB200_OK;
}

int Filter::step_totals(uint64_t* rank_totals, int* exponent) {
  if (!step_.active || peer_world_ < 2) return fail(BB200_ERR_STATE, "no sharded step in progress");
  BB_CHECK(cudaSetDevice(config_.device));
  if (!step_.totals_exchanged) {
    mark("exchange_total");
    const int st = enqueue_exchange(kExchangeTotal, !split_posts_, true);
    if (st != BB200_OK) return st;
    step_.totals_exchanged = true;
  }
  if (rank_totals == nullptr) return BB200_OK;  // enqueue only
  BB_CHECK(cudaStreamSynchronize(stream_));
  if (summary_host_->error != 0) return fail(BB200_ERR_STATE, "shard exchange timed out");
  for (int r = 0; r < peer_world_; ++r) rank_totals[r] = summary_host_->rank_totals[r];
  if (exponent != nullptr) *exponent = summary_host_->exponent;
  return BB200_OK;
}

void Filter::step_set_kld_accepted(uint64_t accepted) { step_.kld_accepted = accepted; }

int Filter::step_end(bb200_estimate* est, double* weight_sum, uint64_t* new_size, double* sum_sq) {
  if (!step_.active) return fail(BB200_ERR_STATE, "step_begin must run first");
  BB_CHECK(cudaSetDevice(config_.device));
  bool done = false;
  if (step_.poll_seq != 0 && step_.resampled) {
    // The resample kernel's last block stored the summary to pinned memory and then the step's ticket: spinning on that
    // word sees the end of the step a few microseconds before a stream synchronisation returns.  Everything later on this
    // stream is ordered behind the kernel anyway.  The stream is queried now and then so that a failed launch cannot hang us.
    const volatile int* seq = &summary_host_->seq;
    for (uint32_t spins = 1; !done; ++spins) {
      if (*seq == step_.poll_seq) {
        done = true;
      } else if ((spins & 0x3fffu) == 0) {
        const cudaError_t q = cudaStreamQuery(stream_);
        if (q == cudaSuccess) break;  // finished: the ticket is there (or the plain path below reports what went wrong)
        if (q != cudaErrorNotReady) break;
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
  }
  if (!done) BB_CHECK(cudaStreamSynchronize(stream_));
  step_.poll_seq = 0;
  finish_marks();
  const bool sharded = peer_world_ > 1;
  if (summary_host_->error != 0) {
    step_.active = false;
    return fail(BB200_ERR_STATE, "shard exchange timed out: a peer rank never posted its value for this step");
  }
  const double* moments = summary_host_->moments;
  step_.total = summary_host_->total;
  step_.exponent = summary_host_->exponent;
  weights_valid_ = summary_host_->valid != 0;
  if (step_.resampled) {
    cur_ ^= 1;
    n_ = sharded ? capacity_ : step_.opts.max_particles;
    if (sharded && step_.kld_accepted != 0) {  // the new set of `accepted` particles in equal contiguous shards
      const uint64_t shard = (step_.kld_accepted + static_cast<uint64_t>(peer_world_) - 1) / static_cast<uint64_t>(peer_world_);
      const uint64_t begin = std::min<uint64_t>(static_cast<uint64_t>(peer_rank_) * shard, step_.kld_accepted);
      n_ = std::min<uint64_t>(shard, step_.kld_accepted - begin);
      first_index_ = static_cast<uint64_t>(peer_rank_) * shard;
    } else if (sharded) {
      first_index_ = config_.first_index;
    }
    ancestors_n_ = n_;
    cdf_valid_ = false;
    step_.active = false;
  } else {
    cdf_valid_ = true;  // kPhaseResample may still follow (selective resampling)
    ++epoch_;           // ... as a new batch of exchanges
  }
  if (new_size != nullptr) *new_size = !sharded ? n_ : (step_.resampled && step_.kld_accepted != 0 ? step_.kld_accepted : global_size_);
  if (sharded && step_.resampled) global_size_ = step_.kld_accepted != 0 ? step_.kld_accepted : config_.global_count;
  if (weight_sum != nullptr) *weight_sum = std::ldexp(static_cast<double>(step_.total), -step_.exponent);
  if (sum_sq != nullptr) *sum_sq = moments[1];
  if (!weights_valid_) error_ = "no positive finite weight (uniform CDF substituted)";
  bb200_estimate local{};
  if (est == nullptr) est = &local;
  estimate_from_moments(moments, est);
  pivot_[0] = est->mean[2];
  pivot_[1] = est->mean[3];
  cloud_ = *est;
  cloud_known_ = step_.resampled;  // unit weights: the estimate describes the raw cloud, the next step can predict its pose bins
  return BB200_OK;
}

int Filter::enqueue_resample_push(const bb200_resample_opts& o, uint64_t global_total, uint64_t cdf_offset, uint64_t slot_begin, uint64_t slot_end,
                                  uint64_t shard, const double pivot[2]) {
  if (peer_world_ == 0) return fail(BB200_ERR_STATE, "open_peers must run before resample_push");
  if (!cdf_valid_) return fail(BB200_ERR_STATE, "build_cdf must run before resample_push");
  if (o.min_particles < o.max_particles) return fail(BB200_ERR_STATE, "sharded resampling does not support KLD");
  if (o.random_state_probability > 0.0 && n_free_ == 0) return fail(BB200_ERR_STATE, "recovery injection needs a map with free cells");
  if (o.scheme != BB200_RESAMPLE_SYSTEMATIC && (slot_begin != 0 || slot_end != o.max_particles))
    return fail(BB200_ERR_INVALID_ARGUMENT, "multinomial push walks all global slots: pass [0, max_particles)");
  BB_CHECK(cudaSetDevice(config_.device));
  ResampleArgs a = make_resample_args(o, 0, slot_end - slot_begin, false);
  a.slot_first = slot_begin;
  if (o.scheme != BB200_RESAMPLE_SYSTEMATIC) {  // draws are independent: every rank filters the global slots by its CDF span
    a.span_filter = 1;
    a.owner_first = first_index_;
    a.owner_count = shard;
  }
  a.global_total = global_total;
  a.cdf_offset = cdf_offset;
  a.weights_out = nullptr;
  a.ancestors = nullptr;
  a.peer_count = peer_world_;
  a.peer_shard = shard;
  a.pivot_x = pivot[0];
  a.pivot_y = pivot[1];
  for (int r = 0; r < peer_world_; ++r) a.peer_out[r] = peer_states_[cur_ ^ 1][r];
  mark("resample_push");
  // slot_count may be 0 (a shard without weight): the kernel still writes its (zero) moment partials.
  pushed_blocks_ = launch_resample(a, scalars_, partials_, stream_);
  BB_LAUNCHED("resample_push");
  return BB200_OK;
}

int Filter::enqueue_resample_push_device(const bb200_resample_opts& o, const uint64_t* rank_totals_device, int rank, int world, uint64_t shard,
                                         const double pivot[2]) {
  if (peer_world_ == 0) return fail(BB200_ERR_STATE, "open_peers must run before resample_push");
  if (!cdf_valid_) return fail(BB200_ERR_STATE, "build_cdf must run before resample_push");
  if (o.min_particles < o.max_particles) return fail(BB200_ERR_STATE, "sharded resampling does not support KLD");
  if (o.random_state_probability > 0.0 && n_free_ == 0) return fail(BB200_ERR_STATE, "recovery injection needs a map with free cells");
  if (rank_totals_device == nullptr || world != peer_world_ || rank < 0 || rank >= world) return fail(BB200_ERR_INVALID_ARGUMENT, "rank totals / rank / world");
  BB_CHECK(cudaSetDevice(config_.device));
  // Systematic: the kernel derives this rank's slot range from the totals; the grid is sized for a shard and strides.
  // Multinomial: all global slots, filtered by this rank's span.
  const bool systematic = o.scheme == BB200_RESAMPLE_SYSTEMATIC;
  ResampleArgs a = make_resample_args(o, 0, systematic ? shard : o.max_particles, false);
  a.slot_first = 0;
  a.weights_out = nullptr;
  a.ancestors = nullptr;
  a.peer_count = peer_world_;
  a.peer_shard = shard;
  a.pivot_x = pivot[0];
  a.pivot_y = pivot[1];
  a.rank_totals = reinterpret_cast<const unsigned long long*>(rank_totals_device);
  a.rank = rank;
  a.world = world;
  if (!systematic) {
    a.span_filter = 1;
    a.owner_first = first_index_;
    a.owner_count = shard;
  }
  for (int r = 0; r < peer_world_; ++r) a.peer_out[r] = peer_states_[cur_ ^ 1][r];
  mark("resample_push");
  pushed_blocks_ = launch_resample(a, scalars_, partials_, stream_);  // a.slot_count only sizes the grid here
  BB_LAUNCHED("resample_push");
  return BB200_OK;
}

int Filter::enqueue_reduce_moments() {
  BB_CHECK(cudaSetDevice(config_.device));
  launch_reduce_partials(partials_, pushed_blocks_, kMomentCount, results_, stream_);
  BB_LAUNCHED("reduce_partials");
  return BB200_OK;
}

int Filter::enqueue_flip_adopt(uint64_t n) {
  cur_ ^= 1;  // the staging buffer, filled by the peers, becomes the particle set
  return enqueue_adopt(n);
}

int Filter::enqueue_adopt(uint64_t n) {
  if (n > capacity_) return fail(BB200_ERR_CAPACITY, "more particles than the filter capacity");
  cloud_known_ = false;
  BB_CHECK(cudaSetDevice(config_.device));
  n_ = n;
  cdf_valid_ = false;
  mark("fill_weights");
  launch_fill(weights_, n, 1.0, stream_);
  BB_LAUNCHED("fill_weights");
  return BB200_OK;
}

int Filter::enqueue_moments(const double pivot[2]) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  BB_CHECK(cudaSetDevice(config_.device));
  mark("moments");
  launch_moments(states_[cur_], weights_, n_, pivot[0], pivot[1], partials_, stream_);
  BB_LAUNCHED("moments");
  launch_reduce_partials(partials_, moments_block_count(n_), kMomentCount, results_, stream_);
  BB_LAUNCHED("reduce_partials");
  return BB200_OK;
}

int Filter::synchronize() {
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  finish_marks();
  return BB200_OK;
}

int Filter::device_pointer(int which, void** ptr, uint64_t* bytes) {
  switch (which) {
    case 0: *ptr = states_[cur_]; *bytes = capacity_ * sizeof(Pose2); return BB200_OK;
    case 1: *ptr = weights_; *bytes = capacity_ * sizeof(double); return BB200_OK;
    case 2: *ptr = cdf_; *bytes = capacity_ * sizeof(unsigned long long); return BB200_OK;
    case 3: *ptr = states_[cur_ ^ 1]; *bytes = capacity_ * sizeof(Pose2); return BB200_OK;
    case 4: *ptr = scalars_; *bytes = sizeof(Scalars); return BB200_OK;
    case 5: *ptr = results_; *bytes = 16 * sizeof(double); return BB200_OK;
    default: return fail(BB200_ERR_INVALID_ARGUMENT, "unknown device pointer id");
  }
}

// ---- maps -----------------------------------------------------------------------------------------

int Filter::set_likelihood_field_map(const bb200_likelihood_field_param& p, const bb200_occupancy_grid& g, bool prob) {
  if (g.cells == nullptr || g.width <= 0 || g.height <= 0 || !(g.resolution > 0.0)) return fail(BB200_ERR_INVALID_ARGUMENT, "invalid occupancy grid");
  if (!(p.sigma_hit > 0.0) || !(p.max_laser_distance > 0.0)) return fail(BB200_ERR_INVALID_ARGUMENT, "invalid likelihood field parameters");
  BB_CHECK(cudaSetDevice(config_.device));
  field_host_ = make_likelihood_field(p, g);
  const size_t count = field_host_.size();
  // Per-cell f(pz) in double: pz^3 (likelihood_field_model.hpp:84-89) or log pz (prob model :84-86).
  if (count + 64 >= (1ull << 32)) return fail(BB200_ERR_CAPACITY, "map too large for 32-bit cell indices");
  std::vector<double> table(count + 1);
  auto f = [prob](float pzf) {
    const double pz = static_cast<double>(pzf);
    return prob ? std::log(pz) : pz * pz * pz;
  };
  for (size_t i = 0; i < count; ++i) table[i] = f(field_host_[i]);
  table[count] = f(static_cast<float>(1. / p.max_laser_distance));  // spare cell for out-of-grid end points
  BB_CHECK(cudaStreamSynchronize(stream_));
  cudaFree(table_);
  table_ = nullptr;
  BB_CHECK(dev_alloc(&table_, count + 1));
  BB_CHECK(cudaMemcpyAsync(table_, table.data(), (count + 1) * sizeof(double), cudaMemcpyHostToDevice, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  // Tiled copy (4x4-cell tiles, Z-order inside) for the beam-parallel lookup kernel.
  const int tiles_x = (g.width + 3) / 4, tiles_y = (g.height + 3) / 4;
  const double unknown = f(static_cast<float>(1. / p.max_laser_distance));
  if (static_cast<size_t>(tiles_x) * tiles_y * 16 + 64 >= (1ull << 32)) return fail(BB200_ERR_CAPACITY, "map too large for 32-bit cell indices");
  std::vector<double> tiled(static_cast<size_t>(tiles_x) * tiles_y * 16 + 1, unknown);
  for (int yi = 0; yi < g.height; ++yi)
    for (int xi = 0; xi < g.width; ++xi) tiled[tiled_index(xi, yi, tiles_x)] = table[static_cast<size_t>(yi) * g.width + xi];
  cudaFree(tiled_);
  tiled_ = nullptr;
  BB_CHECK(dev_alloc(&tiled_, tiled.size()));
  BB_CHECK(cudaMemcpyAsync(tiled_, tiled.data(), tiled.size() * sizeof(double), cudaMemcpyHostToDevice, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  // Bordered tile layout for the fixed-point kernel.
  field_.use_fixed = 0;
  field_.bordered = nullptr;
  field_.bordered_biased = nullptr;
  cudaFree(bordered_);
  bordered_ = nullptr;
  if (fixed_lookup_ && g.width + 2 <= kFixedMaxSide && g.height + 2 <= kFixedMaxSide) {
    int kx = 0;
    while ((1 << kx) < (g.width + 2 + 3) / 4) ++kx;
    const size_t tile_rows = static_cast<size_t>((g.height + 2 + 3) / 4);
    std::vector<double> bordered((tile_rows << (kx + 4)), unknown);
    for (int yi = 0; yi < g.height; ++yi)
      for (int xi = 0; xi < g.width; ++xi)
        bordered[bordered_index(static_cast<uint32_t>(xi + 1), static_cast<uint32_t>(yi + 1), kx)] = table[static_cast<size_t>(yi) * g.width + xi];
    BB_CHECK(dev_alloc(&bordered_, bordered.size()));
    bordered_bytes_ = bordered.size() * sizeof(double);
    BB_CHECK(cudaMemcpyAsync(bordered_, bordered.data(), bordered.size() * sizeof(double), cudaMemcpyHostToDevice, stream_));
    BB_CHECK(cudaStreamSynchronize(stream_));
    field_.bordered = bordered_;
    field_.border_kx = kx;
    field_.border_pitch = 1u << kx;
    field_.border_x_max = static_cast<uint32_t>(4 * (g.width + 1) + 3);
    field_.border_y_max = static_cast<uint32_t>(g.height + 1);
    // The kernel adds the biased 32-bit index to this base, so every index of the table plus the bias must stay below 2^32.
    const uint32_t bias = fixed_index_bias(kx);
    if (static_cast<uint64_t>(bias) + bordered.size() <= (1ull << 32))
      field_.bordered_biased = reinterpret_cast<const double*>(reinterpret_cast<uintptr_t>(bordered_) - static_cast<uintptr_t>(bias) * sizeof(double));
    field_.use_fixed = 1;
  }
  field_.tiled = tiled_;
  field_.tiles_x = tiles_x;
  field_.use_tiled = tiled_layout_ ? 1 : 0;
  field_.spare_index = static_cast<uint32_t>(tiled_layout_ ? tiled.size() - 1 : count);

  field_.table = table_;
  field_.width = g.width;
  field_.height = g.height;
  field_.inv_resolution = 1. / g.resolution;
  field_.unknown_value = f(static_cast<float>(1. / p.max_laser_distance));
  field_.init = prob ? 0.0 : 1.0;
  field_.exp_epilogue = prob ? 1 : 0;
  field_.world_to_field = pose_inverse(pose_from_array(g.origin));
  sensor_ = prob ? BB200_SENSOR_LIKELIHOOD_FIELD_PROB : BB200_SENSOR_LIKELIHOOD_FIELD;

  // Free cells for the recovery random-state generator.
  const std::vector<uint32_t> free = make_free_cells(g);
  cudaFree(free_cells_);
  free_cells_ = nullptr;
  n_free_ = free.size();
  BB_CHECK(dev_alloc(&free_cells_, free.size()));
  if (!free.empty()) BB_CHECK(cudaMemcpy(free_cells_, free.data(), free.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  grid_width_ = g.width;
  grid_height_ = g.height;
  grid_resolution_ = g.resolution;
  grid_origin_ = pose_from_array(g.origin);
  return BB200_OK;
}

int Filter::set_beam_map(const bb200_beam_param& p, const bb200_occupancy_grid& g) {
  if (g.cells == nullptr || g.width <= 0 || g.height <= 0 || !(g.resolution > 0.0)) return fail(BB200_ERR_INVALID_ARGUMENT, "invalid occupancy grid");
  BB_CHECK(cudaSetDevice(config_.device));
  const size_t count = static_cast<size_t>(g.width) * static_cast<size_t>(g.height);
  BB_CHECK(cudaStreamSynchronize(stream_));
  cudaFree(occupancy_);
  occupancy_ = nullptr;
  BB_CHECK(dev_alloc(&occupancy_, count));
  BB_CHECK(cudaMemcpy(occupancy_, g.cells, count, cudaMemcpyHostToDevice));
  const std::vector<uint8_t> free_distance = make_free_distance(g);
  cudaFree(free_distance_);
  free_distance_ = nullptr;
  BB_CHECK(dev_alloc(&free_distance_, count));
  BB_CHECK(cudaMemcpy(free_distance_, free_distance.data(), count, cudaMemcpyHostToDevice));
  // padded copy for the two-pass walk: a border of zeros, power-of-two pitch
  cudaFree(free_padded_);
  free_padded_ = nullptr;
  occupancy_view_.free_padded = nullptr;
  occupancy_view_.pad_shift = 0;
  {
    int shift = 1;
    while ((1 << shift) < g.width + 2) ++shift;
    const size_t rows = static_cast<size_t>(g.height) + 2;
    if (shift <= 16 && g.height <= 65535) {
      std::vector<uint8_t> padded(rows << shift, 0);
      for (int y = 0; y < g.height; ++y)
        std::memcpy(padded.data() + ((static_cast<size_t>(y) + 1) << shift) + 1, free_distance.data() + static_cast<size_t>(y) * g.width, static_cast<size_t>(g.width));
      BB_CHECK(dev_alloc(&free_padded_, padded.size()));
      BB_CHECK(cudaMemcpy(free_padded_, padded.data(), padded.size(), cudaMemcpyHostToDevice));
      occupancy_view_.free_padded = free_padded_;
      occupancy_view_.pad_shift = shift;
    }
  }
  occupancy_view_.cells = occupancy_;
  occupancy_view_.free_distance = free_distance_;
  occupancy_view_.width = g.width;
  occupancy_view_.height = g.height;
  occupancy_view_.resolution = g.resolution;
  occupancy_view_.inv_resolution = 1. / g.resolution;
  occupancy_view_.world_to_grid = pose_inverse(pose_from_array(g.origin));
  beam_ = BeamParams{p.z_hit, p.z_short, p.z_max, p.z_rand, p.sigma_hit, p.lambda_short, p.beam_max_range, nullptr, 0};
  cudaFree(beam_eta_);
  beam_eta_ = nullptr;
  if (const uint32_t entries = beam_eta_table_ ? beam_eta_entries(p.beam_max_range, g.resolution) : 0u) {
    BB_CHECK(dev_alloc(&beam_eta_, entries));
    launch_beam_eta_table(beam_, g.resolution, beam_eta_, entries, stream_);
    BB_LAUNCHED("beam_eta_table");
    BB_CHECK(cudaStreamSynchronize(stream_));
    beam_.eta = beam_eta_;
    beam_.eta_entries = entries;
  }
  sensor_ = BB200_SENSOR_BEAM;
  field_host_.clear();

  const std::vector<uint32_t> free = make_free_cells(g);
  cudaFree(free_cells_);
  free_cells_ = nullptr;
  n_free_ = free.size();
  BB_CHECK(dev_alloc(&free_cells_, free.size()));
  if (!free.empty()) BB_CHECK(cudaMemcpy(free_cells_, free.data(), free.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  grid_width_ = g.width;
  grid_height_ = g.height;
  grid_resolution_ = g.resolution;
  grid_origin_ = pose_from_array(g.origin);
  return BB200_OK;
}

int Filter::get_likelihood_field(float* out, uint64_t capacity) const {
  if (field_host_.empty()) return BB200_ERR_STATE;
  if (capacity < field_host_.size()) return BB200_ERR_CAPACITY;
  std::memcpy(out, field_host_.data(), field_host_.size() * sizeof(float));
  return BB200_OK;
}

// ---- particle access ---------------------------------------------------------------------------------

int Filter::set_particles(const double* states, const double* weights, uint64_t n) {
  if (n > capacity_) return fail(BB200_ERR_CAPACITY, "more particles than the filter capacity");
  if (n > 0 && states == nullptr) return fail(BB200_ERR_INVALID_ARGUMENT, "states is null");
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  if (n > 0) {
    BB_CHECK(cudaMemcpy(states_[cur_], states, n * sizeof(Pose2), cudaMemcpyHostToDevice));
    if (weights != nullptr) {
      BB_CHECK(cudaMemcpy(weights_, weights, n * sizeof(double), cudaMemcpyHostToDevice));
    } else {
      const std::vector<double> ones(n, 1.0);
      BB_CHECK(cudaMemcpy(weights_, ones.data(), n * sizeof(double), cudaMemcpyHostToDevice));
    }
  }
  n_ = n;
  cdf_valid_ = false;
  cloud_known_ = false;
  if (n > 0) {  // the covariance is accumulated about the pivot: keep it inside the cloud (no cancellation for far-away sets)
    pivot_[0] = states[2];
    pivot_[1] = states[3];
  }
  return BB200_OK;
}

int Filter::get_particles(double* states, double* weights, uint64_t capacity) {
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  const uint64_t n = std::min(capacity, n_);
  if (states != nullptr && n > 0) BB_CHECK(cudaMemcpy(states, states_[cur_], n * sizeof(Pose2), cudaMemcpyDeviceToHost));
  if (weights != nullptr && n > 0) BB_CHECK(cudaMemcpy(weights, weights_, n * sizeof(double), cudaMemcpyDeviceToHost));
  return BB200_OK;
}

int Filter::initialize_normal(const double mean[3], const double cov[9], uint64_t n) {
  if (n > capacity_) return fail(BB200_ERR_CAPACITY, "more particles than the filter capacity");
  double transform[9];
  std::string message;
  if (!normal_transform(cov, transform, &message)) return fail(BB200_ERR_INVALID_ARGUMENT, message);
  BB_CHECK(cudaSetDevice(config_.device));
  launch_initialize_normal(states_[cur_], weights_, n, mean, transform, config_.seed, first_index_, stream_);
  BB_LAUNCHED("initialize_normal");
  BB_CHECK(cudaStreamSynchronize(stream_));
  n_ = n;
  cdf_valid_ = false;
  pivot_[0] = mean[0];
  pivot_[1] = mean[1];
  {  // the cloud just drawn is N(mean, cov): the first step can predict its pose bins
    const Pose2 m = pose_from_xytheta(mean[0], mean[1], mean[2]);
    cloud_ = bb200_estimate{{m.c, m.s, m.x, m.y}, {cov[0], cov[1], cov[2], cov[3], cov[4], cov[5], cov[6], cov[7], cov[8]}};
    cloud_known_ = true;
  }
  return BB200_OK;
}

int Filter::initialize_uniform(uint64_t n) {
  if (n > capacity_) return fail(BB200_ERR_CAPACITY, "more particles than the filter capacity");
  if (sensor_ < 0) return fail(BB200_ERR_STATE, "initialize_from_map needs a map (set_*_map first)");
  if (n_free_ == 0) return fail(BB200_ERR_STATE, "the map has no free cell to sample from");
  BB_CHECK(cudaSetDevice(config_.device));
  launch_initialize_uniform(states_[cur_], weights_, n, free_cells_, n_free_, grid_width_, grid_resolution_, grid_origin_, config_.seed,
                            first_index_, stream_);
  BB_LAUNCHED("initialize_uniform");
  BB_CHECK(cudaStreamSynchronize(stream_));
  n_ = n;
  cdf_valid_ = false;
  cloud_known_ = false;
  // pivot of the raw moments: the middle of the map in the global frame
  const double cx = 0.5 * grid_width_ * grid_resolution_, cy = 0.5 * grid_height_ * grid_resolution_;
  pivot_[0] = (grid_origin_.c * cx - grid_origin_.s * cy) + grid_origin_.x;
  pivot_[1] = (grid_origin_.s * cx + grid_origin_.c * cy) + grid_origin_.y;
  return BB200_OK;
}

// ---- per-step operations -----------------------------------------------------------------------------

int Filter::upload_points(const double* points_xy, uint64_t n_points) {
  if (n_points > points_capacity_) {
    cudaFree(points_);
    cudaFreeHost(points_host_);
    points_ = nullptr;
    points_host_ = nullptr;
    points_capacity_ = 0;
    const uint64_t cap = std::max<uint64_t>(n_points, 2048);
    BB_CHECK(dev_alloc(&points_, 2 * cap));
    BB_CHECK(cudaMallocHost(reinterpret_cast<void**>(&points_host_), 2 * cap * sizeof(double)));
    points_capacity_ = cap;
  }
  double radius = 0.0, range_sum = 0.0;
  for (uint64_t i = 0; i < n_points; ++i) {
    const double r = std::fabs(points_xy[2 * i]) + std::fabs(points_xy[2 * i + 1]);
    radius = (r > radius || std::isnan(r)) ? r : radius;  // NaN sticks -> general lookup path
    const double e = std::hypot(points_xy[2 * i], points_xy[2 * i + 1]);
    if (std::isfinite(e)) range_sum += e;
  }
  points_radius_ = radius;
  points_mean_range_ = n_points > 0 ? range_sum / static_cast<double>(n_points) : 1.0;  // lever arm of the heading in the schedule
  if (n_points > 0) {
    // The previous step's copy must have left the staging buffer before it is overwritten.
    std::memcpy(points_host_, points_xy, 2 * n_points * sizeof(double));
    BB_CHECK(cudaMemcpyAsync(points_, points_host_, 2 * n_points * sizeof(double), cudaMemcpyHostToDevice, stream_));
  }
  return BB200_OK;
}

bool Filter::predict_schedule(const MotionSampling& s, Schedule* grid) const {
  // The cloud after this step's propagate, from what the host already knows: the last estimate (the particles carry unit
  // weights, so it describes the raw cloud) composed with the motion means, spread widened by the motion noise.
  if (!cloud_known_ || !predict_schedule_) return false;
  const bb200_estimate& e = cloud_;
  const Pose2 mean = motion_apply(s.model, Pose2{e.mean[0], e.mean[1], e.mean[2], e.mean[3]}, s.mean[0], s.mean[1], s.mean[2], Rot2{s.first_c, s.first_s});
  double var_theta = std::max(e.cov[8], 0.0) + s.stddev[0] * s.stddev[0];
  double spread = s.stddev[1] * s.stddev[1];
  if (s.model == BB200_MOTION_DIFFERENTIAL) var_theta += s.stddev[2] * s.stddev[2];
  if (s.model != BB200_MOTION_DIFFERENTIAL) spread += s.stddev[2] * s.stddev[2];
  if (s.model != BB200_MOTION_STATIONARY) spread += s.mean[1] * s.mean[1] * var_theta;
  const double vx = e.cov[0] + spread, vy = e.cov[4] + spread;
  if (!std::isfinite(var_theta) || !std::isfinite(vx) || !std::isfinite(vy) || !std::isfinite(mean.x) || !std::isfinite(mean.y)) return false;
  const double r = std::exp(-0.5 * var_theta);
  schedule_from_moments(*grid, r * mean.c, r * mean.s, mean.x, mean.y, vx, vy, static_cast<double>(n_), schedule_lever_ * points_mean_range_,
                        0.5 * grid_resolution_, schedule_per_bin_, schedule_x_split_, schedule_equal_mass_);
  return true;
}

int Filter::enqueue_propagate_reweight(const MotionSampling* sampling, uint32_t step, bool do_reweight, uint64_t n_points, bool counters_reset) {
  const bool scheduled = do_reweight && schedule_enabled_ && n_ >= kScheduleMinParticles;
  Schedule grid{};
  const uint32_t* perm = nullptr;
  if (scheduled && counters_reset && sampling != nullptr && predict_schedule(*sampling, &grid)) {
    // Bin grid predicted on the host: propagate histograms its own output, two more launches turn it into the order.
    mark("propagate");
    launch_propagate_binned(states_[cur_], n_, *sampling, config_.seed, step, first_index_, grid, bin_rank_, counters_, sched_, stream_);
    BB_LAUNCHED("propagate");
    mark("schedule");
    launch_finish_schedule(bin_rank_, n_, grid.n_bins, sched_, counters_, perm_, sched_tiles_, stream_);
    BB_LAUNCHED_N("schedule", 2);
    perm = perm_;
  } else if (sampling != nullptr || scheduled) {
    mark("propagate");
    launch_propagate(states_[cur_], n_, sampling != nullptr, sampling != nullptr ? *sampling : MotionSampling{}, config_.seed, step,
                     first_index_, scheduled ? sched_ : nullptr, stream_);
    BB_LAUNCHED_N("propagate", scheduled ? 2 : 1);
  }
  if (scheduled && perm == nullptr) {
    mark("schedule");
    launch_build_schedule(states_[cur_], n_, sched_, bins_, counters_, perm_, sched_tiles_, schedule_lever_ * points_mean_range_, 0.5 * grid_resolution_, schedule_per_bin_, schedule_x_split_, schedule_equal_mass_, stream_);
    BB_LAUNCHED_N("schedule", 4);
    perm = perm_;
  }
  if (do_reweight) {
    if (sensor_ == BB200_SENSOR_BEAM) {
      mark("reweight_beam");
      uint64_t pass = 0;
      // spans of the walk's 32-bit arithmetic: far ends lie within beam_max_range of the source, sources inside the grid
      const double reach_cells = beam_.beam_max_range * occupancy_view_.inv_resolution + 4.0;
      if (beam_two_pass_ && n_points > 0 && occupancy_view_.free_padded != nullptr && reach_cells < static_cast<double>(1 << 21)) {
        // hit words of one pass: at most 3 GiB, whole warps of particles
        pass = std::min<uint64_t>(n_, std::max<uint64_t>(32, ((3ull << 30) / (4ull * n_points)) / 32 * 32));
        const uint64_t words = beam_hit_words(pass, static_cast<uint32_t>(n_points));
        if (words > beam_hits_words_) {
          BB_CHECK(cudaStreamSynchronize(stream_));
          cudaFree(beam_hits_);
          beam_hits_ = nullptr;
          beam_hits_words_ = 0;
          // sized for the filter's capacity so that a growing particle count (KLD) does not reallocate every step
          const uint64_t pass_cap = std::min<uint64_t>(capacity_, std::max<uint64_t>(32, ((3ull << 30) / (4ull * n_points)) / 32 * 32));
          const uint64_t want = beam_hit_words(std::max(pass, pass_cap), static_cast<uint32_t>(n_points));
          if (dev_alloc(&beam_hits_, want) == cudaSuccess) {
            beam_hits_words_ = want;
          } else {
            (void)cudaGetLastError();  // no room for the intermediate: the fused kernel needs none
            pass = 0;
          }
        }
      }
      if (pass > 0) {
        launch_reweight_beam_two_pass(states_[cur_], weights_, n_, perm, occupancy_view_, beam_, points_, static_cast<uint32_t>(n_points), beam_hits_, pass,
                                      scalars_, stream_);
        BB_LAUNCHED_N("reweight_beam", 2 * static_cast<int>((n_ + pass - 1) / pass));
      } else {
        launch_reweight_beam(states_[cur_], weights_, n_, perm, occupancy_view_, beam_, points_, static_cast<uint32_t>(n_points), scalars_, stream_);
        BB_LAUNCHED("reweight_beam");
      }
    } else {
      mark("reweight_lfm");
      launch_reweight_lfm(states_[cur_], weights_, n_, perm, field_, points_, param_points_ ? points_host_ : nullptr, static_cast<uint32_t>(n_points),
                          points_radius_, scalars_, stream_);
      BB_LAUNCHED("reweight_lfm");
    }
  }
  return BB200_OK;
}

int Filter::propagate_reweight(const bb200_motion_sampling* sampling, uint32_t step, const double* points_xy, uint64_t n_points) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  const bool do_reweight = points_xy != nullptr;
  if (do_reweight && sensor_ < 0) return fail(BB200_ERR_STATE, "no sensor model map set");
  if (do_reweight && n_points > 0xffffffffull) return fail(BB200_ERR_INVALID_ARGUMENT, "too many points");
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));  // staging buffer reuse + keeps the fine-grained API simple
  if (do_reweight) {
    const int st = upload_points(points_xy, n_points);
    if (st != BB200_OK) return st;
  }
  MotionSampling s{};
  if (sampling != nullptr) s = to_kernel_sampling(*sampling);
  mark("begin_step");
  launch_begin_step(scalars_, stream_);
  BB_LAUNCHED("begin_step");
  const int st = enqueue_propagate_reweight(sampling != nullptr ? &s : nullptr, step, do_reweight, n_points, false);
  if (st != BB200_OK) return st;
  cdf_valid_ = false;
  cloud_known_ = false;
  finish_marks();
  return BB200_OK;
}

int Filter::max_weight(double* wmax) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  BB_CHECK(cudaSetDevice(config_.device));
  launch_begin_step(scalars_, stream_);
  BB_LAUNCHED("begin_step");
  launch_max_weight(weights_, n_, scalars_, stream_);
  BB_LAUNCHED("max_weight");
  BB_CHECK(cudaMemcpyAsync(scalars_host_, scalars_, sizeof(Scalars), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  double v;
  std::memcpy(&v, &scalars_host_->wmax_bits, sizeof(double));
  *wmax = v;
  return BB200_OK;
}

int Filter::build_cdf(double global_wmax, uint64_t* local_total, int* exponent) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  BB_CHECK(cudaSetDevice(config_.device));
  if (global_wmax < 0.0) {
    launch_begin_step(scalars_, stream_);
    BB_LAUNCHED("begin_step");
    launch_max_weight(weights_, n_, scalars_, stream_);
    BB_LAUNCHED("max_weight");
  }
  mark("prepare_cdf");
  launch_prepare_cdf(scalars_, global_wmax, config_.global_count, tile_state_, scan_tile_count(n_), stream_);
  BB_LAUNCHED("prepare_cdf");
  mark("quantize_scan");
  launch_quantize_scan(weights_, n_, cdf_, scalars_, tile_state_, stream_);
  BB_LAUNCHED("quantize_scan");
  BB_CHECK(cudaMemcpyAsync(scalars_host_, scalars_, sizeof(Scalars), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  finish_marks();
  cdf_valid_ = true;
  if (local_total != nullptr) *local_total = scalars_host_->total;
  if (exponent != nullptr) *exponent = scalars_host_->exponent;
  // No positive finite weight (the reference would divide by zero in normalize.hpp:82): a uniform CDF
  // has been substituted and the weights are left as they are; reported through last_error only.
  weights_valid_ = scalars_host_->valid != 0;
  if (!weights_valid_) error_ = "no positive finite weight (uniform CDF substituted)";
  return BB200_OK;
}

int Filter::normalize_by(uint64_t global_total, double* local_sum_sq) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  if (!cdf_valid_) return fail(BB200_ERR_STATE, "build_cdf must run before normalize_by");
  BB_CHECK(cudaSetDevice(config_.device));
  uint32_t rows = 0;
  mark("normalize");
  launch_normalize(weights_, n_, scalars_, global_total, partials_, &rows, stream_);
  BB_LAUNCHED("normalize");
  launch_reduce_partials(partials_, rows, 1, results_, stream_);
  BB_LAUNCHED("reduce_partials");
  BB_CHECK(cudaMemcpyAsync(results_host_, results_, sizeof(double), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  finish_marks();
  if (local_sum_sq != nullptr) *local_sum_sq = results_host_[0];
  return BB200_OK;
}

int Filter::normalize(double* factor, double* sum_sq) {
  uint64_t total = 0;
  int exponent = 0;
  const int st = build_cdf(-1.0, &total, &exponent);
  if (st != BB200_OK) return st;
  if (factor != nullptr) *factor = std::ldexp(static_cast<double>(total), -exponent);
  return normalize_by(total, sum_sq);
}

int Filter::ensure_cdf_ready() {
  if (cdf_valid_) return BB200_OK;
  return build_cdf(-1.0, nullptr, nullptr);
}

void Filter::estimate_from_moments_static(const double m[kMomentCount], const double pivot[2], bb200_estimate* out) {
  // estimation.hpp:436-475 from raw moments about the pivot: normalised weights w/S,
  // mean of (cos, sin, x, y); cov = (E[d d^T] - E[d] E[d]^T) / (1 - sum (w/S)^2).
  const double sum = m[0];
  const double mc = m[2] / sum, ms = m[3] / sum, mdx = m[4] / sum, mdy = m[5] / sum;
  const double correction = 1.0 - m[1] / (sum * sum);
  for (double& c : out->cov) c = 0.0;
  out->cov[0] = (m[6] / sum - mdx * mdx) / correction;
  out->cov[1] = (m[7] / sum - mdx * mdy) / correction;
  out->cov[3] = out->cov[1];
  out->cov[4] = (m[8] / sum - mdy * mdy) / correction;
  out->mean[2] = pivot[0] + mdx;
  out->mean[3] = pivot[1] + mdy;
  const double norm = std::sqrt(mc * mc + ms * ms);
  if (norm < std::numeric_limits<double>::epsilon()) {
    out->cov[8] = std::numeric_limits<double>::infinity();
    out->mean[0] = 1.0;
    out->mean[1] = 0.0;
  } else {
    out->cov[8] = -2.0 * std::log(norm);
    const double len = std::hypot(mc, ms);
    out->mean[0] = mc / len;
    out->mean[1] = ms / len;
  }
}

void Filter::estimate_from_moments(const double m[kMomentCount], bb200_estimate* out) const { estimate_from_moments_static(m, pivot_, out); }

int Filter::moments(const double pivot[2], double out[9]) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  BB_CHECK(cudaSetDevice(config_.device));
  mark("moments");
  launch_moments(states_[cur_], weights_, n_, pivot[0], pivot[1], partials_, stream_);
  BB_LAUNCHED("moments");
  launch_reduce_partials(partials_, moments_block_count(n_), kMomentCount, results_, stream_);
  BB_LAUNCHED("reduce_partials");
  BB_CHECK(cudaMemcpyAsync(results_host_, results_, kMomentCount * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  finish_marks();
  std::memcpy(out, results_host_, kMomentCount * sizeof(double));
  return BB200_OK;
}

int Filter::estimate(bb200_estimate* out) {
  double m[kMomentCount];
  const int st = moments(pivot_, m);
  if (st != BB200_OK) return st;
  estimate_from_moments(m, out);
  pivot_[0] = out->mean[2];
  pivot_[1] = out->mean[3];
  return BB200_OK;
}

// ---- cluster-based estimate ---------------------------------------------------------------------

int Filter::ensure_cluster_scratch(uint32_t cells) {
  ClusterScratch& c = cluster_;
  if (c.capacity == 0) {
    if (capacity_ >= (1ull << 31)) return fail(BB200_ERR_CAPACITY, "cluster estimate: more than 2^31 particles per filter");
    uint64_t table = 2;
    while (table < 2 * capacity_) table <<= 1;
    const uint32_t tiles = cluster_sort_tiles(capacity_);
    BB_CHECK(dev_alloc(&c.hashes, capacity_));
    BB_CHECK(dev_alloc(&c.keys, table));
    BB_CHECK(dev_alloc(&c.first, table));
    BB_CHECK(dev_alloc(&c.slot_of, capacity_));
    BB_CHECK(dev_alloc(&c.flags, capacity_));
    BB_CHECK(dev_alloc(&c.cell_of, capacity_));
    BB_CHECK(dev_alloc(&c.starts, capacity_ + 1));
    BB_CHECK(dev_alloc(&c.keys_a, capacity_));
    BB_CHECK(dev_alloc(&c.keys_b, capacity_));
    BB_CHECK(dev_alloc(&c.idx_a, capacity_));
    BB_CHECK(dev_alloc(&c.idx_b, capacity_));
    BB_CHECK(dev_alloc(&c.histogram, static_cast<size_t>(256) * tiles));
    BB_CHECK(dev_alloc(&c.tile_state, static_cast<size_t>(scan_tile_count(std::max<uint64_t>(capacity_ + 1, 256ull * tiles)) + 1)));
    BB_CHECK(dev_alloc(&c.words, 4));
    c.table_size = table;
    c.capacity = capacity_;
  }
  if (cells > c.records_capacity) {
    cudaFree(c.records);
    c.records = nullptr;
    c.records_capacity = 0;
    const uint64_t want = std::min<uint64_t>(capacity_, std::max<uint64_t>(1024, 2ull * cells));
    BB_CHECK(dev_alloc(&c.records, want));
    c.records_capacity = want;
  }
  return BB200_OK;
}

int Filter::cell_records(double linear_resolution, double angular_resolution, std::vector<HostCell>* host) {
  // Per-particle half of the clusterizer, also the device-side histogram of the particle cloud: spatial hash ->
  // first-occurrence numbering of the occupied cells -> stable sort of the particle indices by cell -> one record per
  // cell (representative = first particle, count, weight summed in particle order, raw moments).
  BB_CHECK(cudaSetDevice(config_.device));
  {
    const int st = ensure_cluster_scratch(0);
    if (st != BB200_OK) return st;
  }
  mark("cluster_cells");
  launch_cluster_cells_begin(states_[cur_], n_, linear_resolution, angular_resolution, cluster_, stream_);
  BB_LAUNCHED_N("cluster_cells_begin", 3);
  unsigned long long cells64 = 0;
  BB_CHECK(cudaMemcpyAsync(&cells64, cluster_.words + 1, sizeof(cells64), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  const uint32_t cells = static_cast<uint32_t>(cells64);
  {
    const int st = ensure_cluster_scratch(cells);
    if (st != BB200_OK) return st;
  }
  mark("cluster_sort");
  int sort_launches = 0;
  const uint32_t* sorted = launch_cluster_sort(n_, cells, cluster_, stream_, &sort_launches);
  BB_LAUNCHED_N("cluster_sort", sort_launches);
  mark("cluster_records");
  launch_cluster_records(states_[cur_], weights_, sorted, cells, pivot_[0], pivot_[1], cluster_, stream_);
  BB_LAUNCHED("cluster_records");
  host->resize(cells);
  static_assert(sizeof(HostCell) == sizeof(CellRecord), "record layouts must agree");
  BB_CHECK(cudaMemcpyAsync(host->data(), cluster_.records, static_cast<size_t>(cells) * sizeof(CellRecord), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  finish_marks();
  return BB200_OK;
}

int Filter::cluster_estimate(const bb200_cluster_param& p, bb200_estimate* out, uint32_t* cluster_ids, uint64_t ids_capacity, uint32_t* n_cells,
                             uint32_t* n_clusters) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  if (!(p.linear_hash_resolution > 0.0) || !(p.angular_hash_resolution > 0.0) || !(p.weight_cap_percentile >= 0.0) ||
      !(p.weight_cap_percentile < 1.0))
    return fail(BB200_ERR_INVALID_ARGUMENT, "cluster parameters: resolutions must be positive and the percentile in [0, 1)");
  if (cluster_ids != nullptr && ids_capacity < n_) return fail(BB200_ERR_CAPACITY, "cluster id buffer too small");
  std::vector<HostCell> host;
  {
    const int st = cell_records(p.linear_hash_resolution, p.angular_hash_resolution, &host);
    if (st != BB200_OK) return st;
  }
  const uint32_t cells = static_cast<uint32_t>(host.size());
  const ClusterSelection sel = select_cluster(host.data(), host.size(), n_, p.linear_hash_resolution, p.angular_hash_resolution, p.weight_cap_percentile);
  if (out != nullptr) estimate_from_moments(sel.moments, out);
  if (n_cells != nullptr) *n_cells = cells;
  if (n_clusters != nullptr) *n_clusters = sel.clusters;
  if (cluster_ids != nullptr) {
    std::vector<uint32_t> cell_of(n_);
    BB_CHECK(cudaMemcpy(cell_of.data(), cluster_.cell_of, n_ * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < n_; ++i) cluster_ids[i] = sel.cluster_of_cell[cell_of[i]];
  }
  return BB200_OK;
}

int Filter::particle_histogram(double linear_resolution, double angular_resolution, bb200_cluster_cell* bins, uint64_t capacity, uint64_t* n_bins,
                               double* max_bin_weight) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  if (!(linear_resolution > 0.0) || !(angular_resolution > 0.0)) return fail(BB200_ERR_INVALID_ARGUMENT, "histogram resolutions must be positive");
  std::vector<HostCell> host;
  const int st = cell_records(linear_resolution, angular_resolution, &host);
  if (st != BB200_OK) return st;
  if (n_bins != nullptr) *n_bins = host.size();
  double top = 1e-3;  // beluga_ros/particle_cloud.hpp:197
  for (const HostCell& c : host) top = c.weight > top ? c.weight : top;
  if (max_bin_weight != nullptr) *max_bin_weight = top;
  if (bins != nullptr) {
    if (capacity < host.size()) return fail(BB200_ERR_CAPACITY, "histogram bin buffer too small (n_bins has the count)");
    static_assert(sizeof(bb200_cluster_cell) == sizeof(HostCell), "public and internal cell records must agree");
    std::memcpy(bins, host.data(), host.size() * sizeof(HostCell));
  }
  return BB200_OK;
}

int Filter::sample_states(uint64_t count, uint32_t step, double* states_out) {
  // views::sample | take_exactly(count) (beluga_ros/particle_cloud.hpp:141-147): `count` states drawn by weight, the
  // particle set itself untouched.  Counter RNG: the multinomial draws of `step` (the caller picks a step the filter
  // does not use, e.g. 0xFFFFFFFF - publish count).
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  if (count > capacity_) return fail(BB200_ERR_CAPACITY, "more samples than the filter capacity");
  if (count > 0 && states_out == nullptr) return fail(BB200_ERR_INVALID_ARGUMENT, "states_out is null");
  if (count == 0) return BB200_OK;
  int st = ensure_cdf_ready();
  if (st != BB200_OK && !cdf_valid_) return st;
  BB_CHECK(cudaSetDevice(config_.device));
  bb200_resample_opts o{};
  o.scheme = BB200_RESAMPLE_MULTINOMIAL;
  o.step = step;
  o.min_particles = o.max_particles = count;
  ResampleArgs a = make_resample_args(o, 0, count, false);
  a.weights_out = nullptr;  // the weights stay what they are
  a.ancestors = nullptr;
  launch_resample(a, scalars_, partials_, stream_);  // into the staging state buffer; no flip
  BB_LAUNCHED("sample_states");
  BB_CHECK(cudaMemcpyAsync(states_out, states_[cur_ ^ 1], count * sizeof(Pose2), cudaMemcpyDeviceToHost, stream_));
  BB_CHECK(cudaStreamSynchronize(stream_));
  return BB200_OK;
}

ResampleArgs Filter::make_resample_args(const bb200_resample_opts& o, uint64_t slot_begin, uint64_t slot_end, bool with_hashes) const {
  ResampleArgs a{};
  a.states_in = states_[cur_];
  a.cdf = cdf_;
  a.n_in = n_;
  a.states_out = states_[cur_ ^ 1] + slot_begin;
  a.weights_out = weights_ + slot_begin;
  a.ancestors = ancestors_ != nullptr ? ancestors_ + slot_begin : nullptr;
  a.hashes = with_hashes ? hashes_ + slot_begin : nullptr;
  a.slot_first = first_index_ + slot_begin;
  a.slot_count = slot_end - slot_begin;
  a.total_slots = o.max_particles;
  a.scheme = o.scheme;
  a.seed = config_.seed;
  a.step = o.step;
  a.random_state_probability = o.random_state_probability;
  a.free_cells = free_cells_;
  a.n_free = n_free_;
  a.grid_width = grid_width_;
  a.grid_resolution = grid_resolution_;
  a.grid_origin = grid_origin_;
  for (int k = 0; k < 3; ++k) a.hash_resolution[k] = o.spatial_resolution[k];
  a.pivot_x = pivot_[0];
  a.pivot_y = pivot_[1];
  return a;
}

int Filter::resample(const bb200_resample_opts& o, uint64_t* new_size) {
  if (n_ == 0) return fail(BB200_ERR_STATE, "no particles");
  if (o.max_particles == 0 || o.max_particles > capacity_) return fail(BB200_ERR_CAPACITY, "max_particles exceeds the filter capacity");
  if (o.random_state_probability > 0.0 && n_free_ == 0) return fail(BB200_ERR_STATE, "recovery injection needs a map with free cells");
  int st = ensure_cdf_ready();
  if (st != BB200_OK && !cdf_valid_) return st;
  BB_CHECK(cudaSetDevice(config_.device));
  // The weight array is reused for the output (all ones); the CDF already holds what sampling needs.
  uint64_t m = o.max_particles;
  if (o.min_particles >= o.max_particles) {
    // take_while_kld never stops before max when min == max (take_while_kld.hpp:86-87,136).
    mark("resample");
    launch_resample(make_resample_args(o, 0, o.max_particles, false), scalars_, partials_, stream_);
    BB_LAUNCHED("resample");
    BB_CHECK(cudaStreamSynchronize(stream_));
  } else {
    st = resample_kld(o, &m);
    if (st != BB200_OK) return st;
  }
  finish_marks();
  cur_ ^= 1;
  cloud_known_ = false;
  n_ = m;
  ancestors_n_ = n_;
  cdf_valid_ = false;
  if (new_size != nullptr) *new_size = n_;
  return BB200_OK;
}

int Filter::resample_range(const bb200_resample_opts& o, uint64_t global_total, uint64_t cdf_offset, uint64_t slot_begin, uint64_t slot_end) {
  // Sharded filter: this rank produces the output slots [slot_begin, slot_end) -- exactly those whose
  // comb position falls inside its span of the global CDF -- into the staging buffer, in slot order.
  if (!cdf_valid_) return fail(BB200_ERR_STATE, "build_cdf must run before resample_range");
  if (o.scheme != BB200_RESAMPLE_SYSTEMATIC || o.min_particles < o.max_particles)
    return fail(BB200_ERR_STATE, "range resampling supports the systematic comb without KLD (multinomial: bb200_filter_enqueue_resample_push)");
  if (o.random_state_probability > 0.0 && n_free_ == 0) return fail(BB200_ERR_STATE, "recovery injection needs a map with free cells");
  if (slot_end < slot_begin || slot_end - slot_begin > capacity_) return fail(BB200_ERR_CAPACITY, "slot range exceeds the staging buffer");
  BB_CHECK(cudaSetDevice(config_.device));
  if (slot_end > slot_begin) {
    ResampleArgs a = make_resample_args(o, 0, slot_end - slot_begin, false);
    a.slot_first = slot_begin;  // global slot index
    a.global_total = global_total;
    a.cdf_offset = cdf_offset;
    a.weights_out = nullptr;  // the current weights stay untouched; adopt() writes the ones
    mark("resample_range");
    launch_resample(a, scalars_, partials_, stream_);
    BB_LAUNCHED("resample_range");
  }
  BB_CHECK(cudaStreamSynchronize(stream_));
  finish_marks();
  return BB200_OK;
}

int Filter::adopt(uint64_t n, int from_staging) {
  // The caller has placed n particle states into the current (or staging) state buffer, e.g. through
  // an all-to-all: make them the particle set with unit weights (make_from_state, particle_traits.hpp:105).
  if (n > capacity_) return fail(BB200_ERR_CAPACITY, "more particles than the filter capacity");
  BB_CHECK(cudaSetDevice(config_.device));
  if (from_staging) cur_ ^= 1;
  cloud_known_ = false;
  n_ = n;
  cdf_valid_ = false;
  if (n > 0) {
    launch_fill(weights_, n, 1.0, stream_);
    BB_LAUNCHED("fill_weights");
  }
  BB_CHECK(cudaStreamSynchronize(stream_));
  return BB200_OK;
}

int Filter::resample_kld(const bb200_resample_opts& o, uint64_t* accepted) {
  if (config_.global_count != capacity_ || first_index_ != 0) return fail(BB200_ERR_STATE, "KLD-adaptive resampling runs on a single shard");
  if (o.max_particles >= (1ull << 32)) return fail(BB200_ERR_CAPACITY, "KLD-adaptive resampling keeps 32-bit slot indices: max_particles must be below 2^32");
  if (hashes_ == nullptr) {
    BB_CHECK(dev_alloc(&hashes_, capacity_));
    BB_CHECK(dev_alloc(&kld_flags_, capacity_));
    BB_CHECK(dev_alloc(&kld_scan_, capacity_));
    kld_table_size_ = 2;
    while (kld_table_size_ < 2 * capacity_) kld_table_size_ <<= 1;
    BB_CHECK(dev_alloc(&kld_keys_, kld_table_size_));
    BB_CHECK(dev_alloc(&kld_vals_, kld_table_size_));
  }
  mark("kld");
  launch_kld_clear(kld_keys_, kld_vals_, kld_table_size_, stream_);
  const uint64_t max = o.max_particles;
  uint64_t begin = 0, k_before = 0;
  uint64_t end = std::min<uint64_t>(max, std::max<uint64_t>(2 * o.min_particles, 65536));
  *accepted = max;
  while (begin < max) {
    launch_resample(make_resample_args(o, begin, end, true), scalars_, partials_, stream_);
    BB_LAUNCHED("resample");
    KldArgs k{hashes_ + begin, end - begin, begin, k_before, o.min_particles, o.kld_epsilon, o.kld_z};
    launch_kld_chunk(k, kld_keys_, kld_vals_, kld_table_size_, kld_flags_, kld_scan_, scalars_, tile_state_, stream_);
    BB_LAUNCHED_N("kld", 5);
    BB_CHECK(cudaMemcpyAsync(scalars_host_, scalars_, sizeof(Scalars), cudaMemcpyDeviceToHost, stream_));
    BB_CHECK(cudaStreamSynchronize(stream_));
    if (scalars_host_->kld_cutoff != ~0ull) {
      // take_while drops the first element whose condition fails (take_while_kld.hpp:134-136).
      *accepted = std::min<uint64_t>(scalars_host_->kld_cutoff - 1, max);
      break;
    }
    k_before += scalars_host_->pad[1];
    begin = end;
    end = std::min<uint64_t>(max, end * 2);
  }
  return BB200_OK;
}

int Filter::step_resample(const bb200_motion_sampling& sampling, uint32_t step, const double* points_xy, uint64_t n_points,
                          const bb200_resample_opts& o, bb200_estimate* est, double* weight_sum, uint64_t* new_size) {
  int st = step_begin(sampling, step, points_xy, n_points, o, true);
  for (int phase = kPhaseReweight; st == BB200_OK && phase <= kPhaseFinish; ++phase) st = step_phase(phase);
  if (st != BB200_OK) {
    step_.active = false;
    return st;
  }
  return step_end(est, weight_sum, new_size, nullptr);
}

int Filter::ancestors(int64_t* out, uint64_t capacity) {
  if (ancestors_ == nullptr) return fail(BB200_ERR_STATE, "filter was created without record_ancestors");
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  const uint64_t n = std::min(capacity, ancestors_n_);
  if (n > 0) BB_CHECK(cudaMemcpy(out, ancestors_, n * sizeof(int64_t), cudaMemcpyDeviceToHost));
  return BB200_OK;
}

int Filter::cdf(uint64_t* out, uint64_t capacity) {
  if (!cdf_valid_) return fail(BB200_ERR_STATE, "no CDF has been built for the current weights");
  BB_CHECK(cudaSetDevice(config_.device));
  BB_CHECK(cudaStreamSynchronize(stream_));
  const uint64_t n = std::min(capacity, n_);
  if (n > 0) BB_CHECK(cudaMemcpy(out, cdf_, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return BB200_OK;
}

}  // namespace bb200
