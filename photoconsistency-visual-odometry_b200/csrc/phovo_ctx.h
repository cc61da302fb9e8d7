// phovo_ctx.h -- the context object behind the C ABI (one CUDA device + one stream).
#ifndef PHOVO_CTX_H_
#define PHOVO_CTX_H_

#include <cuda_runtime.h>

#include <algorithm>
#include <string>
#include <vector>

#include "phovo_host.h"

struct phovo_batch_state;  // phovo_batch.cu

struct phovo_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  phovo::Stream own_stream;   // the stream phovo_create made; empty once phovo_set_stream names another (and for slots)
  std::string err;
  std::string path_note;   // why the last driver that failed on this context could not run (phovo_graph_error)

  phovo_config cfg;
  double K[9] = {0};
  bool have_K = false;
  bool build_all_levels = false;
  bool have_src = false, have_tgt = false;

  // geometry of the current frames
  int rows = 0, cols = 0;
  int lrows[PHOVO_MAX_LEVELS] = {0}, lcols[PHOVO_MAX_LEVELS] = {0};

  // HBM layout (general path): per active level five dense row-major fp64 images -- bit-identical to the
  // reference's cv::Mat_<double> levels (fp32 storage makes ~15% of trajectories diverge, see DESIGN.md)
  phovo::DeviceArray<double> I0[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> D0[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> I1[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> Gx[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> Gy[PHOVO_MAX_LEVELS];
  // photometric + depth solver: target depth pyramid, Scharr of depth / max_depth, gain per level
  phovo::DeviceArray<double> D1[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> GxD[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> GyD[PHOVO_MAX_LEVELS];
  phovo::DeviceArray<double> d_gain;
  bool have_tgt_depth = false;
  phovo::DeviceArray<int> winner;              // one int per pixel of the largest active level
  phovo::DeviceArray<unsigned char> valid;     // one flag per pixel (K3a -> K3b)
  phovo::DeviceArray<double> scratch64[2];
  phovo::DeviceArray<double> partials;         // [grid][32] per-block normal-equation partials
  phovo::DeviceArray<char> stage_gray[2];
  phovo::DeviceArray<char> stage_depth;
  phovo::DeviceArray<double> dump_res;
  phovo::DeviceArray<double> dump_jac;
  // phovo_warp_image scratch (its keys belong to the batch state)
  phovo::DeviceArray<char> warp_io[3];         // device copies of warped / target / diff for host callers

  // solver state
  double state[6] = {0};
  phovo::DeviceArray<PoseDev> d_pose; phovo::PinnedArray<PoseDev> h_pose;
  phovo::DeviceArray<phovo_iter_stats> d_log; phovo::PinnedArray<phovo_iter_stats> h_log;
  phovo::DeviceArray<phovo_iter_stats> d_eval; phovo::PinnedArray<phovo_iter_stats> h_eval;
  phovo::DeviceArray<double> d_state_in; phovo::PinnedArray<double> h_state_in;
  std::vector<phovo_iter_stats> log;

  // driver of Optimize() (phovo_set_execution): 3 cluster for small levels, 2 (default) persistent cooperative kernel per
  // level, 1 CUDA graph with WHILE nodes, 0 stream launches + host polling.  Bit p of failed_paths: path p could not run
  // on this context, and Optimize() no longer tries it.
  int execution = 2; unsigned failed_paths = 0; int last_path = 0;
  int sm_count = 0;
  cudaGraph_t graph = nullptr; cudaGraphExec_t graph_exec = nullptr;
  int graph_launches_fixed = 0, graph_launches_per_iter = 0;

  // row sharding
  int shard_rank = 0, shard_world = 1, shard_level = -1;
  phovo::DeviceArray<double> d_shard;
  phovo::DeviceArray<double> d_level_dmin;   // [PHOVO_MAX_LEVELS] smallest valid depth per level of the current source frame
  bool level_dmin_valid = false;
  // fused peer-store exchange: own area (device memory, IPC-exported), peers' areas (IPC-opened)
  phovo::DeviceArray<phovo::ShardExchange> xchg_own;
  phovo::ShardExchange* xchg_peer[8] = {nullptr};
  bool xchg_opened[8] = {false};
  phovo::DeviceArray<phovo::ShardExchange*> xchg_peers_dev;   // device copy of xchg_peer[]
  bool xchg_table_dirty = true;
  unsigned long long xchg_epoch = 0;

  // bookkeeping
  phovo::Event ev_copy, ev_time[4];
  bool h2d_pending = false, copy_event_armed = false, setup_timed = false;
  bool defer_device_input_drain = false; // batch slots: the owner of the context keeps device inputs alive and waits itself
  bool device_input_in_flight = false;   // a Set*Frame call was given a device pointer and its kernels are queued
  phovo::LaunchState launch_state;       // per-DEVICE function attributes / occupancy of the persistent kernels
  int64_t launches = 0;

  phovo_batch_state* batch = nullptr;

  // Batch slots (phovo_batch.cu, wave path): a context used for its device side only.  Its level images, winner map,
  // scratch and PoseDev are carved out of ONE allocation owned by the batch state (several hundred slots otherwise
  // cost tens of cudaMalloc / cudaMallocHost calls each: seconds); no stream of its own, no pinned host buffers.
  bool is_slot = false;
  char* arena_base = nullptr; size_t arena_bytes = 0, arena_used = 0;
  void arena_reset(char* base, size_t bytes);   // forget every arena-backed buffer; base == nullptr: leave the arena

  int fail(int code, const std::string& what);
  int cuda_fail(const char* what, cudaError_t e);
  int log_cap() const { return (int)std::min(d_log.capacity(), h_log.capacity()); }   // stats entries Optimize may write
  bool level_active(int l) const;
  LevelParams level_params(int level) const;
  phovo::LevelPtrs level_ptrs(int level) const;
  void invalidate_graph();
};

// The coarse-to-fine walk of every solve (AN:502-503): fn(level, M) for each level with M = max_num_iterations[level] > 0,
// coarsest first; a level without iterations is an empty pass (AN:526).  Stops at, and returns, fn's first non-zero
// return.  It reads the configuration only: batch contexts have no frames.
template <class Fn>
int for_each_level(const phovo_config& cfg, Fn&& fn) {
  for (int level = cfg.num_levels - 1; level >= 0; --level) {
    const int M = cfg.max_num_iterations[level];
    if (M <= 0) continue;
    if (const int rc = fn(level, M)) return rc;
  }
  return 0;
}

void phovo_batch_release(phovo_ctx* ctx);
// phovo::warpImage of `num_pairs` pairs (device pointers in W; rts host or device [num_pairs][16]), enqueued on the
// context stream with the batch state's keys; W.rts is ignored
int phovo_internal_warp_images(phovo_ctx* ctx, phovo::WarpImages W, int src_type, const phovo::WarpIntrinsics& I,
                               int num_pairs, const double* rts);
// a slot context on `device` (see phovo_ctx::is_slot): set the stream and the arena before the first frame
int phovo_internal_create_slot(int device, phovo_ctx** out);
// device bytes a slot needs for rows x cols frames under its current config (upper bound, incl. alignment)
size_t phovo_internal_slot_bytes(const phovo_ctx* ctx, int rows, int cols);

#endif
