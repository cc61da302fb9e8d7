// phovo_kernels.h -- host-callable launchers of the CUDA kernels (one per kernel family).
// Every launcher enqueues on `stream`, returns the number of kernels it launched and never
// synchronises.  Error checking is done by the caller with cudaGetLastError().
#ifndef PHOVO_KERNELS_H_
#define PHOVO_KERNELS_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include "phovo_internal.h"
#include "phovo_lm.h"

namespace phovo {

// ---- frame setup (kernels_pyramid.cu) --------------------------------------------------------
enum SrcType { SRC_U8 = 0, SRC_F64 = 1, SRC_F32 = 2, SRC_U16 = 3 };

// K1: one pyramid level straight from the full-resolution source image (cv::resize INTER_LINEAR
// by 2^-level from the ORIGINAL, AN:132) with the element conversion fused in
// (u8 * 1/255, AN:471; u16 * depth_scale).  Output fp64 scratch (orows x ocols, dense).
int launch_build_level(cudaStream_t stream, const void* src, int src_type, size_t src_step_bytes,
                       double src_scale, int rows, int cols, int level, double* dst, int orows, int ocols);
// K1 (+K2) for every active level of a frame in ONE launch: `dst` (and, with `gradients`, the Scharr
// images `gx`, `gy` with the kernel scaled by grad_scale: ks0 = 3 s, ks1 = 10 s) of each listed level.
// Same arithmetic as launch_build_level + launch_scharr_store, bit for bit; not for blurred levels.
struct PyramidLevels {
  int num;                                  // levels listed
  int level[PHOVO_MAX_LEVELS];              // pyramid level index
  int orows[PHOVO_MAX_LEVELS], ocols[PHOVO_MAX_LEVELS];
  int px_offset[PHOVO_MAX_LEVELS + 1];      // prefix sum of orows * ocols
  double* dst[PHOVO_MAX_LEVELS];
  double* gx[PHOVO_MAX_LEVELS]; double* gy[PHOVO_MAX_LEVELS];
  double ks0[PHOVO_MAX_LEVELS], ks1[PHOVO_MAX_LEVELS];
};
int launch_build_levels(cudaStream_t stream, const void* src, int src_type, size_t src_step_bytes, double src_scale,
                        int rows, int cols, const PyramidLevels& P, bool gradients);
// K2b: cv::GaussianBlur(k x k, sigma) applied once, BORDER_REFLECT_101, fp64 in place via `tmp`.
int launch_gaussian_blur(cudaStream_t stream, double* img, double* tmp, int rows, int cols, int ksize, double sigma);
// dst = src * alpha (Mat::convertTo with a scale), and gain[0] = mean(a) / mean(b) in a fixed summation order
int launch_scale(cudaStream_t stream, const double* src, double alpha, double* dst, size_t n);
int launch_mean_ratio(cudaStream_t stream, const double* a, const double* b, size_t n, double* out);
// K2: Scharr x/y (AN:181-187) from the fp64 level image, same evaluation order as cv::Scharr.
int launch_scharr_store(cudaStream_t stream, const double* img, int rows, int cols, double scale,
                        double* Gx, double* Gy);

// phovo::warpImage (BASE:73-134) for a chunk of pairs of one size.  Device pointers of pair 0; `*_step` bytes between
// rows, `*_pair` bytes between pairs.  warped / target / diff / num_landed / sum_abs_diff may be NULL (diff and
// sum_abs_diff need target); num_landed / sum_abs_diff are added to, so they start at zero.
struct WarpImages {
  int rows, cols;                       // rows * cols < 2^31
  const uint8_t* gray; size_t gray_step, gray_pair;
  const void* depth; size_t depth_step, depth_pair; double depth_scale;   // depth_scale: u16 only
  const double* rts;                    // [pairs][16] row-major 4x4
  const uint8_t* target; size_t target_step, target_pair;
  uint8_t* warped; size_t warped_step, warped_pair;
  uint8_t* diff; size_t diff_step, diff_pair;
  int32_t* num_landed; int64_t* sum_abs_diff;   // [pairs]
};
struct WarpIntrinsics { double fx, fy, ox, oy, inv_fx, inv_fy; };   // K / 2^level (BASE:89-94)
// Splat: key = source linear index + 1, u32 atomicMax per target pixel (raster-order last writer wins).  Resolve:
// gray[key - 1], |target - warped|, per-pair count of landed pixels and sum of their |target - warped|.  `keys`
// [num_pairs][rows * cols] must be zero on entry; with `clear_keys` the resolve leaves them zero again.
int launch_warp_images(cudaStream_t stream, const WarpImages& W, int depth_type /* SRC_* */, const WarpIntrinsics& I,
                       int num_pairs, uint32_t* keys, bool clear_keys);

// ---- alignment (kernels_align.cu) ------------------------------------------------------------
struct LevelPtrs {
  const double* I0; const double* D0; const double* I1; const double* Gx; const double* Gy;
  int* winner;        // rows*cols ints, all -1 between iterations
  unsigned char* valid;  // rows*cols flags written by K3a: pixel is depth-valid and lands in bounds under the current pose
  // photometric + depth solver only (PHOVO_MODE_BIOBJECTIVE); winner then has 2*rows*cols slots
  const double* D1; const double* GxD; const double* GyD; const double* gain;
};

// Batch wave path (phovo_batch.cu): a SLOT is the device side of a child context -- the pyramids of one pair, its
// winner map, its PoseDev.  k_align_slots runs one CTA per slot through every active level (coarse to fine).
struct SlotArgs {
  LevelPtrs P[PHOVO_MAX_LEVELS];
  PoseDev* pose;
  double* partials;              // one row of PHOVO_ACC_STRIDE doubles is used
};
struct SlotLevels {               // kernel parameter: the active levels, coarse to fine (the same for every slot)
  int count;
  LevelParams L[PHOVO_MAX_LEVELS];
  LmParams lm[PHOVO_MAX_LEVELS];  // Ceres mode only
};
int launch_align_slots(cudaStream_t stream, int mode, const SlotLevels& LS, const SlotArgs* slots, int num_slots, const double* init_states,
                       int cluster /* CTAs per slot: 1, 2, 4 or 8 */);   // < 0: the launch failed
int launch_gather_slots(cudaStream_t stream, const SlotArgs* slots, int num_slots, double* states, int32_t* iters);

int launch_set_state(cudaStream_t stream, PoseDev* pose, const double* state_dev_or_null, const double state_host[6], int log_capacity);
int launch_begin_level(cudaStream_t stream, PoseDev* pose, int max_iters);
// K3a + K3b (+ optional dense residual / Jacobian dump) for one iteration; respects pose->done.
// partials: [grid][PHOVO_ACC_STRIDE] doubles.  Returns kernels launched; *grid_out = blocks of K3b.
int launch_iteration_kernels(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, const PoseDev* pose,
                             double* partials, int sm_count, int* grid_out, double* dump_res, double* dump_jac,
                             bool clear_winner_first);
// blocks the per-pixel kernels may use on a device with `sm_count` SMs = rows of `partials` to allocate
int partials_blocks(int sm_count);
// What the launchers of the persistent kernels cache per DEVICE (function attributes are per device
// and per function; a context lives on one device, so the cache lives in the context).
struct LaunchState {
  int coop_blocks_per_sm[5] = {-1, -1, -1, -1, -1};   // k_level_coop<0>, <1>, <3>, and the row-sharded <0>, <1>
  int ceres_blocks_per_sm = -1;
  bool cluster_prepared[2] = {false, false};  // k_level_cluster<0>, <1>
};
// K4: fixed-order sum of the partials, 6x6 solve, state update, termination test, stats log.
// cond_handle != 0: also drives the CUDA-graph WHILE node (cudaGraphSetConditional).
int launch_reduce_solve(cudaStream_t stream, const LevelParams& L, PoseDev* pose, const double* partials, int grid,
                        phovo_iter_stats* log, unsigned long long cond_handle);
// evaluation only: totals -> stats entry `out` (device), no step
int launch_reduce_only(cudaStream_t stream, const LevelParams& L, const PoseDev* pose, const double* partials, int grid,
                       phovo_iter_stats* out);
// row-sharded variant: totals -> 32-double buffer, then solve from the (all-reduced) buffer
int launch_reduce_to_buffer(cudaStream_t stream, const double* partials, int grid, double* buffer);
int launch_solve_from_buffer(cudaStream_t stream, const LevelParams& L, PoseDev* pose, const double* buffer,
                             phovo_iter_stats* log);
int launch_fill_i32(cudaStream_t stream, int* p, int value, size_t n, int sm_count);
// persistent cooperative kernel: the whole iteration loop of one level in one launch (analytic modes)
struct ShardExchange;
// peers_dev != nullptr and world > 1: the row-sharded loop (L.row_begin / row_end = this rank's band) with the sums
// exchanged inside the kernel over NVLink peer memory; epochs epoch_base + 1 ... epoch_base + L.max_iters are used.
int launch_level_coop(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, PoseDev* pose, double* partials,
                      phovo_iter_stats* log, LaunchState* ls, int sm_count, int* grid_out, cudaError_t* err,
                      ShardExchange* const* peers_dev = nullptr, int rank = 0, int world = 1, unsigned long long epoch_base = 0,
                      const double* level_dmin = nullptr);
// out[0] = the smallest depth of the level inside (lo, hi) (+inf / all-ones bits if there is none): the row-sharded loop
// bounds how far a pixel can move between rows with it
int launch_min_valid_depth(cudaStream_t stream, const double* D, int n, double lo, double hi, double* out, int sm_count);

// thread-block-cluster kernel for small levels (analytic modes, <= 8 192 px): the loop of one level inside ONE
// cluster of 16 CTAs, winner map in distributed shared memory.  Returns 1 (launched), 0 (level does not
// qualify: use launch_level_coop), -1 (launch error in *err).
int launch_level_cluster(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, PoseDev* pose, phovo_iter_stats* log, LaunchState* ls, cudaError_t* err);

// Ceres mode: the restated LM loop of one level (phovo_lm.h) in one cooperative launch.
int launch_level_coop_ceres(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, PoseDev* pose, double* partials,
                            phovo_iter_stats* log, const LmParams& lm, LaunchState* ls, int sm_count, cudaError_t* err);

// Exchange area of the fused peer-store all-reduce (one per rank, IPC-shared with the peers).
struct ShardExchange {
  double slots[2][8][32];              // [epoch parity][writer rank][value]
  unsigned long long flags[8];         // flags[w] = last epoch rank w has delivered here
  int error;                           // set when a wait timed out
  int pad;
};
// totals of the local partials -> st.global into every peer's slots -> release flags -> wait for the
// peers -> sum the `world` slots in rank order into `buffer` (32 doubles).
int launch_reduce_exchange(cudaStream_t stream, const PoseDev* pose, const double* partials, int grid, double* buffer,
                           ShardExchange* const* peers_dev /* device array [world] */, int rank, int world,
                           unsigned long long epoch);

}  // namespace phovo
#endif
