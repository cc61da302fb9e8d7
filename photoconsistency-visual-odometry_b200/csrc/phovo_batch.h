// phovo_batch.h -- parameter block and launchers of the batched (one CTA per pair) path.
#ifndef PHOVO_BATCH_H_
#define PHOVO_BATCH_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include "phovo_internal.h"

namespace phovo {

constexpr int kBatchThreads = 480;          // 15 warps, 128 registers per thread; 480 is a multiple of the level widths 160 / 80 / 40 / 20 (640x480) and 240 / 120 / 60 (8K, 960-wide)
constexpr int kBatchThreadsSmall = 160;      // small levels: 3 CTAs of 5 warps per SM (160 is a multiple of 80 / 40 / 20)
constexpr int kBatchSmallLevelPixels = 6400; // largest level that runs 3 CTAs per SM
constexpr int kBatchMaxLevelPixels = 22528; // 10 B/px of shared memory + tables + scratch must fit 227 KB (checked exactly
                                            // by the host); also <= 64 * kBatchThreads (validity mask) and < 65535

// The level kernel prefetches D0 / D32 / I0 up to 8 * kBatchThreads pixels past the end of a level without
// bounds guards (the values are masked); the allocation behind the last record must cover that.
constexpr size_t kBatchStoreSlackBytes = 8 * (size_t)kBatchThreads * sizeof(double) + 1024;

// Everything the two batch kernels need, passed by value (__grid_constant__).
struct BatchParams {
  int num_pairs, rows, cols;
  int num_active;                       // active levels, coarse -> fine
  int mode;
  int log_cap;                          // per-pair stats slots (0: do not record)
  int exact_always;                     // test hook: every pixel takes the exact warp (no estimate shortcut)
  int force_generic;                    // test hook: generic (r, c) bookkeeping even when BT % cols == 0
  int src_period, src_keep_begin, src_keep;   // row compaction of staged inputs (src_period 0: dense frames)
  int level[PHOVO_MAX_LEVELS];          // pyramid level index of active level a
  int lrows[PHOVO_MAX_LEVELS], lcols[PHOVO_MAX_LEVELS];
  int max_iters[PHOVO_MAX_LEVELS];
  int px_offset[PHOVO_MAX_LEVELS + 1];  // prefix sum of level pixel counts (pyramid kernel indexing)
  unsigned long long off_I0[PHOVO_MAX_LEVELS], off_I1[PHOVO_MAX_LEVELS], off_D0[PHOVO_MAX_LEVELS];
  unsigned long long off_D32[PHOVO_MAX_LEVELS];   // fp32 copy of D0, 0 where the depth fails the range test (phase A's estimate)
  unsigned long long record_bytes;      // bytes of one pair's packed level record in HBM
  double fx[PHOVO_MAX_LEVELS], fy[PHOVO_MAX_LEVELS], ox[PHOVO_MAX_LEVELS], oy[PHOVO_MAX_LEVELS];
  double inv_fx[PHOVO_MAX_LEVELS], inv_fy[PHOVO_MAX_LEVELS];
  double lambda[PHOVO_MAX_LEVELS], min_grad[PHOVO_MAX_LEVELS];
  double grad_k[PHOVO_MAX_LEVELS];      // imageGradientsScalingFactor / 1020
  double min_depth, max_depth;
};

// K1b: all active pyramid levels of I0, I1 (as exact u16 tap sums) and D0 (fp64) for every pair,
// one pass over the full-resolution inputs.  depth_type: SRC_F64 / SRC_F32 / SRC_U16.
int launch_batch_pyramid(cudaStream_t stream, const BatchParams& bp, const uint8_t* gray0, const void* depth0,
                         int depth_type, double depth_scale, const uint8_t* gray1, uint8_t* store);
// K3-batch: persistent CTAs, one pair at a time per CTA, the level's images resident in shared
// memory, the whole Gauss-Newton loop of the level on chip; one launch per active level.
// Returns the number of launches.  `next_pair`: PHOVO_MAX_LEVELS zeroed device counters.
int launch_batch_align(cudaStream_t stream, const BatchParams& bp, int sm_count, const uint8_t* store,
                       const double* init_states, double* states, int32_t* iters, phovo_iter_stats* log,
                       int32_t* log_counts, unsigned int* next_pair);
size_t batch_level_smem_bytes(int rows, int cols);

// Normal equations at given states for a chunk of pairs at one pyramid level (kernels_eval.cu).  Level 0 reads the
// caller's dense frames; a level >= 1 reads the records k_batch_pyramid wrote for a BatchParams with that one level.
constexpr int kEvalThreads = 256, kEvalPix = 8, kEvalTile = kEvalThreads * kEvalPix;   // pixels per tile: fixed
struct EvalLevel {
  LevelParams L;                         // K / 2^level, depth range, rows / cols of the level (rows * cols < 2^31)
  double grad_k;                         // imageGradientsScalingFactor / 1020 (gradients from integer tap sums)
  int tiles;                             // ceil(rows * cols / kEvalTile)
  const uint8_t* gray0; const uint8_t* gray1; const void* depth; double depth_scale;   // level 0: [pairs][n] of pair 0
  const uint8_t* store; unsigned long long record_bytes, off_I0, off_I1, off_D0;       // level >= 1: records of pair 0
  const PoseDev* poses;                  // [pairs]
  uint32_t* keys;                        // [pairs][n]: source index + 1 of the winner, 0 = none; zero on entry and exit
  uint8_t* valid;                        // [pairs][n]: the exact warp accepted the source pixel
  double* partials;                      // [pairs][tiles][PHOVO_ACC_STRIDE]
};
// Photometric + depth solver (PHOVO_MODE_BIOBJECTIVE): the target depth of a chunk at the level, and what the kernels
// derive from it.  The level images are built from the caller's full-resolution frames with the per-pair path's
// arithmetic (phovo_level.cuh), so D1, GxD and GyD are the per-pair context's bits.
struct EvalTargetDepth {
  const void* depth1;                    // [pairs][rows][cols] of pair 0, full resolution, element type of depth0
  int rows, cols, level;                 // full-resolution size, pyramid level
  double depth_scale;                    // u16 only (1 otherwise)
  double inv_max_depth;                  // 1 / max_depth: GxD, GyD are the Scharr of D1 / max_depth (BiObjective.h:224-237)
  double ks0, ks1;                       // Scharr kernel scaled by the level's imageGradientsScalingFactor
  int tiles2;                            // ceil(2 rows * cols / kEvalTile) at the level: tiles of the 2N residual slots
  double* D1; double* GxD; double* GyD;  // [pairs][n] at the level
  double* sums;                          // [pairs][tiles][2]: sum of the I1 tap sums, sum of D1 per tile of pixels
  double* gain;                          // [pairs]: mean(I1) / mean(D1) at the level (BiObjective.h:299)
};

// Pose (rotation and trig values) of every state, as the per-pair path derives it: poses[p] from states[p * 6].
int launch_eval_poses(cudaStream_t stream, const double* states, int num_pairs, PoseDev* poses);
// Winner pass, accumulate pass (clears the keys) and the per-pair sums into H [21], g [6], cost, num_valid of pairs
// [0, num_pairs) of E; `out_*` point at the chunk's first pair.  Returns the number of launches.
int launch_eval_normal_equations(cudaStream_t stream, const EvalLevel& E, int src_type /* SRC_*; level 0 */, bool records,
                                 int num_pairs, double* out_H, double* out_g, double* out_cost, int32_t* out_valid);
// The same for the photometric + depth solver: target depth set-up, gain, winner pass over 2N slots (E.keys [pairs][2n]),
// accumulate pass over the 2N Jacobian rows (E.partials [pairs][D.tiles2]) and the per-pair sums.
int launch_eval_normal_equations_bi(cudaStream_t stream, const EvalLevel& E, const EvalTargetDepth& D, int src_type, bool records,
                                    int num_pairs, double* out_H, double* out_g, double* out_cost, int32_t* out_valid);
bool batch_level_is_small(int rows, int cols);
cudaError_t batch_align_prepare();

}  // namespace phovo
#endif
