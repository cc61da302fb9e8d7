/*
 * phovo_b200.h -- C ABI of the B200-native photoconsistency alignment path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch/OpenCV/Eigen types.
 * Every entry point names the reference interface it replaces (paths are relative to the
 * reference tree, MiguelAlgaba/photoconsistency-visual-odometry):
 *
 *   AN  = phovo/include/CPhotoconsistencyOdometryAnalytic.h
 *   CE  = phovo/include/CPhotoconsistencyOdometryCeres.h
 *   BASE= phovo/include/CPhotoconsistencyOdometry.h
 *
 * The C++ adapter `include/CPhotoconsistencyOdometryCuda.h` wraps this ABI behind the
 * reference's own `CPhotoconsistencyOdometry<TPixel,TCoordinate>` virtual interface
 * (BASE:137-179); INTEGRATION.md shows the three-line change in the reference apps.
 *
 * Conventions
 *   - every function returns 0 on success or a negative PHOVO_E_* code; nothing throws or
 *     unwinds across this boundary; `phovo_last_error(ctx)` returns a static/ctx-owned text.
 *   - a context owns one CUDA device + one stream; it is not thread-safe; contexts are
 *     independent (the reference object is single-threaded too, AN:80-113).
 *   - all input buffers are borrowed for the duration of the call only (the reference aliases
 *     the depth buffer, AN:136; we always copy).
 *   - the library has no CPU compute path: if no CUDA device can be opened phovo_create fails.
 */
#ifndef PHOVO_B200_H_
#define PHOVO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHOVO_MAX_LEVELS 10

/* error codes */
#define PHOVO_OK 0
#define PHOVO_E_INVALID   (-1) /* bad argument / call order                            */
#define PHOVO_E_CUDA      (-2) /* CUDA runtime error (text in phovo_last_error)        */
#define PHOVO_E_CONFIG    (-3) /* YAML file missing / malformed                         */
#define PHOVO_E_NOMEM     (-4)
#define PHOVO_E_UNSUPPORTED (-5) /* e.g. batch kernel asked for a level that does not fit SMEM */
#define PHOVO_E_NUMERIC   (-6) /* non-finite state after Optimize (reference would print NaN) */

/* solver variants */
#define PHOVO_MODE_ANALYTIC_REF   0 /* bug-compatible with AN:253 (temp11 = cos*cos + x), default */
#define PHOVO_MODE_ANALYTIC_FIXED 1 /* Maxima-exact Jacobian (phovo/Maxima/derivatives_photoconsistency.wxm) */
#define PHOVO_MODE_CERES          2 /* CE:156-269 residual (bilinear, truncation scatter) + restated LM */
#define PHOVO_MODE_BIOBJECTIVE    3 /* CPhotoconsistencyOdometryBiObjective.h:242-452: photometric + depth rows,
                                       including its row aliasing (depth rows at 2*i collide with intensity rows at i) */

/* depth element types accepted at the boundary */
#define PHOVO_DEPTH_F64 0 /* cv::Mat_<double>, what both reference apps pass */
#define PHOVO_DEPTH_F32 1
#define PHOVO_DEPTH_U16 2 /* raw sensor units; metres = raw * depth_scale (apps: 1/1000, 1/5000) */

/*
 * All run-time parameters of the path, POD.  Fields mirror the members the reference reads from
 * YAML (AN:581-607, CE:526-576) and its constructor defaults (AN:430-443).
 * Per-level arrays are indexed by pyramid level, 0 = full resolution.
 */
typedef struct phovo_config {
  int32_t mode;                                  /* PHOVO_MODE_*                                     */
  int32_t num_levels;                            /* numOptimizationLevels                            */
  int32_t blur_filter_size[PHOVO_MAX_LEVELS];    /* "blurFilterSize (at each level)"                 */
  int32_t max_num_iterations[PHOVO_MAX_LEVELS];  /* "max_num_iterations (at each level)"             */
  double  grad_scale[PHOVO_MAX_LEVELS];          /* "imageGradientsScalingFactor (at each level)"    */
  double  lambda_step[PHOVO_MAX_LEVELS];         /* "lambda_optimization_step (at each level)"       */
  double  min_gradient_norm[PHOVO_MAX_LEVELS];   /* "min_gradient_norm (at each level)"              */
  double  min_depth;                             /* SetMinDepth, default 0.3 (AN:430)                */
  double  max_depth;                             /* SetMaxDepth, default 5.0 (AN:430)                */
  int32_t visualize_iterations;                  /* parsed, ignored (GUI only, AN:551-557)           */
  /* Ceres-mode options (CE:464-477); unused by the analytic modes */
  double  function_tolerance[PHOVO_MAX_LEVELS];
  double  gradient_tolerance[PHOVO_MAX_LEVELS];
  double  parameter_tolerance[PHOVO_MAX_LEVELS];
  double  initial_trust_region_radius[PHOVO_MAX_LEVELS];
  double  max_trust_region_radius[PHOVO_MAX_LEVELS];
  double  min_trust_region_radius[PHOVO_MAX_LEVELS];
  double  min_relative_decrease[PHOVO_MAX_LEVELS];
  int32_t num_threads;                           /* parsed, unused on the GPU                        */
  int32_t num_linear_solver_threads;             /* parsed, unused                                   */
  int32_t minimizer_progress_to_stdout;          /* parsed, unused                                   */
  int32_t reserved;
} phovo_config;

/*
 * One Gauss-Newton (or LM) iteration as executed -- the parity hook.  H holds the 21 unique
 * entries of J^T J in row-major upper-triangular order (00 01 .. 05 11 12 .. 55); g = J^T r.
 * `state_in` is the state the normal equations were evaluated at, `state_out` the state after
 * the step (AN:538-540).  For Ceres mode `cost` = 0.5*|r|^2 and `accepted`/`radius` describe
 * the LM step; analytic modes set cost = 0.5*|r|^2 too (not used by the reference).
 */
typedef struct phovo_iter_stats {
  int32_t level;
  int32_t iteration;      /* 0-based within the level */
  int32_t num_valid;      /* source pixels that were depth-valid and projected in bounds */
  int32_t accepted;       /* LM: step accepted; GN: always 1 */
  double  H[21];
  double  g[6];
  double  grad_norm;      /* |g|_2, the quantity TestTerminationCriteria thresholds (AN:380) */
  double  cost;
  double  radius;         /* LM trust-region radius used for this step (0 for GN) */
  double  state_in[6];
  double  state_out[6];
} phovo_iter_stats;

typedef struct phovo_ctx phovo_ctx;

/* ---- life cycle ------------------------------------------------------------------------- */
/* Replaces constructing phovo::Analytic::CPhotoconsistencyOdometryAnalytic<uchar,double>
 * (AN:430-443: defaults 5 levels, iterations {0,0,5,20,50}, grad scale 0.0625, lambda 1,
 * min gradient norm 300, depth range (0.3, 5.0)). */
int phovo_create(int device, phovo_ctx** out);
int phovo_destroy(phovo_ctx* ctx);
const char* phovo_last_error(const phovo_ctx* ctx); /* ctx may be NULL: text of the last create failure */
const char* phovo_version(void);

/* ---- configuration ---------------------------------------------------------------------- */
int phovo_config_default(phovo_config* cfg);                       /* AN:430-443                */
int phovo_set_config(phovo_ctx* ctx, const phovo_config* cfg);
int phovo_get_config(const phovo_ctx* ctx, phovo_config* cfg);
/* ReadConfigurationFile (AN:581-607, CE:526-576).  `mode` of the context is kept; Ceres keys are
 * read when present.  Missing per-level entries repeat the last given one (the reference reads
 * past the vector, CE:473 with config_5_level_optimization_ceres.yml:11). */
int phovo_load_config_yaml(phovo_ctx* ctx, const char* path);
/* context-free parser, usable without a GPU */
int phovo_parse_config_yaml(const char* path, phovo_config* cfg, char* err, size_t err_len);
int phovo_set_mode(phovo_ctx* ctx, int mode);
/* SetMinDepth / SetMaxDepth (AN:448-457) */
int phovo_set_depth_range(phovo_ctx* ctx, double min_depth, double max_depth);
/* SetIntrinsicMatrix (AN:460-463): row-major 3x3; only K[0],K[2],K[4],K[5] are read (AN:204-207) */
int phovo_set_intrinsics(phovo_ctx* ctx, const double K[9]);

/* ---- frames ----------------------------------------------------------------------------- */
/* SetSourceFrame (AN:466-476): gray u8 rows x cols with byte stride gray_step; depth in metres
 * (F64/F32) or raw u16 * depth_scale, byte stride depth_step.  Uploads and builds the intensity and
 * depth pyramids on the device.  Host pointers may be pageable or pinned; device pointers are
 * accepted too (detected with cudaPointerGetAttributes) and are read in place.
 * Ownership, every frame entry point: inputs are borrowed for the duration of the call only -- when
 * it returns, host buffers have been copied and kernels reading a DEVICE buffer have completed, so
 * the caller may overwrite or free it.  Stream contract for device inputs: the work runs on the
 * context's stream (its own non-blocking stream unless phovo_set_stream was called), which is NOT
 * ordered after whatever produced the buffer.  Either pass the producer's stream to
 * phovo_set_stream first, or synchronise the producer before the call. */
int phovo_set_source(phovo_ctx* ctx, const uint8_t* gray, size_t gray_step,
                     const void* depth, int depth_type, size_t depth_step, double depth_scale,
                     int rows, int cols);
/* SetTargetFrame (AN:479-491): the reference ignores the target depth (only .type(), AN:484);
 * builds the I1 pyramid and the Scharr gradient pyramids (AN:165-189). */
int phovo_set_target(phovo_ctx* ctx, const uint8_t* gray, size_t gray_step, int rows, int cols);
/* Target depth (metres), needed by PHOVO_MODE_BIOBJECTIVE only -- the analytic and Ceres solvers ignore
 * it like the reference does.  Call after phovo_set_target with the same frame size: builds the target
 * depth pyramid, the Scharr pyramids of depth / max_depth and the per-level gain mean(I1)/mean(D1)
 * (CPhotoconsistencyOdometryBiObjective.h:213-239, 299, 567-579). */
int phovo_set_target_depth(phovo_ctx* ctx, const void* depth, int depth_type, size_t depth_step, double depth_scale);
/* VO loop helper (apps/PhotoconsistencyVisualOdometry/PhotoconsistencyVisualOdometry.cpp:222-223,256):
 * the previous target's intensity pyramid becomes the source intensity pyramid on the device;
 * only the depth of that frame has to be supplied. */
int phovo_promote_target_to_source(phovo_ctx* ctx, const void* depth, int depth_type,
                                   size_t depth_step, double depth_scale);

/* ---- solve ------------------------------------------------------------------------------ */
int phovo_set_initial_state(phovo_ctx* ctx, const double state[6]);  /* AN:494-497 x y z yaw pitch roll */
int phovo_optimize(phovo_ctx* ctx);                                  /* AN:500-563 / CE:433-500, blocking */
int phovo_get_state(const phovo_ctx* ctx, double state[6]);          /* AN:566-569 */
int phovo_get_rt(const phovo_ctx* ctx, double rt[16]);               /* AN:572-578 + BASE:47-71, row-major 4x4 */
/* state -> 4x4, usable without a context (BASE:47-71) */
void phovo_state_to_rt(const double state[6], double rt[16]);

/* ---- diagnostics the apps compute after Optimize ----------------------------------------- */
/* phovo::warpImage (BASE:73-134) + the cv::absdiff both apps show (FrameAlignment.cpp:107-110,
 * VisualOdometry.cpp:247-252): forward-splat the source intensities through depth, Rt (row-major
 * 4x4) and K / 2^level into `warped` (zero where nothing lands; truncating cast BASE:119-122,
 * raster-order last writer wins); if `target` and `diff` are given also diff = |target - warped|.
 * Host or device pointers; strides in bytes; depth as in phovo_set_source. */
int phovo_warp_image(phovo_ctx* ctx, const uint8_t* gray, size_t gray_step,
                     const void* depth, int depth_type, size_t depth_step, double depth_scale,
                     int rows, int cols, const double rt[16], const double K[9], int level,
                     uint8_t* warped, size_t warped_step,
                     const uint8_t* target, size_t target_step, uint8_t* diff, size_t diff_step);

/* ---- introspection (parity hooks; not in the reference) --------------------------------- */
int phovo_num_iter_stats(const phovo_ctx* ctx);
int phovo_get_iter_stats(const phovo_ctx* ctx, int index, phovo_iter_stats* out);
/* which: 0 I0, 1 D0, 2 I1, 3 Gx1, 4 Gy1.  dst may be NULL to query the size. */
int phovo_get_level_image(phovo_ctx* ctx, int which, int level, double* dst, int* rows, int* cols);
/* Evaluate the normal equations once at `state` on `level` without stepping (fills H,g,cost,num_valid). */
int phovo_eval_normal_equations(phovo_ctx* ctx, int level, const double state[6], phovo_iter_stats* out);
/* Parity hook: residual vector and Jacobian (row-major, 6 doubles per row) at `state` on `level`, with
 * rows*cols rows of that level in the analytic and Ceres modes (CE:156-269) and 2*rows*cols rows in
 * PHOVO_MODE_BIOBJECTIVE, which stacks the depth rows under the intensity rows (BI:422-452): the residual
 * buffer takes rows*cols or 2*rows*cols doubles, the Jacobian buffer six times that.  Either may be NULL. */
int phovo_eval_residuals(phovo_ctx* ctx, int level, const double state[6], double* residuals, double* jacobian);
/* device time of the last phovo_optimize / frame setup in milliseconds (CUDA events) */
int phovo_get_timings(const phovo_ctx* ctx, float* setup_ms, float* optimize_ms);
/* number of kernels this context has launched so far */
int64_t phovo_launch_count(const phovo_ctx* ctx);
/* use a caller-provided stream (e.g. torch's current stream) instead of the ctx-owned one; required
 * for ordering when device-resident inputs are produced on that stream (see phovo_set_source) */
int phovo_set_stream(phovo_ctx* ctx, void* cuda_stream);
/* enable != 0: path 1 of phovo_set_execution (whole Optimize as one CUDA graph with a conditional
 * WHILE node per level, no host sync inside); 0: path 0 (plain stream launches with host-side
 * convergence polling).  The default is path 2, see phovo_set_execution. */
int phovo_set_use_graph(phovo_ctx* ctx, int enable);
/* How phovo_optimize drives the iteration loop of a level (results agree to rounding; each path is
 * bitwise reproducible run to run):
 *   3           as 2, but a small level (analytic solvers, <= 8 192 px) runs inside ONE thread-block cluster
 *               of 16 CTAs: winner map in distributed shared memory, cluster barriers instead of grid barriers
 *   2 (default) one persistent cooperative kernel per level, grid-wide barriers between the phases
 *   1           one CUDA graph for the whole Optimize with a conditional WHILE node per level
 *   0           plain stream launches, the host polls the termination flag every 4 iterations
 * phovo_set_use_graph(ctx, e) is shorthand for path e ? 1 : 0.  If a path is not available on the
 * device the next one down is used (phovo_graph_error tells why). */
int phovo_set_execution(phovo_ctx* ctx, int path);
int phovo_last_optimize_path(const phovo_ctx* ctx);
/* 1 if the last phovo_optimize ran as the CUDA graph (path 1), else 0 */
int phovo_last_optimize_used_graph(const phovo_ctx* ctx);
/* why the last path that failed on this context (graph, cooperative or cluster launch) was given up; "" if none */
const char* phovo_graph_error(const phovo_ctx* ctx);
/* build every pyramid level, not only those with max_num_iterations > 0 (the reference builds all,
 * AN:474-490, but never reads the others); needed only to inspect them with phovo_get_level_image */
int phovo_set_build_all_levels(phovo_ctx* ctx, int enable);

/* ---- batch of independent pairs (extension; BASELINE config "4096 pairs, sharded by pair") ---- */
/* All pairs share rows/cols/intrinsics/config.  Inputs are strided arrays of `num_pairs` frames:
 * gray0/gray1 u8 [P][rows][cols], depth0 [P][rows][cols] of depth_type.  Pointers may be host
 * (pinned recommended) or device.  Results: states[P][6] doubles, iterations[P][PHOVO_MAX_LEVELS] int32
 * (executed GN iterations per level), both host pointers (may be NULL). */
int phovo_batch_align(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                      const uint8_t* gray0, const void* depth0, int depth_type, double depth_scale,
                      const uint8_t* gray1,
                      const double* initial_states /* [P][6] or NULL = zeros */,
                      double* states, int32_t* iterations);
/* Which implementation the last batch call took: 1 = the shared-memory-resident batch kernels (analytic solvers, no blur,
 * active levels up to ~22 K px: one streaming pyramid pass + one persistent launch per level).  Everything else
 * (Ceres-mode and photometric + depth solver, blurred levels, larger levels): 3 = WAVES of per-pair slots -- the pyramids
 * of a wave are built with the general path's kernels, then one launch aligns the whole wave, one CTA per pair through
 * every level and iteration (a thread-block cluster of 2 / 4 / 8 CTAs per pair while the wave is too small to fill the
 * GPU) -- for batches of 16 (Ceres-mode) / 24 (other solvers) pairs or more; 2 = smaller batches: the pairs go one by one through the general path on a pool of per-pair contexts, one
 * host thread each -- bitwise the results of a loop over the per-pair API.  Paths 2 and 3 give the same iteration counts
 * and states equal up to the grouping of the partial sums (last bits). */
int phovo_batch_last_path(const phovo_ctx* ctx);
/* phovo_batch_align for the photometric + depth solver (PHOVO_MODE_BIOBJECTIVE), which also reads the TARGET depth
 * (depth1 [P][rows][cols], same type / scale as depth0; BiObjective.h:567-579).  Other modes ignore depth1. */
int phovo_batch_align_with_target_depth(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                                        const uint8_t* gray0, const void* depth0, int depth_type, double depth_scale,
                                        const uint8_t* gray1, const void* depth1,
                                        const double* initial_states, double* states, int32_t* iterations);
/* Same work with device-resident inputs and outputs left on the device (states_dev [P][6] f64,
 * iters_dev [P][PHOVO_MAX_LEVELS] i32); asynchronous on the context stream. */
int phovo_batch_align_device(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                             const uint8_t* gray0_dev, const void* depth0_dev, int depth_type,
                             double depth_scale, const uint8_t* gray1_dev,
                             const double* initial_states_dev, double* states_dev, int32_t* iters_dev);
/* phovo_batch_align_device for the photometric + depth solver (PHOVO_MODE_BIOBJECTIVE), which also reads the TARGET
 * depth depth1_dev ([P][rows][cols] on the device, same type / scale as depth0_dev).  In that mode the pairs run through
 * the pool (< 24 pairs) or the slot waves, as phovo_batch_align_with_target_depth takes them, and the call returns once
 * the results are in states_dev / iters_dev.  Other modes ignore depth1_dev and forward to phovo_batch_align_device. */
int phovo_batch_align_device_with_target_depth(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                                               const uint8_t* gray0_dev, const void* depth0_dev, int depth_type,
                                               double depth_scale, const uint8_t* gray1_dev, const void* depth1_dev,
                                               const double* initial_states_dev, double* states_dev, int32_t* iters_dev);
/* per-pair per-iteration stats of the last batch call (only recorded when enabled: costs HBM; what the resident
 * kernels do not take then goes through the pool of per-pair contexts, whose logs these are) */
int phovo_batch_set_record_stats(phovo_ctx* ctx, int enable);
int phovo_batch_get_iter_stats(const phovo_ctx* ctx, int pair, int index, phovo_iter_stats* out);
int phovo_batch_num_iter_stats(const phovo_ctx* ctx, int pair);
/* test hooks of the batch kernel (results must not change): bit 0 = every pixel takes the exact
 * reference warp instead of the estimate-then-verify shortcut; bit 1 = use the generic
 * thread->pixel bookkeeping even when the CTA width is a multiple of the level width; bit 2 / bit 3 = what the
 * resident kernels do not take goes through the pool of per-pair contexts / the slot waves whatever the batch size;
 * bit 4 = the warpImage entries clear their splat keys with a memset per chunk instead of in the resolve pass */
int phovo_batch_set_debug_flags(phovo_ctx* ctx, int flags);
/* phovo::warpImage (BASE:73-134) + the apps' cv::absdiff for P pairs of one size and intrinsics.
 * gray0 / depth0 / gray1 are dense [P][rows][cols], all host or all device (as phovo_batch_align);
 * rts [P][16] row-major 4x4 (host or device) as phovo_state_to_rt / phovo_get_rt return them;
 * outputs may each be NULL, host or device: warped / diff [P][rows][cols] u8,
 * num_landed [P] (source pixels that landed in the target), sum_abs_diff [P] (sum of
 * |gray1 - warped| over those pixels).  diff and sum_abs_diff need gray1.  Blocking.
 * Every image equals what phovo_warp_image gives pair by pair, bit for bit; the summaries are integer sums, the same
 * whatever the chunking.  A source pixel of gray 0 that lands counts in num_landed although `warped` cannot show it.
 * PHOVO_E_INVALID: bad sizes or level, unknown depth type, P < 1, diff / sum_abs_diff without gray1, no output;
 * PHOVO_E_UNSUPPORTED: frames of 2^31 pixels or more.  Pairs run in chunks whose splat keys (4 B per pixel) fit in
 * half of the L2 (640x480 on B200: 51 pairs); debug flag 16 clears the keys with a memset per chunk instead of in the
 * resolve pass (same results). */
int phovo_batch_warp_image(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                           const uint8_t* gray0, const void* depth0, int depth_type, double depth_scale,
                           const double* rts, const double K[9], int level, const uint8_t* gray1,
                           uint8_t* warped, uint8_t* diff, int32_t* num_landed, int64_t* sum_abs_diff);
/* Normal equations of P pairs at given states, at any pyramid level in [0, num_levels) whether or not it has iterations
 * configured (the call builds that level itself).  For pair p it returns what phovo_eval_normal_equations(ctx, level,
 * states[p]) returns on a context with the same configuration and intrinsics after phovo_set_source(gray0[p],
 * depth0[p]) and phovo_set_target(gray1[p]): H [P][21] (the packed upper triangle of J^T J, in the order of
 * phovo_iter_stats.H), g [P][6] = J^T r, cost [P] = 0.5 sum r^2 (over every target pixel some source pixel landed
 * on), num_valid [P].  Agreement is to rounding (the sums are grouped differently); num_valid is exact.
 * What J is: the photometric Jacobian of the analytic solver, with the image gradients multiplied by the configured
 * imageGradientsScalingFactor of the level; in PHOVO_MODE_ANALYTIC_REF it also carries the reference's `temp11`
 * term (AN:253), in PHOVO_MODE_ANALYTIC_FIXED it is the exact derivative.  So H is the reference's J^T J as its
 * Gauss-Newton step uses it, not a calibrated information matrix: scale it by a noise model of your own before
 * using it as one, and mind that in mode 0 its translation-rotation coupling is the reference's.
 * gray0 / depth0 / gray1 are dense [P][rows][cols], all on the host (pageable or pinned) or all on the device;
 * states [P][6] (x y z yaw pitch roll) on the host or the device; each output may be NULL, host or device, at least
 * one must be given.  Blocking; device inputs are read on the context stream (see phovo_set_source).
 * Results are bitwise reproducible and independent of which pairs share a call.
 * PHOVO_E_UNSUPPORTED: Ceres mode and the photometric + depth solver (which has
 * phovo_batch_eval_normal_equations_with_target_depth), blurFilterSize[level] > 1, level 1 of a frame
 * whose size is 3 mod 4, frames of 2^31 pixels or more.  PHOVO_E_INVALID: no intrinsics, P < 1, bad sizes or level,
 * unknown depth type, no output.  Pairs run in chunks whose winner keys, validity flags and level records (5 B per
 * level pixel, + 20 B above level 0) fit in half of the L2. */
int phovo_batch_eval_normal_equations(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                                      const uint8_t* gray0, const void* depth0, int depth_type, double depth_scale,
                                      const uint8_t* gray1, const double* states /* [P][6] */, int level,
                                      double* H /* [P][21] */, double* g /* [P][6] */, double* cost /* [P] */,
                                      int32_t* num_valid /* [P] */);
/* phovo_batch_eval_normal_equations for the photometric + depth solver (PHOVO_MODE_BIOBJECTIVE).  depth1 [P][rows][cols]
 * is the target depth, same type / scale as depth0, host or device like the frames.  For pair p it returns what
 * phovo_eval_normal_equations(ctx, level, states[p]) returns after phovo_set_source(gray0[p], depth0[p]),
 * phovo_set_target(gray1[p]) and phovo_set_target_depth(depth1[p]): H and g of the stacked 2N-row system (intensity and
 * depth rows, the reference's row aliasing included: kernels_align.cu, k_winner_bi), cost = 0.5 sum over the 2N
 * residual slots, num_valid = valid source pixels.  Agreement is to rounding; num_valid is exact.  Inputs, outputs,
 * blocking behaviour, determinism and the other errors are those of phovo_batch_eval_normal_equations.  Pairs run in
 * chunks whose 2N winner keys, validity flags, target depth and its gradients (33 B per level pixel, + 20 B above level 0)
 * fit in half of the L2.  PHOVO_E_INVALID: depth1 NULL.  Other modes ignore depth1 and forward to
 * phovo_batch_eval_normal_equations (Ceres mode: PHOVO_E_UNSUPPORTED). */
int phovo_batch_eval_normal_equations_with_target_depth(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                                                        const uint8_t* gray0, const void* depth0, int depth_type,
                                                        double depth_scale, const uint8_t* gray1, const void* depth1,
                                                        const double* states /* [P][6] */, int level,
                                                        double* H /* [P][21] */, double* g /* [P][6] */,
                                                        double* cost /* [P] */, int32_t* num_valid /* [P] */);
/* The batch entries keep what they allocate between calls: the packed level store, the slots' arena (up to half of the
 * free device memory for frames with large active levels), the pool's contexts, pinned result buffers, the warpImage
 * keys and staging buffers, the keys, level records, target depths, partial sums and results of the batched normal equations.
 * This frees all of it (blocks until the device is idle); the next batch call allocates again.  Debug flags and the
 * record-stats switch return to their defaults. */
int phovo_batch_release_memory(phovo_ctx* ctx);
/* bytes the last phovo_batch_align call copied host -> device.  Host batches are uploaded without
 * the source rows no active pyramid level reads (the levels are point-decimated from the original
 * image, AN:132), so this can be less than the size of the inputs. */
int phovo_batch_get_last_h2d_bytes(const phovo_ctx* ctx, unsigned long long* bytes);
int phovo_synchronize(phovo_ctx* ctx);
/* device time (CUDA events on the context stream) of the two kernels of the last
 * phovo_batch_align_device call: pyramid (K1b) and align (K3-batch); blocks until they finished */
int phovo_batch_get_kernel_times(phovo_ctx* ctx, float* pyramid_ms, float* align_ms);

/* ---- row-sharded single pair across ranks (extension; BASELINE config 7680x4320) -------- */
/* Rank `rank` of `world` evaluates source rows [row_begin,row_end) of each level (the library
 * splits rows evenly) and leaves 27 partial sums (21 H + 6 g) + cost + count in a device buffer
 * the caller all-reduces (NCCL via torch.distributed, or the peer-store kernel) before the step. */
int phovo_shard_configure(phovo_ctx* ctx, int rank, int world);
/* device pointer to the 32-double reduction buffer: [0..20] H, [21..26] g, [27] cost, [28] count */
int phovo_shard_buffer(phovo_ctx* ctx, double** dev_ptr);
/* host-mediated exchange (tests, gloo): copy the buffer out / in through the host (synchronous) */
int phovo_shard_read_buffer(phovo_ctx* ctx, double out[32]);
int phovo_shard_write_buffer(phovo_ctx* ctx, const double in[32]);
int phovo_shard_begin(phovo_ctx* ctx);                           /* uploads the initial state */
int phovo_shard_begin_level(phovo_ctx* ctx, int level);          /* resets the iteration counter */
int phovo_shard_partial(phovo_ctx* ctx);                         /* K3a + K3b + local reduce -> buffer */
int phovo_shard_step(phovo_ctx* ctx, int* done);                 /* solve + update + termination test */
int phovo_shard_finish(phovo_ctx* ctx);                          /* read back state + stats */
/* Fused exchange over NVLink peer memory (one process per GPU): every rank allocates an exchange
 * area and exports its CUDA IPC handle (64 bytes); after importing every peer's handle,
 * phovo_shard_partial_exchange() replaces phovo_shard_partial + the collective: the kernel that
 * reduces the per-block partials stores this rank's 32 sums straight into every peer's area
 * (st.global over NVLink), releases a flag, waits for the peers' flags and sums the `world` slots
 * in rank order -- a one-shot all-reduce in the epilogue of the local reduction, bitwise identical
 * on every rank.  A peer that never arrives makes the wait time out (error flag, PHOVO_E_CUDA
 * from phovo_shard_step) instead of hanging the GPU. */
#define PHOVO_IPC_HANDLE_BYTES 64
#define PHOVO_SHARD_MAX_WORLD 8
int phovo_shard_peer_export(phovo_ctx* ctx, void* handle_out /* PHOVO_IPC_HANDLE_BYTES */);
int phovo_shard_peer_import(phovo_ctx* ctx, int peer_rank, const void* handle);
int phovo_shard_partial_exchange(phovo_ctx* ctx);
/* The whole row-sharded Optimize() (AN:500-563) in ONE call, one persistent cooperative launch per active level on
 * every rank: phase A over the level, phase B over this rank's band of source rows, and the 29 sums exchanged INSIDE
 * the kernel over the imported NVLink exchange areas (flags as the cross-GPU barrier); every rank takes the same
 * step redundantly, nothing returns to the host between iterations.  A level with fewer than `min_shard_pixels`
 * pixels is not sharded: every rank runs the whole level (identical results, no exchange) -- small levels are
 * bound by the latency of an iteration, to which an exchange only adds.  All ranks must call this with the same
 * frames, configuration, initial state and min_shard_pixels; blocks until this rank's result is back.
 * Analytic modes; needs phovo_shard_configure and, for world > 1, the peer areas of every rank imported. */
int phovo_shard_optimize(phovo_ctx* ctx, int min_shard_pixels);

#ifdef __cplusplus
}
#endif
#endif /* PHOVO_B200_H_ */
