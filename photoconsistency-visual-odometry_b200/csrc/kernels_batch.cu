// kernels_batch.cu -- the batched path (BASELINE config "N independent 640x480 pairs"):
//
//   K1b k_batch_pyramid : one streaming pass over the full-resolution inputs of every pair that
//        writes, for each ACTIVE pyramid level only, I0 and I1 as EXACT 10-bit tap sums (u16,
//        value = sum/1020) and D0 as fp64 (the reference's own double average).  HBM-bound.
//        (AN:115-163 with blur 0.)
//   K3-batch k_batch_level : one launch per active pyramid level; persistent CTAs take one pair at a
//        time and run the complete Gauss-Newton loop of that level (AN:504-561) without leaving the
//        SM: winner words, Scharr numerators and I1 resident in shared memory (10 B/px), D0 / I0
//        streamed from the pair's record in L2, estimate-then-verify warp, warp-transposed
//        fixed-order reduction, the 6x6 solve in registers.  No grid-wide synchronisation, no atomics
//        on floating-point data; the thread->pixel mapping is a pure function of the level size,
//        so results are bitwise reproducible and independent of which SM, CTA or GPU processes the
//        pair.
//
// Why exact storage: the residual scatter (AN:358) makes the cost piecewise constant in the
// warp; when a level does not converge (it often runs to max_num_iterations) any 1e-7
// perturbation (e.g. fp32 images) flips a rounding somewhere along the 50-iteration trajectory
// and the final pose moves by >1e-4 in ~15% of pairs.  Integer tap sums + fp64 depth keep the
// device within ~1e-15 of the reference's doubles, so trajectories stay together.
#include "phovo_batch.h"
#include "phovo_device.cuh"
#include "phovo_kernels.h"

namespace phovo {
namespace {


__device__ __forceinline__ void linear_axis(int d, double scale, int ssize, bool is_x, int& s0, float& w1) {
  float f = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= (float)s;
  if (s < 0) { f = 0.f; s = 0; }
  if (is_x && s >= ssize - 1) { f = 0.f; s = ssize - 1; }
  s0 = s; w1 = f;
}

// K1b.  grid = (ceil(pixels of all active levels / 256), pairs).  One thread per level pixel:
// 4 taps from each of gray0, gray1 and depth0 (the central 2x2 of the pixel's 2^level cell).
// Consecutive threads read consecutive cells of the same two source rows, so a warp touches one
// contiguous span per row and every fetched sector is consumed by the warp.
template <typename DT>
__global__ void __launch_bounds__(256) k_batch_pyramid(const __grid_constant__ BatchParams bp,
                                                       const uint8_t* __restrict__ gray0, const DT* __restrict__ depth0,
                                                       double depth_scale, const uint8_t* __restrict__ gray1,
                                                       uint8_t* __restrict__ store) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= bp.px_offset[bp.num_active]) return;
  int a = 0;
  while (j >= bp.px_offset[a + 1]) ++a;
  const int q = j - bp.px_offset[a];
  const int lc = bp.lcols[a];
  const int y = q / lc, x = q - y * lc;
  const int level = bp.level[a];
  const double scale = (double)(1 << level);
  const size_t pair = blockIdx.y;
  // staged host inputs may carry only the source rows the active levels read (see phovo_batch.cu):
  // row y of a frame then lives at compact row (y / period) * keep + (y % period - keep_begin)
  const int period = bp.src_period;
  const size_t frame = period ? (size_t)(bp.rows / period) * bp.src_keep * bp.cols : (size_t)bp.rows * bp.cols;
  const uint8_t* G0 = gray0 + pair * frame;
  const uint8_t* G1 = gray1 + pair * frame;
  const DT* D = depth0 + pair * frame;
  int sx, sy; float fx, fy;
  linear_axis(x, scale, bp.cols, true, sx, fx);
  linear_axis(y, scale, bp.rows, false, sy, fy);
  const int y0 = min(max(sy, 0), bp.rows - 1), y1 = min(max(sy + 1, 0), bp.rows - 1);
  const bool two = sx + 1 < bp.cols;
  const int z0 = period ? (y0 / period) * bp.src_keep + (y0 % period - bp.src_keep_begin) : y0;
  const int z1 = period ? (y1 / period) * bp.src_keep + (y1 % period - bp.src_keep_begin) : y1;
  const size_t o00 = (size_t)z0 * bp.cols + sx, o10 = (size_t)z1 * bp.cols + sx;
  unsigned s0, s1;
  double dv;
  if (level == 0) {  // the image itself: one tap with weight one (value = 4 v / 1020 = v / 255)
    s0 = 4u * (unsigned)__ldg(G0 + o00);
    s1 = 4u * (unsigned)__ldg(G1 + o00);
    dv = depth_at<DT>(D + o00, depth_scale);
  } else if (level == 1) {
    // cv::resize by exactly 1/2 takes the INTER_AREA path: ((S00 + S01) + S10) + S11 times 0.25
    // (kernels_pyramid.cu: level_value).  Sizes with cells cut by the border are rejected by the host.
    s0 = (unsigned)__ldg(G0 + o00) + __ldg(G0 + o00 + 1) + __ldg(G0 + o10) + __ldg(G0 + o10 + 1);
    s1 = (unsigned)__ldg(G1 + o00) + __ldg(G1 + o00 + 1) + __ldg(G1 + o10) + __ldg(G1 + o10 + 1);
    dv = __dmul_rn(__dadd_rn(__dadd_rn(__dadd_rn(depth_at<DT>(D + o00, depth_scale), depth_at<DT>(D + o00 + 1, depth_scale)),
                                       depth_at<DT>(D + o10, depth_scale)), depth_at<DT>(D + o10 + 1, depth_scale)), 0.25);
  } else if (two) {
    s0 = (unsigned)__ldg(G0 + o00) + __ldg(G0 + o00 + 1) + __ldg(G0 + o10) + __ldg(G0 + o10 + 1);
    s1 = (unsigned)__ldg(G1 + o00) + __ldg(G1 + o00 + 1) + __ldg(G1 + o10) + __ldg(G1 + o10 + 1);
    const double a0 = (double)(1.f - fx), a1 = (double)fx;
    const double r0 = __dadd_rn(__dmul_rn(depth_at<DT>(D + o00, depth_scale), a0), __dmul_rn(depth_at<DT>(D + o00 + 1, depth_scale), a1));
    const double r1 = __dadd_rn(__dmul_rn(depth_at<DT>(D + o10, depth_scale), a0), __dmul_rn(depth_at<DT>(D + o10 + 1, depth_scale), a1));
    dv = __dadd_rn(__dmul_rn(r0, (double)(1.f - fy)), __dmul_rn(r1, (double)fy));
  } else {  // right border of an odd-sized image: a single horizontal tap with weight one
    s0 = 2u * ((unsigned)__ldg(G0 + o00) + __ldg(G0 + o10));
    s1 = 2u * ((unsigned)__ldg(G1 + o00) + __ldg(G1 + o10));
    dv = __dadd_rn(__dmul_rn(depth_at<DT>(D + o00, depth_scale), (double)(1.f - fy)), __dmul_rn(depth_at<DT>(D + o10, depth_scale), (double)fy));
  }
  uint8_t* rec = store + pair * bp.record_bytes;
  ((uint16_t*)(rec + bp.off_I0[a]))[q] = (uint16_t)s0;
  ((uint16_t*)(rec + bp.off_I1[a]))[q] = (uint16_t)s1;
  ((double*)(rec + bp.off_D0[a]))[q] = dv;
  // fp32 copy for phase A's estimate; the strict range test of AN:279-280 is decided HERE, in fp64, and
  // encoded as 0 (NaN compares false, so a NaN depth is invalid too); a valid depth that would round
  // to 0 in fp32 cannot occur: the host enables the fp32 estimate only for min_depth >= 2^-100
  ((float*)(rec + bp.off_D32[a]))[q] = (bp.min_depth < dv) & (dv < bp.max_depth) ? (float)dv : 0.f;
}

// ---------------------------------------------------------------------------------------------
// K3-batch building blocks
// ---------------------------------------------------------------------------------------------
static_assert(kBatchThreads % 32 == 0 && kBatchThreadsSmall % 32 == 0, "whole warps: the reduction scratch has one row per warp");
static_assert(kBatchMaxLevelPixels <= 60 * kBatchThreads, "per-thread validity mask is 64 bits (phase A fills it four pixels at a time)");
static_assert(kBatchSmallLevelPixels <= 60 * kBatchThreadsSmall, "per-thread validity mask is 64 bits (phase A fills it four pixels at a time)");
static_assert(kBatchMaxLevelPixels < 65535, "winner word keeps source index + 1 in 16 bits");

// Everything k_batch_level needs about ITS level, at fixed offsets of the kernel parameter block, so
// that every field is a constant-bank operand (indexing BatchParams' per-level arrays with a
// run-time level costs a load and a register per use, inside the pixel loops).
struct BatchLevelParams {
  int num_pairs, rows, cols, n;
  int level, max_iters, first, log_cap;          // first: coarsest active level (starts from the caller's state)
  int exact_always, force_generic;
  int est32;                                     // fp32 estimate of phase A usable for this level (see gn_level)
  int prev_level;                                // pyramid level of the previous (coarser) active level, -1 for the first
  unsigned long long off_I0, off_I1, off_D0, off_D32, record_bytes;
  double fx, fy, ox, oy, inv_fx, inv_fy;
  double lambda, min_grad, grad_k;
  double min_depth, max_depth;
};

static BatchLevelParams level_params(const BatchParams& bp, int a) {
  BatchLevelParams lv;
  lv.num_pairs = bp.num_pairs; lv.rows = bp.lrows[a]; lv.cols = bp.lcols[a]; lv.n = lv.rows * lv.cols;
  lv.level = bp.level[a]; lv.max_iters = bp.max_iters[a]; lv.first = a == 0; lv.log_cap = bp.log_cap;
  lv.exact_always = bp.exact_always; lv.force_generic = bp.force_generic;
  lv.off_I0 = bp.off_I0[a]; lv.off_I1 = bp.off_I1[a]; lv.off_D0 = bp.off_D0[a]; lv.off_D32 = bp.off_D32[a]; lv.record_bytes = bp.record_bytes;
  // the fp32 estimate keeps 14 fraction bits of the displacement in a float: |displacement| < 256 px, so every
  // in-bounds target of a level of at most 256 x 256 px is representable (warp_estimate32)
  lv.est32 = lv.rows <= 256 && lv.cols <= 256 && bp.min_depth >= 0x1p-100 && bp.max_depth <= 0x1p100;
  lv.prev_level = a > 0 ? bp.level[a - 1] : -1;
  lv.fx = bp.fx[a]; lv.fy = bp.fy[a]; lv.ox = bp.ox[a]; lv.oy = bp.oy[a]; lv.inv_fx = bp.inv_fx[a]; lv.inv_fy = bp.inv_fy[a];
  lv.lambda = bp.lambda[a]; lv.min_grad = bp.min_grad[a]; lv.grad_k = bp.grad_k[a];
  lv.min_depth = bp.min_depth; lv.max_depth = bp.max_depth;
  return lv;
}

__device__ __forceinline__ float ldg_f32(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float rcp_approx_f32(float x) {   // MUFU.RCP: at most 1 ulp
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ---------------------------------------------------------------------------------------------
// Phase A in SINGLE precision (column-fixed kernels).  The fp64 estimate (warp_estimate) costs ~17
// instructions of the FP64 pipe per pixel, and an instruction of that pipe costs more than two issue
// cycles (tools/issue_probe.cu: nothing issues in its shadow) -- a third of what the kernel is bound by.
// fp32 cannot resolve t = f X'/Z' + o to the 2^-14 px the certainty test needs (24 bits, |t| < 2^8), but
// it can resolve the DISPLACEMENT t - c of the pixel from its own position, which is small:
//   t_c - c = fx (X' - cxi Z') / Z' + (fx cxi + ox - c),        X' - cxi Z' = d D0 + (x - cxi z),
//   D0 = (R00 cxi + R02) - cxi (R20 cxi + R22) + ryi (R01 - R21 cxi)                      [O(rotation)]
//   t_r - r = fy (Y' - ryi Z') / Z',                            Y' - ryi Z' = d D1 + (y - ryi z),
//   D1 = (R10 cxi + R12) + ryi (R11 - R22 - R20 cxi) - ryi^2 R21
//   Z' = d + (d (M2 - 1) + z),  M2 - 1 = (R20 cxi + R22 - 1) + R21 ryi
// A thread's column is fixed, so the cxi-dependent coefficients are per-thread constants of the
// iteration (computed in fp64, rounded once); the ryi-dependent ones come from a float4 row table.
// floor((displacement + 0.5) 2^14) is read off the mantissa of  q fxs + (0.5 * 2^14 + 1.5 * 2^23)  evaluated
// with round-down (one FFMA.RM): bits 0..13 are the fraction, bits 14.. the whole pixels + 0x12D00.
// Values outside [-2^22, 2^22) leave the binade [2^23, 2^24): the bits then decode to a target >= 256 px
// away, which is out of bounds for a level of at most 256 x 256 px -- as the true target is.
//
// Error budget (u = 2^-24; a valid pixel that passes the guard Z' > d / 2 has d >= dmin = min_depth):
//   every D / M2 - 1 is within 4 u B of its exact value, B = the sum of the magnitudes of its terms
//     (coefficient rounding, ryi rounding, the fused multiply-add, the final add);
//   |num - num*| <= u (6 d B + 2 emax)      (d rounded to fp32, the offset rounded, the fma);   / Z' <= u (12 B + 4 emax / dmin)
//   |Z' - Z'*| / Z' <= u GZ,  GZ = 2 (7 B2 + 1) + 4 |z| / dmin + 1;   reciprocal 2 u, product u, fxs u
//   |displacement| <= D = f (2 B + 2 emax / dmin)
//   E = f u (12 B + 4 emax / dmin) + D u (GZ + 4) + 2^-36          px; the last term covers the ~10 roundings of
//                                                                   the reference's own fp64 evaluation and fx cxi vs c - ox
// A fraction is trusted when it lies at least e = ceil(E 2^14) + 1 units from both ends of [0, 2^14).
// Returns the margins; 2^14 (nothing trusted) if anything is not finite.
// ---------------------------------------------------------------------------------------------
constexpr int kFrac32Bits = 14;
constexpr unsigned kFrac32One = 1u << kFrac32Bits;
constexpr float kMagic32 = 12582912.f + 8192.f;          // 1.5 * 2^23 + 0.5 * 2^14
constexpr int kMagic32Whole = 0x4B400000 >> kFrac32Bits;  // what bits 14.. of the mantissa trick carry for a zero displacement

__device__ __forceinline__ void est32_margins(const Pose& T, double fx, double fy, double rx, double ry, double dmin, unsigned& ex, unsigned& ey) {
  const double u = 0x1p-24;
  const double B0 = (fabs(T.R00 - T.R22) * rx + fabs(T.R20) * rx * rx + fabs(T.R02)) + (fabs(T.R01) + fabs(T.R21) * rx) * ry;
  const double B1 = (fabs(T.R10) * rx + fabs(T.R12)) + (fabs(T.R11 - T.R22) + fabs(T.R20) * rx) * ry + fabs(T.R21) * ry * ry;
  const double B2 = fabs(T.R20) * rx + fabs(T.R22 - 1.0) + fabs(T.R21) * ry;
  const double idmin = 1.0 / dmin;
  const double e0m = fabs(T.x) + rx * fabs(T.z), e1m = fabs(T.y) + ry * fabs(T.z);
  const double GZ = 2.0 * (7.0 * B2 + 1.0) + 4.0 * fabs(T.z) * idmin + 1.0;
  const double Dx = fabs(fx) * (2.0 * B0 + 2.0 * e0m * idmin), Dy = fabs(fy) * (2.0 * B1 + 2.0 * e1m * idmin);
  const double Ex = fabs(fx) * u * (12.0 * B0 + 4.0 * e0m * idmin) + Dx * u * (GZ + 4.0) + 0x1p-36;
  const double Ey = fabs(fy) * u * (12.0 * B1 + 4.0 * e1m * idmin) + Dy * u * (GZ + 4.0) + 0x1p-36;
  const double sx = Ex * (double)kFrac32One, sy = Ey * (double)kFrac32One;
  ex = (sx < 4096.0) ? (unsigned)ceil(sx) + 1u : kFrac32One;     // NaN compares false: nothing trusted
  ey = (sy < 4096.0) ? (unsigned)ceil(sy) + 1u : kFrac32One;
}

struct BatchShared {
  PoseDev pose;          // state + rotation / trig of the current iterate
  double totals[32];
  int done;
  int iteration;
  int pair;
  int pad;
  unsigned ex, ey;       // margins of phase A's fp32 estimate for the current iterate (est32_margins), written with the pose
};

// largest |cxi|, |ryi| of a level: the ray bounds the margins are computed from
__device__ __forceinline__ void est32_publish(const BatchLevelParams& lv, const Pose& P, BatchShared* sh) {
  const double rx = fmax(fabs(lv.ox), fabs((double)(lv.cols - 1) - lv.ox)) * fabs(lv.inv_fx);
  const double ry = fmax(fabs(lv.oy), fabs((double)(lv.rows - 1) - lv.oy)) * fabs(lv.inv_fy);
  unsigned ex, ey;
  est32_margins(P, lv.fx, lv.fy, rx, ry, lv.min_depth, ex, ey);
  sh->ex = ex; sh->ey = ey;
}

// Gauss-Newton step by ONE warp (AN:538-549 + AN:376-392).  Lane L enters with total[L]
// ([0..20] upper triangle of J^T J, [21..26] J^T r, [27] sum r^2, [28] count).  The totals go through
// shared memory and EVERY lane solves the full 6x6 system redundantly in registers: the symmetric
// positive definite system is eliminated without pivoting (LDL^T, i.e. the Cholesky solve the north
// star asks for; the reference's Eigen inverse() is a pivoted LU -- same solution to ~cond*2^-53)
// with one correctly rounded reciprocal per pivot.  No shuffles on the critical path: a serial
// chain of ~50 dependent fp64 operations instead of ~100 shuffle round trips.  Then state update,
// sincos on three lanes, rotation, termination flag.  Lane 0 publishes.
__device__ __forceinline__ void warp_gn_step(double tot, int lane, const BatchLevelParams& lv, int it, int pair,
                                             BatchShared* sh, phovo_iter_stats* log) {
  const unsigned FULL = 0xffffffffu;
  sh->totals[lane] = tot;
  __syncwarp();
  double x[6], n2 = 0.;
  solve6_ldlt(sh->totals, sh->totals + 21, x);
#pragma unroll
  for (int k = 0; k < 6; ++k) n2 = fma(sh->totals[21 + k], sh->totals[21 + k], n2);
  const double lambda = lv.lambda;
  double s_in[6], s_out[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) { s_in[k] = sh->pose.state[k]; s_out[k] = s_in[k] - lambda * x[k]; }   // AN:539-540
  const int which = lane % 3;
  const double ang = which == 0 ? s_out[3] : which == 1 ? s_out[4] : s_out[5];
  double sn, cs;
  sincos(ang, &sn, &cs);
  Pose P;
  P.x = s_out[0]; P.y = s_out[1]; P.z = s_out[2];
  P.sy = __shfl_sync(FULL, sn, 0); P.cy = __shfl_sync(FULL, cs, 0);
  P.sp = __shfl_sync(FULL, sn, 1); P.cp = __shfl_sync(FULL, cs, 1);
  P.sr = __shfl_sync(FULL, sn, 2); P.cr = __shfl_sync(FULL, cs, 2);
  rotation_from_trig(P);
  const double gnorm = sqrt(n2);
  const int done = (it + 1 >= lv.max_iters) || (gnorm < lv.min_grad);   // AN:383-392
  __syncwarp();
  if (lane == 0) {
    if (log && sh->pose.log_count < lv.log_cap) {
      const double* t = sh->totals;
      phovo_iter_stats* e = log + (size_t)pair * lv.log_cap + sh->pose.log_count;
      e->level = lv.level; e->iteration = it; e->num_valid = (int)t[28]; e->accepted = 1;
      for (int k = 0; k < 21; ++k) e->H[k] = t[k];
      for (int k = 0; k < 6; ++k) { e->g[k] = t[21 + k]; e->state_in[k] = s_in[k]; e->state_out[k] = s_out[k]; }
      e->grad_norm = gnorm; e->cost = 0.5 * t[27]; e->radius = 0.;
    }
    sh->pose.log_count += 1;
#pragma unroll
    for (int k = 0; k < 6; ++k) sh->pose.state[k] = s_out[k];
    pose_store(P, &sh->pose);
    est32_publish(lv, P, sh);
    sh->done = done;
    sh->iteration = it + 1;
  }
}

// Per-level / per-iteration lookup tables in shared memory (doubles).  `cols`/`rows` of the level.
//   exact  : cx[c] = fl(c - ox), ry[r] = fl(r - oy)            the reference's own roundings (AN:282-287)
//   ray    : cxi[c] = cx[c] * inv_fx, ryi[r] = ry[r] * inv_fy  back-projected ray (px/d, py/d)
//   colA/B : {R00 cxi, R10 cxi}, {R20 cxi, -cp cxi}            per ITERATION: the column part of R*(ray) and of dZ'/dpitch
//   row    : {R01 ryi + R02, R11 ryi + R12}, {R21 ryi + R22, -(sp sr ryi + sp cr)}, {R22 ryi - R21, R02 ryi - R01}, {R12 ryi - R11, 0},
//            {fxs (R01 ryi + R02), fys (R11 ryi + R12)}          (entry 0 pre-scaled for the fixed-point estimate of phase A)
// so that  R p = d * (col + row)  costs 3 adds + 3 multiplies instead of 4 + 9.
// The row table carries ceil(3 threads / cols) rows of zero padding: the last pixels of a thread's
// last (four-pixel) trip of phase A may lie up to 3 `threads` pixels past the level and are read
// (and masked) without a guard.
constexpr int kRowEntries = 5;
#ifndef PHOVO_PHASE_A_WIDTH
#define PHOVO_PHASE_A_WIDTH 4
#endif
constexpr int kPhaseAWidth = PHOVO_PHASE_A_WIDTH;   // pixels per trip of the fp32 phase A (column-fixed kernels)
struct Tables {
  double* cx; double* ry; double* cxi; double* ryi;
  double2* colA; double2* colB;   // [cols]
  double2* row;                   // [rows + pad][kRowEntries]
  float4* rowf;                   // [rows + pad] per ITERATION, fp32 estimate of phase A: {ryi, y - ryi z, R21 ryi, -R21 ryi^2}
};
__host__ __device__ inline int table_pad_rows(int cols, int threads) { return ((kPhaseAWidth > 4 ? kPhaseAWidth - 1 : 3) * threads + cols - 1) / cols; }
__host__ __device__ inline int table_doubles(int rows, int cols, int threads) {
  return 2 * (rows + cols) + 4 * cols + (2 * kRowEntries + 2) * (rows + table_pad_rows(cols, threads));
}
// shared-memory slots of the three per-pixel arrays: the level plus `threads` slots of padding
__host__ __device__ inline int padded_slots(int n, int threads) { return (n + threads + 7) & ~7; }

struct WarpA { int tj, ti; };   // rounded target column / row; out of the image <=> the pixel does not bid

// The reference's warp of one pixel, AN:279-303: fp64, its operation order, no FMA contraction,
// correctly rounded reciprocal, C round().  Used for the (rare) pixels whose cheap estimate falls
// within 2^-17 px of a rounding boundary, and for everything when bp.exact_always is set.
__device__ __noinline__ WarpA warp_exact(const PoseDev* pose, double cx, double ry, double d, double fx, double fy, double ox, double oy,
                                         double inv_fx, double inv_fy) {
  Pose T;
  pose_load(pose, T);
  const double px = __dmul_rn(__dmul_rn(cx, d), inv_fx);
  const double py = __dmul_rn(__dmul_rn(ry, d), inv_fy);
  const double X = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T.R00, px), __dmul_rn(T.R01, py)), __dmul_rn(T.R02, d)), T.x);
  const double Y = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T.R10, px), __dmul_rn(T.R11, py)), __dmul_rn(T.R12, d)), T.y);
  const double Z = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T.R20, px), __dmul_rn(T.R21, py)), __dmul_rn(T.R22, d)), T.z);
  WarpA w;
  const double az = fabs(Z);
  // |Z| outside the normal range (incl. NaN / 0, where the reference's int cast is undefined) is out of bounds
  if (!((az > 1e-300) & (az < 1e300))) { w.tj = -1; w.ti = -1; return w; }
  const double iz = rcp_rn_normal(Z);                                       // AN:294 `1./Z`
  const double tc = __dadd_rn(__dmul_rn(__dmul_rn(X, fx), iz), ox);
  const double tr = __dadd_rn(__dmul_rn(__dmul_rn(Y, fy), iz), oy);
  // C round(): half away from zero == trunc(x + copysign(0.5, x)) with the add rounded toward zero
  w.tj = __double2int_rz(__dadd_rz(tc, copysign(0.5, tc)));
  w.ti = __double2int_rz(__dadd_rz(tr, copysign(0.5, tr)));   // saturated casts fail the caller's range test
  return w;
}

// Experiment hook (tools/section_clocks.py): -DPHOVO_SECTION_CLOCKS accumulates, from thread 0 of every CTA,
// the clocks between the section boundaries of an iteration.  Not compiled into the product library.
#ifdef PHOVO_SECTION_CLOCKS
__device__ unsigned long long g_section_clocks[2][8];
#define SEC_INIT() long long sec_t = clock64()
#define SEC_MARK(k) do { if (threadIdx.x == 0) { const long long now_ = clock64(); \
  atomicAdd(&g_section_clocks[BT == kBatchThreads ? 1 : 0][k], (unsigned long long)(now_ - sec_t)); sec_t = now_; } } while (0)
#else
#define SEC_INIT() do {} while (0)
#define SEC_MARK(k) do {} while (0)
#endif

struct IterConst {          // per-iteration scalars besides the tables
  double x, y, z, cy, sy, rho;
  double fxs, fys, oxs, oys;   // fx 2^14, fy 2^14, (ox + 0.5) 2^14, (oy + 0.5) 2^14  (phase A fixed point)
  double xs, ys;               // fxs x, fys y
};

struct ColRegs { double2 a, b; double cxix; };   // column entries of the tables for one pixel; cxix = cxi * x (MODE 0 only)
struct ColRegsA { double2 as; double bx; };      // phase A: {fxs R00 cxi, fys R10 cxi}, R20 cxi


// Phase A of one pixel, fast path.  Estimates the warped coordinate from the per-iteration tables as
// floor((t + 0.5) 2^14) in a 32-bit integer.  If the 14-bit fraction is neither 0 nor 2^14 - 1 the
// estimate is at least 2^-14 px away from a rounding boundary, so -- provided estimate and reference
// agree to 2^-14 px -- the rounded pixel is certain and equals the reference's round() (also for t in
// (-0.5, 0), which round() maps to -0 -> column 0); otherwise `uncertain` is set and the caller runs
// warp_exact.  Agreement: both evaluations make ~25 roundings of 2^-53 relative to S, the largest
// summand of X', Y', Z' (see gn_level), so t = f X'/Z' + o differs by at most
// 2^-46 S (f + |t - o|) / |Z'|, which is below 2^-14 px for every t near the image once
// |Z'| >= zmin = 2^-30 S (f + cols + rows + |o| + 2).  Pixels closer to the camera plane than zmin
// (cancellation in Z') are uncertain as well: the caller passes the high word of zmin.  Saturated
// conversions (|t| >= 2^17, inf) land out of bounds, NaN converts to 0 and is therefore
// uncertain.  Straight-line code.
__device__ __forceinline__ WarpA warp_estimate(const IterConst& K, const ColRegsA& col, double2 rs, double r1x, double d,
                                               unsigned unc_thr, unsigned zmin_hi, bool& uncertain) {
  const double M0 = col.as.x + rs.x, M1 = col.as.y + rs.y, M2 = col.bx + r1x;     // M0, M1 carry fxs, fys
  const double X = fma(d, M0, K.xs), Y = fma(d, M1, K.ys), Z = fma(d, M2, K.z);
  const double iz = rcp_1ulp(Z);
  const int lx = __double2int_rd(fma(X, iz, K.oxs));
  const int ly = __double2int_rd(fma(Y, iz, K.oys));
  const unsigned fx_ = (unsigned)lx & (kFracOne - 1u), fy_ = (unsigned)ly & (kFracOne - 1u);
  uncertain = (max(fx_ - 1u, fy_ - 1u) >= unc_thr) | (((unsigned)__double2hiint(Z) & 0x7fffffffu) < zmin_hi);
  WarpA w;
  w.tj = lx >> kFracBits; w.ti = ly >> kFracBits;
  return w;
}

// Prefetch loads of the pixel loops.  `asm volatile`: as plain ld.global.nc (__ldg) the compiler
// treats them as invariant loads and sinks them to their first use one trip later, which turns the
// register prefetch into a load-use stall of a full L2 round trip per trip.  The u16 goes straight
// into a 32-bit register (zero-extended by the load): as an `unsigned short` it would travel in half
// registers and cost a PRMT and a mask per trip.
__device__ __forceinline__ unsigned ldg_u16(const unsigned short* p) {
  unsigned v;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ldg_f64(const double* p) {
  double v;
  asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

// shared-memory max without a result.  Pixels that do not bid are pointed at a per-lane dummy slot
// instead of being branched around (ptxas turns a predicated red into a branch).
__device__ __forceinline__ void smem_red_max(unsigned addr, unsigned v) {
  asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// Phase B of one pixel: J' = J / (gk fx) and the integer residual numerator; the common factors
// are applied once per iteration to the reduced sums.  Everything is computed unconditionally on
// sanitised operands and masked, so that two pixels interleave without branches.  With
// m = col + row (the rotated ray of the pixel, R p = d m) the closed form of AN:243-342 (SURVEY
// appendix C) is written in the products ga d, gb d, J2 d, which needs 27 fp64 operations.
template <int MODE>
__device__ __forceinline__ void jacobian_row(const IterConst& K, const ColRegs& col, double2 r0, double2 r1, double2 r2, double2 r3,
                                             double d, bool valid, unsigned gw, double J[6]) {
  // an invalid pixel contributes a zero row: depth and 1/Z' are forced to 0 (the raw values may be
  // 0, inf or NaN), everything downstream is then a finite table entry times zero
  const double ds = valid ? d : 0.;
  const double m0 = col.a.x + r0.x, m1 = col.a.y + r0.y, m2 = col.b.x + r1.x, m3 = col.b.y + r1.y;
  const double izr = rcp_1ulp(fma(ds, m2, K.z));
  const double iz = valid ? izr : 0.;
  // a' = Gx1[i] / Z', b' = Gy1[i] (fy/fx) / Z'   (gradients at the SOURCE index, AN:346-347)
  const double ga = (double)(short)(gw & 0xffffu) * iz;
  const double gb = (double)((int)gw >> 16) * (iz * K.rho);
  const double gau = ga * ds, gbu = gb * ds;
  // ga X' + gb Y' with X' = d m0 + x (AN:253 reads d (m0 + cxi x): bug-compatible in MODE 0), Y' = d m1 + y
  const double s = MODE == 0 ? fma(gau, m0 + col.cxix, fma(gbu, m1, gb * K.y))
                             : fma(gau, m0, fma(gbu, m1, fma(ga, K.x, gb * K.y)));
  J[0] = ga;
  J[1] = gb;
  J[2] = -(s * iz);
  const double j2d = J[2] * ds;
  J[3] = fma(gbu, m0, -(gau * m1));
  J[4] = fma(m3, j2d, m2 * fma(gau, K.cy, gbu * K.sy));
  J[5] = fma(gau, r2.y, fma(gbu, r3.x, r2.x * j2d));
}

struct LevelCtx {
  int pair;
  const double* gD0; const float* gD32; const unsigned short* gI0;
  unsigned* sWin; const unsigned* sG; const unsigned short* sI1; double* sRed;
  unsigned sWinAddr, sDummyAddr;
  Tables tb;
};

// The Gauss-Newton loop of one level of one pair (AN:504-561).  COLFIX: the CTA width is a multiple
// of the level width, so a thread's pixels t, t+BT, ... all lie in ONE column: the column entries
// of the tables live in registers and only the row advances.  The thread -> pixel mapping is the
// same linear one in both variants, so results are bitwise identical.
template <int MODE, bool COLFIX, int BT, bool STATS>
__device__ __forceinline__ void gn_level(const BatchLevelParams& lv, const LevelCtx& L, BatchShared* sh, phovo_iter_stats* log) {
  constexpr int NW = BT / 32;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int rows = lv.rows, cols = lv.cols, n = lv.n;
  const Tables& tb = L.tb;
  const double fx = lv.fx, fy = lv.fy, ox = lv.ox, oy = lv.oy, inv_fx = lv.inv_fx, inv_fy = lv.inv_fy;
  const double min_depth = lv.min_depth, max_depth = lv.max_depth;
  const int max_iters = lv.max_iters;
  // a fraction f of the estimated coordinate is trusted when f - 1 < unc_thr; the test hook
  // (every pixel takes the exact path) sets the threshold to 0
  const unsigned unc_thr = lv.exact_always ? 0u : kFracOne - 2u;
  unsigned dummy;                                  // opaque, or ptxas rebuilds it from %tid in every trip
  asm volatile("mov.u32 %0, %1;" : "=r"(dummy) : "r"(L.sDummyAddr + 4u * (unsigned)lane));
  // geometry part of zmin (see warp_estimate) and the bound on |ray| of the level
  const double zmin_geo = 0x1p-30 * (fmax(fabs(fx), fabs(fy)) + (double)(cols + rows + 2) + fabs(ox) + fabs(oy));
  const double ray_bound = fmax(fabs(ox), fabs((double)(cols - 1) - ox)) * fabs(inv_fx) + fmax(fabs(oy), fabs((double)(rows - 1) - oy)) * fabs(inv_fy) + 1.0;
  const double depth_bound = fmax(fabs(min_depth), fabs(max_depth));
  // pixel i = tid + k*BT; a trip of the loops handles pixels i and i + BT
  const int r0_first = tid / cols, c0_first = tid - r0_first * cols;
  const int r1_first = (tid + BT) / cols, c1_first = (tid + BT) - r1_first * cols;
  const int dr2 = (2 * BT) / cols, dc2 = 2 * BT - dr2 * cols;
  const int dr4 = (4 * BT) / cols, dc4 = 4 * BT - dr4 * cols;
  int rstep_bytes;                                 // row-table advance of one trip (opaque for the same reason)
  asm volatile("mov.u32 %0, %1;" : "=r"(rstep_bytes) : "r"(kRowEntries * dr2 * (int)sizeof(double2)));
  // common factors of the rows phase B accumulates: J = (gk fx) J', r = r_int / 1020
  const double gkfx = lv.grad_k * fx;
  const double scale = lane < 21 ? gkfx * gkfx : lane < 27 ? gkfx * (1.0 / 1020.0) : lane == 27 ? (1.0 / 1020.0) * (1.0 / 1020.0) : 1.0;
  IterConst K;
  K.rho = fy / fx;
  K.fxs = fx * (double)kFracOne; K.fys = fy * (double)kFracOne;
  K.oxs = (ox + 0.5) * (double)kFracOne; K.oys = (oy + 0.5) * (double)kFracOne;
  const int trips = (n - tid + 2 * BT - 1) / (2 * BT);   // loop trips of this thread (0 if tid >= n)
  const double my_cxi = COLFIX ? tb.cxi[c0_first] : 0., my_cx = COLFIX ? tb.cx[c0_first] : 0.;

  // The first trip of both phases reads the same two pixels in every iteration.  Their loads are
  // issued a whole reduction + solve ahead (before the loop / at the end of phase B) instead of behind
  // the barrier that opens phase A, where every warp of the CTA would wait out the L2 latency at once.
  // (column-fixed kernels: phase A reads the fp32 copy of the depth, phase B the fp64 one)
  constexpr int FW = COLFIX ? kPhaseAWidth : 4;
  double first_d[COLFIX ? 2 : 4]; float first_f[FW]; unsigned first_u[FW];
#pragma unroll
  for (int j = 0; j < FW; ++j) {
    if (COLFIX) first_f[j] = ldg_f32(L.gD32 + tid + j * BT);
    if (!COLFIX || j < 2) first_d[j] = ldg_f64(L.gD0 + tid + j * BT);
    first_u[j] = ldg_u16(L.gI0 + tid + j * BT);
  }

  SEC_INIT();
  for (int it = 0; it < max_iters; ++it) {
    Pose T;
    pose_load(&sh->pose, T);
    // A state that is not finite (a singular solve upstream: tiny or textureless levels) makes every
    // pixel invalid in the reference, whose Jacobian rows then stay zero: H = 0, g = 0, and the level
    // stops as soon as 0 < min_gradient_norm.  Here invalid rows are "finite table entry times zero",
    // so the tables are built from the identity pose instead (warp_exact still reads the real one and
    // rejects every pixel).
    // (balanced sum: a chain of 17 dependent adds is 140 cycles of latency in front of every iteration)
    const bool finite_pose = isfinite((((T.x + T.y) + (T.z + T.R00)) + ((T.R01 + T.R02) + (T.R10 + T.R11))) +
                                      (((T.R12 + T.R20) + (T.R21 + T.R22)) + ((T.sy + T.cy) + (T.sp + T.cp))) + (T.sr + T.cr));
    if (!finite_pose) {
      T.x = T.y = T.z = 0.;
      T.R00 = T.R11 = T.R22 = 1.; T.R01 = T.R02 = T.R10 = T.R12 = T.R20 = T.R21 = 0.;
      T.sy = T.sp = T.sr = 0.; T.cy = T.cp = T.cr = 1.;
    }
    K.x = T.x; K.y = T.y; K.z = T.z; K.cy = T.cy; K.sy = T.sy;
    K.xs = K.fxs * T.x; K.ys = K.fys * T.y;
    // S bounds every summand of X', Y', Z' of a pixel inside the depth range.  If it is not an ordinary
    // number (diverged or NaN state, unbounded depth range) the estimate is not used at all.
    const double S = fma(depth_bound, ray_bound, fmax(fmax(fabs(T.x), fabs(T.y)), fabs(T.z)));
    const double zmin = fmax(S * zmin_geo, 0x1p-500);
    const bool ordinary = (S < 0x1p500) & (zmin_geo < 0x1p100) & (T.x == T.x) & (T.y == T.y) & (T.z == T.z);
    const unsigned thr = (ordinary & finite_pose) ? unc_thr : 0u;
    const unsigned zmin_hi = (unsigned)__double2hiint(zmin) + 1u;
    // ---- per-iteration tables ----
    for (int k = tid; k < (COLFIX ? 0 : cols) + rows; k += BT) {
      if (!COLFIX && k < cols) {
        const double v = tb.cxi[k];
        tb.colA[k] = make_double2(T.R00 * v, T.R10 * v);
        tb.colB[k] = make_double2(T.R20 * v, -(T.cp * v));
      } else {
        const int r = COLFIX ? k : k - cols;
        const double v = tb.ryi[r];
        const double e0 = fma(T.R01, v, T.R02), e1 = fma(T.R11, v, T.R12);
        tb.row[kRowEntries * r + 0] = make_double2(e0, e1);
        tb.row[kRowEntries * r + 1] = make_double2(fma(T.R21, v, T.R22), -fma(T.sp * T.sr, v, T.sp * T.cr));
        tb.row[kRowEntries * r + 2] = make_double2(fma(T.R22, v, -T.R21), fma(T.R02, v, -T.R01));
        tb.row[kRowEntries * r + 3] = make_double2(fma(T.R12, v, -T.R11), 0.);
        if (COLFIX) tb.rowf[r] = make_float4((float)v, (float)fma(-v, T.z, T.y), (float)(T.R21 * v), (float)(-(T.R21 * v) * v));
        else tb.row[kRowEntries * r + 4] = make_double2(K.fxs * e0, K.fys * e1);
      }
    }
    ColRegs mycol;
    mycol.a = make_double2(T.R00 * my_cxi, T.R10 * my_cxi);
    mycol.b = make_double2(T.R20 * my_cxi, -(T.cp * my_cxi));
    mycol.cxix = __dmul_rn(my_cxi, T.x);
    ColRegsA mycolA;
    mycolA.as = make_double2(__dmul_rn(K.fxs, mycol.a.x), __dmul_rn(K.fys, mycol.a.y));
    mycolA.bx = mycol.b.x;
    __syncthreads();
    SEC_MARK(0);
    // ---- phase A: warp every source pixel and bid for its target slot (AN:279-303, 358) ----
    // FOUR pixels per trip (i, i + BT, i + 2 BT, i + 3 BT): this phase has registers to spare, and four
    // independent estimate chains hide more of their own latency than two.  D0 / I0 are read through
    // running pointers WITHOUT bounds guards: the prefetch runs up to 8 BT pixels past the level, into
    // the rest of the record or the slack behind the store (kBatchStoreSlackBytes); whatever comes
    // back there is masked by the in-range tests.
    unsigned long long valid = 0ull;
    const int quads = (trips + 1) >> 1;          // four-pixel trips of this thread
    if (COLFIX) {
      // ---- fp32 estimate (see est32_margins).  Per-thread constants of the iteration, rounded once ----
      unsigned ex = sh->ex, ey = sh->ey;             // computed once, by the thread that published the pose
      // (a pose or depth range that is not an ordinary number makes est32_margins return "nothing trusted" by itself)
      if (!(lv.est32 && finite_pose) || lv.exact_always) ex = ey = kFrac32One;   // nothing trusted: every pixel takes warp_exact
      const unsigned limx = ex < kFrac32One / 2 ? kFrac32One - 2u * ex : 0u, limy = ey < kFrac32One / 2 ? kFrac32One - 2u * ey : 0u;
      const float a0f = (float)(fma(T.R00, my_cxi, T.R02) - my_cxi * fma(T.R20, my_cxi, T.R22)), b0f = (float)fma(-T.R21, my_cxi, T.R01);
      const float a1f = (float)fma(T.R10, my_cxi, T.R12), b1f = (float)((T.R11 - T.R22) - T.R20 * my_cxi);
      const float a2f = (float)fma(T.R20, my_cxi, T.R22 - 1.0), e0f = (float)fma(-my_cxi, T.z, T.x), ztf = (float)T.z;
      const float fxsf = (float)(fx * (double)kFrac32One), fysf = (float)(fy * (double)kFrac32One);
      const int dr1 = BT / cols;                   // rows between two consecutive pixels of a thread
      const int cprime = c0_first - kMagic32Whole;
      int rprime = r0_first - kMagic32Whole;       // row of the trip's first pixel, mantissa offset folded in
      const char* rq = (const char*)(tb.rowf + r0_first);
      constexpr int W = kPhaseAWidth;              // pixels per trip: independent estimate chains in flight per thread
      const int groups = (2 * trips + W - 1) / W;  // W-pixel trips of this thread
      const int rq_step = W * dr1 * (int)sizeof(float4);
      const float* pf = L.gD32 + tid;
      const unsigned short* pu = L.gI0 + tid;
      float p[W], f[W]; unsigned u[W], w[W];
#pragma unroll
      for (int j = 0; j < W; ++j) { p[j] = first_f[j]; u[j] = first_u[j]; f[j] = 0.f; w[j] = 0u; }
      unsigned vhi = 0u, vlo = 0u, uhi = 0u, ulo = 0u;   // validity / "needs the exact warp" bits, shifted in at the top
      unsigned bid = (unsigned)(tid + 1) << 16;
      auto trip = [&](const float (&cd)[W], const unsigned (&cu)[W], float (&nd)[W], unsigned (&nu)[W], const int i) {
#pragma unroll
        for (int j = 0; j < W; ++j) { nd[j] = ldg_f32(pf + (W + j) * BT); nu[j] = ldg_u16(pu + (W + j) * BT); }
        pf += W * BT; pu += W * BT;
        unsigned vbits = 0u, ubits = 0u;
#pragma unroll
        for (int j = 0; j < W; ++j) {
          const float4 rf = *(const float4*)(rq + j * dr1 * (int)sizeof(float4));
          const float d = cd[j];
          const float D0 = fmaf(b0f, rf.x, a0f);
          const float D1 = fmaf(b1f, rf.x, a1f) + rf.w;
          const float Z = d + fmaf(d, a2f + rf.z, ztf);
          const float iz = rcp_approx_f32(Z);
          const unsigned ux = __float_as_uint(__fmaf_rd(fmaf(d, D0, e0f) * iz, fxsf, kMagic32));
          const unsigned uy = __float_as_uint(__fmaf_rd(fmaf(d, D1, rf.y) * iz, fysf, kMagic32));
          const bool dep = (d > 0.f) & (j == 0 || i + j * BT < n);                    // range test of AN:279-280, decided by the pyramid kernel
          const bool sure = (((ux & (kFrac32One - 1u)) - ex) < limx) & (((uy & (kFrac32One - 1u)) - ey) < limy) & (fmaf(d, -0.5f, Z) > 0.f);
          const int tj = (int)(ux >> kFrac32Bits) + cprime, ti = (int)(uy >> kFrac32Bits) + rprime + j * dr1;
          const bool ok = dep & sure & ((unsigned)tj < (unsigned)cols) & ((unsigned)ti < (unsigned)rows);
          smem_red_max(ok ? L.sWinAddr + 4u * (unsigned)(ti * cols + tj) : dummy, bid + ((unsigned)(j * BT) << 16) + cu[j]);
          vbits |= (unsigned)ok << (32 - W + j);
          ubits |= (unsigned)(dep & !sure) << (32 - W + j);
        }
        bid += (unsigned)(W * BT) << 16;
        vlo = __funnelshift_r(vlo, vhi, W); vhi = (vhi >> W) | vbits;
        ulo = __funnelshift_r(ulo, uhi, W); uhi = (uhi >> W) | ubits;
        rq += rq_step; rprime += W * dr1;
      };
      int i = tid;
      if (groups & 1) {
        trip(p, u, f, w, i);
#pragma unroll
        for (int j = 0; j < W; ++j) { p[j] = f[j]; u[j] = w[j]; }
        i += W * BT;
      }
      for (; i < n; i += 2 * W * BT) {
        trip(p, u, f, w, i);
        trip(f, w, p, u, i + W * BT);
      }
      valid = ((unsigned long long)vhi << 32) | vlo;
      valid = groups > 0 ? valid >> (64 - W * groups) : 0ull;
      unsigned long long unsure = ((unsigned long long)uhi << 32) | ulo;
      unsure = groups > 0 ? unsure >> (64 - W * groups) : 0ull;
      // ---- the pixels the estimate could not decide (a few per warp and iteration): the reference's own arithmetic ----
      while (unsure) {
        const int k = __ffsll((long long)unsure) - 1;
        unsure &= unsure - 1ull;
        const int px = tid + k * BT;
        const double d = __ldg(L.gD0 + px);
        const WarpA a = warp_exact(&sh->pose, my_cx, tb.ry[px / cols], d, fx, fy, ox, oy, inv_fx, inv_fy);
        const bool ok = ((unsigned)a.tj < (unsigned)cols) & ((unsigned)a.ti < (unsigned)rows) & (min_depth < d) & (d < max_depth);
        if (ok) {
          smem_red_max(L.sWinAddr + 4u * (unsigned)(a.ti * cols + a.tj), ((unsigned)(px + 1) << 16) + (unsigned)__ldg(L.gI0 + px));
          valid |= 1ull << k;
        }
      }
    } else {
      int rr[4], cc[4];
      const double2* rp[4];                       // COLFIX: the thread's column never changes, the row pointers
#pragma unroll                                    // advance by a constant (rows past the level are zero padding)
      for (int j = 0; j < 4; ++j) {
        rr[j] = (tid + j * BT) / cols; cc[j] = (tid + j * BT) - rr[j] * cols;
        rp[j] = tb.row + kRowEntries * rr[j];
      }
      const double* pd = L.gD0 + tid;
      const unsigned short* pu = L.gI0 + tid;
      // register prefetch: the loads of the next trip are issued at the top of the current one
      double p[4], f[4]; unsigned u[4], w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { p[j] = first_d[j]; u[j] = first_u[j]; f[j] = 0.; w[j] = 0u; }
      unsigned vhi = 0u, vlo = 0u;     // validity bits enter at the top and shift down: bit k of `valid` = pixel k
      unsigned bid = (unsigned)(tid + 1) << 16;   // winner word of pixel i without its I0: (i + 1) << 16
      // one trip: prefetch the next trip's pixels into (nd, nu), process (cd, cu).  Two copies of the
      // trip alternate the roles of the two register sets, so nothing is moved.
      auto trip = [&](const double (&cd)[4], const unsigned (&cu)[4], double (&nd)[4], unsigned (&nu)[4], const int i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { nd[j] = ldg_f64(pd + (4 + j) * BT); nu[j] = ldg_u16(pu + (4 + j) * BT); }
        pd += 4 * BT; pu += 4 * BT;
        WarpA a[4]; bool dep[4], ex[4];
        bool any = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ColRegsA ca = mycolA;
          if (!COLFIX) {
            const double2 t = tb.colA[cc[j]];
            ca.as = make_double2(__dmul_rn(K.fxs, t.x), __dmul_rn(K.fys, t.y)); ca.bx = tb.colB[cc[j]].x;
            rp[j] = tb.row + kRowEntries * rr[j];
          }
          bool unc;
          a[j] = warp_estimate(K, ca, rp[j][4], rp[j][1].x, cd[j], thr, zmin_hi, unc);
          dep[j] = (min_depth < cd[j]) & (cd[j] < max_depth) & (j == 0 || i + j * BT < n);   // strict bounds, AN:279-280
          ex[j] = dep[j] & unc;
          any |= ex[j];
        }
        if (any) {                                                             // rare: ~2e-4 of the pixels
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (ex[j]) {
              const int q = COLFIX ? (i + j * BT) / cols : rr[j];
              a[j] = warp_exact(&sh->pose, COLFIX ? my_cx : tb.cx[cc[j]], tb.ry[q], cd[j], fx, fy, ox, oy, inv_fx, inv_fy);
            }
        }
        unsigned bits = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool ok = ((unsigned)a[j].tj < (unsigned)cols) & ((unsigned)a[j].ti < (unsigned)rows) & dep[j];
          smem_red_max(ok ? L.sWinAddr + 4u * (unsigned)(a[j].ti * cols + a[j].tj) : dummy, bid + ((unsigned)(j * BT) << 16) + cu[j]);
          bits |= (unsigned)ok << (28 + j);
        }
        bid += (unsigned)(4 * BT) << 16;
        vlo = __funnelshift_r(vlo, vhi, 4);
        vhi = (vhi >> 4) | bits;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (COLFIX) rp[j] = (const double2*)((const char*)rp[j] + 2 * rstep_bytes);
          else { cc[j] += dc4; rr[j] += dr4; if (cc[j] >= cols) { cc[j] -= cols; ++rr[j]; } }
        }
      };
      // An odd trip count is peeled off in front, so that the two copies inside the loop form ONE basic
      // block: with an exit test between them ptxas sinks the first copy's prefetch below the test,
      // right in front of its use.
      int i = tid;
      if (quads & 1) {
        trip(p, u, f, w, i);
#pragma unroll
        for (int j = 0; j < 4; ++j) { p[j] = f[j]; u[j] = w[j]; }
        i += 4 * BT;
      }
      for (; i < n; i += 8 * BT) {
        trip(p, u, f, w, i);
        trip(f, w, p, u, i + 4 * BT);
      }
      valid = ((unsigned long long)vhi << 32) | vlo;
      valid = quads > 0 ? valid >> (64 - 4 * quads) : 0ull;
    }
    SEC_MARK(1);
    __syncthreads();
    SEC_MARK(2);
    // ---- phase B: residual + Jacobian + normal equations (AN:308-366, 538-539) ----
    // The second pixel of the last trip may lie past the level: its slots are padding (winner word
    // 0, so residual 0) and its validity bit is 0 (so its Jacobian row is 0).
    double acc[28];
#pragma unroll
    for (int v = 0; v < 28; ++v) acc[v] = 0.;
    {
      int r0 = r0_first, c0 = c0_first, r1 = r1_first, c1 = c1_first;
      const double2* rp0 = tb.row + kRowEntries * r0_first;
      const double2* rp1 = tb.row + kRowEntries * r1_first;
      const double* pd = L.gD0 + tid;
      unsigned* pw = L.sWin + tid;
      const unsigned* pg = L.sG + tid;
      const unsigned short* pi1 = L.sI1 + tid;
      unsigned long long vm = valid;
      double p0 = first_d[0], p1 = first_d[1];
      auto trip = [&](const double c0_, const double c1_, double& n0, double& n1) {
        n0 = ldg_f64(pd + 2 * BT); n1 = ldg_f64(pd + 3 * BT);
        // scheduling fence: at the register limit ptxas otherwise sinks the two loads towards their use.
        // Only the lanes that are here take part (trip counts differ between lanes when n % (2 BT) != 0).
        __syncwarp(__activemask());
        pd += 2 * BT;
        const unsigned wa = pw[0], wb = pw[BT];
        pw[0] = 0u; pw[BT] = 0u;
        const int da = (int)pi1[0] - (int)(wa & 0xffffu), db = (int)pi1[BT] - (int)(wb & 0xffffu);
        const double resa = (double)(wa ? da : 0), resb = (double)(wb ? db : 0);
        ColRegs ca0 = mycol, ca1 = mycol;
        if (!COLFIX) {
          ca0.a = tb.colA[c0]; ca0.b = tb.colB[c0]; ca0.cxix = MODE == 0 ? __dmul_rn(tb.cxi[c0], K.x) : 0.;   // not contracted: same bits as mycol.cxix
          ca1.a = tb.colA[c1]; ca1.b = tb.colB[c1]; ca1.cxix = MODE == 0 ? __dmul_rn(tb.cxi[c1], K.x) : 0.;
          rp0 = tb.row + kRowEntries * r0; rp1 = tb.row + kRowEntries * r1;
        }
        const unsigned vbits = (unsigned)vm;
        double Ja[6], Jb[6];
        jacobian_row<MODE>(K, ca0, rp0[0], rp0[1], rp0[2], rp0[3], c0_, (vbits & 1u) != 0, pg[0], Ja);
        jacobian_row<MODE>(K, ca1, rp1[0], rp1[1], rp1[2], rp1[3], c1_, (vbits & 2u) != 0, pg[BT], Jb);
        if (STATS) acc[27] = fma(resa, resa, acc[27]);   // sum r^2: only the iteration log reports it (the reference has no cost)
        accumulate_row(acc, Ja, resa);
        if (STATS) acc[27] = fma(resb, resb, acc[27]);
        accumulate_row(acc, Jb, resb);
        vm >>= 2;
        pw += 2 * BT; pg += 2 * BT; pi1 += 2 * BT;
        if (COLFIX) { rp0 = (const double2*)((const char*)rp0 + rstep_bytes); rp1 = (const double2*)((const char*)rp1 + rstep_bytes); }
        else {
          c0 += dc2; r0 += dr2; if (c0 >= cols) { c0 -= cols; ++r0; }
          c1 += dc2; r1 += dr2; if (c1 >= cols) { c1 -= cols; ++r1; }
        }
      };
      double f0 = 0., f1 = 0.;
      int i = tid;
      if (trips & 1) {
        trip(p0, p1, f0, f1);
        p0 = f0; p1 = f1; i += 2 * BT;
      }
      for (; i < n; i += 4 * BT) {
        trip(p0, p1, f0, f1);
        trip(f0, f1, p0, p1);
      }
    }
    SEC_MARK(3);
    // first trip of the next iteration: in flight during the reduction and the solve
#pragma unroll
    for (int j = 0; j < FW; ++j) {
      if (COLFIX) first_f[j] = ldg_f32(L.gD32 + tid + j * BT);
      if (!COLFIX || j < 2) first_d[j] = ldg_f64(L.gD0 + tid + j * BT);
      first_u[j] = ldg_u16(L.gI0 + tid + j * BT);
    }
    // ---- deterministic reduction: 31 shuffle-adds per warp, warps summed in index order ----
    {
      double x[32];
#pragma unroll
      for (int v = 0; v < 28; ++v) x[v] = acc[v];
      x[28] = (double)__popcll(valid); x[29] = 0.; x[30] = 0.; x[31] = 0.;
      L.sRed[wid * 32 + lane] = warp_transpose_sum(x, lane);
    }
    __syncthreads();
    SEC_MARK(4);
    if (wid == 0) {
      double t0 = 0., t1 = 0.;   // two interleaved chains, fixed order
#pragma unroll
      for (int w = 0; w < NW; w += 2) { t0 += L.sRed[w * 32 + lane]; if (w + 1 < NW) t1 += L.sRed[(w + 1) * 32 + lane]; }
      warp_gn_step((t0 + t1) * scale, lane, lv, it, L.pair, sh, log);
    }
    SEC_MARK(5);
    __syncthreads();
    if (sh->done) break;
  }
  SEC_MARK(6);
}

// K3-batch, one launch per ACTIVE pyramid level (coarse to fine; the state of every pair travels
// through `states` between launches).  Persistent CTAs fetch pairs from a global counter (iteration
// counts differ between pairs, so static assignment leaves SMs idle at the tail).  A small level
// runs as 3 CTAs of 160 threads per SM, so that the serial part of one pair's iteration (barriers,
// the 6x6 solve) overlaps the pixel loops of two other pairs; a level that needs most of the
// shared memory runs as 1 CTA of 480 threads.  Resident in shared memory for the level:
//   sWin u32[n]  winner word per TARGET slot: (source index + 1) << 16 | I0 tap sum of that source;
//                a native 32-bit shared atomicMax keeps the largest source index == the reference's
//                raster-order last-writer-wins (AN:358) and carries the winner's intensity along
//   sG   u32[n]  Scharr numerators of I1 at the pixel (gx low s16, gy high s16), exact integers,
//                computed once per level from the resident I1 tap sums (AN:165-189)
//   sI1  u16[n]  I1 tap sums (value = sum / 1020)
//   tables       see struct Tables
// D0 (fp64) and I0 (u16) are streamed from the pair's record (L2) with register prefetch.
// Thread t owns pixels t, t+BT, ...; whether pixel k of a thread is valid under the current pose
// stays in a 64-bit register mask between the two phases of an iteration.  The thread -> pixel
// mapping is a pure function of the level size, so results do not depend on grid, batch or GPU.
template <int MODE, int BT, int MINB, bool STATS>
__global__ void __launch_bounds__(BT, MINB) k_batch_level(const __grid_constant__ BatchLevelParams lv,
                                                          const uint8_t* __restrict__ store,
                                                          const double* __restrict__ init_states, double* __restrict__ states,
                                                          int32_t* __restrict__ iters, phovo_iter_stats* __restrict__ log,
                                                          int32_t* __restrict__ log_counts, unsigned int* __restrict__ next_pair) {
  constexpr int NW = BT / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int rows = lv.rows, cols = lv.cols, n = lv.n;
  const int nal = padded_slots(n, BT);
  unsigned* sWin = (unsigned*)smem_raw;
  unsigned* sG = sWin + nal;
  unsigned short* sI1 = (unsigned short*)(sG + nal);
  double* sTab = (double*)(sI1 + nal);
  double* sRed = sTab + ((table_doubles(rows, cols, BT) + 1) & ~1);
  BatchShared* sh = (BatchShared*)(sRed + NW * 32);
  unsigned* sDummy = (unsigned*)(sh + 1);            // 32 slots that absorb the bids of pixels without a target
  const int tid = threadIdx.x;

  // The launches of consecutive levels overlap (programmatic dependent launch): the next level's grid may start
  // as soon as every CTA of this one is running, its CTAs get an SM when this level's persistent CTAs retire, and
  // it waits PER PAIR (below) -- so the SMs that run dry in the tail of this launch (iteration counts differ 4x
  // between pairs) start on the next level instead of idling.  Every CTA of this grid is resident before any
  // CTA of the next one can be scheduled, so the waits below cannot starve this grid.
  asm volatile("griddepcontrol.launch_dependents;");
#ifdef PHOVO_SECTION_CLOCKS
  const long long kernel_t0 = clock64();
#endif
  for (;;) {
    __syncthreads();   // the previous pair's outputs have been read from shared memory
    if (tid == 0) {
      const int pair = (int)atomicAdd(next_pair, 1u);
      sh->pair = pair;
      if (pair < lv.num_pairs) {
        if (lv.prev_level >= 0) {
          // the coarser level publishes its iteration count (>= 1) for the pair LAST, with release semantics
          const int32_t* flag = iters + (size_t)pair * PHOVO_MAX_LEVELS + lv.prev_level;
          int v;
          for (;;) {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
            if (v != 0) break;
            __nanosleep(200);
          }
        }
        double s[6];
        const double* src = lv.first ? init_states : states;     // the first level starts from the caller's state
        for (int k = 0; k < 6; ++k) s[k] = src ? src[(size_t)pair * 6 + k] : 0.;
        Pose P;
        pose_from_state(s, P);
        for (int k = 0; k < 6; ++k) sh->pose.state[k] = s[k];
        pose_store(P, &sh->pose);
        est32_publish(lv, P, sh);
        sh->pose.log_count = (lv.first || !log_counts) ? 0 : log_counts[pair];
        sh->done = 0; sh->iteration = 0;
      }
    }
    __syncthreads();
    const int pair = sh->pair;
    if (pair >= lv.num_pairs) break;
    const uint8_t* rec = store + (size_t)pair * lv.record_bytes;

    LevelCtx L;
    L.pair = pair;
    L.gD0 = (const double*)(rec + lv.off_D0);
    L.gD32 = (const float*)(rec + lv.off_D32);
    L.gI0 = (const unsigned short*)(rec + lv.off_I0);
    L.sWin = sWin; L.sG = sG; L.sI1 = sI1; L.sRed = sRed;
    L.sWinAddr = (unsigned)__cvta_generic_to_shared(sWin);
    L.sDummyAddr = (unsigned)__cvta_generic_to_shared(sDummy);
    const int pad_rows = table_pad_rows(cols, BT);
    Tables& tb = L.tb;
    tb.colA = (double2*)sTab; tb.colB = tb.colA + cols; tb.row = tb.colB + cols;
    tb.rowf = (float4*)(tb.row + kRowEntries * (rows + pad_rows));
    tb.cx = (double*)(tb.rowf + rows + pad_rows); tb.ry = tb.cx + cols; tb.cxi = tb.ry + rows; tb.ryi = tb.cxi + cols;
    {
      // record -> shared memory, 16-byte vectors (record offsets are 16-byte aligned)
      const double ox = lv.ox, oy = lv.oy, inv_fx = lv.inv_fx, inv_fy = lv.inv_fy;
      const uint4* gI1 = (const uint4*)(rec + lv.off_I1);
      uint4* i14 = (uint4*)sI1; uint4* w4 = (uint4*)sWin;
      const int ni = (n * 2 + 15) / 16, nw = nal / 4;
      for (int k = tid; k < ni; k += BT) i14[k] = __ldg(gI1 + k);
      for (int k = tid; k < nw; k += BT) w4[k] = make_uint4(0, 0, 0, 0);                 // level + padding: no winners
      for (int k = n + tid; k < nal; k += BT) sG[k] = 0u;                               // padding slots (read, then masked)
      for (int k = kRowEntries * rows + tid; k < kRowEntries * (rows + pad_rows); k += BT) tb.row[k] = make_double2(0., 0.);
      for (int k = rows + tid; k < rows + pad_rows; k += BT) tb.rowf[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = tid; k < cols; k += BT) { const double v = __dsub_rn((double)k, ox); tb.cx[k] = v; tb.cxi[k] = v * inv_fx; }   // AN:282
      for (int k = tid; k < rows; k += BT) { const double v = __dsub_rn((double)k, oy); tb.ry[k] = v; tb.ryi[k] = v * inv_fy; }   // AN:286
    }
    __syncthreads();
    {
      // Scharr numerators of I1 (AN:181-187), reflect-101: |gx|,|gy| <= 16 * 1020 fits s16
      const int dr = BT / cols, dc = BT - dr * cols;
      int r = tid / cols, c = tid - r * cols;
      for (int i = tid; i < n; i += BT) {
        const int rm = r > 0 ? r - 1 : (rows > 1 ? 1 : 0), rp = r < rows - 1 ? r + 1 : (rows > 1 ? rows - 2 : 0);
        const int cm = c > 0 ? c - 1 : (cols > 1 ? 1 : 0), cp = c < cols - 1 ? c + 1 : (cols > 1 ? cols - 2 : 0);
        const unsigned short* Rm = sI1 + rm * cols; const unsigned short* R0 = sI1 + r * cols; const unsigned short* Rp = sI1 + rp * cols;
        const int a00 = Rm[cm], a01 = Rm[c], a02 = Rm[cp], a10 = R0[cm], a12 = R0[cp], a20 = Rp[cm], a21 = Rp[c], a22 = Rp[cp];
        const int gxn = 10 * (a12 - a10) + 3 * ((a22 - a20) + (a02 - a00));
        const int gyn = (3 * a20 + 10 * a21 + 3 * a22) - (3 * a00 + 10 * a01 + 3 * a02);
        sG[i] = ((unsigned)gxn & 0xffffu) | ((unsigned)gyn << 16);
        c += dc; r += dr;
        if (c >= cols) { c -= cols; ++r; }
      }
    }
    // (the first barrier inside gn_level orders these writes before the pixel loops)
    if (BT % cols == 0 && !lv.force_generic && lv.est32) gn_level<MODE, true, BT, STATS>(lv, L, sh, STATS ? log : nullptr);
    else gn_level<MODE, false, BT, STATS>(lv, L, sh, STATS ? log : nullptr);
    __syncthreads();
    if (tid < 6) states[(size_t)pair * 6 + tid] = sh->pose.state[tid];
    if (tid == 0 && log_counts) log_counts[pair] = sh->pose.log_count;
    __syncthreads();
    if (tid == 0) {   // the pair is ready for the next level: state, log count (and the log) are visible before the count
      __threadfence();
      const int done_iterations = sh->iteration;
      asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(iters + (size_t)pair * PHOVO_MAX_LEVELS + lv.level), "r"(done_iterations) : "memory");
    }
  }
#ifdef PHOVO_SECTION_CLOCKS
  if (tid == 0) atomicAdd(&g_section_clocks[BT == kBatchThreads ? 1 : 0][7], (unsigned long long)(clock64() - kernel_t0));
#endif
}

}  // namespace

#ifdef PHOVO_SECTION_CLOCKS
extern "C" int phovo_debug_section_clocks(unsigned long long* out16, int reset) {
  if (out16 && cudaMemcpyFromSymbol(out16, g_section_clocks, sizeof(g_section_clocks)) != cudaSuccess) return -1;
  if (reset) { unsigned long long z[16] = {}; if (cudaMemcpyToSymbol(g_section_clocks, z, sizeof(z)) != cudaSuccess) return -1; }
  return 0;
}
#endif

// dynamic shared memory of one CTA working on a level of rows x cols pixels with `threads` threads
static size_t level_smem_bytes(int rows, int cols, int threads) {
  const size_t nal = (size_t)padded_slots(rows * cols, threads);
  const size_t tab = ((size_t)table_doubles(rows, cols, threads) + 1) & ~(size_t)1;
  return nal * 10 + tab * sizeof(double) + (size_t)(threads / 32) * 32 * sizeof(double) + sizeof(BatchShared) + 32 * sizeof(unsigned) + 64;
}

// A small level runs as 3 CTAs of kBatchThreadsSmall per SM (each gets a third of the 227 KB).
bool batch_level_is_small(int rows, int cols) {
  return rows * cols <= kBatchSmallLevelPixels && level_smem_bytes(rows, cols, kBatchThreadsSmall) <= (size_t)(227 * 1024) / 3 - 1024;
}

size_t batch_level_smem_bytes(int rows, int cols) {
  return level_smem_bytes(rows, cols, batch_level_is_small(rows, cols) ? kBatchThreadsSmall : kBatchThreads);
}

template <int MODE, int BT, int MINB>
static cudaError_t set_level_smem(int bytes) {
  cudaError_t e = cudaFuncSetAttribute(k_batch_level<MODE, BT, MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k_batch_level<MODE, BT, MINB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

cudaError_t batch_align_prepare() {
  cudaError_t e;
  const int big = 227 * 1024, small = (227 * 1024) / 3 - 1024;
  if ((e = set_level_smem<0, kBatchThreads, 1>(big)) != cudaSuccess) return e;
  if ((e = set_level_smem<1, kBatchThreads, 1>(big)) != cudaSuccess) return e;
  if ((e = set_level_smem<0, kBatchThreadsSmall, 3>(small)) != cudaSuccess) return e;
  return set_level_smem<1, kBatchThreadsSmall, 3>(small);
}

int launch_batch_pyramid(cudaStream_t stream, const BatchParams& bp, const uint8_t* gray0, const void* depth0,
                         int depth_type, double depth_scale, const uint8_t* gray1, uint8_t* store) {
  dim3 grid((bp.px_offset[bp.num_active] + 255) / 256, bp.num_pairs);
  switch (depth_type) {
    case SRC_F32: k_batch_pyramid<float><<<grid, 256, 0, stream>>>(bp, gray0, (const float*)depth0, depth_scale, gray1, store); break;
    case SRC_U16: k_batch_pyramid<uint16_t><<<grid, 256, 0, stream>>>(bp, gray0, (const uint16_t*)depth0, depth_scale, gray1, store); break;
    default:      k_batch_pyramid<double><<<grid, 256, 0, stream>>>(bp, gray0, (const double*)depth0, depth_scale, gray1, store); break;
  }
  return 1;
}

// One launch per active level, coarse to fine.  `next_pair` must hold one zeroed counter per level.
int launch_batch_align(cudaStream_t stream, const BatchParams& bp, int sm_count, const uint8_t* store,
                       const double* init_states, double* states, int32_t* iters, phovo_iter_stats* log, int32_t* log_counts,
                       unsigned int* next_pair) {
  int launches = 0;
  for (int a = 0; a < bp.num_active; ++a) {
    const int rows = bp.lrows[a], cols = bp.lcols[a];
    const BatchLevelParams lv = level_params(bp, a);
    const size_t smem = batch_level_smem_bytes(rows, cols);
    const bool fixed = bp.mode == PHOVO_MODE_ANALYTIC_FIXED;
    // STATS: the kernel that also accumulates sum r^2 and writes the iteration log
#define PHOVO_LAUNCH_LEVEL(MODE, BT, MINB, grid)                                                                                        \
  do {                                                                                                                                  \
    cudaLaunchConfig_t cfg = {};                                                                                                        \
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(BT); cfg.dynamicSmemBytes = smem; cfg.stream = stream;                                \
    cudaLaunchAttribute attr[1];                                                                                                        \
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                                                    \
    attr[0].val.programmaticStreamSerializationAllowed = 1;                                                                             \
    cfg.attrs = attr; cfg.numAttrs = a > 0 ? 1 : 0;   /* levels after the first may start while the previous one drains */             \
    if (log) cudaLaunchKernelEx(&cfg, k_batch_level<MODE, BT, MINB, true>, lv, store, init_states, states, iters, log, log_counts, next_pair + a);   \
    else cudaLaunchKernelEx(&cfg, k_batch_level<MODE, BT, MINB, false>, lv, store, init_states, states, iters, log, log_counts, next_pair + a);      \
  } while (0)
    if (batch_level_is_small(rows, cols)) {
      const int grid = min(bp.num_pairs, 3 * sm_count);
      if (fixed) PHOVO_LAUNCH_LEVEL(1, kBatchThreadsSmall, 3, grid);
      else PHOVO_LAUNCH_LEVEL(0, kBatchThreadsSmall, 3, grid);
    } else {
      const int grid = min(bp.num_pairs, sm_count);
      if (fixed) PHOVO_LAUNCH_LEVEL(1, kBatchThreads, 1, grid);
      else PHOVO_LAUNCH_LEVEL(0, kBatchThreads, 1, grid);
    }
#undef PHOVO_LAUNCH_LEVEL
    ++launches;
  }
  return launches;
}

}  // namespace phovo
