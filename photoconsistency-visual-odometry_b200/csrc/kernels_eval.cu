// kernels_eval.cu -- normal equations of many pairs at given states, at any pyramid level
// (phovo_batch_eval_normal_equations; the analytic modes of k_winner + k_normal_eq for a chunk of pairs).
//
//   k_eval_winner     : grid (tiles, pairs).  Warp every source pixel with the reference's arithmetic
//                       (warp_pixel<false>: round half away, AN:279-303), bid atomicMax(keys[t], i + 1) --
//                       raster-order last writer wins (AN:358) -- and record the pixel's validity.
//   k_eval_accumulate : grid (tiles, pairs).  Residual I1[i] - I0[winner - 1] gathered through the key (the key is
//                       cleared for the next chunk), Jacobian of the valid pixels (analytic_jacobian, shared with
//                       k_normal_eq) with Scharr gradients of I1 at the source index, 29 sums reduced per tile in a
//                       fixed order.
//   k_eval_reduce     : one warp per pair sums its tiles in index order into H, g, cost, num_valid.
//
// The photometric + depth solver (phovo_batch_eval_normal_equations_with_target_depth) has its 2N-row system:
// k_eval_target_depth (D1 and its Scharr / max_depth at the level, per-tile sums for the gain), k_eval_gain,
// k_eval_winner_bi (keys 2i+1 / 2i+2 over 2N slots) and k_eval_accumulate_bi (bi_row_owner + bi_jacobian_core), then
// the same k_eval_reduce over the tiles of the 2N slots.
//
// Intensities are integer tap sums (value = sum / 1020: 4 v at level 0, the pyramid kernel's u16 records above), so
// residuals and gradient numerators are exact integers until the one scaling.  The tile size is a constant and a tile
// never spans two pairs, so the grouping of every sum depends on the level size only: results are bitwise
// reproducible and do not depend on the chunking, the GPU or which pairs share a call.  No floating-point atomics.
#include <type_traits>

#include "phovo_batch.h"
#include "phovo_device.cuh"
#include "phovo_kernels.h"
#include "phovo_level.cuh"

namespace phovo {
namespace {

// Source images of pair p: the caller's frames (level 0) or the pyramid kernel's record (REC, level >= 1).
template <typename DT, bool REC>
__device__ __forceinline__ double ev_depth(const EvalLevel& E, size_t p, int n, int i) {
  if (REC) return __ldg((const double*)(E.store + p * E.record_bytes + E.off_D0) + i);
  return depth_at<DT>((const DT*)E.depth + p * n + i, E.depth_scale);
}
template <bool REC>
__device__ __forceinline__ int ev_i0(const EvalLevel& E, size_t p, int n, int i) {
  if (REC) return __ldg((const uint16_t*)(E.store + p * E.record_bytes + E.off_I0) + i);
  return 4 * (int)__ldg(E.gray0 + p * n + i);
}
template <bool REC>
__device__ __forceinline__ const void* ev_i1_base(const EvalLevel& E, size_t p, int n) {
  if (REC) return E.store + p * E.record_bytes + E.off_I1;
  return E.gray1 + p * n;
}
template <bool REC>
__device__ __forceinline__ int ev_i1(const void* base, int i) {
  if (REC) return __ldg((const uint16_t*)base + i);
  return 4 * (int)__ldg((const uint8_t*)base + i);
}

// Scharr numerators of I1 at level pixel (r, c) (AN:181-187; at the SOURCE index, AN:346-347), reflect-101 borders
template <bool REC>
__device__ __forceinline__ void ev_scharr_i1(const void* I1, int rows, int cols, int r, int c, int& gxn, int& gyn) {
  const int rm = r > 0 ? r - 1 : (rows > 1 ? 1 : 0), rp = r < rows - 1 ? r + 1 : (rows > 1 ? rows - 2 : 0);
  const int cm = c > 0 ? c - 1 : (cols > 1 ? 1 : 0), cp = c < cols - 1 ? c + 1 : (cols > 1 ? cols - 2 : 0);
  const int a00 = ev_i1<REC>(I1, rm * cols + cm), a01 = ev_i1<REC>(I1, rm * cols + c), a02 = ev_i1<REC>(I1, rm * cols + cp);
  const int a10 = ev_i1<REC>(I1, r * cols + cm), a12 = ev_i1<REC>(I1, r * cols + cp);
  const int a20 = ev_i1<REC>(I1, rp * cols + cm), a21 = ev_i1<REC>(I1, rp * cols + c), a22 = ev_i1<REC>(I1, rp * cols + cp);
  gxn = 10 * (a12 - a10) + 3 * ((a22 - a20) + (a02 - a00));
  gyn = (3 * a20 + 10 * a21 + 3 * a22) - (3 * a00 + 10 * a01 + 3 * a02);
}

template <typename DT, bool REC>
__global__ void __launch_bounds__(kEvalThreads) k_eval_winner(const __grid_constant__ EvalLevel E) {
  const size_t p = blockIdx.y;
  const int cols = E.L.cols, n = E.L.rows * cols;
  const int i0 = blockIdx.x * kEvalTile + threadIdx.x;
  double dv[kEvalPix];
#pragma unroll
  for (int j = 0; j < kEvalPix; ++j) {
    const int i = i0 + j * kEvalThreads;
    dv[j] = i < n ? ev_depth<DT, REC>(E, p, n, i) : 0.;
  }
  Pose T;
  pose_load(E.poses + p, T);
  uint32_t* pk = E.keys + p * n;
  uint8_t* pv = E.valid + p * n;
#pragma unroll
  for (int j = 0; j < kEvalPix; ++j) {
    const int i = i0 + j * kEvalThreads;
    if (i >= n) break;
    const int r = i / cols, c = i - r * cols;
    Warped w;
    const bool ok = warp_pixel<false>(E.L, T, r, c, dv[j], w);
    if (ok) atomicMax(pk + w.t, (uint32_t)(i + 1));
    pv[i] = ok;
  }
}

template <int MODE, typename DT, bool REC>
__global__ void __launch_bounds__(kEvalThreads) k_eval_accumulate(const __grid_constant__ EvalLevel E) {
  __shared__ double smem[(kEvalThreads / 32) * PHOVO_ACC_STRIDE];
  const size_t p = blockIdx.y;
  const int rows = E.L.rows, cols = E.L.cols, n = rows * cols;
  const int i0 = blockIdx.x * kEvalTile + threadIdx.x;
  uint32_t* pk = E.keys + p * n;
  const uint8_t* pv = E.valid + p * n;
  const void* I1 = ev_i1_base<REC>(E, p, n);
  Pose T;
  pose_load(E.poses + p, T);
  const double spsr = T.sp * T.sr, spcr = T.sp * T.cr;
  double acc[PHOVO_NACC];
#pragma unroll
  for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
  // not unrolled: eight copies of the Jacobian need 160 registers, one CTA per SM, and run slower (38 vs 28 ms for 4096
  // pairs at 640x480) than one pixel at a time with two CTAs per SM
  for (int j = 0; j < kEvalPix; ++j) {
    const int i = i0 + j * kEvalThreads;
    if (i >= n) break;
    const uint32_t key = pk[i];
    if (key) pk[i] = 0u;                            // clean for the next chunk
    double res = 0.;
    if (key) {
      res = (double)(ev_i1<REC>(I1, i) - ev_i0<REC>(E, p, n, (int)key - 1)) * (1.0 / 1020.0);
      acc[27] = fma(res, res, acc[27]);
    }
    if (!pv[i]) continue;                           // the winner pass decided (exact reference arithmetic)
    const int r = i / cols, c = i - r * cols;
    int gxn, gyn;
    ev_scharr_i1<REC>(I1, rows, cols, r, c, gxn, gyn);
    double J[6];
    analytic_jacobian<MODE>(E.L, T, spsr, spcr, r, c, ev_depth<DT, REC>(E, p, n, i), (double)gxn * E.grad_k,
                            (double)gyn * E.grad_k, J);
    accumulate_row(acc, J, res);
    acc[28] += 1.;
  }
  const double total = block_reduce<kEvalThreads>(acc, smem);
  if (threadIdx.x < PHOVO_NACC) E.partials[(p * E.tiles + blockIdx.x) * PHOVO_ACC_STRIDE + threadIdx.x] = total;
}

// One warp per pair: lane v < 29 sums value v over the pair's tiles in index order.
__global__ void __launch_bounds__(32) k_eval_reduce(const double* __restrict__ partials, int tiles, double* __restrict__ H,
                                                    double* __restrict__ g, double* __restrict__ cost, int32_t* __restrict__ num_valid) {
  const size_t p = blockIdx.x;
  const int v = threadIdx.x;
  if (v >= PHOVO_NACC) return;
  const double* src = partials + p * tiles * PHOVO_ACC_STRIDE + v;
  double s = 0.;
  for (int t = 0; t < tiles; ++t) s += src[(size_t)t * PHOVO_ACC_STRIDE];
  if (v < 21) H[p * 21 + v] = s;
  else if (v < 27) g[p * 6 + (v - 21)] = s;
  else if (v == 27) cost[p] = 0.5 * s;
  else num_valid[p] = (int32_t)s;
}

__global__ void k_eval_poses(const double* __restrict__ states, int num_pairs, PoseDev* __restrict__ poses) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= num_pairs) return;
  double s[6];
  for (int k = 0; k < 6; ++k) s[k] = states[(size_t)p * 6 + k];
  Pose P;
  pose_from_state(s, P);                          // as k_set_state: the same pose bit for bit
  for (int k = 0; k < 6; ++k) poses[p].state[k] = s[k];
  pose_store(P, poses + p);
}

// ---- photometric + depth solver (PHOVO_MODE_BIOBJECTIVE): the stacked 2N-row system of k_winner_bi / k_normal_eq_bi ----

// Target depth of the chunk at the level: D1, and the Scharr of D1 / max_depth scaled as the level's intensity
// gradients -- the per-pair path's launch_build_level, k_scale and k_scharr_store bit for bit (level_value from the
// full-resolution frame, the eight neighbours evaluated again, as k_build_levels does).  Per tile of pixels: the sum of
// the I1 tap sums (exact) and of D1 (fixed order), for the gain.  DT: element type of the caller's depth frames.
template <typename DT, bool REC>
__global__ void __launch_bounds__(kEvalThreads) k_eval_target_depth(const __grid_constant__ EvalLevel E,
                                                                    const __grid_constant__ EvalTargetDepth D) {
  __shared__ double s_sum[2][kEvalThreads / 32];
  const size_t p = blockIdx.y;
  const int lrows = E.L.rows, lcols = E.L.cols, n = lrows * lcols;
  const int i0 = blockIdx.x * kEvalTile + threadIdx.x;
  const size_t step = (size_t)D.cols * sizeof(DT);
  const void* src = (const char*)D.depth1 + p * D.rows * step;
  const double scale = (double)(1 << D.level);
  const void* I1 = ev_i1_base<REC>(E, p, n);
  double sd = 0.;
  int si = 0;
  for (int j = 0; j < kEvalPix; ++j) {
    const int i = i0 + j * kEvalThreads;
    if (i >= n) break;
    const int y = i / lcols, x = i - y * lcols;
    const int ys[3] = {reflect101(y - 1, lrows), y, reflect101(y + 1, lrows)};
    const int xs[3] = {reflect101(x - 1, lcols), x, reflect101(x + 1, lcols)};
    double t[3][3];
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) t[dy][dx] = level_value<DT>(src, step, D.depth_scale, D.rows, D.cols, D.level, scale, ys[dy], xs[dx]);
    const double d1 = t[1][1];
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) t[dy][dx] = __dmul_rn(t[dy][dx], D.inv_max_depth);
    double gx, gy;
    scharr_taps(t, D.ks0, D.ks1, gx, gy);
    D.D1[p * n + i] = d1;
    D.GxD[p * n + i] = gx;
    D.GyD[p * n + i] = gy;
    sd += d1;
    si += ev_i1<REC>(I1, i);
  }
  double si_d = (double)si;                         // < 2^22 per thread: exact
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sd += __shfl_xor_sync(0xffffffffu, sd, o);
    si_d += __shfl_xor_sync(0xffffffffu, si_d, o);
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { s_sum[0][wid] = si_d; s_sum[1][wid] = sd; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double s = 0.;
    for (int w = 0; w < kEvalThreads / 32; ++w) s += s_sum[threadIdx.x][w];
    D.sums[(p * E.tiles + blockIdx.x) * 2 + threadIdx.x] = s;
  }
}

// gain of pair p = mean(I1) / mean(D1) at the level (BiObjective.h:299).  One warp per pair: lane l sums tiles l, l + 32,
// ... in order, then a fixed butterfly over the lanes.
__global__ void __launch_bounds__(32) k_eval_gain(const __grid_constant__ EvalTargetDepth D, int tiles, int n) {
  const size_t p = blockIdx.x;
  const double* s = D.sums + p * tiles * 2;
  double si = 0., sd = 0.;
  for (int t = threadIdx.x; t < tiles; t += 32) { si += s[2 * t]; sd += s[2 * t + 1]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    si += __shfl_xor_sync(0xffffffffu, si, o);
    sd += __shfl_xor_sync(0xffffffffu, sd, o);
  }
  if (threadIdx.x == 0) D.gain[p] = (si / 1020.0 / (double)n) / (sd / (double)n);
}

// Winner pass of the 2N slots (k_winner_bi): key 2 i + 1 for the intensity write to slot t, 2 i + 2 for the depth write
// to slot 2 t, which comes after it; slots 2 t >= N exist, so a pair has 2N keys.
template <typename DT, bool REC>
__global__ void __launch_bounds__(kEvalThreads) k_eval_winner_bi(const __grid_constant__ EvalLevel E) {
  const size_t p = blockIdx.y;
  const int cols = E.L.cols, n = E.L.rows * cols;
  const int i0 = blockIdx.x * kEvalTile + threadIdx.x;
  double dv[kEvalPix];
#pragma unroll
  for (int j = 0; j < kEvalPix; ++j) {
    const int i = i0 + j * kEvalThreads;
    dv[j] = i < n ? ev_depth<DT, REC>(E, p, n, i) : 0.;
  }
  Pose T;
  pose_load(E.poses + p, T);
  uint32_t* pk = E.keys + p * 2 * (size_t)n;
  uint8_t* pv = E.valid + p * n;
#pragma unroll
  for (int j = 0; j < kEvalPix; ++j) {
    const int i = i0 + j * kEvalThreads;
    if (i >= n) break;
    const int r = i / cols, c = i - r * cols;
    Warped w;
    const bool ok = warp_pixel<false>(E.L, T, r, c, dv[j], w);
    if (ok) {
      atomicMax(pk + w.t, 2u * (uint32_t)i + 1u);
      atomicMax(pk + 2 * w.t, 2u * (uint32_t)i + 2u);
    }
    pv[i] = ok;
  }
}

// Accumulate pass over the 2N slots k: residual of slot k through its key (cleared for the next chunk), Jacobian row k
// (bi_row_owner + bi_jacobian_core, as k_normal_eq_bi), 29 sums per tile in a fixed order; valid pixels counted over k < N.
template <typename DT, bool REC>
__global__ void __launch_bounds__(kEvalThreads) k_eval_accumulate_bi(const __grid_constant__ EvalLevel E,
                                                                     const __grid_constant__ EvalTargetDepth D) {
  __shared__ double smem[(kEvalThreads / 32) * PHOVO_ACC_STRIDE];
  const size_t p = blockIdx.y;
  const int rows = E.L.rows, cols = E.L.cols, n = rows * cols;
  const int i0 = blockIdx.x * kEvalTile + threadIdx.x;
  uint32_t* pk = E.keys + p * 2 * (size_t)n;
  const uint8_t* pv = E.valid + p * n;
  const void* I1 = ev_i1_base<REC>(E, p, n);
  const double* D1 = D.D1 + p * n;
  const double gain = __ldg(D.gain + p);
  Pose T;
  pose_load(E.poses + p, T);
  const double spsr = T.sp * T.sr, spcr = T.sp * T.cr;
  double acc[PHOVO_NACC];
#pragma unroll
  for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
  for (int j = 0; j < kEvalPix; ++j) {
    const int k = i0 + j * kEvalThreads;
    if (k >= 2 * n) break;
    const uint32_t key = pk[k];
    if (key) pk[k] = 0u;                            // clean for the next chunk
    double res = 0.;
    if (key) {
      const int src = (int)((key - 1u) >> 1);
      if (((key - 1u) & 1u) == 0u) res = (double)(ev_i1<REC>(I1, k) - ev_i0<REC>(E, p, n, src)) * (1.0 / 1020.0);   // slot k = t
      else res = gain * (__ldg(D1 + (k >> 1)) - ev_depth<DT, REC>(E, p, n, src));                                     // slot k = 2 t
      acc[27] = fma(res, res, acc[27]);
    }
    const bool vk = k < n && pv[k];
    if (vk) acc[28] += 1.;
    bool depth_row;
    const int o = bi_row_owner(k, vk, pv[k >> 1] != 0, &depth_row);
    if (o < 0) continue;
    double gx, gy;
    if (depth_row) {
      gx = __ldg(D.GxD + p * n + o); gy = __ldg(D.GyD + p * n + o);
    } else {
      const int r = o / cols, c = o - r * cols;
      int gxn, gyn;
      ev_scharr_i1<REC>(I1, rows, cols, r, c, gxn, gyn);
      gx = (double)gxn * E.grad_k; gy = (double)gyn * E.grad_k;
    }
    double J[6];
    bi_jacobian_core(E.L, T, spsr, spcr, gain, o, depth_row, ev_depth<DT, REC>(E, p, n, o), gx, gy, J);
    accumulate_row(acc, J, res);
  }
  const double total = block_reduce<kEvalThreads>(acc, smem);
  if (threadIdx.x < PHOVO_NACC) E.partials[(p * D.tiles2 + blockIdx.x) * PHOVO_ACC_STRIDE + threadIdx.x] = total;
}

// DT: depth frames of the call; the source depth comes from the records (double) above level 0
template <typename DT, bool REC>
void launch_passes_bi(cudaStream_t stream, const EvalLevel& E, const EvalTargetDepth& D, int num_pairs) {
  using DT0 = typename std::conditional<REC, double, DT>::type;
  const dim3 grid((unsigned)E.tiles, (unsigned)num_pairs), grid2((unsigned)D.tiles2, (unsigned)num_pairs);
  k_eval_target_depth<DT, REC><<<grid, kEvalThreads, 0, stream>>>(E, D);
  k_eval_gain<<<num_pairs, 32, 0, stream>>>(D, E.tiles, E.L.rows * E.L.cols);
  k_eval_winner_bi<DT0, REC><<<grid, kEvalThreads, 0, stream>>>(E);
  k_eval_accumulate_bi<DT0, REC><<<grid2, kEvalThreads, 0, stream>>>(E, D);
}

template <bool REC>
void launch_bi(cudaStream_t stream, const EvalLevel& E, const EvalTargetDepth& D, int src_type, int num_pairs) {
  switch (src_type) {
    case SRC_F32: launch_passes_bi<float, REC>(stream, E, D, num_pairs); break;
    case SRC_U16: launch_passes_bi<uint16_t, REC>(stream, E, D, num_pairs); break;
    default:      launch_passes_bi<double, REC>(stream, E, D, num_pairs); break;
  }
}

template <int MODE, typename DT, bool REC>
void launch_passes(cudaStream_t stream, const EvalLevel& E, int num_pairs) {
  const dim3 grid((unsigned)E.tiles, (unsigned)num_pairs);
  k_eval_winner<DT, REC><<<grid, kEvalThreads, 0, stream>>>(E);
  k_eval_accumulate<MODE, DT, REC><<<grid, kEvalThreads, 0, stream>>>(E);
}

template <int MODE>
void launch_mode(cudaStream_t stream, const EvalLevel& E, int src_type, bool records, int num_pairs) {
  if (records) { launch_passes<MODE, double, true>(stream, E, num_pairs); return; }
  switch (src_type) {
    case SRC_F32: launch_passes<MODE, float, false>(stream, E, num_pairs); break;
    case SRC_U16: launch_passes<MODE, uint16_t, false>(stream, E, num_pairs); break;
    default:      launch_passes<MODE, double, false>(stream, E, num_pairs); break;
  }
}

}  // namespace

int launch_eval_poses(cudaStream_t stream, const double* states, int num_pairs, PoseDev* poses) {
  k_eval_poses<<<(num_pairs + 127) / 128, 128, 0, stream>>>(states, num_pairs, poses);
  return 1;
}

int launch_eval_normal_equations(cudaStream_t stream, const EvalLevel& E, int src_type, bool records, int num_pairs,
                                 double* out_H, double* out_g, double* out_cost, int32_t* out_valid) {
  if (E.L.mode == PHOVO_MODE_ANALYTIC_FIXED) launch_mode<1>(stream, E, src_type, records, num_pairs);
  else launch_mode<0>(stream, E, src_type, records, num_pairs);
  k_eval_reduce<<<num_pairs, 32, 0, stream>>>(E.partials, E.tiles, out_H, out_g, out_cost, out_valid);
  return 3;
}

int launch_eval_normal_equations_bi(cudaStream_t stream, const EvalLevel& E, const EvalTargetDepth& D, int src_type, bool records,
                                    int num_pairs, double* out_H, double* out_g, double* out_cost, int32_t* out_valid) {
  if (records) launch_bi<true>(stream, E, D, src_type, num_pairs);
  else launch_bi<false>(stream, E, D, src_type, num_pairs);
  k_eval_reduce<<<num_pairs, 32, 0, stream>>>(E.partials, D.tiles2, out_H, out_g, out_cost, out_valid);
  return 5;
}

}  // namespace phovo
