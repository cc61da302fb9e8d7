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
// Intensities are integer tap sums (value = sum / 1020: 4 v at level 0, the pyramid kernel's u16 records above), so
// residuals and gradient numerators are exact integers until the one scaling.  The tile size is a constant and a tile
// never spans two pairs, so the grouping of every sum depends on the level size only: results are bitwise
// reproducible and do not depend on the chunking, the GPU or which pairs share a call.  No floating-point atomics.
#include "phovo_batch.h"
#include "phovo_device.cuh"
#include "phovo_kernels.h"

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
    // Scharr numerators of I1 at the source index (AN:181-187, AN:346-347), reflect-101 borders
    const int rm = r > 0 ? r - 1 : (rows > 1 ? 1 : 0), rp = r < rows - 1 ? r + 1 : (rows > 1 ? rows - 2 : 0);
    const int cm = c > 0 ? c - 1 : (cols > 1 ? 1 : 0), cp = c < cols - 1 ? c + 1 : (cols > 1 ? cols - 2 : 0);
    const int a00 = ev_i1<REC>(I1, rm * cols + cm), a01 = ev_i1<REC>(I1, rm * cols + c), a02 = ev_i1<REC>(I1, rm * cols + cp);
    const int a10 = ev_i1<REC>(I1, r * cols + cm), a12 = ev_i1<REC>(I1, r * cols + cp);
    const int a20 = ev_i1<REC>(I1, rp * cols + cm), a21 = ev_i1<REC>(I1, rp * cols + c), a22 = ev_i1<REC>(I1, rp * cols + cp);
    const int gxn = 10 * (a12 - a10) + 3 * ((a22 - a20) + (a02 - a00));
    const int gyn = (3 * a20 + 10 * a21 + 3 * a22) - (3 * a00 + 10 * a01 + 3 * a02);
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

}  // namespace phovo
