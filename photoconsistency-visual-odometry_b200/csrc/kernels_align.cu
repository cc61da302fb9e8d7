// kernels_align.cu -- the per-level alignment iteration of the general path.
//
//   K3a  k_winner        : warp every source pixel, winner[target] = max(source index)
//                          == the reference's raster-order last-writer-wins residual scatter
//                          (CPhotoconsistencyOdometryAnalytic.h:358; Ceres.h:261)
//   K3b  k_normal_eq     : ONE fused pass per pixel: warp + residual (gathered through the winner
//                          map) + 1x6 Jacobian + 21 J^T J + 6 J^T r products, warp-shuffle then
//                          block reduction into per-block partials (no floating-point atomics)
//                          (AN:271-366 + the Eigen products of AN:538-539)
//   K4   k_reduce_solve  : fixed-order sum of the partials, 6x6 solve, state update, termination
//                          test, stats log, CUDA-graph WHILE condition (AN:538-549, 376-392)
//
// All kernels early-exit when pose->done is set, so an iteration enqueued after convergence is a
// no-op; the integer atomicMax of K3a is order-independent, hence run-to-run reproducible.
#include <cooperative_groups.h>

#include "phovo_device.cuh"
#include "phovo_kernels.h"
#include "phovo_lm.h"

namespace phovo {
namespace {

constexpr int kBlock = 128;

__global__ void k_fill_i32(int* p, int v, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

// state -> Pose -> PoseDev: the state and the rotation and trig values derived from it
__device__ __forceinline__ void pose_set_state(PoseDev* d, const double s[6]) {
  Pose P;
  pose_from_state(s, P);
  for (int k = 0; k < 6; ++k) d->state[k] = s[k];
  pose_store(P, d);
}

__global__ void k_set_state(PoseDev* pose, const double* state_dev, int log_capacity, double s0, double s1, double s2, double s3, double s4, double s5) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double s[6] = {s0, s1, s2, s3, s4, s5};
  if (state_dev) for (int k = 0; k < 6; ++k) s[k] = state_dev[k];
  pose_set_state(pose, s);
  pose->iteration = 0;
  pose->done = 0;
  pose->log_count = 0;
  pose->log_capacity = log_capacity;
  for (int l = 0; l < PHOVO_MAX_LEVELS; ++l) pose->iters_per_level[l] = 0;
}

__global__ void k_begin_level(PoseDev* pose, int max_iters) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  pose->iteration = 0;
  pose->done = max_iters > 0 ? 0 : 1;
}

// K3a.  4 B read (D0) + one 4 B atomicMax per valid pixel.
template <bool CERES>
__global__ void __launch_bounds__(kBlock) k_winner(LevelParams L, LevelPtrs P, const PoseDev* __restrict__ pose) {
  if (pose->done) return;
  Pose T;
  pose_load(pose, T);
  const int n = L.rows * L.cols;
  for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
    const double d = __ldg(P.D0 + i);
    const int r = i / L.cols, c = i - r * L.cols;
    Warped w;
    const bool ok = warp_pixel<CERES>(L, T, r, c, d, w);
    if (ok) atomicMax(P.winner + w.t, i);
    if (!CERES) P.valid[i] = ok;
  }
}

__device__ __forceinline__ void linear_init_axis(double x, int size, int& x1, int& x2, double& dx) {
  // third_party/sample.h:36-50
  const int ix = (int)x;
  if (ix < 0) { x1 = 0; x2 = 0; dx = 1.0; }
  else if (ix > size - 2) { x1 = size - 1; x2 = size - 1; dx = 1.0; }
  else { x1 = ix; x2 = ix + 1; dx = (double)x2 - x; }
}

__device__ __forceinline__ double bilinear(const double* __restrict__ img, int cols, int y1, int y2, int x1, int x2, double dy, double dx) {
  // third_party/sample.h:76-82
  const double a = __ldg(img + (size_t)y1 * cols + x1), b = __ldg(img + (size_t)y1 * cols + x2);
  const double c = __ldg(img + (size_t)y2 * cols + x1), d = __ldg(img + (size_t)y2 * cols + x2);
  return dy * (dx * a + (1.0 - dx) * b) + (1. - dy) * (dx * c + (1.0 - dx) * d);
}

// K3b.  MODE: 0 analytic bug-compatible, 1 analytic Maxima-exact, 2 Ceres residual.
// DUMP: additionally write the dense residual vector / Jacobian (parity hook, never on the hot path).
//
// Analytic (gather form of AN:271-366): thread i owns source pixel i AND residual slot i:
//   res[i] = winner[i] >= 0 ? I1[i] - I0[winner[i]] : 0 ; J_i from D0[i], Gx1[i], Gy1[i]
//   (gradients at the SOURCE index, AN:346-347) ; H += J_i^T J_i ; g += J_i^T res[i].
//   Reads per pixel: D0, winner, I1, I0[winner] (local gather), Gx, Gy -- each array streamed once.
// Ceres (CE:156-269): a source pixel's row survives iff it is the winner of its (truncated) target
//   slot; its residual/Jacobian use bilinear samples of I1/Gx/Gy at the real-valued warp.
// The winner slot is reset to -1 by the thread that consumed it, so the map is clean for the next
// iteration without a separate clear pass.
template <int MODE, bool DUMP>
__global__ void __launch_bounds__(kBlock) k_normal_eq(LevelParams L, LevelPtrs P, const PoseDev* __restrict__ pose,
                                                      double* __restrict__ partials,
                                                      double* __restrict__ dump_res, double* __restrict__ dump_jac) {
  __shared__ double smem[(kBlock / 32) * PHOVO_ACC_STRIDE];
  if (pose->done) return;
  Pose T;
  pose_load(pose, T);
  double acc[PHOVO_NACC];
#pragma unroll
  for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
  const int n = L.rows * L.cols;
  const int i_begin = L.row_begin * L.cols, i_end = L.row_end * L.cols;
  const double spsr = T.sp * T.sr, spcr = T.sp * T.cr;
  for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
    const int r = i / L.cols, c = i - r * L.cols;
    const double d = __ldg(P.D0 + i);
    Warped w;
    if (MODE == 2) {
      const bool ok = warp_pixel<true>(L, T, r, c, d, w);
      if (!ok) continue;
      const bool mine = i >= i_begin && i < i_end;
      if (mine) acc[28] += 1.;
      if (P.winner[w.t] != i) continue;   // overwritten by a later source pixel (CE:261)
      P.winner[w.t] = -1;
      if (!mine) continue;
      int x1, x2, y1, y2; double dx, dy;
      linear_init_axis(w.tr - 0.5, L.rows, y1, y2, dy);   // sample.h:67-71
      linear_init_axis(w.tc - 0.5, L.cols, x1, x2, dx);
      const double s0 = bilinear(P.I1, L.cols, y1, y2, x1, x2, dy, dx);
      const double s1 = bilinear(P.Gx, L.cols, y1, y2, x1, x2, dy, dx);
      const double s2 = bilinear(P.Gy, L.cols, y1, y2, x1, x2, dy, dx);
      const double res = s0 - __ldg(P.I0 + i);
      double Ju[6], Jv[6], J[6];
      projection_jacobian<false>(L, T, w, d, Ju, Jv);
#pragma unroll
      for (int k = 0; k < 6; ++k) J[k] = s1 * Ju[k] + s2 * Jv[k];   // jet_extras.h:87-109
      accumulate_row(acc, J, res);
      acc[27] = fma(res, res, acc[27]);
      if (DUMP) {
        if (dump_res) dump_res[w.t] = res;
        if (dump_jac) for (int k = 0; k < 6; ++k) dump_jac[(size_t)w.t * 6 + k] = J[k];
      }
    } else {
      const int win = P.winner[i];
      P.winner[i] = -1;
      if (i < i_begin || i >= i_end) continue;
      double res = 0.;
      if (win >= 0) {
        res = __ldg(P.I1 + i) - __ldg(P.I0 + win);
        acc[27] = fma(res, res, acc[27]);
      }
      if (DUMP && dump_res) dump_res[i] = res;
      if (!P.valid[i]) continue;                      // K3a decided (exact reference arithmetic)
      double J[6];
      analytic_jacobian<MODE>(L, T, spsr, spcr, r, c, d, __ldg(P.Gx + i), __ldg(P.Gy + i), J);
      accumulate_row(acc, J, res);
      acc[28] += 1.;
      if (DUMP && dump_jac) for (int k = 0; k < 6; ++k) dump_jac[(size_t)i * 6 + k] = J[k];
    }
  }
  const double total = block_reduce<kBlock>(acc, smem);
  if (threadIdx.x < PHOVO_NACC) partials[(size_t)blockIdx.x * PHOVO_ACC_STRIDE + threadIdx.x] = total;
}

// ---------------------------------------------------------------------------------------------
// Photometric + depth solver (CPhotoconsistencyOdometryBiObjective.h:242-452), PHOVO_MODE_BIOBJECTIVE.
//
// The reference stacks 2N rows.  Source pixel i (raster order = time i) writes, in this order:
//   jacobians row i      = intensity Jacobian          residuals slot t(i)     = I1[t] - I0[i]
//   jacobians row 2 i    = depth Jacobian              residuals slot 2 t(i)   = gain (D1[t] - D0[i])
// so depth rows of pixel i collide with intensity rows of pixel 2i and later writers win
// (BiObjective.h:422-442).  Gather form, bit-for-bit in semantics:
//   Jacobian row k = intensity row of pixel k      if k < N, k > 0 and pixel k valid   (time k beats time k/2)
//                  = depth row of pixel k/2        else if k even and pixel k/2 valid   (row 0: depth is written last)
//                  = 0                             otherwise
//   residual slot s = the write with the largest (time, kind) among intensity writes with t(i) = s
//                     and depth writes with 2 t(i) = s  ->  atomicMax of the key 2 i + kind + 1.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_winner_bi(LevelParams L, LevelPtrs P, const PoseDev* __restrict__ pose) {
  if (pose->done) return;
  Pose T;
  pose_load(pose, T);
  const int n = L.rows * L.cols;
  for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
    const double d = __ldg(P.D0 + i);
    const int r = i / L.cols, c = i - r * L.cols;
    Warped w;
    const bool ok = warp_pixel<false>(L, T, r, c, d, w);       // same validity rule as the analytic solver (:279-303)
    if (ok) {
      atomicMax(P.winner + w.t, 2 * i + 1);                     // intensity residual (:433)
      atomicMax(P.winner + 2 * w.t, 2 * i + 2);                 // depth residual (:444-445), written after it
    }
    P.valid[i] = ok;
  }
}

// Jacobian row k of the stacked 2N-row system of the photometric + depth solver (see the comment above k_winner_bi;
// bi_row_owner and bi_jacobian_core are in phovo_device.cuh), loads included (the stream / graph drivers); returns
// false for a zero row.
__device__ __forceinline__ bool bi_jacobian_row(const LevelParams& L, const LevelPtrs& P, const Pose& T, double spsr, double spcr,
                                                double gain, int n, int k, double J[6]) {
  bool depth_row;
  const int p = bi_row_owner(k, k < n && P.valid[k], P.valid[k >> 1] != 0, &depth_row);
  if (p < 0) return false;
  const double gx = depth_row ? __ldg(P.GxD + p) : __ldg(P.Gx + p), gy = depth_row ? __ldg(P.GyD + p) : __ldg(P.Gy + p);
  bi_jacobian_core(L, T, spsr, spcr, gain, p, depth_row, __ldg(P.D0 + p), gx, gy, J);
  return true;
}

template <bool DUMP>
__global__ void __launch_bounds__(kBlock) k_normal_eq_bi(LevelParams L, LevelPtrs P, const PoseDev* __restrict__ pose,
                                                         double* __restrict__ partials,
                                                         double* __restrict__ dump_res, double* __restrict__ dump_jac) {
  __shared__ double smem[(kBlock / 32) * PHOVO_ACC_STRIDE];
  if (pose->done) return;
  Pose T;
  pose_load(pose, T);
  const double gain = __ldg(P.gain);
  double acc[PHOVO_NACC];
#pragma unroll
  for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
  const int n = L.rows * L.cols;
  const double spsr = T.sp * T.sr, spcr = T.sp * T.cr;
  for (int k = blockIdx.x * kBlock + threadIdx.x; k < 2 * n; k += gridDim.x * kBlock) {
    const int wkey = P.winner[k];
    P.winner[k] = -1;
    double res = 0.;
    if (wkey > 0) {
      const int src = (wkey - 1) >> 1;
      if (((wkey - 1) & 1) == 0) res = __ldg(P.I1 + k) - __ldg(P.I0 + src);                     // slot k = t
      else res = gain * (__ldg(P.D1 + (k >> 1)) - __ldg(P.D0 + src));                           // slot k = 2 t
      acc[27] = fma(res, res, acc[27]);
    }
    if (DUMP && dump_res) dump_res[k] = res;
    if (k < n && P.valid[k]) acc[28] += 1.;
    double J[6];
    if (!bi_jacobian_row(L, P, T, spsr, spcr, gain, n, k, J)) continue;
    accumulate_row(acc, J, res);
    if (DUMP && dump_jac) for (int a = 0; a < 6; ++a) dump_jac[(size_t)k * 6 + a] = J[a];
  }
  const double total = block_reduce<kBlock>(acc, smem);
  if (threadIdx.x < PHOVO_NACC) partials[(size_t)blockIdx.x * PHOVO_ACC_STRIDE + threadIdx.x] = total;
}

// Sum partials[0..grid) for each of the PHOVO_NACC values in a fixed order: warp v owns value v,
// lane l adds blocks l, l+32, ... in order, then a fixed butterfly over lanes.  Needs 32 warps.
__device__ __forceinline__ void reduce_partials(const double* __restrict__ partials, int grid, double* totals /* smem[32] */) {
  const int v = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (v < PHOVO_NACC) {
    double s = 0.;
    for (int b = lane; b < grid; b += 32) s += partials[(size_t)b * PHOVO_ACC_STRIDE + v];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) totals[v] = s;
  }
  __syncthreads();
}

// |g|, the quantity the termination test thresholds (AN:380)
__device__ __forceinline__ double grad_norm(const double g[6]) {
  double n2 = 0.;
  for (int k = 0; k < 6; ++k) n2 = fma(g[k], g[k], n2);
  return sqrt(n2);
}

// The fields of a stats entry that an evaluation's totals decide; iteration, accepted and the states are the caller's.
__device__ __forceinline__ void entry_from_totals(phovo_iter_stats* e, int level, const double* totals) {
  e->level = level; e->num_valid = (int)totals[28];
  for (int k = 0; k < 21; ++k) e->H[k] = totals[k];
  for (int k = 0; k < 6; ++k) e->g[k] = totals[21 + k];
  e->grad_norm = grad_norm(totals + 21); e->cost = 0.5 * totals[27]; e->radius = 0.;
}

// The Gauss-Newton step and termination test of AN:538-549 / AN:376-392 for iteration `it` (0-based) of the level,
// single thread: s_out from the totals at s_in.  Returns done.
__device__ __forceinline__ int gn_update(const LevelParams& L, const double* totals, const double s_in[6], int it, double s_out[6]) {
  double g[6], step[6], n2 = 0.;   // (n2 summed here, not by grad_norm after the solve: fewer spills in k_reduce_solve)
  for (int k = 0; k < 6; ++k) { g[k] = totals[21 + k]; n2 = fma(g[k], g[k], n2); }
  solve6_ldlt(totals, g, step);
  for (int k = 0; k < 6; ++k) s_out[k] = s_in[k] - L.lambda * step[k];   // AN:539-540
  return (it + 1 >= L.max_iters) || (sqrt(n2) < L.min_grad_norm);        // AN:383-392, 547
}

// The log entry of that iteration.  (The callers test whether to log after the step: testing before keeps the log
// position live through the solve, which spills in k_reduce_solve.)
__device__ __forceinline__ void gn_entry(phovo_iter_stats* e, const LevelParams& L, const double* totals, int it, const double s_in[6],
                                         const double s_out[6]) {
  entry_from_totals(e, L.level, totals);
  e->iteration = it; e->accepted = 1;
  for (int k = 0; k < 6; ++k) { e->state_in[k] = s_in[k]; e->state_out[k] = s_out[k]; }
}

// One Gauss-Newton iteration of the stream / graph drivers on the PoseDev in global memory.
__device__ void gn_step(const LevelParams& L, PoseDev* pose, const double* totals, phovo_iter_stats* log,
                        unsigned long long cond_handle) {
  double s_in[6], s_out[6];
  for (int k = 0; k < 6; ++k) s_in[k] = pose->state[k];
  const int it = pose->iteration;
  const int done = gn_update(L, totals, s_in, it, s_out);
  if (log && pose->log_count < pose->log_capacity) gn_entry(log + pose->log_count, L, totals, it, s_in, s_out);
  pose->log_count += 1;
  pose_set_state(pose, s_out);
  pose->iteration = it + 1;
  pose->iters_per_level[L.level] = it + 1;
  pose->done = done;
  if (cond_handle) cudaGraphSetConditional((cudaGraphConditionalHandle)cond_handle, done ? 0u : 1u);
}

__global__ void __launch_bounds__(1024) k_reduce_solve(LevelParams L, PoseDev* pose, const double* __restrict__ partials, int grid,
                                                       phovo_iter_stats* log, unsigned long long cond_handle) {
  __shared__ double totals[32];
  if (pose->done) {
    if (cond_handle && threadIdx.x == 0) cudaGraphSetConditional((cudaGraphConditionalHandle)cond_handle, 0u);
    return;
  }
  reduce_partials(partials, grid, totals);
  if (threadIdx.x == 0) gn_step(L, pose, totals, log, cond_handle);
}

__global__ void __launch_bounds__(1024) k_reduce_only(LevelParams L, const PoseDev* pose, const double* __restrict__ partials, int grid,
                                                      phovo_iter_stats* out) {
  __shared__ double totals[32];
  reduce_partials(partials, grid, totals);
  if (threadIdx.x == 0) {
    entry_from_totals(out, L.level, totals);
    out->iteration = 0; out->accepted = 0;
    for (int k = 0; k < 6; ++k) { out->state_in[k] = pose->state[k]; out->state_out[k] = pose->state[k]; }
  }
}

__global__ void __launch_bounds__(1024) k_reduce_to_buffer(const PoseDev* pose, const double* __restrict__ partials, int grid, double* buffer) {
  __shared__ double totals[32];
  reduce_partials(partials, grid, totals);
  if (threadIdx.x < 32) buffer[threadIdx.x] = threadIdx.x < PHOVO_NACC ? totals[threadIdx.x] : 0.;
}

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Fused local reduction + one-shot all-reduce over NVLink peer memory (row-sharded single pair).
// 1024 threads: warps 0..28 reduce the per-block partials (one value each, fixed order); then
// thread (w, v) = (tid / 32, tid % 32), w < world, stores value v into peer w's slot
// [parity][rank][v]; thread w*32 releases peer w's flag[rank] = epoch after a system-scope fence;
// thread w < world acquires the local flag[w] >= epoch (bounded spin); finally thread v < 32 sums the
// slots in rank order.  Two slot parities: a peer can be at most one exchange ahead.
__global__ void __launch_bounds__(1024) k_reduce_exchange(const PoseDev* pose, const double* __restrict__ partials, int grid,
                                                          double* __restrict__ buffer, ShardExchange* const* __restrict__ peers,
                                                          int rank, int world, unsigned long long epoch) {
  __shared__ double totals[32];
  reduce_partials(partials, grid, totals);
  const int w = threadIdx.x >> 5, v = threadIdx.x & 31;
  const int parity = (int)(epoch & 1ull);
  if (w < world) {
    ShardExchange* peer = peers[w];
    peer->slots[parity][rank][v] = v < PHOVO_NACC ? totals[v] : 0.;
    __threadfence_system();
    __syncwarp();
    if (v == 0) st_release_sys(&peer->flags[rank], epoch);
  }
  ShardExchange* mine = peers[rank];
  if (threadIdx.x < world) {
    long long spins = 0;
    while (ld_acquire_sys(&mine->flags[threadIdx.x]) < epoch) {
      if (++spins > (1ll << 22)) { mine->error = 1; break; }   // seconds: a peer never arrived
      __nanosleep(20);
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    double s = 0.;
    for (int r = 0; r < world; ++r) s += mine->slots[parity][r][threadIdx.x];
    buffer[threadIdx.x] = s;
  }
}

__global__ void k_solve_from_buffer(LevelParams L, PoseDev* pose, const double* buffer, phovo_iter_stats* log) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (pose->done) return;
  double totals[32];
  for (int k = 0; k < 32; ++k) totals[k] = buffer[k];
  gn_step(L, pose, totals, log, 0ull);
}

// ---------------------------------------------------------------------------------------------
// Persistent cooperative variant: ONE launch runs the whole Gauss-Newton loop of a level
// (AN:504-561).  Per iteration: phase A (K3a) -> grid.sync -> phase B (K3b, per-block partials) ->
// grid.sync -> every CTA sums ALL partials in the same fixed order and takes the same step
// redundantly (no third barrier, no broadcast); CTA 0 publishes pose and log.  Data written by
// other SMs inside the launch (winner, valid, partials) is read with ld.global.cg.
// ---------------------------------------------------------------------------------------------
constexpr int kCoopBlock = 256;

// Phase A of the analytic loops: whether source pixel i with depth d lands, and on which target slot t.
// Estimate-then-verify (phovo_device.cuh): the exact reference arithmetic runs only for the pixels whose
// estimate lies next to a rounding boundary (~2e-4 of them); the graph / stream drivers (k_winner) run it
// for every pixel.
__device__ __forceinline__ bool phase_a_target(const LevelParams& L, const Pose& T, const EstimateConst& E, int i, double d, int& t) {
  const int r = i / L.cols, c = i - r * L.cols;
  const bool dep = (L.min_depth < d) & (d < L.max_depth);                  // strict bounds, AN:279-280
  int tj, ti;
  const bool unc = estimate_target(L, T, E, r, c, d, tj, ti);
  bool ok = dep & ((unsigned)tj < (unsigned)L.cols) & ((unsigned)ti < (unsigned)L.rows);
  t = L.cols * ti + tj;
  if (dep & unc) {
    Warped w;
    ok = warp_pixel<false>(L, T, r, c, d, w);
    t = w.t;
  }
  return ok;
}

// Every CTA of a persistent loop: the fixed-order sum of all `nblk` CTAs' partials into s_tot (warp g of 8
// takes blocks g, g+8, ..., then the eight warp sums in order).
__device__ __forceinline__ void sum_all_partials(const double* partials, int nblk, double* smem, double* s_tot) {
  const int tid = threadIdx.x, v = tid & 31, g = tid >> 5;
  double s = 0.;
  for (int b = g; b < nblk; b += kCoopBlock / 32) s += __ldcg(partials + (size_t)b * PHOVO_ACC_STRIDE + v);
  smem[g * PHOVO_ACC_STRIDE + v] = s;
  __syncthreads();
  if (tid < 32) {
    double t = 0.;
#pragma unroll
    for (int k = 0; k < kCoopBlock / 32; ++k) t += smem[k * PHOVO_ACC_STRIDE + tid];
    s_tot[tid] = t;
  }
  __syncthreads();
}

// End of a level in a persistent loop (one thread of the pair's first CTA): the pose goes out with the level's
// iteration count and log position.
__device__ __forceinline__ void finish_level(PoseDev* pose, PoseDev& s_pose, int level, int iterations, int log_count) {
  s_pose.iteration = iterations;
  s_pose.iters_per_level[level] = iterations;
  s_pose.done = 1;
  s_pose.log_count = log_count;
  *pose = s_pose;
}

// Row-sharded use (one 8K pair over several GPUs, SURVEY 8(e)): `S.world` > 1.  Every rank runs phase A over the
// whole level (the winner map needs every source pixel), phase B over ITS band of source rows [L.row_begin,
// L.row_end), sums its partials as before -- and then the ranks exchange the 29 sums INSIDE the kernel: CTA 0
// stores them into every peer's exchange area over NVLink and releases a flag, every CTA of every rank waits for
// the `world` flags in its own area and adds the slots in rank order.  All CTAs of all ranks end up with bitwise
// the same totals and take the same step: no broadcast, no third grid barrier, no host in the loop.  The exchange
// areas are double-buffered by epoch parity; a rank can run at most one exchange ahead of the slowest one.
//
// Phase A is sharded too: a source pixel at row r lands at most h rows away, h = ceil(fy (dmin B1 + e1max) / Zlow) + 2
// from the current pose (B1 bounds the coefficient of d in Y' - ryi Z', e1max the offset, Zlow = dmin m2min - |z| <= Z'
// for every valid pixel; (d B1 + e1max) / (d m2min - |z|) decreases in d, so the smallest valid depth of the level
// -- measured once per frame, `dmin` -- gives the maximum).  A rank therefore warps the source rows of its band
// +- h only: every pixel that can bid for a slot of the band is among them; the slots outside the band that those
// pixels may have bid for (+- 2 h) are cleaned after phase B.  No bound (Zlow <= 0, state not finite) => the whole level.
struct ShardArgs {
  ShardExchange* const* peers;     // device array [world] of exchange areas (own one included), or nullptr
  int rank, world;
  unsigned long long epoch_base;   // epoch of iteration `it` of this launch is epoch_base + it + 1
  const double* dmin;              // smallest depth of the level inside (min_depth, max_depth); nullptr: no halo bound
};

__device__ __forceinline__ int shard_halo_rows(const LevelParams& L, const Pose& T, double dmin) {
  const double rx = fmax(fabs(L.ox), fabs((double)(L.cols - 1) - L.ox)) * fabs(L.inv_fx);
  const double ry = fmax(fabs(L.oy), fabs((double)(L.rows - 1) - L.oy)) * fabs(L.inv_fy);
  const double B1 = (fabs(T.R10) * rx + fabs(T.R12)) + (fabs(T.R11 - T.R22) + fabs(T.R20) * rx) * ry + fabs(T.R21) * ry * ry;
  const double e1m = fabs(T.y) + ry * fabs(T.z);
  const double zlow = dmin * (T.R22 - fabs(T.R20) * rx - fabs(T.R21) * ry) - fabs(T.z);
  const double dy = fabs(L.fy) * (dmin * B1 + e1m) / zlow * (1.0 + 0x1p-20) + 0x1p-10;
  if (!(zlow > 0.) || !(dy < (double)L.rows)) return L.rows;      // NaN compares false: no bound
  return (int)ceil(dy) + 2;
}

// SLOT 1: the same loop run by ONE CTA on its own pair (the batch slot kernels below): the grid barriers become block
// barriers, the CTA is "block 0 of a grid of 1".  SLOT 2: by one thread-block CLUSTER per pair (small waves: more CTAs per
// pair than pairs per SM), cluster barriers.  SLOT 0: the cooperative grid.
template <int SLOT>
__device__ __forceinline__ void level_barrier() {
  if (SLOT == 1) __syncthreads();
  else if (SLOT == 2) cooperative_groups::this_cluster().sync();   // release / acquire at cluster scope: orders the global writes too
  else cooperative_groups::this_grid().sync();
}
// the CTA's index among the CTAs that share the pair, and their number
template <int SLOT> __device__ __forceinline__ int level_block_rank() {
  return SLOT == 1 ? 0 : SLOT == 2 ? (int)cooperative_groups::this_cluster().block_rank() : (int)blockIdx.x;
}
template <int SLOT> __device__ __forceinline__ int level_num_blocks() {
  return SLOT == 1 ? 1 : SLOT == 2 ? (int)cooperative_groups::this_cluster().num_blocks() : (int)gridDim.x;
}

template <int MODE, bool SHARD, int SLOT>
__device__ __forceinline__ void level_loop(const LevelParams& L, const LevelPtrs& P, PoseDev* pose, double* partials,
                                           phovo_iter_stats* log, const ShardArgs& S) {
  const int bid = level_block_rank<SLOT>(), nblk = level_num_blocks<SLOT>();
  __shared__ double smem[(kCoopBlock / 32) * PHOVO_ACC_STRIDE];
  __shared__ double s_tot[32];
  __shared__ PoseDev s_pose;
  __shared__ int s_done;
  const int tid = threadIdx.x;
  if (tid == 0) { s_pose = *pose; s_done = 0; }
  __syncthreads();
  int log_count = s_pose.log_count;
  const int log_capacity = s_pose.log_capacity;
  const int n = L.rows * L.cols;
  const int stride = nblk * kCoopBlock;
  int it = 0;
  for (; it < L.max_iters; ++it) {
    Pose T;
    pose_load(&s_pose, T);
    // ---- phase A: winner map + validity ----
    const EstimateConst E = estimate_const(L, T);
    // row-sharded: the source rows that can reach this rank's band (see ShardArgs); otherwise the whole level
    int halo = 0, a_begin = 0, a_end = n;
    if (SHARD && (L.row_begin > 0 || L.row_end < L.rows)) {
      halo = S.dmin ? shard_halo_rows(L, T, __ldg(S.dmin)) : L.rows;
      a_begin = max(0, L.row_begin - halo) * L.cols;
      a_end = min(L.rows, L.row_end + halo) * L.cols;
    }
    for (int i = a_begin + bid * kCoopBlock + tid; i < a_end; i += stride) {
      int t;
      const bool ok = phase_a_target(L, T, E, i, __ldg(P.D0 + i), t);
      if (MODE == 3) {   // photometric + depth solver: two residual slots per pixel, keys 2i+1 / 2i+2 (see k_winner_bi)
        if (ok) { atomicMax(P.winner + t, 2 * i + 1); atomicMax(P.winner + 2 * t, 2 * i + 2); }
      } else if (ok) atomicMax(P.winner + t, i);
      P.valid[i] = ok;
    }
    level_barrier<SLOT>();
    // ---- phase B: residual + Jacobian + normal equations ----
    double acc[PHOVO_NACC];
#pragma unroll
    for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
    const double spsr = T.sp * T.sr, spcr = T.sp * T.cr;
    if (MODE == 3) {
      const double gain = __ldg(P.gain);
      // Every array a row may read is loaded BEFORE anything depends on a loaded value, and ONE TRIP AHEAD: one memory
      // round trip per row (I0 / D0 of the winner) overlapped with the next row's loads, instead of six in a chain
      // (winner -> I0[src]; valid[k] -> valid[k/2] -> D0[p] -> gradient) -- at the price of loads whose values are not
      // used: the loop is latency-bound, not bandwidth-bound.
      struct RowLoads { int wkey; bool vk, vh; double i1, d1, d0k, d0h, gxk, gyk, gxh, gyh; };
      auto load_row = [&](int k, RowLoads& R) {
        const int kh = k >> 1;
        const bool lo = k < n;
        R.wkey = __ldcg(P.winner + k);
        R.vk = lo && __ldcg(P.valid + k) != 0;
        R.vh = __ldcg(P.valid + kh) != 0;
        R.i1 = lo ? __ldg(P.I1 + k) : 0.; R.d1 = __ldg(P.D1 + kh);
        R.d0k = lo ? __ldg(P.D0 + k) : 0.; R.d0h = __ldg(P.D0 + kh);
        R.gxk = lo ? __ldg(P.Gx + k) : 0.; R.gyk = lo ? __ldg(P.Gy + k) : 0.;
        R.gxh = __ldg(P.GxD + kh); R.gyh = __ldg(P.GyD + kh);
      };
      const int k_first = bid * kCoopBlock + tid;
      RowLoads N = {};
      if (k_first < 2 * n) load_row(k_first, N);
      for (int k = k_first; k < 2 * n; k += stride) {
        const RowLoads R = N;
        if (k + stride < 2 * n) load_row(k + stride, N);
        P.winner[k] = -1;
        double res = 0.;
        if (R.wkey > 0) {
          const int src = (R.wkey - 1) >> 1;
          if (((R.wkey - 1) & 1) == 0) res = R.i1 - __ldg(P.I0 + src);                 // slot k = t
          else res = gain * (R.d1 - __ldg(P.D0 + src));                               // slot k = 2 t
          acc[27] = fma(res, res, acc[27]);
        }
        if (R.vk) acc[28] += 1.;
        bool depth_row;
        const int p = bi_row_owner(k, R.vk, R.vh, &depth_row);
        if (p < 0) continue;
        double J[6];
        bi_jacobian_core(L, T, spsr, spcr, gain, p, depth_row, depth_row ? R.d0h : R.d0k, depth_row ? R.gxh : R.gxk, depth_row ? R.gyh : R.gyk, J);
        accumulate_row(acc, J, res);
      }
    } else {
      const int i_begin = L.row_begin * L.cols, i_end = L.row_end * L.cols;   // the whole level unless row-sharded
      if (SHARD) {
        // (a band is a few trips per thread: loading one trip ahead costs more than it hides there -- measured on 4 GPUs,
        // 0.55 vs 0.63 ms for the 8K pair)
        for (int i = i_begin + bid * kCoopBlock + tid; i < i_end; i += stride) {
          const int win = __ldcg(P.winner + i);
          const bool ok = __ldcg(P.valid + i) != 0;
          const double i1 = __ldg(P.I1 + i), d = __ldg(P.D0 + i), gx = __ldg(P.Gx + i), gy = __ldg(P.Gy + i);
          P.winner[i] = -1;
          double res = 0.;
          if (win >= 0) {
            res = i1 - __ldg(P.I0 + win);
            acc[27] = fma(res, res, acc[27]);
          }
          if (!ok) continue;
          const int r = i / L.cols, c = i - r * L.cols;
          double J[6];
          analytic_jacobian<MODE>(L, T, spsr, spcr, r, c, d, gx, gy, J);
          accumulate_row(acc, J, res);
          acc[28] += 1.;
        }
      } else {
        // Everything indexed by i is loaded up front (coalesced, independent) and ONE TRIP AHEAD: while this trip waits for
        // I0[winner] and computes, the next trip's six loads are in flight.  (The winner word of the next trip is final:
        // phase A ended at the barrier, and only this thread resets it.)
        const int b_first = i_begin + bid * kCoopBlock + tid;
        int win_n = -1; bool ok_n = false; double i1_n = 0., d_n = 0., gx_n = 0., gy_n = 0.;
        if (b_first < i_end) {
          win_n = __ldcg(P.winner + b_first); ok_n = __ldcg(P.valid + b_first) != 0;
          i1_n = __ldg(P.I1 + b_first); d_n = __ldg(P.D0 + b_first); gx_n = __ldg(P.Gx + b_first); gy_n = __ldg(P.Gy + b_first);
        }
        for (int i = b_first; i < i_end; i += stride) {
          const int win = win_n; const bool ok = ok_n;
          const double i1 = i1_n, d = d_n, gx = gx_n, gy = gy_n;
          const int j = i + stride;
          if (j < i_end) {
            win_n = __ldcg(P.winner + j); ok_n = __ldcg(P.valid + j) != 0;
            i1_n = __ldg(P.I1 + j); d_n = __ldg(P.D0 + j); gx_n = __ldg(P.Gx + j); gy_n = __ldg(P.Gy + j);
          }
          P.winner[i] = -1;
          double res = 0.;
          if (win >= 0) {
            res = i1 - __ldg(P.I0 + win);
            acc[27] = fma(res, res, acc[27]);
          }
          if (!ok) continue;
          const int r = i / L.cols, c = i - r * L.cols;
          double J[6];
          analytic_jacobian<MODE>(L, T, spsr, spcr, r, c, d, gx, gy, J);
          accumulate_row(acc, J, res);
          acc[28] += 1.;
        }
      }
      // row-sharded: slots outside the band that the warped rows may have bid for must be clean for the next iteration
      if (SHARD && (i_begin > 0 || i_end < n)) {
        const int c_begin = max(0, L.row_begin - 2 * halo) * L.cols, c_end = min(L.rows, L.row_end + 2 * halo) * L.cols;
        for (int i = c_begin + bid * kCoopBlock + tid; i < i_begin; i += stride) P.winner[i] = -1;
        for (int i = i_end + bid * kCoopBlock + tid; i < c_end; i += stride) P.winner[i] = -1;
      }
    }
    {
      const double total = block_reduce<kCoopBlock>(acc, smem);
      if (tid < PHOVO_NACC) partials[(size_t)bid * PHOVO_ACC_STRIDE + tid] = total;
    }
    level_barrier<SLOT>();
    sum_all_partials(partials, nblk, smem, s_tot);
    // ---- row-sharded: all-reduce of the 29 sums over NVLink peer memory, in rank order ----
    if (SHARD && S.world > 1) {
      const unsigned long long epoch = S.epoch_base + (unsigned long long)it + 1ull;
      const int parity = (int)(epoch & 1ull);
      ShardExchange* mine = S.peers[S.rank];
      if (bid == 0) {
        const int w = tid >> 5, v = tid & 31;
        if (w < S.world) {
          ShardExchange* peer = S.peers[w];
          peer->slots[parity][S.rank][v] = v < PHOVO_NACC ? s_tot[v] : 0.;
          __threadfence_system();
          __syncwarp();
          if (v == 0) st_release_sys(&peer->flags[S.rank], epoch);
        }
      }
      if (tid < S.world) {
        long long spins = 0;
        while (ld_acquire_sys(&mine->flags[tid]) < epoch) {
          if (++spins > (1ll << 24)) { mine->error = 1; break; }   // seconds: a peer never arrived
          __nanosleep(20);
        }
      }
      __syncthreads();
      if (tid < 32) {
        double t = 0.;
        for (int r = 0; r < S.world; ++r) t += __ldcg(&mine->slots[parity][r][tid]);
        s_tot[tid] = t;
      }
      __syncthreads();
    }
    // ---- Gauss-Newton step + termination test, one thread per CTA ----
    if (tid == 0) {
      double s_in[6], s_out[6];
      for (int k = 0; k < 6; ++k) s_in[k] = s_pose.state[k];
      const int done = gn_update(L, s_tot, s_in, it, s_out);
      if (bid == 0 && log && log_count < log_capacity) gn_entry(log + log_count, L, s_tot, it, s_in, s_out);
      pose_set_state(&s_pose, s_out);
      s_done = done;
    }
    log_count += 1;
    __syncthreads();
    if (s_done) { ++it; break; }
  }
  if (bid == 0 && tid == 0) finish_level(pose, s_pose, L.level, it, log_count);
}

template <int MODE, bool SHARD>
__global__ void __launch_bounds__(kCoopBlock, 2) k_level_coop(LevelParams L, LevelPtrs P, PoseDev* pose, double* partials,
                                                               phovo_iter_stats* log, ShardArgs S) {
  level_loop<MODE, SHARD, 0>(L, P, pose, partials, log, S);
}

// ---------------------------------------------------------------------------------------------
// Thread-block-cluster variant for SMALL levels (analytic modes): ONE cluster of kClusterSize CTAs runs
// the whole Gauss-Newton loop of a level.  The winner map lives in DISTRIBUTED shared memory: CTA k
// owns the target slots (and the source pixels) [k chunk, (k+1) chunk); phase A bids with a remote
// shared-memory atomicMax into the owner's slice, phase B reads only the CTA's own slice.  The two
// grid-wide barriers of the cooperative kernel (~2.5 us each, which is what a 4 800-px level costs)
// become two cluster barriers (~0.2 us).  Every CTA deposits its 29 partial sums in every CTA's
// shared memory, sums the kClusterSize partials in rank order and takes the same step redundantly.
// Bitwise reproducible; equal to the cooperative kernel up to the grouping of the partial sums.
// ---------------------------------------------------------------------------------------------
constexpr int kClusterBlock = 512;
constexpr int kClusterSize = 16;          // non-portable cluster size (8 is the portable maximum)
constexpr int kClusterMaxPixels = 8192;   // levels up to this size take the cluster kernel (measured: 4 800 px 24.7 vs 30.2 us, 19 200 px 41.9 vs 38.9 us)

template <int MODE>
__global__ void __launch_bounds__(kClusterBlock, 1) k_level_cluster(LevelParams L, LevelPtrs P, PoseDev* pose, phovo_iter_stats* log) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), nblk = (int)cluster.num_blocks();
  extern __shared__ __align__(16) unsigned char cl_smem[];
  const int n = L.rows * L.cols;
  const int chunk = (n + nblk - 1) / nblk;
  double* sPart = (double*)cl_smem;                                   // [nblk][PHOVO_ACC_STRIDE]: partials of every CTA
  double* sRed = sPart + kClusterSize * PHOVO_ACC_STRIDE;             // block_reduce scratch
  int* sWin = (int*)(sRed + (kClusterBlock / 32) * PHOVO_ACC_STRIDE); // [chunk] winner source index per owned target slot
  unsigned char* sValid = (unsigned char*)(sWin + chunk);             // [chunk] validity of the owned source pixels
  __shared__ double s_tot[32];
  __shared__ PoseDev s_pose;
  __shared__ int s_done;
  const int tid = threadIdx.x;
  if (tid == 0) { s_pose = *pose; s_done = 0; }
  for (int k = tid; k < chunk; k += kClusterBlock) sWin[k] = -1;
  __syncthreads();
  cluster.sync();                       // every slice is initialised before anybody bids into it
  int log_count = s_pose.log_count;
  const int log_capacity = s_pose.log_capacity;
  const int begin = rank * chunk, end = min(n, begin + chunk);
  int it = 0;
  for (; it < L.max_iters; ++it) {
    Pose T;
    pose_load(&s_pose, T);
    // ---- phase A: bids of the owned source pixels into the owners of their target slots ----
    const EstimateConst E = estimate_const(L, T);
    for (int i = begin + tid; i < end; i += kClusterBlock) {
      int t;
      const bool ok = phase_a_target(L, T, E, i, __ldg(P.D0 + i), t);
      if (ok) {
        const int owner = t / chunk;
        atomicMax(cluster.map_shared_rank(sWin, owner) + (t - owner * chunk), i);   // raster-order last writer wins (AN:358)
      }
      sValid[i - begin] = ok;
    }
    cluster.sync();
    // ---- phase B: residual + Jacobian + normal equations of the owned pixels ----
    double acc[PHOVO_NACC];
#pragma unroll
    for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
    const double spsr = T.sp * T.sr, spcr = T.sp * T.cr;
    for (int i = begin + tid; i < end; i += kClusterBlock) {
      const int win = sWin[i - begin];
      sWin[i - begin] = -1;
      double res = 0.;
      if (win >= 0) {
        res = __ldg(P.I1 + i) - __ldg(P.I0 + win);
        acc[27] = fma(res, res, acc[27]);
      }
      if (!sValid[i - begin]) continue;
      const int r = i / L.cols, c = i - r * L.cols;
      double J[6];
      analytic_jacobian<MODE>(L, T, spsr, spcr, r, c, __ldg(P.D0 + i), __ldg(P.Gx + i), __ldg(P.Gy + i), J);
      accumulate_row(acc, J, res);
      acc[28] += 1.;
    }
    {
      const double total = block_reduce<kClusterBlock>(acc, sRed);
      if (tid < PHOVO_NACC)
        for (int b = 0; b < nblk; ++b) cluster.map_shared_rank(sPart, b)[rank * PHOVO_ACC_STRIDE + tid] = total;
    }
    cluster.sync();
    // ---- every CTA: partials summed in rank order, same step taken redundantly ----
    if (tid < 32) {
      double t = 0.;
      if (tid < PHOVO_NACC)
        for (int b = 0; b < nblk; ++b) t += sPart[b * PHOVO_ACC_STRIDE + tid];
      s_tot[tid] = t;
    }
    __syncthreads();
    if (tid == 0) {
      double s_in[6], s_out[6];
      for (int k = 0; k < 6; ++k) s_in[k] = s_pose.state[k];
      const int done = gn_update(L, s_tot, s_in, it, s_out);
      if (rank == 0 && log && log_count < log_capacity) gn_entry(log + log_count, L, s_tot, it, s_in, s_out);
      pose_set_state(&s_pose, s_out);
      s_done = done;
    }
    log_count += 1;
    __syncthreads();
    if (s_done) { ++it; break; }
  }
  if (rank == 0 && tid == 0) finish_level(pose, s_pose, L.level, it, log_count);
  cluster.sync();                       // nobody leaves while its shared memory may still be written remotely
}

// ---------------------------------------------------------------------------------------------
// Ceres mode on the device: the restated trust-region Levenberg-Marquardt loop of one level
// (CE:433-500 -> ceres::Solve, SURVEY appendix A) inside ONE persistent cooperative launch.  Every loop
// trip is one evaluation of the CE:156-269 residual + Jacobian at S.xn (phase A winner map by
// truncation, grid.sync, phase B bilinear samples + normal equations, grid.sync, fixed-order sum of
// all partials in every CTA) followed by the LM decision of phovo_lm.h -- the same functions the host
// loop in phovo_api.cu (optimize_ceres) calls.  Thread 0 of every CTA takes the decision redundantly:
// identical inputs, identical arithmetic, so all CTAs stay in lock step without a broadcast.  CTA 0
// writes the log.
// ---------------------------------------------------------------------------------------------
template <int SLOT>
__device__ __forceinline__ void level_loop_ceres(const LevelParams& L, const LevelPtrs& P, PoseDev* pose, double* partials,
                                                 phovo_iter_stats* log, const LmParams& lm) {
  const int bid = level_block_rank<SLOT>(), nblk = level_num_blocks<SLOT>();
  __shared__ double smem[(kCoopBlock / 32) * PHOVO_ACC_STRIDE];
  __shared__ double s_tot[32];
  __shared__ PoseDev s_pose;
  __shared__ LmState S;
  __shared__ int s_first, s_done;
  const int tid = threadIdx.x;
  if (tid == 0) {
    s_pose = *pose;
    for (int k = 0; k < 6; ++k) { S.x[k] = s_pose.state[k]; S.xn[k] = s_pose.state[k]; }
    S.radius = lm.initial_radius; S.decrease_factor = 2.0; S.iteration = 0; s_first = 1; s_done = 0;
  }
  __syncthreads();
  int log_count = s_pose.log_count;
  const int log_capacity = s_pose.log_capacity;
  const int n = L.rows * L.cols;
  const int stride = nblk * kCoopBlock;
  for (;;) {
    // ---- pose of the state to evaluate (every CTA, thread 0) ----
    if (tid == 0) pose_set_state(&s_pose, S.xn);
    __syncthreads();
    Pose T;
    pose_load(&s_pose, T);
    // ---- phase A: winner of each (truncated) target slot, CE:250-254, 261 ----
    for (int i = bid * kCoopBlock + tid; i < n; i += stride) {
      const double d = __ldg(P.D0 + i);
      const int r = i / L.cols, c = i - r * L.cols;
      Warped w;
      if (warp_pixel<true>(L, T, r, c, d, w)) atomicMax(P.winner + w.t, i);
    }
    level_barrier<SLOT>();
    // ---- phase B: CE:156-269 residual + Jacobian rows of the surviving pixels ----
    double acc[PHOVO_NACC];
#pragma unroll
    for (int v = 0; v < PHOVO_NACC; ++v) acc[v] = 0.;
    for (int i = bid * kCoopBlock + tid; i < n; i += stride) {
      const int r = i / L.cols, c = i - r * L.cols;
      const double d = __ldg(P.D0 + i);
      Warped w;
      if (!warp_pixel<true>(L, T, r, c, d, w)) continue;
      acc[28] += 1.;
      // the twelve taps and I0 do not depend on who won the slot: they are issued together with the winner word (one
      // memory round trip instead of two; a loser's taps are wasted, losers are few)
      const int win = __ldcg(P.winner + w.t);
      int x1, x2, y1, y2; double dx, dy;
      linear_init_axis(w.tr - 0.5, L.rows, y1, y2, dy);   // sample.h:67-71
      linear_init_axis(w.tc - 0.5, L.cols, x1, x2, dx);
      const double s0 = bilinear(P.I1, L.cols, y1, y2, x1, x2, dy, dx);
      const double s1 = bilinear(P.Gx, L.cols, y1, y2, x1, x2, dy, dx);
      const double s2 = bilinear(P.Gy, L.cols, y1, y2, x1, x2, dy, dx);
      const double i0 = __ldg(P.I0 + i);
      if (win != i) continue;                        // overwritten by a later source pixel (CE:261)
      P.winner[w.t] = -1;                            // the winner cleans its slot (a loser that reads -1 has lost all the same)
      const double res = s0 - i0;
      double Ju[6], Jv[6], J[6];
      projection_jacobian<false>(L, T, w, d, Ju, Jv);
#pragma unroll
      for (int k = 0; k < 6; ++k) J[k] = s1 * Ju[k] + s2 * Jv[k];   // jet_extras.h:87-109
      accumulate_row(acc, J, res);
      acc[27] = fma(res, res, acc[27]);
    }
    {
      const double total = block_reduce<kCoopBlock>(acc, smem);
      if (tid < PHOVO_NACC) partials[(size_t)bid * PHOVO_ACC_STRIDE + tid] = total;
    }
    level_barrier<SLOT>();   // partials complete, every winner slot back to -1
    sum_all_partials(partials, nblk, smem, s_tot);
    // ---- LM decision (phovo_lm.h) ----
    if (tid == 0) {
      LmLog sink{log, log_count, log_capacity, bid == 0 && log != nullptr};
      bool go;
      if (s_first) {
        s_first = 0;
        entry_from_totals(&S.cur, L.level, s_tot);
        go = lm_start(lm, S) && lm_propose(lm, S, sink);
      } else {
        const int v = lm_judge(lm, S, 0.5 * s_tot[27], sink);
        if (v == LM_ACCEPT) entry_from_totals(&S.cur, L.level, s_tot);
        go = v != LM_STOP && lm_update_radius(lm, S, v == LM_ACCEPT) && lm_propose(lm, S, sink);
      }
      s_done = go ? 0 : 1;
      s_pose.log_count = log_count;
    }
    __syncthreads();
    log_count = s_pose.log_count;
    if (s_done) break;
  }
  if (bid == 0 && tid == 0) {
    pose_set_state(&s_pose, S.x);
    finish_level(pose, s_pose, L.level, S.iteration, log_count);
  }
}

#ifndef PHOVO_CERES_COOP_MINB
#define PHOVO_CERES_COOP_MINB 1   // 255 registers, no spills, one CTA per SM: 0.45 vs 0.49 ms for the 640x480 Ceres configuration (the loop is barrier-bound)
#endif
__global__ void __launch_bounds__(kCoopBlock, PHOVO_CERES_COOP_MINB) k_level_coop_ceres(LevelParams L, LevelPtrs P, PoseDev* pose, double* partials,
                                                                     phovo_iter_stats* log, LmParams lm) {
  level_loop_ceres<0>(L, P, pose, partials, log, lm);
}

// ---------------------------------------------------------------------------------------------
// Batch slot kernels (phovo_batch.cu, wave path): ONE CTA runs the whole coarse-to-fine alignment of ONE pair --
// every active level, every iteration -- on the pair's own pyramids in global memory (a "slot" = the device
// buffers of a child context).  Same loops as the cooperative kernels above with block barriers instead of grid
// barriers, so a wave of several hundred pairs runs with no grid-wide synchronisation at all and pairs that stop
// early make room for the next CTA.  Used for what the shared-memory-resident kernels (kernels_batch.cu) do not
// take: Ceres mode, the photometric + depth solver, blurred or large levels.
// ---------------------------------------------------------------------------------------------
#ifndef PHOVO_SLOT_MINB
#define PHOVO_SLOT_MINB 2
#endif
template <int MODE, bool CLUSTER>
__global__ void __launch_bounds__(kCoopBlock, PHOVO_SLOT_MINB) k_align_slots(const __grid_constant__ SlotLevels LS, const SlotArgs* __restrict__ slots,
                                                                const double* __restrict__ init_states) {
  constexpr int S = CLUSTER ? 2 : 1;
  const int slot = (int)blockIdx.x / level_num_blocks<S>();      // clusters are runs of consecutive blocks
  const SlotArgs& A = slots[slot];
  if (level_block_rank<S>() == 0 && threadIdx.x == 0) {   // k_set_state for this slot: the caller's initial state (zero if none), counters cleared, no log
    double s[6];
    for (int k = 0; k < 6; ++k) s[k] = init_states ? init_states[(size_t)slot * 6 + k] : 0.;
    PoseDev* pose = A.pose;
    pose_set_state(pose, s);
    pose->iteration = 0; pose->done = 0; pose->log_count = 0; pose->log_capacity = 0;
    for (int l = 0; l < PHOVO_MAX_LEVELS; ++l) pose->iters_per_level[l] = 0;
  }
  level_barrier<S>();
  for (int a = 0; a < LS.count; ++a) {
    const LevelParams& L = LS.L[a];
    if (MODE == PHOVO_MODE_CERES) level_loop_ceres<S>(L, A.P[L.level], A.pose, A.partials, nullptr, LS.lm[a]);
    else level_loop<MODE, false, S>(L, A.P[L.level], A.pose, A.partials, nullptr, ShardArgs{nullptr, 0, 1, 0ull, nullptr});
    level_barrier<S>();   // the level's PoseDev is in global memory (written by rank 0, re-read by every CTA of the pair); shared scratch is free again
  }
}

// state + executed iterations per level of every slot -> two dense arrays (one D2H copy per wave)
__global__ void k_gather_slots(const SlotArgs* __restrict__ slots, int n, double* __restrict__ states, int32_t* __restrict__ iters) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const PoseDev* p = slots[s].pose;
  for (int k = 0; k < 6; ++k) states[(size_t)s * 6 + k] = p->state[k];
  for (int l = 0; l < PHOVO_MAX_LEVELS; ++l) iters[(size_t)s * PHOVO_MAX_LEVELS + l] = p->iters_per_level[l];
}

// smallest depth of a level inside (lo, hi), as the bits of a positive double (ordered like unsigned integers)
__global__ void __launch_bounds__(256) k_min_valid_depth(const double* __restrict__ D, int n, double lo, double hi, unsigned long long* out) {
  unsigned long long m = 0x7ff0000000000000ull;   // +inf: no valid pixel
  for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
    const double d = __ldg(D + i);
    if ((lo < d) & (d < hi) & (d > 0.)) m = min(m, (unsigned long long)__double_as_longlong(d));
  }
  for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMin(out, m);
}

inline int grid_for(int n, int sm_count) {
  // one pixel per thread up to 8 CTAs per SM, then a fixed persistent grid (grid-stride loop);
  // the grid is a pure function of the level size and the device, so the partial-sum order is reproducible.
  const int want = (n + kBlock - 1) / kBlock;
  const int cap = sm_count * 8;
  return want < cap ? (want > 0 ? want : 1) : cap;
}

}  // namespace

int partials_blocks(int sm_count) { return (sm_count > 0 ? sm_count : 1) * 8; }

int launch_fill_i32(cudaStream_t stream, int* p, int value, size_t n, int sm_count) {
  const size_t want = (n + 255) / 256, cap = (size_t)partials_blocks(sm_count);
  const int blocks = (int)(want < cap ? (want ? want : 1) : cap);
  k_fill_i32<<<blocks, 256, 0, stream>>>(p, value, n);
  return 1;
}

int launch_min_valid_depth(cudaStream_t stream, const double* D, int n, double lo, double hi, double* out, int sm_count) {
  cudaMemsetAsync(out, 0xff, sizeof(double), stream);                 // all ones: larger than any positive double's bits
  const int want = (n + 255) / 256, cap = partials_blocks(sm_count);
  k_min_valid_depth<<<want < cap ? (want > 0 ? want : 1) : cap, 256, 0, stream>>>(D, n, lo, hi, (unsigned long long*)out);
  return 1;
}

int launch_set_state(cudaStream_t stream, PoseDev* pose, const double* state_dev, const double s[6], int log_capacity) {
  if (state_dev) k_set_state<<<1, 32, 0, stream>>>(pose, state_dev, log_capacity, 0, 0, 0, 0, 0, 0);
  else k_set_state<<<1, 32, 0, stream>>>(pose, nullptr, log_capacity, s[0], s[1], s[2], s[3], s[4], s[5]);
  return 1;
}

int launch_begin_level(cudaStream_t stream, PoseDev* pose, int max_iters) {
  k_begin_level<<<1, 32, 0, stream>>>(pose, max_iters);
  return 1;
}

int launch_iteration_kernels(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, const PoseDev* pose,
                             double* partials, int sm_count, int* grid_out, double* dump_res, double* dump_jac,
                             bool clear_winner_first) {
  const int n = L.rows * L.cols;
  const int grid = grid_for(n, sm_count);
  int launches = 0;
  if (clear_winner_first) launches += launch_fill_i32(stream, P.winner, -1, (size_t)n, sm_count);
  if (L.mode == PHOVO_MODE_BIOBJECTIVE) {
    k_winner_bi<<<grid, kBlock, 0, stream>>>(L, P, pose);
    const int grid2 = grid_for(2 * n, sm_count);
    if (dump_res || dump_jac) k_normal_eq_bi<true><<<grid2, kBlock, 0, stream>>>(L, P, pose, partials, dump_res, dump_jac);
    else k_normal_eq_bi<false><<<grid2, kBlock, 0, stream>>>(L, P, pose, partials, nullptr, nullptr);
    *grid_out = grid2;
    return launches + 2;
  }
  if (L.mode == PHOVO_MODE_CERES) k_winner<true><<<grid, kBlock, 0, stream>>>(L, P, pose);
  else k_winner<false><<<grid, kBlock, 0, stream>>>(L, P, pose);
  const bool dump = dump_res || dump_jac;
  switch (L.mode) {
    case PHOVO_MODE_ANALYTIC_REF:
      if (dump) k_normal_eq<0, true><<<grid, kBlock, 0, stream>>>(L, P, pose, partials, dump_res, dump_jac);
      else k_normal_eq<0, false><<<grid, kBlock, 0, stream>>>(L, P, pose, partials, nullptr, nullptr);
      break;
    case PHOVO_MODE_ANALYTIC_FIXED:
      if (dump) k_normal_eq<1, true><<<grid, kBlock, 0, stream>>>(L, P, pose, partials, dump_res, dump_jac);
      else k_normal_eq<1, false><<<grid, kBlock, 0, stream>>>(L, P, pose, partials, nullptr, nullptr);
      break;
    default:
      if (dump) k_normal_eq<2, true><<<grid, kBlock, 0, stream>>>(L, P, pose, partials, dump_res, dump_jac);
      else k_normal_eq<2, false><<<grid, kBlock, 0, stream>>>(L, P, pose, partials, nullptr, nullptr);
      break;
  }
  *grid_out = grid;
  return launches + 2;
}

// One cooperative launch for the whole iteration loop of a level.  Returns the number of launches
// (1) or -1 if cooperative launch is not available (the caller falls back to the graph path).
int launch_level_coop(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, PoseDev* pose, double* partials,
                      phovo_iter_stats* log, LaunchState* ls, int sm_count, int* grid_out, cudaError_t* err,
                      ShardExchange* const* peers_dev, int rank, int world, unsigned long long epoch_base, const double* level_dmin) {
  int* g_coop_blocks_per_sm = ls->coop_blocks_per_sm;
  const bool shard = peers_dev != nullptr && world > 1 && L.mode != PHOVO_MODE_BIOBJECTIVE;
  const int m = shard ? (L.mode == PHOVO_MODE_ANALYTIC_FIXED ? 4 : 3)
                      : L.mode == PHOVO_MODE_BIOBJECTIVE ? 2 : L.mode == PHOVO_MODE_ANALYTIC_FIXED ? 1 : 0;
  void* fn = m == 4 ? (void*)k_level_coop<1, true> : m == 3 ? (void*)k_level_coop<0, true>
           : m == 2 ? (void*)k_level_coop<3, false> : m ? (void*)k_level_coop<1, false> : (void*)k_level_coop<0, false>;
  if (g_coop_blocks_per_sm[m] < 0) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kCoopBlock, 0) != cudaSuccess) nb = 0;
    g_coop_blocks_per_sm[m] = nb;
  }
  if (g_coop_blocks_per_sm[m] < 1) { *err = cudaErrorCooperativeLaunchTooLarge; return -1; }
  const int n = L.rows * L.cols;
  int grid = (n + kCoopBlock - 1) / kCoopBlock;
  const int cap = sm_count * (g_coop_blocks_per_sm[m] < 2 ? g_coop_blocks_per_sm[m] : 2);
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  LevelParams Lc = L; LevelPtrs Pc = P;
  ShardArgs Sc; Sc.peers = shard ? peers_dev : nullptr; Sc.rank = rank; Sc.world = shard ? world : 1; Sc.epoch_base = epoch_base; Sc.dmin = level_dmin;
  void* args[] = {&Lc, &Pc, &pose, &partials, &log, &Sc};
  *err = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kCoopBlock), args, 0, stream);
  if (*err != cudaSuccess) return -1;
  *grid_out = grid;
  return 1;
}

// One cluster per level launch.  Returns 1, 0 if the level does not qualify (mode, size), -1 on a launch error.
int launch_level_cluster(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, PoseDev* pose, phovo_iter_stats* log, LaunchState* ls,
                         cudaError_t* err) {
  *err = cudaSuccess;
  const int n = L.rows * L.cols;
  if (n > kClusterMaxPixels || (L.mode != PHOVO_MODE_ANALYTIC_REF && L.mode != PHOVO_MODE_ANALYTIC_FIXED)) return 0;
  if (L.row_begin != 0 || L.row_end != L.rows) return 0;
  void (*fn)(LevelParams, LevelPtrs, PoseDev*, phovo_iter_stats*) = L.mode == PHOVO_MODE_ANALYTIC_FIXED ? k_level_cluster<1> : k_level_cluster<0>;
  const int chunk = (n + kClusterSize - 1) / kClusterSize;
  const size_t smem = sizeof(double) * PHOVO_ACC_STRIDE * (kClusterSize + kClusterBlock / 32) + (size_t)chunk * 5 + 16;
  bool* prepared = ls->cluster_prepared;
  const int m = L.mode == PHOVO_MODE_ANALYTIC_FIXED ? 1 : 0;
  if (!prepared[m]) {
    if ((*err = cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1)) != cudaSuccess) return -1;
    if ((*err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * PHOVO_ACC_STRIDE * (kClusterSize + kClusterBlock / 32) + (size_t)((kClusterMaxPixels + kClusterSize - 1) / kClusterSize) * 5 + 16))) != cudaSuccess) return -1;
    prepared[m] = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(kClusterSize); cfg.blockDim = dim3(kClusterBlock); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kClusterSize; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  *err = cudaLaunchKernelEx(&cfg, fn, L, P, pose, log);
  return *err == cudaSuccess ? 1 : -1;
}

int launch_level_coop_ceres(cudaStream_t stream, const LevelParams& L, const LevelPtrs& P, PoseDev* pose, double* partials,
                            phovo_iter_stats* log, const LmParams& lm, LaunchState* ls, int sm_count, cudaError_t* err) {
  int& blocks_per_sm = ls->ceres_blocks_per_sm;
  void* fn = (void*)k_level_coop_ceres;
  if (blocks_per_sm < 0) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kCoopBlock, 0) != cudaSuccess) nb = 0;
    blocks_per_sm = nb;
  }
  if (blocks_per_sm < 1) { *err = cudaErrorCooperativeLaunchTooLarge; return -1; }
  const int n = L.rows * L.cols;
  int grid = (n + kCoopBlock - 1) / kCoopBlock;
  const int cap = sm_count * (blocks_per_sm < 2 ? blocks_per_sm : 2);
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  LevelParams Lc = L; LevelPtrs Pc = P; LmParams lmc = lm;
  void* args[] = {&Lc, &Pc, &pose, &partials, &log, &lmc};
  *err = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kCoopBlock), args, 0, stream);
  return *err == cudaSuccess ? 1 : -1;
}

int launch_reduce_solve(cudaStream_t stream, const LevelParams& L, PoseDev* pose, const double* partials, int grid,
                        phovo_iter_stats* log, unsigned long long cond_handle) {
  k_reduce_solve<<<1, 1024, 0, stream>>>(L, pose, partials, grid, log, cond_handle);
  return 1;
}

int launch_reduce_only(cudaStream_t stream, const LevelParams& L, const PoseDev* pose, const double* partials, int grid,
                       phovo_iter_stats* out) {
  k_reduce_only<<<1, 1024, 0, stream>>>(L, pose, partials, grid, out);
  return 1;
}

int launch_reduce_to_buffer(cudaStream_t stream, const double* partials, int grid, double* buffer) {
  k_reduce_to_buffer<<<1, 1024, 0, stream>>>(nullptr, partials, grid, buffer);
  return 1;
}

int launch_reduce_exchange(cudaStream_t stream, const PoseDev* pose, const double* partials, int grid, double* buffer,
                           ShardExchange* const* peers_dev, int rank, int world, unsigned long long epoch) {
  k_reduce_exchange<<<1, 1024, 0, stream>>>(pose, partials, grid, buffer, peers_dev, rank, world, epoch);
  return 1;
}

int launch_solve_from_buffer(cudaStream_t stream, const LevelParams& L, PoseDev* pose, const double* buffer,
                             phovo_iter_stats* log) {
  k_solve_from_buffer<<<1, 32, 0, stream>>>(L, pose, buffer, log);
  return 1;
}

template <int MODE>
static cudaError_t launch_align_slots_mode(cudaStream_t stream, const SlotLevels& LS, const SlotArgs* slots, int num_slots, const double* init_states, int cluster) {
  if (cluster <= 1) {
    k_align_slots<MODE, false><<<num_slots, kCoopBlock, 0, stream>>>(LS, slots, init_states);
    return cudaGetLastError();
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(num_slots * cluster)); cfg.blockDim = dim3(kCoopBlock); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_align_slots<MODE, true>, LS, slots, init_states);
}

// `cluster` CTAs per slot (1, 2, 4 or 8: the portable cluster sizes)
int launch_align_slots(cudaStream_t stream, int mode, const SlotLevels& LS, const SlotArgs* slots, int num_slots, const double* init_states, int cluster) {
  if (num_slots < 1) return 0;   // (no active level: the kernel still writes the initial state into every slot's PoseDev)
  cudaError_t e;
  switch (mode) {
    case PHOVO_MODE_ANALYTIC_REF:   e = launch_align_slots_mode<0>(stream, LS, slots, num_slots, init_states, cluster); break;
    case PHOVO_MODE_ANALYTIC_FIXED: e = launch_align_slots_mode<1>(stream, LS, slots, num_slots, init_states, cluster); break;
    case PHOVO_MODE_CERES:          e = launch_align_slots_mode<2>(stream, LS, slots, num_slots, init_states, cluster); break;
    default:                        e = launch_align_slots_mode<3>(stream, LS, slots, num_slots, init_states, cluster); break;
  }
  return e == cudaSuccess ? 1 : -1;
}

int launch_gather_slots(cudaStream_t stream, const SlotArgs* slots, int num_slots, double* states, int32_t* iters) {
  k_gather_slots<<<(num_slots + 127) / 128, 128, 0, stream>>>(slots, num_slots, states, iters);
  return 1;
}

}  // namespace phovo
