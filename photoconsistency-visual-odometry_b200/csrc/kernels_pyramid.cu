// kernels_pyramid.cu -- frame setup for the general (any resolution, any config) path:
// K1 pyramid level from the full-resolution source, K2b Gaussian blur, K2 Scharr.  All level images are fp64, bit-identical
// to the reference's cv::Mat_<double> pyramids as OpenCV's portable C++ code computes them (same
// operation order, no FMA contraction; pinned against cv2 with its IPP / SIMD dispatch switched off).
// Replaces CPhotoconsistencyOdometryAnalytic.h:115-189 (BuildPyramid / BuildDerivativesPyramids).
// The batched path has its own fused, shared-memory version (kernels_batch.cu).
#include <math.h>

#include "phovo_kernels.h"
#include "phovo_level.cuh"

namespace phovo {
namespace {

// K1.  One thread per output pixel (level_value, phovo_level.cuh).  A warp reads one contiguous span of each of two
// source rows, so every 32-byte sector fetched is used by the warp.
template <typename T>
__global__ void __launch_bounds__(256) k_build_level(const void* __restrict__ src, size_t step, double src_scale,
                                                     int rows, int cols, int level, double scale,
                                                     double* __restrict__ dst, int orows, int ocols) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= ocols || y >= orows) return;
  dst[(size_t)y * ocols + x] = level_value<T>(src, step, src_scale, rows, cols, level, scale, y, x);
}

// K1+K2 fused over ALL active levels of one frame: one thread per level pixel (levels laid end to end
// in the thread index).  Every level is resized from the ORIGINAL image (AN:132), so the levels do not
// depend on each other; with GRAD the thread also evaluates its eight level neighbours (the same
// four-tap function, so the same bits as the stored image; the taps come from L1/L2) and applies
// cv::Scharr's arithmetic (AN:181-187) -- one launch instead of two per level, which is what a
// VO frame's set-up time consists of.
template <typename T, bool GRAD>
__global__ void __launch_bounds__(256) k_build_levels(const void* __restrict__ src, size_t step, double src_scale,
                                                      int rows, int cols, const __grid_constant__ PyramidLevels P) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= P.px_offset[P.num]) return;
  int a = 0;
  while (j >= P.px_offset[a + 1]) ++a;
  const int q = j - P.px_offset[a];
  const int oc = P.ocols[a], orr = P.orows[a], level = P.level[a];
  const int y = q / oc, x = q - y * oc;
  const double scale = (double)(1 << level);
  if (!GRAD) {
    P.dst[a][q] = level_value<T>(src, step, src_scale, rows, cols, level, scale, y, x);
    return;
  }
  const int ym = reflect101(y - 1, orr), yp = reflect101(y + 1, orr), xm = reflect101(x - 1, oc), xp = reflect101(x + 1, oc);
  double t[3][3];
  const int ys[3] = {ym, y, yp}, xs[3] = {xm, x, xp};
#pragma unroll
  for (int dy = 0; dy < 3; ++dy)
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) t[dy][dx] = level_value<T>(src, step, src_scale, rows, cols, level, scale, ys[dy], xs[dx]);
  double gx, gy;
  scharr_taps(t, P.ks0[a], P.ks1[a], gx, gy);
  P.dst[a][q] = t[1][1];
  P.gx[a][q] = gx;
  P.gy[a][q] = gy;
}

struct GaussTaps { double k[32]; int n; };

// K2b row pass: generic cv RowFilter order (taps accumulated left to right).
__global__ void __launch_bounds__(256) k_gauss_rows(const double* __restrict__ src, double* __restrict__ dst, int rows, int cols, GaussTaps t) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= cols) return;
  const double* S = src + (size_t)r * cols;
  const int a = t.n / 2;
  double s = __dmul_rn(t.k[0], S[reflect101(c - a, cols)]);
  for (int k = 1; k < t.n; ++k) s = __dadd_rn(s, __dmul_rn(t.k[k], S[reflect101(c - a + k, cols)]));
  dst[(size_t)r * cols + c] = s;
}
// K2b column pass: cv SymmColumnFilter order (centre tap, then symmetric pairs).
__global__ void __launch_bounds__(256) k_gauss_cols(const double* __restrict__ src, double* __restrict__ dst, int rows, int cols, GaussTaps t) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= cols) return;
  const int a = t.n / 2;
  double s = __dmul_rn(t.k[a], src[(size_t)r * cols + c]);
  for (int k = 1; k <= a; ++k) {
    const double p = src[(size_t)reflect101(r + k, rows) * cols + c], q = src[(size_t)reflect101(r - k, rows) * cols + c];
    s = __dadd_rn(s, __dmul_rn(t.k[a + k], __dadd_rn(p, q)));
  }
  dst[(size_t)r * cols + c] = s;
}

// K2: Scharr in x and y with cv::Scharr's separable evaluation order (derivative kernel [-1 0 1],
// smoothing kernel [3 10 3]*scale).  32x8 tiles with a
// 1-pixel halo staged in shared memory so every level pixel is read from global memory once
// (plus halo), then 18 shared-memory reads per pixel.
#define SCH_TW 32
#define SCH_TH 8
__global__ void __launch_bounds__(SCH_TW * SCH_TH) k_scharr_store(const double* __restrict__ img, int rows, int cols,
                                                                   double ks0, double ks1,
                                                                   double* __restrict__ Gx, double* __restrict__ Gy) {
  __shared__ double tile[SCH_TH + 2][SCH_TW + 2];
  const int x0 = blockIdx.x * SCH_TW, y0 = blockIdx.y * SCH_TH;
  for (int i = threadIdx.y * SCH_TW + threadIdx.x; i < (SCH_TH + 2) * (SCH_TW + 2); i += SCH_TW * SCH_TH) {
    const int ty = i / (SCH_TW + 2), tx = i % (SCH_TW + 2);
    const int gy = reflect101(min(y0 + ty - 1, rows), rows), gx = reflect101(min(x0 + tx - 1, cols), cols);
    tile[ty][tx] = img[(size_t)gy * cols + gx];
  }
  __syncthreads();
  const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
  if (x >= cols || y >= rows) return;
  const int tx = threadIdx.x + 1, ty = threadIdx.y + 1;
  // dx: row filter [-1 0 1] on three rows, then column filter centre-first
  const double dm = __dsub_rn(tile[ty - 1][tx + 1], tile[ty - 1][tx - 1]);
  const double d0 = __dsub_rn(tile[ty][tx + 1], tile[ty][tx - 1]);
  const double dp = __dsub_rn(tile[ty + 1][tx + 1], tile[ty + 1][tx - 1]);
  const double gx = __dadd_rn(__dmul_rn(ks1, d0), __dmul_rn(ks0, __dadd_rn(dp, dm)));
  // dy: row filter [3 10 3]*scale left-to-right on rows y-1 and y+1, then column [-1 0 1]
  const double sm = __dadd_rn(__dadd_rn(__dmul_rn(ks0, tile[ty - 1][tx - 1]), __dmul_rn(ks1, tile[ty - 1][tx])), __dmul_rn(ks0, tile[ty - 1][tx + 1]));
  const double sp = __dadd_rn(__dadd_rn(__dmul_rn(ks0, tile[ty + 1][tx - 1]), __dmul_rn(ks1, tile[ty + 1][tx])), __dmul_rn(ks0, tile[ty + 1][tx + 1]));
  const double gy = __dsub_rn(sp, sm);
  const size_t o = (size_t)y * cols + x;

  Gx[o] = gx;
  Gy[o] = gy;
}

}  // namespace

int launch_build_level(cudaStream_t stream, const void* src, int src_type, size_t step, double src_scale,
                       int rows, int cols, int level, double* dst, int orows, int ocols) {
  dim3 block(64, 4), grid((ocols + 63) / 64, (orows + 3) / 4);
  const double scale = ldexp(1.0, level);
  switch (src_type) {
    case SRC_U8:  k_build_level<uint8_t><<<grid, block, 0, stream>>>(src, step, src_scale, rows, cols, level, scale, dst, orows, ocols); break;
    case SRC_U16: k_build_level<uint16_t><<<grid, block, 0, stream>>>(src, step, src_scale, rows, cols, level, scale, dst, orows, ocols); break;
    case SRC_F32: k_build_level<float><<<grid, block, 0, stream>>>(src, step, src_scale, rows, cols, level, scale, dst, orows, ocols); break;
    default:      k_build_level<double><<<grid, block, 0, stream>>>(src, step, src_scale, rows, cols, level, scale, dst, orows, ocols); break;
  }
  return 1;
}

int launch_build_levels(cudaStream_t stream, const void* src, int src_type, size_t step, double src_scale,
                        int rows, int cols, const PyramidLevels& P, bool gradients) {
  const int total = P.px_offset[P.num];
  if (total <= 0) return 0;
  const int grid = (total + 255) / 256;
#define PHOVO_BUILD_LEVELS(T)                                                                                   \
  if (gradients) k_build_levels<T, true><<<grid, 256, 0, stream>>>(src, step, src_scale, rows, cols, P);        \
  else k_build_levels<T, false><<<grid, 256, 0, stream>>>(src, step, src_scale, rows, cols, P)
  switch (src_type) {
    case SRC_U8:  PHOVO_BUILD_LEVELS(uint8_t); break;
    case SRC_U16: PHOVO_BUILD_LEVELS(uint16_t); break;
    case SRC_F32: PHOVO_BUILD_LEVELS(float); break;
    default:      PHOVO_BUILD_LEVELS(double); break;
  }
#undef PHOVO_BUILD_LEVELS
  return 1;
}

int launch_gaussian_blur(cudaStream_t stream, double* img, double* tmp, int rows, int cols, int ksize, double sigma) {
  if (ksize <= 1) return 0;
  GaussTaps t; t.n = ksize;
  // cv::getGaussianKernel(ksize, sigma, CV_64F)
  const double sigmaX = sigma > 0 ? sigma : ((ksize - 1) * 0.5 - 1) * 0.3 + 0.8;
  const double scale2X = -0.5 / (sigmaX * sigmaX);
  double sum = 0;
  for (int i = 0; i < ksize; ++i) { const double x = i - (ksize - 1) * 0.5; t.k[i] = exp(scale2X * x * x); sum += t.k[i]; }
  sum = 1. / sum;
  for (int i = 0; i < ksize; ++i) t.k[i] *= sum;
  dim3 block(256), grid((cols + 255) / 256, rows);
  k_gauss_rows<<<grid, block, 0, stream>>>(img, tmp, rows, cols, t);
  k_gauss_cols<<<grid, block, 0, stream>>>(tmp, img, rows, cols, t);
  return 2;
}

int launch_scharr_store(cudaStream_t stream, const double* img, int rows, int cols, double scale,
                        double* Gx, double* Gy) {
  double ks0 = 3., ks1 = 10.;
  if (scale != 1.) { ks0 *= scale; ks1 *= scale; }
  dim3 block(SCH_TW, SCH_TH), grid((cols + SCH_TW - 1) / SCH_TW, (rows + SCH_TH - 1) / SCH_TH);
  k_scharr_store<<<grid, block, 0, stream>>>(img, rows, cols, ks0, ks1, Gx, Gy);
  return 1;
}


// ---------------------------------------------------------------------------------------------
// helpers of the photometric + depth solver (BiObjective.h:213-239, 299)
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) k_scale(const double* __restrict__ src, double alpha, double* __restrict__ dst, size_t n) {
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) dst[i] = __dmul_rn(src[i], alpha);
}
// one CTA, fixed order: thread t sums elements t, t+1024, ...; then a fixed tree over the threads
__global__ void __launch_bounds__(1024) k_mean_ratio(const double* __restrict__ a, const double* __restrict__ b, size_t n, double* out) {
  __shared__ double sa[1024], sb[1024];
  double x = 0., y = 0.;
  for (size_t i = threadIdx.x; i < n; i += 1024) { x += a[i]; y += b[i]; }
  sa[threadIdx.x] = x; sb[threadIdx.x] = y;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { sa[threadIdx.x] += sa[threadIdx.x + o]; sb[threadIdx.x] += sb[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (sa[0] / (double)n) / (sb[0] / (double)n);   // cv::mean(I).val[0] / cv::mean(D).val[0]
}
}  // namespace

int launch_scale(cudaStream_t stream, const double* src, double alpha, double* dst, size_t n) {
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  k_scale<<<blocks > 0 ? blocks : 1, 256, 0, stream>>>(src, alpha, dst, n);
  return 1;
}
int launch_mean_ratio(cudaStream_t stream, const double* a, const double* b, size_t n, double* out) {
  k_mean_ratio<<<1, 1024, 0, stream>>>(a, b, n, out);
  return 1;
}

// ---------------------------------------------------------------------------------------------
// phovo::warpImage, CPhotoconsistencyOdometry.h:73-134 (post-hoc visualisation of both apps), for a chunk of pairs:
// blockIdx.y is the pair, so no block spans two pairs and every pair reads its own Rt
// ---------------------------------------------------------------------------------------------
namespace {
// Each thread takes kWarpPix pixels kWarpThreads apart and issues all their loads before it uses any: one pixel per
// thread leaves a single dependent memory access in flight per thread, and both kernels then wait on latency.
constexpr int kWarpThreads = 256, kWarpPix = 8, kWarpTile = kWarpThreads * kWarpPix;

template <typename DT>
__global__ void __launch_bounds__(kWarpThreads) k_warp_splat(const __grid_constant__ WarpImages W, const __grid_constant__ WarpIntrinsics I,
                                                             uint32_t* __restrict__ keys) {
  const int p = blockIdx.y;
  const int n = W.rows * W.cols;                                                       // < 2^31: 32-bit index arithmetic
  const int i0 = blockIdx.x * kWarpTile + threadIdx.x;
  const char* dbase = (const char*)W.depth + p * W.depth_pair;
  double dv[kWarpPix];
#pragma unroll
  for (int j = 0; j < kWarpPix; ++j) {
    const int i = i0 + j * kWarpThreads;
    dv[j] = 0.;
    if (i < n) {
      const int r = i / W.cols, c = i - r * W.cols;
      dv[j] = (double)__ldg((const DT*)(dbase + (size_t)r * W.depth_step) + c);
    }
  }
  const double* R = W.rts + (size_t)p * 16;
  double M[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) M[k] = __ldg(R + k);
  uint32_t* pk = keys + (size_t)p * n;
#pragma unroll
  for (int j = 0; j < kWarpPix; ++j) {
    const int i = i0 + j * kWarpThreads;
    double d = dv[j];
    if (sizeof(DT) == 2) d = __dmul_rn(d, W.depth_scale);
    if (!(d > 0.)) continue;                                                           // BASE:106 (also i >= n: d = 0)
    const int r = i / W.cols, c = i - r * W.cols;
    // BASE:109-112, fp64, the reference's operation order, no FMA contraction
    const double px = __dmul_rn(__dmul_rn(__dsub_rn((double)c, I.ox), d), I.inv_fx);
    const double py = __dmul_rn(__dmul_rn(__dsub_rn((double)r, I.oy), d), I.inv_fy);
    // Eigen 4x4 * 4x1 (BASE:115): sum over k = 0..3 in order, the homogeneous 1 multiplies the translation
    const double X = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(M[0], px), __dmul_rn(M[1], py)), __dmul_rn(M[2], d)), M[3]);
    const double Y = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(M[4], px), __dmul_rn(M[5], py)), __dmul_rn(M[6], d)), M[7]);
    const double Z = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(M[8], px), __dmul_rn(M[9], py)), __dmul_rn(M[10], d)), M[11]);
    const double tc = __dadd_rn(__ddiv_rn(__dmul_rn(X, I.fx), Z), I.ox);               // BASE:118-121: true division
    const double tr = __dadd_rn(__ddiv_rn(__dmul_rn(Y, I.fy), Z), I.oy);
    // static_cast<int>: truncation toward zero; NaN / out-of-range (undefined in the reference) -> skipped
    if (!(tc > -1. && tc < (double)W.cols && tr > -1. && tr < (double)W.rows)) continue;
    const int tj = (int)tc, ti = (int)tr;
    // raster-order last writer wins: the largest source index; 0 = nothing landed
    atomicMax(pk + ti * W.cols + tj, (uint32_t)(i + 1));
  }
}

// CLEAR: leave the keys zero for the next chunk (instead of a memset before the splat)
template <bool CLEAR>
__global__ void __launch_bounds__(kWarpThreads) k_warp_resolve(const __grid_constant__ WarpImages W, uint32_t* __restrict__ keys) {
  const int p = blockIdx.y;
  const int n = W.rows * W.cols;
  const int i0 = blockIdx.x * kWarpTile + threadIdx.x;
  uint32_t* pk = keys + (size_t)p * n;
  const uint8_t* gray = W.gray + p * W.gray_pair;
  const uint8_t* target = W.target ? W.target + p * W.target_pair : nullptr;
  uint32_t kv[kWarpPix];
  int tv[kWarpPix];
#pragma unroll
  for (int j = 0; j < kWarpPix; ++j) {
    const int i = i0 + j * kWarpThreads;
    kv[j] = 0; tv[j] = 0;
    if (i < n) {
      kv[j] = pk[i];
      if (target) { const int r = i / W.cols; tv[j] = __ldg(target + (size_t)r * W.target_step + (i - r * W.cols)); }
    }
  }
  int gv[kWarpPix];
#pragma unroll
  for (int j = 0; j < kWarpPix; ++j) {                                                 // BASE:98 zeros()
    gv[j] = 0;
    if (kv[j]) {
      const int s = (int)(kv[j] - 1), sr = s / W.cols;
      gv[j] = __ldg(gray + (size_t)sr * W.gray_step + (s - sr * W.cols));
    }
  }
  unsigned landed = 0, absdiff = 0;
#pragma unroll
  for (int j = 0; j < kWarpPix; ++j) {
    const int i = i0 + j * kWarpThreads;
    if (i >= n) continue;
    if (CLEAR && kv[j]) pk[i] = 0;
    const int r = i / W.cols, c = i - r * W.cols, v = gv[j];
    if (W.warped) W.warped[p * W.warped_pair + (size_t)r * W.warped_step + c] = (uint8_t)v;
    const unsigned a = (unsigned)(tv[j] > v ? tv[j] - v : v - tv[j]);
    if (W.diff) W.diff[p * W.diff_pair + (size_t)r * W.diff_step + c] = (uint8_t)a;
    if (kv[j]) { landed += 1; absdiff += a; }
  }
  if (!W.num_landed) return;
  // block sums, then one integer atomic per block and quantity: the totals do not depend on the order
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    landed += __shfl_down_sync(0xffffffffu, landed, o);
    absdiff += __shfl_down_sync(0xffffffffu, absdiff, o);
  }
  __shared__ unsigned s_landed[kWarpThreads / 32], s_abs[kWarpThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_landed[warp] = landed; s_abs[warp] = absdiff; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned a = 0, b = 0;
    for (int w = 0; w < kWarpThreads / 32; ++w) { a += s_landed[w]; b += s_abs[w]; }
    if (a) atomicAdd((unsigned*)W.num_landed + p, a);
    if (b && W.sum_abs_diff) atomicAdd((unsigned long long*)W.sum_abs_diff + p, (unsigned long long)b);
  }
}
}  // namespace

int launch_warp_images(cudaStream_t stream, const WarpImages& W, int depth_type, const WarpIntrinsics& I, int num_pairs,
                       uint32_t* keys, bool clear_keys) {
  const int n = W.rows * W.cols;
  const dim3 grid((unsigned)((n + kWarpTile - 1) / kWarpTile), (unsigned)num_pairs);
  switch (depth_type) {
    case SRC_F32: k_warp_splat<float><<<grid, kWarpThreads, 0, stream>>>(W, I, keys); break;
    case SRC_U16: k_warp_splat<uint16_t><<<grid, kWarpThreads, 0, stream>>>(W, I, keys); break;
    default:      k_warp_splat<double><<<grid, kWarpThreads, 0, stream>>>(W, I, keys); break;
  }
  if (clear_keys) k_warp_resolve<true><<<grid, kWarpThreads, 0, stream>>>(W, keys);
  else k_warp_resolve<false><<<grid, kWarpThreads, 0, stream>>>(W, keys);
  return 2;
}

}  // namespace phovo
