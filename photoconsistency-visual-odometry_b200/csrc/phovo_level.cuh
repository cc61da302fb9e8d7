// phovo_level.cuh -- one pyramid level pixel straight from the full-resolution image, and cv::Scharr at it.
// The frame set-up kernels (kernels_pyramid.cu) and the target depth of the batched normal equations (kernels_eval.cu)
// use these, so that both produce the per-pair path's level images bit for bit: fp64 with OpenCV's portable C++
// operation order, no FMA contraction.
#ifndef PHOVO_LEVEL_CUH_
#define PHOVO_LEVEL_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

namespace phovo {

__device__ __forceinline__ int reflect101(int p, int len) {
  if (len == 1) return 0;
  while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
  return p;
}

template <typename T>
__device__ __forceinline__ double load_src(const void* base, size_t step_bytes, int r, int c, double scale);
template <>
__device__ __forceinline__ double load_src<uint8_t>(const void* base, size_t step, int r, int c, double scale) {
  return __dmul_rn((double)__ldg((const uint8_t*)base + (size_t)r * step + c), scale);
}
template <>
__device__ __forceinline__ double load_src<uint16_t>(const void* base, size_t step, int r, int c, double scale) {
  return __dmul_rn((double)__ldg((const uint16_t*)((const char*)base + (size_t)r * step) + c), scale);
}
template <>
__device__ __forceinline__ double load_src<float>(const void* base, size_t step, int r, int c, double) {
  return (double)__ldg((const float*)((const char*)base + (size_t)r * step) + c);
}
template <>
__device__ __forceinline__ double load_src<double>(const void* base, size_t step, int r, int c, double) {
  return __ldg((const double*)((const char*)base + (size_t)r * step) + c);
}

// One axis of OpenCV's INTER_LINEAR table: f = (float)((d+0.5)*scale - 0.5); s = floor(f); f -= s.
__device__ __forceinline__ void linear_axis(int d, double scale, int ssize, bool is_x, int& s0, float& w1) {
  float f = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= (float)s;
  if (s < 0) { f = 0.f; s = 0; }
  if (is_x && s >= ssize - 1) { f = 0.f; s = ssize - 1; }
  s0 = s; w1 = f;
}

// For the exact factor 2^-level, level >= 2, the four taps are the central 2x2 of the pixel's 2^level cell with
// weights 1/2 (horizontal pair first, then vertical) -- cv::resize INTER_LINEAR from the ORIGINAL image, AN:132; level 1
// is OpenCV's area path (below).
// value of level pixel (y, x): the conversion of the source pixel at level 0, else cv::resize's four taps
template <typename T>
__device__ __forceinline__ double level_value(const void* __restrict__ src, size_t step, double src_scale,
                                              int rows, int cols, int level, double scale, int y, int x) {
  if (level == 0) return load_src<T>(src, step, y, x, src_scale);
  if (level == 1) {
    // cv::resize by exactly 1/2 is NOT bilinear: resize.cpp switches INTER_LINEAR to INTER_AREA when
    // both integer scale factors are 2 (resizeAreaFast_Invoker<double,double>): a whole 2x2 cell is
    // ((S00 + S01) + S10) + S11 times 0.25f; a cell cut by the right / bottom edge (sizes = 3 mod 4:
    // the output size is cvRound(size / 2)) sums its taps inside the image in raster order and
    // divides by their count IN SINGLE PRECISION ((float)sum / count).
    const int sy0 = 2 * y, sx0 = 2 * x;
    if (sy0 + 2 <= rows && x < cols / 2) {
      const double a = load_src<T>(src, step, sy0, sx0, src_scale), b = load_src<T>(src, step, sy0, sx0 + 1, src_scale);
      const double c = load_src<T>(src, step, sy0 + 1, sx0, src_scale), d = load_src<T>(src, step, sy0 + 1, sx0 + 1, src_scale);
      return __dmul_rn(__dadd_rn(__dadd_rn(__dadd_rn(a, b), c), d), 0.25);
    }
    double sum = 0.; int count = 0;
    for (int sy = 0; sy < 2 && sy0 + sy < rows; ++sy)
      for (int sx = 0; sx < 2 && sx0 + sx < cols; ++sx) { sum = __dadd_rn(sum, load_src<T>(src, step, sy0 + sy, sx0 + sx, src_scale)); ++count; }
    return (double)__fdiv_rn(__double2float_rn(sum), (float)count);
  }
  int sx, sy; float fx, fy;
  linear_axis(x, scale, cols, true, sx, fx);
  linear_axis(y, scale, rows, false, sy, fy);
  const int y0 = min(max(sy, 0), rows - 1), y1 = min(max(sy + 1, 0), rows - 1);
  double r0, r1;
  if (sx + 1 < cols) {
    const double a0 = (double)(1.f - fx), a1 = (double)fx;
    r0 = __dadd_rn(__dmul_rn(load_src<T>(src, step, y0, sx, src_scale), a0), __dmul_rn(load_src<T>(src, step, y0, sx + 1, src_scale), a1));
    r1 = __dadd_rn(__dmul_rn(load_src<T>(src, step, y1, sx, src_scale), a0), __dmul_rn(load_src<T>(src, step, y1, sx + 1, src_scale), a1));
  } else {
    r0 = load_src<T>(src, step, y0, sx, src_scale);
    r1 = load_src<T>(src, step, y1, sx, src_scale);
  }
  const double b0 = (double)(1.f - fy), b1 = (double)fy;
  return __dadd_rn(__dmul_rn(r0, b0), __dmul_rn(r1, b1));
}

// cv::Scharr (AN:181-187) of the 3x3 neighbourhood t (rows y-1, y, y+1; reflect-101 already applied) with the kernel
// scaled: ks0 = 3 s, ks1 = 10 s.  cv::Scharr's separable evaluation order.
__device__ __forceinline__ void scharr_taps(const double (&t)[3][3], double ks0, double ks1, double& gx, double& gy) {
  // dx: row filter [-1 0 1] on three rows, then column filter centre-first
  const double dm = __dsub_rn(t[0][2], t[0][0]);
  const double d0 = __dsub_rn(t[1][2], t[1][0]);
  const double dp = __dsub_rn(t[2][2], t[2][0]);
  gx = __dadd_rn(__dmul_rn(ks1, d0), __dmul_rn(ks0, __dadd_rn(dp, dm)));
  // dy: row filter [3 10 3]*scale left-to-right on rows y-1 and y+1, then column [-1 0 1]
  const double sm = __dadd_rn(__dadd_rn(__dmul_rn(ks0, t[0][0]), __dmul_rn(ks1, t[0][1])), __dmul_rn(ks0, t[0][2]));
  const double sp = __dadd_rn(__dadd_rn(__dmul_rn(ks0, t[2][0]), __dmul_rn(ks1, t[2][1])), __dmul_rn(ks0, t[2][2]));
  gy = __dsub_rn(sp, sm);
}

}  // namespace phovo
#endif
