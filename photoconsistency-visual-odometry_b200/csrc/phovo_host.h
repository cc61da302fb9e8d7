// phovo_host.h -- host-only helpers of phovo_api.cu and phovo_batch.cu: owners of device / pinned memory, streams and
// events (the only place that allocates or frees them), and the small functions both translation units need.
#ifndef PHOVO_HOST_H_
#define PHOVO_HOST_H_

#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <memory>
#include <string>
#include <utility>

#include "phovo_internal.h"
#include "phovo_kernels.h"

// return ctx->cuda_fail(...) from the enclosing function when `call` fails
#define CK(call)                                                      \
  do {                                                                \
    cudaError_t e_ = (call);                                          \
    if (e_ != cudaSuccess) return ctx->cuda_fail((std::string(__func__) + ": " #call).c_str(), e_); \
  } while (0)

namespace phovo {

// Storage for `capacity()` elements of T in device or pinned host memory that only grows.  It either owns its allocation
// or is a view of memory owned elsewhere (a slot context's buffers carved out of the batch state's arena): the
// destructor frees only what it owns.
template <class T, bool kPinned>
class Array {
 public:
  Array() = default;
  ~Array() { reset(); }
  Array(const Array&) = delete;
  Array& operator=(const Array&) = delete;

  // at least `n` elements; the capacity is recorded only once the allocation succeeded.  *fresh: the storage is new
  // (contents undefined) -- possibly at the address of the old one, so comparing pointers does not tell
  cudaError_t ensure(size_t n, bool* fresh = nullptr) {
    if (fresh) *fresh = false;
    if (p_ && cap_ >= n) return cudaSuccess;
    reset();
    void* p = nullptr;
    const cudaError_t e = kPinned ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
    if (e != cudaSuccess) return e;
    p_ = (T*)p; cap_ = n; owned_ = true;
    if (fresh) *fresh = true;
    return cudaSuccess;
  }
  void view(T* p, size_t n) { reset(); p_ = p; cap_ = n; }
  void reset() {
    if (owned_) kPinned ? cudaFreeHost(p_) : cudaFree(p_);
    p_ = nullptr; cap_ = 0; owned_ = false;
  }
  void swap(Array& o) { std::swap(p_, o.p_); std::swap(cap_, o.cap_); std::swap(owned_, o.owned_); }
  T* get() const { return p_; }
  size_t capacity() const { return cap_; }

 private:
  T* p_ = nullptr;
  size_t cap_ = 0;
  bool owned_ = false;
};
template <class T> using DeviceArray = Array<T, false>;
template <class T> using PinnedArray = Array<T, true>;

struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;

inline cudaError_t create_stream(Stream& s) {
  cudaStream_t h = nullptr;
  const cudaError_t e = cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking);
  if (e == cudaSuccess) s.reset(h);
  return e;
}
inline cudaError_t create_event(Event& ev, unsigned flags = cudaEventDefault) {
  cudaEvent_t h = nullptr;
  const cudaError_t e = cudaEventCreateWithFlags(&h, flags);
  if (e == cudaSuccess) ev.reset(h);
  return e;
}

// Two classifications of a caller's pointer that differ on managed memory, kept apart because each call site relies
// on its own answer: is_device_pointer counts managed memory as device memory (the kernels read it in place), and a
// pointer the runtime does not know as host memory.  host_readable counts managed memory, and a pointer the runtime
// does not know, as host memory (the host may read it, a cudaMemcpyDefault may copy it).
inline bool is_device_pointer(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}
inline bool host_readable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return a.type != cudaMemoryTypeDevice;
}

inline void level_size(int rows, int cols, int level, int* orows, int* ocols) {
  // cv::resize(img, Size(0,0), f, f): dsize = cvRound(ssize * f), f = 2^-level (AN:132,159)
  if (level == 0) { *orows = rows; *ocols = cols; return; }
  const double f = ldexp(1.0, -level);
  *orows = (int)lrint(rows * f);
  *ocols = (int)lrint(cols * f);
}

inline int src_type_of_depth(int depth_type) {
  switch (depth_type) {
    case PHOVO_DEPTH_F64: return SRC_F64;
    case PHOVO_DEPTH_F32: return SRC_F32;
    case PHOVO_DEPTH_U16: return SRC_U16;
  }
  return -1;
}
inline size_t depth_elt(int depth_type) { return depth_type == PHOVO_DEPTH_F64 ? 8 : depth_type == PHOVO_DEPTH_F32 ? 4 : 2; }

// The pinhole K / 2^level.  The reference writes it three ways: K / 2^level with 1. / fx in Ceres mode
// (CPhotoconsistencyOdometryCeres.h:163-168), K * (1 / 2^level) with 1.f / fx in the analytic modes
// (CPhotoconsistencyOdometryAnalytic.h:203-209) and K / 2^level with 1.f / fx in warpImage (BASE:89-94).  They agree
// bit for bit for normal K: scaling by a power of two is exact either way, and 1.f / double is a double division.
inline WarpIntrinsics scaled_intrinsics(const double K[9], int level) {
  const double p = pow(2, (double)level);
  WarpIntrinsics I;
  I.fx = K[0] / p; I.fy = K[4] / p; I.ox = K[2] / p; I.oy = K[5] / p;
  I.inv_fx = 1. / I.fx; I.inv_fy = 1. / I.fy;
  return I;
}

// LevelParams of pyramid level `level`, rows x cols at that level, under cfg and K; all of its rows
inline LevelParams make_level_params(const phovo_config& cfg, const double K[9], int level, int rows, int cols) {
  LevelParams L;
  memset(&L, 0, sizeof(L));
  const WarpIntrinsics I = scaled_intrinsics(K, level);
  L.fx = I.fx; L.fy = I.fy; L.ox = I.ox; L.oy = I.oy; L.inv_fx = I.inv_fx; L.inv_fy = I.inv_fy;
  L.min_depth = cfg.min_depth; L.max_depth = cfg.max_depth;
  L.lambda = cfg.lambda_step[level]; L.min_grad_norm = cfg.min_gradient_norm[level];
  L.rows = rows; L.cols = cols;
  L.max_iters = cfg.max_num_iterations[level];
  L.mode = cfg.mode; L.level = level;
  L.row_begin = 0; L.row_end = rows;
  return L;
}

}  // namespace phovo

#endif
