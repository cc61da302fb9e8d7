// phovo_api.cu -- context object and C ABI (include/phovo_b200.h) of the general path.
// The batch extension lives in phovo_batch.cu and shares the context through phovo_ctx.h.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "phovo_ctx.h"
#include "phovo_lm.h"

using namespace phovo;

static std::string g_create_error;

// ---------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------
int phovo_ctx::fail(int code, const std::string& what) {
  err = what;
  return code;
}
int phovo_ctx::cuda_fail(const char* what, cudaError_t e) {
  err = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  return PHOVO_E_CUDA;
}

bool phovo_ctx::level_active(int l) const {
  return l < cfg.num_levels && (build_all_levels || cfg.max_num_iterations[l] > 0);
}

LevelParams phovo_ctx::level_params(int level) const {
  LevelParams L = make_level_params(cfg, K, level, lrows[level], lcols[level]);
  if (shard_world > 1) {
    L.row_begin = (int)((long long)L.rows * shard_rank / shard_world);
    L.row_end = (int)((long long)L.rows * (shard_rank + 1) / shard_world);
  }
  return L;
}

LevelPtrs phovo_ctx::level_ptrs(int level) const {
  LevelPtrs P;
  P.I0 = I0[level].get(); P.D0 = D0[level].get(); P.I1 = I1[level].get(); P.Gx = Gx[level].get(); P.Gy = Gy[level].get();
  P.winner = winner.get();
  P.valid = valid.get();
  P.D1 = D1[level].get(); P.GxD = GxD[level].get(); P.GyD = GyD[level].get(); P.gain = d_gain.get() ? d_gain.get() + level : nullptr;
  return P;
}

// slots take views of their arena (bump pointer; arena_reset starts over), everything else allocates; *fresh as in
// Array::ensure
template <class T>
static cudaError_t ctx_ensure(phovo_ctx* ctx, DeviceArray<T>& a, size_t want, bool* fresh = nullptr) {
  if (!ctx->arena_base) return a.ensure(want, fresh);
  if (fresh) *fresh = false;
  if (a.capacity() >= want && a.get()) return cudaSuccess;
  const size_t off = (ctx->arena_used + 255) & ~(size_t)255, bytes = want * sizeof(T);
  if (off + bytes > ctx->arena_bytes) return cudaErrorMemoryAllocation;
  a.view((T*)(ctx->arena_base + off), want);
  if (fresh) *fresh = true;
  ctx->arena_used = off + bytes;
  return cudaSuccess;
}

void phovo_ctx::arena_reset(char* base, size_t bytes) {
  for (int l = 0; l < PHOVO_MAX_LEVELS; ++l) {
    I0[l].reset(); D0[l].reset(); I1[l].reset(); Gx[l].reset(); Gy[l].reset();
    D1[l].reset(); GxD[l].reset(); GyD[l].reset();
  }
  winner.reset(); valid.reset(); scratch64[0].reset(); scratch64[1].reset(); partials.reset();
  d_gain.reset(); d_pose.reset();
  have_src = have_tgt = have_tgt_depth = false;
  rows = cols = 0;
  arena_base = base; arena_bytes = bytes; arena_used = 0;
  if (base) {
    d_pose.view((PoseDev*)base, 1);
    d_gain.view((double*)(base + 256), PHOVO_MAX_LEVELS);
    arena_used = 512;
    static_assert(sizeof(PoseDev) <= 256 && sizeof(double) * PHOVO_MAX_LEVELS <= 256, "slot header layout");
  }
}

size_t phovo_internal_slot_bytes(const phovo_ctx* ctx, int rows, int cols) {
  size_t total = 512, max_px = 1;
  auto add = [&](size_t bytes) { total = ((total + 255) & ~(size_t)255) + bytes; };
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (!ctx->level_active(l)) continue;
    int r, c;
    level_size(rows, cols, l, &r, &c);
    const size_t n = (size_t)(r > 0 ? r : 1) * (c > 0 ? c : 1);
    if (n > max_px) max_px = n;
    for (int a = 0; a < 8; ++a) add(n * sizeof(double));      // I0 D0 I1 Gx Gy (+ D1 GxD GyD)
  }
  add(2 * max_px * sizeof(int)); add(max_px);                 // winner (2N slots), valid
  add(max_px * sizeof(double)); add(max_px * sizeof(double)); // scratch
  add((size_t)partials_blocks(ctx->sm_count) * PHOVO_ACC_STRIDE * sizeof(double));
  return (total + 4095) & ~(size_t)4095;
}

void phovo_ctx::invalidate_graph() {
  if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
  if (graph) { cudaGraphDestroy(graph); graph = nullptr; }
}

// (re)allocate per-level storage for a rows x cols frame under the current config
static int prepare_levels(phovo_ctx* ctx, int rows, int cols) {
  if (rows <= 0 || cols <= 0) return ctx->fail(PHOVO_E_INVALID, "frame size must be positive");
  if (ctx->cfg.num_levels < 1 || ctx->cfg.num_levels > PHOVO_MAX_LEVELS) return ctx->fail(PHOVO_E_INVALID, "num_levels out of range");
  bool changed = rows != ctx->rows || cols != ctx->cols;
  ctx->rows = rows; ctx->cols = cols;
  size_t max_px = 0;
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    level_size(rows, cols, l, &ctx->lrows[l], &ctx->lcols[l]);
    if (ctx->lrows[l] < 1 || ctx->lcols[l] < 1) return ctx->fail(PHOVO_E_INVALID, "image too small for the number of pyramid levels");
    if (!ctx->level_active(l)) continue;
    const size_t n = (size_t)ctx->lrows[l] * ctx->lcols[l];
    if (n > max_px) max_px = n;
    DeviceArray<double>* arrs[5] = {&ctx->I0[l], &ctx->D0[l], &ctx->I1[l], &ctx->Gx[l], &ctx->Gy[l]};
    for (int a = 0; a < 5; ++a) {
      bool fresh;
      CK(ctx_ensure(ctx, *arrs[a], n, &fresh));
      changed |= fresh;
    }
  }
  if (max_px == 0) max_px = 1;
  // new storage <=> refill with -1.  NOT "the pointer changed": cudaFree + cudaMalloc may hand the same address back
  // with a larger extent, whose tail is garbage -- winner indices nobody wrote (found by the randomised sweep on a
  // pool of 8 contexts: illegal addresses in phase B after a frame-size change)
  bool fresh;
  CK(ctx_ensure(ctx, ctx->winner, 2 * max_px, &fresh));   // the photometric + depth solver stacks 2N rows
  if (fresh) {
    changed = true;
    launch_fill_i32(ctx->stream, ctx->winner.get(), -1, ctx->winner.capacity(), ctx->sm_count);
    ctx->launches += 1;
  }
  CK(ctx_ensure(ctx, ctx->valid, max_px, &fresh));
  changed |= fresh;
  for (int s = 0; s < 2; ++s) CK(ctx_ensure(ctx, ctx->scratch64[s], max_px));
  CK(ctx_ensure(ctx, ctx->partials, (size_t)partials_blocks(ctx->sm_count) * PHOVO_ACC_STRIDE, &fresh));
  changed |= fresh;
  if (changed) ctx->invalidate_graph();
  return PHOVO_OK;
}

// copy a strided host/device image into a dense device staging buffer (or use it in place)
static int stage_image(phovo_ctx* ctx, const void* src, size_t step, size_t elt, int rows, int cols,
                       DeviceArray<char>& stage, const void** dev_out, size_t* dev_step) {
  if (is_device_pointer(src)) {
    // used in place; the kernels that read it are drained before the call returns (wait_uploads), so the
    // caller may overwrite or free the buffer afterwards, exactly as with a host buffer.  Ordering
    // BEFORE the call is the caller's: the data must be complete on the context's stream
    // (phovo_set_stream(producer stream)) or the producer stream must have been synchronised.
    *dev_out = src; *dev_step = step;
    ctx->device_input_in_flight = true;
    return PHOVO_OK;
  }
  const size_t bytes = (size_t)rows * cols * elt;
  CK(stage.ensure(bytes));
  CK(cudaMemcpy2DAsync(stage.get(), (size_t)cols * elt, src, step, (size_t)cols * elt, rows, cudaMemcpyHostToDevice, ctx->stream));
  *dev_out = stage.get(); *dev_step = (size_t)cols * elt;
  ctx->h2d_pending = true;
  return PHOVO_OK;
}

static int finish_uploads(phovo_ctx* ctx) {
  // inputs are borrowed for the duration of the call only: wait for the copies (not the kernels)
  if (ctx->h2d_pending) {
    CK(cudaEventRecord(ctx->ev_copy.get(), ctx->stream));
    ctx->h2d_pending = false;
    ctx->copy_event_armed = true;
  }
  return PHOVO_OK;
}

static int wait_uploads(phovo_ctx* ctx) {
  if (ctx->device_input_in_flight) {   // kernels are still reading the caller's device buffer: drain them
    ctx->device_input_in_flight = false;
    ctx->copy_event_armed = false;
    if (!ctx->defer_device_input_drain) CK(cudaStreamSynchronize(ctx->stream));
    return PHOVO_OK;
  }
  if (ctx->copy_event_armed) { CK(cudaEventSynchronize(ctx->ev_copy.get())); ctx->copy_event_armed = false; }
  return PHOVO_OK;
}

// the active levels of the current size as a PyramidLevels block; false if one of them is blurred
// (the fused kernel has no blur stage) or if the frame is big: one launch for all levels wins while
// launch latency dominates (640x480: set-up 0.18 -> 0.10 ms); on an 8K frame the per-level launches
// with 2-D tiles and the shared-memory Scharr are faster (0.58 vs 0.77-0.92 ms)
static bool fused_levels(const phovo_ctx* ctx, PyramidLevels* P) {
  memset(P, 0, sizeof(*P));
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (!ctx->level_active(l)) continue;
    if (ctx->cfg.blur_filter_size[l] > 1) return false;
    const int a = P->num++;
    P->level[a] = l; P->orows[a] = ctx->lrows[l]; P->ocols[a] = ctx->lcols[l];
    P->px_offset[a + 1] = P->px_offset[a] + ctx->lrows[l] * ctx->lcols[l];
    const double s = ctx->cfg.grad_scale[l];
    P->ks0[a] = s != 1. ? 3. * s : 3.; P->ks1[a] = s != 1. ? 10. * s : 10.;   // launch_scharr_store's kernel
  }
  return P->px_offset[P->num] <= (1 << 20);
}

// intensity pyramid (+ gradients for the target) of one frame; AN:471-474 / AN:484-490
static int build_intensity(phovo_ctx* ctx, const void* dev_gray, size_t step, bool target) {
  PyramidLevels P;
  if (fused_levels(ctx, &P)) {
    for (int a = 0; a < P.num; ++a) {
      const int l = P.level[a];
      P.dst[a] = target ? ctx->I1[l].get() : ctx->I0[l].get();
      P.gx[a] = target ? ctx->Gx[l].get() : nullptr; P.gy[a] = target ? ctx->Gy[l].get() : nullptr;
    }
    ctx->launches += launch_build_levels(ctx->stream, dev_gray, SRC_U8, step, 1. / 255, ctx->rows, ctx->cols, P, target);
    CK(cudaGetLastError());
    return PHOVO_OK;
  }
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (!ctx->level_active(l)) continue;
    const int r = ctx->lrows[l], c = ctx->lcols[l];
    double* img = target ? ctx->I1[l].get() : ctx->I0[l].get();
    ctx->launches += launch_build_level(ctx->stream, dev_gray, SRC_U8, step, 1. / 255, ctx->rows, ctx->cols, l, img, r, c);
    const int k = ctx->cfg.blur_filter_size[l];
    if (k > 1) {  // AN:144-148: GaussianBlur(k, sigma 3) twice
      ctx->launches += launch_gaussian_blur(ctx->stream, img, ctx->scratch64[0].get(), r, c, k, 3.);
      ctx->launches += launch_gaussian_blur(ctx->stream, img, ctx->scratch64[0].get(), r, c, k, 3.);
    }
    if (target) ctx->launches += launch_scharr_store(ctx->stream, img, r, c, ctx->cfg.grad_scale[l], ctx->Gx[l].get(), ctx->Gy[l].get());
  }
  CK(cudaGetLastError());
  return PHOVO_OK;
}

static int build_depth(phovo_ctx* ctx, const void* dev_depth, int depth_type, size_t step, double depth_scale) {
  PyramidLevels P;   // the depth pyramid is never blurred (AN:471-476)
  memset(&P, 0, sizeof(P));
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (!ctx->level_active(l)) continue;
    const int a = P.num++;
    P.level[a] = l; P.orows[a] = ctx->lrows[l]; P.ocols[a] = ctx->lcols[l];
    P.px_offset[a + 1] = P.px_offset[a] + ctx->lrows[l] * ctx->lcols[l];
    P.dst[a] = ctx->D0[l].get();
  }
  if (P.px_offset[P.num] <= (1 << 20)) {   // small frame: every active level in one launch (see fused_levels)
    ctx->launches += launch_build_levels(ctx->stream, dev_depth, src_type_of_depth(depth_type), step, depth_scale, ctx->rows, ctx->cols, P, false);
  } else {
    for (int a = 0; a < P.num; ++a)
      ctx->launches += launch_build_level(ctx->stream, dev_depth, src_type_of_depth(depth_type), step, depth_scale, ctx->rows, ctx->cols,
                                          P.level[a], P.dst[a], P.orows[a], P.ocols[a]);
  }
  CK(cudaGetLastError());
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// life cycle
// ---------------------------------------------------------------------------------------------
extern "C" const char* phovo_version(void) { return "phovo-b200 0.1 (sm_100a)"; }

extern "C" const char* phovo_last_error(const phovo_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

static int create_context(int device, phovo_ctx** out, bool slot) {
  if (!out) return PHOVO_E_INVALID;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) + "); this library has no CPU path";
    cudaGetLastError();
    return PHOVO_E_CUDA;
  }
  if (device < 0 || device >= ndev) { g_create_error = "device index out of range"; return PHOVO_E_INVALID; }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) { g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e); return PHOVO_E_CUDA; }
  phovo_ctx* ctx = new phovo_ctx();   // on failure, `delete ctx` frees whatever was made so far
  ctx->device = device;
  {
    cudaDeviceProp prop;
    memset(&prop, 0, sizeof(prop));
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { cudaGetLastError(); prop.multiProcessorCount = 0; prop.cooperativeLaunch = 0; }
    ctx->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 1;
    if (!prop.cooperativeLaunch) ctx->failed_paths |= 1u << 2;
  }
  phovo_internal_default_config(&ctx->cfg);
  auto bail = [&](const char* what, cudaError_t err) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
    delete ctx;
    return PHOVO_E_CUDA;
  };
  ctx->is_slot = slot;
  if (!slot) {
    if ((e = create_stream(ctx->own_stream)) != cudaSuccess) return bail("cudaStreamCreate", e);
    ctx->stream = ctx->own_stream.get();
  }
  if ((e = create_event(ctx->ev_copy)) != cudaSuccess) return bail("cudaEventCreate", e);
  for (int i = 0; i < 4; ++i)
    if ((e = create_event(ctx->ev_time[i])) != cudaSuccess) return bail("cudaEventCreate", e);
  if (slot) { *out = ctx; return PHOVO_OK; }   // device buffers come from the arena, results are gathered by the batch state
  if ((e = ctx->d_pose.ensure(1)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMemset(ctx->d_pose.get(), 0, sizeof(PoseDev))) != cudaSuccess) return bail("cudaMemset", e);
  if ((e = ctx->d_log.ensure(1024)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = ctx->d_state_in.ensure(6)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = ctx->d_shard.ensure(32)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = ctx->d_eval.ensure(1)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = ctx->h_pose.ensure(1)) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = ctx->h_log.ensure(1024)) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = ctx->h_state_in.ensure(8)) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = ctx->h_eval.ensure(1)) != cudaSuccess) return bail("cudaMallocHost", e);
  memset(ctx->h_pose.get(), 0, sizeof(PoseDev));
  *out = ctx;
  return PHOVO_OK;
}

extern "C" int phovo_create(int device, phovo_ctx** out) { return create_context(device, out, false); }
int phovo_internal_create_slot(int device, phovo_ctx** out) { return create_context(device, out, true); }

extern "C" int phovo_destroy(phovo_ctx* ctx) {
  if (!ctx) return PHOVO_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream || !ctx->is_slot) cudaStreamSynchronize(ctx->stream);
  if (ctx->arena_base) ctx->arena_reset(nullptr, 0);   // arena-backed buffers belong to the batch state
  ctx->invalidate_graph();
  phovo_batch_release(ctx);
  for (int r = 0; r < 8; ++r)   // peers' areas are mappings, not allocations of this context
    if (ctx->xchg_opened[r]) cudaIpcCloseMemHandle(ctx->xchg_peer[r]);
  delete ctx;
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// configuration
// ---------------------------------------------------------------------------------------------
extern "C" int phovo_config_default(phovo_config* cfg) {
  if (!cfg) return PHOVO_E_INVALID;
  phovo_internal_default_config(cfg);
  return PHOVO_OK;
}

static int validate_config(phovo_ctx* ctx, const phovo_config* cfg) {
  if (cfg->num_levels < 1 || cfg->num_levels > PHOVO_MAX_LEVELS) return ctx->fail(PHOVO_E_INVALID, "num_levels must be in [1, PHOVO_MAX_LEVELS]");
  if (cfg->mode < 0 || cfg->mode > 3) return ctx->fail(PHOVO_E_INVALID, "unknown mode");
  long total = 0;
  for (int l = 0; l < cfg->num_levels; ++l) {
    const int k = cfg->blur_filter_size[l];
    if (k < 0 || k > 31 || (k > 0 && k % 2 == 0)) return ctx->fail(PHOVO_E_INVALID, "blur_filter_size must be 0 or odd and <= 31");
    if (cfg->max_num_iterations[l] < 0) return ctx->fail(PHOVO_E_INVALID, "max_num_iterations must be >= 0");
    total += cfg->max_num_iterations[l];
  }
  if (total > 1000000) return ctx->fail(PHOVO_E_INVALID, "sum of max_num_iterations too large");
  return PHOVO_OK;
}

extern "C" int phovo_set_config(phovo_ctx* ctx, const phovo_config* cfg) {
  if (!ctx || !cfg) return PHOVO_E_INVALID;
  int rc = validate_config(ctx, cfg);
  if (rc) return rc;
  ctx->cfg = *cfg;
  for (int l = cfg->num_levels; l < PHOVO_MAX_LEVELS; ++l) ctx->cfg.max_num_iterations[l] = 0;
  ctx->have_src = ctx->have_tgt = false;  // pyramids depend on the config (AN:474: m_NumOptimizationLevels)
  ctx->level_dmin_valid = false;
  ctx->invalidate_graph();
  return PHOVO_OK;
}

extern "C" int phovo_get_config(const phovo_ctx* ctx, phovo_config* cfg) {
  if (!ctx || !cfg) return PHOVO_E_INVALID;
  *cfg = ctx->cfg;
  return PHOVO_OK;
}

extern "C" int phovo_parse_config_yaml(const char* path, phovo_config* cfg, char* err, size_t err_len) {
  if (!path || !cfg) return PHOVO_E_INVALID;
  std::string e;
  int rc = phovo_internal_parse_yaml(path, cfg, &e);
  if (rc && err && err_len) { strncpy(err, e.c_str(), err_len - 1); err[err_len - 1] = 0; }
  return rc;
}

extern "C" int phovo_load_config_yaml(phovo_ctx* ctx, const char* path) {
  if (!ctx || !path) return PHOVO_E_INVALID;
  phovo_config cfg = ctx->cfg;
  std::string e;
  int rc = phovo_internal_parse_yaml(path, &cfg, &e);
  if (rc) return ctx->fail(rc, e);
  return phovo_set_config(ctx, &cfg);
}

extern "C" int phovo_set_mode(phovo_ctx* ctx, int mode) {
  if (!ctx || mode < 0 || mode > 3) return PHOVO_E_INVALID;
  if (ctx->cfg.mode != mode) {
    ctx->cfg.mode = mode;
    ctx->invalidate_graph();
  }
  return PHOVO_OK;
}

extern "C" int phovo_set_depth_range(phovo_ctx* ctx, double min_depth, double max_depth) {
  if (!ctx) return PHOVO_E_INVALID;
  ctx->cfg.min_depth = min_depth; ctx->cfg.max_depth = max_depth;
  ctx->level_dmin_valid = false;     // the smallest VALID depth of a level depends on the range
  ctx->invalidate_graph();
  return PHOVO_OK;
}

extern "C" int phovo_set_intrinsics(phovo_ctx* ctx, const double K[9]) {
  if (!ctx || !K) return PHOVO_E_INVALID;
  if (memcmp(ctx->K, K, sizeof(double) * 9) != 0) ctx->invalidate_graph();
  memcpy(ctx->K, K, sizeof(double) * 9);
  ctx->have_K = true;
  return PHOVO_OK;
}

extern "C" int phovo_set_build_all_levels(phovo_ctx* ctx, int enable) {
  if (!ctx) return PHOVO_E_INVALID;
  ctx->build_all_levels = enable != 0;
  ctx->have_src = ctx->have_tgt = false;
  return PHOVO_OK;
}

extern "C" int phovo_set_stream(phovo_ctx* ctx, void* cuda_stream) {
  if (!ctx) return PHOVO_E_INVALID;
  cudaStreamSynchronize(ctx->stream);
  ctx->own_stream.reset();
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->invalidate_graph();
  return PHOVO_OK;
}

extern "C" int phovo_set_use_graph(phovo_ctx* ctx, int enable) {
  if (!ctx) return PHOVO_E_INVALID;
  ctx->execution = enable ? 1 : 0;
  return PHOVO_OK;
}

extern "C" int phovo_set_execution(phovo_ctx* ctx, int path) {
  if (!ctx || path < 0 || path > 3) return PHOVO_E_INVALID;
  ctx->execution = path;
  return PHOVO_OK;
}

extern "C" int phovo_last_optimize_path(const phovo_ctx* ctx) { return ctx ? ctx->last_path : -1; }

// ---------------------------------------------------------------------------------------------
// frames
// ---------------------------------------------------------------------------------------------
extern "C" int phovo_set_source(phovo_ctx* ctx, const uint8_t* gray, size_t gray_step, const void* depth,
                                int depth_type, size_t depth_step, double depth_scale, int rows, int cols) {
  if (!ctx || !gray || !depth) return PHOVO_E_INVALID;
  if (src_type_of_depth(depth_type) < 0) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if (gray_step < (size_t)cols || depth_step < (size_t)cols * depth_elt(depth_type)) return ctx->fail(PHOVO_E_INVALID, "row stride smaller than a row");
  CK(cudaSetDevice(ctx->device));
  int rc = prepare_levels(ctx, rows, cols);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev_time[0].get(), ctx->stream));
  const void* dg; size_t dgs; const void* dd; size_t dds;
  if ((rc = stage_image(ctx, gray, gray_step, 1, rows, cols, ctx->stage_gray[0], &dg, &dgs))) return rc;
  if ((rc = stage_image(ctx, depth, depth_step, depth_elt(depth_type), rows, cols, ctx->stage_depth, &dd, &dds))) return rc;
  if ((rc = finish_uploads(ctx))) return rc;
  if ((rc = build_intensity(ctx, dg, dgs, false))) return rc;
  if ((rc = build_depth(ctx, dd, depth_type, dds, depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0))) return rc;
  CK(cudaEventRecord(ctx->ev_time[1].get(), ctx->stream));
  ctx->have_src = true;
  ctx->setup_timed = true;
  ctx->level_dmin_valid = false;
  return wait_uploads(ctx);
}

extern "C" int phovo_set_target(phovo_ctx* ctx, const uint8_t* gray, size_t gray_step, int rows, int cols) {
  if (!ctx || !gray) return PHOVO_E_INVALID;
  if (gray_step < (size_t)cols) return ctx->fail(PHOVO_E_INVALID, "row stride smaller than a row");
  // the reference reads the Scharr ddepth from m_IntensityPyramid0[0] (AN:171): source first
  if (!ctx->have_src) return ctx->fail(PHOVO_E_INVALID, "SetSourceFrame must be called before SetTargetFrame");
  if (rows != ctx->rows || cols != ctx->cols) return ctx->fail(PHOVO_E_INVALID, "target frame size differs from the source frame");
  CK(cudaSetDevice(ctx->device));
  const void* dg; size_t dgs;
  int rc;
  if (!ctx->setup_timed) CK(cudaEventRecord(ctx->ev_time[0].get(), ctx->stream));
  if ((rc = stage_image(ctx, gray, gray_step, 1, rows, cols, ctx->stage_gray[1], &dg, &dgs))) return rc;
  if ((rc = finish_uploads(ctx))) return rc;
  if ((rc = build_intensity(ctx, dg, dgs, true))) return rc;
  CK(cudaEventRecord(ctx->ev_time[1].get(), ctx->stream));
  ctx->have_tgt = true;
  ctx->have_tgt_depth = false;
  return wait_uploads(ctx);
}

extern "C" int phovo_set_target_depth(phovo_ctx* ctx, const void* depth, int depth_type, size_t depth_step, double depth_scale) {
  if (!ctx || !depth) return PHOVO_E_INVALID;
  if (!ctx->have_tgt) return ctx->fail(PHOVO_E_INVALID, "SetTargetFrame must be called before the target depth is set");
  if (src_type_of_depth(depth_type) < 0) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if (depth_step < (size_t)ctx->cols * depth_elt(depth_type)) return ctx->fail(PHOVO_E_INVALID, "row stride smaller than a row");
  CK(cudaSetDevice(ctx->device));
  CK(ctx->d_gain.ensure(PHOVO_MAX_LEVELS));   // (a slot's is a view of its arena)
  const void* dd; size_t dds; int rc;
  if ((rc = stage_image(ctx, depth, depth_step, depth_elt(depth_type), ctx->rows, ctx->cols, ctx->stage_depth, &dd, &dds))) return rc;
  if ((rc = finish_uploads(ctx))) return rc;
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (!ctx->level_active(l)) continue;
    const int r = ctx->lrows[l], c = ctx->lcols[l];
    const size_t n = (size_t)r * c;
    DeviceArray<double>* arrs[3] = {&ctx->D1[l], &ctx->GxD[l], &ctx->GyD[l]};
    for (int a = 0; a < 3; ++a) {
      bool fresh;
      CK(ctx_ensure(ctx, *arrs[a], n, &fresh));
      if (fresh) ctx->invalidate_graph();
    }
    // BiObjective.h:574 (depth pyramid, no blur), :224-237 (Scharr of depth / m_MaxDepth), :299 (gain)
    ctx->launches += launch_build_level(ctx->stream, dd, src_type_of_depth(depth_type), dds, depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0,
                                        ctx->rows, ctx->cols, l, ctx->D1[l].get(), r, c);
    ctx->launches += launch_scale(ctx->stream, ctx->D1[l].get(), 1. / ctx->cfg.max_depth, ctx->scratch64[0].get(), n);
    ctx->launches += launch_scharr_store(ctx->stream, ctx->scratch64[0].get(), r, c, ctx->cfg.grad_scale[l], ctx->GxD[l].get(), ctx->GyD[l].get());
    ctx->launches += launch_mean_ratio(ctx->stream, ctx->I1[l].get(), ctx->D1[l].get(), n, ctx->d_gain.get() + l);
  }
  CK(cudaGetLastError());
  ctx->have_tgt_depth = true;
  return wait_uploads(ctx);
}

extern "C" int phovo_promote_target_to_source(phovo_ctx* ctx, const void* depth, int depth_type, size_t depth_step, double depth_scale) {
  if (!ctx || !depth) return PHOVO_E_INVALID;
  if (!ctx->have_tgt) return ctx->fail(PHOVO_E_INVALID, "no target frame to promote");
  if (src_type_of_depth(depth_type) < 0) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  CK(cudaSetDevice(ctx->device));
  // the I1 pyramid of frame k is bit-identical to the I0 pyramid of frame k as a source
  // (same convert + resize + blur, AN:471-474 vs AN:484-487): swap the level buffers.
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (!ctx->level_active(l)) continue;
    ctx->I0[l].swap(ctx->I1[l]);
  }
  ctx->invalidate_graph();
  CK(cudaEventRecord(ctx->ev_time[0].get(), ctx->stream));
  const void* dd; size_t dds; int rc;
  if ((rc = stage_image(ctx, depth, depth_step, depth_elt(depth_type), ctx->rows, ctx->cols, ctx->stage_depth, &dd, &dds))) return rc;
  if ((rc = finish_uploads(ctx))) return rc;
  if ((rc = build_depth(ctx, dd, depth_type, dds, depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0))) return rc;
  ctx->have_src = true; ctx->have_tgt = false; ctx->setup_timed = true;
  ctx->level_dmin_valid = false;
  return wait_uploads(ctx);
}

// ---------------------------------------------------------------------------------------------
// solve
// ---------------------------------------------------------------------------------------------
extern "C" int phovo_set_initial_state(phovo_ctx* ctx, const double state[6]) {
  if (!ctx || !state) return PHOVO_E_INVALID;
  memcpy(ctx->state, state, sizeof(double) * 6);
  return PHOVO_OK;
}

static int ready_to_solve(phovo_ctx* ctx) {
  if (!ctx->have_K) return ctx->fail(PHOVO_E_INVALID, "SetIntrinsicMatrix has not been called");
  if (!ctx->have_src || !ctx->have_tgt) return ctx->fail(PHOVO_E_INVALID, "source and target frames must be set before Optimize");
  if (ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE && !ctx->have_tgt_depth)
    return ctx->fail(PHOVO_E_INVALID, "the photometric + depth solver needs the target depth (phovo_set_target_depth)");
  return PHOVO_OK;
}

static int total_iterations(const phovo_ctx* ctx) {
  int t = 0;
  for (int l = 0; l < ctx->cfg.num_levels; ++l) t += ctx->cfg.max_num_iterations[l];
  return t;
}

static int ensure_log(phovo_ctx* ctx, int want) {
  if (want <= ctx->log_cap()) return PHOVO_OK;
  ctx->invalidate_graph();   // it writes to d_log
  CK(ctx->d_log.ensure(want));
  CK(ctx->h_log.ensure(want));
  return PHOVO_OK;
}

// The start of every solve: the inputs are complete, the log has room for a whole run, the optimize timer starts.  The
// initial state is uploaded by the driver (upload_state), because the graph driver captures its own upload.
static int begin_solve(phovo_ctx* ctx) {
  int rc = ready_to_solve(ctx);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  if ((rc = ensure_log(ctx, total_iterations(ctx) + 1))) return rc;
  ctx->setup_timed = false;
  CK(cudaEventRecord(ctx->ev_time[2].get(), ctx->stream));
  return PHOVO_OK;
}

static void upload_state(phovo_ctx* ctx) {
  ctx->launches += launch_set_state(ctx->stream, ctx->d_pose.get(), nullptr, ctx->state, ctx->log_cap());
}

static int read_back(phovo_ctx* ctx) {
  const int cap = total_iterations(ctx);
  CK(cudaMemcpyAsync(ctx->h_pose.get(), ctx->d_pose.get(), sizeof(PoseDev), cudaMemcpyDeviceToHost, ctx->stream));
  if (cap > 0) CK(cudaMemcpyAsync(ctx->h_log.get(), ctx->d_log.get(), sizeof(phovo_iter_stats) * (size_t)std::min(cap, ctx->log_cap()), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaEventRecord(ctx->ev_time[3].get(), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  memcpy(ctx->state, ctx->h_pose.get()->state, sizeof(double) * 6);
  int n = ctx->h_pose.get()->log_count;
  if (n > cap) n = cap;
  ctx->log.assign(ctx->h_log.get(), ctx->h_log.get() + n);
  for (int k = 0; k < 6; ++k)
    if (!isfinite(ctx->state[k])) return ctx->fail(PHOVO_E_NUMERIC, "non-finite state after Optimize (singular normal equations?)");
  return PHOVO_OK;
}

// The end of a row-sharded solve: the read-back, then whether a wait for a peer timed out.
static int end_solve(phovo_ctx* ctx) {
  const int rc = read_back(ctx);
  if (ctx->xchg_own.get()) {
    int err = 0;
    CK(cudaMemcpy(&err, &ctx->xchg_own.get()->error, sizeof(int), cudaMemcpyDeviceToHost));
    if (err) return ctx->fail(PHOVO_E_CUDA, "peer exchange timed out waiting for another rank");
  }
  return rc;
}

// What a driver returns when its path cannot run on this context: positive, so never a PHOVO_* code.  phovo_optimize
// then starts the solve over on the next path down.
static const int kPathUnavailable = 1;

static bool path_failed(const phovo_ctx* ctx, int path) { return (ctx->failed_paths >> path) & 1u; }

// A launch of `path` was refused: clears the launch error, keeps the reason for phovo_graph_error, marks the path so that
// no later Optimize() on this context tries it, and drains the stream.
static int path_unavailable(phovo_ctx* ctx, int path, const char* launch, cudaError_t e) {
  cudaGetLastError();
  ctx->path_note = std::string(launch) + " unavailable: " + cudaGetErrorString(e);
  ctx->failed_paths |= 1u << path;
  CK(cudaStreamSynchronize(ctx->stream));
  return kPathUnavailable;
}

// Plain stream launches; the host polls the device-side termination flag every `poll` iterations.
static int optimize_stream(phovo_ctx* ctx) {
  upload_state(ctx);
  const int poll = 4;
  return for_each_level(ctx->cfg, [&](int level, int M) {
    const LevelParams L = ctx->level_params(level);
    const LevelPtrs P = ctx->level_ptrs(level);
    ctx->launches += launch_begin_level(ctx->stream, ctx->d_pose.get(), M);
    for (int it = 0; it < M;) {
      int chunk = M - it < poll ? M - it : poll;
      for (int k = 0; k < chunk; ++k) {
        int grid = 0;
        ctx->launches += launch_iteration_kernels(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->sm_count, &grid, nullptr, nullptr, false);
        ctx->launches += launch_reduce_solve(ctx->stream, L, ctx->d_pose.get(), ctx->partials.get(), grid, ctx->d_log.get(), 0ull);
      }
      it += chunk;
      if (it < M) {
        CK(cudaMemcpyAsync(&ctx->h_pose.get()->done, &ctx->d_pose.get()->done, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (ctx->h_pose.get()->done) break;
      }
    }
    return PHOVO_OK;
  });
}

// One CUDA graph for the whole Optimize(): set-state -> for each active level { begin-level ->
// WHILE(handle) { K3a, K3b, K4 (sets handle = !done) } }.  No host involvement between the
// first kernel and the final read-back.
static int build_graph(phovo_ctx* ctx) {
  ctx->invalidate_graph();
  cudaGraph_t g = nullptr;
  CK(cudaGraphCreate(&g, 0));
  ctx->graph = g;
  cudaGraphNode_t tail = nullptr;
  bool have_tail = false;
  int launches_per_run = 0;

  auto capture = [&](cudaGraph_t target, bool chain, auto&& fn) -> cudaError_t {
    cudaError_t e = cudaStreamBeginCaptureToGraph(ctx->stream, target, (chain && have_tail) ? &tail : nullptr, nullptr,
                                                  (chain && have_tail) ? 1 : 0, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) return e;
    fn();
    cudaStreamCaptureStatus st; const cudaGraphNode_t* deps = nullptr; size_t ndeps = 0;
    e = cudaStreamGetCaptureInfo(ctx->stream, &st, nullptr, nullptr, &deps, &ndeps);
    cudaGraphNode_t last = (e == cudaSuccess && ndeps > 0) ? deps[ndeps - 1] : nullptr;
    cudaGraph_t out = nullptr;
    cudaError_t e2 = cudaStreamEndCapture(ctx->stream, &out);
    if (e != cudaSuccess) return e;
    if (e2 != cudaSuccess) return e2;
    if (chain && last) { tail = last; have_tail = true; }
    return cudaSuccess;
  };

  CK(capture(g, true, [&] { launches_per_run += launch_set_state(ctx->stream, ctx->d_pose.get(), ctx->d_state_in.get(), ctx->state, ctx->log_cap()); }));
  const int rc = for_each_level(ctx->cfg, [&](int level, int M) {
    const LevelParams L = ctx->level_params(level);
    const LevelPtrs P = ctx->level_ptrs(level);
    CK(capture(g, true, [&] { launches_per_run += launch_begin_level(ctx->stream, ctx->d_pose.get(), M); }));
    cudaGraphConditionalHandle handle;
    CK(cudaGraphConditionalHandleCreate(&handle, g, 1, cudaGraphCondAssignDefault));
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = handle;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t cond_node;
    CK(cudaGraphAddNode(&cond_node, g, have_tail ? &tail : nullptr, have_tail ? 1 : 0, &np));
    cudaGraph_t body = np.conditional.phGraph_out[0];
    int per_iter = 0;
    CK(capture(body, false, [&] {
      int grid = 0;
      per_iter += launch_iteration_kernels(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->sm_count, &grid, nullptr, nullptr, false);
      per_iter += launch_reduce_solve(ctx->stream, L, ctx->d_pose.get(), ctx->partials.get(), grid, ctx->d_log.get(), (unsigned long long)handle);
    }));
    ctx->graph_launches_per_iter = per_iter;
    tail = cond_node; have_tail = true;
    return PHOVO_OK;
  });
  if (rc) return rc;
  ctx->graph_launches_fixed = launches_per_run;
  CK(cudaGraphInstantiate(&ctx->graph_exec, g, 0));
  return PHOVO_OK;
}

static int run_graph(phovo_ctx* ctx) {
  if (!ctx->graph_exec) {
    int rc = build_graph(ctx);
    if (rc) return rc;
  }
  memcpy(ctx->h_state_in.get(), ctx->state, sizeof(double) * 6);
  CK(cudaMemcpyAsync(ctx->d_state_in.get(), ctx->h_state_in.get(), sizeof(double) * 6, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaGraphLaunch(ctx->graph_exec, ctx->stream));
  return read_back(ctx);
}

// The graph driver reads back itself: when building, launching or running the graph fails, the context stops using
// graphs and the solve starts over on plain launches.
static int optimize_graph(phovo_ctx* ctx) {
  const int rc = run_graph(ctx);
  if (rc == PHOVO_OK || rc == PHOVO_E_NUMERIC) {
    int iters = 0;
    for (int l = 0; l < ctx->cfg.num_levels; ++l) iters += ctx->h_pose.get()->iters_per_level[l];
    ctx->launches += ctx->graph_launches_fixed + (int64_t)iters * ctx->graph_launches_per_iter;
    return rc;
  }
  ctx->failed_paths |= 1u << 1;
  ctx->path_note = ctx->err;
  ctx->invalidate_graph();
  cudaGetLastError();
  cudaStreamCaptureStatus st;
  if (cudaStreamIsCapturing(ctx->stream, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone) {
    cudaGraph_t junk = nullptr;
    cudaStreamEndCapture(ctx->stream, &junk);
    if (junk) cudaGraphDestroy(junk);
  }
  cudaGetLastError();
  return kPathUnavailable;
}

// One cooperative persistent launch per active level (path 2); path 3 runs a level that qualifies inside one
// thread-block cluster instead.
static int optimize_coop(phovo_ctx* ctx, int path) {
  upload_state(ctx);
  return for_each_level(ctx->cfg, [&](int level, int) {
    const LevelParams L = ctx->level_params(level);
    const LevelPtrs P = ctx->level_ptrs(level);
    // (no k_begin_level: the persistent kernel keeps iteration / done in registers and shared memory
    // and writes the whole PoseDev back when the level ends)
    int grid = 0; cudaError_t e = cudaSuccess;
    if (path == 3 && !path_failed(ctx, 3)) {      // small level: one thread-block cluster, cluster barriers
      const int n = launch_level_cluster(ctx->stream, L, P, ctx->d_pose.get(), ctx->d_log.get(), &ctx->launch_state, &e);
      if (n > 0) { ctx->launches += n; return PHOVO_OK; }
      if (n < 0) {   // refused: this level and the rest take path 2
        const int r = path_unavailable(ctx, 3, "cluster launch", e);
        if (r != kPathUnavailable) return r;
      }
    }
    const int n = launch_level_coop(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->d_log.get(), &ctx->launch_state, ctx->sm_count, &grid, &e);
    if (n < 0) return path_unavailable(ctx, 2, "cooperative launch", e);
    ctx->launches += n;
    return PHOVO_OK;
  });
}

// Ceres mode with the LM loop on the device: one cooperative launch per active level (CE:437).
static int optimize_ceres_coop(phovo_ctx* ctx) {
  upload_state(ctx);
  return for_each_level(ctx->cfg, [&](int level, int) {
    cudaError_t e = cudaSuccess;
    const int n = launch_level_coop_ceres(ctx->stream, ctx->level_params(level), ctx->level_ptrs(level), ctx->d_pose.get(), ctx->partials.get(),
                                          ctx->d_log.get(), lm_params(ctx->cfg, level), &ctx->launch_state, ctx->sm_count, &e);
    if (n < 0) return path_unavailable(ctx, 2, "cooperative launch", e);
    ctx->launches += n;
    return PHOVO_OK;
  });
}

static int optimize_ceres(phovo_ctx* ctx);

// The driver of this Optimize(): the path phovo_set_execution asks for, or the next one down that has not failed on this
// context.  Analytic and photometric + depth solvers: 3 -> 2 -> 1 (graph) -> 0 (stream); the cooperative paths need a
// world of one.  Ceres mode: 3 and 2 run the device LM (path 2) and fall back to the host LM (path 0), which 1 and 0 select.
static int choose_path(const phovo_ctx* ctx) {
  const bool coop = ctx->execution >= 2 && ctx->shard_world == 1 && !path_failed(ctx, 2);
  if (ctx->cfg.mode == PHOVO_MODE_CERES) return coop ? 2 : 0;
  if (coop) return ctx->execution == 3 && !path_failed(ctx, 3) ? 3 : 2;
  return ctx->execution >= 1 && !path_failed(ctx, 1) ? 1 : 0;
}

extern "C" int phovo_optimize(phovo_ctx* ctx) {
  if (!ctx) return PHOVO_E_INVALID;
  int rc = begin_solve(ctx);
  if (rc) return rc;
  const bool ceres = ctx->cfg.mode == PHOVO_MODE_CERES;
  ctx->last_path = 0;
  int path;
  do {   // a driver that cannot run marks its path failed, and the solve starts over on the next one down
    path = choose_path(ctx);
    if (ceres && path == 0) return optimize_ceres(ctx);   // host-driven LM over GPU evaluations
    if (ceres) rc = optimize_ceres_coop(ctx);
    else if (path >= 2) rc = optimize_coop(ctx, path);
    else if (path == 1) rc = optimize_graph(ctx);
    else rc = optimize_stream(ctx);
  } while (rc == kPathUnavailable);
  if (rc == PHOVO_OK && path != 1) {   // (the graph driver has read back)
    CK(cudaGetLastError());
    rc = read_back(ctx);
  }
  // a cluster launch refused during this solve: path 2 ran that level and the rest
  if (rc == PHOVO_OK || rc == PHOVO_E_NUMERIC) ctx->last_path = path == 3 && path_failed(ctx, 3) ? 2 : path;
  return rc;
}

extern "C" int phovo_last_optimize_used_graph(const phovo_ctx* ctx) { return ctx ? ctx->last_path == 1 : 0; }
extern "C" const char* phovo_graph_error(const phovo_ctx* ctx) { return ctx ? ctx->path_note.c_str() : ""; }

extern "C" int phovo_get_state(const phovo_ctx* ctx, double state[6]) {
  if (!ctx || !state) return PHOVO_E_INVALID;
  memcpy(state, ctx->state, sizeof(double) * 6);
  return PHOVO_OK;
}

extern "C" void phovo_state_to_rt(const double s[6], double P[16]) {
  // CPhotoconsistencyOdometry.h:47-71 eigenPose
  const double x = s[0], y = s[1], z = s[2], yaw = s[3], pitch = s[4], roll = s[5];
  P[0] = cos(yaw) * cos(pitch);
  P[1] = cos(yaw) * sin(pitch) * sin(roll) - sin(yaw) * cos(roll);
  P[2] = cos(yaw) * sin(pitch) * cos(roll) + sin(yaw) * sin(roll);
  P[3] = x;
  P[4] = sin(yaw) * cos(pitch);
  P[5] = sin(yaw) * sin(pitch) * sin(roll) + cos(yaw) * cos(roll);
  P[6] = sin(yaw) * sin(pitch) * cos(roll) - cos(yaw) * sin(roll);
  P[7] = y;
  P[8] = -sin(pitch);
  P[9] = cos(pitch) * sin(roll);
  P[10] = cos(pitch) * cos(roll);
  P[11] = z;
  P[12] = 0; P[13] = 0; P[14] = 0; P[15] = 1;
}

extern "C" int phovo_get_rt(const phovo_ctx* ctx, double rt[16]) {
  if (!ctx || !rt) return PHOVO_E_INVALID;
  phovo_state_to_rt(ctx->state, rt);
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// diagnostics: phovo::warpImage + absdiff (BASE:73-134; apps :107-110 / :247-252)
// ---------------------------------------------------------------------------------------------
extern "C" int phovo_warp_image(phovo_ctx* ctx, const uint8_t* gray, size_t gray_step, const void* depth, int depth_type,
                                size_t depth_step, double depth_scale, int rows, int cols, const double rt[16],
                                const double K[9], int level, uint8_t* warped, size_t warped_step,
                                const uint8_t* target, size_t target_step, uint8_t* diff, size_t diff_step) {
  if (!ctx || !gray || !depth || !rt || !K || !warped) return PHOVO_E_INVALID;
  if (rows < 1 || cols < 1 || level < 0 || level > 30) return ctx->fail(PHOVO_E_INVALID, "bad image size or level");
  if (src_type_of_depth(depth_type) < 0) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if ((diff != nullptr) != (target != nullptr)) return ctx->fail(PHOVO_E_INVALID, "target and diff must be given together");
  if (gray_step < (size_t)cols || warped_step < (size_t)cols || depth_step < (size_t)cols * depth_elt(depth_type) ||
      (diff && (target_step < (size_t)cols || diff_step < (size_t)cols)))
    return ctx->fail(PHOVO_E_INVALID, "row stride smaller than a row");
  const size_t n = (size_t)rows * cols;
  if (n > (size_t)INT32_MAX) return ctx->fail(PHOVO_E_UNSUPPORTED, "warpImage: frames of 2^31 pixels or more");
  CK(cudaSetDevice(ctx->device));
  const void* dg; size_t dgs; const void* dd; size_t dds; int rc;
  if ((rc = stage_image(ctx, gray, gray_step, 1, rows, cols, ctx->stage_gray[0], &dg, &dgs))) return rc;
  if ((rc = stage_image(ctx, depth, depth_step, depth_elt(depth_type), rows, cols, ctx->stage_depth, &dd, &dds))) return rc;
  const void* dt = nullptr; size_t dts = 0;
  if (target && (rc = stage_image(ctx, target, target_step, 1, rows, cols, ctx->warp_io[1], &dt, &dts))) return rc;
  ctx->h2d_pending = false; ctx->device_input_in_flight = false;   // this call ends with a stream synchronise
  // outputs: write in place for device callers, through a dense device buffer for host callers
  uint8_t* dw = warped; size_t dws = warped_step; uint8_t* ddf = diff; size_t ddfs = diff_step;
  const bool w_host = !is_device_pointer(warped), d_host = diff && !is_device_pointer(diff);
  if (w_host) { CK(ctx->warp_io[0].ensure(n)); dw = (uint8_t*)ctx->warp_io[0].get(); dws = cols; }
  if (d_host) { CK(ctx->warp_io[2].ensure(n)); ddf = (uint8_t*)ctx->warp_io[2].get(); ddfs = cols; }
  WarpImages W;
  memset(&W, 0, sizeof(W));
  W.rows = rows; W.cols = cols;
  W.gray = (const uint8_t*)dg; W.gray_step = dgs;
  W.depth = dd; W.depth_step = dds; W.depth_scale = depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0;
  W.target = (const uint8_t*)dt; W.target_step = dts;
  W.warped = dw; W.warped_step = dws;
  W.diff = ddf; W.diff_step = ddfs;
  if ((rc = phovo_internal_warp_images(ctx, W, src_type_of_depth(depth_type), scaled_intrinsics(K, level), 1, rt))) return rc;
  if (w_host) CK(cudaMemcpy2DAsync(warped, warped_step, dw, dws, cols, rows, cudaMemcpyDeviceToHost, ctx->stream));
  if (d_host) CK(cudaMemcpy2DAsync(diff, diff_step, ddf, ddfs, cols, rows, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// introspection
// ---------------------------------------------------------------------------------------------
extern "C" int phovo_num_iter_stats(const phovo_ctx* ctx) { return ctx ? (int)ctx->log.size() : PHOVO_E_INVALID; }

extern "C" int phovo_get_iter_stats(const phovo_ctx* ctx, int index, phovo_iter_stats* out) {
  if (!ctx || !out || index < 0 || index >= (int)ctx->log.size()) return PHOVO_E_INVALID;
  *out = ctx->log[index];
  return PHOVO_OK;
}

extern "C" int phovo_get_level_image(phovo_ctx* ctx, int which, int level, double* dst, int* rows, int* cols) {
  if (!ctx || which < 0 || which > 4 || level < 0 || level >= ctx->cfg.num_levels) return PHOVO_E_INVALID;
  if (!ctx->level_active(level)) return ctx->fail(PHOVO_E_INVALID, "level was not built (no iterations configured; see phovo_set_build_all_levels)");
  if ((which <= 1 && !ctx->have_src) || (which >= 2 && !ctx->have_tgt)) return ctx->fail(PHOVO_E_INVALID, "frame not set");
  if (rows) *rows = ctx->lrows[level];
  if (cols) *cols = ctx->lcols[level];
  if (!dst) return PHOVO_OK;
  CK(cudaSetDevice(ctx->device));
  const double* src = which == 0 ? ctx->I0[level].get() : which == 1 ? ctx->D0[level].get() : which == 2 ? ctx->I1[level].get() : which == 3 ? ctx->Gx[level].get() : ctx->Gy[level].get();
  CK(cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)ctx->lrows[level] * ctx->lcols[level], cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

static int eval_at(phovo_ctx* ctx, int level, const double state[6], phovo_iter_stats* out, double* dres, double* djac) {
  const LevelParams L = ctx->level_params(level);
  const LevelPtrs P = ctx->level_ptrs(level);
  ctx->launches += launch_set_state(ctx->stream, ctx->d_pose.get(), nullptr, state, 0);
  int grid = 0;
  ctx->launches += launch_iteration_kernels(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->sm_count, &grid, dres, djac, false);
  ctx->launches += launch_reduce_only(ctx->stream, L, ctx->d_pose.get(), ctx->partials.get(), grid, ctx->d_eval.get());
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->h_eval.get(), ctx->d_eval.get(), sizeof(phovo_iter_stats), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *out = *ctx->h_eval.get();
  return PHOVO_OK;
}

extern "C" int phovo_eval_normal_equations(phovo_ctx* ctx, int level, const double state[6], phovo_iter_stats* out) {
  if (!ctx || !state || !out) return PHOVO_E_INVALID;
  int rc = ready_to_solve(ctx);
  if (rc) return rc;
  if (level < 0 || level >= ctx->cfg.num_levels || !ctx->level_active(level)) return ctx->fail(PHOVO_E_INVALID, "level not built");
  CK(cudaSetDevice(ctx->device));
  return eval_at(ctx, level, state, out, nullptr, nullptr);
}

extern "C" int phovo_eval_residuals(phovo_ctx* ctx, int level, const double state[6], double* residuals, double* jacobian) {
  if (!ctx || !state) return PHOVO_E_INVALID;
  int rc = ready_to_solve(ctx);
  if (rc) return rc;
  if (level < 0 || level >= ctx->cfg.num_levels || !ctx->level_active(level)) return ctx->fail(PHOVO_E_INVALID, "level not built");
  CK(cudaSetDevice(ctx->device));
  const size_t n = (size_t)ctx->lrows[level] * ctx->lcols[level] * (ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE ? 2 : 1);
  CK(ctx->dump_res.ensure(n));
  CK(ctx->dump_jac.ensure(n * 6));
  CK(cudaMemsetAsync(ctx->dump_res.get(), 0, sizeof(double) * n, ctx->stream));
  CK(cudaMemsetAsync(ctx->dump_jac.get(), 0, sizeof(double) * n * 6, ctx->stream));
  phovo_iter_stats tmp;
  if ((rc = eval_at(ctx, level, state, &tmp, ctx->dump_res.get(), ctx->dump_jac.get()))) return rc;
  if (residuals) CK(cudaMemcpy(residuals, ctx->dump_res.get(), sizeof(double) * n, cudaMemcpyDeviceToHost));
  if (jacobian) CK(cudaMemcpy(jacobian, ctx->dump_jac.get(), sizeof(double) * n * 6, cudaMemcpyDeviceToHost));
  return PHOVO_OK;
}

extern "C" int phovo_get_timings(const phovo_ctx* ctx, float* setup_ms, float* optimize_ms) {
  if (!ctx) return PHOVO_E_INVALID;
  float a = 0, b = 0;
  if (setup_ms) { if (cudaEventElapsedTime(&a, ctx->ev_time[0].get(), ctx->ev_time[1].get()) != cudaSuccess) { a = -1; cudaGetLastError(); } *setup_ms = a; }
  if (optimize_ms) { if (cudaEventElapsedTime(&b, ctx->ev_time[2].get(), ctx->ev_time[3].get()) != cudaSuccess) { b = -1; cudaGetLastError(); } *optimize_ms = b; }
  return PHOVO_OK;
}

extern "C" int64_t phovo_launch_count(const phovo_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int phovo_synchronize(phovo_ctx* ctx) {
  if (!ctx) return PHOVO_E_INVALID;
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// Ceres mode: restated trust-region Levenberg-Marquardt driving the GPU evaluation
// (CPhotoconsistencyOdometryCeres.h:433-500 -> ceres::Solve; SURVEY appendix A).  The solver
// itself is third-party and absent from the reference tree: trajectory parity is UNPINNED, the
// residual/Jacobian kernel (K5) is pinned against the oracle.
// ---------------------------------------------------------------------------------------------
static int optimize_ceres(phovo_ctx* ctx) {
  ctx->log.clear();
  int log_count = 0;
  LmLog log{ctx->h_log.get(), log_count, ctx->log_cap(), true};
  LmState S;
  memcpy(S.x, ctx->state, sizeof(S.x));
  const int status = for_each_level(ctx->cfg, [&](int level, int) {   // CE:437
    const LmParams lm = lm_params(ctx->cfg, level);
    S.radius = lm.initial_radius; S.decrease_factor = 2.0; S.iteration = 0;
    int rc = eval_at(ctx, level, S.x, &S.cur, nullptr, nullptr);
    if (rc) return rc;
    bool go = lm_start(lm, S);
    while (go && lm_propose(lm, S, log)) {
      phovo_iter_stats cand;
      if ((rc = eval_at(ctx, level, S.xn, &cand, nullptr, nullptr))) return rc;
      const int v = lm_judge(lm, S, cand.cost, log);
      if (v == LM_ACCEPT) S.cur = cand;
      go = v != LM_STOP && lm_update_radius(lm, S, v == LM_ACCEPT);
    }
    return PHOVO_OK;
  });
  if (status) return status;
  ctx->log.assign(ctx->h_log.get(), ctx->h_log.get() + std::min(log_count, ctx->log_cap()));
  memcpy(ctx->state, S.x, sizeof(S.x));
  CK(cudaEventRecord(ctx->ev_time[3].get(), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 6; ++k)
    if (!isfinite(ctx->state[k])) return ctx->fail(PHOVO_E_NUMERIC, "non-finite state after Optimize");
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// row-sharded single pair (BASELINE config 5): each rank evaluates a band of source rows; the
// caller all-reduces the 32-double buffer between phovo_shard_partial and phovo_shard_step.
// ---------------------------------------------------------------------------------------------
static int upload_peer_table(phovo_ctx* ctx);

extern "C" int phovo_shard_configure(phovo_ctx* ctx, int rank, int world) {
  if (!ctx || world < 1 || rank < 0 || rank >= world) return PHOVO_E_INVALID;
  ctx->shard_rank = rank; ctx->shard_world = world;
  ctx->invalidate_graph();
  return PHOVO_OK;
}

extern "C" int phovo_shard_buffer(phovo_ctx* ctx, double** dev_ptr) {
  if (!ctx || !dev_ptr) return PHOVO_E_INVALID;
  *dev_ptr = ctx->d_shard.get();
  return PHOVO_OK;
}

extern "C" int phovo_shard_read_buffer(phovo_ctx* ctx, double out[32]) {
  if (!ctx || !out) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(out, ctx->d_shard.get(), sizeof(double) * 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

extern "C" int phovo_shard_write_buffer(phovo_ctx* ctx, const double in[32]) {
  if (!ctx || !in) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(ctx->d_shard.get(), in, sizeof(double) * 32, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

extern "C" int phovo_shard_begin(phovo_ctx* ctx) {
  if (!ctx) return PHOVO_E_INVALID;
  const int rc = begin_solve(ctx);
  if (rc) return rc;
  upload_state(ctx);
  ctx->shard_level = -1;
  return PHOVO_OK;
}

extern "C" int phovo_shard_begin_level(phovo_ctx* ctx, int level) {
  if (!ctx || level < 0 || level >= ctx->cfg.num_levels) return PHOVO_E_INVALID;
  if (!ctx->level_active(level)) return ctx->fail(PHOVO_E_INVALID, "level not built");
  CK(cudaSetDevice(ctx->device));
  ctx->shard_level = level;
  ctx->launches += launch_begin_level(ctx->stream, ctx->d_pose.get(), ctx->cfg.max_num_iterations[level]);
  return PHOVO_OK;
}

extern "C" int phovo_shard_partial(phovo_ctx* ctx) {
  if (!ctx || ctx->shard_level < 0) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  const LevelParams L = ctx->level_params(ctx->shard_level);
  const LevelPtrs P = ctx->level_ptrs(ctx->shard_level);
  int grid = 0;
  ctx->launches += launch_iteration_kernels(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->sm_count, &grid, nullptr, nullptr, false);
  ctx->launches += launch_reduce_to_buffer(ctx->stream, ctx->partials.get(), grid, ctx->d_shard.get());
  CK(cudaGetLastError());
  return PHOVO_OK;
}

extern "C" int phovo_shard_peer_export(phovo_ctx* ctx, void* handle_out) {
  if (!ctx || !handle_out) return PHOVO_E_INVALID;
  static_assert(sizeof(cudaIpcMemHandle_t) == PHOVO_IPC_HANDLE_BYTES, "IPC handle size");
  CK(cudaSetDevice(ctx->device));
  if (!ctx->xchg_own.get()) {
    CK(ctx->xchg_own.ensure(1));
    CK(cudaMemset(ctx->xchg_own.get(), 0, sizeof(ShardExchange)));
    CK(cudaDeviceSynchronize());
  }
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, ctx->xchg_own.get()));
  memcpy(handle_out, &h, sizeof(h));
  ctx->xchg_peer[ctx->shard_rank] = ctx->xchg_own.get();
  ctx->xchg_table_dirty = true;
  return PHOVO_OK;
}

extern "C" int phovo_shard_peer_import(phovo_ctx* ctx, int peer_rank, const void* handle) {
  if (!ctx || !handle || peer_rank < 0 || peer_rank >= PHOVO_SHARD_MAX_WORLD) return PHOVO_E_INVALID;
  if (peer_rank == ctx->shard_rank) return PHOVO_OK;   // own area: no IPC round trip
  CK(cudaSetDevice(ctx->device));
  if (ctx->xchg_opened[peer_rank]) { cudaIpcCloseMemHandle(ctx->xchg_peer[peer_rank]); ctx->xchg_opened[peer_rank] = false; }
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  ctx->xchg_peer[peer_rank] = (ShardExchange*)p;
  ctx->xchg_opened[peer_rank] = true;
  ctx->xchg_table_dirty = true;
  return PHOVO_OK;
}

extern "C" int phovo_shard_partial_exchange(phovo_ctx* ctx) {
  if (!ctx || ctx->shard_level < 0) return PHOVO_E_INVALID;
  if (ctx->shard_world > PHOVO_SHARD_MAX_WORLD) return ctx->fail(PHOVO_E_UNSUPPORTED, "peer exchange supports up to 8 ranks");
  CK(cudaSetDevice(ctx->device));
  { int rc = upload_peer_table(ctx); if (rc) return rc; }
  const LevelParams L = ctx->level_params(ctx->shard_level);
  const LevelPtrs P = ctx->level_ptrs(ctx->shard_level);
  int grid = 0;
  ctx->launches += launch_iteration_kernels(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->sm_count, &grid, nullptr, nullptr, false);
  ctx->xchg_epoch += 1;
  ctx->launches += launch_reduce_exchange(ctx->stream, ctx->d_pose.get(), ctx->partials.get(), grid, ctx->d_shard.get(), ctx->xchg_peers_dev.get(),
                                          ctx->shard_rank, ctx->shard_world, ctx->xchg_epoch);
  CK(cudaGetLastError());
  return PHOVO_OK;
}

static int upload_peer_table(phovo_ctx* ctx) {
  for (int r = 0; r < ctx->shard_world; ++r)
    if (!ctx->xchg_peer[r]) return ctx->fail(PHOVO_E_INVALID, "peer exchange areas are not all imported (phovo_shard_peer_export / _import)");
  CK(ctx->xchg_peers_dev.ensure(PHOVO_SHARD_MAX_WORLD));
  if (ctx->xchg_table_dirty) {
    CK(cudaMemcpyAsync(ctx->xchg_peers_dev.get(), ctx->xchg_peer, sizeof(ShardExchange*) * PHOVO_SHARD_MAX_WORLD, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->xchg_table_dirty = false;
  }
  return PHOVO_OK;
}

extern "C" int phovo_shard_optimize(phovo_ctx* ctx, int min_shard_pixels) {
  if (!ctx) return PHOVO_E_INVALID;
  if (ctx->cfg.mode != PHOVO_MODE_ANALYTIC_REF && ctx->cfg.mode != PHOVO_MODE_ANALYTIC_FIXED)
    return ctx->fail(PHOVO_E_UNSUPPORTED, "the row-sharded loop implements the analytic solver only");
  if (path_failed(ctx, 2)) return ctx->fail(PHOVO_E_UNSUPPORTED, "cooperative launch is not available on this device");
  if (ctx->shard_world > PHOVO_SHARD_MAX_WORLD) return ctx->fail(PHOVO_E_UNSUPPORTED, "peer exchange supports up to 8 ranks");
  int rc = begin_solve(ctx);
  if (rc) return rc;
  if (ctx->shard_world > 1 && (rc = upload_peer_table(ctx))) return rc;
  if (ctx->shard_world > 1 && !ctx->level_dmin_valid) {   // once per source frame: what bounds the row displacement (ShardArgs)
    CK(ctx->d_level_dmin.ensure(PHOVO_MAX_LEVELS));
    for (int level = 0; level < ctx->cfg.num_levels; ++level)
      if (ctx->cfg.max_num_iterations[level] > 0)
        ctx->launches += launch_min_valid_depth(ctx->stream, ctx->D0[level].get(), ctx->lrows[level] * ctx->lcols[level], ctx->cfg.min_depth,
                                                ctx->cfg.max_depth, ctx->d_level_dmin.get() + level, ctx->sm_count);
    ctx->level_dmin_valid = true;
  }
  upload_state(ctx);
  rc = for_each_level(ctx->cfg, [&](int level, int M) {
    LevelParams L = ctx->level_params(level);                          // carries this rank's row band
    const LevelPtrs P = ctx->level_ptrs(level);
    const bool shard = ctx->shard_world > 1 && (long long)L.rows * L.cols >= (long long)min_shard_pixels;
    if (!shard) { L.row_begin = 0; L.row_end = L.rows; }
    int grid = 0; cudaError_t e = cudaSuccess;
    const int n = launch_level_coop(ctx->stream, L, P, ctx->d_pose.get(), ctx->partials.get(), ctx->d_log.get(), &ctx->launch_state, ctx->sm_count, &grid, &e,
                                    shard ? ctx->xchg_peers_dev.get() : nullptr, ctx->shard_rank, ctx->shard_world, ctx->xchg_epoch,
                                    shard ? ctx->d_level_dmin.get() + level : nullptr);
    if (n < 0) { cudaGetLastError(); return ctx->cuda_fail("cooperative launch of the sharded level loop", e); }
    ctx->launches += n;
    if (shard) ctx->xchg_epoch += (unsigned long long)M;               // every rank advances by the same amount
    return PHOVO_OK;
  });
  if (rc) return rc;
  CK(cudaGetLastError());
  ctx->last_path = 2;
  return end_solve(ctx);
}

extern "C" int phovo_shard_step(phovo_ctx* ctx, int* done) {
  if (!ctx || ctx->shard_level < 0) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  const LevelParams L = ctx->level_params(ctx->shard_level);
  ctx->launches += launch_solve_from_buffer(ctx->stream, L, ctx->d_pose.get(), ctx->d_shard.get(), ctx->d_log.get());
  CK(cudaGetLastError());
  if (done) {
    CK(cudaMemcpyAsync(&ctx->h_pose.get()->done, &ctx->d_pose.get()->done, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *done = ctx->h_pose.get()->done;
  }
  return PHOVO_OK;
}

extern "C" int phovo_shard_finish(phovo_ctx* ctx) {
  if (!ctx) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  return end_solve(ctx);
}
