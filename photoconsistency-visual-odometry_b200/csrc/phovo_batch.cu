// phovo_batch.cu -- host side of the batch-of-pairs extension (phovo_batch_* in phovo_b200.h).
//
// HBM layout: inputs stay in the caller's layout ([P][rows][cols] u8 / depth); the pyramid kernel
// writes one packed record per pair holding, for each ACTIVE level, I0 and I1 as u16 tap sums and
// D0 as fp64 (12 B/px; 288 000 B per 640x480 pair under the 4-level config).  The align kernel
// reads each record exactly once.  Host inputs are streamed in chunks through two device staging
// slots on two streams so that the PCIe copy of chunk k+1 overlaps the kernels of chunk k.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

#include "phovo_batch.h"
#include "phovo_ctx.h"

using namespace phovo;

constexpr int kWaveSetupThreads = 4;   // host threads (and streams) that build the pyramids of a wave's slots

struct phovo_batch_state {
  // packed level records
  uint8_t* store = nullptr; size_t store_cap = 0;
  // outputs of the last call (device)
  double* states = nullptr; size_t states_cap = 0;
  int32_t* iters = nullptr; size_t iters_cap = 0;
  double* init = nullptr; size_t init_cap = 0;
  phovo_iter_stats* log = nullptr; size_t log_cap_entries = 0;
  int32_t* log_counts = nullptr; size_t log_counts_cap = 0;
  // host mirrors of the stats (filled on demand)
  std::vector<phovo_iter_stats> h_log; std::vector<int32_t> h_log_counts;
  int log_per_pair = 0; int last_pairs = 0; bool log_fetched = false;
  bool record_stats = false;
  int debug_flags = 0;
  unsigned long long last_h2d_bytes = 0;
  // staging for host inputs: two slots
  uint8_t* stage_g0[2] = {nullptr, nullptr}; uint8_t* stage_g1[2] = {nullptr, nullptr}; char* stage_d[2] = {nullptr, nullptr};
  size_t stage_cap_g[2] = {0, 0}, stage_cap_g1[2] = {0, 0}, stage_cap_d[2] = {0, 0};
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  double* h_states_pinned = nullptr; int32_t* h_iters_pinned = nullptr; size_t h_out_cap = 0;
  size_t prepared_smem = 0;
  unsigned int* next_pair = nullptr;   // work counter of the persistent align kernel
  int sm_count = 0;
  cudaEvent_t ev_k[3] = {nullptr, nullptr, nullptr};   // before pyramid / between / after align
  bool timed = false;
  // batches the shared-memory-resident kernels cannot take (Ceres / photometric + depth solver, blurred levels, levels
  // beyond the shared-memory budget) run pair by pair on a small pool of per-pair contexts, one host thread each
  std::vector<phovo_ctx*> pool;
  int last_path = 0;                                   // 1: shared-memory-resident batch kernels, 2: pool of per-pair contexts, 3: slot waves
  // slot waves (batch_waves): two halves of per-pair slots; one half aligns while the other is being set up
  std::vector<phovo_ctx*> slots;
  cudaStream_t setup_stream[kWaveSetupThreads] = {}; cudaEvent_t ev_setup[kWaveSetupThreads] = {};
  cudaStream_t align_stream[2] = {nullptr, nullptr}; cudaEvent_t ev_wave_done[2] = {nullptr, nullptr}; cudaEvent_t ev_wave_in[2] = {nullptr, nullptr};
  char* arena = nullptr; size_t arena_cap = 0, slot_bytes = 0; int arena_rows = 0, arena_cols = 0, arena_slots = 0, wave_half = 0; phovo_config arena_cfg = {};
  SlotArgs* d_slot_args = nullptr; size_t slot_args_cap = 0; std::vector<SlotArgs> h_slot_args;
  double* d_wave_init[2] = {nullptr, nullptr}; double* d_wave_states[2] = {nullptr, nullptr}; int32_t* d_wave_iters[2] = {nullptr, nullptr};
  double* h_wave_states[2] = {nullptr, nullptr}; int32_t* h_wave_iters[2] = {nullptr, nullptr}; size_t wave_cap = 0;
  uint8_t* wave_g0[2] = {nullptr, nullptr}; uint8_t* wave_g1[2] = {nullptr, nullptr}; char* wave_d0[2] = {nullptr, nullptr}; char* wave_d1[2] = {nullptr, nullptr};
  size_t wave_g_cap[2] = {0, 0}, wave_g1_cap[2] = {0, 0}, wave_d0_cap[2] = {0, 0}, wave_d1_cap[2] = {0, 0};
  // warpImage (phovo_batch_warp_image, phovo_warp_image): splat keys of one chunk of pairs (zero between calls while
  // warp_keys_clean), Rt of the pairs, per-pair summaries, device copies of host inputs and outputs of one chunk
  uint32_t* warp_keys = nullptr; size_t warp_keys_cap = 0; bool warp_keys_clean = false;
  double* warp_rts = nullptr; size_t warp_rts_cap = 0;
  int32_t* warp_landed = nullptr; size_t warp_landed_cap = 0;
  int64_t* warp_sum = nullptr; size_t warp_sum_cap = 0;
  uint8_t* warp_io[4] = {nullptr, nullptr, nullptr, nullptr}; size_t warp_io_cap[4] = {0, 0, 0, 0};   // gray0, gray1, warped, diff
  char* warp_depth = nullptr; size_t warp_depth_cap = 0;
  int l2_bytes = 0;
  // normal equations at given states (phovo_batch_eval_normal_equations): winner keys (zero between calls while
  // eval_keys_clean) and validity of one chunk, its level records and tile partials; states, poses and results of
  // every pair.  Host inputs are staged through warp_io[0] / warp_io[1] / warp_depth.
  uint32_t* eval_keys = nullptr; size_t eval_keys_cap = 0; bool eval_keys_clean = false;
  uint8_t* eval_valid = nullptr; size_t eval_valid_cap = 0;
  uint8_t* eval_store = nullptr; size_t eval_store_cap = 0;
  double* eval_partials = nullptr; size_t eval_partials_cap = 0;
  double* eval_states = nullptr; size_t eval_states_cap = 0;
  PoseDev* eval_poses = nullptr; size_t eval_poses_cap = 0;
  double* eval_out = nullptr; size_t eval_out_cap = 0;        // [P][21] H, [P][6] g, [P] cost
  int32_t* eval_nvalid = nullptr; size_t eval_nvalid_cap = 0;
};

#define CK(call)                                                      \
  do {                                                                \
    cudaError_t e_ = (call);                                          \
    if (e_ != cudaSuccess) return ctx->cuda_fail((std::string(__func__) + ": " #call).c_str(), e_); \
  } while (0)

template <class T>
static cudaError_t ensure(T** p, size_t* cap, size_t want) {
  if (*cap >= want && *p) return cudaSuccess;
  if (*p) cudaFree(*p);
  *p = nullptr; *cap = 0;
  cudaError_t e = cudaMalloc((void**)p, want * sizeof(T));
  if (e == cudaSuccess) *cap = want;
  return e;
}

void phovo_batch_release(phovo_ctx* ctx) {
  phovo_batch_state* b = ctx->batch;
  if (!b) return;
  cudaFree(b->next_pair);
  cudaFree(b->store); cudaFree(b->states); cudaFree(b->iters); cudaFree(b->init); cudaFree(b->log); cudaFree(b->log_counts);
  for (int s = 0; s < 2; ++s) {
    cudaFree(b->stage_g0[s]); cudaFree(b->stage_g1[s]); cudaFree(b->stage_d[s]);
    if (b->ev_copied[s]) cudaEventDestroy(b->ev_copied[s]);
    if (b->ev_consumed[s]) cudaEventDestroy(b->ev_consumed[s]);
  }
  if (b->copy_stream) cudaStreamDestroy(b->copy_stream);
  cudaFreeHost(b->h_states_pinned); cudaFreeHost(b->h_iters_pinned);
  for (phovo_ctx* c : b->pool) phovo_destroy(c);
  for (phovo_ctx* c : b->slots) phovo_destroy(c);      // (their streams are the setup streams below: not owned)
  for (int t = 0; t < kWaveSetupThreads; ++t) {
    if (b->setup_stream[t]) cudaStreamDestroy(b->setup_stream[t]);
    if (b->ev_setup[t]) cudaEventDestroy(b->ev_setup[t]);
  }
  for (int h = 0; h < 2; ++h) {
    if (b->align_stream[h]) cudaStreamDestroy(b->align_stream[h]);
    if (b->ev_wave_done[h]) cudaEventDestroy(b->ev_wave_done[h]);
    if (b->ev_wave_in[h]) cudaEventDestroy(b->ev_wave_in[h]);
    cudaFree(b->d_wave_init[h]); cudaFree(b->d_wave_states[h]); cudaFree(b->d_wave_iters[h]);
    cudaFreeHost(b->h_wave_states[h]); cudaFreeHost(b->h_wave_iters[h]);
    cudaFree(b->wave_g0[h]); cudaFree(b->wave_g1[h]); cudaFree(b->wave_d0[h]); cudaFree(b->wave_d1[h]);
  }
  cudaFree(b->d_slot_args);
  cudaFree(b->arena);
  cudaFree(b->warp_keys); cudaFree(b->warp_rts); cudaFree(b->warp_landed); cudaFree(b->warp_sum); cudaFree(b->warp_depth);
  for (int k = 0; k < 4; ++k) cudaFree(b->warp_io[k]);
  cudaFree(b->eval_keys); cudaFree(b->eval_valid); cudaFree(b->eval_store); cudaFree(b->eval_partials);
  cudaFree(b->eval_states); cudaFree(b->eval_poses); cudaFree(b->eval_out); cudaFree(b->eval_nvalid);
  delete b;
  ctx->batch = nullptr;
}

static int get_state(phovo_ctx* ctx, phovo_batch_state** out) {
  if (!ctx->batch) {
    ctx->batch = new phovo_batch_state();
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->batch->sm_count = prop.multiProcessorCount;
    ctx->batch->l2_bytes = prop.l2CacheSize;
    CK(cudaStreamCreateWithFlags(&ctx->batch->copy_stream, cudaStreamNonBlocking));
    CK(cudaMalloc((void**)&ctx->batch->next_pair, sizeof(unsigned int) * PHOVO_MAX_LEVELS));
    for (int s = 0; s < 2; ++s) {
      CK(cudaEventCreateWithFlags(&ctx->batch->ev_copied[s], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&ctx->batch->ev_consumed[s], cudaEventDisableTiming));
    }
  }
  *out = ctx->batch;
  return PHOVO_OK;
}

static void level_size(int rows, int cols, int level, int* orows, int* ocols) {
  const double f = ldexp(1.0, -level);
  *orows = level == 0 ? rows : (int)lrint(rows * f);
  *ocols = level == 0 ? cols : (int)lrint(cols * f);
}

// Active level `a` of bp = pyramid level `level` of a rows x cols frame under the context's config: size, record
// offsets (appended at *off), intrinsics, step and gradient scale.  Fails on what the pyramid kernel cannot build.
static int fill_level(phovo_ctx* ctx, int rows, int cols, int level, int a, BatchParams* bp, unsigned long long* off) {
  if (ctx->cfg.blur_filter_size[level] > 1) return ctx->fail(PHOVO_E_UNSUPPORTED, "batch kernel: blurFilterSize > 0 is only supported by the per-pair API");
  // cv::resize by 1/2 averages cells cut by the image border in single precision (sizes = 3 mod 4):
  // not representable in the exact integer tap sums the batch records keep
  if (level == 1 && (rows % 4 == 3 || cols % 4 == 3))
    return ctx->fail(PHOVO_E_UNSUPPORTED, "batch kernel: level 1 of an image whose size is 3 mod 4 is only supported by the per-pair API");
  int lr, lc;
  level_size(rows, cols, level, &lr, &lc);
  if (lr < 1 || lc < 1) return ctx->fail(PHOVO_E_INVALID, "image too small for the number of pyramid levels");
  const int n = lr * lc;
  bp->level[a] = level; bp->lrows[a] = lr; bp->lcols[a] = lc;
  bp->px_offset[a + 1] = bp->px_offset[a] + n;
  const unsigned long long n16 = ((unsigned long long)n * 2 + 15) & ~15ull, n64 = ((unsigned long long)n * 8 + 15) & ~15ull;
  bp->off_D0[a] = *off; *off += n64;
  bp->off_I0[a] = *off; *off += n16;
  bp->off_I1[a] = *off; *off += n16;
  bp->off_D32[a] = *off; *off += ((unsigned long long)n * 4 + 15) & ~15ull;
  // CPhotoconsistencyOdometryAnalytic.h:203-209
  const double scaleFactor = 1.0 / pow(2, level);
  bp->fx[a] = ctx->K[0] * scaleFactor; bp->fy[a] = ctx->K[4] * scaleFactor;
  bp->ox[a] = ctx->K[2] * scaleFactor; bp->oy[a] = ctx->K[5] * scaleFactor;
  bp->inv_fx[a] = 1.f / bp->fx[a]; bp->inv_fy[a] = 1.f / bp->fy[a];
  bp->lambda[a] = ctx->cfg.lambda_step[level]; bp->min_grad[a] = ctx->cfg.min_gradient_norm[level];
  bp->grad_k[a] = ctx->cfg.grad_scale[level] / 1020.0;
  return PHOVO_OK;
}

// Parameter block for a rows x cols batch under the context's config; fails loudly when a
// configuration cannot run in the shared-memory-resident kernel (there is no slower fallback
// inside this entry point: the caller is told to use the per-pair API).
static int make_params(phovo_ctx* ctx, int num_pairs, int rows, int cols, int log_cap, BatchParams* bp, size_t* smem_out) {
  if (!ctx->have_K) return ctx->fail(PHOVO_E_INVALID, "SetIntrinsicMatrix has not been called");
  if (num_pairs < 1 || rows < 1 || cols < 1) return ctx->fail(PHOVO_E_INVALID, "empty batch");
  if (ctx->cfg.mode == PHOVO_MODE_CERES || ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE)
    return ctx->fail(PHOVO_E_UNSUPPORTED, "the shared-memory-resident batch kernels implement the analytic solver only");
  memset(bp, 0, sizeof(*bp));
  bp->num_pairs = num_pairs; bp->rows = rows; bp->cols = cols;
  bp->mode = ctx->cfg.mode; bp->log_cap = log_cap;
  bp->exact_always = ctx->batch ? (ctx->batch->debug_flags & 1) : 0;
  bp->force_generic = ctx->batch ? ((ctx->batch->debug_flags >> 1) & 1) : 0;
  bp->min_depth = ctx->cfg.min_depth; bp->max_depth = ctx->cfg.max_depth;
  int a = 0, nmax = 0;
  unsigned long long off = 0;
  for (int level = ctx->cfg.num_levels - 1; level >= 0; --level) {
    if (ctx->cfg.max_num_iterations[level] <= 0) continue;
    const int rc = fill_level(ctx, rows, cols, level, a, bp, &off);
    if (rc) return rc;
    const int n = bp->lrows[a] * bp->lcols[a];
    if (n > kBatchMaxLevelPixels) return ctx->fail(PHOVO_E_UNSUPPORTED, "batch kernel: an active level exceeds the shared-memory budget (about 20K px); use the per-pair API");
    nmax = std::max(nmax, n);
    bp->max_iters[a] = ctx->cfg.max_num_iterations[level];
    ++a;
  }
  bp->num_active = a;
  bp->record_bytes = off ? off : 16;
  *smem_out = 0;
  for (int k = 0; k < a; ++k) {
    const size_t need = batch_level_smem_bytes(bp->lrows[k], bp->lcols[k]);
    if (need > 227 * 1024) return ctx->fail(PHOVO_E_UNSUPPORTED, "batch kernel: an active level exceeds the shared-memory budget; use the per-pair API");
    *smem_out = std::max(*smem_out, need);
  }
  return PHOVO_OK;
}

// Which source rows do the active levels read?  Level l >= 1 of an image whose height is a
// multiple of 2^l reads rows 2^l y + 2^(l-1) - 1 and 2^l y + 2^(l-1) only (central 2x2 taps of
// cv::resize at an exact power-of-two factor, AN:132).  If, within the period 2^lmax, the rows read
// form one contiguous run [begin, begin + keep), a host batch is uploaded with one strided 2-D copy
// that skips the other rows (640x480, levels 2+3: rows 1..6 of every 8, 25 % less PCIe traffic).
static void row_compaction(const phovo_ctx* ctx, int rows, int* period, int* begin, int* keep) {
  *period = 0; *begin = 0; *keep = 0;
  int lmax = 0;
  for (int l = 0; l < ctx->cfg.num_levels; ++l) {
    if (ctx->cfg.max_num_iterations[l] <= 0) continue;
    if (l == 0) return;                       // level 0 reads every row
    lmax = std::max(lmax, l);
  }
  if (lmax == 0 || lmax > 6) return;
  const int P = 1 << lmax;
  if (rows % P != 0) return;                  // border taps would break the pattern
  std::vector<char> need(P, 0);
  for (int l = 1; l <= lmax; ++l) {
    if (ctx->cfg.max_num_iterations[l] <= 0) continue;
    for (int y = 0; y < P >> l; ++y) { need[(y << l) + (1 << (l - 1)) - 1] = 1; need[(y << l) + (1 << (l - 1))] = 1; }
  }
  int first = 0; while (first < P && !need[first]) ++first;
  int last = P - 1; while (last >= 0 && !need[last]) --last;
  if (first > last || (first == 0 && last == P - 1)) return;   // nothing to skip
  for (int r = first; r <= last; ++r) if (!need[r]) return;     // holes inside the run: keep it simple, copy everything
  *period = P; *begin = first; *keep = last - first + 1;
}

static int run_device(phovo_ctx* ctx, phovo_batch_state* b, const BatchParams& bp, size_t smem, cudaStream_t stream,
                      const uint8_t* g0, const void* d0, int depth_type, double depth_scale, const uint8_t* g1,
                      uint8_t* store, const double* init, double* states, int32_t* iters,
                      phovo_iter_stats* log, int32_t* log_counts) {
  CK(cudaMemsetAsync(iters, 0, sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)bp.num_pairs, stream));
  if (bp.num_active == 0) {  // nothing to optimise: the state passes through (AN:526)
    if (init) CK(cudaMemcpyAsync(states, init, sizeof(double) * 6 * (size_t)bp.num_pairs, cudaMemcpyDeviceToDevice, stream));
    else CK(cudaMemsetAsync(states, 0, sizeof(double) * 6 * (size_t)bp.num_pairs, stream));
    return PHOVO_OK;
  }
  if (!b->prepared_smem) {
    CK(batch_align_prepare());
    b->prepared_smem = 1;
  }
  const int src = depth_type == PHOVO_DEPTH_F64 ? SRC_F64 : depth_type == PHOVO_DEPTH_F32 ? SRC_F32 : SRC_U16;
  if (!b->ev_k[0]) for (int i = 0; i < 3; ++i) CK(cudaEventCreate(&b->ev_k[i]));
  CK(cudaEventRecord(b->ev_k[0], stream));
  ctx->launches += launch_batch_pyramid(stream, bp, g0, d0, src, depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0, g1, store);
  CK(cudaEventRecord(b->ev_k[1], stream));
  CK(cudaMemsetAsync(b->next_pair, 0, sizeof(unsigned int) * PHOVO_MAX_LEVELS, stream));
  ctx->launches += launch_batch_align(stream, bp, b->sm_count, store, init, states, iters, log, log_counts, b->next_pair);
  CK(cudaEventRecord(b->ev_k[2], stream));
  b->timed = true;
  CK(cudaGetLastError());
  return PHOVO_OK;
}

extern "C" int phovo_batch_get_last_h2d_bytes(const phovo_ctx* ctx, unsigned long long* bytes) {
  if (!ctx || !bytes || !ctx->batch) return PHOVO_E_INVALID;
  *bytes = ctx->batch->last_h2d_bytes;
  return PHOVO_OK;
}

extern "C" int phovo_batch_get_kernel_times(phovo_ctx* ctx, float* pyramid_ms, float* align_ms) {
  if (!ctx || !ctx->batch || !ctx->batch->timed) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventSynchronize(ctx->batch->ev_k[2]));
  float a = 0, c = 0;
  CK(cudaEventElapsedTime(&a, ctx->batch->ev_k[0], ctx->batch->ev_k[1]));
  CK(cudaEventElapsedTime(&c, ctx->batch->ev_k[1], ctx->batch->ev_k[2]));
  if (pyramid_ms) *pyramid_ms = a;
  if (align_ms) *align_ms = c;
  return PHOVO_OK;
}

static size_t depth_elt(int t) { return t == PHOVO_DEPTH_F64 ? 8 : t == PHOVO_DEPTH_F32 ? 4 : 2; }

extern "C" int phovo_batch_set_record_stats(phovo_ctx* ctx, int enable) {
  if (!ctx) return PHOVO_E_INVALID;
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  b->record_stats = enable != 0;
  return PHOVO_OK;
}

extern "C" int phovo_batch_release_memory(phovo_ctx* ctx) {
  if (!ctx) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  phovo_batch_release(ctx);
  return PHOVO_OK;
}

extern "C" int phovo_batch_set_debug_flags(phovo_ctx* ctx, int flags) {
  if (!ctx) return PHOVO_E_INVALID;
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  b->debug_flags = flags;
  return PHOVO_OK;
}

static int prepare_log(phovo_ctx* ctx, phovo_batch_state* b, int num_pairs, int* log_cap) {
  *log_cap = 0;
  b->last_pairs = num_pairs; b->log_fetched = false; b->log_per_pair = 0;
  if (!b->record_stats) return PHOVO_OK;
  int total = 0;
  for (int l = 0; l < ctx->cfg.num_levels; ++l) total += ctx->cfg.max_num_iterations[l];
  if (total < 1) total = 1;
  CK(ensure(&b->log, &b->log_cap_entries, (size_t)num_pairs * total));
  CK(ensure(&b->log_counts, &b->log_counts_cap, (size_t)num_pairs));
  b->log_per_pair = total;
  *log_cap = total;
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// The pool path.  phovo_batch_align never refuses a configuration: what the shared-memory-resident kernels cannot
// take goes, pair by pair, through the general path (phovo_set_source / phovo_set_target / phovo_optimize: the
// persistent cooperative kernels of kernels_align.cu) on kPoolContexts child contexts of the same device, each driven
// by its own host thread, so that the frame set-up of one pair overlaps the iteration loop of another.  Same results
// as calling the per-pair API in a loop, by construction.
// ---------------------------------------------------------------------------------------------
constexpr int kPoolContexts = 8;   // measured: 1 / 2 / 4 / 8 contexts 2.5 / 4.8 / 8.9 / 12.2 K pairs/s; beyond the 8 hardware queues it collapses
constexpr int kPoolContextsMax = 32;
// PHOVO_POOL_CONTEXTS overrides the number of child contexts (1..32): a tuning knob, results do not depend on it
static int pool_contexts() {
  const char* e = getenv("PHOVO_POOL_CONTEXTS");
  const int v = e ? atoi(e) : 0;
  return v >= 1 && v <= kPoolContextsMax ? v : kPoolContexts;
}

static bool host_readable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return a.type != cudaMemoryTypeDevice;
}

static int batch_general(phovo_ctx* ctx, phovo_batch_state* b, int num_pairs, int rows, int cols, const uint8_t* gray0,
                         const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1, const void* depth1,
                         const double* initial_states, double* states, int32_t* iterations) {
  if (!ctx->have_K) return ctx->fail(PHOVO_E_INVALID, "SetIntrinsicMatrix has not been called");
  if (num_pairs < 1 || rows < 1 || cols < 1) return ctx->fail(PHOVO_E_INVALID, "empty batch");
  if (ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE && !depth1)
    return ctx->fail(PHOVO_E_INVALID, "the photometric + depth solver needs the target depth: use phovo_batch_align_with_target_depth");
  // the pool's contexts run on their own streams: device-resident inputs produced on this context's stream must be complete
  CK(cudaStreamSynchronize(ctx->stream));
  const int workers = std::min(pool_contexts(), num_pairs);
  while ((int)b->pool.size() < workers) {
    phovo_ctx* c = nullptr;
    if (phovo_create(ctx->device, &c) != PHOVO_OK) return ctx->fail(PHOVO_E_CUDA, std::string("batch pool: ") + phovo_last_error(nullptr));
    b->pool.push_back(c);
  }
  std::vector<double> init_host;
  if (initial_states && !host_readable(initial_states)) {
    init_host.resize((size_t)num_pairs * 6);
    CK(cudaMemcpy(init_host.data(), initial_states, sizeof(double) * init_host.size(), cudaMemcpyDeviceToHost));
    initial_states = init_host.data();
  }
  const size_t frame = (size_t)rows * cols, delt = depth_type == PHOVO_DEPTH_F64 ? 8 : depth_type == PHOVO_DEPTH_F32 ? 4 : 2;
  // per-pair per-iteration stats (phovo_batch_set_record_stats): the children's logs, kept in the host mirrors
  int log_per_pair = 0;
  if (b->record_stats) {
    for (int l = 0; l < ctx->cfg.num_levels; ++l) log_per_pair += ctx->cfg.max_num_iterations[l];
    log_per_pair += 1;
    b->h_log.assign((size_t)num_pairs * log_per_pair, phovo_iter_stats{});
    b->h_log_counts.assign(num_pairs, 0);
  }
  std::atomic<int> next(0), first_rc(PHOVO_OK);
  std::mutex mu; std::string message;
  auto work = [&](phovo_ctx* c) {
    auto fail = [&](int rc) {
      std::lock_guard<std::mutex> g(mu);
      if (first_rc.load() == PHOVO_OK) { first_rc.store(rc); message = phovo_last_error(c); }
    };
    int rc = phovo_set_config(c, &ctx->cfg);
    if (!rc) rc = phovo_set_intrinsics(c, ctx->K);
    if (!rc) rc = phovo_set_execution(c, ctx->execution);
    { const char* e = getenv("PHOVO_POOL_SM_SHARE"); const int d = e ? atoi(e) : 1; if (d > 1) c->sm_count = std::max(4, ctx->sm_count / d); }
    if (rc) { fail(rc); return; }
    const double zeros[6] = {0, 0, 0, 0, 0, 0};
    for (;;) {
      const int p = next.fetch_add(1);
      if (p >= num_pairs || first_rc.load() != PHOVO_OK) return;
      rc = phovo_set_source(c, gray0 + (size_t)p * frame, cols, (const char*)depth0 + (size_t)p * frame * delt, depth_type, cols * delt,
                            depth_scale, rows, cols);
      if (!rc) rc = phovo_set_target(c, gray1 + (size_t)p * frame, cols, rows, cols);
      if (!rc && ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE)
        rc = phovo_set_target_depth(c, (const char*)depth1 + (size_t)p * frame * delt, depth_type, cols * delt, depth_scale);
      if (!rc) rc = phovo_set_initial_state(c, initial_states ? initial_states + (size_t)p * 6 : zeros);
      if (!rc) rc = phovo_optimize(c);
      if (rc && rc != PHOVO_E_NUMERIC) { fail(rc); return; }     // a non-finite state is a result (the reference returns NaN too)
      if (states) phovo_get_state(c, states + (size_t)p * 6);
      if (iterations || log_per_pair) {
        int32_t* it = iterations ? iterations + (size_t)p * PHOVO_MAX_LEVELS : nullptr;
        for (int l = 0; it && l < PHOVO_MAX_LEVELS; ++l) it[l] = 0;
        phovo_iter_stats e;
        const int n = phovo_num_iter_stats(c);
        for (int k = 0; k < n; ++k) {
          if (phovo_get_iter_stats(c, k, &e) != PHOVO_OK) continue;
          if (it && e.level >= 0 && e.level < PHOVO_MAX_LEVELS) it[e.level] += 1;
          if (k < log_per_pair) b->h_log[(size_t)p * log_per_pair + k] = e;      // (distinct pairs: no two threads share an entry)
        }
        if (log_per_pair) b->h_log_counts[p] = std::min(n, log_per_pair);
      }
    }
  };
  std::vector<std::thread> threads;
  for (int w = 1; w < workers; ++w) threads.emplace_back(work, b->pool[w]);
  work(b->pool[0]);
  for (auto& t : threads) t.join();
  for (int w = 0; w < workers; ++w) ctx->launches += b->pool[w]->launches, b->pool[w]->launches = 0;
  b->last_pairs = log_per_pair ? num_pairs : 0; b->log_per_pair = log_per_pair; b->log_fetched = log_per_pair > 0;
  b->last_h2d_bytes = 0; b->timed = false; b->last_path = 2;
  if (first_rc.load() != PHOVO_OK) return ctx->fail(first_rc.load(), "batch pool: " + message);
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// The wave path: what the shared-memory-resident kernels cannot take (Ceres mode, the photometric + depth solver,
// blurred or large levels) runs in WAVES of slots.  A slot is a child context used for its device side only: its
// pyramids are built with the general path's kernels (phovo_set_source / phovo_set_target / phovo_set_target_depth,
// asynchronously, kWaveSetupThreads host threads each on a stream of its own), then ONE launch of k_align_slots runs
// the complete coarse-to-fine alignment of every pair of the wave, one CTA per pair (kernels_align.cu).  The slots
// come in two halves: while one half aligns, the other is being set up.  Results equal the per-pair API's up to the
// grouping of the partial sums (one CTA instead of a grid), i.e. to the last bits of the normal equations.
// ---------------------------------------------------------------------------------------------
#ifndef PHOVO_SLOT_MINB
#define PHOVO_SLOT_MINB 2
#endif
static int wave_slots_per_half(const phovo_batch_state* b) { return PHOVO_SLOT_MINB * std::max(1, b->sm_count); }   // CTAs of k_align_slots resident per SM

static int wave_resources(phovo_ctx* ctx, phovo_batch_state* b, int num_pairs, int rows, int cols, int* half_out) {
  for (int t = 0; t < kWaveSetupThreads; ++t)
    if (!b->setup_stream[t]) {
      CK(cudaStreamCreateWithFlags(&b->setup_stream[t], cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&b->ev_setup[t], cudaEventDisableTiming));
    }
  for (int h = 0; h < 2; ++h)
    if (!b->align_stream[h]) {
      CK(cudaStreamCreateWithFlags(&b->align_stream[h], cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&b->ev_wave_done[h], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&b->ev_wave_in[h], cudaEventDisableTiming));
    }
  auto add_slots = [&](int want) -> int {
    while ((int)b->slots.size() < want) {
      phovo_ctx* c = nullptr;
      if (phovo_internal_create_slot(ctx->device, &c) != PHOVO_OK) return ctx->fail(PHOVO_E_CUDA, std::string("batch slots: ") + phovo_last_error(nullptr));
      c->defer_device_input_drain = true;   // the wave's inputs outlive its kernels (batch_waves waits for the wave before they go)
      b->slots.push_back(c);
    }
    return PHOVO_OK;
  };
  int rc = add_slots(1);
  if (rc) return rc;
  // ---- bytes per slot under this configuration and frame size ----
  phovo_ctx* c0 = b->slots[0];
  if (memcmp(&c0->cfg, &ctx->cfg, sizeof(phovo_config)) != 0 && (rc = phovo_set_config(c0, &ctx->cfg))) return ctx->fail(rc, phovo_last_error(c0));
  const size_t need = phovo_internal_slot_bytes(c0, rows, cols);
  // ---- slots per half: the CTAs of k_align_slots one wave keeps resident -- fewer if two halves of them would take more
  // than half of the device memory that is free (counting what the arena already holds) ----
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  size_t budget = (free_b + b->arena_cap) / 2;
  if (const char* e = getenv("PHOVO_WAVE_BUDGET_MB")) budget = std::min(budget, (size_t)std::max(1LL, atoll(e)) << 20);   // test hook
  int half = wave_slots_per_half(b);
  if ((size_t)2 * half * need > budget) half = (int)std::max<size_t>(1, budget / need / 2);
  const int want = num_pairs > half ? 2 * half : num_pairs;
  if ((rc = add_slots(want))) return rc;
  // ---- the arena: ONE allocation, slot s at s * slot_bytes; laid out again whenever configuration, frame size or slot count change ----
  const bool same = want <= b->arena_slots && half == b->wave_half && need == b->slot_bytes && rows == b->arena_rows && cols == b->arena_cols &&
                    memcmp(&b->arena_cfg, &ctx->cfg, sizeof(phovo_config)) == 0;
  if (!same) {
    CK(cudaDeviceSynchronize());                       // nothing of an earlier call is still running on the old layout
    const size_t total = need * (size_t)want;
    if (total > b->arena_cap) {
      cudaFree(b->arena); b->arena = nullptr; b->arena_cap = 0;
      CK(cudaMalloc((void**)&b->arena, total));
      b->arena_cap = total;
    }
    for (size_t s = 0; s < b->slots.size(); ++s) {
      if ((int)s < want) b->slots[s]->arena_reset(b->arena + s * need, need);
      else b->slots[s]->arena_reset(nullptr, 0);       // not part of this layout (never used until the next one)
    }
    b->slot_bytes = need; b->arena_rows = rows; b->arena_cols = cols; b->arena_cfg = ctx->cfg; b->arena_slots = want; b->wave_half = half;
    for (auto& a : b->h_slot_args) memset(&a, 0, sizeof(a));
  }
  if (b->wave_cap < (size_t)half) {
    for (int h = 0; h < 2; ++h) {
      cudaFree(b->d_wave_init[h]); cudaFree(b->d_wave_states[h]); cudaFree(b->d_wave_iters[h]);
      cudaFreeHost(b->h_wave_states[h]); cudaFreeHost(b->h_wave_iters[h]);
      CK(cudaMalloc((void**)&b->d_wave_init[h], sizeof(double) * 6 * half));
      CK(cudaMalloc((void**)&b->d_wave_states[h], sizeof(double) * 6 * half));
      CK(cudaMalloc((void**)&b->d_wave_iters[h], sizeof(int32_t) * PHOVO_MAX_LEVELS * half));
      CK(cudaMallocHost((void**)&b->h_wave_states[h], sizeof(double) * 6 * half));
      CK(cudaMallocHost((void**)&b->h_wave_iters[h], sizeof(int32_t) * PHOVO_MAX_LEVELS * half));
    }
    b->wave_cap = half;
  }
  CK(ensure(&b->d_slot_args, &b->slot_args_cap, (size_t)2 * half));
  if (b->h_slot_args.size() < (size_t)2 * half) b->h_slot_args.resize((size_t)2 * half);
  *half_out = half;
  return PHOVO_OK;
}

static int batch_waves(phovo_ctx* ctx, phovo_batch_state* b, int num_pairs, int rows, int cols, const uint8_t* gray0,
                       const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1, const void* depth1,
                       const double* initial_states, double* states, int32_t* iterations) {
  if (!ctx->have_K) return ctx->fail(PHOVO_E_INVALID, "SetIntrinsicMatrix has not been called");
  if (num_pairs < 1 || rows < 1 || cols < 1) return ctx->fail(PHOVO_E_INVALID, "empty batch");
  const bool bi = ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE;
  if (bi && !depth1)
    return ctx->fail(PHOVO_E_INVALID, "the photometric + depth solver needs the target depth: use phovo_batch_align_with_target_depth");
  // device-resident inputs produced on this context's stream must be complete: the slots run on streams of their own
  CK(cudaStreamSynchronize(ctx->stream));
  int half = 0;
  int rc = wave_resources(ctx, b, num_pairs, rows, cols, &half);
  if (rc) return rc;
  const int waves = (num_pairs + half - 1) / half;
  const size_t frame = (size_t)rows * cols, delt = depth_type == PHOVO_DEPTH_F64 ? 8 : depth_type == PHOVO_DEPTH_F32 ? 4 : 2;
  b->last_h2d_bytes = 0;
  const bool host_in = host_readable(gray0) || host_readable(depth0) || host_readable(gray1) || (bi && host_readable(depth1));

  // the active levels, coarse to fine (AN:502-503; CE:437 skips levels without iterations)
  SlotLevels LS;
  memset(&LS, 0, sizeof(LS));
  bool levels_known = false;

  struct Pending { int start = 0, n = 0; bool active = false; } pend[2];
  const bool trace = getenv("PHOVO_WAVE_TRACE") != nullptr;   // stderr: host set-up time and device align time per wave
  cudaEvent_t tr0[2] = {nullptr, nullptr}, tr1[2] = {nullptr, nullptr};
  if (trace) for (int h = 0; h < 2; ++h) { cudaEventCreate(&tr0[h]); cudaEventCreate(&tr1[h]); }
  auto harvest = [&](int h) -> int {
    if (!pend[h].active) return PHOVO_OK;
    CK(cudaEventSynchronize(b->ev_wave_done[h]));
    if (trace) { float ms = 0.f; cudaEventElapsedTime(&ms, tr0[h], tr1[h]); fprintf(stderr, "[wave] start %d n %d align %.3f ms\n", pend[h].start, pend[h].n, ms); }
    if (states) memcpy(states + (size_t)pend[h].start * 6, b->h_wave_states[h], sizeof(double) * 6 * (size_t)pend[h].n);
    if (iterations) memcpy(iterations + (size_t)pend[h].start * PHOVO_MAX_LEVELS, b->h_wave_iters[h], sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)pend[h].n);
    pend[h].active = false;
    return PHOVO_OK;
  };

  for (int k = 0; k < waves; ++k) {
    const int h = k & 1, start = k * half, n = std::min(half, num_pairs - start);
    if ((rc = harvest(h))) return rc;          // wave k - 2 used these slots (and these input buffers)
    // ---- inputs of the wave on the device ----
    const uint8_t* g0 = gray0 + (size_t)start * frame; const uint8_t* g1 = gray1 + (size_t)start * frame;
    const char* d0 = (const char*)depth0 + (size_t)start * frame * delt;
    const char* d1 = bi ? (const char*)depth1 + (size_t)start * frame * delt : nullptr;
    if (host_in) {
      const size_t nb = (size_t)n * frame;
      CK(ensure(&b->wave_g0[h], &b->wave_g_cap[h], nb)); CK(ensure(&b->wave_g1[h], &b->wave_g1_cap[h], nb));
      CK(ensure(&b->wave_d0[h], &b->wave_d0_cap[h], nb * delt));
      if (bi) CK(ensure(&b->wave_d1[h], &b->wave_d1_cap[h], nb * delt));
      cudaStream_t cs = b->align_stream[h];
      CK(cudaMemcpyAsync(b->wave_g0[h], g0, nb, cudaMemcpyDefault, cs));
      CK(cudaMemcpyAsync(b->wave_g1[h], g1, nb, cudaMemcpyDefault, cs));
      CK(cudaMemcpyAsync(b->wave_d0[h], d0, nb * delt, cudaMemcpyDefault, cs));
      if (bi) CK(cudaMemcpyAsync(b->wave_d1[h], d1, nb * delt, cudaMemcpyDefault, cs));
      CK(cudaEventRecord(b->ev_wave_in[h], cs));
      for (int t = 0; t < kWaveSetupThreads; ++t) CK(cudaStreamWaitEvent(b->setup_stream[t], b->ev_wave_in[h], 0));
      g0 = b->wave_g0[h]; g1 = b->wave_g1[h]; d0 = b->wave_d0[h]; d1 = bi ? b->wave_d1[h] : nullptr;
      b->last_h2d_bytes += nb * (2 + delt * (bi ? 2 : 1));
    }
    // ---- pyramids of the wave's slots: kWaveSetupThreads host threads, each on its own stream ----
    const auto t_setup = std::chrono::steady_clock::now();
    std::atomic<int> first_rc(PHOVO_OK);
    std::mutex mu; std::string message;
    auto work = [&](int t) {
      for (int s = t; s < n; s += kWaveSetupThreads) {
        if (first_rc.load() != PHOVO_OK) return;
        phovo_ctx* c = b->slots[(size_t)h * half + s];
        c->stream = b->setup_stream[t];      // not owned: this thread's stream
        int r = PHOVO_OK;
        if (memcmp(&c->cfg, &ctx->cfg, sizeof(phovo_config)) != 0) r = phovo_set_config(c, &ctx->cfg);
        if (!r) r = phovo_set_intrinsics(c, ctx->K);
        if (!r) r = phovo_set_source(c, g0 + (size_t)s * frame, cols, d0 + (size_t)s * frame * delt, depth_type, cols * delt, depth_scale, rows, cols);
        if (!r) r = phovo_set_target(c, g1 + (size_t)s * frame, cols, rows, cols);
        if (!r && bi) r = phovo_set_target_depth(c, d1 + (size_t)s * frame * delt, depth_type, cols * delt, depth_scale);
        if (r) {
          std::lock_guard<std::mutex> g(mu);
          if (first_rc.load() == PHOVO_OK) { first_rc.store(r); message = phovo_last_error(c); }
          return;
        }
      }
    };
    {
      std::vector<std::thread> threads;
      const int nt = std::min(kWaveSetupThreads, n);
      for (int t = 1; t < nt; ++t) threads.emplace_back(work, t);
      work(0);
      for (auto& t : threads) t.join();
    }
    if (first_rc.load() != PHOVO_OK) {
      cudaDeviceSynchronize();
      return ctx->fail(first_rc.load(), "batch slots: " + message);
    }
    if (trace) fprintf(stderr, "[wave] start %d n %d host set-up %.3f ms\n", start, n, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_setup).count());
    cudaStream_t as = b->align_stream[h];
    for (int t = 0; t < kWaveSetupThreads; ++t) {
      CK(cudaEventRecord(b->ev_setup[t], b->setup_stream[t]));
      CK(cudaStreamWaitEvent(as, b->ev_setup[t], 0));
    }
    // ---- slot table (the buffers of a slot stay where they are once allocated for a frame size) ----
    bool table_changed = false;
    for (int s = 0; s < n; ++s) {
      phovo_ctx* c = b->slots[(size_t)h * half + s];
      SlotArgs A;
      memset(&A, 0, sizeof(A));
      for (int l = 0; l < c->cfg.num_levels; ++l) A.P[l] = c->level_ptrs(l);
      A.pose = c->d_pose; A.partials = c->partials;
      SlotArgs& cached = b->h_slot_args[(size_t)h * half + s];
      if (memcmp(&cached, &A, sizeof(A)) != 0) { cached = A; table_changed = true; }
      ctx->launches += c->launches; c->launches = 0;
    }
    if (table_changed) {
      CK(cudaMemcpyAsync(b->d_slot_args + (size_t)h * half, b->h_slot_args.data() + (size_t)h * half, sizeof(SlotArgs) * (size_t)n, cudaMemcpyHostToDevice, as));
      CK(cudaStreamSynchronize(as));   // pageable source: keep it simple, this happens once per frame size
    }
    if (!levels_known) {
      const phovo_ctx* c0 = b->slots[(size_t)h * half];
      for (int level = ctx->cfg.num_levels - 1; level >= 0; --level) {
        const int M = ctx->cfg.max_num_iterations[level];
        if (!(M > 0)) continue;
        const int a = LS.count++;
        LS.L[a] = c0->level_params(level);
        LmParams& lm = LS.lm[a];
        lm.function_tolerance = ctx->cfg.function_tolerance[level]; lm.gradient_tolerance = ctx->cfg.gradient_tolerance[level];
        lm.parameter_tolerance = ctx->cfg.parameter_tolerance[level]; lm.initial_radius = ctx->cfg.initial_trust_region_radius[level];
        lm.max_radius = ctx->cfg.max_trust_region_radius[level]; lm.min_radius = ctx->cfg.min_trust_region_radius[level];
        lm.min_relative_decrease = ctx->cfg.min_relative_decrease[level]; lm.max_iterations = M;
      }
      levels_known = true;
    }
    // ---- one launch aligns the wave; results to pinned memory ----
    const double* d_init = nullptr;
    if (initial_states) {
      CK(cudaMemcpyAsync(b->d_wave_init[h], initial_states + (size_t)start * 6, sizeof(double) * 6 * (size_t)n, cudaMemcpyDefault, as));
      d_init = b->d_wave_init[h];
    }
    if (trace) cudaEventRecord(tr0[h], as);
    // CTAs per pair: one when the wave fills the GPU; a small wave gives every pair a thread-block cluster (2, 4 or 8 CTAs,
    // cluster barriers) so that the SMs it would leave idle shorten the wave instead
    int cluster = 1;
    for (int c = 8; c > 1; c >>= 1)
      if (n * c <= PHOVO_SLOT_MINB * b->sm_count) { cluster = c; break; }
    if (const char* e = getenv("PHOVO_WAVE_CLUSTER")) { const int v = atoi(e); if (v == 1 || v == 2 || v == 4 || v == 8) cluster = v; }   // experiment hook
    int launched = launch_align_slots(as, ctx->cfg.mode, LS, b->d_slot_args + (size_t)h * half, n, d_init, cluster);
    if (launched < 0 && cluster > 1) { cudaGetLastError(); launched = launch_align_slots(as, ctx->cfg.mode, LS, b->d_slot_args + (size_t)h * half, n, d_init, 1); }
    if (launched < 0) return ctx->cuda_fail("k_align_slots", cudaGetLastError());
    ctx->launches += launched;
    if (trace) cudaEventRecord(tr1[h], as);
    ctx->launches += launch_gather_slots(as, b->d_slot_args + (size_t)h * half, n, b->d_wave_states[h], b->d_wave_iters[h]);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(b->h_wave_states[h], b->d_wave_states[h], sizeof(double) * 6 * (size_t)n, cudaMemcpyDeviceToHost, as));
    CK(cudaMemcpyAsync(b->h_wave_iters[h], b->d_wave_iters[h], sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)n, cudaMemcpyDeviceToHost, as));
    CK(cudaEventRecord(b->ev_wave_done[h], as));
    pend[h].start = start; pend[h].n = n; pend[h].active = true;
  }
  // in wave order: the older half first
  const int last = (waves - 1) & 1;
  if ((rc = harvest(1 - last))) return rc;
  if ((rc = harvest(last))) return rc;
  if (trace) for (int h = 0; h < 2; ++h) { cudaEventDestroy(tr0[h]); cudaEventDestroy(tr1[h]); }
  b->last_pairs = 0; b->log_per_pair = 0; b->log_fetched = false; b->timed = false; b->last_path = 3;
  return PHOVO_OK;
}

// What the shared-memory-resident kernels do not take.  A wave gives every pair one CTA -- or, while the wave is too small
// to fill the GPU, one thread-block cluster of 2 / 4 / 8 CTAs -- and lasts as long as its slowest pair takes on that.  The
// pool of per-pair contexts gives every pair the whole GPU, one after the other (about 0.1-0.2 ms per pair).  Measured on
// B200 at 640x480 (tools/wave_cluster_sweep.py, profiles/r02_wave_cluster_sweep.jsonl): the pool wins below about 12 pairs
// (Ceres-mode solver) / 24 pairs (photometric + depth solver), the waves above.  Debug flag 4 forces the pool, 8 the
// waves.  Same iteration counts either way, states equal to the last bits.
static int batch_other(phovo_ctx* ctx, phovo_batch_state* b, int num_pairs, int rows, int cols, const uint8_t* gray0,
                       const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1, const void* depth1,
                       const double* initial_states, double* states, int32_t* iterations) {
  const int min_pairs = ctx->cfg.mode == PHOVO_MODE_CERES ? 16 : 24;
  // (the per-iteration stats are a debugging aid: a batch that records them takes the pool, whose children keep logs)
  const bool pool = (b->debug_flags & 4) || b->record_stats || (!(b->debug_flags & 8) && num_pairs < min_pairs);
  if (pool) return batch_general(ctx, b, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, depth1, initial_states, states, iterations);
  return batch_waves(ctx, b, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, depth1, initial_states, states, iterations);
}

// true if the batch must take the wave (or pool) path (see make_params for what the shared-memory-resident kernels accept)
static bool needs_pool(phovo_ctx* ctx, int num_pairs, int rows, int cols, int log_cap, BatchParams* bp, size_t* smem, int* rc_out) {
  if (ctx->cfg.mode == PHOVO_MODE_CERES || ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE) { *rc_out = PHOVO_OK; return true; }
  *rc_out = make_params(ctx, num_pairs, rows, cols, log_cap, bp, smem);
  if (*rc_out == PHOVO_E_UNSUPPORTED) { *rc_out = PHOVO_OK; return true; }
  return false;
}

extern "C" int phovo_batch_last_path(const phovo_ctx* ctx) { return ctx && ctx->batch ? ctx->batch->last_path : 0; }

extern "C" int phovo_batch_align_device(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0,
                                        const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1,
                                        const double* initial_states, double* states, int32_t* iters) {
  if (!ctx || !gray0 || !depth0 || !gray1 || !states || !iters) return PHOVO_E_INVALID;
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  CK(cudaSetDevice(ctx->device));
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  int log_cap = 0;
  if ((rc = prepare_log(ctx, b, num_pairs, &log_cap))) return rc;
  BatchParams bp; size_t smem = 0;
  if (needs_pool(ctx, num_pairs, rows, cols, log_cap, &bp, &smem, &rc)) {
    // pool path: synchronous; results go to the caller's device arrays through host temporaries
    std::vector<double> hs((size_t)num_pairs * 6); std::vector<int32_t> hi((size_t)num_pairs * PHOVO_MAX_LEVELS);
    if ((rc = batch_other(ctx, b, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, nullptr, initial_states, hs.data(), hi.data()))) return rc;
    CK(cudaMemcpyAsync(states, hs.data(), sizeof(double) * hs.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(iters, hi.data(), sizeof(int32_t) * hi.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return PHOVO_OK;
  }
  if (rc) return rc;
  b->last_path = 1;
  CK(ensure(&b->store, &b->store_cap, (size_t)bp.record_bytes * num_pairs + kBatchStoreSlackBytes));
  return run_device(ctx, b, bp, smem, ctx->stream, gray0, depth0, depth_type, depth_scale, gray1, b->store,
                    initial_states, states, iters, log_cap ? b->log : nullptr, log_cap ? b->log_counts : nullptr);
}

static bool is_device_pointer(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

extern "C" int phovo_batch_align(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0,
                                 const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1,
                                 const double* initial_states, double* states, int32_t* iterations) {
  if (!ctx || !gray0 || !depth0 || !gray1) return PHOVO_E_INVALID;
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  CK(cudaSetDevice(ctx->device));
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  int log_cap = 0;
  if ((rc = prepare_log(ctx, b, num_pairs, &log_cap))) return rc;
  BatchParams bp; size_t smem = 0;
  if (needs_pool(ctx, num_pairs, rows, cols, log_cap, &bp, &smem, &rc))
    return batch_other(ctx, b, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, nullptr, initial_states, states, iterations);
  if (rc) return rc;
  b->last_path = 1;
  CK(ensure(&b->states, &b->states_cap, (size_t)num_pairs * 6));
  CK(ensure(&b->iters, &b->iters_cap, (size_t)num_pairs * PHOVO_MAX_LEVELS));
  CK(ensure(&b->store, &b->store_cap, (size_t)bp.record_bytes * num_pairs + kBatchStoreSlackBytes));
  const double* d_init = nullptr;
  if (initial_states) {
    CK(ensure(&b->init, &b->init_cap, (size_t)num_pairs * 6));
    CK(cudaMemcpyAsync(b->init, initial_states, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
    d_init = b->init;
  }
  if (b->h_out_cap < (size_t)num_pairs) {
    cudaFreeHost(b->h_states_pinned); cudaFreeHost(b->h_iters_pinned);
    b->h_states_pinned = nullptr; b->h_iters_pinned = nullptr; b->h_out_cap = 0;
    CK(cudaMallocHost((void**)&b->h_states_pinned, sizeof(double) * 6 * (size_t)num_pairs));
    CK(cudaMallocHost((void**)&b->h_iters_pinned, sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs));
    b->h_out_cap = num_pairs;
  }
  const bool on_device = is_device_pointer(gray0) && is_device_pointer(depth0) && is_device_pointer(gray1);
  const size_t frame = (size_t)rows * cols, delt = depth_elt(depth_type);
  if (on_device) {
    rc = run_device(ctx, b, bp, smem, ctx->stream, gray0, depth0, depth_type, depth_scale, gray1, b->store, d_init,
                    b->states, b->iters, log_cap ? b->log : nullptr, log_cap ? b->log_counts : nullptr);
    if (rc) return rc;
  } else {
    // chunked, double-buffered upload: copies run on copy_stream, kernels on ctx->stream
    // a chunk is four waves of persistent CTAs: large enough to amortise the ragged tail of a
    // wave (pairs need different iteration counts), small enough to overlap with the next copy
    const int chunk = std::max(1, std::min(num_pairs, 4 * b->sm_count));
    for (int s = 0; s < 2; ++s) {
      CK(ensure(&b->stage_g0[s], &b->stage_cap_g[s], frame * chunk));
      CK(ensure(&b->stage_g1[s], &b->stage_cap_g1[s], frame * chunk));
      CK(ensure(&b->stage_d[s], &b->stage_cap_d[s], frame * chunk * delt));
    }
    CK(cudaMemsetAsync(b->iters, 0, sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs, ctx->stream));
    int period, keep_begin, keep;
    row_compaction(ctx, rows, &period, &keep_begin, &keep);
    b->last_h2d_bytes = 0;
    int slot = 0, used[2] = {0, 0};
    for (int p0 = 0; p0 < num_pairs; p0 += chunk, slot ^= 1) {
      const int np = std::min(chunk, num_pairs - p0);
      if (used[slot]) CK(cudaStreamWaitEvent(b->copy_stream, b->ev_consumed[slot], 0));
      if (period) {
        // one strided copy per image stack: `keep` of every `period` rows, frames are back to back
        const size_t groups = (size_t)(rows / period) * np;
        const size_t gw = (size_t)keep * cols, gp = (size_t)period * cols, go = (size_t)keep_begin * cols;
        CK(cudaMemcpy2DAsync(b->stage_g0[slot], gw, gray0 + (size_t)p0 * frame + go, gp, gw, groups, cudaMemcpyHostToDevice, b->copy_stream));
        CK(cudaMemcpy2DAsync(b->stage_g1[slot], gw, gray1 + (size_t)p0 * frame + go, gp, gw, groups, cudaMemcpyHostToDevice, b->copy_stream));
        CK(cudaMemcpy2DAsync(b->stage_d[slot], gw * delt, (const char*)depth0 + ((size_t)p0 * frame + go) * delt, gp * delt, gw * delt, groups, cudaMemcpyHostToDevice, b->copy_stream));
        b->last_h2d_bytes += groups * gw * (2 + delt);
      } else {
        CK(cudaMemcpyAsync(b->stage_g0[slot], gray0 + (size_t)p0 * frame, frame * np, cudaMemcpyHostToDevice, b->copy_stream));
        CK(cudaMemcpyAsync(b->stage_g1[slot], gray1 + (size_t)p0 * frame, frame * np, cudaMemcpyHostToDevice, b->copy_stream));
        CK(cudaMemcpyAsync(b->stage_d[slot], (const char*)depth0 + (size_t)p0 * frame * delt, frame * np * delt, cudaMemcpyHostToDevice, b->copy_stream));
        b->last_h2d_bytes += (size_t)frame * np * (2 + delt);
      }
      CK(cudaEventRecord(b->ev_copied[slot], b->copy_stream));
      CK(cudaStreamWaitEvent(ctx->stream, b->ev_copied[slot], 0));
      BatchParams cp = bp;
      cp.num_pairs = np;
      cp.src_period = period; cp.src_keep_begin = keep_begin; cp.src_keep = keep;
      rc = run_device(ctx, b, cp, smem, ctx->stream, b->stage_g0[slot], b->stage_d[slot], depth_type, depth_scale, b->stage_g1[slot],
                      b->store + (size_t)p0 * bp.record_bytes, d_init ? d_init + (size_t)p0 * 6 : nullptr,
                      b->states + (size_t)p0 * 6, b->iters + (size_t)p0 * PHOVO_MAX_LEVELS,
                      log_cap ? b->log + (size_t)p0 * log_cap : nullptr, log_cap ? b->log_counts + p0 : nullptr);
      if (rc) return rc;
      CK(cudaEventRecord(b->ev_consumed[slot], ctx->stream));
      used[slot] = 1;
    }
  }
  CK(cudaMemcpyAsync(b->h_states_pinned, b->states, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(b->h_iters_pinned, b->iters, sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (states) memcpy(states, b->h_states_pinned, sizeof(double) * 6 * (size_t)num_pairs);
  if (iterations) memcpy(iterations, b->h_iters_pinned, sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs);
  return PHOVO_OK;
}

static int fetch_log(const phovo_ctx* cctx) {
  phovo_ctx* ctx = const_cast<phovo_ctx*>(cctx);
  phovo_batch_state* b = ctx->batch;
  if (!b || !b->log_per_pair) return PHOVO_E_INVALID;
  if (b->log_fetched) return PHOVO_OK;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  b->h_log.resize((size_t)b->last_pairs * b->log_per_pair);
  b->h_log_counts.resize(b->last_pairs);
  CK(cudaMemcpy(b->h_log.data(), b->log, sizeof(phovo_iter_stats) * b->h_log.size(), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(b->h_log_counts.data(), b->log_counts, sizeof(int32_t) * b->last_pairs, cudaMemcpyDeviceToHost));
  b->log_fetched = true;
  return PHOVO_OK;
}

extern "C" int phovo_batch_num_iter_stats(const phovo_ctx* ctx, int pair) {
  if (!ctx || !ctx->batch) return 0;
  if (fetch_log(ctx) != PHOVO_OK) return 0;
  if (pair < 0 || pair >= ctx->batch->last_pairs) return 0;
  return std::min(ctx->batch->h_log_counts[pair], ctx->batch->log_per_pair);
}

extern "C" int phovo_batch_get_iter_stats(const phovo_ctx* ctx, int pair, int index, phovo_iter_stats* out) {
  if (!ctx || !out || !ctx->batch) return PHOVO_E_INVALID;
  const int n = phovo_batch_num_iter_stats(ctx, pair);
  if (index < 0 || index >= n) return PHOVO_E_INVALID;
  *out = ctx->batch->h_log[(size_t)pair * ctx->batch->log_per_pair + index];
  return PHOVO_OK;
}

extern "C" int phovo_batch_align_with_target_depth(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0,
                                                   const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1,
                                                   const void* depth1, const double* initial_states, double* states, int32_t* iterations) {
  if (!ctx || !gray0 || !depth0 || !gray1 || !depth1) return PHOVO_E_INVALID;
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if (ctx->cfg.mode != PHOVO_MODE_BIOBJECTIVE)      // the other solvers ignore the target depth, like the reference (AN:484)
    return phovo_batch_align(ctx, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, initial_states, states, iterations);
  CK(cudaSetDevice(ctx->device));
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  return batch_other(ctx, b, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, depth1, initial_states, states, iterations);
}

// ---------------------------------------------------------------------------------------------
// phovo::warpImage (BASE:73-134) + the apps' cv::absdiff for many pairs (kernels_pyramid.cu: k_warp_splat, k_warp_resolve)
// ---------------------------------------------------------------------------------------------
// Pairs per chunk: the chunk's keys (4 B per pixel) fit in half of the L2, so that they are cleared, bid on and read back
// there and HBM sees only the images (640x480 on a 126 MB L2: 51 pairs).
static int warp_chunk_pairs(const phovo_batch_state* b, size_t n, int num_pairs) {
  const size_t fit = (size_t)std::max(b->l2_bytes, 1) / 2 / (n * sizeof(uint32_t));
  return (int)std::max<size_t>(1, std::min<size_t>({fit, (size_t)num_pairs, 65535}));
}

static WarpImages offset_pairs(WarpImages W, int p0) {
  W.gray += p0 * W.gray_pair;
  W.depth = (const char*)W.depth + p0 * W.depth_pair;
  if (W.target) W.target += p0 * W.target_pair;
  if (W.warped) W.warped += p0 * W.warped_pair;
  if (W.diff) W.diff += p0 * W.diff_pair;
  if (W.num_landed) W.num_landed += p0;
  if (W.sum_abs_diff) W.sum_abs_diff += p0;
  return W;
}

// Enqueues the warp of `num_pairs` pairs described by W (device pointers; W.rts is set here from `rts`, host or device
// [num_pairs][16]) in chunks of warp_chunk_pairs.  Debug flag 16: the keys are cleared with a memset before each chunk
// instead of by the resolve pass (same results; a measurement hook).
int phovo_internal_warp_images(phovo_ctx* ctx, WarpImages W, int src_type, const WarpIntrinsics& I, int num_pairs, const double* rts) {
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  const size_t n = (size_t)W.rows * W.cols;
  const int chunk = warp_chunk_pairs(b, n, num_pairs);
  if (b->warp_keys_cap < (size_t)chunk * n) {
    CK(ensure(&b->warp_keys, &b->warp_keys_cap, (size_t)chunk * n));
    b->warp_keys_clean = false;
  }
  const bool memset_each = (b->debug_flags & 16) != 0;
  if (!b->warp_keys_clean && !memset_each) CK(cudaMemsetAsync(b->warp_keys, 0, b->warp_keys_cap * sizeof(uint32_t), ctx->stream));
  b->warp_keys_clean = false;   // until every launch below has been enqueued
  CK(ensure(&b->warp_rts, &b->warp_rts_cap, (size_t)num_pairs * 16));
  CK(cudaMemcpyAsync(b->warp_rts, rts, sizeof(double) * 16 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  for (int p0 = 0; p0 < num_pairs; p0 += chunk) {
    const int np = std::min(chunk, num_pairs - p0);
    WarpImages C = offset_pairs(W, p0);
    C.rts = b->warp_rts + (size_t)p0 * 16;
    if (memset_each) CK(cudaMemsetAsync(b->warp_keys, 0, (size_t)np * n * sizeof(uint32_t), ctx->stream));
    ctx->launches += launch_warp_images(ctx->stream, C, src_type, I, np, b->warp_keys, !memset_each) + (memset_each ? 1 : 0);
    CK(cudaGetLastError());
  }
  b->warp_keys_clean = !memset_each;
  return PHOVO_OK;
}

extern "C" int phovo_batch_warp_image(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0, const void* depth0,
                                      int depth_type, double depth_scale, const double* rts, const double K[9], int level,
                                      const uint8_t* gray1, uint8_t* warped, uint8_t* diff, int32_t* num_landed, int64_t* sum_abs_diff) {
  if (!ctx) return PHOVO_E_INVALID;
  if (!gray0 || !depth0 || !rts || !K) return ctx->fail(PHOVO_E_INVALID, "gray0, depth0, rts and K are required");
  if (num_pairs < 1 || rows < 1 || cols < 1 || level < 0 || level > 30) return ctx->fail(PHOVO_E_INVALID, "bad batch size, image size or level");
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if ((diff || sum_abs_diff) && !gray1) return ctx->fail(PHOVO_E_INVALID, "diff and sum_abs_diff need gray1");
  if (!warped && !diff && !num_landed && !sum_abs_diff) return ctx->fail(PHOVO_E_INVALID, "no output requested");
  const size_t n = (size_t)rows * cols;
  if (n > (size_t)INT32_MAX) return ctx->fail(PHOVO_E_UNSUPPORTED, "warpImage: frames of 2^31 pixels or more");
  CK(cudaSetDevice(ctx->device));
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  const size_t delt = depth_elt(depth_type);
  const bool want_sum = sum_abs_diff != nullptr, want_summary = num_landed || sum_abs_diff;
  const uint8_t* target = diff || want_sum ? gray1 : nullptr;
  const bool in_dev = is_device_pointer(gray0) && is_device_pointer(depth0) && (!target || is_device_pointer(target));
  const bool w_host = warped && !is_device_pointer(warped), d_host = diff && !is_device_pointer(diff);
  if (want_summary) {
    CK(ensure(&b->warp_landed, &b->warp_landed_cap, (size_t)num_pairs));
    CK(ensure(&b->warp_sum, &b->warp_sum_cap, (size_t)num_pairs));
    CK(cudaMemsetAsync(b->warp_landed, 0, sizeof(int32_t) * num_pairs, ctx->stream));
    CK(cudaMemsetAsync(b->warp_sum, 0, sizeof(int64_t) * num_pairs, ctx->stream));
  }
  WarpImages W;
  memset(&W, 0, sizeof(W));
  W.rows = rows; W.cols = cols;
  W.gray = gray0; W.gray_step = cols; W.gray_pair = n;
  W.depth = depth0; W.depth_step = cols * delt; W.depth_pair = n * delt;
  W.depth_scale = depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0;
  W.target = target; W.target_step = cols; W.target_pair = n;
  W.warped = warped; W.warped_step = cols; W.warped_pair = n;
  W.diff = diff; W.diff_step = cols; W.diff_pair = n;
  W.num_landed = want_summary ? b->warp_landed : nullptr;
  W.sum_abs_diff = want_sum ? b->warp_sum : nullptr;
  const double s = pow(2, level);                                  // BASE:89-94: K / 2^level
  WarpIntrinsics I;
  I.fx = K[0] / s; I.fy = K[4] / s; I.ox = K[2] / s; I.oy = K[5] / s;
  I.inv_fx = 1.f / I.fx; I.inv_fy = 1.f / I.fy;                    // BASE:91-92
  const int src = depth_type == PHOVO_DEPTH_F64 ? SRC_F64 : depth_type == PHOVO_DEPTH_F32 ? SRC_F32 : SRC_U16;
  if (in_dev && !w_host && !d_host) {
    if ((rc = phovo_internal_warp_images(ctx, W, src, I, num_pairs, rts))) return rc;
  } else {
    // host inputs (all rows: the warp reads every one) and host outputs go through device buffers of one chunk
    const int chunk = warp_chunk_pairs(b, n, num_pairs);
    const size_t cn = (size_t)chunk * n;
    if (!in_dev) {
      CK(ensure(&b->warp_io[0], &b->warp_io_cap[0], cn));
      CK(ensure(&b->warp_depth, &b->warp_depth_cap, cn * delt));
      if (target) CK(ensure(&b->warp_io[1], &b->warp_io_cap[1], cn));
    }
    if (w_host) CK(ensure(&b->warp_io[2], &b->warp_io_cap[2], cn));
    if (d_host) CK(ensure(&b->warp_io[3], &b->warp_io_cap[3], cn));
    for (int p0 = 0; p0 < num_pairs; p0 += chunk) {
      const int np = std::min(chunk, num_pairs - p0);
      WarpImages C = offset_pairs(W, p0);
      if (!in_dev) {
        CK(cudaMemcpyAsync(b->warp_io[0], C.gray, n * np, cudaMemcpyDefault, ctx->stream));
        CK(cudaMemcpyAsync(b->warp_depth, C.depth, n * np * delt, cudaMemcpyDefault, ctx->stream));
        if (target) CK(cudaMemcpyAsync(b->warp_io[1], C.target, n * np, cudaMemcpyDefault, ctx->stream));
        C.gray = b->warp_io[0]; C.depth = b->warp_depth;
        if (target) C.target = b->warp_io[1];
      }
      if (w_host) C.warped = b->warp_io[2];
      if (d_host) C.diff = b->warp_io[3];
      if ((rc = phovo_internal_warp_images(ctx, C, src, I, np, rts + (size_t)p0 * 16))) return rc;
      if (w_host) CK(cudaMemcpyAsync(warped + (size_t)p0 * n, C.warped, n * np, cudaMemcpyDeviceToHost, ctx->stream));
      if (d_host) CK(cudaMemcpyAsync(diff + (size_t)p0 * n, C.diff, n * np, cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  if (num_landed) CK(cudaMemcpyAsync(num_landed, b->warp_landed, sizeof(int32_t) * num_pairs, cudaMemcpyDefault, ctx->stream));
  if (sum_abs_diff) CK(cudaMemcpyAsync(sum_abs_diff, b->warp_sum, sizeof(int64_t) * num_pairs, cudaMemcpyDefault, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// Normal equations of many pairs at given states (kernels_eval.cu): what phovo_eval_normal_equations gives pair by pair
// ---------------------------------------------------------------------------------------------
// Pairs per chunk: the chunk's winner keys (4 B per pixel), validity flags (1 B) and, above level 0, its level records
// fit in half of the L2, so that the two passes find them there (640x480 level 0 on a 126 MB L2: 41 pairs).
static int eval_chunk_pairs(const phovo_batch_state* b, size_t n, unsigned long long record_bytes, int num_pairs) {
  const size_t fit = (size_t)std::max(b->l2_bytes, 1) / 2 / (n * (sizeof(uint32_t) + 1) + record_bytes);
  return (int)std::max<size_t>(1, std::min<size_t>({fit, (size_t)num_pairs, 65535}));
}

extern "C" int phovo_batch_eval_normal_equations(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0,
                                                 const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1,
                                                 const double* states, int level, double* H, double* g, double* cost,
                                                 int32_t* num_valid) {
  if (!ctx) return PHOVO_E_INVALID;
  if (!gray0 || !depth0 || !gray1 || !states) return ctx->fail(PHOVO_E_INVALID, "gray0, depth0, gray1 and states are required");
  if (!ctx->have_K) return ctx->fail(PHOVO_E_INVALID, "SetIntrinsicMatrix has not been called");
  if (ctx->cfg.mode == PHOVO_MODE_CERES || ctx->cfg.mode == PHOVO_MODE_BIOBJECTIVE)
    return ctx->fail(PHOVO_E_UNSUPPORTED, "batched normal equations: analytic modes only");
  if (num_pairs < 1 || rows < 1 || cols < 1 || level < 0 || level >= ctx->cfg.num_levels)
    return ctx->fail(PHOVO_E_INVALID, "bad batch size, image size or level");
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if (!H && !g && !cost && !num_valid) return ctx->fail(PHOVO_E_INVALID, "no output requested");
  const size_t n = (size_t)rows * cols;
  if (n > (size_t)INT32_MAX) return ctx->fail(PHOVO_E_UNSUPPORTED, "batched normal equations: frames of 2^31 pixels or more");
  BatchParams bp;
  memset(&bp, 0, sizeof(bp));
  bp.rows = rows; bp.cols = cols; bp.num_active = 1; bp.mode = ctx->cfg.mode;
  bp.min_depth = ctx->cfg.min_depth; bp.max_depth = ctx->cfg.max_depth;
  unsigned long long record_bytes = 0;
  int rc = fill_level(ctx, rows, cols, level, 0, &bp, &record_bytes);
  if (rc) return rc;
  bp.record_bytes = record_bytes;
  const bool records = level > 0;                   // level 0 is read straight from the caller's frames
  CK(cudaSetDevice(ctx->device));
  phovo_batch_state* b;
  if ((rc = get_state(ctx, &b))) return rc;
  const int ln = bp.lrows[0] * bp.lcols[0];
  EvalLevel E;
  memset(&E, 0, sizeof(E));
  E.L.fx = bp.fx[0]; E.L.fy = bp.fy[0]; E.L.ox = bp.ox[0]; E.L.oy = bp.oy[0]; E.L.inv_fx = bp.inv_fx[0]; E.L.inv_fy = bp.inv_fy[0];
  E.L.min_depth = bp.min_depth; E.L.max_depth = bp.max_depth;
  E.L.lambda = bp.lambda[0]; E.L.min_grad_norm = bp.min_grad[0];
  E.L.rows = bp.lrows[0]; E.L.cols = bp.lcols[0];
  E.L.mode = bp.mode; E.L.level = level; E.L.row_begin = 0; E.L.row_end = E.L.rows;
  E.grad_k = bp.grad_k[0];
  E.tiles = (ln + kEvalTile - 1) / kEvalTile;
  E.depth_scale = depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0;
  E.record_bytes = record_bytes; E.off_I0 = bp.off_I0[0]; E.off_I1 = bp.off_I1[0]; E.off_D0 = bp.off_D0[0];
  const int src = depth_type == PHOVO_DEPTH_F64 ? SRC_F64 : depth_type == PHOVO_DEPTH_F32 ? SRC_F32 : SRC_U16;
  const size_t delt = depth_elt(depth_type);
  const int chunk = eval_chunk_pairs(b, (size_t)ln, records ? record_bytes : 0, num_pairs);
  const size_t ck = (size_t)chunk * ln;
  if (b->eval_keys_cap < ck) {
    CK(ensure(&b->eval_keys, &b->eval_keys_cap, ck));
    b->eval_keys_clean = false;
  }
  CK(ensure(&b->eval_valid, &b->eval_valid_cap, ck));
  CK(ensure(&b->eval_partials, &b->eval_partials_cap, (size_t)chunk * E.tiles * PHOVO_ACC_STRIDE));
  if (records) CK(ensure(&b->eval_store, &b->eval_store_cap, (size_t)chunk * record_bytes));
  CK(ensure(&b->eval_states, &b->eval_states_cap, (size_t)num_pairs * 6));
  CK(ensure(&b->eval_poses, &b->eval_poses_cap, (size_t)num_pairs));
  CK(ensure(&b->eval_out, &b->eval_out_cap, (size_t)num_pairs * 28));
  CK(ensure(&b->eval_nvalid, &b->eval_nvalid_cap, (size_t)num_pairs));
  const bool in_dev = is_device_pointer(gray0) && is_device_pointer(depth0) && is_device_pointer(gray1);
  if (!in_dev) {   // host frames go through device buffers of one chunk (every row: level 0 and the pyramid read them all)
    CK(ensure(&b->warp_io[0], &b->warp_io_cap[0], (size_t)chunk * n));
    CK(ensure(&b->warp_io[1], &b->warp_io_cap[1], (size_t)chunk * n));
    CK(ensure(&b->warp_depth, &b->warp_depth_cap, (size_t)chunk * n * delt));
  }
  if (!b->eval_keys_clean) CK(cudaMemsetAsync(b->eval_keys, 0, b->eval_keys_cap * sizeof(uint32_t), ctx->stream));
  b->eval_keys_clean = false;   // until every launch below has been enqueued
  CK(cudaMemcpyAsync(b->eval_states, states, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  ctx->launches += launch_eval_poses(ctx->stream, b->eval_states, num_pairs, b->eval_poses);
  double* dH = b->eval_out; double* dg = dH + (size_t)num_pairs * 21; double* dcost = dg + (size_t)num_pairs * 6;
  E.keys = b->eval_keys; E.valid = b->eval_valid; E.partials = b->eval_partials; E.store = b->eval_store;
  for (int p0 = 0; p0 < num_pairs; p0 += chunk) {
    const int np = std::min(chunk, num_pairs - p0);
    const uint8_t* c_g0 = gray0 + (size_t)p0 * n; const uint8_t* c_g1 = gray1 + (size_t)p0 * n;
    const void* c_d = (const char*)depth0 + (size_t)p0 * n * delt;
    if (!in_dev) {
      CK(cudaMemcpyAsync(b->warp_io[0], c_g0, n * np, cudaMemcpyDefault, ctx->stream));
      CK(cudaMemcpyAsync(b->warp_io[1], c_g1, n * np, cudaMemcpyDefault, ctx->stream));
      CK(cudaMemcpyAsync(b->warp_depth, c_d, n * np * delt, cudaMemcpyDefault, ctx->stream));
      c_g0 = b->warp_io[0]; c_g1 = b->warp_io[1]; c_d = b->warp_depth;
    }
    if (records) {
      bp.num_pairs = np;
      ctx->launches += launch_batch_pyramid(ctx->stream, bp, c_g0, c_d, src, E.depth_scale, c_g1, b->eval_store);
    } else {
      E.gray0 = c_g0; E.gray1 = c_g1; E.depth = c_d;
    }
    E.poses = b->eval_poses + p0;
    ctx->launches += launch_eval_normal_equations(ctx->stream, E, src, records, np, dH + (size_t)p0 * 21, dg + (size_t)p0 * 6,
                                                  dcost + p0, b->eval_nvalid + p0);
    CK(cudaGetLastError());
  }
  b->eval_keys_clean = true;
  if (H) CK(cudaMemcpyAsync(H, dH, sizeof(double) * 21 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  if (g) CK(cudaMemcpyAsync(g, dg, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  if (cost) CK(cudaMemcpyAsync(cost, dcost, sizeof(double) * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  if (num_valid) CK(cudaMemcpyAsync(num_valid, b->eval_nvalid, sizeof(int32_t) * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}
