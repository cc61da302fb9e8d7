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
#include <memory>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

#include "phovo_batch.h"
#include "phovo_ctx.h"

using namespace phovo;

constexpr int kWaveSetupThreads = 4;   // host threads (and streams) that build the pyramids of a wave's slots

// [pairs][rows * cols] frame stacks of a call: gray0, gray1, depth0, depth1 (nullptr: not part of the call)
struct Frames {
  const uint8_t* gray0; const uint8_t* gray1; const void* depth0; const void* depth1;
  Frames offset(size_t p0, size_t frame, size_t delt) const {
    return {gray0 + p0 * frame, gray1 ? gray1 + p0 * frame : nullptr, (const char*)depth0 + p0 * frame * delt,
            depth1 ? (const char*)depth1 + p0 * frame * delt : nullptr};
  }
};

// Device copies of a chunk of host frames, for the stacks a call has
struct FrameStage {
  DeviceArray<uint8_t> gray0, gray1;
  DeviceArray<char> depth0, depth1;
  cudaError_t reserve(const Frames& which, size_t pairs, size_t frame, size_t delt) {
    cudaError_t e = gray0.ensure(pairs * frame);
    if (e == cudaSuccess && which.gray1) e = gray1.ensure(pairs * frame);
    if (e == cudaSuccess) e = depth0.ensure(pairs * frame * delt);
    if (e == cudaSuccess && which.depth1) e = depth1.ensure(pairs * frame * delt);
    return e;
  }
  // Pairs [p0, p0 + np) of `in` on the device: with `copy` copied in here on `stream`, otherwise used in place
  cudaError_t stage(bool copy, const Frames& in, size_t frame, size_t delt, int p0, int np, cudaStream_t stream, Frames* out) {
    const Frames f = in.offset(p0, frame, delt);
    *out = f;
    if (!copy) return cudaSuccess;
    const size_t nb = frame * np;
    cudaError_t e = reserve(in, np, frame, delt);
    if (e == cudaSuccess) e = cudaMemcpyAsync(gray0.get(), f.gray0, nb, cudaMemcpyDefault, stream);
    if (e == cudaSuccess && f.gray1) e = cudaMemcpyAsync(gray1.get(), f.gray1, nb, cudaMemcpyDefault, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(depth0.get(), f.depth0, nb * delt, cudaMemcpyDefault, stream);
    if (e == cudaSuccess && f.depth1) e = cudaMemcpyAsync(depth1.get(), f.depth1, nb * delt, cudaMemcpyDefault, stream);
    *out = {gray0.get(), f.gray1 ? gray1.get() : nullptr, depth0.get(), f.depth1 ? depth1.get() : nullptr};
    return e;
  }
};

struct ContextDestroy { void operator()(phovo_ctx* c) const { phovo_destroy(c); } };
using ContextPtr = std::unique_ptr<phovo_ctx, ContextDestroy>;

struct phovo_batch_state {
  int sm_count = 0, l2_bytes = 0;
  int debug_flags = 0;
  bool record_stats = false;
  int last_path = 0;                                   // 1: shared-memory-resident batch kernels, 2: pool of per-pair contexts, 3: slot waves
  unsigned long long last_h2d_bytes = 0;
  // host mirrors of the per-pair stats of the last call (filled on demand)
  std::vector<phovo_iter_stats> h_log; std::vector<int32_t> h_log_counts;
  int log_per_pair = 0; int last_pairs = 0; bool log_fetched = false;

  // the shared-memory-resident kernels (phovo_batch_align, phovo_batch_align_device)
  struct Resident {
    DeviceArray<uint8_t> store;                        // packed level records
    DeviceArray<double> states, init;                  // outputs / inputs of the last call
    DeviceArray<int32_t> iters;
    DeviceArray<phovo_iter_stats> log;
    DeviceArray<int32_t> log_counts;
    PinnedArray<double> h_states; PinnedArray<int32_t> h_iters;
    FrameStage stage[2];                               // host inputs: two staging slots
    Stream copy_stream;
    Event ev_copied[2], ev_consumed[2];
    DeviceArray<unsigned int> next_pair;               // work counter of the persistent align kernel
    Event ev_k[3];                                     // before pyramid / between / after align
    bool timed = false;
    size_t prepared_smem = 0;
  } res;

  // batches the shared-memory-resident kernels cannot take (Ceres / photometric + depth solver, blurred levels, levels
  // beyond the shared-memory budget) run pair by pair on a small pool of per-pair contexts, one host thread each
  std::vector<ContextPtr> pool;

  // slot waves (batch_waves): two halves of per-pair slots; one half aligns while the other is being set up
  struct Waves {
    Stream setup_stream[kWaveSetupThreads]; Event ev_setup[kWaveSetupThreads];
    Stream align_stream[2]; Event ev_wave_done[2], ev_wave_in[2];
    DeviceArray<char> arena;
    size_t slot_bytes = 0; int arena_rows = 0, arena_cols = 0, arena_slots = 0, wave_half = 0; phovo_config arena_cfg = {};
    DeviceArray<SlotArgs> d_slot_args; std::vector<SlotArgs> h_slot_args;
    DeviceArray<double> d_init[2], d_states[2]; DeviceArray<int32_t> d_iters[2];
    PinnedArray<double> h_states[2]; PinnedArray<int32_t> h_iters[2];
    FrameStage stage[2];
    // Declared last, so destroyed first: phovo_destroy synchronises a slot's stream, one of setup_stream, and the
    // slot's buffers are views of the arena.
    std::vector<ContextPtr> slots;
  } waves;

  // warpImage (phovo_batch_warp_image, phovo_warp_image): splat keys of one chunk of pairs (zero between calls while
  // keys_clean), Rt of the pairs, per-pair summaries, device copies of host outputs of one chunk
  struct Warp {
    DeviceArray<uint32_t> keys; bool keys_clean = false;
    DeviceArray<double> rts;
    DeviceArray<int32_t> landed;
    DeviceArray<int64_t> sum;
    DeviceArray<uint8_t> warped, diff;
  } warp;

  // normal equations at given states (phovo_batch_eval_normal_equations): winner keys (zero between calls while
  // keys_clean) and validity of one chunk, its level records and tile partials; states, poses and results of every pair
  struct Eval {
    DeviceArray<uint32_t> keys; bool keys_clean = false;
    DeviceArray<uint8_t> valid, store;
    DeviceArray<double> partials, states;
    DeviceArray<PoseDev> poses;
    DeviceArray<double> out;                           // [P][21] H, [P][6] g, [P] cost
    DeviceArray<int32_t> nvalid;
    // photometric + depth solver: the chunk's target depth at the level (D1, its gradients), per-tile sums and gains
    DeviceArray<double> d1, gxd, gyd, sums, gain;
  } eval;

  // device copies of one chunk of host frames, for warpImage and the normal equations alike
  FrameStage chunk_frames;
};

void phovo_batch_release(phovo_ctx* ctx) {
  delete ctx->batch;
  ctx->batch = nullptr;
}

static int get_state(phovo_ctx* ctx, phovo_batch_state** out) {
  if (!ctx->batch) {
    std::unique_ptr<phovo_batch_state> b(new phovo_batch_state());
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    b->sm_count = prop.multiProcessorCount;
    b->l2_bytes = prop.l2CacheSize;
    CK(create_stream(b->res.copy_stream));
    CK(b->res.next_pair.ensure(PHOVO_MAX_LEVELS));
    for (int s = 0; s < 2; ++s) {
      CK(create_event(b->res.ev_copied[s], cudaEventDisableTiming));
      CK(create_event(b->res.ev_consumed[s], cudaEventDisableTiming));
    }
    ctx->batch = b.release();
  }
  *out = ctx->batch;
  return PHOVO_OK;
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
  const WarpIntrinsics I = scaled_intrinsics(ctx->K, level);
  bp->fx[a] = I.fx; bp->fy[a] = I.fy; bp->ox[a] = I.ox; bp->oy[a] = I.oy; bp->inv_fx[a] = I.inv_fx; bp->inv_fy[a] = I.inv_fy;
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
  const int status = for_each_level(ctx->cfg, [&](int level, int M) {
    const int rc = fill_level(ctx, rows, cols, level, a, bp, &off);
    if (rc) return rc;
    const int n = bp->lrows[a] * bp->lcols[a];
    if (n > kBatchMaxLevelPixels) return ctx->fail(PHOVO_E_UNSUPPORTED, "batch kernel: an active level exceeds the shared-memory budget (about 20K px); use the per-pair API");
    nmax = std::max(nmax, n);
    bp->max_iters[a] = M;
    ++a;
    return PHOVO_OK;
  });
  if (status) return status;
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
  auto& r = b->res;
  if (!r.prepared_smem) {
    CK(batch_align_prepare());
    r.prepared_smem = 1;
  }
  for (int i = 0; i < 3; ++i)
    if (!r.ev_k[i]) CK(create_event(r.ev_k[i]));
  CK(cudaEventRecord(r.ev_k[0].get(), stream));
  ctx->launches += launch_batch_pyramid(stream, bp, g0, d0, src_type_of_depth(depth_type), depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0, g1, store);
  CK(cudaEventRecord(r.ev_k[1].get(), stream));
  CK(cudaMemsetAsync(r.next_pair.get(), 0, sizeof(unsigned int) * PHOVO_MAX_LEVELS, stream));
  ctx->launches += launch_batch_align(stream, bp, b->sm_count, store, init, states, iters, log, log_counts, r.next_pair.get());
  CK(cudaEventRecord(r.ev_k[2].get(), stream));
  r.timed = true;
  CK(cudaGetLastError());
  return PHOVO_OK;
}

extern "C" int phovo_batch_get_last_h2d_bytes(const phovo_ctx* ctx, unsigned long long* bytes) {
  if (!ctx || !bytes || !ctx->batch) return PHOVO_E_INVALID;
  *bytes = ctx->batch->last_h2d_bytes;
  return PHOVO_OK;
}

extern "C" int phovo_batch_get_kernel_times(phovo_ctx* ctx, float* pyramid_ms, float* align_ms) {
  if (!ctx || !ctx->batch || !ctx->batch->res.timed) return PHOVO_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  const Event* ev = ctx->batch->res.ev_k;
  CK(cudaEventSynchronize(ev[2].get()));
  float a = 0, c = 0;
  CK(cudaEventElapsedTime(&a, ev[0].get(), ev[1].get()));
  CK(cudaEventElapsedTime(&c, ev[1].get(), ev[2].get()));
  if (pyramid_ms) *pyramid_ms = a;
  if (align_ms) *align_ms = c;
  return PHOVO_OK;
}

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
  CK(b->res.log.ensure((size_t)num_pairs * total));
  CK(b->res.log_counts.ensure((size_t)num_pairs));
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
    b->pool.emplace_back(c);
  }
  std::vector<double> init_host;
  if (initial_states && !host_readable(initial_states)) {
    init_host.resize((size_t)num_pairs * 6);
    CK(cudaMemcpy(init_host.data(), initial_states, sizeof(double) * init_host.size(), cudaMemcpyDeviceToHost));
    initial_states = init_host.data();
  }
  const size_t frame = (size_t)rows * cols, delt = depth_elt(depth_type);
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
  for (int w = 1; w < workers; ++w) threads.emplace_back(work, b->pool[w].get());
  work(b->pool[0].get());
  for (auto& t : threads) t.join();
  for (int w = 0; w < workers; ++w) ctx->launches += b->pool[w]->launches, b->pool[w]->launches = 0;
  b->last_pairs = log_per_pair ? num_pairs : 0; b->log_per_pair = log_per_pair; b->log_fetched = log_per_pair > 0;
  b->last_h2d_bytes = 0; b->res.timed = false; b->last_path = 2;
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
  auto& w = b->waves;
  for (int t = 0; t < kWaveSetupThreads; ++t) {
    if (!w.setup_stream[t]) CK(create_stream(w.setup_stream[t]));
    if (!w.ev_setup[t]) CK(create_event(w.ev_setup[t], cudaEventDisableTiming));
  }
  for (int h = 0; h < 2; ++h) {
    if (!w.align_stream[h]) CK(create_stream(w.align_stream[h]));
    if (!w.ev_wave_done[h]) CK(create_event(w.ev_wave_done[h], cudaEventDisableTiming));
    if (!w.ev_wave_in[h]) CK(create_event(w.ev_wave_in[h], cudaEventDisableTiming));
  }
  auto add_slots = [&](int want) -> int {
    while ((int)w.slots.size() < want) {
      phovo_ctx* c = nullptr;
      if (phovo_internal_create_slot(ctx->device, &c) != PHOVO_OK) return ctx->fail(PHOVO_E_CUDA, std::string("batch slots: ") + phovo_last_error(nullptr));
      c->defer_device_input_drain = true;   // the wave's inputs outlive its kernels (batch_waves waits for the wave before they go)
      w.slots.emplace_back(c);
    }
    return PHOVO_OK;
  };
  int rc = add_slots(1);
  if (rc) return rc;
  // ---- bytes per slot under this configuration and frame size ----
  phovo_ctx* c0 = w.slots[0].get();
  if (memcmp(&c0->cfg, &ctx->cfg, sizeof(phovo_config)) != 0 && (rc = phovo_set_config(c0, &ctx->cfg))) return ctx->fail(rc, phovo_last_error(c0));
  const size_t need = phovo_internal_slot_bytes(c0, rows, cols);
  // ---- slots per half: the CTAs of k_align_slots one wave keeps resident -- fewer if two halves of them would take more
  // than half of the device memory that is free (counting what the arena already holds) ----
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  size_t budget = (free_b + w.arena.capacity()) / 2;
  if (const char* e = getenv("PHOVO_WAVE_BUDGET_MB")) budget = std::min(budget, (size_t)std::max(1LL, atoll(e)) << 20);   // test hook
  int half = wave_slots_per_half(b);
  if ((size_t)2 * half * need > budget) half = (int)std::max<size_t>(1, budget / need / 2);
  const int want = num_pairs > half ? 2 * half : num_pairs;
  if ((rc = add_slots(want))) return rc;
  // ---- the arena: ONE allocation, slot s at s * slot_bytes; laid out again whenever configuration, frame size or slot count change ----
  const bool same = want <= w.arena_slots && half == w.wave_half && need == w.slot_bytes && rows == w.arena_rows && cols == w.arena_cols &&
                    memcmp(&w.arena_cfg, &ctx->cfg, sizeof(phovo_config)) == 0;
  if (!same) {
    CK(cudaDeviceSynchronize());                       // nothing of an earlier call is still running on the old layout
    CK(w.arena.ensure(need * (size_t)want));
    for (size_t s = 0; s < w.slots.size(); ++s) {
      if ((int)s < want) w.slots[s]->arena_reset(w.arena.get() + s * need, need);
      else w.slots[s]->arena_reset(nullptr, 0);       // not part of this layout (never used until the next one)
    }
    w.slot_bytes = need; w.arena_rows = rows; w.arena_cols = cols; w.arena_cfg = ctx->cfg; w.arena_slots = want; w.wave_half = half;
    for (auto& a : w.h_slot_args) memset(&a, 0, sizeof(a));
  }
  for (int h = 0; h < 2; ++h) {
    CK(w.d_init[h].ensure((size_t)6 * half));
    CK(w.d_states[h].ensure((size_t)6 * half));
    CK(w.d_iters[h].ensure((size_t)PHOVO_MAX_LEVELS * half));
    CK(w.h_states[h].ensure((size_t)6 * half));
    CK(w.h_iters[h].ensure((size_t)PHOVO_MAX_LEVELS * half));
  }
  CK(w.d_slot_args.ensure((size_t)2 * half));
  if (w.h_slot_args.size() < (size_t)2 * half) w.h_slot_args.resize((size_t)2 * half);
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
  auto& w = b->waves;
  const int waves = (num_pairs + half - 1) / half;
  const size_t frame = (size_t)rows * cols, delt = depth_elt(depth_type);
  const Frames in = {gray0, gray1, depth0, bi ? depth1 : nullptr};
  b->last_h2d_bytes = 0;
  const bool host_in = host_readable(gray0) || host_readable(depth0) || host_readable(gray1) || (bi && host_readable(depth1));

  // the active levels, coarse to fine (AN:502-503; CE:437 skips levels without iterations)
  SlotLevels LS;
  memset(&LS, 0, sizeof(LS));
  bool levels_known = false;

  struct Pending { int start = 0, n = 0; bool active = false; } pend[2];
  const bool trace = getenv("PHOVO_WAVE_TRACE") != nullptr;   // stderr: host set-up time and device align time per wave
  Event tr0[2], tr1[2];
  if (trace) for (int h = 0; h < 2; ++h) { create_event(tr0[h]); create_event(tr1[h]); }
  auto harvest = [&](int h) -> int {
    if (!pend[h].active) return PHOVO_OK;
    CK(cudaEventSynchronize(w.ev_wave_done[h].get()));
    if (trace) { float ms = 0.f; cudaEventElapsedTime(&ms, tr0[h].get(), tr1[h].get()); fprintf(stderr, "[wave] start %d n %d align %.3f ms\n", pend[h].start, pend[h].n, ms); }
    if (states) memcpy(states + (size_t)pend[h].start * 6, w.h_states[h].get(), sizeof(double) * 6 * (size_t)pend[h].n);
    if (iterations) memcpy(iterations + (size_t)pend[h].start * PHOVO_MAX_LEVELS, w.h_iters[h].get(), sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)pend[h].n);
    pend[h].active = false;
    return PHOVO_OK;
  };

  for (int k = 0; k < waves; ++k) {
    const int h = k & 1, start = k * half, n = std::min(half, num_pairs - start);
    if ((rc = harvest(h))) return rc;          // wave k - 2 used these slots (and these input buffers)
    // ---- inputs of the wave on the device ----
    cudaStream_t as = w.align_stream[h].get();
    Frames f;
    CK(w.stage[h].stage(host_in, in, frame, delt, start, n, as, &f));
    if (host_in) {
      CK(cudaEventRecord(w.ev_wave_in[h].get(), as));
      for (int t = 0; t < kWaveSetupThreads; ++t) CK(cudaStreamWaitEvent(w.setup_stream[t].get(), w.ev_wave_in[h].get(), 0));
      b->last_h2d_bytes += (size_t)n * frame * (2 + delt * (bi ? 2 : 1));
    }
    const uint8_t* g0 = f.gray0; const uint8_t* g1 = f.gray1;
    const char* d0 = (const char*)f.depth0; const char* d1 = (const char*)f.depth1;
    // ---- pyramids of the wave's slots: kWaveSetupThreads host threads, each on its own stream ----
    const auto t_setup = std::chrono::steady_clock::now();
    std::atomic<int> first_rc(PHOVO_OK);
    std::mutex mu; std::string message;
    auto work = [&](int t) {
      for (int s = t; s < n; s += kWaveSetupThreads) {
        if (first_rc.load() != PHOVO_OK) return;
        phovo_ctx* c = w.slots[(size_t)h * half + s].get();
        c->stream = w.setup_stream[t].get();   // not owned: this thread's stream
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
    for (int t = 0; t < kWaveSetupThreads; ++t) {
      CK(cudaEventRecord(w.ev_setup[t].get(), w.setup_stream[t].get()));
      CK(cudaStreamWaitEvent(as, w.ev_setup[t].get(), 0));
    }
    // ---- slot table (the buffers of a slot stay where they are once allocated for a frame size) ----
    bool table_changed = false;
    for (int s = 0; s < n; ++s) {
      phovo_ctx* c = w.slots[(size_t)h * half + s].get();
      SlotArgs A;
      memset(&A, 0, sizeof(A));
      for (int l = 0; l < c->cfg.num_levels; ++l) A.P[l] = c->level_ptrs(l);
      A.pose = c->d_pose.get(); A.partials = c->partials.get();
      SlotArgs& cached = w.h_slot_args[(size_t)h * half + s];
      if (memcmp(&cached, &A, sizeof(A)) != 0) { cached = A; table_changed = true; }
      ctx->launches += c->launches; c->launches = 0;
    }
    if (table_changed) {
      CK(cudaMemcpyAsync(w.d_slot_args.get() + (size_t)h * half, w.h_slot_args.data() + (size_t)h * half, sizeof(SlotArgs) * (size_t)n, cudaMemcpyHostToDevice, as));
      CK(cudaStreamSynchronize(as));   // pageable source: keep it simple, this happens once per frame size
    }
    if (!levels_known) {
      const phovo_ctx* c0 = w.slots[(size_t)h * half].get();
      for_each_level(ctx->cfg, [&](int level, int) {
        const int a = LS.count++;
        LS.L[a] = c0->level_params(level);
        LS.lm[a] = lm_params(ctx->cfg, level);
        return 0;
      });
      levels_known = true;
    }
    // ---- one launch aligns the wave; results to pinned memory ----
    const double* d_init = nullptr;
    if (initial_states) {
      CK(cudaMemcpyAsync(w.d_init[h].get(), initial_states + (size_t)start * 6, sizeof(double) * 6 * (size_t)n, cudaMemcpyDefault, as));
      d_init = w.d_init[h].get();
    }
    if (trace) cudaEventRecord(tr0[h].get(), as);
    // CTAs per pair: one when the wave fills the GPU; a small wave gives every pair a thread-block cluster (2, 4 or 8 CTAs,
    // cluster barriers) so that the SMs it would leave idle shorten the wave instead
    int cluster = 1;
    for (int c = 8; c > 1; c >>= 1)
      if (n * c <= PHOVO_SLOT_MINB * b->sm_count) { cluster = c; break; }
    if (const char* e = getenv("PHOVO_WAVE_CLUSTER")) { const int v = atoi(e); if (v == 1 || v == 2 || v == 4 || v == 8) cluster = v; }   // experiment hook
    SlotArgs* args = w.d_slot_args.get() + (size_t)h * half;
    int launched = launch_align_slots(as, ctx->cfg.mode, LS, args, n, d_init, cluster);
    if (launched < 0 && cluster > 1) { cudaGetLastError(); launched = launch_align_slots(as, ctx->cfg.mode, LS, args, n, d_init, 1); }
    if (launched < 0) return ctx->cuda_fail("k_align_slots", cudaGetLastError());
    ctx->launches += launched;
    if (trace) cudaEventRecord(tr1[h].get(), as);
    ctx->launches += launch_gather_slots(as, args, n, w.d_states[h].get(), w.d_iters[h].get());
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(w.h_states[h].get(), w.d_states[h].get(), sizeof(double) * 6 * (size_t)n, cudaMemcpyDeviceToHost, as));
    CK(cudaMemcpyAsync(w.h_iters[h].get(), w.d_iters[h].get(), sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)n, cudaMemcpyDeviceToHost, as));
    CK(cudaEventRecord(w.ev_wave_done[h].get(), as));
    pend[h].start = start; pend[h].n = n; pend[h].active = true;
  }
  // in wave order: the older half first
  const int last = (waves - 1) & 1;
  if ((rc = harvest(1 - last))) return rc;
  if ((rc = harvest(last))) return rc;
  b->last_pairs = 0; b->log_per_pair = 0; b->log_fetched = false; b->res.timed = false; b->last_path = 3;
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
  auto& r = b->res;
  CK(r.store.ensure((size_t)bp.record_bytes * num_pairs + kBatchStoreSlackBytes));
  return run_device(ctx, b, bp, smem, ctx->stream, gray0, depth0, depth_type, depth_scale, gray1, r.store.get(),
                    initial_states, states, iters, log_cap ? r.log.get() : nullptr, log_cap ? r.log_counts.get() : nullptr);
}

extern "C" int phovo_batch_align_device_with_target_depth(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0,
                                                          const void* depth0, int depth_type, double depth_scale, const uint8_t* gray1,
                                                          const void* depth1, const double* initial_states, double* states,
                                                          int32_t* iters) {
  if (!ctx || !gray0 || !depth0 || !gray1 || !depth1 || !states || !iters) return PHOVO_E_INVALID;
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if (ctx->cfg.mode != PHOVO_MODE_BIOBJECTIVE)      // the other solvers ignore the target depth, like the reference (AN:484)
    return phovo_batch_align_device(ctx, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, initial_states, states, iters);
  CK(cudaSetDevice(ctx->device));
  phovo_batch_state* b; int rc = get_state(ctx, &b);
  if (rc) return rc;
  // the pool (< 24 pairs) or the slot waves, as phovo_batch_align_device takes them for the other solvers: synchronous;
  // results go to the caller's device arrays through host temporaries
  std::vector<double> hs((size_t)num_pairs * 6); std::vector<int32_t> hi((size_t)num_pairs * PHOVO_MAX_LEVELS);
  if ((rc = batch_other(ctx, b, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, depth1, initial_states, hs.data(), hi.data()))) return rc;
  CK(cudaMemcpyAsync(states, hs.data(), sizeof(double) * hs.size(), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(iters, hi.data(), sizeof(int32_t) * hi.size(), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
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
  auto& r = b->res;
  CK(r.states.ensure((size_t)num_pairs * 6));
  CK(r.iters.ensure((size_t)num_pairs * PHOVO_MAX_LEVELS));
  CK(r.store.ensure((size_t)bp.record_bytes * num_pairs + kBatchStoreSlackBytes));
  const double* d_init = nullptr;
  if (initial_states) {
    CK(r.init.ensure((size_t)num_pairs * 6));
    CK(cudaMemcpyAsync(r.init.get(), initial_states, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
    d_init = r.init.get();
  }
  CK(r.h_states.ensure((size_t)num_pairs * 6));
  CK(r.h_iters.ensure((size_t)num_pairs * PHOVO_MAX_LEVELS));
  const bool on_device = is_device_pointer(gray0) && is_device_pointer(depth0) && is_device_pointer(gray1);
  const size_t frame = (size_t)rows * cols, delt = depth_elt(depth_type);
  phovo_iter_stats* log = log_cap ? r.log.get() : nullptr;
  int32_t* log_counts = log_cap ? r.log_counts.get() : nullptr;
  if (on_device) {
    rc = run_device(ctx, b, bp, smem, ctx->stream, gray0, depth0, depth_type, depth_scale, gray1, r.store.get(), d_init,
                    r.states.get(), r.iters.get(), log, log_counts);
    if (rc) return rc;
  } else {
    // chunked, double-buffered upload: copies run on copy_stream, kernels on ctx->stream
    // a chunk is four waves of persistent CTAs: large enough to amortise the ragged tail of a
    // wave (pairs need different iteration counts), small enough to overlap with the next copy
    const int chunk = std::max(1, std::min(num_pairs, 4 * b->sm_count));
    for (int s = 0; s < 2; ++s) CK(r.stage[s].reserve({gray0, gray1, depth0, nullptr}, chunk, frame, delt));
    CK(cudaMemsetAsync(r.iters.get(), 0, sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs, ctx->stream));
    int period, keep_begin, keep;
    row_compaction(ctx, rows, &period, &keep_begin, &keep);
    b->last_h2d_bytes = 0;
    int slot = 0, used[2] = {0, 0};
    for (int p0 = 0; p0 < num_pairs; p0 += chunk, slot ^= 1) {
      const int np = std::min(chunk, num_pairs - p0);
      FrameStage& st = r.stage[slot];
      cudaStream_t cs = r.copy_stream.get();
      if (used[slot]) CK(cudaStreamWaitEvent(cs, r.ev_consumed[slot].get(), 0));
      if (period) {
        // one strided copy per image stack: `keep` of every `period` rows, frames are back to back
        const size_t groups = (size_t)(rows / period) * np;
        const size_t gw = (size_t)keep * cols, gp = (size_t)period * cols, go = (size_t)keep_begin * cols;
        CK(cudaMemcpy2DAsync(st.gray0.get(), gw, gray0 + (size_t)p0 * frame + go, gp, gw, groups, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpy2DAsync(st.gray1.get(), gw, gray1 + (size_t)p0 * frame + go, gp, gw, groups, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpy2DAsync(st.depth0.get(), gw * delt, (const char*)depth0 + ((size_t)p0 * frame + go) * delt, gp * delt, gw * delt, groups, cudaMemcpyHostToDevice, cs));
        b->last_h2d_bytes += groups * gw * (2 + delt);
      } else {
        CK(cudaMemcpyAsync(st.gray0.get(), gray0 + (size_t)p0 * frame, frame * np, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(st.gray1.get(), gray1 + (size_t)p0 * frame, frame * np, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(st.depth0.get(), (const char*)depth0 + (size_t)p0 * frame * delt, frame * np * delt, cudaMemcpyHostToDevice, cs));
        b->last_h2d_bytes += (size_t)frame * np * (2 + delt);
      }
      CK(cudaEventRecord(r.ev_copied[slot].get(), cs));
      CK(cudaStreamWaitEvent(ctx->stream, r.ev_copied[slot].get(), 0));
      BatchParams cp = bp;
      cp.num_pairs = np;
      cp.src_period = period; cp.src_keep_begin = keep_begin; cp.src_keep = keep;
      rc = run_device(ctx, b, cp, smem, ctx->stream, st.gray0.get(), st.depth0.get(), depth_type, depth_scale, st.gray1.get(),
                      r.store.get() + (size_t)p0 * bp.record_bytes, d_init ? d_init + (size_t)p0 * 6 : nullptr,
                      r.states.get() + (size_t)p0 * 6, r.iters.get() + (size_t)p0 * PHOVO_MAX_LEVELS,
                      log ? log + (size_t)p0 * log_cap : nullptr, log_counts ? log_counts + p0 : nullptr);
      if (rc) return rc;
      CK(cudaEventRecord(r.ev_consumed[slot].get(), ctx->stream));
      used[slot] = 1;
    }
  }
  CK(cudaMemcpyAsync(r.h_states.get(), r.states.get(), sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(r.h_iters.get(), r.iters.get(), sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (states) memcpy(states, r.h_states.get(), sizeof(double) * 6 * (size_t)num_pairs);
  if (iterations) memcpy(iterations, r.h_iters.get(), sizeof(int32_t) * PHOVO_MAX_LEVELS * (size_t)num_pairs);
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
  CK(cudaMemcpy(b->h_log.data(), b->res.log.get(), sizeof(phovo_iter_stats) * b->h_log.size(), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(b->h_log_counts.data(), b->res.log_counts.get(), sizeof(int32_t) * b->last_pairs, cudaMemcpyDeviceToHost));
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
  auto& w = b->warp;
  bool fresh;
  CK(w.keys.ensure((size_t)chunk * n, &fresh));
  if (fresh) w.keys_clean = false;
  const bool memset_each = (b->debug_flags & 16) != 0;
  if (!w.keys_clean && !memset_each) CK(cudaMemsetAsync(w.keys.get(), 0, w.keys.capacity() * sizeof(uint32_t), ctx->stream));
  w.keys_clean = false;   // until every launch below has been enqueued
  CK(w.rts.ensure((size_t)num_pairs * 16));
  CK(cudaMemcpyAsync(w.rts.get(), rts, sizeof(double) * 16 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  for (int p0 = 0; p0 < num_pairs; p0 += chunk) {
    const int np = std::min(chunk, num_pairs - p0);
    WarpImages C = offset_pairs(W, p0);
    C.rts = w.rts.get() + (size_t)p0 * 16;
    if (memset_each) CK(cudaMemsetAsync(w.keys.get(), 0, (size_t)np * n * sizeof(uint32_t), ctx->stream));
    ctx->launches += launch_warp_images(ctx->stream, C, src_type, I, np, w.keys.get(), !memset_each) + (memset_each ? 1 : 0);
    CK(cudaGetLastError());
  }
  w.keys_clean = !memset_each;
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
  auto& w = b->warp;
  if (want_summary) {
    CK(w.landed.ensure((size_t)num_pairs));
    CK(w.sum.ensure((size_t)num_pairs));
    CK(cudaMemsetAsync(w.landed.get(), 0, sizeof(int32_t) * num_pairs, ctx->stream));
    CK(cudaMemsetAsync(w.sum.get(), 0, sizeof(int64_t) * num_pairs, ctx->stream));
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
  W.num_landed = want_summary ? w.landed.get() : nullptr;
  W.sum_abs_diff = want_sum ? w.sum.get() : nullptr;
  const WarpIntrinsics I = scaled_intrinsics(K, level);
  const int src = src_type_of_depth(depth_type);
  if (in_dev && !w_host && !d_host) {
    if ((rc = phovo_internal_warp_images(ctx, W, src, I, num_pairs, rts))) return rc;
  } else {
    // host inputs (all rows: the warp reads every one) and host outputs go through device buffers of one chunk
    const int chunk = warp_chunk_pairs(b, n, num_pairs);
    const Frames in = {gray0, target, depth0, nullptr};
    if (w_host) CK(w.warped.ensure((size_t)chunk * n));
    if (d_host) CK(w.diff.ensure((size_t)chunk * n));
    for (int p0 = 0; p0 < num_pairs; p0 += chunk) {
      const int np = std::min(chunk, num_pairs - p0);
      WarpImages C = offset_pairs(W, p0);
      Frames f;
      CK(b->chunk_frames.stage(!in_dev, in, n, delt, p0, np, ctx->stream, &f));
      C.gray = f.gray0; C.target = f.gray1; C.depth = f.depth0;
      if (w_host) C.warped = w.warped.get();
      if (d_host) C.diff = w.diff.get();
      if ((rc = phovo_internal_warp_images(ctx, C, src, I, np, rts + (size_t)p0 * 16))) return rc;
      if (w_host) CK(cudaMemcpyAsync(warped + (size_t)p0 * n, C.warped, n * np, cudaMemcpyDeviceToHost, ctx->stream));
      if (d_host) CK(cudaMemcpyAsync(diff + (size_t)p0 * n, C.diff, n * np, cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  if (num_landed) CK(cudaMemcpyAsync(num_landed, w.landed.get(), sizeof(int32_t) * num_pairs, cudaMemcpyDefault, ctx->stream));
  if (sum_abs_diff) CK(cudaMemcpyAsync(sum_abs_diff, w.sum.get(), sizeof(int64_t) * num_pairs, cudaMemcpyDefault, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
}

// ---------------------------------------------------------------------------------------------
// Normal equations of many pairs at given states (kernels_eval.cu): what phovo_eval_normal_equations gives pair by pair
// ---------------------------------------------------------------------------------------------
// Pairs per chunk: the chunk's winner keys (4 B per pixel; 8 B for the 2N slots of the photometric + depth solver, which
// also keeps D1, GxD and GyD: 24 B), validity flags (1 B) and, above level 0, its level records fit in half of the L2,
// so that the passes find them there (640x480 level 0 on a 126 MB L2: 41 pairs, 6 for the photometric + depth solver).
static int eval_chunk_pairs(const phovo_batch_state* b, size_t n, size_t px_bytes, unsigned long long record_bytes, int num_pairs) {
  const size_t fit = (size_t)std::max(b->l2_bytes, 1) / 2 / (n * px_bytes + record_bytes);
  return (int)std::max<size_t>(1, std::min<size_t>({fit, (size_t)num_pairs, 65535}));
}

// depth1 == nullptr: the analytic modes (k_eval_*); otherwise the photometric + depth solver (k_eval_*_bi)
static int eval_normal_equations(phovo_ctx* ctx, int num_pairs, int rows, int cols, const uint8_t* gray0, const void* depth0,
                                 int depth_type, double depth_scale, const uint8_t* gray1, const void* depth1,
                                 const double* states, int level, double* H, double* g, double* cost, int32_t* num_valid) {
  if (num_pairs < 1 || rows < 1 || cols < 1 || level < 0 || level >= ctx->cfg.num_levels)
    return ctx->fail(PHOVO_E_INVALID, "bad batch size, image size or level");
  if (depth_type < 0 || depth_type > 2) return ctx->fail(PHOVO_E_INVALID, "unknown depth_type");
  if (!H && !g && !cost && !num_valid) return ctx->fail(PHOVO_E_INVALID, "no output requested");
  const size_t n = (size_t)rows * cols;
  if (n > (size_t)INT32_MAX) return ctx->fail(PHOVO_E_UNSUPPORTED, "batched normal equations: frames of 2^31 pixels or more");
  const bool bi = depth1 != nullptr;
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
  E.L = make_level_params(ctx->cfg, ctx->K, level, bp.lrows[0], bp.lcols[0]);
  E.grad_k = bp.grad_k[0];
  E.tiles = (ln + kEvalTile - 1) / kEvalTile;
  E.depth_scale = depth_type == PHOVO_DEPTH_U16 ? depth_scale : 1.0;
  E.record_bytes = record_bytes; E.off_I0 = bp.off_I0[0]; E.off_I1 = bp.off_I1[0]; E.off_D0 = bp.off_D0[0];
  const int src = src_type_of_depth(depth_type);
  const size_t delt = depth_elt(depth_type);
  const size_t slots = bi ? 2 : 1;                  // residual slots per level pixel
  const size_t px_bytes = slots * sizeof(uint32_t) + 1 + (bi ? 3 * sizeof(double) : 0);
  const int chunk = eval_chunk_pairs(b, (size_t)ln, px_bytes, records ? record_bytes : 0, num_pairs);
  const size_t ck = (size_t)chunk * ln;
  auto& v = b->eval;
  EvalTargetDepth D;
  memset(&D, 0, sizeof(D));
  if (bi) {
    D.rows = rows; D.cols = cols; D.level = level; D.depth_scale = E.depth_scale;
    D.inv_max_depth = 1. / ctx->cfg.max_depth;    // as phovo_set_target_depth: k_scale by 1 / max_depth, then k_scharr_store
    D.ks0 = 3.; D.ks1 = 10.;
    if (ctx->cfg.grad_scale[level] != 1.) { D.ks0 *= ctx->cfg.grad_scale[level]; D.ks1 *= ctx->cfg.grad_scale[level]; }
    D.tiles2 = (int)((2 * (size_t)ln + kEvalTile - 1) / kEvalTile);
    CK(v.d1.ensure(ck)); CK(v.gxd.ensure(ck)); CK(v.gyd.ensure(ck));
    CK(v.sums.ensure((size_t)chunk * E.tiles * 2));
    CK(v.gain.ensure((size_t)chunk));
    D.D1 = v.d1.get(); D.GxD = v.gxd.get(); D.GyD = v.gyd.get(); D.sums = v.sums.get(); D.gain = v.gain.get();
  }
  bool fresh;
  CK(v.keys.ensure(ck * slots, &fresh));
  if (fresh) v.keys_clean = false;
  CK(v.valid.ensure(ck));
  CK(v.partials.ensure((size_t)chunk * (bi ? D.tiles2 : E.tiles) * PHOVO_ACC_STRIDE));
  if (records) CK(v.store.ensure((size_t)chunk * record_bytes));
  CK(v.states.ensure((size_t)num_pairs * 6));
  CK(v.poses.ensure((size_t)num_pairs));
  CK(v.out.ensure((size_t)num_pairs * 28));
  CK(v.nvalid.ensure((size_t)num_pairs));
  const bool in_dev = is_device_pointer(gray0) && is_device_pointer(depth0) && is_device_pointer(gray1) &&
                      (!bi || is_device_pointer(depth1));
  const Frames in = {gray0, gray1, depth0, depth1};
  if (!v.keys_clean) CK(cudaMemsetAsync(v.keys.get(), 0, v.keys.capacity() * sizeof(uint32_t), ctx->stream));
  v.keys_clean = false;   // until every launch below has been enqueued
  CK(cudaMemcpyAsync(v.states.get(), states, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  ctx->launches += launch_eval_poses(ctx->stream, v.states.get(), num_pairs, v.poses.get());
  double* dH = v.out.get(); double* dg = dH + (size_t)num_pairs * 21; double* dcost = dg + (size_t)num_pairs * 6;
  E.keys = v.keys.get(); E.valid = v.valid.get(); E.partials = v.partials.get(); E.store = v.store.get();
  for (int p0 = 0; p0 < num_pairs; p0 += chunk) {
    const int np = std::min(chunk, num_pairs - p0);
    Frames f;
    CK(b->chunk_frames.stage(!in_dev, in, n, delt, p0, np, ctx->stream, &f));   // host frames: every row (level 0 and the pyramid read them all)
    if (records) {
      bp.num_pairs = np;
      ctx->launches += launch_batch_pyramid(ctx->stream, bp, f.gray0, f.depth0, src, E.depth_scale, f.gray1, v.store.get());
    } else {
      E.gray0 = f.gray0; E.gray1 = f.gray1; E.depth = f.depth0;
    }
    E.poses = v.poses.get() + p0;
    if (bi) {
      D.depth1 = f.depth1;
      ctx->launches += launch_eval_normal_equations_bi(ctx->stream, E, D, src, records, np, dH + (size_t)p0 * 21, dg + (size_t)p0 * 6,
                                                       dcost + p0, v.nvalid.get() + p0);
    } else {
      ctx->launches += launch_eval_normal_equations(ctx->stream, E, src, records, np, dH + (size_t)p0 * 21, dg + (size_t)p0 * 6,
                                                    dcost + p0, v.nvalid.get() + p0);
    }
    CK(cudaGetLastError());
  }
  v.keys_clean = true;
  if (H) CK(cudaMemcpyAsync(H, dH, sizeof(double) * 21 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  if (g) CK(cudaMemcpyAsync(g, dg, sizeof(double) * 6 * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  if (cost) CK(cudaMemcpyAsync(cost, dcost, sizeof(double) * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  if (num_valid) CK(cudaMemcpyAsync(num_valid, v.nvalid.get(), sizeof(int32_t) * (size_t)num_pairs, cudaMemcpyDefault, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return PHOVO_OK;
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
  return eval_normal_equations(ctx, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, nullptr, states, level,
                               H, g, cost, num_valid);
}

extern "C" int phovo_batch_eval_normal_equations_with_target_depth(phovo_ctx* ctx, int num_pairs, int rows, int cols,
                                                                   const uint8_t* gray0, const void* depth0, int depth_type,
                                                                   double depth_scale, const uint8_t* gray1, const void* depth1,
                                                                   const double* states, int level, double* H, double* g,
                                                                   double* cost, int32_t* num_valid) {
  if (!ctx) return PHOVO_E_INVALID;
  if (!gray0 || !depth0 || !gray1 || !depth1 || !states)
    return ctx->fail(PHOVO_E_INVALID, "gray0, depth0, gray1, depth1 and states are required");
  if (ctx->cfg.mode != PHOVO_MODE_BIOBJECTIVE)      // the other solvers ignore the target depth, like the reference (AN:484)
    return phovo_batch_eval_normal_equations(ctx, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, states,
                                             level, H, g, cost, num_valid);
  if (!ctx->have_K) return ctx->fail(PHOVO_E_INVALID, "SetIntrinsicMatrix has not been called");
  return eval_normal_equations(ctx, num_pairs, rows, cols, gray0, depth0, depth_type, depth_scale, gray1, depth1, states, level,
                               H, g, cost, num_valid);
}
