// phovo_lm.h -- the Levenberg-Marquardt decision of Ceres mode: the restated trust-region loop of one level
// (CPhotoconsistencyOdometryCeres.h:433-500 -> ceres::Solve, SURVEY appendix A), defined once.
//
// Two drivers run it.  The device loop (kernels_align.cu, level_loop_ceres) evaluates the residuals inside one
// persistent launch and takes each decision in thread 0 of every CTA.  The host loop (phovo_api.cu, optimize_ceres)
// evaluates through stream launches and decides on the CPU; it is the fallback when cooperative launch is not
// available.  Both call the functions below in the same order:
//
//   S.cur = evaluation at x;  go = lm_start(...)
//   while (go && lm_propose(...)) {                          // S.xn = x + step, or the level ends
//     v = lm_judge(..., cost at S.xn, ...)                   // stop / accept / reject, one log entry
//     if (v == LM_ACCEPT) S.cur = evaluation at S.xn
//     go = v != LM_STOP && lm_update_radius(...)
//   }
//
// nvcc compiles the device copy; the host compiler builds the host copy (x86-64 baseline, no FMA).  S.cur comes from
// the device in both drivers, so the log entries' H, g, grad_norm, cost and num_valid are the evaluation's.
// Include from .cu files only.
#ifndef PHOVO_LM_H_
#define PHOVO_LM_H_

#include <math.h>

#include "phovo_internal.h"

namespace phovo {

// Levenberg-Marquardt options of one level (CE:464-477)
struct LmParams {
  double function_tolerance, gradient_tolerance, parameter_tolerance;
  double initial_radius, max_radius, min_radius, min_relative_decrease;
  int max_iterations;
};

inline LmParams lm_params(const phovo_config& cfg, int level) {
  LmParams lm;
  lm.function_tolerance = cfg.function_tolerance[level];
  lm.gradient_tolerance = cfg.gradient_tolerance[level];
  lm.parameter_tolerance = cfg.parameter_tolerance[level];
  lm.initial_radius = cfg.initial_trust_region_radius[level];
  lm.max_radius = cfg.max_trust_region_radius[level];
  lm.min_radius = cfg.min_trust_region_radius[level];
  lm.min_relative_decrease = cfg.min_relative_decrease[level];
  lm.max_iterations = cfg.max_num_iterations[level];
  return lm;
}

struct LmState {
  phovo_iter_stats cur;             // the evaluation at x: H, g, grad_norm, cost, num_valid, level
  double x[6], xn[6], scale[6];     // current state, candidate, Jacobi scaling of the columns
  double step_norm, x_norm, model_cost_change, rho;
  double radius, decrease_factor;
  int iteration;                    // LM iterations of the level so far
};

// Where the log entries go: base[count] while count < capacity and `write`; count advances with every entry.
struct LmLog {
  phovo_iter_stats* base;
  int& count;
  int capacity;
  bool write;
};

__host__ __device__ inline void expand_sym(const double H[21], double M[36]) {
  int k = 0;
  for (int a = 0; a < 6; ++a) for (int b = a; b < 6; ++b) { M[a * 6 + b] = H[k]; M[b * 6 + a] = H[k]; ++k; }
}

__host__ __device__ inline bool chol_solve6(const double M[36], const double b[6], double x[6]) {
  double Lm[36];
  for (int i = 0; i < 36; ++i) Lm[i] = 0.;
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j <= i; ++j) {
      double sum = M[i * 6 + j];
      for (int k = 0; k < j; ++k) sum -= Lm[i * 6 + k] * Lm[j * 6 + k];
      if (i == j) { if (!(sum > 0)) return false; Lm[i * 6 + i] = sqrt(sum); }
      else Lm[i * 6 + j] = sum / Lm[j * 6 + j];
    }
  double y[6];
  for (int i = 0; i < 6; ++i) { double sum = b[i]; for (int k = 0; k < i; ++k) sum -= Lm[i * 6 + k] * y[k]; y[i] = sum / Lm[i * 6 + i]; }
  for (int i = 5; i >= 0; --i) { double sum = y[i]; for (int k = i + 1; k < 6; ++k) sum -= Lm[k * 6 + i] * x[k]; x[i] = sum / Lm[i * 6 + i]; }
  return true;
}

__host__ __device__ inline double lm_gmax(const LmState& S) {
  double gmax = 0; for (int a = 0; a < 6; ++a) gmax = fmax(gmax, fabs(S.cur.g[a]));
  return gmax;
}

// log entry of the iteration being decided
__host__ __device__ inline void lm_log(const LmState& S, LmLog& log, int accepted, const double* state_out) {
  if (log.write && log.count < log.capacity) {
    phovo_iter_stats* e = log.base + log.count;
    *e = S.cur;
    e->iteration = S.iteration - 1; e->accepted = accepted; e->radius = S.radius;
    for (int k = 0; k < 6; ++k) { e->state_in[k] = S.x[k]; e->state_out[k] = state_out[k]; }
  }
  log.count += 1;
}

// After the first evaluation of a level (S.cur at x): the scaling, and false when the gradient is already small.
__host__ __device__ inline bool lm_start(const LmParams& lm, LmState& S) {
  double M[36]; expand_sym(S.cur.H, M);
  for (int a = 0; a < 6; ++a) S.scale[a] = 1.0 / (1.0 + sqrt(M[a * 6 + a]));
  return !(lm_gmax(S) <= lm.gradient_tolerance);
}

// Proposes LM iteration S.iteration + 1 from S.cur: S.xn and the norms lm_judge needs.  False when the level ends here.
__host__ __device__ inline bool lm_propose(const LmParams& lm, LmState& S, LmLog& log) {
  if (S.iteration >= lm.max_iterations) return false;
  S.iteration += 1;
  double M[36], Ms[36], gs[6], A[36], step[6];
  expand_sym(S.cur.H, M);
  for (int a = 0; a < 6; ++a) { gs[a] = S.cur.g[a] * S.scale[a]; for (int b = 0; b < 6; ++b) Ms[a * 6 + b] = M[a * 6 + b] * S.scale[a] * S.scale[b]; }
  for (int k = 0; k < 36; ++k) A[k] = Ms[k];
  for (int a = 0; a < 6; ++a) { double d = Ms[a * 6 + a]; if (d < 1e-6) d = 1e-6; if (d > 1e32) d = 1e32; A[a * 6 + a] += d / S.radius; }
  bool ok = chol_solve6(A, gs, step);
  for (int a = 0; a < 6; ++a) step[a] = -step[a];
  double model_cost_change = 0;
  if (ok) {
    double dg = 0, dMd = 0;
    for (int a = 0; a < 6; ++a) { dg += step[a] * gs[a]; double t = 0; for (int b = 0; b < 6; ++b) t += Ms[a * 6 + b] * step[b]; dMd += step[a] * t; }
    model_cost_change = -(dg + 0.5 * dMd);
    for (int a = 0; a < 6; ++a) if (!isfinite(step[a])) ok = false;
  }
  if (!ok || !(model_cost_change > 0)) { lm_log(S, log, 0, S.x); return false; }   // max_num_consecutive_invalid_steps = 0 (CE:477)
  double step_norm = 0, x_norm = 0;
  for (int a = 0; a < 6; ++a) { const double d = step[a] * S.scale[a]; S.xn[a] = S.x[a] + d; step_norm += d * d; x_norm += S.x[a] * S.x[a]; }
  S.step_norm = sqrt(step_norm); S.x_norm = sqrt(x_norm); S.model_cost_change = model_cost_change;
  return true;
}

enum { LM_STOP = 0, LM_ACCEPT = 1, LM_REJECT = 2 };

// After the evaluation of the candidate S.xn: convergence tests, then accept (x = xn) or reject.  Logs the iteration.
// On LM_ACCEPT the caller replaces S.cur by the candidate's evaluation before lm_update_radius.
__host__ __device__ inline int lm_judge(const LmParams& lm, LmState& S, double cand_cost, LmLog& log) {
  if (S.step_norm <= lm.parameter_tolerance * (S.x_norm + lm.parameter_tolerance)) { lm_log(S, log, 0, S.x); return LM_STOP; }
  const double cost_change = S.cur.cost - cand_cost;
  if (fabs(cost_change) < lm.function_tolerance * S.cur.cost) { lm_log(S, log, 0, S.x); return LM_STOP; }
  S.rho = cost_change / S.model_cost_change;
  if (S.rho > lm.min_relative_decrease) {
    lm_log(S, log, 1, S.xn);
    for (int k = 0; k < 6; ++k) S.x[k] = S.xn[k];
    return LM_ACCEPT;
  }
  lm_log(S, log, 0, S.x);
  return LM_REJECT;
}

// Trust-region update after an accepted or a rejected step.  False when the level ends here.
__host__ __device__ inline bool lm_update_radius(const LmParams& lm, LmState& S, bool accepted) {
  if (accepted) {
    if (lm_gmax(S) <= lm.gradient_tolerance) return false;
    const double t = 2.0 * S.rho - 1.0;
    double f = 1.0 - t * t * t; if (f < 1.0 / 3.0) f = 1.0 / 3.0;
    S.radius = S.radius / f; if (S.radius > lm.max_radius) S.radius = lm.max_radius;
    S.decrease_factor = 2.0;
  } else {
    S.radius = S.radius / S.decrease_factor; S.decrease_factor *= 2.0;
  }
  return !(S.radius < lm.min_radius);
}

}  // namespace phovo
#endif
