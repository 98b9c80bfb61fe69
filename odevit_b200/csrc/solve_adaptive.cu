// Adaptive Dormand-Prince 5(4) solve with per-image step control (odevit_solve_adaptive[_record|_attn]) and its reverse
// sweep over the accepted steps (odevit_solve_adaptive_bwd[_attn]).
//
// Every image b runs torchdiffeq's dopri5 (_impl/dopri5.py, rk_common.py, interp.py, misc.py) on its own N*D
// elements: its own t, dt, error norm, accept/reject decision and dense output.  A batch of one is the published
// algorithm; an image's result does not depend on its batch-mates (torchdiffeq takes one RMS norm over the whole
// batch instead).
//
// A ROUND is one attempted step of every image, six field evaluations for the whole batch through eval_forward:
//   u2 = y0 + dt_b/5 k1                         rk_apply_rows (per-image step)
//   k2..k6 = f(u2..u6)                          each evaluation's last GEMM epilogue forms the next stage input
//                                               u_{m+1} = y0 + dt_b * sum_l beta[m][l] k_l  (EPI_RK | EPI_ROWDT)
//                                               and, after k6, y1 = y0 + dt_b * sum_l c_sol[l] k_l
//   k7 = f(y1)                                  (FSAL: next step's k1)
//   ad_rowsq_kernel<ERR>                        per-row sums of (err / tol)^2
//   ad_control_kernel                           per image: fixed-order sum -> ratio -> accept, next t / dt (double
//                                               buffer: this round's kernels read slot r & 1, it writes the other)
//   ad_commit_kernel                            accepted images: dense output for every output time in (t0, t1],
//                                               y0 <- y1, k1 <- k7
// An image that has finished has dt_b = 0: its stage inputs equal y0 and its round is a no-op.
//
// The host cannot know the number of rounds: after enqueuing round r + 1 it waits for round r's active-image count
// (copied to pinned host memory right after round r, before round r + 1's launches), so the GPU always has the next
// round queued while the host decides.
//
// Attention outputs (odevit_solve_adaptive_attn), torchdiffeq's meaning taken per image: p_last[b] is the map of image
// b's last field evaluation, k7 = f(y1) of its last accepted step (one extra evaluation at y0 after the last round
// repeats it bit for bit); the JaSMin window of b is the statistic of b's own last min(W, nfe_b) evaluations -- f(x0),
// the probe, the 6 stages of every attempted step, rejected ones included, not the identity rounds after b finished --
// filed per evaluation by ad_jas_push_kernel into a ring [W, B, H].
//
// odevit_solve_adaptive_record also records every image's accepted steps (ad_control_kernel); odevit_solve_adaptive_bwd
// differentiates the solve along them, frozen: it replays the steps into checkpoints (optionally onto a tape), then runs
// the reverse sweep step by step -- the dense output's VJP (ad_interp_vjp_kernel), the stage VJPs whose mu epilogues form
// the next lambda with the per-image dt (EPI_RK | EPI_ROWDT), and one VJP at the step's start row (DESIGN.md 4.5).
#include <cmath>
#include <vector>

#include "dopri5.cuh"
#include "epilogue.cuh"
#include "host.h"
#include "internal.h"

namespace odevit {
namespace {

__constant__ float kCErr[7] = {kDopri5Err[0], kDopri5Err[1], kDopri5Err[2], kDopri5Err[3],
                               kDopri5Err[4], kDopri5Err[5], kDopri5Err[6]};
__constant__ float kCMid[7] = {kDopri5Mid[0], kDopri5Mid[1], kDopri5Mid[2], kDopri5Mid[3],
                               kDopri5Mid[4], kDopri5Mid[5], kDopri5Mid[6]};

constexpr int kMaxOut = 4096;        // output times a workspace holds (32 KB of fp64)
constexpr int kRedThreads = 256;     // per-image reductions: one block per image
constexpr int kErrRecord = 3;
constexpr int kNoError = 0x7fffffff;

// sync words: [0], [1] active-image count of rounds with r & 1 == 0 / 1; [2] min(b * 4 + kind) over failed images
struct AdBufs {
  WeightBufs w;
  StageCtx ctx;
  float *P, *sq;
  float *y0, *y1, *u;
  float* k[7];
  double *row0, *row1;      // [M] per-row partial sums
  double *t, *dt;           // [2][B] double-buffered per-image time and step (dt 0: image inactive)
  int* out_next;            // [2][B] first output index not yet written
  double *h0, *d1;          // [B] initial-step selection
  double* t_out;            // [kMaxOut]
  int *accept, *attempts, *n_acc, *n_rej;   // [B]
  int* sync;                // [4]
  float* jas;               // [B, H] JaSMin statistic of one evaluation
};

AdBufs layout_adaptive(const Plan& p, Arena& a) {
  AdBufs f;
  const size_t MD = (size_t)p.M * p.D;
  f.w = take_weights(p, a);
  f.ctx = take_ctx(p, a, false);
  f.P = a.f32(p.BHNN);
  f.sq = (p.variant == ODEVIT_FIELD_PARALLEL_L2) ? a.f32((size_t)2 * p.B * p.H * p.N) : nullptr;
  f.y0 = a.f32(MD);
  f.y1 = a.f32(MD);
  f.u = a.f32(MD);
  for (int i = 0; i < 7; ++i) f.k[i] = a.f32(MD);
  f.row0 = reinterpret_cast<double*>(a.take((size_t)p.M * 8));
  f.row1 = reinterpret_cast<double*>(a.take((size_t)p.M * 8));
  f.t = reinterpret_cast<double*>(a.take((size_t)2 * p.B * 8));
  f.dt = reinterpret_cast<double*>(a.take((size_t)2 * p.B * 8));
  f.out_next = reinterpret_cast<int*>(a.take((size_t)2 * p.B * 4));
  f.h0 = reinterpret_cast<double*>(a.take((size_t)p.B * 8));
  f.d1 = reinterpret_cast<double*>(a.take((size_t)p.B * 8));
  f.t_out = reinterpret_cast<double*>(a.take((size_t)kMaxOut * 8));
  f.accept = reinterpret_cast<int*>(a.take((size_t)4 * p.B * 4));
  f.attempts = f.accept ? f.accept + p.B : nullptr;
  f.n_acc = f.accept ? f.accept + 2 * p.B : nullptr;
  f.n_rej = f.accept ? f.accept + 3 * p.B : nullptr;
  f.sync = reinterpret_cast<int*>(a.take(16));
  split_scratch(p, a);
  f.jas = a.f32((size_t)p.B * p.H);
  return f;
}

// ---- device code ---------------------------------------------------------------------------------------------------
__global__ void ad_init_kernel(double* t, double* dt, int* out_next, int* counters, int* sync, const double* t_out,
                               double first_step, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) { sync[0] = 0; sync[1] = 0; sync[2] = kNoError; }
  if (b >= B) return;
  t[b] = t_out[0];
  dt[b] = first_step;     // <= 0: replaced by the initial-step selection
  out_next[b] = 1;
  for (int i = 0; i < 4; ++i) counters[i * B + b] = 0;
}

// JaSMin window: the statistic of one evaluation (jas [B, H]) goes to slot count[b] mod W of image b's ring [W, B, H],
// then count[b] += 1 -- for the images that took part in it: all (dt == null: f(x0), the probe) or those with dt_b != 0
// (a round's stages; a finished image's identity rounds are not evaluations of it).
__global__ void ad_jas_push_kernel(const float* __restrict__ jas, const double* dt, float* ring, int* count, int B,
                                   int H, int W) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B || (dt && dt[b] == 0.0)) return;
  const int c = count[b];
  float* dst = ring + ((long long)(c % W) * B + b) * H;
  for (int h = 0; h < H; ++h) dst[h] = jas[(long long)b * H + h];
  count[b] = c + 1;
}

enum { RS_INIT = 0, RS_D2 = 1, RS_ERR = 2 };
// One warp per row, lanes stride over D in a fixed order, fixed shuffle tree: a deterministic per-row partial.
//   RS_INIT: row0 = sum (y0 / sc)^2, row1 = sum (f0 / sc)^2,  sc = atol + rtol |y0|       (misc._select_initial_step)
//   RS_D2:   row0 = sum ((f1 - f0) / sc)^2
//   RS_ERR:  row0 = sum (err / tol)^2, err = dt_b sum_l c_err[l] k_l, tol = atol + rtol max(|y0|, |y1|)
//            (rk_common._runge_kutta_step, misc._compute_error_ratio)
template <int MODE>
__global__ void __launch_bounds__(256) ad_rowsq_kernel(const float* __restrict__ y0, const float* __restrict__ y1,
                                                       const float* __restrict__ f0, const float* __restrict__ f1,
                                                       const float* k3, const float* k4, const float* k5,
                                                       const float* k6, const float* k7, const double* dt, float rtol,
                                                       float atol, int rows, int N, int D, double* row0,
                                                       double* row1) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const long long base = (long long)row * D;
  double s0 = 0.0, s1 = 0.0;
  float dtb = 0.f;
  if constexpr (MODE == RS_ERR) dtb = (float)dt[row / N];
  for (int c = lane; c < D; c += 32) {
    const long long i = base + c;
    const float a = y0[i];
    if constexpr (MODE == RS_INIT) {
      const float sc = atol + fabsf(a) * rtol;
      const float q0 = a / sc, q1 = f0[i] / sc;
      s0 += (double)(q0 * q0);
      s1 += (double)(q1 * q1);
    } else if constexpr (MODE == RS_D2) {
      const float sc = atol + fabsf(a) * rtol;
      const float q = (f1[i] - f0[i]) / sc;
      s0 += (double)(q * q);
    } else {
      float e = kCErr[0] * f0[i];
      e = fmaf(kCErr[2], k3[i], e);
      e = fmaf(kCErr[3], k4[i], e);
      e = fmaf(kCErr[4], k5[i], e);
      e = fmaf(kCErr[5], k6[i], e);
      e = fmaf(kCErr[6], k7[i], e);
      e *= dtb;
      const float tol = atol + rtol * fmaxf(fabsf(a), fabsf(y1[i]));
      const float q = e / tol;
      s0 += (double)(q * q);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    if constexpr (MODE == RS_INIT) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (lane == 0) {
    row0[row] = s0;
    if constexpr (MODE == RS_INIT) row1[row] = s1;
  }
}

// sum of v[0..n) in a fixed order: thread j sums j, j + 256, ... in sequence, then a fixed shared-memory tree
__device__ __forceinline__ double block_sum_fixed(const double* v, int n, double* red) {
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += kRedThreads) s += v[i];
  red[threadIdx.x] = s;
  __syncthreads();
#pragma unroll
  for (int w = kRedThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  return red[0];
}

// Initial step (torchdiffeq misc._select_initial_step with order 4), one block per image.
//   phase 0: d0, d1 -> h0 (the probe is y0 + h0 f0);  phase 1: d2 -> h1 -> dt = min(100 h0, h1)
__global__ void __launch_bounds__(kRedThreads) ad_init_step_kernel(int phase, const double* row0, const double* row1,
                                                                   int N, int D, double* h0, double* d1v, double* dt) {
  __shared__ double red[kRedThreads];
  const int b = blockIdx.x;
  const double nel = (double)N * D;
  const double s0 = block_sum_fixed(row0 + (long long)b * N, N, red);
  if (phase == 0) {
    __syncthreads();
    const double s1 = block_sum_fixed(row1 + (long long)b * N, N, red);
    if (threadIdx.x == 0) dp5_probe_step(s0, s1, nel, h0[b], d1v[b]);
  } else if (threadIdx.x == 0) {
    dt[b] = dp5_first_step(s0, nel, h0[b], d1v[b]);
  }
}

// Per image: error ratio from the row partials (fixed order), accept / reject, the next t / dt / output index into the
// other half of the double buffer, counters, limits.  One block per image.
// rec_t0 != null: an accepted step is recorded at [n_acc[b], b] of rec_t0 / rec_dt / rec_out ([rec_cap, B]).
__global__ void __launch_bounds__(kRedThreads) ad_control_kernel(
    const double* row0, int N, int D, int B, const double* t_cur, const double* dt_cur, const int* on_cur,
    double* t_nxt, double* dt_nxt, int* on_nxt, int* accept, int* attempts, int* n_acc, int* n_rej, const double* t_out,
    int n_out, int max_steps, int nfe_base, int* nfe, int* acc_out, int* rej_out, int* active_slot, int* err,
    double* rec_t0, double* rec_dt, int* rec_out, int rec_cap) {
  __shared__ double red[kRedThreads];
  const int b = blockIdx.x;
  const double dt = dt_cur[b];
  if (dt == 0.0) {   // finished (or failed) before this round
    if (threadIdx.x == 0) { t_nxt[b] = t_cur[b]; dt_nxt[b] = 0.0; on_nxt[b] = on_cur[b]; accept[b] = 0; }
    return;
  }
  const double s = block_sum_fixed(row0 + (long long)b * N, N, red);
  if (threadIdx.x != 0) return;
  const double ratio = sqrt(s / ((double)N * D));
  const double t0 = t_cur[b];
  const int att = attempts[b] + 1;
  attempts[b] = att;
  int on = on_cur[b];
  double t1 = t0, dt_new = 0.0;
  int fail = -1;
  const bool ok = ratio <= 1.0;
  if (!isfinite(ratio)) {
    fail = kErrNonFinite;
  } else {
    if (ok) {
      t1 = t0 + dt;
      while (on < n_out && t_out[on] <= t1) ++on;
      if (rec_t0) {
        const int i = n_acc[b];
        if (i >= rec_cap) {
          fail = kErrRecord;
        } else {
          rec_t0[(long long)i * B + b] = t0;
          rec_dt[(long long)i * B + b] = dt;
          rec_out[(long long)i * B + b] = on;
        }
      }
      n_acc[b] += 1;
    } else {
      n_rej[b] += 1;
    }
    // _optimal_step_size(dt, ratio, safety 0.9, ifactor 10, dfactor 0.2, order 5)
    dt_new = dp5_next_step(dt, ratio);
    if (fail < 0 && on < n_out) {
      if (att >= max_steps) fail = kErrMax;
      else if (t1 + dt_new == t1) fail = kErrUnderflow;
    }
  }
  accept[b] = (fail < 0 && ok) ? 1 : 0;
  t_nxt[b] = t1;
  on_nxt[b] = on;
  const bool active = fail < 0 && on < n_out;
  dt_nxt[b] = active ? dt_new : 0.0;
  if (active) atomicAdd(active_slot, 1);
  if (fail >= 0) atomicMin(err, b * 4 + fail);
  if (nfe) nfe[b] = nfe_base + 6 * att;
  if (acc_out) acc_out[b] = n_acc[b];
  if (rej_out) rej_out[b] = n_rej[b];
}

// Accepted images: every output time in (t0, t1] from the quartic of interp._interp_fit / _interp_evaluate, then
// y0 <- y1 and k1 <- k7.  Rejected or inactive images: untouched.
__global__ void __launch_bounds__(256) ad_commit_kernel(float* y0, const float* __restrict__ y1, float* k1,
                                                        const float* k3, const float* k4, const float* k5,
                                                        const float* k6, const float* k7, const int* accept,
                                                        const double* t_cur, const double* dt_cur, const int* on_cur,
                                                        const int* on_nxt, const double* t_out, float* states,
                                                        long long MD, long long per_image) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < MD; i += stride) {
    const int b = (int)(i / per_image);
    if (!accept[b]) continue;
    const int lo = on_cur[b], hi = on_nxt[b];
    const float a0 = y0[i], a1 = y1[i], f0 = k1[i], f1 = k7[i];
    if (lo < hi) {
      const double t0 = t_cur[b], dtd = dt_cur[b];
      const float dt = (float)dtd;
      float m = kCMid[0] * f0;
      m = fmaf(kCMid[2], k3[i], m);
      m = fmaf(kCMid[3], k4[i], m);
      m = fmaf(kCMid[4], k5[i], m);
      m = fmaf(kCMid[5], k6[i], m);
      m = fmaf(kCMid[6], f1, m);
      const Dp5Quartic qa(a0, a1, f0, f1, m, dt);
      for (int j = lo; j < hi; ++j) states[(long long)j * MD + i] = qa.at((float)((t_out[j] - t0) / dtd));
    }
    y0[i] = a1;
    k1[i] = f1;
  }
}

// Cotangents the dense output of one reverse step hands to the stages.  Row r = ckpt[s] is y0 of step s and y1 of step
// s - 1, and its evaluation f(ckpt[s]) is k1 of step s and k7 of step s - 1 (FSAL): one buffer each.
struct InterpCot {
  float* y;      // of row s: g_y0 of step s + g_y1 of step s - 1 (+ g_states[0] when s == 0)
  float* k17;    // of f(row s): g_k1 of step s + g_k7 of step s - 1
  float* k[4];   // g_k3 .. g_k6 of step s
};

// VJP of the quartic dense output of step s (interp._interp_fit / _interp_evaluate, as ad_commit_kernel forms it).  With
// S_p = sum_j x_j^p g_j over the outputs j of the step (step_out of steps s - 1 and s bound them) and the coefficients
// [e, d, c, b, a] of interp_fit:  g_a = S4, g_b = S3, g_c = S2, g_d = S1, g_e = S0, hence
//   g_y0 = S0 - 11 S2 + 18 S3 - 8 S4,  g_y1 = -5 S2 + 14 S3 - 8 S4,  g_ymid = 16 S2 - 32 S3 + 16 S4,
//   g_f0 = dt (S1 - 4 S2 + 5 S3 - 2 S4),  g_f1 = dt (S2 - 3 S3 + 2 S4),
// and y_mid = y0 + dt sum_l c_mid[l] k_l spreads g_ymid onto y0 and onto k_l with dt c_mid[l].  Writes `cur` (step s's
// own cotangents; zeros for an image without an output in the step) and adds g_y1, g_k7 into `nxt` (row s + 1).
__global__ void __launch_bounds__(256) ad_interp_vjp_kernel(const float* __restrict__ g_states, const double* t_out,
                                                            const double* step_t0, const double* step_dt,
                                                            const int* step_out, int s, int B, InterpCot cur,
                                                            InterpCot nxt, long long MD, long long per_image) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < MD; i += stride) {
    const int b = (int)(i / per_image);
    const long long sb = (long long)s * B + b;
    const int lo = s == 0 ? 1 : step_out[sb - B], hi = step_out[sb];
    float S0 = 0.f, S1 = 0.f, S2 = 0.f, S3 = 0.f, S4 = 0.f;
    if (lo < hi) {
      const double t0 = step_t0[sb], dtd = step_dt[sb];
      for (int j = lo; j < hi; ++j) {
        const float x = (float)((t_out[j] - t0) / dtd);
        const float g = g_states[(long long)j * MD + i];
        const float x2 = x * x;
        S0 += g;
        S1 = fmaf(x, g, S1);
        S2 = fmaf(x2, g, S2);
        S3 = fmaf(x2 * x, g, S3);
        S4 = fmaf(x2 * x2, g, S4);
      }
    }
    const float dt = lo < hi ? (float)step_dt[sb] : 0.f;
    const float gm = 16.f * S2 - 32.f * S3 + 16.f * S4;
    const float dgm = dt * gm;
    float gy0 = S0 - 11.f * S2 + 18.f * S3 - 8.f * S4 + gm;
    if (s == 0) gy0 += g_states[i];
    cur.y[i] = gy0;
    cur.k17[i] = fmaf(kCMid[0], dgm, dt * (S1 - 4.f * S2 + 5.f * S3 - 2.f * S4));
    for (int l = 0; l < 4; ++l) cur.k[l][i] = kCMid[l + 2] * dgm;
    if (lo < hi) {
      nxt.y[i] += -5.f * S2 + 14.f * S3 - 8.f * S4;
      nxt.k17[i] += fmaf(kCMid[6], dgm, dt * (S2 - 3.f * S3 + 2.f * S4));
    }
  }
}

int grid_for(long long n) {
  const long long b = (n + 255) / 256;
  return (int)(b < 148 * 8 ? (b > 0 ? b : 1) : 148 * 8);
}

// u = y0 + dt_b * c * v  (the first stage input of a round, and the initial-step probe)
int row_axpy(const Plan& p, const float* y0, const float* v, float c, const double* dt, float* u, cudaStream_t s) {
  Epi e;
  e.y = y0; e.y_coef = 1.f; e.c_new = c; e.out = u;
  e.row_dt = dt; e.rows_per_image = p.N;
  return rk_apply_rows(e, v, p.M, p.D, s);
}

// The JaSMin window of the forward solve: every evaluation forms its statistic in `tmp` (inside the fused attention
// kernel, else from the exported map: attention_forward) and push() files it in the evaluating images' rings.
struct JasWindow {
  float* tmp;
  float* ring;   // [W, B, H]
  int* count;    // [B]
  int k, W, B, H;
  int push(const double* dt, cudaStream_t s) const {
    ad_jas_push_kernel<<<(B + 127) / 128, 128, 0, s>>>(tmp, dt, ring, count, B, H, W);
    ODV_LAUNCH_CHECK();
    return 0;
  }
};

// f(u) -> out (plain store); with a window, filed for the images with dt_b != 0 (dt == null: all)
int eval_plain(const Plan& p, AdBufs& f, const float* u, float* out, cudaStream_t s, const JasWindow* jw = nullptr,
               const double* dt = nullptr) {
  Epi e;
  e.out = out; e.c_new = 1.f;
  ODV_TRY(eval_forward(p, f.w, f.ctx, u, f.P, nullptr, f.sq, nullptr, 0, &e, s, jw ? jw->tmp : nullptr, jw ? jw->k : 0));
  return jw ? jw->push(dt, s) : 0;
}

// The stages k2..k6 of one step of every image from y0 and k[0] = k1 (FSAL): u2 by a row pass, then the evaluation of
// u_{m+1} stores k_{m+1} and its epilogue forms u_{m+2} in u (y1 after k6).  ctx(m): the intermediates of that
// evaluation.  y1 == nullptr recomputes the intermediates only: k6's output GEMM is skipped.  jw: the forward solve's
// JaSMin window (null in the reverse sweep).
template <class Ctx>
int dp_stages(const Plan& p, const WeightBufs& w, Ctx ctx, float* P, float* sq, const float* y0, float* const* k,
              const double* dt, float* u, float* y1, cudaStream_t s, const JasWindow* jw = nullptr) {
  ODV_TRY(row_axpy(p, y0, k[0], kDopri5.a[1][0], dt, u, s));
  for (int m = 1; m <= 5; ++m) {
    if (!y1 && m == 5) return eval_forward(p, w, ctx(m), u, P, nullptr, sq, nullptr, 0, nullptr, s);
    Epi e = rk_epilogue(kDopri5, m, 1.f, y0, k, m == 5 ? y1 : u);   // dt_b is applied per image in the epilogue
    e.row_dt = dt; e.rows_per_image = p.N;
    e.k_store = k[m];
    ODV_TRY(eval_forward(p, w, ctx(m), u, P, nullptr, sq, nullptr, 0, &e, s, jw ? jw->tmp : nullptr, jw ? jw->k : 0));
    if (jw) ODV_TRY(jw->push(dt, s));
  }
  return 0;
}

struct Host {
  int* pinned = nullptr;             // [2][4] sync words of rounds with r & 1 == 0 / 1
  cudaEvent_t ev[2] = {nullptr, nullptr};
  ~Host() {
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
  }
};
int* pinned_slots() {
  static thread_local int* p = nullptr;
  if (!p && cudaHostAlloc(reinterpret_cast<void**>(&p), 8 * sizeof(int), cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    p = nullptr;
  }
  return p;
}

// the output times as fp64, checked: 2..kMaxOut finite, strictly increasing values
int read_t_out(const float* t_out_host, int n_out, std::vector<double>& t_out) {
  if (!t_out_host || n_out < 2 || n_out > kMaxOut)
    return set_error(ODEVIT_ERR_INVALID_ARG, "t_out must hold 2..%d host values, got %d", kMaxOut, (int)n_out);
  t_out.resize(n_out);
  for (int i = 0; i < n_out; ++i) {
    t_out[i] = (double)t_out_host[i];
    if (!std::isfinite(t_out[i])) return set_error(ODEVIT_ERR_INVALID_ARG, "t_out[%d] is not finite", i);
    if (i > 0 && !(t_out[i] > t_out[i - 1]))
      return set_error(ODEVIT_ERR_INVALID_ARG, "t_out must be strictly increasing (t_out[%d]=%g, t_out[%d]=%g)", i - 1,
                       t_out[i - 1], i, t_out[i]);
  }
  return 0;
}

// ---- reverse sweep (odevit_solve_adaptive_bwd) ---------------------------------------------------------------------
struct AdBwdBufs {
  BwdBufs b;          // the fixed-grid reverse-sweep buffers: folded weights, VJP scratch, G (b.gy), dd, accumulators
  StageCtx ctx[6];    // without a tape: f(ckpt[s]) (ctx[0] = b.ctx[0], also every replay evaluation) and k2..k6 of step s
  float* k[6];        // k1..k6 of the step being replayed or recomputed
  float* mu[6];       // [1..5]: mu of the evaluations k2..k6 of the reverse step
  InterpCot cot[2];   // dense-output cotangents of rows with s & 1 == 0 / 1
  double* t_out;      // [kMaxOut]
};

AdBwdBufs layout_adaptive_bwd(const Plan& p, Arena& a) {
  AdBwdBufs f;
  const size_t MD = (size_t)p.M * p.D;
  f.b = layout_bwd(p, a, 1);
  f.ctx[0] = f.b.ctx[0];
  for (int i = 1; i < 6; ++i) f.ctx[i] = take_ctx(p, a, true);
  for (int i = 0; i < 6; ++i) f.k[i] = a.f32(MD);
  f.mu[0] = nullptr;
  for (int i = 1; i < 6; ++i) f.mu[i] = a.f32(MD);
  for (InterpCot& c : f.cot) {
    c.y = a.f32(MD);
    c.k17 = a.f32(MD);
    for (float*& k : c.k) k = a.f32(MD);
  }
  f.t_out = reinterpret_cast<double*>(a.take((size_t)kMaxOut * 8));
  return f;
}

}  // namespace

size_t solve_adaptive_workspace_bytes(const Plan& p) {
  Arena a(nullptr);
  layout_adaptive(p, a);
  return a.off;
}

size_t solve_adaptive_bwd_workspace_bytes(const Plan& p) {
  Arena a(nullptr);
  layout_adaptive_bwd(p, a);
  return a.off;
}

}  // namespace odevit

using namespace odevit;

namespace {
// The accepted-step record of odevit_solve_adaptive_record ([cap, B] each; t0 == nullptr: no record).
struct StepRecord {
  double* t0 = nullptr;
  double* dt = nullptr;
  int32_t* out = nullptr;
  int cap = 0;
};

// The attention outputs of odevit_solve_adaptive_attn (all null: none).
struct AttnOut {
  float* p_last = nullptr;    // [B, H, N, N]
  float* ring = nullptr;      // [W, B, H]
  int32_t* count = nullptr;   // [B]
  int k = 0, window = 0;
};

int solve_adaptive_impl(const odevit_desc* desc, const odevit_weights* w, const float* x0, const float* t_out_host,
                        int32_t n_out, double rtol, double atol, double first_step, int32_t max_num_steps,
                        float* states, int32_t* nfe, int32_t* accepted, int32_t* rejected, const StepRecord& rec,
                        const AttnOut& at, void* workspace, size_t workspace_bytes, odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  if (p.any_drop) return set_error(ODEVIT_ERR_INVALID_ARG, "the adaptive solve is inference-only: dropout must be 0");
  if ((at.p_last || at.ring) && p.variant == ODEVIT_FIELD_MACARON)
    return set_error(ODEVIT_ERR_INVALID_ARG, "MACARON exposes no attention map (need_weights=False, macaron.py:60-65)");
  if (at.p_last) ODV_TRY(check_device_ptr(at.p_last, "p_last"));
  if (at.ring) {
    ODV_TRY(check_device_ptr(at.ring, "jas_ring"));
    if (!at.count) return set_error(ODEVIT_ERR_INVALID_ARG, "jas_count is NULL");
    ODV_TRY(check_device_ptr(at.count, "jas_count"));
    if (at.k < 0 || at.k > p.N || at.window < 1)
      return set_error(ODEVIT_ERR_INVALID_ARG, "jas_k %d (0..tokens) / jas_window %d (>= 1) out of range", at.k,
                       at.window);
  }
  ODV_TRY(check_device_ptr(x0, "x0"));
  ODV_TRY(check_device_ptr(states, "states"));
  if (nfe) ODV_TRY(check_device_ptr(nfe, "nfe"));
  if (accepted) ODV_TRY(check_device_ptr(accepted, "accepted"));
  if (rejected) ODV_TRY(check_device_ptr(rejected, "rejected"));
  if (rec.t0) {
    if (rec.cap < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "step_cap %d < 1", rec.cap);
    ODV_TRY(check_device_ptr(rec.t0, "step_t0"));
    ODV_TRY(check_device_ptr(rec.dt, "step_dt"));
    ODV_TRY(check_device_ptr(rec.out, "step_out"));
  }
  std::vector<double> t_out;
  ODV_TRY(read_t_out(t_out_host, n_out, t_out));
  if (!(rtol >= 0.0 && atol >= 0.0 && rtol + atol > 0.0 && std::isfinite(rtol) && std::isfinite(atol)))
    return set_error(ODEVIT_ERR_INVALID_ARG, "rtol %g / atol %g: both >= 0, finite, not both 0", rtol, atol);
  if (!std::isfinite(first_step)) return set_error(ODEVIT_ERR_INVALID_ARG, "first_step is not finite");
  if (max_num_steps < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "max_num_steps %d < 1", (int)max_num_steps);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  ODV_CUDA(cudaStreamIsCapturing(s, &cap));
  if (cap != cudaStreamCaptureStatusNone)
    return set_error(ODEVIT_ERR_UNSUPPORTED, "the adaptive solve synchronises once per round: it cannot be captured");
  Arena a(workspace);
  AdBufs f = layout_adaptive(p, a);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  Host h;
  h.pinned = pinned_slots();
  if (!h.pinned) return set_error(ODEVIT_ERR_CUDA, "cudaHostAlloc of the round counters failed");
  for (cudaEvent_t& e : h.ev) ODV_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));

  const int B = p.B, N = p.N, D = p.D;
  const long long MD = (long long)p.M * D;
  const float frtol = (float)rtol, fatol = (float)atol;
  ODV_TRY(prepare_weights(p, w, f.w, s));
  ODV_CUDA(cudaMemcpyAsync(f.t_out, t_out.data(), (size_t)n_out * 8, cudaMemcpyHostToDevice, s));
  ODV_CUDA(cudaMemcpyAsync(states, x0, (size_t)MD * 4, cudaMemcpyDeviceToDevice, s));
  ODV_CUDA(cudaMemcpyAsync(f.y0, x0, (size_t)MD * 4, cudaMemcpyDeviceToDevice, s));
  if (rec.t0) {   // entries past an image's count stay zero: row s of step_dt is then the dt of reverse step s
    const size_t n = (size_t)rec.cap * B;
    ODV_CUDA(cudaMemsetAsync(rec.t0, 0, n * 8, s));
    ODV_CUDA(cudaMemsetAsync(rec.dt, 0, n * 8, s));
    ODV_CUDA(cudaMemsetAsync(rec.out, 0, n * 4, s));
  }
  const JasWindow jas{f.jas, at.ring, at.count, at.k, at.window, B, p.H};
  const JasWindow* jw = at.ring ? &jas : nullptr;
  if (jw) {
    ODV_CUDA(cudaMemsetAsync(at.ring, 0, (size_t)at.window * B * p.H * 4, s));
    ODV_CUDA(cudaMemsetAsync(at.count, 0, (size_t)B * 4, s));
  }
  ad_init_kernel<<<(B + 255) / 256, 256, 0, s>>>(f.t, f.dt, f.out_next, f.accept, f.sync, f.t_out,
                                                  first_step > 0 ? first_step : 0.0, B);
  ODV_LAUNCH_CHECK();
  ODV_TRY(eval_plain(p, f, f.y0, f.k[0], s, jw));   // f0
  const int row_blocks = (p.M + 7) / 8;
  if (!(first_step > 0)) {
    ad_rowsq_kernel<RS_INIT><<<row_blocks, 256, 0, s>>>(f.y0, nullptr, f.k[0], nullptr, nullptr, nullptr, nullptr,
                                                       nullptr, nullptr, nullptr, frtol, fatol, p.M, N, D, f.row0, f.row1);
    ODV_LAUNCH_CHECK();
    ad_init_step_kernel<<<B, kRedThreads, 0, s>>>(0, f.row0, f.row1, N, D, f.h0, f.d1, f.dt);
    ODV_LAUNCH_CHECK();
    ODV_TRY(row_axpy(p, f.y0, f.k[0], 1.f, f.h0, f.u, s));   // probe y0 + h0 f0
    ODV_TRY(eval_plain(p, f, f.u, f.k[1], s, jw));
    ad_rowsq_kernel<RS_D2><<<row_blocks, 256, 0, s>>>(f.y0, nullptr, f.k[0], f.k[1], nullptr, nullptr, nullptr, nullptr,
                                                     nullptr, nullptr, frtol, fatol, p.M, N, D, f.row0, nullptr);
    ODV_LAUNCH_CHECK();
    ad_init_step_kernel<<<B, kRedThreads, 0, s>>>(1, f.row0, nullptr, N, D, f.h0, f.d1, f.dt);
    ODV_LAUNCH_CHECK();
  }
  const int nfe_base = first_step > 0 ? 1 : 2;

  // one round: attempted step of every image; reads scalar slot r & 1, the control kernel writes the other
  auto round = [&](long long r) -> int {
    const int c = (int)(r & 1), n = c ^ 1;
    const double* dt = f.dt + (size_t)c * B;
    ODV_CUDA(cudaMemsetAsync(f.sync + c, 0, sizeof(int), s));
    ODV_TRY(dp_stages(p, f.w, [&](int) { return f.ctx; }, f.P, f.sq, f.y0, f.k, dt, f.u, f.y1, s, jw));
    ODV_TRY(eval_plain(p, f, f.y1, f.k[6], s, jw, dt));   // k7 = f(y1)
    ad_rowsq_kernel<RS_ERR><<<row_blocks, 256, 0, s>>>(f.y0, f.y1, f.k[0], nullptr, f.k[2], f.k[3], f.k[4], f.k[5],
                                                       f.k[6], dt, frtol, fatol, p.M, N, D, f.row0, nullptr);
    ODV_LAUNCH_CHECK();
    ad_control_kernel<<<B, kRedThreads, 0, s>>>(f.row0, N, D, B, f.t + (size_t)c * B, dt, f.out_next + (size_t)c * B,
                                                f.t + (size_t)n * B, f.dt + (size_t)n * B, f.out_next + (size_t)n * B,
                                                f.accept, f.attempts, f.n_acc, f.n_rej, f.t_out, n_out, max_num_steps,
                                                nfe_base, nfe, accepted, rejected, f.sync + c, f.sync + 2, rec.t0,
                                                rec.dt, rec.out, rec.cap);
    ODV_LAUNCH_CHECK();
    ad_commit_kernel<<<grid_for(MD), 256, 0, s>>>(f.y0, f.y1, f.k[0], f.k[2], f.k[3], f.k[4], f.k[5], f.k[6], f.accept,
                                                  f.t + (size_t)c * B, dt, f.out_next + (size_t)c * B,
                                                  f.out_next + (size_t)n * B, f.t_out, states, MD, (long long)N * D);
    ODV_LAUNCH_CHECK();
    ODV_CUDA(cudaMemcpyAsync(h.pinned + 4 * c, f.sync, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
    ODV_CUDA(cudaEventRecord(h.ev[c], s));
    return 0;
  };

  ODV_TRY(round(0));
  for (long long r = 0;; ++r) {
    ODV_TRY(round(r + 1));   // keeps the queue fed while round r's count comes back
    ODV_CUDA(cudaEventSynchronize(h.ev[r & 1]));
    const int* hs = h.pinned + 4 * (r & 1);
    const int active = hs[r & 1], err = hs[2];
    if (err != kNoError) {
      ODV_CUDA(cudaStreamSynchronize(s));
      const int b = err / 4, kind = err % 4;
      if (kind == kErrMax)
        return set_error(ODEVIT_ERR_NOT_CONVERGED, "image %d: max_num_steps (%d) exceeded before t_out[-1]", b,
                         (int)max_num_steps);
      if (kind == kErrNonFinite) return set_error(ODEVIT_ERR_NOT_CONVERGED, "image %d: non-finite error ratio", b);
      if (kind == kErrRecord)
        return set_error(ODEVIT_ERR_WORKSPACE, "image %d: more than step_cap (%d) accepted steps: the step record is full",
                         b, rec.cap);
      return set_error(ODEVIT_ERR_NOT_CONVERGED, "image %d: underflow in dt (t + dt == t)", b);
    }
    if (active == 0) {
      // the look-ahead round r + 1 is a no-op for every image; wait for it so that its copy into the pinned slots
      // cannot land in a later call's
      ODV_CUDA(cudaEventSynchronize(h.ev[(r + 1) & 1]));
      break;
    }
    if (r > (long long)max_num_steps + 1) {
      ODV_CUDA(cudaStreamSynchronize(s));
      return set_error(ODEVIT_ERR_CUDA, "adaptive solve: %d images still active after %lld rounds", active, r + 1);
    }
  }
  // block.attentions is the map of each image's last evaluation, k7 = f(y1) of its last accepted step; y0 holds that y1
  // (finished images repeat it).  The forward's kernels have no order-dependent reduction, so this evaluation repeats
  // that map bit for bit.  It is not counted in nfe and not filed in the window.
  if (at.p_last) ODV_TRY(eval_forward(p, f.w, f.ctx, f.y0, f.P, at.p_last, f.sq, nullptr, 0, nullptr, s));
  return 0;
}
}  // namespace

extern "C" int odevit_solve_adaptive(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                     const float* t_out_host, int32_t n_out, double rtol, double atol,
                                     double first_step, int32_t max_num_steps, float* states, int32_t* nfe,
                                     int32_t* accepted, int32_t* rejected, void* workspace, size_t workspace_bytes,
                                     odevit_stream_t stream) {
  return solve_adaptive_impl(desc, w, x0, t_out_host, n_out, rtol, atol, first_step, max_num_steps, states, nfe,
                             accepted, rejected, StepRecord{}, AttnOut{}, workspace, workspace_bytes, stream);
}

extern "C" int odevit_solve_adaptive_record(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                            const float* t_out_host, int32_t n_out, double rtol, double atol,
                                            double first_step, int32_t max_num_steps, float* states, int32_t* nfe,
                                            int32_t* accepted, int32_t* rejected, int32_t step_cap, double* step_t0,
                                            double* step_dt, int32_t* step_out, void* workspace,
                                            size_t workspace_bytes, odevit_stream_t stream) {
  if (!step_t0 || !step_dt || !step_out) return set_error(ODEVIT_ERR_INVALID_ARG, "step_t0 / step_dt / step_out is NULL");
  StepRecord rec;
  rec.t0 = step_t0; rec.dt = step_dt; rec.out = step_out; rec.cap = step_cap;
  return solve_adaptive_impl(desc, w, x0, t_out_host, n_out, rtol, atol, first_step, max_num_steps, states, nfe,
                             accepted, rejected, rec, AttnOut{}, workspace, workspace_bytes, stream);
}

extern "C" int odevit_solve_adaptive_attn(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                          const float* t_out_host, int32_t n_out, double rtol, double atol,
                                          double first_step, int32_t max_num_steps, float* states, int32_t* nfe,
                                          int32_t* accepted, int32_t* rejected, int32_t step_cap, double* step_t0,
                                          double* step_dt, int32_t* step_out, float* p_last, int32_t jas_k,
                                          int32_t jas_window, float* jas_ring, int32_t* jas_count, void* workspace,
                                          size_t workspace_bytes, odevit_stream_t stream) {
  StepRecord rec;
  if (step_t0 || step_dt || step_out) {
    if (!step_t0 || !step_dt || !step_out)
      return set_error(ODEVIT_ERR_INVALID_ARG, "step_t0 / step_dt / step_out: give all three or none");
    rec.t0 = step_t0; rec.dt = step_dt; rec.out = step_out; rec.cap = step_cap;
  }
  AttnOut at;
  at.p_last = p_last;
  at.ring = jas_ring; at.count = jas_count; at.k = jas_k; at.window = jas_window;
  return solve_adaptive_impl(desc, w, x0, t_out_host, n_out, rtol, atol, first_step, max_num_steps, states, nfe,
                             accepted, rejected, rec, at, workspace, workspace_bytes, stream);
}

namespace {
struct AdResBufs {
  WeightBufs w;
  float* kbuf;
  int* next_image;
};
AdResBufs layout_adaptive_resident(const Plan& p, Arena& a) {
  AdResBufs f;
  f.w = take_weights(p, a);
  f.kbuf = a.f32(solve_resident_adaptive_scratch_floats(p));
  f.next_image = reinterpret_cast<int*>(a.take(16));
  return f;
}
}  // namespace

size_t odevit::solve_adaptive_resident_workspace_bytes(const Plan& p) {
  Arena a(nullptr);
  layout_adaptive_resident(p, a);
  return a.off;
}

extern "C" int odevit_solve_adaptive_resident(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                              const float* t_out_host, int32_t n_out, double rtol, double atol,
                                              double first_step, int32_t max_num_steps, float* states, int32_t* nfe,
                                              int32_t* accepted, int32_t* rejected, int32_t* status, void* workspace,
                                              size_t workspace_bytes, odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  if (p.any_drop) return set_error(ODEVIT_ERR_INVALID_ARG, "the adaptive solve is inference-only: dropout must be 0");
  if (const char* why = solve_resident_adaptive_envelope(p))
    return set_error(ODEVIT_ERR_UNSUPPORTED, "the on-chip adaptive solve covers this shape only with %s", why);
  ODV_TRY(check_device_ptr(x0, "x0"));
  ODV_TRY(check_device_ptr(states, "states"));
  if (!status) return set_error(ODEVIT_ERR_INVALID_ARG, "status is NULL");
  ODV_TRY(check_device_ptr(status, "status"));
  if (nfe) ODV_TRY(check_device_ptr(nfe, "nfe"));
  if (accepted) ODV_TRY(check_device_ptr(accepted, "accepted"));
  if (rejected) ODV_TRY(check_device_ptr(rejected, "rejected"));
  std::vector<double> t_out;
  if (n_out > kResidentMaxGrid)
    return set_error(ODEVIT_ERR_INVALID_ARG, "t_out must hold 2..%d host values on the chip, got %d", kResidentMaxGrid,
                     (int)n_out);
  ODV_TRY(read_t_out(t_out_host, n_out, t_out));
  if (!(rtol >= 0.0 && atol >= 0.0 && rtol + atol > 0.0 && std::isfinite(rtol) && std::isfinite(atol)))
    return set_error(ODEVIT_ERR_INVALID_ARG, "rtol %g / atol %g: both >= 0, finite, not both 0", rtol, atol);
  if (!std::isfinite(first_step)) return set_error(ODEVIT_ERR_INVALID_ARG, "first_step is not finite");
  if (max_num_steps < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "max_num_steps %d < 1", (int)max_num_steps);
  Arena a(workspace);
  AdResBufs f = layout_adaptive_resident(p, a);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  ODV_TRY(prepare_weights(p, w, f.w, s));
  ODV_CUDA(cudaMemcpyAsync(states, x0, (size_t)p.M * p.D * 4, cudaMemcpyDeviceToDevice, s));
  return solve_resident_adaptive(p, f.w, x0, t_out.data(), n_out, rtol, atol, first_step > 0 ? first_step : 0.0,
                                 max_num_steps, states, nfe, accepted, rejected, status, f.kbuf, f.next_image, s);
}

extern "C" size_t odevit_adaptive_tape_bytes(const odevit_desc* desc, int32_t S) {
  Plan p{};
  if (make_plan(desc, &p)) return 0;
  if (S < 1) { set_error(ODEVIT_ERR_INVALID_ARG, "S %d < 1", (int)S); return 0; }
  return tape_bytes(p, 6LL * S + 1);
}

// Reverse sweep with the recorded steps frozen.  Evaluation e = 6 s + i of the replay is f(ckpt[s]) for i = 0 (k1 of step
// s, k7 of step s - 1) and k_{i+1} of step s for i = 1..5.  With G the cotangent of ckpt[s + 1] (everything downstream of
// it), reverse step s runs
//   lambda_6 = g_k6 + dt_b c_sol[5] G                                   (a row pass: rk_apply_rows with EPI_ROWDT)
//   VJP of k6 .. k2 (rk_step_vjp with row_dt): mu_m, and in the mu GEMM's EPI_RK | EPI_ROWDT epilogue
//     lambda_{m-1} = g_k{m-1} + dt_b (beta[m-1][m-1] mu_m + sum_{l>m} beta[l-1][m-1] mu_l + c_sol[m-1] G)
//   VJP of f(ckpt[s]) with lambda_1 + g_k7 of step s - 1 (the same evaluation):  G <- G + sum mu + g of row s
// where the g_* are the dense output's cotangents (ad_interp_vjp_kernel).  Reverse step S is that last VJP alone, at each
// image's end state.  A finished image has dt_b = 0 and no outputs in its remaining steps: lambda = 0 there.
// f(ckpt[S]) is also the evaluation whose map is p_last (each image's last one): g_p_last enters its attention VJP.
namespace {
int solve_adaptive_bwd_impl(const odevit_desc* desc, const odevit_weights* w, const float* x0, const float* t_out_host,
                            int32_t n_out, const double* step_t0, const double* step_dt, const int32_t* step_out,
                            int32_t step_cap, const int32_t* n_steps_host, const float* g_states,
                            const float* g_p_last, float* g_x0, const odevit_weight_grads* gw, float* ckpt, void* tape,
                            size_t tape_bytes, void* workspace, size_t workspace_bytes, odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  if (p.any_drop) return set_error(ODEVIT_ERR_INVALID_ARG, "the adaptive solve has no dropout: dropout must be 0");
  if (!gw) return set_error(ODEVIT_ERR_INVALID_ARG, "weight-gradient struct is NULL");
  if (g_p_last) {
    if (p.variant == ODEVIT_FIELD_MACARON)
      return set_error(ODEVIT_ERR_INVALID_ARG, "MACARON exposes no attention map (need_weights=False, macaron.py:60-65)");
    ODV_TRY(check_device_ptr(g_p_last, "g_p_last"));
  }
  ODV_TRY(check_device_ptr(x0, "x0"));
  ODV_TRY(check_device_ptr(g_states, "g_states"));
  ODV_TRY(check_device_ptr(g_x0, "g_x0"));
  ODV_TRY(check_device_ptr(ckpt, "ckpt"));
  ODV_TRY(check_device_ptr(step_t0, "step_t0"));
  ODV_TRY(check_device_ptr(step_dt, "step_dt"));
  ODV_TRY(check_device_ptr(step_out, "step_out"));
  std::vector<double> t_out;
  ODV_TRY(read_t_out(t_out_host, n_out, t_out));
  if (step_cap < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "step_cap %d < 1", (int)step_cap);
  if (!n_steps_host) return set_error(ODEVIT_ERR_INVALID_ARG, "n_steps_host is NULL");
  int S = 0;
  for (int b = 0; b < p.B; ++b) {
    const int n = n_steps_host[b];
    if (n < 0 || n > step_cap)
      return set_error(ODEVIT_ERR_INVALID_ARG, "n_steps[%d] = %d outside [0, step_cap = %d]", b, n, (int)step_cap);
    S = n > S ? n : S;
  }
  if (S < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "no image has an accepted step");
  if (tape) ODV_TRY(check_tape(p, tape, tape_bytes, 6LL * S + 1));
  Arena a(workspace);
  AdBwdBufs f = layout_adaptive_bwd(p, a);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  BwdBufs& b = f.b;
  const int B = p.B, N = p.N;
  const long long MD = (long long)p.M * p.D;
  const bool need_c2 = wants_c2(gw);
  float* G = b.gy;
  ODV_TRY(prepare_weights(p, w, b.w, s));
  ODV_CUDA(cudaMemcpyAsync(f.t_out, t_out.data(), (size_t)n_out * 8, cudaMemcpyHostToDevice, s));
  ODV_CUDA(cudaMemsetAsync(b.G1, 0, b.acc_bytes, s));
  ODV_CUDA(cudaMemcpyAsync(ckpt, x0, (size_t)MD * 4, cudaMemcpyDeviceToDevice, s));

  auto row = [&](int r) { return ckpt + (size_t)r * MD; };
  auto dt_of = [&](int st) { return step_dt + (size_t)st * B; };
  // context of evaluation 6 st + i: its tape slot, else the recompute buffer (the replay's own evaluations all go to
  // ctx[0], which leaves f(ckpt[S]) there for reverse step S)
  auto ctx_of = [&](int st, int i) -> StageCtx {
    return tape ? tape_ctx(p, tape, 6LL * st + i) : f.ctx[i];
  };
  auto eval_k1 = [&](int r, const StageCtx& c) -> int {   // k1 = f(ckpt[r])
    Epi e;
    e.out = f.k[0]; e.c_new = 1.f;
    return eval_forward(p, b.w, c, row(r), b.P, nullptr, b.sq, nullptr, 0, &e, s);
  };
  // the stages k2..k6 of step st from ckpt[st] and k1.  replay: the k6 evaluation's epilogue writes ckpt[st + 1];
  // recompute: only the contexts are needed
  auto stages = [&](int st, bool replay) -> int {
    auto ctx = [&](int m) { return tape ? ctx_of(st, m) : f.ctx[replay ? 0 : m]; };
    return dp_stages(p, b.w, ctx, b.P, b.sq, row(st), f.k, dt_of(st), b.u, replay ? row(st + 1) : nullptr, s);
  };

  // ---- replay: ckpt[1..S] (and the tape) ----
  ODV_TRY(eval_k1(0, tape ? ctx_of(0, 0) : f.ctx[0]));
  for (int st = 0; st < S; ++st) {
    ODV_TRY(stages(st, true));
    ODV_TRY(eval_k1(st + 1, tape ? ctx_of(st + 1, 0) : f.ctx[0]));
  }

  // ---- reverse ----
  auto interp_vjp = [&](int st) -> int {   // step st's own cotangents into cot[st & 1], g_y1 / g_k7 added to row st + 1's
    ad_interp_vjp_kernel<<<grid_for(MD), 256, 0, s>>>(g_states, f.t_out, step_t0, step_dt, step_out, st, B,
                                                      f.cot[st & 1], f.cot[(st + 1) & 1], MD, (long long)N * p.D);
    ODV_LAUNCH_CHECK();
    return 0;
  };
  auto seed = [&](const float* gk, float c, const double* dt) -> int {   // dd = scaler * (gk + dt_b c G)
    Epi e;
    e.y = gk; e.y_coef = 1.f; e.c_new = c;
    e.row_dt = dt; e.rows_per_image = N;
    e.out2 = b.dd; e.out2_scale = p.scaler; e.aux_type = p.dd_type;
    return rk_apply_rows(e, G, p.M, p.D, s);
  };
  const Tableau& tb = kDopri5;

  ODV_CUDA(cudaMemsetAsync(G, 0, (size_t)MD * 4, s));
  ODV_CUDA(cudaMemsetAsync(f.cot[S & 1].y, 0, (size_t)MD * 4, s));
  ODV_CUDA(cudaMemsetAsync(f.cot[S & 1].k17, 0, (size_t)MD * 4, s));
  ODV_TRY(interp_vjp(S - 1));
  ODV_TRY(seed(f.cot[S & 1].k17, 0.f, dt_of(S - 1)));   // G = 0: dd = scaler * g_k7 of step S - 1
  {   // reverse step S: f(ckpt[S]) alone, G <- G + its mu + g of row S
    Epi e = rk_vjp_row_epilogue(G, f.mu, 0, &f.cot[S & 1].y, 1, G);
    e.aux_type = p.dd_type;
    ODV_TRY(eval_vjp(p, b.w, ctx_of(S, 0), b, g_p_last, need_c2, gw, 6LL * S, e, s));
  }
  for (int st = S - 1; st >= 0; --st) {
    ODV_TRY(seed(f.cot[st & 1].k[3], tb.b[5], dt_of(st)));   // lambda_6
    if (!tape) {
      ODV_TRY(eval_k1(st, f.ctx[0]));
      ODV_TRY(stages(st, false));
    }
    if (st > 0) ODV_TRY(interp_vjp(st - 1));
    // the dense output's cotangents of k1 .. k5 (k2 has no dense-output weight: c_mid[1] = 0) and of row st
    const InterpCot& cot = f.cot[st & 1];
    const float* g[5] = {cot.k17, nullptr, cot.k[0], cot.k[1], cot.k[2]};
    StageCtx ctx[6];
    for (int i = 0; i < 6; ++i) ctx[i] = ctx_of(st, i);
    ODV_TRY(rk_step_vjp(p, b, tb, 1.f, dt_of(st), g, f.mu, ctx, 6LL * st, nullptr, need_c2, gw,
                        rk_vjp_row_epilogue(G, f.mu, 5, &cot.y, 1, st == 0 ? g_x0 : G), s));
  }
  return finish_grads(p, w, gw, b, s);
}
}  // namespace

extern "C" int odevit_solve_adaptive_bwd(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                         const float* t_out_host, int32_t n_out, const double* step_t0,
                                         const double* step_dt, const int32_t* step_out, int32_t step_cap,
                                         const int32_t* n_steps_host, const float* g_states, float* g_x0,
                                         const odevit_weight_grads* gw, float* ckpt, void* tape, size_t tape_bytes,
                                         void* workspace, size_t workspace_bytes, odevit_stream_t stream) {
  return solve_adaptive_bwd_impl(desc, w, x0, t_out_host, n_out, step_t0, step_dt, step_out, step_cap, n_steps_host,
                                 g_states, nullptr, g_x0, gw, ckpt, tape, tape_bytes, workspace, workspace_bytes, stream);
}

extern "C" int odevit_solve_adaptive_bwd_attn(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                              const float* t_out_host, int32_t n_out, const double* step_t0,
                                              const double* step_dt, const int32_t* step_out, int32_t step_cap,
                                              const int32_t* n_steps_host, const float* g_states,
                                              const float* g_p_last, float* g_x0, const odevit_weight_grads* gw,
                                              float* ckpt, void* tape, size_t tape_bytes, void* workspace,
                                              size_t workspace_bytes, odevit_stream_t stream) {
  if (!g_p_last) return set_error(ODEVIT_ERR_INVALID_ARG, "g_p_last is NULL (odevit_solve_adaptive_bwd takes none)");
  return solve_adaptive_bwd_impl(desc, w, x0, t_out_host, n_out, step_t0, step_dt, step_out, step_cap, n_steps_host,
                                 g_states, g_p_last, g_x0, gw, ckpt, tape, tape_bytes, workspace, workspace_bytes, stream);
}
