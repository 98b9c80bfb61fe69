// Host-side orchestration structs shared by api.cu (solver loops, PARALLEL / PARALLEL_L2 fields) and
// field_macaron.cu (MACARON field).  Not part of the ABI.
#pragma once
#include "internal.h"

namespace odevit {

struct Plan {
  int B, N, D, H, hid, d, M;
  int variant, precision, act;  // act = DType of activation buffers
  int dd_type;                  // DType of the cotangent buffer entering a field VJP
  float scaler;
  long long BHNN;
  // training-mode dropout (0 = off) and the per-call seed of the mask generator
  float p_attn, p_proj, p_mlp;
  uint32_t seed_lo, seed_hi;
  const uint32_t* seed_dev;   // device-resident seed (or null): keys come from `drop_keys`
  uint32_t* drop_keys;        // [kDropKeyEvals * DS_SITES] key table in the workspace (device seed only)
  bool any_drop;
  bool split_out;   // proj / mlp dropout on: out-proj and fc2 run as two GEMMs (their outputs take different masks)
  // fp32 mode on the tensor core: scratch for the bf16 hi / lo split of a GEMM's operands (api.cu::gemm_split3); set by
  // the workspace layouts (null: the FFMA kernel runs)
  mutable void* split_a = nullptr;
  mutable void* split_b = nullptr;
  mutable size_t split_a_bytes = 0, split_b_bytes = 0;
  // deterministic mode: scratch for the partial slabs of the fixed-order reductions; set by layout_bwd (null otherwise)
  mutable float* det_ws = nullptr;
  mutable size_t det_ws_bytes = 0;
};
// mask of dropout site `site` in field evaluation `e` (e = step * stages + stage)
Drop make_drop(const Plan& p, int site, long long e);

struct Arena {
  char* base;
  size_t off = 0;
  explicit Arena(void* b) : base(reinterpret_cast<char*>(b)) {}
  void* take(size_t bytes) {
    off = (off + 1023) & ~size_t(1023);
    void* p = base ? base + off : nullptr;
    off += bytes;
    return p;
  }
  float* f32(size_t n) { return reinterpret_cast<float*>(take(n * 4)); }
};

// Activation-typed copies of the weights, laid out the same way for every variant:
//   w1cat  [3D+hid, D]  = [in-proj rows (q rows carry 1/sqrt(d)) ; fc1 rows]     (+ transpose [D, 3D+hid])
//   w2cat  [D, D+hid]   = [out-proj | fc2] along K                              (+ transpose [D+hid, D])
// PARALLEL / PARALLEL_L2 fold the CenterNorm affines into w1cat and run each concatenation as ONE
// GEMM; MACARON uses the four blocks as separate operands (views with the concatenated leading dim).
struct WeightBufs {
  void *w1cat, *w1catT, *w2cat, *w2catT;
  float *b1cat, *b2;
  float* fmean;   // [3D+hid] row means of W1cat (what the transposed copy subtracts)
  const odevit_weights* user;  // the caller's fp32 parameters (biases, LayerNorm affines, res_scale)
};

// Intermediates of ONE field evaluation that its VJP needs (a tape slot or a recompute buffer).
struct StageCtx {
  void *xc, *qkv, *oh, *hpre;
  float* lse;  // [B,H,N] log2-domain row log-sum-exp of the attention (reverse sweep only)
  // MACARON only: xc = LN1(u), hpre/oh[:, D:] = first half-FFN; the rest of the chain:
  float *x0, *x1, *x2;   // [M,D] fp32: the stage input, after the first half-FFN, after attention
  void *n2, *n3;         // [M,D] LN2(x1), LN3(x2)
  void *hpre3, *h3;      // [M,hid] second half-FFN
};

struct BwdBufs {
  uint32_t* drop_keys;   // device-seeded dropout: key table (head of the workspace) or null
  WeightBufs w;
  StageCtx ctx[4];
  float *P, *dP;
  float* u;
  float* k[3];
  void *dd, *dO, *dz;
  float* mu[4];
  float* gy;
  float *delta, *dq_scratch;
  float *G1, *c1, *G2, *c2, *c3;
  size_t acc_bytes;  // G1..c3 are contiguous: one memset
  // MACARON / L2 scratch
  float* dn;    // [M,D] fp32: cotangent of a LayerNorm output
  void* ddc;    // [M,D] act: cast/scaled copy of the running cotangent (GEMM operand)
  float* sq;    // [2,B,H,N] fp32: |q|^2, |k|^2 per head (L2 attention)
  float* tmp;   // [M,D] fp32: masked fc2 output waiting for the out-proj GEMM (split_out)
  void *dd1, *dd2;  // [M,D] act: the cotangent under the fc2-output / out-proj-output masks (split_out)
};

// GEMM dispatch: tcgen05 in bf16 mode where the kernel covers the problem, FFMA otherwise.
int gemm(const Plan& p, const GemmArgs& g, cudaStream_t s);

// Plan, workspace pieces, argument checks and weight preparation shared by the solve entry points (api.cu).
int make_plan(const odevit_desc* desc, Plan* p);
WeightBufs take_weights(const Plan& p, Arena& a);
StageCtx take_ctx(const Plan& p, Arena& a, bool with_hpre);
void split_scratch(const Plan& p, Arena& a);   // fp32 mode: bf16 split scratch of the tensor-core GEMMs
int check_ws(const void* ws, size_t have, size_t need);
int check_device_ptr(const void* p, const char* what);
int check_weights(const Plan& p, const odevit_weights* w);
int prepare_weights(const Plan& p, const odevit_weights* w, WeightBufs& wb, cudaStream_t s);

// Butcher tableau of an explicit Runge-Kutta method: the fixed-grid methods (api.cu, up to 4 stages) and Dormand-Prince
// (solve_adaptive.cu, 6 stages)
struct Tableau {
  int S;
  float a[6][6];  // u_m = y + dt * sum_l a[m][l] * k_l   (m >= 1)
  float b[6];     // y_next = y + dt * sum_l b[l] * k_l
};
// Epilogue of stage `st` of a step starting at y with step dt (api.cu): produces the next stage input (or the step result
// when st == S-1) into `out`; stores k_st into k[st] when a later stage needs it.  k[l] is null where no buffer exists.
Epi rk_epilogue(const Tableau& tb, int st, float dt, const float* y, float* const* k, float* out);
// Its reverse (api.cu): the epilogue of stage m's mu GEMM (m >= 1) with t = m - 1,
//   lambda_t = g_t + h (a[m][t] mu_m + sum_{l>m} a[l][t] mu_l + b[t] G),
// keeping mu_m in mu[m]; the caller routes lambda_t (to dd).  h is the scalar dt, or with row_dt (non-null: dt unused)
// each image's step (EPI_ROWDT).  g_t (nullable, row_dt only) is the dense output's cotangent of stage t.
Epi rk_vjp_epilogue(const Tableau& tb, int m, float dt, const double* row_dt, int rows_per_image, const float* G,
                    float* const* mu, const float* g_t);
// The epilogue of stage 0's mu GEMM: out = G + mu_0 + mu_1 + ... + mu_{n_mu} + rows[0] + ... + rows[n_rows - 1].
Epi rk_vjp_row_epilogue(const float* G, float* const* mu, int n_mu, const float* const* rows, int n_rows, float* out);

// One forward field evaluation at `u` (api.cu); `rk` (nullable) is the epilogue of its last GEMM.
int eval_forward(const Plan& p, const WeightBufs& wb, const StageCtx& c, const float* u, float* P,
                 float* p_copy, float* sq, float* tmp, long long e, const Epi* rk, cudaStream_t s,
                 float* jas_out = nullptr, int jas_k = 0);

// softmax(q k^T) v per (image, head) from the packed qkv buffer into oh[:, h*d ...] (leading dim ld_oh).
// P: [B,H,N,N] fp32 scratch (unfused path); p_copy: optional export; lse: optional row log-sum-exp.
int attention_forward(const Plan& p, const void* qkv, void* oh, long long ld_oh, float* P, float* p_copy,
                      float* lse, float* sq, Drop drop, cudaStream_t s,
                      float* jas_out = nullptr, int jas_k = 0);
// Its VJP: dO [M,D] (act) -> dq|dk|dv into dz (leading dim R, act).  g_p: optional cotangent of P.
// dq_colsum / colsum_done: the fused kernel can add the column sums of dq (the q-row bias gradient) into dq_colsum [D]
// on its way out; *colsum_done says whether it did.
int attention_vjp(const Plan& p, const void* qkv, const void* oh, long long ld_oh, const float* lse, BwdBufs& b,
                  const float* g_p, void* dz, int R, Drop drop, cudaStream_t s, float* dq_colsum = nullptr,
                  bool* colsum_done = nullptr);

constexpr int kResidentMaxGrid = 129;   // grid points / output times the on-chip-state kernel carries in its arguments

// On-chip-state solver for small-token shapes (solve_resident.cu): one persistent CTA per image runs
// every step of the solve with the ODE state in shared memory.  Inference, PARALLEL field, bf16 mode.
bool solve_resident_shape_ok(const Plan& p);
bool solve_resident_supports(const Plan& p, int n_grid, bool wants_p_traj, bool has_tape);
size_t solve_resident_scratch_floats(const Plan& p);
int solve_resident(const Plan& p, const WeightBufs& wb, const Tableau& tb, const float* x0, const float* t_host,
                   int n_grid, float* states, float* final_state, float* p_last, float* kbuf, cudaStream_t s);
// Its adaptive mode (odevit_solve_adaptive_resident): per-image Dormand-Prince, one launch, no host round trip.
// envelope: null when the shape is covered, else what is out of range.  t_out [n_out] fp64 host, 2 <= n_out <= 129;
// next_image: one device int (the image dealer); status [B] device, never null.
const char* solve_resident_adaptive_envelope(const Plan& p);
size_t solve_resident_adaptive_scratch_floats(const Plan& p);
int solve_resident_adaptive(const Plan& p, const WeightBufs& wb, const float* x0, const double* t_out, int n_out,
                            double rtol, double atol, double first_step, int max_steps, float* states, int* nfe,
                            int* accepted, int* rejected, int* status, float* kbuf, int* next_image, cudaStream_t s);

// Reverse-sweep pieces shared by odevit_solve_bwd and odevit_solve_adaptive_bwd (api.cu):
//   layout_bwd: the fixed-grid workspace for S stages;  tape_bytes / check_tape / tape_ctx: the size of a tape of n_evals
//   evaluations, the check of a caller's tape against it, and the context of evaluation e in it;  eval_vjp: VJP of one
//   field evaluation, mu delivered through `mu_epi` (the EPI_RK epilogue of its last GEMM);  rk_step_vjp: the reverse
//   of one step;  finish_grads: the accumulators unfolded into the caller's gradients, once per call
BwdBufs layout_bwd(const Plan& p, Arena& a, int S);
size_t tape_bytes(const Plan& p, long long n_evals);
int check_tape(const Plan& p, const void* tape, size_t bytes, long long n_evals);
StageCtx tape_ctx(const Plan& p, const void* tape, long long e);
int eval_vjp(const Plan& p, const WeightBufs& wb, const StageCtx& c, BwdBufs& b, const float* g_p, bool need_c2,
             const odevit_weight_grads* gw, long long ev, const Epi& mu_epi, cudaStream_t s);
// The stage VJPs of one step, S-1 down to 0, G in b.gy: evaluation e0 + st with the intermediates ctx[st].  On entry dd
// holds scaler * lambda_{S-1}.  Stages S-1 .. 1 combine with rk_vjp_epilogue (dt / row_dt, g[t] of g (nullable)) and
// leave scaler * lambda_{st-1} in dd; stage 0 runs the caller's `row_epi` (rk_vjp_row_epilogue and any dd seed it
// adds).  g_p (nullable): the attention-map cotangent of stage S-1.
int rk_step_vjp(const Plan& p, BwdBufs& b, const Tableau& tb, float dt, const double* row_dt, const float* const* g,
                float* const* mu, const StageCtx* ctx, long long e0, const float* g_p, bool need_c2,
                const odevit_weight_grads* gw, Epi row_epi, cudaStream_t s);
int finish_grads(const Plan& p, const odevit_weights* w, const odevit_weight_grads* gw, const BwdBufs& b, cudaStream_t s);
bool wants_c2(const odevit_weight_grads* gw);

// Adaptive Dormand-Prince solve (solve_adaptive.cu): bytes of its workspace layouts (ODEVIT_WS_SOLVE_ADAPTIVE,
// ODEVIT_WS_SOLVE_ADAPTIVE_BWD)
size_t solve_adaptive_workspace_bytes(const Plan& p);
size_t solve_adaptive_bwd_workspace_bytes(const Plan& p);
size_t solve_adaptive_resident_workspace_bytes(const Plan& p);   // ODEVIT_WS_SOLVE_ADAPTIVE_RESIDENT

// MACARON field (field_macaron.cu)
int macaron_forward(const Plan& p, const WeightBufs& wb, const StageCtx& c, const float* u, float* P,
                    const Epi* rk, long long e, cudaStream_t s);
int macaron_vjp(const Plan& p, const WeightBufs& wb, const StageCtx& c, BwdBufs& b,
                const odevit_weight_grads* gw, const Epi& mu_epi, long long e, cudaStream_t s);

// Pre-LN encoder stack, forward only (field_macaron.cu): the distillation teacher
int encoder_forward(const Plan& p, const WeightBufs* layers, int n_layers, float ln_eps, const float* x0, float* hidden,
                    float* p_out, int p_mode, const StageCtx& c, float* P_scratch, cudaStream_t s);

}  // namespace odevit
