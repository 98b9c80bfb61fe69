// Internal declarations shared by the translation units of libodevit.so.
// Not part of the ABI (that is include/odevit.h).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "../../include/odevit.h"

namespace odevit {

// ---------------------------------------------------------------------------------------------
// error handling + launch accounting (thread-local: the ABI is thread-safe for distinct streams)
// ---------------------------------------------------------------------------------------------
int set_error(int code, const char* fmt, ...);
void count_launch(int n = 1);

#define ODV_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (call);                                                             \
    if (_e != cudaSuccess)                                                               \
      return ::odevit::set_error(ODEVIT_ERR_CUDA, "%s failed: %s (%s:%d)", #call,        \
                                 cudaGetErrorString(_e), __FILE__, __LINE__);            \
  } while (0)

#define ODV_TRY(call)          \
  do {                         \
    int _s = (call);           \
    if (_s != 0) return _s;    \
  } while (0)

#define ODV_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    cudaError_t _e = cudaGetLastError();                                                 \
    if (_e != cudaSuccess)                                                               \
      return ::odevit::set_error(ODEVIT_ERR_CUDA, "kernel launch failed: %s (%s:%d)",    \
                                 cudaGetErrorString(_e), __FILE__, __LINE__);            \
    ::odevit::count_launch();                                                            \
  } while (0)

// ---------------------------------------------------------------------------------------------
// per-kernel-class device timing (bench.py's roofline numbers): when enabled through
// odevit_profile_enable(), every launch site brackets its launch with a CUDA event pair on the
// launching stream; odevit_profile_read() sums the pairs per class.  Off by default (no events).
// ---------------------------------------------------------------------------------------------
enum KClass : int {
  KC_CENTER = 0,   // center_rows
  KC_GEMM_IN,      // xc @ W1cat^T (packed in-proj + fc1, GELU epilogue)
  KC_ATTN_S,       // q k^T per (image, head)
  KC_SOFTMAX,      // softmax rows (+ P export)
  KC_ATTN_PV,      // P v per (image, head)
  KC_GEMM_OUT,     // [O|h] @ [Wo|W2]^T + RK stage-combine epilogue
  KC_BWD_GEMM_DOH, // dd @ [Wo|W2]   (+ GELU' epilogue)
  KC_BWD_GEMM_G2,  // G2 += dd^T [O|h]
  KC_BWD_ATTN,     // attention VJP products (dP, dq, dk, dv)
  KC_BWD_SOFTMAX,  // softmax VJP rows
  KC_BWD_GEMM_DX,  // mu = dz @ centred(W1cat) (+ RK stage-combine epilogue)
  KC_BWD_GEMM_G1,  // G1 += dz^T xc
  KC_BWD_COLSUM,   // bias-gradient column sums
  KC_COMBINE,      // reverse-mode stage combine / axpy
  KC_WEIGHTS,      // weight fold / gradient unfold
  KC_FUSED_ATTN,   // fused attention (S, softmax, PV in one kernel)
  KC_FUSED_ATTN_BWD,  // fused attention VJP (delta + dq/dk/dv in one kernel)
  KC_FD_BOUND,        // finite-difference curvature of the trajectory (single pass)
  KC_FUSED_ATTN_EXPORT,  // fused attention forward that also writes the fp32 attention map
  KC_RESIDENT,        // on-chip-state solver: the whole solve of an image in one persistent CTA
  KC_OTHER,
  KC_COUNT
};
struct ProfScope {
  int cls;
  cudaStream_t s;
  int slot;
  ProfScope(int cls, cudaStream_t s);
  ~ProfScope();
};

// ---------------------------------------------------------------------------------------------
// element types of activation buffers
// ---------------------------------------------------------------------------------------------
enum DType : int { DT_F32 = 0, DT_BF16 = 1 };
static inline size_t dtype_size(int t) { return t == DT_F32 ? 4 : 2; }

// ---------------------------------------------------------------------------------------------
// GEMM:  C[m,n] = sum_k A(m,k) * B(n,k)   (both operands addressed by element strides)
// ---------------------------------------------------------------------------------------------
enum EpiMode : int {
  EPI_STORE = 0,  // out[m,n] = alpha*acc + bias[n]
  EPI_FWD1 = 1,   // n <  split: out[m,n] = acc + bias[n]          (q|k|v)
                  // n >= split: out3[m,n-split] = v (opt), out2[m,n-split] = gelu(v)   (fc1)
  EPI_RK = 2,     // v = alpha*(acc + bias[n]); kstore (opt) = v;
                  // r = y_coef*y[m,n] + c_new*v + sum_i c_k[i]*kin[i][m,n]
                  // out (opt, fp32) = r;  out2 (opt, aux_type) = out2_scale * r
  EPI_BWD3 = 3,   // n <  split: out[m,n] = acc                    (dO)
                  // n >= split: out2[m,n-split] = acc * gelu'(aux[m,n-split])   (d h_pre)
  EPI_ACCUM = 4,  // out[m,n] += alpha*acc   (fp32; atomic when split-K)
  EPI_TOKENS = 5, // patch projection straight into the token tensor (ode_transformer_gpt.py:148-182): with P = split
                  // rows per image, out[(m / P) * out_bo + (m % P + out_bi) * ld_out + n] = acc + y[(m % P) * ld_out + n]
                  // (y = bias + positional rows of the patch tokens, [P, D] fp32)
  // template-only flag: the epilogue applies Epi::drop (kernels without it carry no mask code at all)
  EPI_DROP = 8,
  // template-only flag (EPI_RK): the epilogue also folds the second finite difference of the trajectory into
  // Epi::fd_out (trajectory-free inference: ode_transformer_gpt.py:529-543 without the [T,B,N,D] tensor)
  EPI_FD = 16,
  // template-only flag (EPI_FWD1 / EPI_BWD3): erf-form GELU instead of the fitted logistic form (the fp32 mode)
  EPI_EXACT = 32,
  // template-only flag (EPI_RK): per-image step size, r = y_coef*y + dt_b*(c_new*v + sum_i c_k[i]*kin[i]) with
  // dt_b = (float)Epi::row_dt[m / rows_per_image] (the adaptive solve: the host passes the tableau without dt)
  EPI_ROWDT = 64
};

// One dropout site of one field evaluation: element (r, c) is kept iff hash(key, r, c) >= thresh and then
// multiplied by scale = 1/(1-p).  thresh == 0: no dropout.
// key_ptr != null: the key is read from device memory (a table the library fills from a device-resident seed at the
// start of the call, rows.cu::resolve_drop_keys) instead of being formed on the host.
struct Drop {
  uint32_t key = 0;
  uint32_t thresh = 0;
  float scale = 1.f;
  const uint32_t* key_ptr = nullptr;
};
// sites of one field evaluation (MACARON: the second half-FFN has its own two)
enum DropSite : int { DS_ATTN = 0, DS_PROJ = 1, DS_MLP_H = 2, DS_MLP_OUT = 3, DS_MLP_H2 = 4, DS_MLP_OUT2 = 5, DS_SITES = 8 };
constexpr int kDropKeyEvals = 1024;   // evaluations a device-seeded call can address (key table: 32 KB of workspace)

struct Epi {
  float alpha = 1.f;
  const float* bias = nullptr;
  void* out = nullptr;
  int out_type = DT_F32;
  long long ld_out = 0, out_bo = 0, out_bi = 0;
  int split = 0;
  void* out2 = nullptr;
  long long ld_out2 = 0;
  void* out3 = nullptr;
  long long ld_out3 = 0;
  int aux_type = DT_F32;  // type of out2/out3/aux buffers
  const float* y = nullptr;
  static constexpr int kMaxTerms = 6;
  const float* kin[kMaxTerms] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  float y_coef = 1.f, c_new = 0.f, c_k[kMaxTerms] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float out2_scale = 1.f;
  float* k_store = nullptr;
  const void* aux = nullptr;
  long long ld_aux = 0;
  // device-resident scalar factor on the accumulator (macaron.py:104 `res_scale`, a learnable [1]
  // parameter the host must not read back): EPI_STORE / EPI_RK / EPI_BWD3 multiply by *dev_scale
  const float* dev_scale = nullptr;
  // EPI_RK: v += resid_coef * resid[m,n] before k_store / the stage combine (the Macaron field
  // returns scaler * (x2 + half-FFN), macaron.py:118-123, :148)
  const float* resid = nullptr;
  float resid_coef = 0.f;
  // dropout on the epilogue's value: EPI_FWD1 after GELU, EPI_RK on v (before resid), EPI_BWD3 on d h
  Drop drop;
  // EPI_RK, when r is the NEXT trajectory row and y the current one: fd_out[m] = max(fd_out[m], max_n |r - 2 y + fd_prev|)
  // with fd_prev the row before y ([M] fp32 maxima, atomicMax on the bit pattern of non-negative floats)
  const float* fd_prev = nullptr;
  float* fd_out = nullptr;
  // the tcgen05 epilogues use GELU's erf form (set by the fp32 mode's split-bf16 GEMMs; the bf16 mode's fitted form is
  // 2.6e-5 off, inside bf16 rounding but not inside the fp32 mode's 1e-4)
  bool exact_gelu = false;
  // EPI_FWD1 stores GELU'(pre-activation) instead of the pre-activation in out3, and EPI_BWD3 finds it in aux: the
  // VJP's epilogue multiplies by it instead of evaluating the derivative again (~14 instructions and two MUFU
  // operations per element less in an epilogue that was as long as its K = D main loop).  Both GEMMs of a field
  // evaluation must agree on it.
  bool aux_gelu_grad = false;
  // EPI_BWD3 (tcgen05 kernel): column sums of the stored values over the rows m, added atomically to colsum_a[n] for the
  // columns n < split and to colsum_b[n - split] for the rest (bias gradients without a second pass over the outputs;
  // needs N % 32 == 0 and split % 32 == 0: whole warps reduce)
  float* colsum_a = nullptr;
  float* colsum_b = nullptr;
  // EPI_RK with EPI_ROWDT: per-image step sizes [B] (fp64, cast to fp32 as torchdiffeq casts dt to the state's type);
  // row m belongs to image m / rows_per_image.  Needs y.
  const double* row_dt = nullptr;
  int rows_per_image = 1;
};

struct GemmArgs {
  int M = 0, N = 0, K = 0;
  const void* A = nullptr;
  int a_type = DT_F32;
  long long a_rs = 0, a_cs = 1, a_bo = 0, a_bi = 0;
  const void* B = nullptr;
  int b_type = DT_F32;
  long long b_rs = 0, b_cs = 1, b_bo = 0, b_bi = 0;
  int batch_outer = 1, batch_inner = 1;
  int epi_mode = EPI_STORE;
  Epi epi;
  int kclass = KC_OTHER;
};

// CUDA-core (FFMA) GEMM: any strides, any M/N/K, fp32 or bf16 operands, fp32 accumulate.
int gemm_simt(const GemmArgs& g, cudaStream_t s);

// tcgen05 / TMA GEMM (bf16 operands, fp32 accumulate in TMEM).  Returns ODEVIT_ERR_UNSUPPORTED
// for shapes/layouts it does not cover (caller then reports the error; there is no silent
// fallback in the bf16 product path except for the batched per-head attention products).
int gemm_tc(const GemmArgs& g, cudaStream_t s);
bool gemm_tc_supports(const GemmArgs& g);

// Fused tcgen05 attention forward (attn_tc.cu): qkv [B,N,3D] bf16 -> O into oh[:, h*64..] (bf16),
// optional fp32 P export.  Covers head dim 64, N <= 256.
bool attn_fwd_tc_supports(int N, int D, int H, int act_type, long long ld_oh);
int attn_fwd_tc(const void* qkv, void* oh, long long ld_oh, float* p_out, float* lse_out, int B, int N, int H, int D,
                Drop drop, cudaStream_t s, float* jas_out = nullptr, int jas_k = 0);
bool attn_fwd_tc_jasmin_supports(int N, int k);
// Fused attention VJP; needs the forward's lse2 [B,H,N]; writes delta [B,H,N] and dq|dk|dv into dz.
size_t attn_bwd_tc_scratch_floats(int B, int N, int H);
int attn_bwd_tc(const void* qkv, const void* dO, const void* oh, long long ld_oh, const float* lse2, float* delta,
                void* dz, int R, float* dq_scratch, int B, int N, int H, int D, Drop drop, cudaStream_t s, const float* gp = nullptr,
                const float* dext = nullptr, float* dq_colsum = nullptr);   // dq_colsum [D] += column sums of dq

// ---------------------------------------------------------------------------------------------
// row-wise / elementwise kernels (odevit_rows.cu)
// ---------------------------------------------------------------------------------------------
// xc[r,:] = x[r,:] - mean(x[r,:]);  if rstd_out: also divide by sqrt(var+eps) (LayerNorm core)
int center_rows(const float* x, void* xc, int xc_type, float* rstd_out, float eps, int rows,
                int D, cudaStream_t s);
// in-place softmax over rows of length n (fp32); optional second copy
int softmax_rows(float* p, float* copy_to, long long rows, int n, cudaStream_t s);
// ds = p * (dp + dpx - sum_j p*(dp+dpx)), written over dp.  dpx nullable.
int softmax_bwd_rows(const float* p, float* dp, const float* dpx, long long rows, int n,
                     cudaStream_t s);
// acc[j] += sum_r X[r, j]
int colsum_accum(const void* X, int x_type, long long ld, int rows, int cols, float* acc,
                 cudaStream_t s);

// Reverse-mode stage combine (the seed and overflow passes of the reverse sweeps, the MACARON VJP):
// v = sum_i coef[i]*term[i] ; writes out_f32 = v and/or out_dd = cast(dd_scale*v)
struct CombineArgs {
  int n_terms = 0;
  const float* term[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  float coef[6] = {0, 0, 0, 0, 0, 0};
  float* out_f32 = nullptr;
  void* out_dd = nullptr;
  int dd_type = DT_F32;
  float dd_scale = 1.f;
};
int vjp_combine(const CombineArgs& a, int rows, int D, cudaStream_t s);

// per_seq[r] = max_j max_d |s[j+2,r,d] - 2 s[j+1,r,d] + s[j,r,d]| / dt2   (states [T, rows, D])
int fd_curvature(const float* states, int T, long long rows, int D, float dt2, float* per_seq, cudaStream_t s);
// per [N x N] attention-map slice: max over rows of the JaSMin row value (rows.cu)
// out[row] = sum_j P[row, j] * G[row, j]   (rows.cu)
int rowdot_rows(const float* P, const float* G, float* out, long long rows, int n, cudaStream_t s);
int jasmin_rowmax(const float* P, long long n_slices, int N, int k, float* out, cudaStream_t s);

// out1 = x o mask(d1), out2 = x o mask(d2)  (x, out*: [rows, D] of type `type`; the two masked copies of
// the cotangent that enter the fc2 and the out-proj branch when their output dropouts differ)
int drop_pair_rows(const void* x, void* out1, void* out2, int type, Drop d1, Drop d2, int rows, int D, cudaStream_t s);
// p[r, c] = keep(r, c) ? p[r, c] * scale : 0   (fp32 [rows, n]; the attention map of the CUDA-core path)
int drop_inplace_f32(float* p, float* copy_to, Drop d, long long rows, int n, cudaStream_t s);
// x <- x o mask(d) in place on an [rows, D] activation-typed buffer
int drop_rows_inplace(void* x, int type, Drop d, int rows, int D, cudaStream_t s);
// table[i] = key of (evaluation i / DS_SITES, site i % DS_SITES) from the 64-bit seed at seed_dev
int resolve_drop_keys(const uint32_t* seed_dev, uint32_t* table, int n, cudaStream_t s);
int drop_state_advance(unsigned long long* state, cudaStream_t s);

// tokens.cu: token assembly around the patch GEMM, head + cross-entropy
int tokens_special_rows(const float* rows, const int* index, int n_special, int B, int N, int D, float* x0, cudaStream_t s);
int head_ce_fwd(const float* x, long long x_stride, const float* W, const float* bias, const long long* labels, int B, int C, int D,
                float eps, float* logits, float* loss, float* lse, cudaStream_t s);
int head_ce_bwd(const float* x, long long x_stride, const float* W, const long long* labels, const float* logits, const float* lse,
                const float* g_logits, const float* g_loss, int B, int C, int D, float eps, float* dz, float* g_x,
                long long gx_stride, float* g_W, float* g_bias, cudaStream_t s);

// mass.cu: the L1-attention front-end (loss_trainer.py:80-117), forward and exact VJP
int extract_mass_fwd(const float* a, int B, int H, int n, float threshold, int smooth, float scale, float* out_mean,
                     float* out_heads, float* out_mask, cudaStream_t s);
int extract_mass_bwd(const float* a, int B, int H, int n, float threshold, int smooth, float scale, const float* g_mean,
                     const float* g_heads, float* g_a, cudaStream_t s);

// preprocess.cu: PIL-exact bilinear resize of uint8 HWC images + rescale + normalise -> fp32 NCHW
int preprocess_u8(const uint8_t* images, int B, int H, int W, int So_h, int So_w, const int32_t* bounds_h,
                  const int32_t* kk_h, int ksize_h, const int32_t* bounds_v, const int32_t* kk_v, int ksize_v,
                  float rescale, const float* mean, const float* stdv, uint8_t* tmp, float* out, uint8_t* out_u8,
                  cudaStream_t s);
int pil_bilinear_ksize(int in_size, int out_size);
void pil_bilinear_tables(int in_size, int out_size, int32_t* bounds, int32_t* kk);

// dst (bf16) = bf16 pieces of the fp32 matrix src [rows, cols] (row stride ld): x = hi + mid + lo with hi = bf16(x),
// mid = bf16(x - hi), lo = bf16(x - hi - mid); segment i of the output holds piece[i] (0 hi, 1 mid, 2 lo), the segments
// concatenated along the columns (concat_rows = 0: dst [rows, nseg cols]) or along the rows (dst [nseg rows, cols])
int split_bf16(const float* src, long long ld, int rows, int cols, int concat_rows, int nseg, const int* piece, void* dst,
               cudaStream_t s);

// start of the reverse sweep in one pass: gy = sum of the injected cotangents, dd = cast(dd_coef * gy)
int seed_sweep(const float* const* terms, int n_terms, float* gy, void* dd, int dd_type, float dd_coef, long long n, cudaStream_t s);

// y[i] += a * x[i]
int axpy_f32(float* y, const float* x, float a, long long n, cudaStream_t s);

// Weight preparation / gradient assembly for the PARALLEL variant (folded CenterNorm affine).
struct FoldArgs {
  int D, hid, heads;
  float q_scale;   // factor on the Wq rows / bq: 1/sqrt(d) for nn.MultiheadAttention, 1 for L2SelfAttention
  bool fold_norm;  // fold the CenterNorm affines (PARALLEL*) or copy the weights as they are (MACARON)
  const odevit_weights* w;
  void* w1cat; int w_type;   // [3D+hid, D]
  void* w1catT;              // [D, 3D+hid] or null; each W1cat row is CENTRED over D here (so that
                             // dz @ W1cat directly yields the centring VJP mu = zsum - mean_D zsum)
  float* b1cat;              // [3D+hid]
  float* fmean;              // [3D+hid] scratch: row means of W1cat (fold_w1_kernel -> fold_w1_transpose_kernel)
  void* w2cat;               // [D, D+hid]
  void* w2catT;              // [D+hid, D] or null
  float* b2;                 // [D] (out_proj_b + fc2_b) -- zero if absent
};
int fold_weights_parallel(const FoldArgs& a, cudaStream_t s);

struct UnfoldArgs {
  int D, hid, heads;
  float q_scale;
  const float* c3 = nullptr;  // MACARON: colsum of the fc2 cotangent (c2 is the out-proj one)
  const odevit_weights* w;
  const odevit_weight_grads* gw;
  const float* G1;  // [3D+hid, D]   = sum dz^T xc
  const float* c1;  // [3D+hid]      = colsum dz
  const float* G2;  // [D, D+hid]    = sum dd^T [O|h]
  const float* c2;  // [D]           = colsum dd
};
int unfold_grads_parallel(const UnfoldArgs& a, cudaStream_t s);
// MACARON (no folded norms; G2/c2/c3 were accumulated WITHOUT res_scale, macaron.py:104):
//   dW_in += q_scale_row*G1[:3D], dW_fc1 += G1[3D:], dWo += rs*G2[:, :D], dW_fc2 += rs*G2[:, D:],
//   d res_scale += <Wo, G2[:, :D]> + <bo, c2> + <W2, G2[:, D:]> + <b2, c3>
int unfold_grads_macaron(const UnfoldArgs& a, cudaStream_t s);

// LayerNorm rows (nn.LayerNorm, eps inside the sqrt; macaron.py:80-82): out = (x-mean)*rstd*w + b
int ln_rows(const float* x, const float* w, const float* b, void* out, int out_type, float eps, int rows, int D,
            cudaStream_t s);
// Its VJP fused with the residual add:  g_out = g_in + dLN(x)^T dn ;  dw += sum dn*xhat ; db += sum dn ;
// optional dd_out = cast(dd_coef * g_out) (the next GEMM's operand).  g_out may alias g_in.
struct LnBwdArgs {
  const float* x = nullptr;
  const float* dn = nullptr;
  const float* w = nullptr;
  const float* g_in = nullptr;
  float* g_out = nullptr;
  void* dd_out = nullptr;
  int dd_type = DT_F32;
  float dd_coef = 1.f;
  float* dw = nullptr;
  float* db = nullptr;
  float eps = 1e-5f;
};
int ln_bwd_rows(const LnBwdArgs& a, int rows, int D, cudaStream_t s);
// EPI_RK applied to a plain [rows, D] fp32 array v (alpha/bias ignored): the stage combine when the
// producer of v is not a GEMM.
int rk_apply_rows(const Epi& e, const float* v, int rows, int D, cudaStream_t s);

// L2SelfAttention pieces (ode_transformer_gpt.py:34-63)
// sq[0][b,h,i] = |q_i|^2, sq[1][b,h,j] = |k_j|^2 from the packed qkv rows
int head_sqnorm(const void* qkv, int type, float* sq, int B, int N, int H, int D, cudaStream_t s);
// S[b,h,i,j] = q_i.k_j in place -> P = exp(-(|q_i|^2+|k_j|^2-2S)*scale) / (rowsum + 1e-8)
int l2_prob_rows(float* S, const float* sq, float scale, float* copy_to, int B, int H, int N, cudaStream_t s);
// dq_i -= coef * rowsum_i(ds) * q_i ;  dk_j -= coef * colsum_j(ds) * k_j   (the |q|^2, |k|^2 terms)
int l2_vjp_fix(const float* ds, const void* qkv, int type, void* dz, int R, float coef, int B, int N, int H, int D,
               cudaStream_t s);

}  // namespace odevit
