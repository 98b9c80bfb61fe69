// The MACARON vector field (models/macaron.py:106-123, :146-150):
//
//   x1 = x  + 1/2 rs * FFN(LN1 x)        FFN = fc2(GELU(fc1 .)), biases on, SHARED by both halves
//   x2 = x1 +     rs * MHA(LN2 x1)       nn.MultiheadAttention(bias=True), need_weights=False
//   x3 = x2 + 1/2 rs * FFN(LN3 x2)
//   f(t, x) = scaler * x3                (a state, not a derivative: SURVEY 2.3 quirk 14)
//
// `rs` = res_scale is a learnable [1] parameter: it stays on the device (Epi::dev_scale), the host
// never reads it.  Each residual update is the epilogue of its GEMM (EPI_RK with y = the running
// state); the last one also carries `scaler`, the x2 term (Epi::resid) and the caller's Runge-Kutta
// stage combine.  LayerNorm needs whole-row statistics, so it is a row kernel between the GEMMs.
//
// VJP: the cotangent g runs down the fp32 residual chain x3 -> x2 -> x1 -> x.  For every branch
// (coefficient c = 1/2, 1, 1/2) the GEMM operand is ddc = cast(c * g), WITHOUT rs: the weight-gradient
// accumulators G2 / c2 / c3 are therefore the rs = 1 sums, from which both dW = rs * G and
// d rs = <W, G> + <b, c> follow at the end (rows.cu::unfold_w2_macaron_kernel) -- no division by rs.
#include "host.h"

namespace odevit {

namespace {

constexpr float kLnEps = 1e-5f;  // nn.LayerNorm default (macaron.py:80-82)

inline void* off(void* p, size_t elems, int type) { return reinterpret_cast<char*>(p) + elems * dtype_size(type); }

// h = drop(GELU(n @ W1^T + b1))  (hpre kept for the VJP)
int ffn_up(const Plan& p, const WeightBufs& wb, const void* n, void* h, long long ld_h, void* hpre, Drop drop, cudaStream_t s) {
  const int D = p.D, hid = p.hid;
  GemmArgs g;
  g.M = p.M; g.N = hid; g.K = D;
  g.A = n; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
  g.B = off(wb.w1cat, (size_t)3 * D * D, p.act); g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
  g.epi_mode = EPI_FWD1;
  g.kclass = KC_GEMM_IN;
  g.epi.bias = wb.user->fc1_b;
  g.epi.split = 0;
  g.epi.out2 = h; g.epi.ld_out2 = ld_h;
  g.epi.out3 = hpre; g.epi.ld_out3 = hid;
  g.epi.aux_type = p.act;
  g.epi.drop = drop;   // macaron.py:88-94: Dropout(mlp_drop) after GELU
  return gemm(p, g, s);
}

// out-projection-like GEMM with the residual epilogue `e` (EPI_RK)
int proj_down(const Plan& p, const void* A, long long lda, int K, const void* W, long long ldw, const Epi& e,
              cudaStream_t s) {
  GemmArgs g;
  g.M = p.M; g.N = p.D; g.K = K;
  g.A = A; g.a_type = p.act; g.a_rs = lda; g.a_cs = 1;
  g.B = W; g.b_type = p.act; g.b_rs = ldw; g.b_cs = 1;
  g.epi_mode = EPI_RK;
  g.kclass = KC_GEMM_OUT;
  g.epi = e;
  g.epi.ld_out = p.D;
  return gemm(p, g, s);
}

}  // namespace

int macaron_forward(const Plan& p, const WeightBufs& wb, const StageCtx& c, const float* u, float* P,
                    const Epi* rk, long long ev, cudaStream_t s) {
  const int D = p.D, hid = p.hid, K2 = D + hid;
  const odevit_weights* w = wb.user;
  const size_t MD = (size_t)p.M * D;
  void* h1 = off(c.oh, D, p.act);  // [O | h1] rows of K2
  // the VJP of LN1 needs the stage input; it is an RK intermediate that does not outlive the step
  if (cudaMemcpyAsync(c.x0, u, MD * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
    return set_error(ODEVIT_ERR_CUDA, "macaron_forward: stage-input copy failed");
  // ---- first half-FFN ----
  ODV_TRY(ln_rows(u, w->norm_a_w, w->norm_a_b, c.xc, p.act, kLnEps, p.M, D, s));
  ODV_TRY(ffn_up(p, wb, c.xc, h1, K2, c.hpre, make_drop(p, DS_MLP_H, ev), s));
  {
    Epi e;
    e.bias = w->fc2_b; e.alpha = 1.f; e.dev_scale = w->res_scale;
    e.drop = make_drop(p, DS_MLP_OUT, ev);   // Dropout(mlp_drop) after ffn.3, before the residual
    e.c_new = 0.5f; e.y = u; e.y_coef = 1.f; e.out = c.x1;
    ODV_TRY(proj_down(p, h1, K2, hid, off(wb.w2cat, D, p.act), K2, e, s));
  }
  // ---- attention ----
  ODV_TRY(ln_rows(c.x1, w->norm_b_w, w->norm_b_b, c.n2, p.act, kLnEps, p.M, D, s));
  {
    GemmArgs g;
    g.M = p.M; g.N = 3 * D; g.K = D;
    g.A = c.n2; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
    g.B = wb.w1cat; g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
    g.epi_mode = EPI_STORE;
    g.kclass = KC_GEMM_IN;
    g.epi.bias = wb.b1cat;  // [q_scale*bq ; bk ; bv | fc1_b]: the first 3D entries
    g.epi.out = c.qkv; g.epi.out_type = p.act; g.epi.ld_out = 3 * D;
    ODV_TRY(gemm(p, g, s));
  }
  ODV_TRY(attention_forward(p, c.qkv, c.oh, K2, P, nullptr, c.lse, nullptr, make_drop(p, DS_ATTN, ev), s));
  {
    Epi e;
    e.bias = w->out_proj_b; e.alpha = 1.f; e.dev_scale = w->res_scale;
    e.drop = make_drop(p, DS_PROJ, ev);      // macaron.py:58-61: proj_drop after the out-projection
    e.c_new = 1.f; e.y = c.x1; e.y_coef = 1.f; e.out = c.x2;
    ODV_TRY(proj_down(p, c.oh, K2, D, wb.w2cat, K2, e, s));
  }
  // ---- second half-FFN ----
  ODV_TRY(ln_rows(c.x2, w->norm_c_w, w->norm_c_b, c.n3, p.act, kLnEps, p.M, D, s));
  ODV_TRY(ffn_up(p, wb, c.n3, c.h3, hid, c.hpre3, make_drop(p, DS_MLP_H2, ev), s));
  if (rk) {
    // k = scaler * (x2 + 1/2 rs drop(h3 W2^T + b2)), then the caller's stage combine on k
    Epi e = *rk;
    e.bias = w->fc2_b; e.alpha = 0.5f * p.scaler; e.dev_scale = w->res_scale;
    e.drop = make_drop(p, DS_MLP_OUT2, ev);
    e.resid = c.x2; e.resid_coef = p.scaler;
    ODV_TRY(proj_down(p, c.h3, hid, hid, off(wb.w2cat, D, p.act), K2, e, s));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Pre-LayerNorm transformer encoder stack, forward only: the frozen TEACHER of the distillation step
// (loss_trainer.py:318-321 calls a HF ViT with output_hidden_states / output_attentions; SURVEY
// section 8 row (f)3).  Per layer l, on the fp32 residual stream:
//     x' = x  + MHA(LN_a x)                 (q/k/v/out Linears with bias, softmax(q k^T / sqrt(d)) v)
//     x  = x' + fc2(GELU_erf(fc1(LN_b x')))
// built from the Macaron field's pieces: LayerNorm row kernel, one GEMM per projection with the bias /
// GELU / residual in its epilogue, the fused attention kernel.  hidden[l] receives every layer's output
// (it IS the residual stream: layer l+1 reads hidden[l]); p_out the attention maps of the layers asked for.
// ------------------------------------------------------------------------------------------------
int encoder_forward(const Plan& p, const WeightBufs* layers, int n_layers, float ln_eps, const float* x0, float* hidden,
                    float* p_out, int p_mode, const StageCtx& c, float* P_scratch, cudaStream_t s) {
  const int D = p.D, hid = p.hid, K2 = D + hid;
  const size_t MD = (size_t)p.M * D;
  void* h1 = off(c.oh, D, p.act);  // [O | h] rows of K2
  const float* x = x0;
  for (int l = 0; l < n_layers; ++l) {
    const WeightBufs& wb = layers[l];
    const odevit_weights* w = wb.user;
    float* x_out = hidden + (size_t)l * MD;
    float* p_copy = nullptr;
    if (p_out && (p_mode == 2 || (p_mode == 1 && l == n_layers - 1)))
      p_copy = p_out + (p_mode == 2 ? (size_t)l * (size_t)p.BHNN : 0);
    // ---- attention block ----
    ODV_TRY(ln_rows(x, w->norm_a_w, w->norm_a_b, c.xc, p.act, ln_eps, p.M, D, s));
    {
      GemmArgs g;
      g.M = p.M; g.N = 3 * D; g.K = D;
      g.A = c.xc; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
      g.B = wb.w1cat; g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
      g.epi_mode = EPI_STORE;
      g.kclass = KC_GEMM_IN;
      g.epi.bias = wb.b1cat;
      g.epi.out = c.qkv; g.epi.out_type = p.act; g.epi.ld_out = 3 * D;
      ODV_TRY(gemm(p, g, s));
    }
    ODV_TRY(attention_forward(p, c.qkv, c.oh, K2, P_scratch, p_copy, nullptr, nullptr, Drop{}, s));
    {
      Epi e;
      e.bias = w->out_proj_b; e.alpha = 1.f;
      e.c_new = 1.f; e.y = x; e.y_coef = 1.f; e.out = c.x1;
      ODV_TRY(proj_down(p, c.oh, K2, D, wb.w2cat, K2, e, s));
    }
    // ---- MLP block ----
    ODV_TRY(ln_rows(c.x1, w->norm_b_w, w->norm_b_b, c.xc, p.act, ln_eps, p.M, D, s));
    ODV_TRY(ffn_up(p, wb, c.xc, h1, K2, nullptr, Drop{}, s));
    {
      Epi e;
      e.bias = w->fc2_b; e.alpha = 1.f;
      e.c_new = 1.f; e.y = c.x1; e.y_coef = 1.f; e.out = x_out;
      ODV_TRY(proj_down(p, h1, K2, hid, off(wb.w2cat, D, p.act), K2, e, s));
    }
    x = x_out;
  }
  return 0;
}

namespace {

// One half-FFN branch of the VJP.  In: b.ddc = cast(1/2 g) [M,D] (act).  Out: b.dn = cotangent of
// the LayerNorm output feeding this branch (fp32 [M,D]); G1 / c1 (fc1 rows) and G2 / c3 accumulate.
int ffn_vjp(const Plan& p, const WeightBufs& wb, BwdBufs& b, const void* n, const void* h, long long ld_h,
            const void* hpre, Drop drop_h, Drop drop_out, cudaStream_t s) {
  const int D = p.D, hid = p.hid, R = 3 * D + hid, K2 = D + hid;
  void* dh = off(b.dz, 0, p.act);  // [M, hid] scratch inside dz ([M, R])
  // the branch output went through drop_out before the residual: its cotangent is ddc o mask
  if (drop_out.thresh) ODV_TRY(drop_rows_inplace(b.ddc, p.act, drop_out, p.M, D, s));
  {  // dh = rs * (ddc @ W2) o mask_h o GELU'(hpre)
    GemmArgs g;
    g.M = p.M; g.N = hid; g.K = D;
    g.A = b.ddc; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
    g.B = off(wb.w2catT, (size_t)D * D, p.act); g.b_type = p.act; g.b_rs = D; g.b_cs = 1;  // W2^T [hid, D]
    g.epi_mode = EPI_BWD3;
    g.kclass = KC_BWD_GEMM_DOH;
    g.epi.split = 0;
    g.epi.out2 = dh; g.epi.ld_out2 = hid;
    g.epi.aux = hpre; g.epi.ld_aux = hid; g.epi.aux_type = p.act;
    g.epi.dev_scale = wb.user->res_scale;
    g.epi.drop = drop_h;
    ODV_TRY(gemm(p, g, s));
  }
  {  // G2[:, D:] += ddc^T @ h      (the rs = 1 sum; h as the forward left it: after its dropout)
    GemmArgs g;
    g.M = D; g.N = hid; g.K = p.M;
    g.A = b.ddc; g.a_type = p.act; g.a_rs = 1; g.a_cs = D;
    g.B = h; g.b_type = p.act; g.b_rs = 1; g.b_cs = ld_h;
    g.epi_mode = EPI_ACCUM;
    g.epi.out = b.G2 + D; g.epi.ld_out = K2;
    g.kclass = KC_BWD_GEMM_G2;
    ODV_TRY(gemm(p, g, s));
  }
  ODV_TRY(colsum_accum(b.ddc, p.act, D, p.M, D, b.c3, s, p.det_ws));
  {  // dn = dh @ W1
    GemmArgs g;
    g.M = p.M; g.N = D; g.K = hid;
    g.A = dh; g.a_type = p.act; g.a_rs = hid; g.a_cs = 1;
    g.B = off(wb.w1catT, (size_t)3 * D, p.act); g.b_type = p.act; g.b_rs = R; g.b_cs = 1;  // W1^T view [D, hid], ld R
    g.epi_mode = EPI_STORE;
    g.kclass = KC_BWD_GEMM_DX;
    g.epi.out = b.dn; g.epi.out_type = DT_F32; g.epi.ld_out = D;
    ODV_TRY(gemm(p, g, s));
  }
  {  // G1[3D:, :] += dh^T @ n
    GemmArgs g;
    g.M = hid; g.N = D; g.K = p.M;
    g.A = dh; g.a_type = p.act; g.a_rs = 1; g.a_cs = hid;
    g.B = n; g.b_type = p.act; g.b_rs = 1; g.b_cs = D;
    g.epi_mode = EPI_ACCUM;
    g.epi.out = b.G1 + (size_t)3 * D * D; g.epi.ld_out = D;
    g.kclass = KC_BWD_GEMM_G1;
    ODV_TRY(gemm(p, g, s));
  }
  return colsum_accum(dh, p.act, hid, p.M, hid, b.c1 + 3 * D, s, p.det_ws);
}

}  // namespace

// In: b.dd = g3 = scaler * lambda (fp32 [M,D], cotangent of x3).  Out: mu = J(u)^T lambda through mu_epi.
int macaron_vjp(const Plan& p, const WeightBufs& wb, const StageCtx& c, BwdBufs& b, const odevit_weight_grads* gw,
                const Epi& mu_epi, long long ev, cudaStream_t s) {
  const int D = p.D, hid = p.hid, R = 3 * D + hid, K2 = D + hid;
  const odevit_weights* w = wb.user;
  float* g = reinterpret_cast<float*>(b.dd);
  const void* h1 = off(c.oh, D, p.act);
  {  // ddc = cast(1/2 g3)
    CombineArgs c0;
    c0.n_terms = 1; c0.term[0] = g; c0.coef[0] = 0.5f;
    c0.out_dd = b.ddc; c0.dd_type = p.act; c0.dd_scale = 1.f;
    ODV_TRY(vjp_combine(c0, p.M, D, s));
  }
  // ---- second half-FFN:  g2 = g3 + LN3'(x2)^T dn3 ----
  ODV_TRY(ffn_vjp(p, wb, b, c.n3, c.h3, hid, c.hpre3, make_drop(p, DS_MLP_H2, ev), make_drop(p, DS_MLP_OUT2, ev), s));
  {
    LnBwdArgs a;
    a.x = c.x2; a.dn = b.dn; a.w = w->norm_c_w; a.g_in = g; a.g_out = g;
    a.dd_out = b.ddc; a.dd_type = p.act; a.dd_coef = 1.f;  // attention branch coefficient
    a.dw = gw->norm_c_w; a.db = gw->norm_c_b; a.eps = kLnEps;
    a.part = p.det_ws;
    ODV_TRY(ln_bwd_rows(a, p.M, D, s));
  }
  // ---- attention:  g1 = g2 + LN2'(x1)^T dn2 ----
  {
    const Drop dp = make_drop(p, DS_PROJ, ev);   // the out-projection's output went through proj_drop
    if (dp.thresh) ODV_TRY(drop_rows_inplace(b.ddc, p.act, dp, p.M, D, s));
  }
  {  // dO = rs * (ddc @ Wo)
    GemmArgs gm;
    gm.M = p.M; gm.N = D; gm.K = D;
    gm.A = b.ddc; gm.a_type = p.act; gm.a_rs = D; gm.a_cs = 1;
    gm.B = wb.w2catT; gm.b_type = p.act; gm.b_rs = D; gm.b_cs = 1;  // Wo^T [D, D]
    gm.epi_mode = EPI_STORE;
    gm.kclass = KC_BWD_GEMM_DOH;
    gm.epi.out = b.dO; gm.epi.out_type = p.act; gm.epi.ld_out = D;
    gm.epi.dev_scale = w->res_scale;
    ODV_TRY(gemm(p, gm, s));
  }
  {  // G2[:, :D] += ddc^T @ O
    GemmArgs gm;
    gm.M = D; gm.N = D; gm.K = p.M;
    gm.A = b.ddc; gm.a_type = p.act; gm.a_rs = 1; gm.a_cs = D;
    gm.B = c.oh; gm.b_type = p.act; gm.b_rs = 1; gm.b_cs = K2;
    gm.epi_mode = EPI_ACCUM;
    gm.epi.out = b.G2; gm.epi.ld_out = K2;
    gm.kclass = KC_BWD_GEMM_G2;
    ODV_TRY(gemm(p, gm, s));
  }
  ODV_TRY(colsum_accum(b.ddc, p.act, D, p.M, D, b.c2, s, p.det_ws));
  ODV_TRY(attention_vjp(p, c.qkv, c.oh, K2, c.lse, b, nullptr, b.dz, R, make_drop(p, DS_ATTN, ev), s));  // dq|dk|dv -> dz[:, :3D] (ld R)
  {  // dn2 = dz[:, :3D] @ W_in (q rows scaled)
    GemmArgs gm;
    gm.M = p.M; gm.N = D; gm.K = 3 * D;
    gm.A = b.dz; gm.a_type = p.act; gm.a_rs = R; gm.a_cs = 1;
    gm.B = wb.w1catT; gm.b_type = p.act; gm.b_rs = R; gm.b_cs = 1;  // W_in^T view [D, 3D], ld R
    gm.epi_mode = EPI_STORE;
    gm.kclass = KC_BWD_GEMM_DX;
    gm.epi.out = b.dn; gm.epi.out_type = DT_F32; gm.epi.ld_out = D;
    ODV_TRY(gemm(p, gm, s));
  }
  {  // G1[:3D, :] += dz[:, :3D]^T @ n2
    GemmArgs gm;
    gm.M = 3 * D; gm.N = D; gm.K = p.M;
    gm.A = b.dz; gm.a_type = p.act; gm.a_rs = 1; gm.a_cs = R;
    gm.B = c.n2; gm.b_type = p.act; gm.b_rs = 1; gm.b_cs = D;
    gm.epi_mode = EPI_ACCUM;
    gm.epi.out = b.G1; gm.epi.ld_out = D;
    gm.kclass = KC_BWD_GEMM_G1;
    ODV_TRY(gemm(p, gm, s));
  }
  ODV_TRY(colsum_accum(b.dz, p.act, R, p.M, 3 * D, b.c1, s, p.det_ws));
  {
    LnBwdArgs a;
    a.x = c.x1; a.dn = b.dn; a.w = w->norm_b_w; a.g_in = g; a.g_out = g;
    a.dd_out = b.ddc; a.dd_type = p.act; a.dd_coef = 0.5f;  // first half-FFN coefficient
    a.dw = gw->norm_b_w; a.db = gw->norm_b_b; a.eps = kLnEps;
    a.part = p.det_ws;
    ODV_TRY(ln_bwd_rows(a, p.M, D, s));
  }
  // ---- first half-FFN:  g0 = g1 + LN1'(x0)^T dn1 ----
  ODV_TRY(ffn_vjp(p, wb, b, c.xc, h1, K2, c.hpre, make_drop(p, DS_MLP_H, ev), make_drop(p, DS_MLP_OUT, ev), s));
  {
    LnBwdArgs a;
    a.x = c.x0; a.dn = b.dn; a.w = w->norm_a_w; a.g_in = g; a.g_out = g;
    a.dw = gw->norm_a_w; a.db = gw->norm_a_b; a.eps = kLnEps;
    a.part = p.det_ws;
    ODV_TRY(ln_bwd_rows(a, p.M, D, s));
  }
  // mu = g0; the reverse-mode stage combine (may rewrite b.dd in place: element-wise, read before write)
  return rk_apply_rows(mu_epi, g, p.M, D, s);
}

}  // namespace odevit
