/*
 * odevit.h -- C ABI of libodevit.so: the B200-native (sm_100a) implementation of ODE-ViT's hot
 * path, the vector field f(t, x) evaluated by a fixed-step solver over the integration grid.
 *
 * The reference (Bycarkos/ODE-ViT) is pure Python: it has no FFI layer, its "plugin" surface is
 * the nn.Module API.  This header declares what a binding for the hot path binds; each entry
 * point names the reference interface it replaces (paths relative to the reference root):
 *
 *   odevit_field_fwd   <-  ViT_ODEFunc.forward(t, x)            models/ode_transformer_gpt.py:317-330
 *                          (= ParallelAttentionMLP.forward :274-277, CenterNorm :79-83,
 *                             MultiheadSelfAttention :226-232, MLP :193-200, L2SelfAttention :34-63)
 *                          and macaron ViT_ODEFunc.forward       models/macaron.py:106-123, :146-150
 *   odevit_solve_fwd   <-  odeint(odefunc, tokens, t_grid, method=solver)
 *                                                                models/ode_transformer_gpt.py:571-578
 *                                                                models/macaron.py:323, :326
 *                          (third-party torchdiffeq fixed-grid euler / midpoint / rk4 = 3/8 rule)
 *   odevit_solve_bwd   <-  loss.backward() through that call     train.py:57-67, loss_trainer.py:365
 *                          (reference gradient mode: autograd through the unrolled solver; here a
 *                           reverse sweep that recomputes each step from the stored trajectory row)
 *   odevit_solve_adaptive[_record] / odevit_solve_adaptive_bwd
 *                      <-  odeint(..., method="dopri5") with the error norm taken per image, and loss.backward()
 *                          through it with the accepted steps frozen (not part of the reference)
 *
 * Conventions (SURVEY.md section 8b):
 *   - plain pointers and sizes only; no torch types; every device buffer, including the workspace,
 *     is owned by the caller; the library never allocates device memory and never synchronises
 *     (except odevit_solve_adaptive[_record], which cannot know its number of rounds in advance);
 *   - all work is enqueued on `stream` and is asynchronous with respect to the host;
 *   - `t_grid` is a HOST pointer (the per-step dt = t[i+1]-t[i] is formed on the host in fp32,
 *     exactly as torchdiffeq forms it);
 *   - weights are read at call time (modules may be re-assigned between calls);
 *   - returns 0 on success, a negative odevit_status otherwise; never throws across the ABI;
 *     odevit_last_error_string() describes the last failure on the calling thread;
 *   - there is NO CPU fallback: a host pointer where a device pointer is expected is an error.
 *
 * Tensor layouts: tokens are row-major [B, N, D] fp32 (rows = B*N); attention maps [B, H, N, N]
 * fp32; trajectories [T, B, N, D] fp32.  Weights use the reference's state_dict layouts
 * (nn.Linear: [out, in]; packed in_proj_weight [3D, D] with rows [Wq; Wk; Wv]).
 */
#ifndef ODEVIT_H_
#define ODEVIT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ODEVIT_ABI_VERSION 8

typedef struct CUstream_st* odevit_stream_t; /* == cudaStream_t */

typedef enum {
  ODEVIT_OK = 0,
  ODEVIT_ERR_INVALID_ARG = -1,   /* bad shape / null pointer / unsupported combination        */
  ODEVIT_ERR_WORKSPACE = -2,     /* workspace too small or misaligned                          */
  ODEVIT_ERR_CUDA = -3,          /* a CUDA runtime / driver call failed (sticky errors too)    */
  ODEVIT_ERR_UNSUPPORTED = -4,   /* shape outside what the kernels cover                       */
  ODEVIT_ERR_NOT_DEVICE_PTR = -5, /* a host pointer was passed where device memory is required */
  ODEVIT_ERR_NOT_CONVERGED = -6   /* adaptive solve: max_num_steps, a non-finite error ratio or dt
                                     underflow (the message names the image)                     */
} odevit_status;

typedef enum {
  ODEVIT_FIELD_PARALLEL = 0, /* MLP(CN x) + MHA(CN x)          ode_transformer_gpt.py:274-277 */
  ODEVIT_FIELD_PARALLEL_L2 = 1, /* same with L2SelfAttention   ode_transformer_gpt.py:34-63   */
  ODEVIT_FIELD_MACARON = 2   /* half-FFN, MHA, half-FFN        macaron.py:106-123             */
} odevit_variant;

typedef enum {
  ODEVIT_FP32 = 0, /* fp32 storage and FFMA arithmetic: <= 1e-4 of the reference              */
  ODEVIT_BF16 = 1  /* bf16 operands on tcgen05 tensor cores, fp32 accumulate/state: <= 2e-2   */
} odevit_precision;

typedef enum {
  ODEVIT_EULER = 0,
  ODEVIT_MIDPOINT = 1,
  ODEVIT_RK4_38 = 2 /* torchdiffeq method="rk4" (rk4_alt_step_func, Kutta 3/8 rule)           */
} odevit_method;

/* Problem descriptor. */
typedef struct {
  int32_t abi_version; /* ODEVIT_ABI_VERSION */
  int32_t batch;       /* B: images in this call                                              */
  int32_t tokens;      /* N: tokens per image (cls + patches + registers [+ dist])            */
  int32_t dim;         /* D: embed_dim                                                        */
  int32_t heads;       /* H: num_heads (head dim d = D/H, d <= 128, d % 8 == 0)               */
  int32_t hidden;      /* int(D * mlp_ratio)                                                  */
  int32_t variant;     /* odevit_variant                                                      */
  int32_t precision;   /* odevit_precision                                                    */
  float scaler;        /* ViT_ODEFunc.scaler (emulate_depth if time_interval == 1 else 1)     */
  /* Training-mode dropout (0 = off): on the attention map (the returned P is post-dropout), after out_proj, and
   * after GELU + after fc2 (ode_transformer_gpt.py:56, :61, :196-199, :217-231; MACARON: after GELU and after
   * ffn.3 of BOTH half steps with separate masks, on the attention map, after out_proj -- macaron.py:58-61, :88-94).
   * Masks are re-drawn at every field evaluation from a counter-based generator keyed by (seed, evaluation
   * index, site, element): the reverse sweep regenerates them, nothing is stored.  Not bit-compatible with
   * PyTorch's Philox stream (SURVEY 2.3 quirk 16).
   * The 64-bit seed is either given here (drop_seed_lo/hi) or READ FROM DEVICE MEMORY at kernel time
   * (drop_seed_dev != NULL: two uint32, lo then hi): a step captured in a CUDA graph then draws new masks at every
   * replay when something on the device advances the seed (odevit_drop_state_advance).  The forward and the
   * backward call of one step must see the same value. */
  float attn_drop;
  float proj_drop;
  float mlp_drop;
  uint32_t drop_seed_lo;
  uint32_t drop_seed_hi;
  const uint32_t* drop_seed_dev; /* device pointer or NULL */
} odevit_desc;

/* Weights of the vector field, fp32 device pointers in state_dict layout; unused = NULL.
 *   PARALLEL:    norm_a = block.norm_attn, norm_b = block.norm_mlp (CenterNorm, no eps);
 *                in_proj_w [3D,D], out_proj_w [D,D], fc1_w [hid,D], fc2_w [D,hid]; no biases.
 *   PARALLEL_L2: in_proj_w/in_proj_b hold [q_proj;k_proj;v_proj] stacked ([3D,D] / [3D]);
 *                out_proj_w/out_proj_b = out_proj.
 *   MACARON:     norm_a = norm1, norm_b = norm2, norm_c = norm3 (LayerNorm, eps 1e-5);
 *                fc1 = ffn.0, fc2 = ffn.3 (shared by both half steps), all biases present;
 *                res_scale [1].
 * mod_*: optional per-call modulation vectors [D] from models/time_emb.py::ScaleShift applied to
 * the normalised activations as n*(1+scale)+shift (NULL = off, the reference's behaviour). */
typedef struct {
  const float* norm_a_w; const float* norm_a_b;
  const float* norm_b_w; const float* norm_b_b;
  const float* norm_c_w; const float* norm_c_b;
  const float* in_proj_w; const float* in_proj_b;
  const float* out_proj_w; const float* out_proj_b;
  const float* fc1_w; const float* fc1_b;
  const float* fc2_w; const float* fc2_b;
  const float* res_scale;
  const float* mod_attn_scale; const float* mod_attn_shift;
  const float* mod_mlp_scale; const float* mod_mlp_shift;
  const void* reserved[5];
} odevit_weights;

/* Gradient accumulators, same layouts; the library ADDS into them (caller zero-fills). */
typedef struct {
  float* norm_a_w; float* norm_a_b;
  float* norm_b_w; float* norm_b_b;
  float* norm_c_w; float* norm_c_b;
  float* in_proj_w; float* in_proj_b;
  float* out_proj_w; float* out_proj_b;
  float* fc1_w; float* fc1_b;
  float* fc2_w; float* fc2_b;
  float* res_scale;
  void* reserved[9];
} odevit_weight_grads;

/* What a workspace is sized for. */
typedef enum {
  ODEVIT_WS_FIELD = 0,     /* odevit_field_fwd                                                 */
  ODEVIT_WS_SOLVE_FWD = 1, /* odevit_solve_fwd                                                 */
  ODEVIT_WS_SOLVE_BWD = 2, /* odevit_solve_bwd                                                 */
  ODEVIT_WS_ENCODER_FWD = 3, /* odevit_encoder_fwd (method ignored)                            */
  ODEVIT_WS_SOLVE_ADAPTIVE = 4, /* odevit_solve_adaptive[_record] (method ignored)              */
  ODEVIT_WS_SOLVE_ADAPTIVE_BWD = 5 /* odevit_solve_adaptive_bwd (method ignored)                */
} odevit_ws_kind;

/* ABI / build identification. */
int odevit_abi_version(void);
const char* odevit_build_info(void);             /* "sm_100a, nvcc x.y, <date>"                */
const char* odevit_last_error_string(void);      /* thread-local, never NULL                    */

/* Bytes of device workspace needed (0 on invalid desc; then see odevit_last_error_string). The
 * workspace must be 1024-byte aligned. `method` matters for the solve kinds (stage buffers). */
size_t odevit_workspace_bytes(const odevit_desc* desc, int32_t ws_kind, int32_t method);

/* One evaluation of the vector field: dx = f(t, x).  Replaces ViT_ODEFunc.forward(t, x).
 *   x   [B,N,D] in, dx [B,N,D] out (may not alias);
 *   p_out [B,H,N,N] or NULL: the attention map P of this evaluation (block.attentions). */
int odevit_field_fwd(const odevit_desc* desc, const odevit_weights* w,
                     const float* x, float* dx, float* p_out,
                     void* workspace, size_t workspace_bytes, odevit_stream_t stream);

/* The fixed-grid solve.  Replaces odeint(odefunc, x0, t_grid, method=...).
 *   t_grid_host [T] fp32, strictly monotonic, HOST memory;
 *   states [T,B,N,D] or NULL.  If given, row 0 := x0 and row j := state after step j (what odeint
 *          returns).  If NULL only final_state is produced (inference without trajectory);
 *   final_state [B,N,D] or NULL (required when states == NULL);
 *   p_last [B,H,N,N] or NULL: P of the LAST field evaluation (block.attentions after the solve);
 *   p_traj [(n_evals - p_traj_first_eval), B,H,N,N] or NULL: P of every evaluation e >=
 *          p_traj_first_eval, e = step*stages + stage (odefunc.attention_trajectory);
 *   jas_traj [(n_evals - jas_first_eval), B,H] or NULL: the JaSMin statistic (see odevit_jasmin_rowmax) of
 *          the map of every evaluation e >= jas_first_eval with parameter jas_k, WITHOUT exporting the maps:
 *          what ViTNeuralODE.forward needs of attention_trajectory[-int(0.85 T):] (:614-618).  k <= 3 in the
 *          fused bf16 attention kernel is formed on chip; every other case exports to scratch and reduces;
 *   tape (odevit_tape_bytes() bytes, 1024-aligned) or NULL: when given, the intermediates of every
 *          field evaluation (centred rows, q|k|v, [O|h], fc1 pre-activation, softmax row log-sums)
 *          are kept there for odevit_solve_bwd -- what autograd's saved tensors are in the reference
 *          (train.py:57-67), in bf16 in the bf16 mode -- followed by the folded weights of this call: the reverse
 *          sweep of a tape uses the WEIGHTS AS THEY WERE at the forward call (as autograd's saved tensors do) and reads
 *          `w` only for the parameters that are not folded (biases, LayerNorm affines, res_scale). */
int odevit_solve_fwd(const odevit_desc* desc, const odevit_weights* w, int32_t method,
                     const float* x0, const float* t_grid_host, int32_t n_grid,
                     float* states, float* final_state,
                     float* p_last, float* p_traj, int32_t p_traj_first_eval,
                     float* jas_traj, int32_t jas_first_eval, int32_t jas_k,
                     void* tape, size_t tape_bytes,
                     void* workspace, size_t workspace_bytes, odevit_stream_t stream);

/* Bytes of the tape of a solve over n_grid points (0 on invalid arguments). */
size_t odevit_tape_bytes(const odevit_desc* desc, int32_t method, int32_t n_grid);

/* Reverse sweep through the solve (backprop-through-solver semantics).  With `tape` (written by the
 * forward call of the same desc/method/grid) the stage intermediates are read back; with tape ==
 * NULL each step is recomputed from its stored trajectory row (no stage tensor is kept).
 *   states [T,B,N,D]: the trajectory odevit_solve_fwd produced (row j = input of step j);
 *   g_states [T,B,N,D] or NULL: cotangent of every trajectory row;
 *   g_rows [n_g_rows,B,N,D] + g_row_index_host [n_g_rows] (HOST ints, may repeat): cotangents of
 *          selected rows (final state, control points) -- added on top of g_states;
 *   g_p_last [B,H,N,N] or NULL: cotangent of p_last (the `attentions` output);
 *   g_x0 [B,N,D] out: cotangent of x0 (flows on into the patch embedding);
 *   gw: weight-gradient accumulators (+=). */
int odevit_solve_bwd(const odevit_desc* desc, const odevit_weights* w, int32_t method,
                     const float* t_grid_host, int32_t n_grid, const float* states,
                     const float* g_states,
                     const float* g_rows, const int32_t* g_row_index_host, int32_t n_g_rows,
                     const float* g_p_last,
                     float* g_x0, const odevit_weight_grads* gw,
                     const void* tape, size_t tape_bytes,
                     void* workspace, size_t workspace_bytes, odevit_stream_t stream);

/* Vector-Jacobian product of ONE field evaluation (autograd of odevit_field_fwd):
 *   g_dx [B,N,D] cotangent of dx, g_p [B,H,N,N] or NULL cotangent of p_out;
 *   g_x [B,N,D] out; gw accumulators (+=). Workspace kind ODEVIT_WS_SOLVE_BWD with EULER. */
int odevit_field_bwd(const odevit_desc* desc, const odevit_weights* w,
                     const float* x, const float* g_dx, const float* g_p,
                     float* g_x, const odevit_weight_grads* gw,
                     void* workspace, size_t workspace_bytes, odevit_stream_t stream);

/* Finite-difference curvature of a trajectory in one pass.  Replaces the tensor arithmetic of
 * ViTNeuralODE.compute_upper_bound_by_fininte_difference (ode_transformer_gpt.py:529-543 with
 * finite_difference_second_derivative_sequence :458-468):
 *   per_seq[b,n] = max_j max_d |s[j+2,b,n,d] - 2 s[j+1,b,n,d] + s[j,b,n,d]| / delta_t^2
 * states [T,B,N,D], T >= 3, D % 4 == 0; per_seq [B,N] out.  The caller applies the scalar prefactor and
 * the maxima over n and b (tiny). */
int odevit_fd_curvature(const float* states, int32_t n_grid, int32_t batch, int32_t tokens, int32_t dim,
                        double delta_t, float* per_seq, odevit_stream_t stream);

/* Pre-LayerNorm transformer encoder stack, forward only, no tape: the frozen TEACHER of the distillation
 * step.  Replaces `self.teacher(**inputs, output_hidden_states=True, output_attentions=True)` under
 * torch.no_grad() (loss_trainer.py:318-321; a HF ViTModel encoder: ViTLayer = x + MHA(LN x), x + MLP(LN x))
 * from the embedding output on.  desc: batch, tokens, dim, heads, hidden, precision (variant ignored,
 * dropout must be 0).  layers[l] uses norm_a_* (LayerNorm before attention), norm_b_* (before the MLP),
 * in_proj_w/b = [Wq; Wk; Wv] / [bq; bk; bv] packed [3D, D] / [3D], out_proj_w/b, fc1_w/b, fc2_w/b.
 *   x0 [B,N,D] fp32 in;  hidden [L,B,N,D] fp32 out: the output of every layer (HF's hidden_states[1:]);
 *   p_out: attention maps, p_mode 0 none | 1 last layer only [B,H,N,N] | 2 all layers [L,B,H,N,N].
 * wcache (odevit_encoder_cache_bytes) holds the activation-typed weight copies: pass wcache_valid = 0 whenever the
 * weights changed since the last call with this cache, 1 to reuse them (a frozen teacher: every call but the
 * first).  Workspace kind ODEVIT_WS_ENCODER_FWD. */
size_t odevit_encoder_cache_bytes(const odevit_desc* desc, int32_t n_layers);
int odevit_encoder_fwd(const odevit_desc* desc, const odevit_weights* layers, int32_t n_layers, float ln_eps,
                       const float* x0, float* hidden, float* p_out, int32_t p_mode, void* wcache,
                       size_t wcache_bytes, int32_t wcache_valid, void* workspace, size_t workspace_bytes,
                       odevit_stream_t stream);

/* JaSMin statistic of exported attention maps in one pass.  Replaces the sort-based tensor arithmetic of
 * ViTNeuralODE.jasmin_loss / g_k (ode_transformer_gpt.py:419-456; the reference calls it on detached maps,
 * :614-618): for each [tokens x tokens] slice (evaluation, image, head) of p_maps
 *   out[slice] = max over query rows of log(g_1 / (g_k + 1e-12) + 1e-12)        (k = 0: log(g_1 + 1e-12))
 * with g_j = x_(j) (1 - x_(j) + x_(j+1)), x_(j) the j-th largest entry of the row after clamp to
 * [1e-12, 1] and renormalisation by (row sum + 1e-12).  The caller takes the means over heads, images and
 * evaluations (tiny).  1 <= tokens <= 1024, 0 <= k <= tokens. */
int odevit_jasmin_rowmax(const float* p_maps, int64_t n_slices, int32_t tokens, int32_t k, float* out,
                         odevit_stream_t stream);

/* The fixed-grid solve WITHOUT a materialised trajectory (inference: the reference returns `states` only on
 * request, ode_transformer_gpt.py:628-630, but always needs the finite-difference bound :529-543 and may need the
 * control-point rows :632-639).  The states live in a ring of three inside the workspace.
 *   final_state [B,N,D]: the last state (required);
 *   rows_out [n_rows,B,N,D] or NULL: trajectory rows row_index_host[0..n_rows) (host array, repeats allowed);
 *   fd_max [B*N] or NULL: max over steps j and features d of |s[j+2] - 2 s[j+1] + s[j]| (NOT divided by dt^2),
 *          folded into the epilogue of the step's last GEMM; zero when the grid has fewer than 3 points;
 *   p_last, jas_traj, jas_first_eval, jas_k: as in odevit_solve_fwd.  Workspace: ODEVIT_WS_SOLVE_FWD. */
int odevit_solve_fwd_lean(const odevit_desc* desc, const odevit_weights* w, int32_t method, const float* x0,
                          const float* t_grid_host, int32_t n_grid, float* final_state, float* rows_out,
                          const int32_t* row_index_host, int32_t n_rows, float* fd_max, float* p_last,
                          float* jas_traj, int32_t jas_first_eval, int32_t jas_k, void* workspace,
                          size_t workspace_bytes, odevit_stream_t stream);

/* Adaptive Dormand-Prince 5(4) solve with PER-IMAGE step control, inference only.  Replaces
 * torchdiffeq.odeint(func, x0, t_out, method="dopri5", rtol, atol, options={first_step, max_num_steps}) with one
 * difference of substance: torchdiffeq takes ONE RMS error norm over the whole batch, here every image b is solved on
 * its own N*D elements (its own t, dt, accept/reject decisions and dense output), so a batch of one is the published
 * algorithm and an image's result does not depend on its batch-mates.  Per image (torchdiffeq _impl/dopri5.py,
 * rk_common.py, interp.py, misc.py): FSAL Dormand-Prince with Shampine's error estimate, ratio = RMS(err / (atol +
 * rtol max(|y0|, |y1|))), accept iff ratio <= 1, _optimal_step_size(safety 0.9, ifactor 10, dfactor 0.2, order 5),
 * _select_initial_step(order 4) when first_step <= 0, outputs written from the quartic interpolant of the accepted
 * step that covers them (the solver does not step to them).  Time and dt are fp64 on the device; stage combines run
 * in fp32 with dt cast, as torchdiffeq does.
 *   t_out_host [n_out] fp32 HOST, strictly increasing, 2 <= n_out <= 4096 (decreasing grids are not supported);
 *   max_num_steps: attempted steps per image over the WHOLE solve (torchdiffeq counts per output interval);
 *   states [n_out,B,N,D] out: row 0 = x0, row i = the solution at t_out[i];
 *   nfe, accepted, rejected [B] device int32 or NULL: field evaluations per image
 *          (1 + (first_step <= 0) + 6 * (accepted + rejected)) and step counts.
 * desc must have no dropout.  Workspace kind ODEVIT_WS_SOLVE_ADAPTIVE.  Returns ODEVIT_ERR_NOT_CONVERGED when an
 * image exceeds max_num_steps, meets a non-finite error ratio or a dt that no longer advances t.
 * SYNCHRONISATION: the one entry point of the library that waits for the device.  Each round (one attempted step of
 * every image, six field evaluations of the batch) ends with a copy of its active-image count to pinned host memory;
 * the host enqueues round r + 1 and then waits for round r's count (an event), so the device always has one round
 * queued, and the last round enqueued is a no-op that the call also waits for.  A finished image keeps dt = 0 (its
 * rounds are identity steps) until every image has finished.  Refused (ODEVIT_ERR_UNSUPPORTED) while `stream` is being
 * captured into a CUDA graph. */
int odevit_solve_adaptive(const odevit_desc* desc, const odevit_weights* w, const float* x0, const float* t_out_host,
                          int32_t n_out, double rtol, double atol, double first_step /* <= 0: select */,
                          int32_t max_num_steps, float* states /* [n_out,B,N,D] */, int32_t* nfe, int32_t* accepted,
                          int32_t* rejected /* [B] device, or NULL */, void* workspace, size_t workspace_bytes,
                          odevit_stream_t stream);

/* odevit_solve_adaptive that also records every image's ACCEPTED steps, the schedule odevit_solve_adaptive_bwd
 * differentiates.  step_t0, step_dt [step_cap, B] fp64 and step_out [step_cap, B] int32, device: entry [s, b] is image
 * b's s-th accepted step (its start time, its dt, the first output index not yet written after it); entries past an
 * image's count are zero, so row s of step_dt is the per-image dt of reverse step s.  Everything else, including the
 * states and counts, is bitwise what odevit_solve_adaptive gives.  An image that accepts more than step_cap steps stops
 * the solve with ODEVIT_ERR_WORKSPACE (the message names the image); the solve is deterministic, so a retry with a
 * larger record gives the same result. */
int odevit_solve_adaptive_record(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                                 const float* t_out_host, int32_t n_out, double rtol, double atol, double first_step,
                                 int32_t max_num_steps, float* states, int32_t* nfe, int32_t* accepted,
                                 int32_t* rejected, int32_t step_cap, double* step_t0, double* step_dt,
                                 int32_t* step_out, void* workspace, size_t workspace_bytes, odevit_stream_t stream);

/* Bytes of the tape of odevit_solve_adaptive_bwd for S = max accepted steps: 6 S + 1 field evaluations. */
size_t odevit_adaptive_tape_bytes(const odevit_desc* desc, int32_t S);

/* Reverse sweep through the adaptive solve with the recorded steps FROZEN (discretise-then-optimise): the exact
 * derivative, with respect to x0 and the field's weights, of the computation that maps x0 to `states` along each
 * image's accepted steps -- FSAL Dormand-Prince stages, stage combines in fp32 with dt cast, the quartic dense output at
 * x = (t_out[j] - t0) / dt (fp64, cast).  The step times, dt, x and the choice of step per output are constants: rejected
 * attempts, the error estimate, the step-size controller and the initial-step selection contribute nothing.  (Neither
 * the continuous adjoint nor autograd through an unrolled torchdiffeq dopri5, whose graph also reaches y through the
 * error ratio that sets the next dt.)
 *   x0, t_out_host, n_out: as given to odevit_solve_adaptive_record;  step_t0, step_dt, step_out, step_cap: its record;
 *   n_steps_host [B] HOST int32: accepted steps per image (0 <= n_b <= step_cap);  S = max n_b >= 1;
 *   g_states [n_out,B,N,D]: cotangent of states;  g_x0 [B,N,D] out;  gw: weight-gradient accumulators (+=);
 *   ckpt [S+1,B,N,D] fp32 caller scratch: the state at the start of every reverse step (a replay of the recorded steps
 *        writes it; a finished image's rows repeat its last state);
 *   tape (odevit_adaptive_tape_bytes(desc, S) bytes, 1024-aligned) or NULL: the replay keeps every evaluation's
 *        intermediates there; with NULL the reverse sweep recomputes each step from its checkpoint.
 * 6 S + 1 evaluations replay the steps, 6 S + 1 VJPs run the reverse sweep, plus 6 S recomputed evaluations without a
 * tape.  desc must have no dropout.  Workspace kind ODEVIT_WS_SOLVE_ADAPTIVE_BWD.  Does not synchronise. */
int odevit_solve_adaptive_bwd(const odevit_desc* desc, const odevit_weights* w, const float* x0,
                              const float* t_out_host, int32_t n_out, const double* step_t0, const double* step_dt,
                              const int32_t* step_out, int32_t step_cap, const int32_t* n_steps_host,
                              const float* g_states, float* g_x0, const odevit_weight_grads* gw, float* ckpt,
                              void* tape, size_t tape_bytes, void* workspace, size_t workspace_bytes,
                              odevit_stream_t stream);

/* 1 when odevit_solve_fwd runs this inference solve in the on-chip-state kernel (one persistent CTA per image,
 * trajectory rows written from shared memory): the caller then has no reason to prefer the trajectory-free form. */
int odevit_solve_uses_resident(const odevit_desc* desc, int32_t method, int32_t n_grid);

/* Token assembly, ode_transformer_gpt.py:148-182 (PatchEmbed.forward): the patch projection written straight into
 * the token tensor.
 *   cols_bf16 [B*P, k] bf16: im2col rows of the images (k = C * patch^2, order (c, i, j) as Conv2d's weight);
 *   w_bf16 [dim, k] bf16: proj.weight reshaped;  patch_add [P, dim] fp32: proj.bias + the positional rows of the patch
 *   tokens;  x0 [B, tokens, dim] fp32 out: rows [first_patch_row, first_patch_row + P) of every image come from the
 *   GEMM's epilogue; special_rows [n_special, dim] fp32 (cls / distillation / register rows, positional rows already
 *   added where the reference adds them) go to token positions special_index [n_special] (device int32) of every image. */
int odevit_tokens_fwd(const void* cols_bf16, const void* w_bf16, int32_t batch, int32_t patches, int32_t k, int32_t dim,
                      int32_t tokens, int32_t first_patch_row, const float* patch_add, const float* special_rows,
                      const int32_t* special_index, int32_t n_special, float* x0, odevit_stream_t stream);

/* Head + loss, ode_transformer_gpt.py:588-589, :626: logits = head(final[:, 0]), F.cross_entropy(label_smoothing).
 *   x: first CLS row, x_stride = elements between the CLS rows of consecutive images (tokens * dim for final[:, 0]);
 *   w [classes, dim], bias [classes] or NULL;  logits [B, classes] out;
 *   loss_rows [B] or NULL: the per-image smoothed loss (the module's `loss` is its mean), lse [B] kept for the backward.
 * odevit_head_ce_bwd: dz [B, classes] scratch/out = g_logits (or 0) + g_loss[0] / B * d loss_rows / d logits;
 *   g_x (stride gx_stride) or NULL = dz @ w;  g_w, g_bias (or NULL): += dz^T @ x, += column sums (caller zero-fills). */
int odevit_head_ce_fwd(const float* x, int64_t x_stride, const float* w, const float* bias, const int64_t* labels,
                       int32_t batch, int32_t classes, int32_t dim, float label_smoothing, float* logits, float* loss_rows,
                       float* lse, odevit_stream_t stream);
int odevit_head_ce_bwd(const float* x, int64_t x_stride, const float* w, const int64_t* labels, const float* logits,
                       const float* lse, const float* g_logits, const float* g_loss, int32_t batch, int32_t classes,
                       int32_t dim, float label_smoothing, float* dz, float* g_x, int64_t gx_stride, float* g_w, float* g_bias,
                       odevit_stream_t stream);

/* The L1-attention-loss front-end, loss_trainer.py:80-117 (`ImageDistilTrainer.extract_mass`), one launch:
 *   attn_rows [B,H,n] fp32: the CLS query's attention over the n = side^2 patches (contiguous);
 *   per row: ascending sort, normalise by (sum + 1e-8), cumulative sum c, mask = sigmoid((c - (1 - threshold)) *
 *   scale_factor) (smooth != 0) or [c > 1 - threshold]; the mask goes back to the original positions, multiplies the
 *   row, the [side, side] tile is blurred (3 x 3 gaussian, sigma 0.5, reflect padding; smooth only);
 *   out_mean [B,n]: mean over heads; out_heads [B,H,n] or NULL: per head; out_mask [B,n] or NULL: mean mask.
 * odevit_extract_mass_bwd: g_rows [B,H,n] = VJP for the cotangents g_mean [B,n] and/or g_heads [B,H,n] (smooth: through
 * the blur, the mask and the normalised cumulative sum; hard mask: through the product only, as autograd does). */
int odevit_extract_mass_fwd(const float* attn_rows, int32_t batch, int32_t heads, int32_t n, float threshold, int32_t smooth,
                            float scale_factor, float* out_mean, float* out_heads, float* out_mask, odevit_stream_t stream);
int odevit_extract_mass_bwd(const float* attn_rows, int32_t batch, int32_t heads, int32_t n, float threshold, int32_t smooth,
                            float scale_factor, const float* g_mean, const float* g_heads, float* g_rows,
                            odevit_stream_t stream);

/* GPU-side image preprocessing: what the reference's collator asks of HF `ViTImageProcessor`
 * (datasets/collator.py:11-22): resize to out_h x out_w with Pillow's BILINEAR resampling (bit-exact: fixed point,
 * horizontal then vertical pass, uint8 rounding after each), multiply by `rescale` (1/255), subtract mean, divide by std.
 *   images [B,H,W,3] uint8 (RGB, the layout of np.asarray(PIL image)), device;
 *   bounds_h [out_w,2], kk_h [out_w, ksize(W,out_w)], bounds_v [out_h,2], kk_v [out_h, ksize(H,out_h)]: Pillow's
 *          coefficient tables, built on the HOST by odevit_pil_bilinear_tables and copied to the device by the caller;
 *   tmp [B,H,out_w,3] uint8 device scratch;  out [B,3,out_h,out_w] fp32;  out_u8 [B,out_h,out_w,3] or NULL: the
 *          resized uint8 image itself (what PIL.Image.resize returns). */
int odevit_pil_bilinear_ksize(int32_t in_size, int32_t out_size);
int odevit_pil_bilinear_tables(int32_t in_size, int32_t out_size, int32_t* bounds_host, int32_t* kk_host);
int odevit_preprocess_u8(const uint8_t* images, int32_t batch, int32_t height, int32_t width, int32_t out_h, int32_t out_w,
                         const int32_t* bounds_h, const int32_t* kk_h, const int32_t* bounds_v, const int32_t* kk_v,
                         float rescale, const float* mean3_host, const float* std3_host, uint8_t* tmp, float* out,
                         uint8_t* out_u8, odevit_stream_t stream);

/* Advances a device-resident dropout state by one step (a 1-thread kernel, capturable in a CUDA graph):
 *   state[0] base seed (set once by the caller), state[1] step counter += 1, state[2] = the seed of this step
 *   (a 64-bit mix of base and counter; pass &state[2] as odevit_desc.drop_seed_dev, or a copy of it). */
int odevit_drop_state_advance(uint64_t* state, odevit_stream_t stream);

/* Number of kernels the library launched (process-wide, all threads) since the last reset (bench.py's
 * gpu_launches claim is counted, not estimated). */
int64_t odevit_launch_count(void);
void odevit_reset_launch_count(void);

/* Diagnostic entry (no reference counterpart): the GEMM kernel on its own, for unit parity tests.
 *   C[M,N] (fp32, row-major) = or += sum_k A(m,k) * B(n,k), bf16 operands.
 *   mn_major == 0: A is [M,K], B is [N,K] row-major (K contiguous);
 *   mn_major == 1: A is [K,M], B is [K,N] row-major (the weight-gradient products, split-K).
 *   engine: 0 = CUDA-core FFMA kernel, 1 = tcgen05/TMA kernel (ODEVIT_ERR_UNSUPPORTED if the shape
 *   is outside what it covers). */
int odevit_gemm_bf16(int32_t M, int32_t N, int32_t K, int32_t mn_major, const void* A, const void* B,
                     float* C, int32_t accumulate, int32_t engine, odevit_stream_t stream);

/* Per-kernel-class device timing for bench.py's roofline line (no reference counterpart).
 * While enabled, each launch is bracketed by a CUDA event pair on its stream (a few microseconds
 * of host time per launch).  odevit_profile_read synchronises on the recorded events, so call it
 * after the work has been enqueued; it returns the summed milliseconds and the launch count of
 * class `kclass` since the last enable, or a negative status.  Process-wide like the counter. */
int odevit_profile_enable(int32_t on);
int odevit_profile_reserve(int32_t pairs); /* pre-create event pairs (keeps cudaEventCreate out of timed regions) */
int odevit_profile_num_classes(void);
const char* odevit_profile_class_name(int32_t kclass);
int odevit_profile_read(int32_t kclass, double* total_ms, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* ODEVIT_H_ */
