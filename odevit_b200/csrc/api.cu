// libodevit.so -- orchestration of the hot path and the C ABI (include/odevit.h).
//
// One vector-field evaluation f(u) of the PARALLEL variant (ode_transformer_gpt.py:274-277,
// :317-330) is four launches groups here:
//   1. center_rows        xc = u - mean_D(u)                        (CenterNorm core, :80-81)
//   2. GEMM1 + EPI_FWD1   [q|k|v|h] = xc @ W1cat^T + b1cat, GELU on the fc1 columns
//                         (both CenterNorm affines, the 1/sqrt(d) of MHA and both projections folded
//                          into one weight: see rows.cu::fold_w1_kernel)
//   3. attention          P = softmax(q k^T), O = P v  per (image, head)
//   4. GEMM2 + EPI_RK     scaler * ([O|h] @ [Wo|W2]^T)  fused with the Runge-Kutta stage combine
//                         (writes the next stage input / the next trajectory row directly)
// The solver loop (torchdiffeq fixed grid: euler, midpoint, rk4 = 3/8 rule) runs on the host and
// only enqueues launches; dt_j = t[j+1]-t[j] is formed in fp32 on the host like torchdiffeq does.
//
// The reverse sweep recomputes each step's stage intermediates from the stored trajectory row
// (no stage tensor survives the forward) and applies the exact VJP of the unrolled RK step.
#include <atomic>
#include <cmath>
#include <cstring>
#include <mutex>

#include "epilogue.cuh"
#include "host.h"
#include "internal.h"

#define ODEVIT_STR2(x) #x
#define ODEVIT_STR(x) ODEVIT_STR2(x)

namespace odevit {

// ------------------------------------------------------------------------------------------------
// thread-local error text + launch counter
// ------------------------------------------------------------------------------------------------
// The error text is thread-local; the launch counter and the profiling state are process-wide
// (PyTorch runs the backward on its own autograd thread, which must be counted too).
static thread_local char g_err[512] = "ok";
static std::atomic<int64_t> g_launches{0};
// Process-wide like torch.use_deterministic_algorithms, which the Python layer mirrors into it (and like the counter:
// the backward runs on PyTorch's autograd thread)
static std::atomic<int> g_deterministic{0};

bool deterministic() { return g_deterministic.load(std::memory_order_relaxed) != 0; }

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-class event timing ------------------------------------------------------------------
namespace {
constexpr int kMaxProfPairs = 1 << 16;
struct ProfState {
  std::mutex mu;
  bool on = false;
  int used = 0;
  int cap = 0;
  cudaEvent_t* ev = nullptr;  // 2 per pair
  int* cls = nullptr;
};
ProfState g_prof;
const char* const kClassNames[KC_COUNT] = {
    "center_rows", "gemm_in_qkv_fc1", "attn_qk", "softmax", "attn_pv", "gemm_out_rk",
    "bwd_gemm_doh", "bwd_gemm_g2", "bwd_attn", "bwd_softmax", "bwd_gemm_dx", "bwd_gemm_g1",
    "bwd_colsum", "combine", "weights", "fused_attn", "fused_attn_bwd", "fd_curvature", "fused_attn_export", "resident_solve", "det_sum", "other"};
}  // namespace

ProfScope::ProfScope(int c, cudaStream_t st) : cls(c), s(st), slot(-1) {
  ProfState& p = g_prof;
  if (!p.on) return;
  std::lock_guard<std::mutex> lock(p.mu);
  if (p.used >= p.cap) {
    if (p.cap >= kMaxProfPairs) return;
    if (cudaEventCreate(&p.ev[2 * p.cap]) != cudaSuccess || cudaEventCreate(&p.ev[2 * p.cap + 1]) != cudaSuccess) return;
    ++p.cap;
  }
  slot = p.used++;
  p.cls[slot] = c;
  cudaEventRecord(p.ev[2 * slot], s);
}
ProfScope::~ProfScope() {
  if (slot >= 0) cudaEventRecord(g_prof.ev[2 * slot + 1], s);
}

namespace {

// ------------------------------------------------------------------------------------------------
// Butcher tableaux of the fixed-grid methods (torchdiffeq _impl/fixed_grid.py, rk_common.py)
// ------------------------------------------------------------------------------------------------
const Tableau kEuler = {1, {{0}}, {1.f}};
const Tableau kMidpoint = {2, {{0}, {0.5f}}, {0.f, 1.f}};
const Tableau kRk38 = {4,
                       {{0}, {1.f / 3.f}, {-1.f / 3.f, 1.f}, {1.f, -1.f, 1.f}},
                       {0.125f, 0.375f, 0.375f, 0.125f}};

const Tableau* tableau_for(int method) {
  switch (method) {
    case ODEVIT_EULER: return &kEuler;
    case ODEVIT_MIDPOINT: return &kMidpoint;
    case ODEVIT_RK4_38: return &kRk38;
    default: return nullptr;
  }
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// plan + workspace arena (structs in host.h)
// ------------------------------------------------------------------------------------------------
int make_plan(const odevit_desc* desc, Plan* p) {
  if (!desc) return set_error(ODEVIT_ERR_INVALID_ARG, "desc is NULL");
  if (desc->abi_version != ODEVIT_ABI_VERSION)
    return set_error(ODEVIT_ERR_INVALID_ARG, "abi_version %d != %d", desc->abi_version, ODEVIT_ABI_VERSION);
  p->B = desc->batch; p->N = desc->tokens; p->D = desc->dim; p->H = desc->heads; p->hid = desc->hidden;
  p->variant = desc->variant; p->precision = desc->precision; p->scaler = desc->scaler;
  if (p->B <= 0 || p->N <= 0 || p->D <= 1 || p->H <= 0 || p->hid <= 0)
    return set_error(ODEVIT_ERR_INVALID_ARG, "non-positive dimension (B=%d N=%d D=%d H=%d hid=%d)", p->B, p->N,
                     p->D, p->H, p->hid);
  if (p->D % p->H) return set_error(ODEVIT_ERR_INVALID_ARG, "dim %d not divisible by heads %d", p->D, p->H);
  if (p->D > 1024 || p->N > 1024)
    return set_error(ODEVIT_ERR_UNSUPPORTED, "dim %d / tokens %d above 1024", p->D, p->N);
  if (p->precision != ODEVIT_FP32 && p->precision != ODEVIT_BF16)
    return set_error(ODEVIT_ERR_INVALID_ARG, "unknown precision %d", p->precision);
  if (p->variant != ODEVIT_FIELD_PARALLEL && p->variant != ODEVIT_FIELD_PARALLEL_L2 &&
      p->variant != ODEVIT_FIELD_MACARON)
    return set_error(ODEVIT_ERR_INVALID_ARG, "unknown variant %d", p->variant);
  p->d = p->D / p->H;
  p->M = p->B * p->N;
  p->act = (p->precision == ODEVIT_BF16) ? DT_BF16 : DT_F32;
  // MACARON: the cotangent runs along the fp32 residual chain x -> x1 -> x2 -> x3
  p->dd_type = (p->variant == ODEVIT_FIELD_MACARON) ? DT_F32 : p->act;
  p->p_attn = desc->attn_drop; p->p_proj = desc->proj_drop; p->p_mlp = desc->mlp_drop;
  p->seed_lo = desc->drop_seed_lo; p->seed_hi = desc->drop_seed_hi;
  for (float q : {p->p_attn, p->p_proj, p->p_mlp})
    if (!(q >= 0.f && q < 1.f)) return set_error(ODEVIT_ERR_INVALID_ARG, "dropout probability %g outside [0, 1)", q);
  p->any_drop = (p->p_attn > 0.f || p->p_proj > 0.f || p->p_mlp > 0.f);
  p->seed_dev = p->any_drop ? desc->drop_seed_dev : nullptr;
  p->drop_keys = nullptr;
  // PARALLEL: out-proj and fc2 share one GEMM unless their outputs take different masks.  MACARON runs them as
  // separate GEMMs anyway.
  p->split_out = (p->variant != ODEVIT_FIELD_MACARON) && (p->p_proj > 0.f || p->p_mlp > 0.f);
  p->BHNN = (long long)p->B * p->H * p->N * p->N;
  return 0;
}

// Device-seeded dropout: the key table sits at the head of every workspace layout.
uint32_t* take_drop_keys(const Plan& p, Arena& a) {
  return p.seed_dev ? reinterpret_cast<uint32_t*>(a.take((size_t)kDropKeyEvals * DS_SITES * 4)) : nullptr;
}

WeightBufs take_weights(const Plan& p, Arena& a) {
  const size_t e = dtype_size(p.act);
  const size_t R = 3 * (size_t)p.D + p.hid, K2 = (size_t)p.D + p.hid;
  WeightBufs w;
  w.w1cat = a.take(R * p.D * e);
  w.w1catT = a.take(R * p.D * e);
  w.w2cat = a.take(K2 * p.D * e);
  w.w2catT = a.take(K2 * p.D * e);
  w.b1cat = a.f32(R);
  w.b2 = a.f32(p.D);
  w.fmean = a.f32(R);
  w.user = nullptr;
  return w;
}
StageCtx take_ctx(const Plan& p, Arena& a, bool with_hpre) {
  const size_t e = dtype_size(p.act);
  const size_t MD = (size_t)p.M * p.D, Mh = (size_t)p.M * p.hid;
  const bool mac = (p.variant == ODEVIT_FIELD_MACARON);
  if (mac) with_hpre = true;  // the chain x -> x1 -> x2 is written either way; keep one layout
  StageCtx c{};
  c.xc = a.take(MD * e);
  c.qkv = a.take(3 * MD * e);
  c.oh = a.take((MD + Mh) * e);
  c.hpre = with_hpre ? a.take(Mh * e) : nullptr;
  c.lse = with_hpre ? a.f32((size_t)p.B * p.H * p.N) : nullptr;
  if (mac) {
    c.x0 = a.f32(MD);
    c.x1 = a.f32(MD);
    c.x2 = a.f32(MD);
    c.n2 = a.take(MD * e);
    c.n3 = a.take(MD * e);
    c.hpre3 = a.take(Mh * e);
    c.h3 = a.take(Mh * e);
  }
  return c;
}

// deterministic mode: one scratch region for the partial slabs of whichever reduction runs (they run one after another
// on the call's stream, each finished by its det_sum before the next starts)
void det_scratch(const Plan& p, Arena& a) {
  p.det_ws = nullptr;
  p.det_ws_bytes = 0;
  if (!deterministic()) return;
  const int R = 3 * p.D + p.hid;
  size_t f = gemm_tc_det_bytes() / 4;
  auto at_least = [&f](size_t n) { if (n > f) f = n; };
  at_least(colsum_part_floats(p.M, R));
  at_least(ln_bwd_part_floats(p.M, p.D));
  at_least(unfold_part_floats(p.D, p.hid));
  p.det_ws_bytes = f * 4;
  p.det_ws = a.f32(f);
}

void split_scratch(const Plan& p, Arena& a) {
  p.split_a = p.split_b = nullptr;
  p.split_a_bytes = p.split_b_bytes = 0;
  static const bool off = [] { const char* e = getenv("ODEVIT_FP32_SPLIT"); return e && e[0] == '0'; }();
  if (p.precision != ODEVIT_FP32 || off) return;
  const size_t R = 3 * (size_t)p.D + p.hid, K2 = (size_t)p.D + p.hid;
  const size_t mk2 = (size_t)p.M * K2, rd = R * (size_t)p.D;
  p.split_a_bytes = 3 * (size_t)p.M * R * 2;   // three segments of the mu GEMM's K = 3D + hid
  p.split_b_bytes = 3 * (mk2 > 2 * rd ? mk2 : 2 * rd) * 2;
  p.split_a = a.take(p.split_a_bytes);
  p.split_b = a.take(p.split_b_bytes);
}

struct FwdBufs {
  uint32_t* drop_keys;
  WeightBufs w;
  StageCtx ctx;
  float* P;
  float* u;
  float* k[3];
  float* ytmp[3];   // trajectory-free solves: a ring of three states (the finite-difference window)
  float* sq;
  float* tmp;
  float* kbuf;
};
FwdBufs layout_fwd(const Plan& p, Arena& a, int S) {
  FwdBufs f;
  f.drop_keys = take_drop_keys(p, a);
  f.w = take_weights(p, a);
  f.ctx = take_ctx(p, a, false);
  f.P = a.f32(p.BHNN);
  f.u = a.f32((size_t)p.M * p.D);
  for (int i = 0; i < 3; ++i) f.k[i] = (i < S - 1) ? a.f32((size_t)p.M * p.D) : nullptr;
  for (int i = 0; i < 3; ++i) f.ytmp[i] = a.f32((size_t)p.M * p.D);
  f.sq = (p.variant == ODEVIT_FIELD_PARALLEL_L2) ? a.f32((size_t)2 * p.B * p.H * p.N) : nullptr;
  f.tmp = p.split_out ? a.f32((size_t)p.M * p.D) : nullptr;
  f.kbuf = (S > 1 && solve_resident_shape_ok(p)) ? a.f32(solve_resident_scratch_floats(p)) : nullptr;
  split_scratch(p, a);
  return f;
}

BwdBufs layout_bwd(const Plan& p, Arena& a, int S) {
  const size_t e = dtype_size(p.act);
  const size_t MD = (size_t)p.M * p.D;
  const size_t R = 3 * (size_t)p.D + p.hid, K2 = (size_t)p.D + p.hid;
  BwdBufs b;
  b.drop_keys = take_drop_keys(p, a);
  b.w = take_weights(p, a);
  for (int i = 0; i < 4; ++i) b.ctx[i] = (i < S) ? take_ctx(p, a, true) : StageCtx{};
  b.P = a.f32(p.BHNN);
  b.dP = a.f32(p.BHNN);
  b.u = a.f32(MD);
  for (int i = 0; i < 3; ++i) b.k[i] = (i < S - 1) ? a.f32(MD) : nullptr;
  b.dd = a.take(MD * dtype_size(p.dd_type));
  b.dO = a.take(MD * e);
  b.dz = a.take((size_t)p.M * R * e);
  for (int i = 0; i < 4; ++i) b.mu[i] = (i >= 1 && i < S) ? a.f32(MD) : nullptr;
  b.gy = a.f32(MD);
  b.delta = a.f32((size_t)p.B * p.H * p.N);
  {
    const size_t n = attn_bwd_tc_scratch_floats(p.B, p.N, p.H);
    b.dq_scratch = n ? a.f32(n) : nullptr;
  }
  // accumulators, contiguous (sizes are multiples of 4 bytes; keep them packed for one memset)
  const size_t acc_floats = R * p.D + R + K2 * p.D + 2 * (size_t)p.D;
  float* acc = a.f32(acc_floats);
  b.G1 = acc;
  b.c1 = acc ? acc + R * p.D : nullptr;
  b.G2 = acc ? acc + R * p.D + R : nullptr;
  b.c2 = acc ? acc + R * p.D + R + K2 * p.D : nullptr;
  b.c3 = acc ? b.c2 + p.D : nullptr;
  b.acc_bytes = acc_floats * 4;
  const bool mac = (p.variant == ODEVIT_FIELD_MACARON);
  b.dn = mac ? a.f32(MD) : nullptr;
  b.ddc = mac ? a.take(MD * e) : nullptr;
  b.sq = (p.variant == ODEVIT_FIELD_PARALLEL_L2) ? a.f32((size_t)2 * p.B * p.H * p.N) : nullptr;
  b.tmp = p.split_out ? a.f32(MD) : nullptr;
  b.dd1 = p.split_out ? a.take(MD * e) : nullptr;
  b.dd2 = p.split_out ? a.take(MD * e) : nullptr;
  split_scratch(p, a);
  det_scratch(p, a);
  return b;
}

// The tape: one StageCtx per field evaluation e = step*S + stage, written by the forward solve and
// read by the reverse sweep instead of recomputing the step (HBM is 180 GB: at the C100 bench shape
// the tape is 3.3 GB).  Layout is a pure function of (plan, n_evals): n_evals slots of tape_slot_bytes,
// then the folded weights of the forward (tape_weights).
size_t tape_slot_bytes(const Plan& p) {
  Arena a(nullptr);
  take_ctx(p, a, true);
  return (a.off + 1023) & ~size_t(1023);
}

size_t tape_bytes(const Plan& p, long long n_evals) {
  Arena aw(nullptr);
  take_weights(p, aw);
  return tape_slot_bytes(p) * (size_t)n_evals + ((aw.off + 1023) & ~size_t(1023));
}

StageCtx tape_ctx(const Plan& p, const void* tape, long long e) {
  Arena a(const_cast<char*>(reinterpret_cast<const char*>(tape)) + tape_slot_bytes(p) * (size_t)e);
  return take_ctx(p, a, true);
}

// The folded / transposed weights of the forward solve, stored behind the tape's evaluation slots: the reverse sweep of
// the same step reads them instead of folding the (unchanged) parameters a second time.
WeightBufs tape_weights(const Plan& p, const void* tape, long long n_evals) {
  Arena a(const_cast<char*>(reinterpret_cast<const char*>(tape)) + tape_slot_bytes(p) * (size_t)n_evals);
  return take_weights(p, a);
}

int check_ws(const void* ws, size_t have, size_t need) {
  if (!ws) return set_error(ODEVIT_ERR_WORKSPACE, "workspace is NULL");
  if (reinterpret_cast<uintptr_t>(ws) & 1023) return set_error(ODEVIT_ERR_WORKSPACE, "workspace not 1024-byte aligned");
  if (have < need) return set_error(ODEVIT_ERR_WORKSPACE, "workspace too small: %zu < %zu bytes", have, need);
  return 0;
}

int check_tape(const Plan& p, const void* tape, size_t bytes, long long n_evals) {
  ODV_TRY(check_device_ptr(tape, "tape"));
  return check_ws(tape, bytes, tape_bytes(p, n_evals));
}

int check_device_ptr(const void* p, const char* what) {
  if (!p) return set_error(ODEVIT_ERR_INVALID_ARG, "%s is NULL", what);
  cudaPointerAttributes attr;
  cudaError_t e = cudaPointerGetAttributes(&attr, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return set_error(ODEVIT_ERR_NOT_DEVICE_PTR, "%s: cudaPointerGetAttributes failed: %s", what, cudaGetErrorString(e));
  }
  if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
    return set_error(ODEVIT_ERR_NOT_DEVICE_PTR, "%s is not device memory (no CPU fallback)", what);
  // this library carries its own (static) CUDA runtime: follow the caller's device
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess || cur != attr.device) {
    cudaError_t e2 = cudaSetDevice(attr.device);
    if (e2 != cudaSuccess)
      return set_error(ODEVIT_ERR_CUDA, "cudaSetDevice(%d) failed: %s", attr.device, cudaGetErrorString(e2));
  }
  return 0;
}

int check_weights(const Plan& p, const odevit_weights* w) {
  if (!w) return set_error(ODEVIT_ERR_INVALID_ARG, "weights is NULL");
  if (!w->norm_a_w || !w->norm_a_b || !w->norm_b_w || !w->norm_b_b || !w->in_proj_w || !w->out_proj_w ||
      !w->fc1_w || !w->fc2_w)
    return set_error(ODEVIT_ERR_INVALID_ARG, "the field needs norm_a/norm_b/in_proj/out_proj/fc1/fc2 weights");
  if (p.variant == ODEVIT_FIELD_PARALLEL_L2 && (!w->in_proj_b || !w->out_proj_b))
    return set_error(ODEVIT_ERR_INVALID_ARG, "PARALLEL_L2 needs in_proj_b ([bq;bk;bv]) and out_proj_b");
  if (p.variant == ODEVIT_FIELD_MACARON &&
      (!w->norm_c_w || !w->norm_c_b || !w->in_proj_b || !w->out_proj_b || !w->fc1_b || !w->fc2_b || !w->res_scale))
    return set_error(ODEVIT_ERR_INVALID_ARG, "MACARON needs norm_c, all four biases and res_scale");
  return check_device_ptr(w->in_proj_w, "weights.in_proj_w");
}

float q_scale_of(const Plan& p) {
  // nn.MultiheadAttention scales q by 1/sqrt(d) (folded into the Wq rows); L2SelfAttention applies its
  // scale to the squared distance instead (ode_transformer_gpt.py:24, :54)
  return (p.variant == ODEVIT_FIELD_PARALLEL_L2) ? 1.f : 1.f / sqrtf((float)p.d);
}

int prepare_weights(const Plan& p, const odevit_weights* w, WeightBufs& wb, cudaStream_t s) {
  FoldArgs f;
  f.D = p.D; f.hid = p.hid; f.heads = p.H; f.w = w;
  f.q_scale = q_scale_of(p);
  f.fold_norm = (p.variant != ODEVIT_FIELD_MACARON);
  f.w1cat = wb.w1cat; f.w1catT = wb.w1catT; f.w_type = p.act;
  f.b1cat = wb.b1cat; f.w2cat = wb.w2cat; f.w2catT = wb.w2catT; f.b2 = wb.b2;
  f.fmean = wb.fmean;
  wb.user = w;
  return fold_weights_parallel(f, s);
}

namespace {
// q / k / v views of the packed qkv buffer for batch z = (image b, head h)
struct HeadView {
  long long bo, bi, rs;
};
HeadView qkv_view(const Plan& p) { return {(long long)p.N * 3 * p.D, (long long)p.d, (long long)3 * p.D}; }

}  // namespace

// ------------------------------------------------------------------------------------------------
// GEMM dispatch: tcgen05 in bf16 mode where the kernel covers the shape, FFMA otherwise
// ------------------------------------------------------------------------------------------------
Drop make_drop(const Plan& p, int site, long long e) {
  Drop d;
  const float q = (site == DS_ATTN) ? p.p_attn : (site == DS_PROJ) ? p.p_proj : p.p_mlp;
  if (!(q > 0.f)) return d;
  const double t = (double)q * 4294967296.0;
  d.thresh = t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
  if (d.thresh == 0) d.thresh = 1;
  d.scale = 1.f / (1.f - q);
  if (p.drop_keys) d.key_ptr = p.drop_keys + e * DS_SITES + site;   // resolved on the device from the resident seed
  else d.key = drop_site_key(p.seed_lo, p.seed_hi, e, site);
  return d;
}

// Device-seeded dropout: the key table (head of every workspace layout) is filled at the start of the call.
static int prepare_drop_keys(Plan& p, uint32_t* table, long long n_evals, cudaStream_t s) {
  if (!p.seed_dev) return 0;
  if (n_evals > kDropKeyEvals)
    return set_error(ODEVIT_ERR_UNSUPPORTED, "device-seeded dropout addresses %d field evaluations per call, %lld asked", kDropKeyEvals, n_evals);
  ODV_TRY(check_device_ptr(p.seed_dev, "drop_seed_dev"));
  p.drop_keys = table;
  return resolve_drop_keys(p.seed_dev, table, (int)(n_evals > 0 ? n_evals : 1) * DS_SITES, s);
}

// The fp32 mode on the tensor core: every fp32 operand x is split into bf16 pieces hi = bf16(x), mid = bf16(x - hi),
// lo = bf16(x - hi - mid) (8 mantissa bits each) and the leading cross products are ONE bf16 GEMM over a longer
// contraction axis -- e.g. A' = [hi | hi | mid], B' = [hi | mid | hi] -- with fp32 accumulation in tensor memory and the
// usual fused epilogue (erf-form GELU).  Three products leave 2^-18 relative per term.  Against the reference's goldens final states, logits, losses and
// bounds stay inside 1e-4 and gradients inside 2e-3; the exported attention maps (the state error of the whole solve
// sits in the softmax's exponent) reach 1.6e-4 (tests/test_gpu_parity.py).  ODEVIT_FP32_SPLIT=0 selects the FFMA kernel.  Operands the tcgen05 kernel cannot take
// (batched per-head products, odd strides) stay on the FFMA kernel.
static int gemm_split3(const Plan& p, const GemmArgs& g, cudaStream_t s, bool* taken) {
  *taken = false;
  if (!p.split_a || !p.split_b || g.a_type != DT_F32 || g.b_type != DT_F32 || g.batch_outer * g.batch_inner != 1) return 0;
  const bool a_k = (g.a_cs == 1), a_mn = (g.a_rs == 1 && g.a_cs != 1);
  const bool b_k = (g.b_cs == 1), b_mn = (g.b_rs == 1 && g.b_cs != 1);
  if (!((a_k && !a_mn && b_k && !b_mn) || (a_mn && b_mn))) return 0;
  const bool mn = a_mn;
  if (g.K % 8 || (mn && (g.M % 8 || g.N % 8))) return 0;
  if ((mn ? g.a_cs : g.a_rs) % 4 || (mn ? g.b_cs : g.b_rs) % 4) return 0;
  if ((reinterpret_cast<uintptr_t>(g.A) | reinterpret_cast<uintptr_t>(g.B)) & 15) return 0;
  // products kept: (hi,hi) (hi,mid) (mid,hi).  Six products (adding (hi,lo) (mid,mid) (lo,hi): 2^-26 per term) were
  // measured and are NOT more accurate here: the tensor core's fp32 accumulation is not round-to-nearest, its error
  // grows with the length of the contraction, and the doubled axis cost more than the extra terms bought (exported
  // attention map of the 224 px RK4 case: 1.6e-4 with three segments, 2.2e-4 with six).
  static const int pa[3] = {0, 0, 1}, pb[3] = {0, 1, 0};
  constexpr int ns = 3;
  if ((size_t)ns * g.M * g.K * 2 > p.split_a_bytes || (size_t)ns * g.N * g.K * 2 > p.split_b_bytes) return 0;
  GemmArgs t = g;
  t.K = ns * g.K;
  t.A = p.split_a; t.a_type = DT_BF16;
  t.B = p.split_b; t.b_type = DT_BF16;
  if (!mn) { t.a_rs = (long long)ns * g.K; t.a_cs = 1; t.b_rs = (long long)ns * g.K; t.b_cs = 1; }
  else { t.a_rs = 1; t.a_cs = g.M; t.b_rs = 1; t.b_cs = g.N; }
  t.epi.exact_gelu = true;
  if (!gemm_tc_supports(t)) return 0;
  const float* A = reinterpret_cast<const float*>(g.A);
  const float* B = reinterpret_cast<const float*>(g.B);
  if (!mn) {
    ODV_TRY(split_bf16(A, g.a_rs, g.M, g.K, 0, ns, pa, p.split_a, s));
    ODV_TRY(split_bf16(B, g.b_rs, g.N, g.K, 0, ns, pb, p.split_b, s));
  } else {   // element (m, k) at A[k * cs + m]: a [K, M] matrix, pieces stacked along k
    ODV_TRY(split_bf16(A, g.a_cs, g.K, g.M, 1, ns, pa, p.split_a, s));
    ODV_TRY(split_bf16(B, g.b_cs, g.K, g.N, 1, ns, pb, p.split_b, s));
  }
  *taken = true;
  return gemm_tc(t, s);
}

int gemm(const Plan& p, const GemmArgs& g_in, cudaStream_t s) {
  GemmArgs g = g_in;
  g.det_ws = p.det_ws;
  g.det_ws_bytes = p.det_ws_bytes;
  if (p.precision == ODEVIT_BF16 && gemm_tc_supports(g)) return gemm_tc(g, s);
  if (p.precision == ODEVIT_FP32) {
    bool taken = false;
    ODV_TRY(gemm_split3(p, g, s, &taken));
    if (taken) return 0;
  }
  return gemm_simt(g, s);
}

// ------------------------------------------------------------------------------------------------
// attention per (image, head): fused tcgen05 kernels in bf16 mode (head dim 64, N <= 256), else
// batched FFMA products + row kernels.  PARALLEL_L2 swaps the softmax for the L2 weights (:48-56).
// ------------------------------------------------------------------------------------------------
int attention_forward(const Plan& p, const void* qkv_v, void* oh, long long ld_oh, float* P, float* p_copy,
                      float* lse, float* sq, Drop drop, cudaStream_t s, float* jas_out, int jas_k) {
  const int D = p.D;
  const bool l2 = (p.variant == ODEVIT_FIELD_PARALLEL_L2);
  if (!l2 && p.precision == ODEVIT_BF16 && attn_fwd_tc_supports(p.N, D, p.H, p.act, ld_oh)) {
    if (jas_out && !p_copy && !drop.thresh && attn_fwd_tc_jasmin_supports(p.N, jas_k))
      return attn_fwd_tc(qkv_v, oh, ld_oh, nullptr, lse, p.B, p.N, p.H, D, drop, s, jas_out, jas_k);   // statistic in-kernel
    float* pc = (jas_out && !p_copy) ? P : p_copy;     // JaSMin wanted but not built in-kernel for this case: export + row kernel
    ODV_TRY(attn_fwd_tc(qkv_v, oh, ld_oh, pc, lse, p.B, p.N, p.H, D, drop, s));
    if (jas_out) ODV_TRY(jasmin_rowmax(pc, (long long)p.B * p.H, p.N, jas_k, jas_out, s));
    return 0;
  }
  const HeadView hv = qkv_view(p);
  const char* qkv = reinterpret_cast<const char*>(qkv_v);
  const size_t e = dtype_size(p.act);
  {  // S = q k^T  (MHA: the 1/sqrt(d) is folded into the Wq rows)
    GemmArgs g;
    g.M = p.N; g.N = p.N; g.K = p.d;
    g.A = qkv; g.a_type = p.act; g.a_rs = hv.rs; g.a_cs = 1; g.a_bo = hv.bo; g.a_bi = hv.bi;
    g.B = qkv + (size_t)D * e; g.b_type = p.act; g.b_rs = hv.rs; g.b_cs = 1; g.b_bo = hv.bo; g.b_bi = hv.bi;
    g.batch_outer = p.B; g.batch_inner = p.H;
    g.epi_mode = EPI_STORE;
    g.epi.out = P; g.epi.out_type = DT_F32; g.epi.ld_out = p.N;
    g.epi.out_bo = (long long)p.H * p.N * p.N; g.epi.out_bi = (long long)p.N * p.N;
    g.kclass = KC_ATTN_S;
    ODV_TRY(gemm_simt(g, s));
  }
  if (l2) {
    if (!sq) return set_error(ODEVIT_ERR_WORKSPACE, "L2 attention: squared-norm scratch missing");
    ODV_TRY(head_sqnorm(qkv_v, p.act, sq, p.B, p.N, p.H, D, s));
    ODV_TRY(l2_prob_rows(P, sq, 1.f / sqrtf((float)p.d), drop.thresh ? nullptr : p_copy, p.B, p.H, p.N, s));
  } else {
    ODV_TRY(softmax_rows(P, drop.thresh ? nullptr : p_copy, (long long)p.B * p.H * p.N, p.N, s));
  }
  // attention-map dropout: what the caller sees (p_copy) and what multiplies v are both post-dropout
  if (drop.thresh) ODV_TRY(drop_inplace_f32(P, p_copy, drop, (long long)p.B * p.H * p.N, p.N, s));
  {  // O = P v  -> columns [h*d, (h+1)*d) of the output buffer
    GemmArgs g;
    g.M = p.N; g.N = p.d; g.K = p.N;
    g.A = P; g.a_type = DT_F32; g.a_rs = p.N; g.a_cs = 1;
    g.a_bo = (long long)p.H * p.N * p.N; g.a_bi = (long long)p.N * p.N;
    g.B = qkv + (size_t)2 * D * e; g.b_type = p.act; g.b_rs = 1; g.b_cs = hv.rs; g.b_bo = hv.bo; g.b_bi = hv.bi;
    g.batch_outer = p.B; g.batch_inner = p.H;
    g.epi_mode = EPI_STORE;
    g.epi.out = oh; g.epi.out_type = p.act; g.epi.ld_out = ld_oh;
    g.epi.out_bo = (long long)p.N * ld_oh; g.epi.out_bi = p.d;
    g.kclass = KC_ATTN_PV;
    ODV_TRY(gemm_simt(g, s));
  }
  if (jas_out) ODV_TRY(jasmin_rowmax(P, (long long)p.B * p.H, p.N, jas_k, jas_out, s));   // P holds the (post-dropout) map
  return 0;
}

// dq_colsum / colsum_done: the fused kernel can add the column sums of dq (the q-row bias gradient) into dq_colsum
// on its way out; *colsum_done says whether it did
int attention_vjp(const Plan& p, const void* qkv_v, const void* oh, long long ld_oh, const float* lse, BwdBufs& b,
                  const float* g_p, void* dz_v, int R, Drop drop, cudaStream_t s, float* dq_colsum, bool* colsum_done) {
  if (colsum_done) *colsum_done = false;
  const int D = p.D;
  const bool l2 = (p.variant == ODEVIT_FIELD_PARALLEL_L2);
  const size_t e = dtype_size(p.act);
  char* dz = reinterpret_cast<char*>(dz_v);
  if (!l2 && p.precision == ODEVIT_BF16 && !g_p && lse && attn_fwd_tc_supports(p.N, D, p.H, p.act, ld_oh)) {
    // fused tcgen05 kernel (P recomputed on chip from q, k and the saved row log-sum-exp)
    if (colsum_done) *colsum_done = dq_colsum != nullptr;
    return attn_bwd_tc(qkv_v, b.dO, oh, ld_oh, lse, b.delta, dz_v, R, b.dq_scratch, p.B, p.N, p.H, D, drop, s, nullptr, nullptr,
                       dq_colsum);
  }
  if (!l2 && p.precision == ODEVIT_BF16 && g_p && lse && !drop.thresh && b.P && b.delta &&
      attn_fwd_tc_supports(p.N, D, p.H, p.act, ld_oh)) {
    // a cotangent on the exported map (the `attentions` output, last evaluation): its row term
    // sum_j P_ij g_ij needs the normalised map once -- re-exported by the forward kernel (which rewrites O with
    // the very same values) -- then the fused kernel adds g to dP on the fly
    ODV_TRY(attn_fwd_tc(qkv_v, const_cast<void*>(oh), ld_oh, b.P, nullptr, p.B, p.N, p.H, D, Drop{}, s));
    ODV_TRY(rowdot_rows(b.P, g_p, b.delta, (long long)p.B * p.H * p.N, p.N, s));
    if (colsum_done) *colsum_done = dq_colsum != nullptr;
    return attn_bwd_tc(qkv_v, b.dO, oh, ld_oh, lse, b.delta, dz_v, R, b.dq_scratch, p.B, p.N, p.H, D, drop, s, g_p, b.delta, dq_colsum);
  }
  const HeadView hv = qkv_view(p);
  const char* qkv = reinterpret_cast<const char*>(qkv_v);
  const long long pbo = (long long)p.H * p.N * p.N, pbi = (long long)p.N * p.N;
  auto head_gemm = [&](GemmArgs& g) {
    g.batch_outer = p.B; g.batch_inner = p.H;
    g.kclass = KC_BWD_ATTN;
    return gemm_simt(g, s);
  };
  {  // S
    GemmArgs g;
    g.M = p.N; g.N = p.N; g.K = p.d;
    g.A = qkv; g.a_type = p.act; g.a_rs = hv.rs; g.a_cs = 1; g.a_bo = hv.bo; g.a_bi = hv.bi;
    g.B = qkv + (size_t)D * e; g.b_type = p.act; g.b_rs = hv.rs; g.b_cs = 1; g.b_bo = hv.bo; g.b_bi = hv.bi;
    g.epi.out = b.P; g.epi.ld_out = p.N; g.epi.out_bo = pbo; g.epi.out_bi = pbi;
    ODV_TRY(head_gemm(g));
  }
  float ds_coef = 1.f;  // d(q k^T) = ds_coef * ds
  if (l2) {
    if (!b.sq) return set_error(ODEVIT_ERR_WORKSPACE, "L2 attention: squared-norm scratch missing");
    ODV_TRY(head_sqnorm(qkv_v, p.act, b.sq, p.B, p.N, p.H, D, s));
    ODV_TRY(l2_prob_rows(b.P, b.sq, 1.f / sqrtf((float)p.d), nullptr, p.B, p.H, p.N, s));
    ds_coef = 2.f / sqrtf((float)p.d);
  } else {
    ODV_TRY(softmax_rows(b.P, nullptr, (long long)p.B * p.H * p.N, p.N, s));
  }
  {  // dP = dO v^T
    GemmArgs g;
    g.M = p.N; g.N = p.N; g.K = p.d;
    g.A = b.dO; g.a_type = p.act; g.a_rs = D; g.a_cs = 1; g.a_bo = (long long)p.N * D; g.a_bi = p.d;
    g.B = qkv + (size_t)2 * D * e; g.b_type = p.act; g.b_rs = hv.rs; g.b_cs = 1; g.b_bo = hv.bo; g.b_bi = hv.bi;
    g.epi.out = b.dP; g.epi.ld_out = p.N; g.epi.out_bo = pbo; g.epi.out_bi = pbi;
    ODV_TRY(head_gemm(g));
  }
  if (drop.thresh) {
    // O = drop(P) v and the exported map is drop(P):  cotangent of P = mask o (dO v^T + g_p)
    if (g_p) ODV_TRY(axpy_f32(b.dP, g_p, 1.f, p.BHNN, s));
    ODV_TRY(drop_inplace_f32(b.dP, nullptr, drop, (long long)p.B * p.H * p.N, p.N, s));
    g_p = nullptr;
  }
  // ds = P o (dP - sum_j P dP): also the L2 weights' VJP w.r.t. -scale*dist^2 (the +1e-8 drops out)
  ODV_TRY(softmax_bwd_rows(b.P, b.dP, g_p, (long long)p.B * p.H * p.N, p.N, s));
  if (drop.thresh) ODV_TRY(drop_inplace_f32(b.P, nullptr, drop, (long long)p.B * p.H * p.N, p.N, s));  // dv uses drop(P)
  {  // dq = ds k      (MHA: dq is the cotangent of the already-scaled q, the scale lives in W1cat)
    GemmArgs g;
    g.M = p.N; g.N = p.d; g.K = p.N;
    g.A = b.dP; g.a_type = DT_F32; g.a_rs = p.N; g.a_cs = 1; g.a_bo = pbo; g.a_bi = pbi;
    g.B = qkv + (size_t)D * e; g.b_type = p.act; g.b_rs = 1; g.b_cs = hv.rs; g.b_bo = hv.bo; g.b_bi = hv.bi;
    g.epi.alpha = ds_coef;
    g.epi.out = dz; g.epi.out_type = p.act; g.epi.ld_out = R; g.epi.out_bo = (long long)p.N * R; g.epi.out_bi = p.d;
    ODV_TRY(head_gemm(g));
  }
  {  // dk = ds^T q
    GemmArgs g;
    g.M = p.N; g.N = p.d; g.K = p.N;
    g.A = b.dP; g.a_type = DT_F32; g.a_rs = 1; g.a_cs = p.N; g.a_bo = pbo; g.a_bi = pbi;
    g.B = qkv; g.b_type = p.act; g.b_rs = 1; g.b_cs = hv.rs; g.b_bo = hv.bo; g.b_bi = hv.bi;
    g.epi.alpha = ds_coef;
    g.epi.out = dz + (size_t)D * e; g.epi.out_type = p.act; g.epi.ld_out = R;
    g.epi.out_bo = (long long)p.N * R; g.epi.out_bi = p.d;
    ODV_TRY(head_gemm(g));
  }
  {  // dv = P^T dO
    GemmArgs g;
    g.M = p.N; g.N = p.d; g.K = p.N;
    g.A = b.P; g.a_type = DT_F32; g.a_rs = 1; g.a_cs = p.N; g.a_bo = pbo; g.a_bi = pbi;
    g.B = b.dO; g.b_type = p.act; g.b_rs = 1; g.b_cs = D; g.b_bo = (long long)p.N * D; g.b_bi = p.d;
    g.epi.out = dz + (size_t)2 * D * e; g.epi.out_type = p.act; g.epi.ld_out = R;
    g.epi.out_bo = (long long)p.N * R; g.epi.out_bi = p.d;
    ODV_TRY(head_gemm(g));
  }
  // L2: dist^2 = |q|^2 + |k|^2 - 2 q.k -- the squared-norm terms add -ds_coef*rowsum(ds) q, -ds_coef*colsum(ds) k
  if (l2) ODV_TRY(l2_vjp_fix(b.dP, qkv_v, p.act, dz_v, R, ds_coef, p.B, p.N, p.H, D, s));
  return 0;
}

// Forward evaluation at stage input `u`.  `rk` (nullable) is the epilogue of the last GEMM.
int eval_forward(const Plan& p, const WeightBufs& wb, const StageCtx& c, const float* u, float* P,
                 float* p_copy, float* sq, float* tmp, long long e, const Epi* rk, cudaStream_t s,
                 float* jas_out, int jas_k) {
  if (p.variant == ODEVIT_FIELD_MACARON) return macaron_forward(p, wb, c, u, P, rk, e, s);
  const int D = p.D, hid = p.hid, R = 3 * D + hid, K2 = D + hid;
  ODV_TRY(center_rows(u, c.xc, p.act, nullptr, 0.f, p.M, D, s));
  {
    GemmArgs g;
    g.M = p.M; g.N = R; g.K = D;
    g.A = c.xc; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
    g.B = wb.w1cat; g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
    g.epi_mode = EPI_FWD1;
    g.kclass = KC_GEMM_IN;
    g.epi.bias = wb.b1cat;
    g.epi.out = c.qkv; g.epi.out_type = p.act; g.epi.ld_out = 3 * D;
    g.epi.split = 3 * D;
    g.epi.out2 = reinterpret_cast<char*>(c.oh) + (size_t)D * dtype_size(p.act); g.epi.ld_out2 = K2;
    g.epi.out3 = c.hpre; g.epi.ld_out3 = hid;   // (holds GELU'(pre-activation): Epi::aux_gelu_grad)
    g.epi.aux_gelu_grad = true;
    g.epi.aux_type = p.act;
    g.epi.drop = make_drop(p, DS_MLP_H, e);   // dropout after GELU (:196-197)
    ODV_TRY(gemm(p, g, s));
  }
  ODV_TRY(attention_forward(p, c.qkv, c.oh, K2, P, p_copy, c.lse, sq, make_drop(p, DS_ATTN, e), s, jas_out, jas_k));
  if (rk && p.split_out) {
    // out-proj and fc2 outputs take different dropout masks (:231 proj_drop, :199 mlp drop): two GEMMs,
    // the first parks scaler * drop(h W2^T) in `tmp`, the second adds it (Epi::resid) before the stage combine
    const size_t es = dtype_size(p.act);
    if (!tmp) return set_error(ODEVIT_ERR_WORKSPACE, "dropout: scratch for the split output projection missing");
    {
      GemmArgs g;
      g.M = p.M; g.N = D; g.K = hid;
      g.A = reinterpret_cast<const char*>(c.oh) + (size_t)D * es; g.a_type = p.act; g.a_rs = K2; g.a_cs = 1;
      g.B = reinterpret_cast<const char*>(wb.w2cat) + (size_t)D * es; g.b_type = p.act; g.b_rs = K2; g.b_cs = 1;
      g.epi_mode = EPI_RK;
      g.kclass = KC_GEMM_OUT;
      g.epi.alpha = p.scaler;
      g.epi.c_new = 1.f;
      g.epi.out = tmp;
      g.epi.ld_out = D;
      g.epi.drop = make_drop(p, DS_MLP_OUT, e);
      ODV_TRY(gemm(p, g, s));
    }
    {
      GemmArgs g;
      g.M = p.M; g.N = D; g.K = D;
      g.A = c.oh; g.a_type = p.act; g.a_rs = K2; g.a_cs = 1;
      g.B = wb.w2cat; g.b_type = p.act; g.b_rs = K2; g.b_cs = 1;
      g.epi_mode = EPI_RK;
      g.kclass = KC_GEMM_OUT;
      g.epi = *rk;
      g.epi.bias = wb.b2;
      g.epi.alpha = p.scaler;
      g.epi.ld_out = D;
      g.epi.drop = make_drop(p, DS_PROJ, e);
      g.epi.resid = tmp; g.epi.resid_coef = 1.f;
      ODV_TRY(gemm(p, g, s));
    }
  } else if (rk) {
    GemmArgs g;
    g.M = p.M; g.N = D; g.K = K2;
    g.A = c.oh; g.a_type = p.act; g.a_rs = K2; g.a_cs = 1;
    g.B = wb.w2cat; g.b_type = p.act; g.b_rs = K2; g.b_cs = 1;
    g.epi_mode = EPI_RK;
    g.kclass = KC_GEMM_OUT;
    g.epi = *rk;
    g.epi.bias = wb.b2;
    g.epi.alpha = p.scaler;
    g.epi.ld_out = D;
    ODV_TRY(gemm(p, g, s));
  }
  return 0;
}

Epi rk_epilogue(const Tableau& tb, int st, float dt, const float* y, float* const* k, float* out) {
  Epi e;
  e.out = out;
  e.y = y;
  e.y_coef = 1.f;
  const bool last = (st == tb.S - 1);
  const float* row = last ? tb.b : tb.a[st + 1];
  e.c_new = dt * row[st];
  for (int l = 0; l < st; ++l) {
    if (row[l] != 0.f) { e.kin[l] = k[l]; e.c_k[l] = dt * row[l]; }
  }
  e.k_store = last ? nullptr : k[st];
  return e;
}

Epi rk_vjp_epilogue(const Tableau& tb, int m, float dt, const double* row_dt, int rows_per_image, const float* G,
                    float* const* mu, const float* g_t) {
  const int t = m - 1;
  const float h = row_dt ? 1.f : dt;
  Epi e;
  e.k_store = mu[m];
  e.c_new = h * tb.a[m][t];
  int n = 0;
  for (int l = m + 1; l < tb.S; ++l)
    if (tb.a[l][t] != 0.f) { e.kin[n] = mu[l]; e.c_k[n] = h * tb.a[l][t]; ++n; }
  // The branch follows the epilogue's arithmetic, not the caller: EPI_ROWDT scales every term by the image's step
  // except y, so y carries the unscaled g_t (or G with coefficient 0 where there is none) and G joins the kin terms.
  // A scalar dt is folded into the coefficients and G takes the y slot.
  if (row_dt) {
    e.row_dt = row_dt; e.rows_per_image = rows_per_image;
    if (tb.b[t] != 0.f) { e.kin[n] = G; e.c_k[n] = tb.b[t]; }
    e.y = g_t ? g_t : G; e.y_coef = g_t ? 1.f : 0.f;
  } else {
    e.y = G; e.y_coef = dt * tb.b[t];
  }
  return e;
}

Epi rk_vjp_row_epilogue(const float* G, float* const* mu, int n_mu, const float* const* rows, int n_rows, float* out) {
  Epi e;
  e.y = G; e.y_coef = 1.f; e.c_new = 1.f;
  int n = 0;
  for (int m = 1; m <= n_mu; ++m) { e.kin[n] = mu[m]; e.c_k[n] = 1.f; ++n; }
  for (int i = 0; i < n_rows; ++i) { e.kin[n] = rows[i]; e.c_k[n] = 1.f; ++n; }
  e.out = out;
  return e;
}

// What one forward evaluation of a fixed-grid step keeps besides its stage combine: its intermediates (a tape slot or
// the workspace's context) and, when wanted, its attention map and JaSMin statistic.
struct EvalOut {
  StageCtx ctx;
  float* p_copy = nullptr;
  float* jas_out = nullptr;
  int jas_k = 0;
};

// The S stages of step j from row y with step dt: evaluation e = j*S + st (the dropout masks are keyed by it).  Stage 0
// reads y, the later stages the stage buffer b.u; the epilogues (rk_epilogue) form each next stage input in b.u and the
// step result in y_next.  out(e, st) gives each evaluation's EvalOut.  With fd_prev and fd_out, the last stage also folds
// the finite-difference maxima of (fd_prev, y, y_next) into fd_out.  y_next == nullptr recomputes the intermediates
// only: the last stage runs without its output GEMM.
template <class Bufs, class Out>
int rk_step(const Plan& p, const Bufs& b, const Tableau& tb, int j, float dt, const float* y, float* y_next,
            const float* fd_prev, float* fd_out, Out out, cudaStream_t s) {
  for (int st = 0; st < tb.S; ++st) {
    const long long e = (long long)j * tb.S + st;
    const bool last = (st == tb.S - 1);
    const EvalOut o = out(e, st);
    Epi rk = rk_epilogue(tb, st, dt, y, b.k, last ? y_next : b.u);
    if (last && fd_prev && fd_out) { rk.fd_prev = fd_prev; rk.fd_out = fd_out; }
    const Epi* epi = (last && !y_next) ? nullptr : &rk;
    ODV_TRY(eval_forward(p, b.w, o.ctx, st == 0 ? y : b.u, b.P, o.p_copy, b.sq, b.tmp, e, epi, s, o.jas_out, o.jas_k));
  }
  return 0;
}

// VJP of one field evaluation: given dd = scaler * lambda (cotangent of the pre-scaler output, in
// the activation type) and the stage intermediates `c`, accumulate G1, c1, G2, c2 and deliver
// mu = J(u)^T lambda = centre_D(dz @ W1cat) through `mu_epi`, the EPI_RK epilogue of the last GEMM
// (W1cat^T is stored row-centred, so the GEMM yields the centred value directly; the reverse-mode
// stage combination rides in that epilogue instead of a separate pass over [M, D]).
int eval_vjp(const Plan& p, const WeightBufs& wb, const StageCtx& c, BwdBufs& b, const float* g_p,
             bool need_c2, const odevit_weight_grads* gw, long long ev, const Epi& mu_epi, cudaStream_t s) {
  if (p.variant == ODEVIT_FIELD_MACARON) {
    if (g_p) return set_error(ODEVIT_ERR_UNSUPPORTED, "MACARON has no attention-map output (macaron.py:60-65)");
    return macaron_vjp(p, wb, c, b, gw, mu_epi, ev, s);
  }
  const int D = p.D, hid = p.hid, R = 3 * D + hid, K2 = D + hid;
  const size_t e = dtype_size(p.act);
  char* dz = reinterpret_cast<char*>(b.dz);
  // (softmax attention, no attention-map dropout, the single-GEMM form of d[O|h]: see below)
  // (the deterministic mode sums every bias-gradient block in colsum_accum, which adds its partials in a fixed order)
  bool fused_colsum = p.variant == ODEVIT_FIELD_PARALLEL && p.p_attn == 0.f && !p.split_out && !deterministic();
  if (p.split_out) {
    // the cotangent enters the out-proj branch under the proj mask and the fc2 branch under the mlp-output mask
    if (gw->fc2_b) return set_error(ODEVIT_ERR_UNSUPPORTED, "dropout with an fc2 bias is not built (the reference has none)");
    ODV_TRY(drop_pair_rows(b.dd, b.dd1, b.dd2, p.act, make_drop(p, DS_MLP_OUT, ev), make_drop(p, DS_PROJ, ev), p.M, D, s));
    const char* w2T = reinterpret_cast<const char*>(wb.w2catT);
    {  // dO = dd2 @ Wo
      GemmArgs g;
      g.M = p.M; g.N = D; g.K = D;
      g.A = b.dd2; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
      g.B = w2T; g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
      g.epi_mode = EPI_STORE;
      g.kclass = KC_BWD_GEMM_DOH;
      g.epi.out = b.dO; g.epi.out_type = p.act; g.epi.ld_out = D;
      ODV_TRY(gemm(p, g, s));
    }
    {  // d h_pre = (dd1 @ W2) o mask_h o GELU'
      GemmArgs g;
      g.M = p.M; g.N = hid; g.K = D;
      g.A = b.dd1; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
      g.B = w2T + (size_t)D * D * e; g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
      g.epi_mode = EPI_BWD3;
      g.kclass = KC_BWD_GEMM_DOH;
      g.epi.split = 0;
      g.epi.out2 = dz + (size_t)3 * D * e; g.epi.ld_out2 = R;
      g.epi.aux = c.hpre; g.epi.ld_aux = hid; g.epi.aux_type = p.act;
      g.epi.aux_gelu_grad = true;
      g.epi.drop = make_drop(p, DS_MLP_H, ev);
      ODV_TRY(gemm(p, g, s));
    }
    {  // G2[:, :D] += dd2^T O
      GemmArgs g;
      g.M = D; g.N = D; g.K = p.M;
      g.A = b.dd2; g.a_type = p.act; g.a_rs = 1; g.a_cs = D;
      g.B = c.oh; g.b_type = p.act; g.b_rs = 1; g.b_cs = K2;
      g.epi_mode = EPI_ACCUM;
      g.epi.out = b.G2; g.epi.ld_out = K2;
      g.kclass = KC_BWD_GEMM_G2;
      ODV_TRY(gemm(p, g, s));
    }
    {  // G2[:, D:] += dd1^T h   (h as the forward left it: after its dropout)
      GemmArgs g;
      g.M = D; g.N = hid; g.K = p.M;
      g.A = b.dd1; g.a_type = p.act; g.a_rs = 1; g.a_cs = D;
      g.B = reinterpret_cast<const char*>(c.oh) + (size_t)D * e; g.b_type = p.act; g.b_rs = 1; g.b_cs = K2;
      g.epi_mode = EPI_ACCUM;
      g.epi.out = b.G2 + D; g.epi.ld_out = K2;
      g.kclass = KC_BWD_GEMM_G2;
      ODV_TRY(gemm(p, g, s));
    }
    if (need_c2) ODV_TRY(colsum_accum(b.dd2, p.act, D, p.M, D, b.c2, s, p.det_ws));
  } else {
  {  // d[O|h] = dd @ [Wo|W2];  GELU' on the h half
    GemmArgs g;
    g.M = p.M; g.N = K2; g.K = D;
    g.A = b.dd; g.a_type = p.act; g.a_rs = D; g.a_cs = 1;
    g.B = wb.w2catT; g.b_type = p.act; g.b_rs = D; g.b_cs = 1;
    g.epi_mode = EPI_BWD3;
    g.kclass = KC_BWD_GEMM_DOH;
    g.epi.out = b.dO; g.epi.out_type = p.act; g.epi.ld_out = D;
    g.epi.split = D;
    g.epi.out2 = dz + (size_t)3 * D * e; g.epi.ld_out2 = R;
    g.epi.aux = c.hpre; g.epi.ld_aux = hid; g.epi.aux_type = p.act;
    g.epi.aux_gelu_grad = true;
    // Bias-gradient column sums without a pass over dz (81 MB at the bench shape).  Softmax attention without map
    // dropout gives two of the four blocks for free:  sum_j dK_j = sum_i q_i (sum_j dS_ij) = 0  (rows of the softmax
    // Jacobian sum to zero) and  sum_j dV_j = sum_i (sum_j P_ij) dO_i = sum_i dO_i;  dO and d h_pre are summed in the
    // epilogue that produces them, and only the dq block is left for colsum_accum below.
    if (fused_colsum) {
      g.epi.colsum_a = b.c1 + 2 * D;   // the v rows of c1
      g.epi.colsum_b = b.c1 + 3 * D;   // the fc1 rows of c1
      if (!(p.precision == ODEVIT_BF16 && gemm_tc_supports(g))) { g.epi.colsum_a = g.epi.colsum_b = nullptr; fused_colsum = false; }
    }
    ODV_TRY(gemm(p, g, s));
  }
  {  // G2 += dd^T @ [O|h]
    GemmArgs g;
    g.M = D; g.N = K2; g.K = p.M;
    g.A = b.dd; g.a_type = p.act; g.a_rs = 1; g.a_cs = D;
    g.B = c.oh; g.b_type = p.act; g.b_rs = 1; g.b_cs = K2;
    g.epi_mode = EPI_ACCUM;
    g.epi.out = b.G2; g.epi.ld_out = K2;
    g.kclass = KC_BWD_GEMM_G2;
    ODV_TRY(gemm(p, g, s));
  }
  if (need_c2) ODV_TRY(colsum_accum(b.dd, p.act, D, p.M, D, b.c2, s, p.det_ws));
  }

  // ---- attention VJP per (image, head) ----------------------------------------------------------
  bool dq_colsum_done = false;   // the fused attention VJP sums the dq block on its way out
  ODV_TRY(attention_vjp(p, c.qkv, c.oh, K2, c.lse, b, g_p, b.dz, R, make_drop(p, DS_ATTN, ev), s, fused_colsum ? b.c1 : nullptr,
                        &dq_colsum_done));
  {  // mu = dz @ centred(W1cat), consumed by the caller's stage-combine epilogue
    GemmArgs g;
    g.M = p.M; g.N = D; g.K = R;
    g.A = b.dz; g.a_type = p.act; g.a_rs = R; g.a_cs = 1;
    g.B = wb.w1catT; g.b_type = p.act; g.b_rs = R; g.b_cs = 1;
    g.epi_mode = EPI_RK;
    g.epi = mu_epi;
    g.epi.alpha = 1.f;
    g.epi.bias = nullptr;
    g.epi.ld_out = D;
    g.epi.aux_type = p.dd_type;
    g.kclass = KC_BWD_GEMM_DX;
    ODV_TRY(gemm(p, g, s));
  }
  {  // G1 += dz^T @ xc
    GemmArgs g;
    g.M = R; g.N = D; g.K = p.M;
    g.A = b.dz; g.a_type = p.act; g.a_rs = 1; g.a_cs = R;
    g.B = c.xc; g.b_type = p.act; g.b_rs = 1; g.b_cs = D;
    g.epi_mode = EPI_ACCUM;
    g.epi.out = b.G1; g.epi.ld_out = D;
    g.kclass = KC_BWD_GEMM_G1;
    ODV_TRY(gemm(p, g, s));
  }
  if (!fused_colsum) ODV_TRY(colsum_accum(b.dz, p.act, R, p.M, R, b.c1, s, p.det_ws));
  else if (!dq_colsum_done) ODV_TRY(colsum_accum(b.dz, p.act, R, p.M, D, b.c1, s, p.det_ws));     // the dq block only
  return 0;
}

int rk_step_vjp(const Plan& p, BwdBufs& b, const Tableau& tb, float dt, const double* row_dt, const float* const* g,
                float* const* mu, const StageCtx* ctx, long long e0, const float* g_p, bool need_c2,
                const odevit_weight_grads* gw, Epi row_epi, cudaStream_t s) {
  for (int m = tb.S - 1; m >= 1; --m) {
    Epi e = rk_vjp_epilogue(tb, m, dt, row_dt, p.N, b.gy, mu, g ? g[m - 1] : nullptr);
    e.aux_type = p.dd_type;
    e.out2 = b.dd; e.out2_scale = p.scaler;
    ODV_TRY(eval_vjp(p, b.w, ctx[m], b, m == tb.S - 1 ? g_p : nullptr, need_c2, gw, e0 + m, e, s));
  }
  row_epi.aux_type = p.dd_type;
  return eval_vjp(p, b.w, ctx[0], b, tb.S == 1 ? g_p : nullptr, need_c2, gw, e0, row_epi, s);
}

int finish_grads(const Plan& p, const odevit_weights* w, const odevit_weight_grads* gw, const BwdBufs& b,
                 cudaStream_t s) {
  UnfoldArgs u;
  u.D = p.D; u.hid = p.hid; u.heads = p.H; u.w = w; u.gw = gw;
  u.G1 = b.G1; u.c1 = b.c1; u.G2 = b.G2; u.c2 = b.c2;
  u.q_scale = q_scale_of(p);
  u.part = p.det_ws;
  if (p.variant == ODEVIT_FIELD_MACARON) {
    u.c3 = b.c3;
    return unfold_grads_macaron(u, s);
  }
  return unfold_grads_parallel(u, s);
}

bool wants_c2(const odevit_weight_grads* gw) { return gw && (gw->out_proj_b || gw->fc2_b); }

}  // namespace odevit

// ================================================================================================
// C ABI
// ================================================================================================
using namespace odevit;

extern "C" {

int odevit_abi_version(void) { return ODEVIT_ABI_VERSION; }

const char* odevit_build_info(void) {
  return "libodevit sm_100a (nvcc " ODEVIT_STR(__CUDACC_VER_MAJOR__) "." ODEVIT_STR(__CUDACC_VER_MINOR__) ", " __DATE__ ")";
}

const char* odevit_last_error_string(void) { return g_err; }

int odevit_drop_state_advance(uint64_t* state, odevit_stream_t stream) {
  ODV_TRY(check_device_ptr(state, "state"));
  return drop_state_advance(reinterpret_cast<unsigned long long*>(state), reinterpret_cast<cudaStream_t>(stream));
}

int64_t odevit_launch_count(void) { return g_launches.load(); }

int odevit_set_deterministic(int32_t on) {
  g_deterministic.store(on ? 1 : 0);
  return 0;
}
int32_t odevit_deterministic(void) { return g_deterministic.load(); }
void odevit_reset_launch_count(void) { g_launches.store(0); }

int odevit_gemm_bf16(int32_t M, int32_t N, int32_t K, int32_t mn_major, const void* A, const void* B, float* C,
                     int32_t accumulate, int32_t engine, odevit_stream_t stream) {
  ODV_TRY(check_device_ptr(A, "A"));
  ODV_TRY(check_device_ptr(B, "B"));
  ODV_TRY(check_device_ptr(C, "C"));
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.a_type = DT_BF16;
  g.B = B; g.b_type = DT_BF16;
  if (mn_major) { g.a_rs = 1; g.a_cs = M; g.b_rs = 1; g.b_cs = N; }
  else { g.a_rs = K; g.a_cs = 1; g.b_rs = K; g.b_cs = 1; }
  g.epi_mode = accumulate ? EPI_ACCUM : EPI_STORE;
  g.epi.out = C; g.epi.out_type = DT_F32; g.epi.ld_out = N;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (engine == 1) return gemm_tc(g, s);
  return gemm_simt(g, s);
}

int odevit_profile_enable(int32_t on) {
  ProfState& p = g_prof;
  std::lock_guard<std::mutex> lock(p.mu);
  if (on) {
    if (!p.ev) {
      p.ev = new cudaEvent_t[2 * kMaxProfPairs];
      p.cls = new int[kMaxProfPairs];
      p.cap = 0;
    }
    p.used = 0;
    p.on = true;
  } else {
    p.on = false;
  }
  return 0;
}
int odevit_profile_reserve(int32_t pairs) {
  // create the event pairs up front, so that cudaEventCreate never lands inside a timed region
  ProfState& p = g_prof;
  std::lock_guard<std::mutex> lock(p.mu);
  if (!p.ev) {
    p.ev = new cudaEvent_t[2 * kMaxProfPairs];
    p.cls = new int[kMaxProfPairs];
    p.cap = 0;
  }
  if (pairs > kMaxProfPairs) pairs = kMaxProfPairs;
  while (p.cap < pairs) {
    if (cudaEventCreate(&p.ev[2 * p.cap]) != cudaSuccess || cudaEventCreate(&p.ev[2 * p.cap + 1]) != cudaSuccess)
      return set_error(ODEVIT_ERR_CUDA, "odevit_profile_reserve: cudaEventCreate failed at pair %d", p.cap);
    ++p.cap;
  }
  return 0;
}
int odevit_profile_num_classes(void) { return KC_COUNT; }
const char* odevit_profile_class_name(int32_t k) { return (k >= 0 && k < KC_COUNT) ? kClassNames[k] : "?"; }
int odevit_profile_read(int32_t kclass, double* total_ms, int64_t* launches) {
  ProfState& p = g_prof;
  if (kclass < 0 || kclass >= KC_COUNT || !total_ms || !launches)
    return set_error(ODEVIT_ERR_INVALID_ARG, "odevit_profile_read: bad arguments");
  double t = 0;
  int64_t n = 0;
  for (int i = 0; i < p.used; ++i) {
    if (p.cls[i] != kclass) continue;
    float ms = 0.f;
    ODV_CUDA(cudaEventSynchronize(p.ev[2 * i + 1]));
    ODV_CUDA(cudaEventElapsedTime(&ms, p.ev[2 * i], p.ev[2 * i + 1]));
    t += ms;
    ++n;
  }
  *total_ms = t;
  *launches = n;
  return 0;
}

// ---- encoder stack (the distillation teacher): workspace and prepared-weight cache layouts ----
namespace odevit {
namespace {
struct EncBufs {
  StageCtx ctx;
  float* P;
};
EncBufs layout_encoder(const Plan& p, Arena& a) {
  const size_t e = dtype_size(p.act);
  const size_t MD = (size_t)p.M * p.D, Mh = (size_t)p.M * p.hid;
  EncBufs b{};
  b.ctx.xc = a.take(MD * e);
  b.ctx.qkv = a.take(3 * MD * e);
  b.ctx.oh = a.take((MD + Mh) * e);
  b.ctx.x1 = a.f32(MD);
  b.P = a.f32((size_t)p.BHNN);
  return b;
}
// activation-typed [3D+hid, D] and [D, D+hid] blocks + fp32 biases per layer, no transposes (forward only)
WeightBufs take_encoder_weights(const Plan& p, Arena& a) {
  const size_t e = dtype_size(p.act);
  const size_t R = 3 * (size_t)p.D + p.hid, K2 = (size_t)p.D + p.hid;
  WeightBufs w{};
  w.w1cat = a.take(R * p.D * e);
  w.w2cat = a.take(K2 * p.D * e);
  w.b1cat = a.f32(R);
  w.b2 = a.f32(p.D);
  return w;
}
int encoder_plan(const odevit_desc* desc, Plan* p) {
  ODV_TRY(make_plan(desc, p));
  p->variant = ODEVIT_FIELD_MACARON;   // the four weight blocks unfolded, biases on
  p->dd_type = DT_F32;
  if (p->any_drop) return set_error(ODEVIT_ERR_UNSUPPORTED, "the encoder stack is inference-only: dropout must be 0");
  p->split_out = false;
  return 0;
}
}  // namespace
}  // namespace odevit

size_t odevit_workspace_bytes(const odevit_desc* desc, int32_t ws_kind, int32_t method) {
  Plan p{};
  if (make_plan(desc, &p)) return 0;
  Arena a(nullptr);
  if (ws_kind == ODEVIT_WS_FIELD) {
    layout_fwd(p, a, 1);
  } else if (ws_kind == ODEVIT_WS_ENCODER_FWD) {
    if (encoder_plan(desc, &p)) return 0;
    layout_encoder(p, a);
  } else if (ws_kind == ODEVIT_WS_SOLVE_ADAPTIVE) {
    a.off = solve_adaptive_workspace_bytes(p);
  } else if (ws_kind == ODEVIT_WS_SOLVE_ADAPTIVE_BWD) {
    a.off = solve_adaptive_bwd_workspace_bytes(p);
  } else if (ws_kind == ODEVIT_WS_SOLVE_ADAPTIVE_RESIDENT) {
    a.off = solve_adaptive_resident_workspace_bytes(p);
  } else {
    const Tableau* tb = tableau_for(method);
    if (!tb) { set_error(ODEVIT_ERR_INVALID_ARG, "unknown method %d", method); return 0; }
    if (ws_kind == ODEVIT_WS_SOLVE_FWD) layout_fwd(p, a, tb->S);
    else if (ws_kind == ODEVIT_WS_SOLVE_BWD) layout_bwd(p, a, tb->S);
    else { set_error(ODEVIT_ERR_INVALID_ARG, "unknown workspace kind %d", ws_kind); return 0; }
  }
  return a.off + 1024;
}

size_t odevit_tape_bytes(const odevit_desc* desc, int32_t method, int32_t n_grid) {
  Plan p{};
  if (make_plan(desc, &p)) return 0;
  const Tableau* tb = tableau_for(method);
  if (!tb || n_grid < 1) { set_error(ODEVIT_ERR_INVALID_ARG, "unknown method %d / empty grid", method); return 0; }
  return tape_bytes(p, (long long)(n_grid - 1) * tb->S);
}

int odevit_field_fwd(const odevit_desc* desc, const odevit_weights* w, const float* x, float* dx,
                     float* p_out, void* workspace, size_t workspace_bytes, odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  ODV_TRY(check_device_ptr(x, "x"));
  ODV_TRY(check_device_ptr(dx, "dx"));
  if (x == dx) return set_error(ODEVIT_ERR_INVALID_ARG, "x and dx may not alias");
  if (p.variant == ODEVIT_FIELD_MACARON && p_out)
    return set_error(ODEVIT_ERR_INVALID_ARG, "MACARON exposes no attention map (need_weights=False, macaron.py:60-65)");
  Arena a(workspace);
  FwdBufs f = layout_fwd(p, a, 1);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  ODV_TRY(prepare_drop_keys(p, f.drop_keys, 1, s));
  ODV_TRY(prepare_weights(p, w, f.w, s));
  Epi rk;
  rk.out = dx;
  rk.y = nullptr;
  rk.c_new = 1.f;
  return eval_forward(p, f.w, f.ctx, x, f.P, p_out, f.sq, f.tmp, 0, &rk, s);
}

namespace {
// Trajectory-free outputs (odevit_solve_fwd_lean): selected trajectory rows and the finite-difference maxima.
struct LeanOut {
  float* rows_out;
  const int32_t* row_index;
  int n_rows;
  float* fd_max;
};

// The fixed-grid forward solve.  lean == nullptr: the trajectory into `states` and, when given, a tape for the reverse
// sweep.  Otherwise trajectory-free: the rows live in a ring of three (the finite-difference window), in the caller's
// slots of `rows_out` when they are control points, in `final_state` when last.
int solve_fwd_impl(const odevit_desc* desc, const odevit_weights* w, int32_t method, const float* x0,
                   const float* t_grid_host, int32_t n_grid, float* states, float* final_state,
                   float* p_last, float* p_traj, int32_t p_traj_first_eval, float* jas_traj,
                   int32_t jas_first_eval, int32_t jas_k, void* tape, size_t tape_bytes,
                   void* workspace, size_t workspace_bytes, odevit_stream_t stream, const LeanOut* lean) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  if (jas_traj) {
    ODV_TRY(check_device_ptr(jas_traj, "jas_traj"));
    if (jas_k < 0 || jas_k > p.N || jas_first_eval < 0)
      return set_error(ODEVIT_ERR_INVALID_ARG, "jas_k %d / jas_first_eval %d out of range", jas_k, jas_first_eval);
    if (p.variant == ODEVIT_FIELD_MACARON) return set_error(ODEVIT_ERR_UNSUPPORTED, "MACARON has no attention-map output");
  }
  const Tableau* tb = tableau_for(method);
  if (!tb) return set_error(ODEVIT_ERR_INVALID_ARG, "unknown method %d", method);
  if (!t_grid_host || n_grid < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "t_grid must hold >= 1 point");
  const long long n_evals = (long long)(n_grid - 1) * tb->S;
  if (tape) ODV_TRY(check_tape(p, tape, tape_bytes, n_evals));
  if (!states && !final_state) return set_error(ODEVIT_ERR_INVALID_ARG, "states and final_state both NULL");
  if (p.variant == ODEVIT_FIELD_MACARON && (p_last || p_traj))
    return set_error(ODEVIT_ERR_INVALID_ARG, "MACARON exposes no attention map (need_weights=False, macaron.py:60-65)");
  ODV_TRY(check_device_ptr(x0, "x0"));
  if (states) ODV_TRY(check_device_ptr(states, "states"));
  for (int j = 0; j + 2 < n_grid; ++j) {
    const float d0 = t_grid_host[j + 1] - t_grid_host[j], d1 = t_grid_host[j + 2] - t_grid_host[j + 1];
    if (!(d0 * d1 > 0.f)) return set_error(ODEVIT_ERR_INVALID_ARG, "t must be strictly increasing or decreasing");
  }
  if (n_grid == 2 && t_grid_host[1] == t_grid_host[0])
    return set_error(ODEVIT_ERR_INVALID_ARG, "t must be strictly increasing or decreasing");
  if (lean && (states || tape)) return set_error(ODEVIT_ERR_INVALID_ARG, "the trajectory-free solve keeps neither states nor a tape");
  const LeanOut lo = lean ? *lean : LeanOut{nullptr, nullptr, 0, nullptr};
  for (int i = 0; i < lo.n_rows; ++i)
    if (lo.row_index[i] < 0 || lo.row_index[i] >= n_grid)
      return set_error(ODEVIT_ERR_INVALID_ARG, "row_index[%d]=%d outside [0,%d)", i, lo.row_index[i], n_grid);
  Arena a(workspace);
  FwdBufs f = layout_fwd(p, a, tb->S);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t MD = (size_t)p.M * p.D;
  ODV_TRY(prepare_drop_keys(p, f.drop_keys, n_evals, s));
  if (tape) f.w = tape_weights(p, tape, n_evals);   // fold once per step: the reverse sweep reuses them
  ODV_TRY(prepare_weights(p, w, f.w, s));

  const float* y = x0;   // row j
  if (states) {
    ODV_CUDA(cudaMemcpyAsync(states, x0, MD * 4, cudaMemcpyDeviceToDevice, s));
    y = states;
  }
  // small-token shapes: the whole solve of an image in one persistent CTA, state resident on the chip.  It writes
  // neither rows_out nor fd_max, so the trajectory-free mode never takes it.
  if (!lean && solve_resident_supports(p, n_grid, p_traj != nullptr || jas_traj != nullptr, tape != nullptr) &&
      (tb->S == 1 || f.kbuf))
    return solve_resident(p, f.w, *tb, x0, t_grid_host, n_grid, states, final_state, p_last, f.kbuf, s);

  if (lo.fd_max) ODV_CUDA(cudaMemsetAsync(lo.fd_max, 0, (size_t)p.M * 4, s));
  auto next_row = [&](int j) -> float* {   // where row j + 1 goes
    if (states) return states + (size_t)(j + 1) * MD;
    for (int i = 0; i < lo.n_rows; ++i)    // the first caller slot that names it
      if (lo.row_index[i] == j + 1) return lo.rows_out + (size_t)i * MD;
    if (j + 2 == n_grid && final_state) return final_state;
    return f.ytmp[(j + 1) % 3];            // rows j - 1 and j stay readable
  };
  auto fan_out = [&](int j, const float* src) -> int {   // row j into every further slot that names it
    bool first = true;
    for (int i = 0; i < lo.n_rows; ++i) {
      if (lo.row_index[i] != j) continue;
      float* dst = lo.rows_out + (size_t)i * MD;
      if (first && dst == src) { first = false; continue; }
      first = false;
      ODV_CUDA(cudaMemcpyAsync(dst, src, MD * 4, cudaMemcpyDeviceToDevice, s));
    }
    return 0;
  };
  auto p_slot = [&](long long e) -> float* {   // where the attention map of evaluation e goes
    if (p_traj && e >= p_traj_first_eval) return p_traj + (size_t)(e - p_traj_first_eval) * p.BHNN;
    return (p_last && e == n_evals - 1) ? p_last : nullptr;
  };
  auto out = [&](long long e, int) {
    EvalOut o;
    o.ctx = tape ? tape_ctx(p, tape, e) : f.ctx;
    o.p_copy = p_slot(e);
    if (jas_traj && e >= jas_first_eval) o.jas_out = jas_traj + (size_t)(e - jas_first_eval) * p.B * p.H;
    o.jas_k = jas_k;
    return o;
  };
  ODV_TRY(fan_out(0, x0));
  const float* y_prev = nullptr;   // row j - 1
  for (int j = 0; j + 1 < n_grid; ++j) {
    float* y_next = next_row(j);
    ODV_TRY(rk_step(p, f, *tb, j, t_grid_host[j + 1] - t_grid_host[j], y, y_next, y_prev, lo.fd_max, out, s));
    ODV_TRY(fan_out(j + 1, y_next));
    y_prev = y;
    y = y_next;
  }
  if (p_last && n_evals > 0 && p_slot(n_evals - 1) != p_last)   // p_traj holds the last evaluation's map
    ODV_CUDA(cudaMemcpyAsync(p_last, p_slot(n_evals - 1), (size_t)p.BHNN * 4, cudaMemcpyDeviceToDevice, s));
  if (final_state && y != final_state) ODV_CUDA(cudaMemcpyAsync(final_state, y, MD * 4, cudaMemcpyDeviceToDevice, s));
  return 0;
}
}  // namespace

int odevit_solve_fwd(const odevit_desc* desc, const odevit_weights* w, int32_t method, const float* x0,
                     const float* t_grid_host, int32_t n_grid, float* states, float* final_state,
                     float* p_last, float* p_traj, int32_t p_traj_first_eval, float* jas_traj,
                     int32_t jas_first_eval, int32_t jas_k, void* tape, size_t tape_bytes,
                     void* workspace, size_t workspace_bytes, odevit_stream_t stream) {
  return solve_fwd_impl(desc, w, method, x0, t_grid_host, n_grid, states, final_state, p_last, p_traj, p_traj_first_eval,
                        jas_traj, jas_first_eval, jas_k, tape, tape_bytes, workspace, workspace_bytes, stream, nullptr);
}

int odevit_solve_fwd_lean(const odevit_desc* desc, const odevit_weights* w, int32_t method, const float* x0,
                          const float* t_grid_host, int32_t n_grid, float* final_state, float* rows_out,
                          const int32_t* row_index_host, int32_t n_rows, float* fd_max, float* p_last,
                          float* jas_traj, int32_t jas_first_eval, int32_t jas_k, void* workspace,
                          size_t workspace_bytes, odevit_stream_t stream) {
  if (!final_state) return set_error(ODEVIT_ERR_INVALID_ARG, "final_state is NULL");
  if (n_rows < 0 || (n_rows > 0 && (!rows_out || !row_index_host)))
    return set_error(ODEVIT_ERR_INVALID_ARG, "rows_out / row_index_host missing");
  if (rows_out) ODV_TRY(check_device_ptr(rows_out, "rows_out"));
  if (fd_max) ODV_TRY(check_device_ptr(fd_max, "fd_max"));
  const LeanOut lean{rows_out, row_index_host, n_rows, fd_max};
  return solve_fwd_impl(desc, w, method, x0, t_grid_host, n_grid, nullptr, final_state, p_last, nullptr, 0, jas_traj,
                        jas_first_eval, jas_k, nullptr, 0, workspace, workspace_bytes, stream, &lean);
}

int odevit_solve_uses_resident(const odevit_desc* desc, int32_t method, int32_t n_grid) {
  Plan p{};
  if (make_plan(desc, &p) != 0) return 0;
  const Tableau* tb = tableau_for(method);
  if (!tb) return 0;
  return solve_resident_supports(p, n_grid, false, false) ? 1 : 0;
}

int odevit_solve_bwd(const odevit_desc* desc, const odevit_weights* w, int32_t method,
                     const float* t_grid_host, int32_t n_grid, const float* states, const float* g_states,
                     const float* g_rows, const int32_t* g_row_index_host, int32_t n_g_rows,
                     const float* g_p_last, float* g_x0, const odevit_weight_grads* gw, const void* tape,
                     size_t tape_bytes, void* workspace, size_t workspace_bytes, odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  const Tableau* tb = tableau_for(method);
  if (!tb) return set_error(ODEVIT_ERR_INVALID_ARG, "unknown method %d", method);
  if (!t_grid_host || n_grid < 1) return set_error(ODEVIT_ERR_INVALID_ARG, "t_grid must hold >= 1 point");
  if (!gw) return set_error(ODEVIT_ERR_INVALID_ARG, "weight-gradient struct is NULL");
  ODV_TRY(check_device_ptr(states, "states"));
  ODV_TRY(check_device_ptr(g_x0, "g_x0"));
  if (n_g_rows > 0 && (!g_rows || !g_row_index_host))
    return set_error(ODEVIT_ERR_INVALID_ARG, "g_rows / g_row_index_host missing");
  for (int i = 0; i < n_g_rows; ++i)
    if (g_row_index_host[i] < 0 || g_row_index_host[i] >= n_grid)
      return set_error(ODEVIT_ERR_INVALID_ARG, "g_row_index[%d]=%d outside [0,%d)", i, g_row_index_host[i], n_grid);
  if (tape) ODV_TRY(check_tape(p, tape, tape_bytes, (long long)(n_grid - 1) * tb->S));
  Arena a(workspace);
  BwdBufs b = layout_bwd(p, a, tb->S);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t MD = (size_t)p.M * p.D;
  const int S = tb->S;
  const bool need_c2 = wants_c2(gw);
  ODV_TRY(prepare_drop_keys(p, b.drop_keys, (long long)(n_grid - 1) * S, s));
  if (tape) {   // the forward of this step left its folded weights behind the tape's slots
    b.w = tape_weights(p, tape, (long long)(n_grid - 1) * S);
    b.w.user = w;
  } else {
    ODV_TRY(prepare_weights(p, w, b.w, s));
  }
  ODV_CUDA(cudaMemsetAsync(b.G1, 0, b.acc_bytes, s));

  // cotangent of trajectory row j = g_states[j] + sum of g_rows whose index is j
  auto injected_terms = [&](int row, const float** out, int cap) -> int {
    int n = 0;
    if (g_states) { if (n < cap) out[n] = g_states + (size_t)row * MD; ++n; }
    for (int i = 0; i < n_g_rows; ++i)
      if (g_row_index_host[i] == row) { if (n < cap) out[n] = g_rows + (size_t)i * MD; ++n; }
    return n;
  };
  auto inject = [&](int row) -> int {
    if (g_states) ODV_TRY(axpy_f32(b.gy, g_states + (size_t)row * MD, 1.f, (long long)MD, s));
    for (int i = 0; i < n_g_rows; ++i)
      if (g_row_index_host[i] == row) ODV_TRY(axpy_f32(b.gy, g_rows + (size_t)i * MD, 1.f, (long long)MD, s));
    return 0;
  };
  // dd = scaler * dt * b[S-1] * G : the cotangent entering the last stage of a step
  auto seed_dd = [&](float dt) -> int {
    CombineArgs c0;
    c0.n_terms = 1; c0.term[0] = b.gy; c0.coef[0] = dt * tb->b[S - 1];
    c0.out_dd = b.dd; c0.dd_type = p.dd_type; c0.dd_scale = p.scaler;
    return vjp_combine(c0, p.M, p.D, s);
  };
  {
    // G = the cotangent injected at the last row, dd = scaler * dt * b[S-1] * G: one pass (it used to be a memset, an axpy
    // per term and a combine: 260 MB of traffic and four launches at the bench shape instead of 100 MB and one)
    const float* terms[4];
    const int nt_inj = injected_terms(n_grid - 1, terms, 4);
    if (nt_inj <= 4 && MD % 4 == 0) {
      const bool seed = n_grid >= 2;
      const float coef = seed ? p.scaler * (t_grid_host[n_grid - 1] - t_grid_host[n_grid - 2]) * tb->b[S - 1] : 0.f;
      ODV_TRY(seed_sweep(terms, nt_inj, b.gy, seed ? b.dd : nullptr, p.dd_type, coef, (long long)MD, s));
    } else {
      ODV_CUDA(cudaMemsetAsync(b.gy, 0, MD * 4, s));
      ODV_TRY(inject(n_grid - 1));
      if (n_grid >= 2) ODV_TRY(seed_dd(t_grid_host[n_grid - 1] - t_grid_host[n_grid - 2]));
    }
  }

  for (int j = n_grid - 2; j >= 0; --j) {
    const float dt = t_grid_host[j + 1] - t_grid_host[j];
    const float* y = states + (size_t)j * MD;
    // (1) the stage intermediates of this step: read back from the tape when the forward kept one,
    //     else recomputed from the trajectory row (the last stage skips GEMM2)
    StageCtx ctx[4];
    for (int st = 0; st < S; ++st)
      ctx[st] = tape ? tape_ctx(p, tape, (long long)j * S + st) : b.ctx[st];
    if (!tape)
      ODV_TRY(rk_step(p, b, *tb, j, dt, y, nullptr, nullptr, nullptr,
                      [&](long long, int st) { return EvalOut{b.ctx[st]}; }, s));
    // (2) reverse through the stages: G <- G + sum_st mu_st + the cotangents injected at row j, and the row epilogue
    //     seeds dd for step j-1 -- unless the terms overflow it: then the injection and the seed follow as passes
    const float* inj[Epi::kMaxTerms];
    const int n_inj = injected_terms(j, inj, Epi::kMaxTerms);
    const bool fits = (S - 1 + n_inj <= Epi::kMaxTerms);
    Epi row = rk_vjp_row_epilogue(b.gy, b.mu, S - 1, inj, fits ? n_inj : 0, b.gy);
    if (fits && j > 0) {
      row.out2 = b.dd;
      row.out2_scale = p.scaler * (t_grid_host[j] - t_grid_host[j - 1]) * tb->b[S - 1];
    }
    ODV_TRY(rk_step_vjp(p, b, *tb, dt, nullptr, nullptr, b.mu, ctx, (long long)j * S,
                        j == n_grid - 2 ? g_p_last : nullptr, need_c2, gw, row, s));
    if (!fits) ODV_TRY(inject(j));
    if (!fits && j > 0) ODV_TRY(seed_dd(t_grid_host[j] - t_grid_host[j - 1]));
  }
  ODV_CUDA(cudaMemcpyAsync(g_x0, b.gy, MD * 4, cudaMemcpyDeviceToDevice, s));
  return finish_grads(p, w, gw, b, s);
}

int odevit_fd_curvature(const float* states, int32_t n_grid, int32_t batch, int32_t tokens, int32_t dim,
                        double delta_t, float* per_seq, odevit_stream_t stream) {
  if (n_grid < 3) return set_error(ODEVIT_ERR_INVALID_ARG, "fd_curvature needs >= 3 grid points, got %d", n_grid);
  if (batch <= 0 || tokens <= 0 || dim <= 0) return set_error(ODEVIT_ERR_INVALID_ARG, "non-positive dimension");
  ODV_TRY(check_device_ptr(states, "states"));
  ODV_TRY(check_device_ptr(per_seq, "per_seq"));
  return fd_curvature(states, n_grid, (long long)batch * tokens, dim, (float)(delta_t * delta_t), per_seq,
                      reinterpret_cast<cudaStream_t>(stream));
}

size_t odevit_encoder_cache_bytes(const odevit_desc* desc, int32_t n_layers) {
  Plan p{};
  if (encoder_plan(desc, &p) || n_layers < 1) return 0;
  Arena a(nullptr);
  for (int l = 0; l < n_layers; ++l) take_encoder_weights(p, a);
  return a.off + 1024;
}

int odevit_encoder_fwd(const odevit_desc* desc, const odevit_weights* layers, int32_t n_layers, float ln_eps,
                       const float* x0, float* hidden, float* p_out, int32_t p_mode, void* wcache,
                       size_t wcache_bytes, int32_t wcache_valid, void* workspace, size_t workspace_bytes,
                       odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(encoder_plan(desc, &p));
  if (!layers || n_layers < 1 || n_layers > 64) return set_error(ODEVIT_ERR_INVALID_ARG, "encoder: 1 <= n_layers <= 64 and a layer array");
  if (p_mode < 0 || p_mode > 2) return set_error(ODEVIT_ERR_INVALID_ARG, "encoder: p_mode %d (0 none, 1 last layer, 2 all)", p_mode);
  if (p_mode && !p_out) return set_error(ODEVIT_ERR_INVALID_ARG, "encoder: p_mode %d without p_out", p_mode);
  ODV_TRY(check_device_ptr(x0, "x0"));
  ODV_TRY(check_device_ptr(hidden, "hidden"));
  if (p_out) ODV_TRY(check_device_ptr(p_out, "p_out"));
  for (int l = 0; l < n_layers; ++l) {
    const odevit_weights& w = layers[l];
    if (!w.norm_a_w || !w.norm_a_b || !w.norm_b_w || !w.norm_b_b || !w.in_proj_w || !w.in_proj_b || !w.out_proj_w ||
        !w.out_proj_b || !w.fc1_w || !w.fc1_b || !w.fc2_w || !w.fc2_b)
      return set_error(ODEVIT_ERR_INVALID_ARG, "encoder layer %d: norm_a, norm_b, in_proj, out_proj, fc1, fc2 with biases are required", l);
    ODV_TRY(check_device_ptr(w.in_proj_w, "layers[].in_proj_w"));
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  Arena ca(wcache);
  WeightBufs wbs[64];
  for (int l = 0; l < n_layers; ++l) {
    wbs[l] = take_encoder_weights(p, ca);
    wbs[l].user = &layers[l];
  }
  ODV_TRY(check_ws(wcache, wcache_bytes, ca.off));
  if (!wcache_valid)
    for (int l = 0; l < n_layers; ++l) ODV_TRY(prepare_weights(p, &layers[l], wbs[l], s));
  Arena a(workspace);
  EncBufs b = layout_encoder(p, a);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  return encoder_forward(p, wbs, n_layers, ln_eps, x0, hidden, p_out, p_mode, b.ctx, b.P, s);
}

int odevit_jasmin_rowmax(const float* p_maps, int64_t n_slices, int32_t tokens, int32_t k, float* out,
                         odevit_stream_t stream) {
  if (n_slices < 0 || tokens <= 0) return set_error(ODEVIT_ERR_INVALID_ARG, "non-positive dimension");
  if (n_slices == 0) return 0;
  ODV_TRY(check_device_ptr(p_maps, "p_maps"));
  ODV_TRY(check_device_ptr(out, "out"));
  return jasmin_rowmax(p_maps, n_slices, tokens, k, out, reinterpret_cast<cudaStream_t>(stream));
}

int odevit_tokens_fwd(const void* cols_bf16, const void* w_bf16, int32_t batch, int32_t patches, int32_t k, int32_t dim,
                      int32_t tokens, int32_t first_patch_row, const float* patch_add, const float* special_rows,
                      const int32_t* special_index, int32_t n_special, float* x0, odevit_stream_t stream) {
  if (batch <= 0 || patches <= 0 || k <= 0 || dim <= 0 || tokens < patches + n_special || first_patch_row < 0 ||
      first_patch_row + patches > tokens || n_special < 0)
    return set_error(ODEVIT_ERR_INVALID_ARG, "tokens_fwd: inconsistent sizes");
  ODV_TRY(check_device_ptr(cols_bf16, "cols"));
  ODV_TRY(check_device_ptr(w_bf16, "w"));
  ODV_TRY(check_device_ptr(patch_add, "patch_add"));
  ODV_TRY(check_device_ptr(x0, "x0"));
  if (n_special) {
    ODV_TRY(check_device_ptr(special_rows, "special_rows"));
    ODV_TRY(check_device_ptr(special_index, "special_index"));
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  GemmArgs g;
  g.M = batch * patches; g.N = dim; g.K = k;
  g.A = cols_bf16; g.a_type = DT_BF16; g.a_rs = k; g.a_cs = 1;
  g.B = w_bf16; g.b_type = DT_BF16; g.b_rs = k; g.b_cs = 1;
  g.epi_mode = EPI_TOKENS;
  g.kclass = KC_OTHER;
  g.epi.out = x0; g.epi.out_type = DT_F32; g.epi.ld_out = dim;
  g.epi.split = patches; g.epi.out_bo = (long long)tokens * dim; g.epi.out_bi = first_patch_row;
  g.epi.y = patch_add;
  if (gemm_tc_supports(g)) ODV_TRY(gemm_tc(g, s));
  else ODV_TRY(gemm_simt(g, s));
  return tokens_special_rows(special_rows, special_index, n_special, batch, tokens, dim, x0, s);
}

int odevit_head_ce_fwd(const float* x, int64_t x_stride, const float* w, const float* bias, const int64_t* labels,
                       int32_t batch, int32_t classes, int32_t dim, float label_smoothing, float* logits, float* loss_rows,
                       float* lse, odevit_stream_t stream) {
  if (batch <= 0 || classes <= 0 || dim <= 0) return set_error(ODEVIT_ERR_INVALID_ARG, "head_ce: non-positive dimension");
  if ((size_t)(dim + classes) * 4 > 48 * 1024) return set_error(ODEVIT_ERR_UNSUPPORTED, "head_ce: dim + classes > 12288 is not built");
  ODV_TRY(check_device_ptr(x, "x"));
  ODV_TRY(check_device_ptr(w, "w"));
  ODV_TRY(check_device_ptr(logits, "logits"));
  if (loss_rows) {
    ODV_TRY(check_device_ptr(labels, "labels"));
    ODV_TRY(check_device_ptr(loss_rows, "loss_rows"));
    ODV_TRY(check_device_ptr(lse, "lse"));
  }
  return head_ce_fwd(x, x_stride, w, bias, reinterpret_cast<const long long*>(labels), batch, classes, dim, label_smoothing,
                     logits, loss_rows, lse, reinterpret_cast<cudaStream_t>(stream));
}

int odevit_head_ce_bwd(const float* x, int64_t x_stride, const float* w, const int64_t* labels, const float* logits,
                       const float* lse, const float* g_logits, const float* g_loss, int32_t batch, int32_t classes,
                       int32_t dim, float label_smoothing, float* dz, float* g_x, int64_t gx_stride, float* g_w, float* g_bias,
                       odevit_stream_t stream) {
  if (batch <= 0 || classes <= 0 || dim <= 0) return set_error(ODEVIT_ERR_INVALID_ARG, "head_ce: non-positive dimension");
  if ((size_t)classes * 4 > 48 * 1024) return set_error(ODEVIT_ERR_UNSUPPORTED, "head_ce: more than 12288 classes are not built");
  if (!g_logits && !g_loss) return set_error(ODEVIT_ERR_INVALID_ARG, "head_ce_bwd: no cotangent given");
  ODV_TRY(check_device_ptr(x, "x"));
  ODV_TRY(check_device_ptr(w, "w"));
  ODV_TRY(check_device_ptr(dz, "dz"));
  if (g_loss) {
    ODV_TRY(check_device_ptr(g_loss, "g_loss"));
    ODV_TRY(check_device_ptr(labels, "labels"));
    ODV_TRY(check_device_ptr(logits, "logits"));
    ODV_TRY(check_device_ptr(lse, "lse"));
  }
  return head_ce_bwd(x, x_stride, w, reinterpret_cast<const long long*>(labels), logits, lse, g_logits, g_loss, batch, classes, dim,
                     label_smoothing, dz, g_x, gx_stride, g_w, g_bias, reinterpret_cast<cudaStream_t>(stream));
}

int odevit_extract_mass_fwd(const float* attn_rows, int32_t batch, int32_t heads, int32_t n, float threshold, int32_t smooth,
                            float scale_factor, float* out_mean, float* out_heads, float* out_mask, odevit_stream_t stream) {
  if (batch <= 0 || heads <= 0 || n <= 0) return set_error(ODEVIT_ERR_INVALID_ARG, "extract_mass: non-positive dimension");
  ODV_TRY(check_device_ptr(attn_rows, "attn_rows"));
  ODV_TRY(check_device_ptr(out_mean, "out_mean"));
  if (out_heads) ODV_TRY(check_device_ptr(out_heads, "out_heads"));
  if (out_mask) ODV_TRY(check_device_ptr(out_mask, "out_mask"));
  return extract_mass_fwd(attn_rows, batch, heads, n, threshold, smooth, scale_factor, out_mean, out_heads, out_mask,
                          reinterpret_cast<cudaStream_t>(stream));
}

int odevit_extract_mass_bwd(const float* attn_rows, int32_t batch, int32_t heads, int32_t n, float threshold, int32_t smooth,
                            float scale_factor, const float* g_mean, const float* g_heads, float* g_rows,
                            odevit_stream_t stream) {
  if (batch <= 0 || heads <= 0 || n <= 0) return set_error(ODEVIT_ERR_INVALID_ARG, "extract_mass: non-positive dimension");
  if (!g_mean && !g_heads) return set_error(ODEVIT_ERR_INVALID_ARG, "extract_mass: no cotangent given");
  ODV_TRY(check_device_ptr(attn_rows, "attn_rows"));
  ODV_TRY(check_device_ptr(g_rows, "g_rows"));
  if (g_mean) ODV_TRY(check_device_ptr(g_mean, "g_mean"));
  if (g_heads) ODV_TRY(check_device_ptr(g_heads, "g_heads"));
  return extract_mass_bwd(attn_rows, batch, heads, n, threshold, smooth, scale_factor, g_mean, g_heads, g_rows,
                          reinterpret_cast<cudaStream_t>(stream));
}

int odevit_pil_bilinear_ksize(int32_t in_size, int32_t out_size) {
  if (in_size <= 0 || out_size <= 0) return 0;
  return pil_bilinear_ksize(in_size, out_size);
}

int odevit_pil_bilinear_tables(int32_t in_size, int32_t out_size, int32_t* bounds_host, int32_t* kk_host) {
  if (in_size <= 0 || out_size <= 0 || !bounds_host || !kk_host)
    return set_error(ODEVIT_ERR_INVALID_ARG, "pil_bilinear_tables: bad arguments");
  if (pil_bilinear_ksize(in_size, out_size) > 64)
    return set_error(ODEVIT_ERR_UNSUPPORTED, "pil_bilinear_tables: down-scaling by more than 31x is not built");
  pil_bilinear_tables(in_size, out_size, bounds_host, kk_host);
  return 0;
}

int odevit_preprocess_u8(const uint8_t* images, int32_t batch, int32_t height, int32_t width, int32_t out_h, int32_t out_w,
                         const int32_t* bounds_h, const int32_t* kk_h, const int32_t* bounds_v, const int32_t* kk_v,
                         float rescale, const float* mean3_host, const float* std3_host, uint8_t* tmp, float* out,
                         uint8_t* out_u8, odevit_stream_t stream) {
  if (batch <= 0 || height <= 0 || width <= 0 || out_h <= 0 || out_w <= 0 || !mean3_host || !std3_host)
    return set_error(ODEVIT_ERR_INVALID_ARG, "preprocess_u8: bad arguments");
  ODV_TRY(check_device_ptr(images, "images"));
  ODV_TRY(check_device_ptr(bounds_h, "bounds_h"));
  ODV_TRY(check_device_ptr(kk_h, "kk_h"));
  ODV_TRY(check_device_ptr(bounds_v, "bounds_v"));
  ODV_TRY(check_device_ptr(kk_v, "kk_v"));
  ODV_TRY(check_device_ptr(tmp, "tmp"));
  ODV_TRY(check_device_ptr(out, "out"));
  if (out_u8) ODV_TRY(check_device_ptr(out_u8, "out_u8"));
  return preprocess_u8(images, batch, height, width, out_h, out_w, bounds_h, kk_h, pil_bilinear_ksize(width, out_w), bounds_v,
                       kk_v, pil_bilinear_ksize(height, out_h), rescale, mean3_host, std3_host, tmp, out, out_u8,
                       reinterpret_cast<cudaStream_t>(stream));
}

int odevit_field_bwd(const odevit_desc* desc, const odevit_weights* w, const float* x, const float* g_dx,
                     const float* g_p, float* g_x, const odevit_weight_grads* gw, void* workspace,
                     size_t workspace_bytes, odevit_stream_t stream) {
  Plan p{};
  ODV_TRY(make_plan(desc, &p));
  ODV_TRY(check_weights(p, w));
  if (!gw) return set_error(ODEVIT_ERR_INVALID_ARG, "weight-gradient struct is NULL");
  ODV_TRY(check_device_ptr(x, "x"));
  ODV_TRY(check_device_ptr(g_dx, "g_dx"));
  ODV_TRY(check_device_ptr(g_x, "g_x"));
  Arena a(workspace);
  BwdBufs b = layout_bwd(p, a, 1);
  ODV_TRY(check_ws(workspace, workspace_bytes, a.off));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  ODV_TRY(prepare_drop_keys(p, b.drop_keys, 1, s));
  ODV_TRY(prepare_weights(p, w, b.w, s));
  ODV_CUDA(cudaMemsetAsync(b.G1, 0, b.acc_bytes, s));
  ODV_TRY(eval_forward(p, b.w, b.ctx[0], x, b.P, nullptr, b.sq, b.tmp, 0, nullptr, s));
  {
    CombineArgs c0;
    c0.n_terms = 1; c0.term[0] = g_dx; c0.coef[0] = 1.f;
    c0.out_dd = b.dd; c0.dd_type = p.dd_type; c0.dd_scale = p.scaler;
    ODV_TRY(vjp_combine(c0, p.M, p.D, s));
  }
  {
    Epi e;
    e.c_new = 1.f;
    e.out = g_x;
    ODV_TRY(eval_vjp(p, b.w, b.ctx[0], b, g_p, wants_c2(gw), gw, 0, e, s));
  }
  return finish_grads(p, w, gw, b, s);
}

}  // extern "C"
