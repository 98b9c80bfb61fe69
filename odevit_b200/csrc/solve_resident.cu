// The on-chip-state solver for small-token shapes (CIFAR: N ~ 65-69 tokens, D = 64..192, head dim 64):
// ONE persistent CTA per image runs EVERY solver step of odeint(odefunc, x0, t, method)
// (ode_transformer_gpt.py:571-578 with the parallel field :274-277, :317-330), inference only.
//
// What stays on the chip for the whole solve of an image:
//   shared memory   the ODE state y [N, D] fp32 (row-padded), the centred stage input xc as the bf16
//                   A-operand tile, per-head q/k/v/O tiles, the GELU(fc1) chunk tile, a ring of weight
//                   tiles, the biases
//   tensor memory   R0 [0,192): q|k|v accumulator of a head -> S -> P (bf16 in place) -> O;
//                   R1 [192,192+D): the field output accumulator, summed over all heads' out-projections
//                   and all fc2 chunks;  HB [192+D, +128): the fc1 chunk accumulator
// HBM / L2 sees only: the weights (streamed by TMA, L2 hits after the first CTA), x0 once, each
// trajectory row once (if requested), the last attention map (if requested), and -- for multi-stage
// methods -- the k_l stage vectors in a per-CTA L2-resident scratch.
//
// One evaluation is a fixed list of JOBS (built on the host, `Sched`): a group of tcgen05.mma issued by
// the producer warp, then a compute phase on its result by all compute warps.  Two chains are
// interleaved so that the tensor core works on one while the CUDA cores work on the other:
//   attention chain, per head h:  Q_h  [q|k|v]_h = xc W^T (+ OUT += O_{h-1} Wo)   -> bias, bf16 tiles
//                                 S_h  S = q k^T                                  -> softmax, P in TMEM
//                                 PV_h O = P v (TS-mode)                          -> O / rowsum, bf16 tile
//   MLP chain, per 128-wide hidden chunk c:  FC_c  (OUT += G_{c-1} W2) ; HB = xc W1_c^T  -> GELU tile G_c
//   F: OUT += O_{H-1} Wo + G_{C-1} W2  -> k = scaler (OUT + b2), Butcher stage combine on the resident
//      state, trajectory row, centred next stage input.
// The group of job i is issued as soon as the compute phase of the previous job OF ITS CHAIN is done,
// i.e. while the compute warps are still busy with job i-1 of the other chain.
//
//   loader warp (elected lane)     TMA weight units into the ring
//   producer warp (elected lane)   every tcgen05.mma
//   warps 0-15               quadrant q = warp & 3 owns token rows [32q, 32q+32) (the TMEM lanes a warp
//                            may touch), column share cw = warp >> 2 owns a quarter of the columns of
//                            every phase; thread = (row, column quarter).  Row-wise reductions (softmax
//                            max / sum, CenterNorm mean) are exchanged through shared memory between the
//                            four warps of a quadrant (named barrier 1+q).  Quadrants without rows idle.
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstddef>
#include <cstdlib>
#include <type_traits>

#include "dopri5.cuh"
#include "epilogue.cuh"
#include "host.h"
#include "ptx.cuh"

namespace odevit {

int make_tmap_2d_bf16(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                      uint32_t box_inner, uint32_t box_outer);

namespace {

int num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  return sms;
}

// Warps 0-15 are (quadrant, column share) slots.  With N <= 96 tokens quadrant 3 holds no rows: the MMA
// issuer and the weight loader take slots 3 and 7 (a scheduler of their own) and 512 threads leave 128
// registers each; with more tokens they are warps 16 and 17 (FULL).
__host__ __device__ constexpr int res_threads(bool full) { return full ? 576 : 512; }
__host__ __device__ constexpr int res_producer(bool full) { return full ? 16 : 3; }
__host__ __device__ constexpr int res_loader(bool full) { return full ? 17 : 7; }
constexpr int NU = 10;                               // weight-ring slots of 8 KB
constexpr int T_R0 = 0, T_O = 128, T_R1 = 192;
constexpr int kMaxGrid = kResidentMaxGrid;           // grid points carried in the kernel parameters
constexpr int kMaxJobs = 64, kMaxAllocs = 112;
constexpr int NB = 8;                                // barrier pairs of the weight ring (>= allocations in flight)

enum JobKind : uint8_t { JOB_QKV = 0, JOB_S = 1, JOB_PV = 2, JOB_FC = 3, JOB_F = 4 };

// The job list of one evaluation and the weight ALLOCATIONS it consumes, in issue order.  An allocation is
// one B operand of a run of 4 MMAs (one 64-wide k-atom): `size` consecutive 8 KB ring slots, each filled by
// one [64 x 64] TMA box:
//   kind 0  rows {q, k, v} of head `arg` of W1cat, k-atom ka   -> [192 x 64], N = 192 into R0
//   kind 1  fc1 rows of hidden chunk `arg`, k-atom ka          -> [128 x 64], N = 128 into HB
//   kind 2  W2cat k-atom starting at column `arg`              -> [D x 64],   N = D   into R1
// The slot offsets come from a host-side walk of the ring (an allocation never wraps; every evaluation
// starts at slot 0, so the pattern repeats); `back` = how many allocations before this one the latest
// allocation is whose slots (or barrier pair) it reuses: the loader waits for that one's release.
struct Alloc {
  uint16_t arg;
  uint8_t kind, ka, off, size, back, pad;
};
struct Sched {
  int n_jobs, n_allocs;
  uint8_t kind[kMaxJobs];
  uint8_t arg[kMaxJobs];     // head or hidden chunk
  int8_t dep[kMaxJobs];      // job of this evaluation whose compute phase must be done first; -1: the
                             // previous evaluation's F (or the image's initial phase)
  Alloc alloc[kMaxAllocs];
};

struct ResArgs {
  int B, N, RA, NK, D, H, hid;
  int n_grid, S;
  float scaler;
  float dt[kMaxGrid - 1];
  float a[4][4], b[4];
  const float* x0;       // [B, N, D]
  float* states;         // [T, B, N, D] or null (row 0 written by the host wrapper)
  float* final_state;    // [B, N, D] or null
  float* p_last;         // [B, H, N, N] or null
  const float* b1cat;    // [3D + hid]
  const float* b2;       // [D]
  float* kbuf;           // [grid][3][D][128] fp32 scratch (stage vectors of multi-stage methods)
  Sched sc;
};

// The adaptive mode's arguments (odevit_solve_adaptive_resident): the output times and the Dormand-Prince tableau take
// the place of the fixed grid's step sizes and Butcher tableau.
struct ResArgsAd {
  int B, N, RA, NK, D, H, hid;
  int n_out, max_steps;
  float scaler, rtol, atol;
  double first_step;     // <= 0: selected per image (one probe evaluation)
  float a[6][6], b[6], c_err[7], c_mid[7];
  const float* x0;       // [B, N, D]
  float* states;         // [n_out, B, N, D] (row 0 written by the host wrapper)
  const float* b1cat;
  const float* b2;
  float* kbuf;           // [grid][8][D][RA] fp32 scratch: k1..k7 (k1 and k7 swap slots 0 and 6) and y1 (slot 7)
  int* next_image;       // the image dealer (zeroed by the host wrapper)
  int *nfe, *accepted, *rejected, *status;   // [B] or null (status: never null)
  Sched sc;
  // Last, and not copied to shared memory (1 KB the C10 shape does not have there): read from the parameter space,
  // only when a step is accepted
  double t_out[kMaxGrid];
};
// bytes of the arguments the kernel copies to shared memory
template <class Args> __host__ __device__ constexpr int res_smem_args() { return (int)sizeof(Args); }
template <> __host__ __device__ constexpr int res_smem_args<ResArgsAd>() { return (int)offsetof(ResArgsAd, t_out); }
__device__ __forceinline__ int res_stages(const ResArgs& a) { return a.S; }
__device__ __forceinline__ int res_stages(const ResArgsAd&) { return 1; }
__device__ __forceinline__ int res_evals(const ResArgs& a) { return (a.n_grid - 1) * a.S; }
__device__ __forceinline__ int res_evals(const ResArgsAd&) { return 0; }
// What the compute warps announce with the last compute phase of an evaluation (adaptive mode): the image steps on, its
// solve is over and the next image's initial phase follows, or the CTA has no image left
enum : int { CTL_RUN = 0, CTL_NEXT = 1, CTL_DONE = 2 };

struct Smem {
  int xc_atom;           // bytes of one 64-column atom of RA rows
  int off_xc, off_q, off_k, off_v, off_g, off_ring, off_y, off_b1, off_b2, off_ex, off_args, off_bars, total;
};
__host__ __device__ inline Smem smem_layout(int RA, int N, int D, int hid, int args_bytes = (int)sizeof(ResArgs)) {
  Smem s;
  s.xc_atom = RA * 128;
  int o = 0;
  s.off_xc = o; o += (D / 64) * s.xc_atom;
  s.off_q = o; o += s.xc_atom;      // q; later the O tile of the same head (q is dead once S is formed)
  s.off_k = o; o += s.xc_atom;
  s.off_v = o; o += s.xc_atom;
  s.off_g = o; o += 2 * s.xc_atom;  // GELU(fc1) chunk: two atoms
  o = (o + 1023) & ~1023;
  s.off_ring = o; o += NU * 8192;
  s.off_y = o; o += N * (D + 4) * 4;
  o = (o + 15) & ~15;
  s.off_b1 = o; o += (3 * D + hid) * 4;
  s.off_b2 = o; o += D * 4;
  s.off_ex = o; o += 2 * 4 * 128 * 4;   // row-reduction exchange: [max or mean | sum][column share][row]
  s.off_args = o; o += (args_bytes + 15) / 16 * 16;   // the kernel arguments (see the kernel's first lines)
  s.off_bars = o; o += 256;
  s.total = o;
  return s;
}

// bf16 row of a K-major SWIZZLE_128B tile: 8 consecutive columns [col, col+8) of row r
__device__ __forceinline__ void st_tile8(uint8_t* atom0, int atom_bytes, int r, int col, const float* v) {
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    w[j] = *reinterpret_cast<uint32_t*>(&hh);
  }
  const int atom = col >> 6, chunk = (col & 63) >> 3;
  *reinterpret_cast<uint4*>(atom0 + atom * atom_bytes + r * 128 + ((chunk ^ (r & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st4u(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st16f(uint32_t taddr, const float* v) {
  uint32_t r[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(v[i]);
  ptx::tmem_st16(taddr, r);
}
// 16 consecutive fp32 values of shared memory (64-byte aligned; every lane reads the same address: broadcast)
__device__ __forceinline__ void lds16(const float* p, float* b) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 f = reinterpret_cast<const float4*>(p)[j];
    b[4 * j] = f.x; b[4 * j + 1] = f.y; b[4 * j + 2] = f.z; b[4 * j + 3] = f.w;
  }
}
// Two GELUs at once in half precision (11-bit significand, finer than the bf16 the tile stores):
// GELU(x) = hx + hx tanh(x (c0 + c1 x^2)), hx = x/2, coefficients fitted to the erf form (|formula error|
// <= 2.8e-4 absolute over the reals), ONE MUFU.TANH per pair.  x^2 overflowing to inf gives tanh = +-1, the
// right limit.  Returns the pair packed as bf16x2 (low half = first argument).
__device__ __forceinline__ uint32_t gelu2_bf16(float x0, float x1) {
  const __half2 x = __floats2half2_rn(x0, x1);
  const __half2 x2 = __hmul2(x, x);
  const __half2 p = __hfma2(x2, __float2half2_rn(0.034700893432451876f), __float2half2_rn(0.8001570785469041f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 t = *reinterpret_cast<const __half2*>(&ti);
  const __half2 hx = __hmul2(x, __float2half2_rn(0.5f));
  const float2 g = __half22float2(__hfma2(hx, t, hx));
  const __nv_bfloat162 o = __floats2bfloat162_rn(g.x, g.y);
  return *reinterpret_cast<const uint32_t*>(&o);
}
// 8 consecutive bf16 columns (4 packed words) of row r of a K-major SWIZZLE_128B tile
__device__ __forceinline__ void st_tile8w(uint8_t* atom0, int atom_bytes, int r, int col, const uint32_t* w) {
  const int atom = col >> 6, chunk = (col & 63) >> 3;
  *reinterpret_cast<uint4*>(atom0 + atom * atom_bytes + r * 128 + ((chunk ^ (r & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// shared memory -> global memory through the bulk-copy engine (16-byte aligned, size a multiple of 16)
__device__ __forceinline__ void bulk_store(float* gdst, const float* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ptx::smem_u32(ssrc)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// the four warps of token-row quadrant q
__device__ __forceinline__ void quad_sync(int q) { asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory"); }

#ifdef RES_TRACE
// clock stamps of CTA 0, second evaluation of its first image: class 0 = compute thread 0, 1 = producer
__device__ uint32_t rtr[2][256];
__device__ uint16_t rtr_id[2][256];
__device__ int rtr_n[2];
#define RTR(cls, slot) do { if (rtr_on && rtr_cnt < 256) { rtr[cls][rtr_cnt] = (uint32_t)clock(); rtr_id[cls][rtr_cnt] = (uint16_t)(slot); ++rtr_cnt; rtr_n[cls] = rtr_cnt; } } while (0)
#else
#define RTR(cls, slot) do { } while (0)
#endif

template <bool FULL, bool ADAPTIVE>
__global__ void __launch_bounds__(res_threads(FULL), 1)
solve_resident_kernel(const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                      const __grid_constant__ std::conditional_t<ADAPTIVE, ResArgsAd, ResArgs> a_param) {
  using Args = std::conditional_t<ADAPTIVE, ResArgsAd, ResArgs>;
  extern __shared__ __align__(1024) uint8_t smem[];
  const Smem L = smem_layout(a_param.RA, a_param.N, a_param.D, a_param.hid, res_smem_args<Args>());
  // The arguments are read from a shared-memory copy: the job list, step sizes and tableau are indexed
  // dynamically all through the solve, and the constant cache does not hold them next to the instruction
  // stream's own constants (measured: ~2000 cycles per 150-instruction loop iteration with LDC in it).
  const Args& a = *reinterpret_cast<const Args*>(smem + L.off_args);
  uint8_t* sXC = smem + L.off_xc;
  uint8_t* sQ = smem + L.off_q;
  uint8_t* sK = smem + L.off_k;
  uint8_t* sV = smem + L.off_v;
  uint8_t* sG = smem + L.off_g;
  uint8_t* sRing = smem + L.off_ring;
  float* sY = reinterpret_cast<float*>(smem + L.off_y);
  float* sB1 = reinterpret_cast<float*>(smem + L.off_b1);
  float* sB2 = reinterpret_cast<float*>(smem + L.off_b2);
  float* sEx = reinterpret_cast<float*>(smem + L.off_ex);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bars);
  uint64_t* bar_full = bars;              // [NB] the boxes of a weight allocation landed
  uint64_t* bar_free = bars + NB;         // [NB] the MMAs that read the allocation have retired
  uint64_t* bar_mma = bars + 2 * NB;      // [2] the MMA group of job (parity of the job counter) has retired
  uint64_t* bar_cmp = bars + 2 * NB + 2;  // [2] the compute phase (parity of the phase counter) is finished
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NB + 4);
  // adaptive mode: [0] CTL_* of the last compute phase, [1] the image just dealt, [2] 1 once the CTA has no image left
  // (the loader stops), [3] weight allocations the producer consumed (teardown)
  volatile int* ctl = reinterpret_cast<volatile int*>(bars + 2 * NB + 6);

  constexpr int RES_THREADS = res_threads(FULL), PRODUCER = res_producer(FULL), LOADER = res_loader(FULL);
  const int warp = threadIdx.x >> 5;
#ifdef RES_TRACE
  if (threadIdx.x == 0 && blockIdx.x == 0) { rtr_n[0] = 0; rtr_n[1] = 0; }
  bool rtr_on = false;
  int rtr_cnt = 0;
#endif
  const int D = a_param.D, H = a_param.H, N = a_param.N, NK = a_param.NK;
  const int T_HB = T_R1 + D;
  const int nJ = a_param.sc.n_jobs;
  const int n_evals = res_evals(a_param);
  const int n_mine = (a_param.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int n_quads = (N + 31) >> 5;           // token-row quadrants that hold rows

  if (threadIdx.x == 0) {
    for (int i = 0; i < NB; ++i) { ptx::mbar_init(bar_full + i, 1); ptx::mbar_init(bar_free + i, 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(bar_mma + i, 1); ptx::mbar_init(bar_cmp + i, n_quads * 128); }
    ptx::fence_barrier_init();
    if constexpr (ADAPTIVE) ctl[2] = 0;
  }
  if (warp == PRODUCER) ptx::tmem_alloc(tmem_slot, 512);
  // biases -> shared memory; operand tiles zeroed once (rows [N, RA) stay zero: a thread only writes its own row)
  for (int i = threadIdx.x; i < 3 * D + a_param.hid; i += RES_THREADS) sB1[i] = a_param.b1cat[i];
  for (int i = threadIdx.x; i < D; i += RES_THREADS) sB2[i] = a_param.b2[i];
  for (int i = threadIdx.x; i < res_smem_args<Args>() / 4; i += RES_THREADS)
    reinterpret_cast<uint32_t*>(smem + L.off_args)[i] = reinterpret_cast<const uint32_t*>(&a_param)[i];
  for (int i = threadIdx.x; i < L.off_ring / 16; i += RES_THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  ptx::fence_async_shared();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  uint32_t ld_issued = 0;                   // adaptive mode: weight allocations the loader issued
  if (warp == PRODUCER) {
    // ======================= producer: weight units + every MMA =======================
    // The ring moves UNITS: one [64 x 64] bf16 box (8 KB).  A tile of the job list is D/64 consecutive units
    // (the k-atoms of 64 W1cat rows, or the 64-row blocks of one W2cat k-atom), so a stage is refilled as
    // soon as 4 MMAs retire and the ring always holds NU units in flight whatever the job boundaries are.
    // Every lane runs the same instruction stream; the tcgen05 instructions carry the election as a
    // predicate, so the warp never diverges and needs no __syncwarp.
    const uint32_t lead = ptx::elect_one() ? 1u : 0u;
    uint32_t cg = 0;                          // allocations consumed (global count: barrier pair and phase)
    int ci = 0;                               // ... and the index of the next one in the evaluation's list
    const int n_allocs = a.sc.n_allocs;
    uint32_t waited = 0;                      // compute phases consumed
    uint32_t gm = 0;                          // MMA groups committed
    const int UPT = D / 64;                   // k-atoms of the model dimension
    // K-major SWIZZLE_128B descriptors differ only in their 14-bit address field: desc(addr) = DESC0 + (addr >> 4)
    const uint64_t DESC0 = ptx::smem_desc_sw128(0, 16, 1024);
    const uint32_t ring_lo = ptx::smem_u32(sRing) >> 4;
    const uint32_t full0 = ptx::smem_u32(bar_full), free0 = ptx::smem_u32(bar_free);
    const uint32_t id_qkv = ptx::idesc_bf16(128, 192, 0, 0), id_fc1 = ptx::idesc_bf16(128, 128, 0, 0);
    const uint32_t id_out = ptx::idesc_bf16(128, D, 0, 0);

    // the next weight allocation [N x 64]: D[128 x N] (+)= A[128 x 64] (descriptor address field a_lo) * alloc^T
    auto alloc_mma = [&](uint32_t d_tmem, uint32_t a_lo, uint32_t idesc, uint32_t acc_first) {
      const uint32_t b = cg & (NB - 1);
      const uint32_t fb = full0 + b * 8;
      for (uint32_t spins = 0; !ptx::mbar_try_wait_addr(fb, (cg / NB) & 1);)
        if (++spins > (1u << 24)) __trap();   // a protocol bug must surface as a launch failure, never as a hung GPU
      const uint64_t da = DESC0 + a_lo, db = DESC0 + (ring_lo + (uint32_t)a.sc.alloc[ci].off * 512);
      ptx::mma_ss_pred(d_tmem, da, db, idesc, acc_first, lead);
      ptx::mma_ss_pred(d_tmem, da + 2, db + 2, idesc, 1u, lead);
      ptx::mma_ss_pred(d_tmem, da + 4, db + 4, idesc, 1u, lead);
      ptx::mma_ss_pred(d_tmem, da + 6, db + 6, idesc, 1u, lead);
      ptx::commit_pred(free0 + b * 8, lead);
      ++cg;
      if (++ci == n_allocs) ci = 0;
    };
    // all compute phases up to and including `phase` are finished
    auto need = [&](uint32_t phase) {
      while (waited <= phase) {
        ptx::mbar_wait(bar_cmp + (int)(waited & 1), (uint32_t)((waited >> 1) & 1));
        ++waited;
      }
      ptx::tc_fence_after();
    };
    const uint32_t xc_lo = ptx::smem_u32(sXC) >> 4, q_lo = ptx::smem_u32(sQ) >> 4, k_lo = ptx::smem_u32(sK) >> 4;
    const uint32_t g_lo = ptx::smem_u32(sG) >> 4, atom_lo = (uint32_t)L.xc_atom >> 4;
    const uint32_t v_addr = ptx::smem_u32(sV);
    const uint32_t id_s = ptx::idesc_bf16(128, NK, 0, 0);
    const uint32_t id_pv = ptx::idesc_bf16(128, 64, 0, 1);
    uint32_t r1_acc = 0;                      // 0: the next MMAs into R1 start a new field output
    // D[128 x N] = xc[128 x D] * W^T over the k-atoms of the model dimension (q|k|v of a head, or an fc1 chunk)
    auto mma_xc = [&](uint32_t d_tmem, uint32_t idesc) {
      for (int ka = 0; ka < UPT; ++ka) alloc_mma(d_tmem, xc_lo + ka * atom_lo, idesc, ka > 0 ? 1u : 0u);
    };
    // OUT[128 x D] += A[128 x 64] (one 64-column atom, address field a_lo) * W2cat k-atom [D x 64]^T
    auto mma_into_out = [&](uint32_t a_lo) {
      alloc_mma(tmem + T_R1, a_lo, id_out, r1_acc);
      r1_acc = 1u;
    };

    // the MMA group of one job, committed to bar_mma
    auto issue = [&](int kind, int arg) {
      if (kind == JOB_QKV) {
        if (arg > 0) mma_into_out(q_lo);                         // O of the previous head (in the q tile)
        mma_xc(tmem + T_R0, id_qkv);
      } else if (kind == JOB_S) {
        const uint64_t da = DESC0 + q_lo, db = DESC0 + k_lo;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) ptx::mma_ss_pred(tmem + T_R0, da + 2 * kk, db + 2 * kk, id_s, kk > 0 ? 1u : 0u, lead);
      } else if (kind == JOB_PV) {
        for (int ks = 0; ks < NK / 16; ++ks)
          ptx::mma_ts_pred(tmem + T_O, tmem + T_R0 + ks * 8, ptx::smem_desc_sw128(v_addr + ks * 2048, 8192, 1024), id_pv,
                      ks > 0 ? 1u : 0u, lead);
      } else if (kind == JOB_FC) {
        if (arg > 0)
          for (int m = 0; m < 2; ++m) mma_into_out(g_lo + m * atom_lo);      // fc2 of the previous chunk
        mma_xc(tmem + T_HB, id_fc1);
      } else {  // JOB_F
        mma_into_out(q_lo);                                      // O of the last head
        for (int m = 0; m < 2; ++m) mma_into_out(g_lo + m * atom_lo);
      }
      ptx::commit_pred(ptx::smem_u32(bar_mma + (int)(gm & 1)), lead);
      ++gm;
    };

    if constexpr (ADAPTIVE) {
      // The number of evaluations is decided on the chip: the compute warps announce with each F phase whether the
      // image steps on, the next image's initial phase follows, or the CTA is done (ctl[0]).  The next evaluation's
      // first job waits for that phase anyway (dep < 0), so reading the word there costs nothing.
      uint32_t P = 0;                         // phase that formed the current evaluation's stage input
      need(P);
      if (ctl[0] != CTL_DONE) {
        for (;;) {
          r1_acc = 0u;
#pragma unroll 1
          for (int j = 0; j < nJ; ++j) {
            const int dep = a.sc.dep[j];
            need(dep < 0 ? P : P + 1 + (uint32_t)dep);
            issue(a.sc.kind[j], a.sc.arg[j]);
          }
          P += nJ;
          need(P);
          const int f = ctl[0];
          if (f == CTL_DONE) break;
          if (f == CTL_NEXT) ++P;             // the next image's initial phase
        }
      }
      ctl[3] = (int)cg;
    }
    for (int idx = 0; idx < n_mine && !ADAPTIVE; ++idx) {
      const uint32_t base = (uint32_t)idx * (1u + (uint32_t)n_evals * nJ);   // phase of the image's initial xc
      for (int ev = 0; ev < n_evals; ++ev) {
        r1_acc = 0u;
#ifdef RES_TRACE
        rtr_on = (blockIdx.x == 0 && idx == 0 && ev == 1 && (threadIdx.x & 31) == 0);
#endif
#pragma unroll 1
        for (int j = 0; j < nJ; ++j) {
          const int kind = a.sc.kind[j], arg = a.sc.arg[j], dep = a.sc.dep[j];
          RTR(1, j * 4 + 0);
          need(dep < 0 ? base + (uint32_t)ev * nJ : base + 1 + (uint32_t)ev * nJ + dep);
          RTR(1, j * 4 + 1);
          issue(kind, arg);
          RTR(1, j * 4 + 2);
        }
      }
    }
  } else if (warp == LOADER) {
    // ======================= loader: streams the weight units of every evaluation through the ring =======================
    // Walks the evaluation's allocation list (struct Alloc) over and over: NU slots of 8 KB, up to NB
    // allocations in flight, each refilled as soon as the 4 MMAs that read its predecessor retire.
    const bool leader = ptx::elect_one();
    if (leader) { ptx::prefetch_tensormap(&tmW1); ptx::prefetch_tensormap(&tmW2); }
    const int n_allocs = a.sc.n_allocs;
    const uint32_t total = ADAPTIVE ? 0xffffffffu : (uint32_t)n_mine * n_evals * n_allocs;
    int li = 0;
    uint32_t g = 0;
    // adaptive mode: the allocation cycle is the same whatever the evaluation boundaries are, so the loader streams it
    // until the CTA has no image left; the waits of the allocations nobody will consume end on that flag
    int lead_lane = 0;
    if constexpr (ADAPTIVE) lead_lane = __ffs(__ballot_sync(0xffffffffu, leader)) - 1;
    for (; g < total; ++g) {
      const Alloc al = a.sc.alloc[li];
      if (g >= al.back) {   // the allocation whose slots / barrier pair this one reuses has been released
        const uint32_t w = g - al.back;
        if constexpr (ADAPTIVE) {
          int st = 0;   // the leader's view, for the whole warp: 1 released, 2 the CTA is done
          for (uint32_t spins = 0; st == 0;) {
            st = ptx::mbar_try_wait(bar_free + (w & (NB - 1)), (w / NB) & 1) ? 1 : (ctl[2] ? 2 : 0);
            st = __shfl_sync(0xffffffffu, st, lead_lane);
            if (++spins > (1u << 24)) __trap();
          }
          if (st == 2) break;
        } else {
          ptx::mbar_wait(bar_free + (w & (NB - 1)), (w / NB) & 1);
        }
      }
      if (leader) {
        uint64_t* fb = bar_full + (g & (NB - 1));
        uint8_t* dst = sRing + (int)al.off * 8192;
        ptx::mbar_expect_tx(fb, (uint32_t)al.size * 8192);
        if (al.kind == 0) {
          for (int m = 0; m < 3; ++m) ptx::tma_load_2d(dst + m * 8192, &tmW1, fb, al.ka * 64, m * D + al.arg * 64);
        } else if (al.kind == 1) {
          for (int m = 0; m < 2; ++m) ptx::tma_load_2d(dst + m * 8192, &tmW1, fb, al.ka * 64, 3 * D + al.arg * 128 + m * 64);
        } else {
          for (int nb = 0; nb < (int)al.size; ++nb) ptx::tma_load_2d(dst + nb * 8192, &tmW2, fb, al.arg, nb * 64);
        }
      }
      __syncwarp();
      if (++li == n_allocs) li = 0;
    }
    ld_issued = g;
  } else if (warp < 16 && (warp & 3) < n_quads) {
    // ======================= compute warps: thread = (token row, column quarter) =======================
    const int q = warp & 3, cw = warp >> 2;
    const int r = q * 32 + (threadIdx.x & 31);
    const bool row_ok = r < N;
    const uint32_t t_lane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    uint32_t gm = 0, gc = 0;                   // only their two low bits matter (barrier index, phase parity)
    auto wait_mma = [&]() {
      ptx::mbar_wait(bar_mma + (gm & 1), (gm >> 1) & 1);
      ++gm;
      ptx::tc_fence_after();
    };
    auto done = [&]() {   // shared-memory writes -> async proxy, tensor-memory traffic ordered, then signal
      ptx::fence_async_shared();
      ptx::tc_fence_before();
      ptx::mbar_arrive(bar_cmp + (gc & 1));
      ++gc;
    };
    float* yrow = sY + (size_t)(row_ok ? r : 0) * (D + 4);   // row stride D+4 floats: conflict-free 16-byte accesses
    float* kb = a_param.kbuf + (size_t)blockIdx.x * (ADAPTIVE ? 8 * D * a_param.RA : 3 * D * 128);
    float* ex_max = sEx;          // softmax row max; between evaluations the CenterNorm row sums
    float* ex_sum = sEx + 512;
    float* ex_mean = sEx;
    constexpr float LOG2E = 1.4426950408889634f;
    const int DQ = D / 4;                      // columns of a D-wide row this thread owns: [cw*DQ, +DQ), 16 | DQ
    const int ngq = DQ / 16;
    float inv_sum = 0.f;                       // 1 / softmax row sum of the current head

    // The stage input u sits in R1 (this thread's columns, fp32): partial row sum -> mean over D (exchange
    // between the four warps of the quadrant) -> centred bf16 row into the xc tile.
    auto centre_from_r1 = [&](float part) {
      ex_mean[cw * 128 + r] = part;
      ptx::tmem_st_wait();
      quad_sync(q);
      const float mean = ((ex_mean[r] + ex_mean[128 + r]) + (ex_mean[256 + r] + ex_mean[384 + r])) / (float)D;
#pragma unroll 1
      for (int g = 0; g < ngq; ++g) {
        float v[16];
        ptx::tmem_ld16(t_lane + T_R1 + cw * DQ + g * 16, v);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) v[jj] -= mean;
        if (row_ok) {
          st_tile8(sXC, L.xc_atom, r, cw * DQ + g * 16, v);
          st_tile8(sXC, L.xc_atom, r, cw * DQ + g * 16 + 8, v + 8);
        }
      }
    };

    // ---- adaptive mode ----
    // CTA-wide sums over the compute warps in a fixed order (rows, then warps): accept / reject never varies between runs
    auto cta_sum = [&](double& s0, double& s1) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      }
      double* red = reinterpret_cast<double*>(ex_sum);   // the softmax sums are dead until the next S phase
      if ((threadIdx.x & 31) == 0) { red[2 * warp] = s0; red[2 * warp + 1] = s1; }
      asm volatile("bar.sync 5, %0;" ::"r"(n_quads * 128) : "memory");
      s0 = 0.0; s1 = 0.0;
      for (int w = 0; w < 16; ++w)
        if ((w & 3) < n_quads) { s0 += red[2 * w]; s1 += red[2 * w + 1]; }
    };
    // the next image for this CTA (>= B: none left): images cost different numbers of steps, so they are dealt as CTAs
    // become free, and an image's result does not depend on which CTA runs it
    auto fetch = [&](const auto& ap) -> int {
      if (threadIdx.x == 0) ctl[1] = atomicAdd(ap.next_image, 1);
      asm volatile("bar.sync 5, %0;" ::"r"(n_quads * 128) : "memory");
      return ctl[1];
    };
    int img = 0;
    // the image's controller, the same in every compute thread (each forms it from the same CTA-wide sums).  stage s
    // evaluates k_{s+1} (s = 0..6) or the initial-step probe (kProbe); k1 and k7 swap slots 0 and 6 on accept (FSAL)
    constexpr int kProbe = 7;
    double t = 0.0, dt = 0.0, h0 = 0.0, d1 = 0.0;
    int on = 1, att = 0, n_acc = 0, n_rej = 0, stage = 0, k1s = 0, nfe_base = 1;
    bool stepping = false;
    auto kslot = [&](int l) { return l == 0 ? k1s : (l == 6 ? 6 - k1s : l); };
    auto kld = [&](int l, int col) { return kb[((size_t)kslot(l) * D + col) * a_param.RA + r]; };
    // u2 = y0 + dt a21 k1 -> R1: the first stage input of an attempt; returns the partial row sum
    auto form_u2 = [&]() -> float {
      float part = 0.f;
#pragma unroll 1
      for (int g = 0; g < ngq; ++g) {
        const int col0 = cw * DQ + g * 16;
        float v[16];
        lds16(yrow + col0, v);
        const float dtf = (float)dt;
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
          const float k1 = row_ok ? kld(0, col0 + jj) : 0.f;
          v[jj] = fmaf(dtf, a.a[1][0] * k1, v[jj]);
          part += v[jj];
        }
        tmem_st16f(t_lane + T_R1 + col0, v);
      }
      return part;
    };
    if constexpr (ADAPTIVE) {
      img = fetch(a_param);
      if (img >= a_param.B) {   // nothing for this CTA: release the producer and the loader
        if (threadIdx.x == 0) { ctl[0] = CTL_DONE; ctl[2] = 1; }
        done();
      } else if (threadIdx.x == 0) {
        ctl[0] = CTL_RUN;
      }
    }

    for (int idx = 0; ADAPTIVE ? img < a_param.B : idx < n_mine; ++idx) {
      if constexpr (ADAPTIVE) {
        t = a_param.t_out[0];
        dt = a.first_step > 0 ? a.first_step : 0.0;
        nfe_base = a.first_step > 0 ? 1 : 2;
        on = 1; att = 0; n_acc = 0; n_rej = 0; stage = 0; k1s = 0;
        stepping = true;
      } else {
        img = (int)blockIdx.x + idx * (int)gridDim.x;
      }
      // ---- x0 -> resident state, first xc ----
      {
        if (cw == 0) bulk_wait_read();   // the previous image's last row stores have read the state
        quad_sync(q);   // ... and its last mean exchange has been read by every warp of the quadrant
        float part = 0.f;
        const float* src = a_param.x0 + ((size_t)img * N + (row_ok ? r : 0)) * D + cw * DQ;
#pragma unroll 1
        for (int g = 0; g < ngq; ++g) {
          float v[16];
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float4 f = row_ok ? *reinterpret_cast<const float4*>(src + g * 16 + jj * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            v[4 * jj] = f.x; v[4 * jj + 1] = f.y; v[4 * jj + 2] = f.z; v[4 * jj + 3] = f.w;
          }
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) part += v[jj];
          if (row_ok) {
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
              reinterpret_cast<float4*>(yrow + cw * DQ + g * 16)[jj] = make_float4(v[4 * jj], v[4 * jj + 1], v[4 * jj + 2], v[4 * jj + 3]);
          }
          tmem_st16f(t_lane + T_R1 + cw * DQ + g * 16, v);
        }
        centre_from_r1(part);
        done();
      }
      for (int ev = 0; ADAPTIVE ? stepping : ev < n_evals; ++ev) {
        const int step = ev / res_stages(a), st = ev - step * res_stages(a);
        const bool last_eval = (ev == n_evals - 1);
#ifdef RES_TRACE
        rtr_on = (blockIdx.x == 0 && idx == 0 && ev == 1 && threadIdx.x == 0);
#endif
#pragma unroll 1
        for (int j = 0; j < nJ; ++j) {
          const int kind = a.sc.kind[j], arg = a.sc.arg[j];
          RTR(0, j * 4 + 0);
          wait_mma();
          RTR(0, j * 4 + 1);
          if (j == 0 && cw == 0) bulk_wait_read();   // the row stores of the previous step have read the state
          if (kind == JOB_FC) {
            // ---- fc1 chunk -> bias -> GELU -> bf16 tile: 32 of the 128 columns ----
            const float* bias = sB1 + 3 * D + arg * 128 + cw * 32;
#pragma unroll 1
            for (int g = 0; g < 2; ++g) {
              float v[16];
              ptx::tmem_ld16(t_lane + T_HB + cw * 32 + g * 16, v);
              float bv[16];
              lds16(bias + g * 16, bv);
              ptx::tmem_ld_wait();
              uint32_t w[8];
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) w[jj] = gelu2_bf16(v[2 * jj] + bv[2 * jj], v[2 * jj + 1] + bv[2 * jj + 1]);
              if (row_ok) {
                st_tile8w(sG, L.xc_atom, r, cw * 32 + g * 16, w);
                st_tile8w(sG, L.xc_atom, r, cw * 32 + g * 16 + 8, w + 4);
              }
            }
          } else if (kind == JOB_QKV) {
            // ---- q | k | v accumulators -> bias -> bf16 tiles: this thread's 48 of the 192 columns ----
#pragma unroll 1
            for (int g = 0; g < 3; ++g) {
              const int G = cw * 3 + g, m = G >> 2, c = G & 3;
              float v[16];
              ptx::tmem_ld16(t_lane + T_R0 + G * 16, v);
              float bv[16];
              lds16(sB1 + m * D + arg * 64 + c * 16, bv);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) v[jj] += bv[jj];
              if (row_ok) {
                uint8_t* dst = sQ + m * L.xc_atom;     // q, k, v tiles are consecutive
                st_tile8(dst, L.xc_atom, r, c * 16, v);
                st_tile8(dst, L.xc_atom, r, c * 16 + 8, v + 8);
              }
            }
          } else if (kind == JOB_S) {
            // ---- softmax over the keys of this row; 8-key groups g = cw, cw+4, ...; P packed in place ----
            float v[4][8];
            const int ng = NK / 8;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (cw + 4 * i < ng) tmem_ld8(t_lane + T_R0 + (cw + 4 * i) * 8, v[i]);
            ptx::tmem_ld_wait();
            float mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (cw + 4 * i < ng) {
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                  if ((cw + 4 * i) * 8 + jj >= N) v[i][jj] = -INFINITY;
                  mx = fmaxf(mx, v[i][jj]);
                }
              }
            ex_max[cw * 128 + r] = mx;
            quad_sync(q);     // every warp of the quadrant holds its S values in registers from here on
            mx = fmaxf(fmaxf(ex_max[r], ex_max[128 + r]), fmaxf(ex_max[256 + r], ex_max[384 + r]));
            const float mxs = mx * LOG2E;
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (cw + 4 * i < ng) {
                uint32_t packed[4];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                  v[i][jj] = ex2f(fmaf(v[i][jj], LOG2E, -mxs));
                  sum += v[i][jj];
                }
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                  __nv_bfloat162 hh = __floats2bfloat162_rn(v[i][2 * jj], v[i][2 * jj + 1]);
                  packed[jj] = *reinterpret_cast<uint32_t*>(&hh);
                }
                tmem_st4u(t_lane + T_R0 + (cw + 4 * i) * 4, packed);
              }
            ex_sum[cw * 128 + r] = sum;
            quad_sync(q);
            inv_sum = 1.f / ((ex_sum[r] + ex_sum[128 + r]) + (ex_sum[256 + r] + ex_sum[384 + r]));
            if constexpr (!ADAPTIVE) {
              if (last_eval && a_param.p_last && row_ok) {
                float* p_row = a_param.p_last + (((size_t)img * H + arg) * N + r) * N;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  if (cw + 4 * i < ng) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                      const int col = (cw + 4 * i) * 8 + jj;
                      if (col < N) p_row[col] = v[i][jj] * inv_sum;
                    }
                  }
              }
            }
            ptx::tmem_st_wait();
          } else if (kind == JOB_PV) {
            // ---- O row * 1/sum -> bf16 tile (over the q tile): 16 of the 64 columns ----
            float v[16];
            ptx::tmem_ld16(t_lane + T_O + cw * 16, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) v[jj] *= inv_sum;
            if (row_ok) {
              st_tile8(sQ, L.xc_atom, r, cw * 16, v);
              st_tile8(sQ, L.xc_atom, r, cw * 16 + 8, v + 8);
            }
          } else if constexpr (ADAPTIVE) {
            // ---- k = scaler (OUT + b2) kept in the scratch; a stage combine, or norm partials -> the step decision ----
            const double nel = (double)N * D;
            const bool combine = (stage >= 1 && stage <= 5) || (stage == 0 && a.first_step > 0);
            const float* coef = stage == 5 ? a.b : a.a[stage + 1 < 6 ? stage + 1 : 0];
            const float dtf = (float)dt;
            float part = 0.f;
            double s0 = 0.0, s1 = 0.0;
#pragma unroll 1
            for (int g = 0; g < ngq; ++g) {
              const int col0 = cw * DQ + g * 16;
              float v[16];
              ptx::tmem_ld16(t_lane + T_R1 + col0, v);
              float bv[16];
              lds16(sB2 + col0, bv);
              float yv[16];
              lds16(yrow + col0, yv);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) v[jj] = a.scaler * (v[jj] + bv[jj]);
              if (stage != kProbe && row_ok) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) kb[((size_t)kslot(stage) * D + col0 + jj) * a_param.RA + r] = v[jj];
              }
              if (combine) {   // u_{s+2} = y0 + dt sum_l a[s+1][l] k_l  (after k6: y1 with b = c_sol, kept in slot 7)
                float acc[16];
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) acc[jj] = coef[stage] * v[jj];
#pragma unroll 1
                for (int l = 0; l < stage; ++l) {
                  const float cl = coef[l];
                  if (cl != 0.f && row_ok) {
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) acc[jj] = fmaf(cl, kld(l, col0 + jj), acc[jj]);
                  }
                }
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                  v[jj] = fmaf(dtf, acc[jj], yv[jj]);
                  part += v[jj];
                }
                if (stage == 5 && row_ok) {
#pragma unroll
                  for (int jj = 0; jj < 16; ++jj) kb[((size_t)7 * D + col0 + jj) * a_param.RA + r] = v[jj];
                }
                tmem_st16f(t_lane + T_R1 + col0, v);
              } else if (row_ok) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                  const float sc = a.atol + fabsf(yv[jj]) * a.rtol;
                  if (stage == 0) {            // initial-step selection: |y0 / sc|^2, |f0 / sc|^2
                    const float q0 = yv[jj] / sc, q1 = v[jj] / sc;
                    s0 += (double)(q0 * q0);
                    s1 += (double)(q1 * q1);
                  } else if (stage == kProbe) {   // |(f1 - f0) / sc|^2
                    const float q = (v[jj] - kld(0, col0 + jj)) / sc;
                    s0 += (double)(q * q);
                  } else {                     // |err / tol|^2, err = dt sum_l c_err[l] k_l, k7 = v
                    float e = a.c_err[0] * kld(0, col0 + jj);
                    e = fmaf(a.c_err[2], kld(2, col0 + jj), e);
                    e = fmaf(a.c_err[3], kld(3, col0 + jj), e);
                    e = fmaf(a.c_err[4], kld(4, col0 + jj), e);
                    e = fmaf(a.c_err[5], kld(5, col0 + jj), e);
                    e = fmaf(a.c_err[6], v[jj], e);
                    e *= dtf;
                    const float tol = a.atol + a.rtol * fmaxf(fabsf(yv[jj]), fabsf(kld(7, col0 + jj)));
                    const float q = e / tol;
                    s0 += (double)(q * q);
                  }
                }
              }
            }
            bool finished = false;
            if (combine) {
              ++stage;
            } else if (stage == 0) {
              cta_sum(s0, s1);
              dp5_probe_step(s0, s1, nel, h0, d1);
              const float hf = (float)h0;
              part = 0.f;
#pragma unroll 1
              for (int g = 0; g < ngq; ++g) {   // the probe y0 + h0 f0
                const int col0 = cw * DQ + g * 16;
                float v[16];
                lds16(yrow + col0, v);
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                  v[jj] = fmaf(hf, 1.f * (row_ok ? kld(0, col0 + jj) : 0.f), v[jj]);
                  part += v[jj];
                }
                tmem_st16f(t_lane + T_R1 + col0, v);
              }
              stage = kProbe;
            } else if (stage == kProbe) {
              cta_sum(s0, s1);
              dt = dp5_first_step(s0, nel, h0, d1);
              part = form_u2();
              stage = 1;
            } else {
              // ---- the step decision (ad_control_kernel's arithmetic) ----
              cta_sum(s0, s1);
              const double ratio = sqrt(s0 / nel);
              ++att;
              int fail = -1, on1 = on;
              const bool ok = ratio <= 1.0;
              double t1 = t, dt_new = 0.0;
              if (!isfinite(ratio)) {
                fail = kErrNonFinite;
              } else {
                if (ok) {
                  t1 = t + dt;
                  while (on1 < a.n_out && a_param.t_out[on1] <= t1) ++on1;
                  ++n_acc;
                } else {
                  ++n_rej;
                }
                dt_new = dp5_next_step(dt, ratio);
                if (on1 < a.n_out) {
                  if (att >= a.max_steps) fail = kErrMax;
                  else if (t1 + dt_new == t1) fail = kErrUnderflow;
                }
              }
              const size_t MD = (size_t)a.B * N * D;
              float* srow = a_param.states + ((size_t)img * N + r) * D;
              if (fail < 0 && ok) {
                // dense output for every output time in (t, t1] (ad_commit_kernel's arithmetic), then y0 <- y1
                if (row_ok) {
#pragma unroll 1
                  for (int c4 = 0; c4 < DQ / 4; ++c4) {
                    const int col = cw * DQ + c4 * 4;
                    Dp5Quartic qa[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                      const float f0 = kld(0, col + i), f1 = kld(6, col + i), y1 = kld(7, col + i);
                      float m = a.c_mid[0] * f0;
                      m = fmaf(a.c_mid[2], kld(2, col + i), m);
                      m = fmaf(a.c_mid[3], kld(3, col + i), m);
                      m = fmaf(a.c_mid[4], kld(4, col + i), m);
                      m = fmaf(a.c_mid[5], kld(5, col + i), m);
                      m = fmaf(a.c_mid[6], f1, m);
                      qa[i] = Dp5Quartic(yrow[col + i], y1, f0, f1, m, dtf);
                      yrow[col + i] = y1;
                    }
                    for (int jo = on; jo < on1; ++jo) {
                      const float x = (float)((a_param.t_out[jo] - t) / dt);
                      *reinterpret_cast<float4*>(srow + (size_t)jo * MD + col) = make_float4(qa[0].at(x), qa[1].at(x), qa[2].at(x), qa[3].at(x));
                    }
                  }
                }
                k1s = 6 - k1s;
                t = t1;
                on = on1;
              }
              if (fail >= 0 && row_ok) {   // a failed image stops: the rows it has not reached are NaN
                for (int jo = on; jo < a.n_out; ++jo)
                  for (int c = 0; c < DQ; c += 4)
                    *reinterpret_cast<float4*>(srow + (size_t)jo * MD + cw * DQ + c) = make_float4(NAN, NAN, NAN, NAN);
              }
              dt = dt_new;
              finished = fail >= 0 || on >= a.n_out;
              if (finished) {
                if (threadIdx.x == 0) {
                  if (a_param.nfe) a_param.nfe[img] = nfe_base + 6 * att;
                  if (a_param.accepted) a_param.accepted[img] = n_acc;
                  if (a_param.rejected) a_param.rejected[img] = n_rej;
                  a_param.status[img] = fail + 1;
                }
                img = fetch(a_param);
                if (threadIdx.x == 0) {
                  ctl[0] = img < a_param.B ? CTL_NEXT : CTL_DONE;
                  if (img >= a_param.B) ctl[2] = 1;
                }
                stepping = false;
              } else {
                part = form_u2();
                stage = 1;
              }
            }
            if (!finished) {
              if (threadIdx.x == 0) ctl[0] = CTL_RUN;
              centre_from_r1(part);
            }
          } else {
            // ---- k = scaler (OUT + b2); stage combine on the resident state; next stage input -> xc ----
            const float dt = a.dt[step];
            const bool last_stage = (st == a.S - 1);
            const float* coef = last_stage ? a.b : a.a[st + 1];
            const float c_self = coef[st];
            float* srow = (last_stage && a_param.states && row_ok) ? a_param.states + (((size_t)(step + 1) * a_param.B + img) * N + r) * D : nullptr;
            float* frow = (last_eval && a_param.final_state && row_ok) ? a_param.final_state + ((size_t)img * N + r) * D : nullptr;
            float part = 0.f;
#pragma unroll 1
            for (int g = 0; g < ngq; ++g) {
              const int col0 = cw * DQ + g * 16;
              float v[16], acc[16];
              ptx::tmem_ld16(t_lane + T_R1 + col0, v);
              float bv[16];
              lds16(sB2 + col0, bv);
              float yv[16];
              lds16(yrow + col0, yv);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) {
                v[jj] = a.scaler * (v[jj] + bv[jj]);      // k of this stage
                acc[jj] = c_self * v[jj];
              }
              if (!last_stage && row_ok) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) kb[((size_t)st * D + col0 + jj) * 128 + r] = v[jj];   // a later stage combines it
              }
#pragma unroll 1
              for (int l = 0; l < st; ++l) {
                const float cl = coef[l];
                if (cl != 0.f && row_ok) {
#pragma unroll
                  for (int jj = 0; jj < 16; ++jj) acc[jj] = fmaf(cl, kb[((size_t)l * D + col0 + jj) * 128 + r], acc[jj]);
                }
              }
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) {
                v[jj] = fmaf(dt, acc[jj], yv[jj]);
                part += v[jj];
              }
              if (last_stage && row_ok) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj)
                  reinterpret_cast<float4*>(yrow + col0)[jj] = make_float4(v[4 * jj], v[4 * jj + 1], v[4 * jj + 2], v[4 * jj + 3]);
              }
              tmem_st16f(t_lane + T_R1 + col0, v);
            }
            centre_from_r1(part);
            // The updated state row is complete in shared memory (all four column shares, ordered by the
            // quadrant barrier inside centre_from_r1): one thread per row hands it to the bulk-copy engine.
            // Per-lane stores of 64 bytes at a 768-byte stride cost ~4600 LSU cycles per step here.
            if (cw == 0 && row_ok && (srow || frow)) {
              ptx::fence_async_shared();
              if (srow) bulk_store(srow, yrow, (uint32_t)D * 4);
              if (frow) bulk_store(frow, yrow, (uint32_t)D * 4);
              bulk_commit();
            }
          }
          done();
          RTR(0, j * 4 + 2);
        }
      }
    }
    if (cw == 0) bulk_wait_all();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (ADAPTIVE) {
    // no TMA write may land after the CTA exits: wait for the allocations issued past the last one consumed
    if (warp == LOADER)
      for (uint32_t g = (uint32_t)ctl[3]; g < ld_issued; ++g) ptx::mbar_wait(bar_full + (g & (NB - 1)), (g / NB) & 1);
  }
#ifdef RES_TRACE
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (int w = 0; w < 2; ++w)
      for (int i = 0; i < rtr_n[w]; ++i) printf("RTR %d %d %d %u\n", w, (int)rtr_id[w][i] >> 2, (int)rtr_id[w][i] & 3, rtr[w][i]);
#endif
  if (warp == PRODUCER) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem, 512);
  }
}

// Job list of one evaluation: per head [Q_h, MLP jobs, S_h, MLP jobs, PV_h], the C hidden chunks spread
// evenly over the 2H gaps, then F.  Adjacent jobs of one chain serialise (the second group waits for the
// first's compute phase): with C >= 2H only PV_h -> Q_{h+1} is left (measured 3 % faster than S_h -> PV_h).
bool build_sched(int D, int H, int C, Sched& sc) {
  int nj = 0, na = 0, last_a = -1, last_b = -1, c = 0;
  const int U = D / 64;
  auto push = [&](uint8_t kind, int arg, int dep) { sc.kind[nj] = kind; sc.arg[nj] = (uint8_t)arg; sc.dep[nj] = (int8_t)dep; return nj++; };
  auto add = [&](int kind, int ka, int arg, int size) {
    if (na < kMaxAllocs) sc.alloc[na] = Alloc{(uint16_t)arg, (uint8_t)kind, (uint8_t)ka, 0, (uint8_t)size, 0, 0};
    ++na;
  };
  auto w2 = [&](int col0) { add(2, 0, col0, U); };
  auto mlp_jobs = [&](int slot) {
    const int upto = (slot + 1) * C / (2 * H);
    for (; c < upto; ++c) {
      if (c > 0) { w2(D + (c - 1) * 128); w2(D + (c - 1) * 128 + 64); }
      for (int ka = 0; ka < U; ++ka) add(1, ka, c, 2);
      last_b = push(JOB_FC, c, last_b);
    }
  };
  for (int h = 0; h < H; ++h) {
    if (h > 0) w2((h - 1) * 64);
    for (int ka = 0; ka < U; ++ka) add(0, ka, h, 3);
    last_a = push(JOB_QKV, h, last_a);
    mlp_jobs(2 * h);
    last_a = push(JOB_S, h, last_a);
    mlp_jobs(2 * h + 1);
    last_a = push(JOB_PV, h, last_a);
  }
  w2((H - 1) * 64); w2(D + (C - 1) * 128); w2(D + (C - 1) * 128 + 64);
  push(JOB_F, 0, nj - 1);
  sc.n_jobs = nj;
  sc.n_allocs = na;
  if (na > kMaxAllocs) return false;
  // ring walk: no allocation wraps; every evaluation starts at slot 0
  int pos = 0;
  for (int i = 0; i < na; ++i) {
    if (pos + sc.alloc[i].size > NU) pos = 0;
    sc.alloc[i].off = (uint8_t)pos;
    pos += sc.alloc[i].size;
  }
  // steady state (allocation i of an evaluation, the previous evaluation before it): distance to the latest
  // older allocation that overlaps its slots, capped by the reuse distance of the barrier pair
  for (int i = 0; i < na; ++i) {
    int back = NB;
    for (int d = 1; d < NB; ++d) {
      const Alloc& o = sc.alloc[((i - d) % na + na) % na];
      if (o.off < sc.alloc[i].off + sc.alloc[i].size && sc.alloc[i].off < o.off + o.size) { back = d; break; }
    }
    sc.alloc[i].back = (uint8_t)back;
  }
  return true;
}

// null when the kernel covers the shape with `args_bytes` of arguments in shared memory, else what is out of range
const char* resident_envelope(const Plan& p, int args_bytes) {
  if (p.variant != ODEVIT_FIELD_PARALLEL) return "the PARALLEL field only";
  if (p.precision != ODEVIT_BF16) return "bf16 precision only";
  if (p.d != 64) return "head dim 64 only";
  if (p.D % 64 || p.D > 192) return "dim a multiple of 64, <= 192";
  if (p.hid % 128 || p.hid < 128) return "hidden a multiple of 128";
  if (p.N > 128 || p.N < 1) return "1..128 tokens";
  if (3 * p.H + p.hid / 128 + 1 > kMaxJobs || 4 * p.H + 5 * (p.hid / 128) > kMaxAllocs || 3 * p.D + p.hid > 0x7fff)
    return "the job list of one evaluation is too long";
  const int RA = (p.N + 15) / 16 * 16;
  if (smem_layout(RA, p.N, p.D, p.hid, args_bytes).total > 227 * 1024) return "the state does not fit in shared memory";
  return nullptr;
}

template <bool FULL, bool ADAPTIVE, class Args>
int launch_resident(const Args& a, const CUtensorMap& t1, const CUtensorMap& t2, int grid, cudaStream_t s) {
  const int bytes = smem_layout(a.RA, a.N, a.D, a.hid, res_smem_args<Args>()).total;
  static int configured_bytes = 0;
  if (bytes > configured_bytes) {
    ODV_CUDA(cudaFuncSetAttribute(solve_resident_kernel<FULL, ADAPTIVE>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    configured_bytes = bytes;
  }
  solve_resident_kernel<FULL, ADAPTIVE><<<grid, res_threads(FULL), bytes, s>>>(t1, t2, a);
  ODV_LAUNCH_CHECK();
  return 0;
}

int resident_tmaps(const Plan& p, const WeightBufs& wb, CUtensorMap* t1, CUtensorMap* t2) {
  const int R = 3 * p.D + p.hid, K2 = p.D + p.hid;
  ODV_TRY(make_tmap_2d_bf16(t1, wb.w1cat, p.D, R, p.D, 64, 64));
  ODV_TRY(make_tmap_2d_bf16(t2, wb.w2cat, K2, p.D, K2, 64, 64));
  return 0;
}

}  // namespace

size_t solve_resident_scratch_floats(const Plan& p) {
  const int sms = num_sms();
  const int grid = p.B < sms ? p.B : sms;
  return (size_t)grid * 3 * p.D * 128;
}

bool solve_resident_shape_ok(const Plan& p) { return resident_envelope(p, res_smem_args<ResArgs>()) == nullptr; }

const char* solve_resident_adaptive_envelope(const Plan& p) { return resident_envelope(p, res_smem_args<ResArgsAd>()); }

size_t solve_resident_adaptive_scratch_floats(const Plan& p) {
  const int sms = num_sms();
  const int grid = p.B < sms ? p.B : sms;
  return (size_t)grid * 8 * p.D * ((p.N + 15) / 16 * 16);
}

int solve_resident_adaptive(const Plan& p, const WeightBufs& wb, const float* x0, const double* t_out, int n_out,
                            double rtol, double atol, double first_step, int max_steps, float* states, int* nfe,
                            int* accepted, int* rejected, int* status, float* kbuf, int* next_image, cudaStream_t s) {
  ProfScope prof(KC_RESIDENT, s);
  ResArgsAd a;
  a.B = p.B; a.N = p.N; a.D = p.D; a.H = p.H; a.hid = p.hid;
  a.RA = (p.N + 15) / 16 * 16;
  a.NK = a.RA;
  a.n_out = n_out; a.max_steps = max_steps;
  a.scaler = p.scaler; a.rtol = (float)rtol; a.atol = (float)atol;
  a.first_step = first_step;
  for (int i = 0; i < 6; ++i) {
    a.b[i] = kDopri5.b[i];
    for (int j = 0; j < 6; ++j) a.a[i][j] = kDopri5.a[i][j];
  }
  for (int i = 0; i < 7; ++i) { a.c_err[i] = kDopri5Err[i]; a.c_mid[i] = kDopri5Mid[i]; }
  for (int i = 0; i < kMaxGrid; ++i) a.t_out[i] = i < n_out ? t_out[i] : 0.0;
  a.x0 = x0; a.states = states; a.b1cat = wb.b1cat; a.b2 = wb.b2; a.kbuf = kbuf; a.next_image = next_image;
  a.nfe = nfe; a.accepted = accepted; a.rejected = rejected; a.status = status;
  if (!build_sched(p.D, p.H, p.hid / 128, a.sc)) return set_error(ODEVIT_ERR_INVALID_ARG, "resident solver: allocation list too long");
  CUtensorMap t1, t2;
  ODV_TRY(resident_tmaps(p, wb, &t1, &t2));
  const int sms = num_sms();
  const int grid = p.B < sms ? p.B : sms;
  ODV_CUDA(cudaMemsetAsync(next_image, 0, sizeof(int), s));
  return p.N > 96 ? launch_resident<true, true>(a, t1, t2, grid, s) : launch_resident<false, true>(a, t1, t2, grid, s);
}

bool solve_resident_supports(const Plan& p, int n_grid, bool wants_p_traj, bool has_tape) {
  const char* env = getenv("ODEVIT_RESIDENT");
  if (env && env[0] == '0') return false;
  if (wants_p_traj || has_tape || p.split_out || p.p_attn > 0.f) return false;
  if (n_grid < 2 || n_grid > kMaxGrid) return false;
  return solve_resident_shape_ok(p);
}

int solve_resident(const Plan& p, const WeightBufs& wb, const Tableau& tb, const float* x0, const float* t_host,
                   int n_grid, float* states, float* final_state, float* p_last, float* kbuf, cudaStream_t s) {
  ProfScope prof(KC_RESIDENT, s);
  ResArgs a;
  a.B = p.B; a.N = p.N; a.D = p.D; a.H = p.H; a.hid = p.hid;
  a.RA = (p.N + 15) / 16 * 16;
  a.NK = a.RA;
  a.n_grid = n_grid; a.S = tb.S; a.scaler = p.scaler;
  for (int j = 0; j + 1 < n_grid; ++j) a.dt[j] = t_host[j + 1] - t_host[j];
  for (int i = 0; i < 4; ++i) {
    a.b[i] = tb.b[i];
    for (int j = 0; j < 4; ++j) a.a[i][j] = tb.a[i][j];
  }
  a.x0 = x0; a.states = states; a.final_state = final_state; a.p_last = p_last;
  a.b1cat = wb.b1cat; a.b2 = wb.b2; a.kbuf = kbuf;
  if (!build_sched(p.D, p.H, p.hid / 128, a.sc)) return set_error(ODEVIT_ERR_INVALID_ARG, "resident solver: allocation list too long");
  CUtensorMap t1, t2;
  ODV_TRY(resident_tmaps(p, wb, &t1, &t2));
  const int sms = num_sms();
  const int grid = p.B < sms ? p.B : sms;
  return p.N > 96 ? launch_resident<true, false>(a, t1, t2, grid, s) : launch_resident<false, false>(a, t1, t2, grid, s);
}

}  // namespace odevit
