// Row-wise and element-wise kernels of the hot path: all HBM-bound, one warp per token row,
// coalesced 128-byte warp accesses, no shared memory (no reuse beyond a row held in registers).
//
//   center_rows        CenterNorm / LayerNorm core       ode_transformer_gpt.py:79-83, macaron.py:80-82
//   softmax_rows       softmax over key positions        nn.MultiheadAttention explicit path (:228)
//   softmax_bwd_rows   its VJP (+ injected dP for the `attentions` output)
//   colsum_accum       bias-gradient column sums
//   vjp_combine        reverse-mode Runge-Kutta stage combination
//   fold / unfold      CenterNorm affine folded into the GEMM weights, and the chain rule back
#include "epilogue.cuh"
#include "internal.h"

namespace odevit {

namespace {

constexpr int MAX_PER_LANE = 32;  // rows up to 1024 elements are held in registers

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__global__ void __launch_bounds__(256) center_rows_kernel(const float* __restrict__ x, void* xc,
                                                          int xc_type, float* rstd_out, float eps,
                                                          int rows, int D) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (long long)row * D;
  float v[MAX_PER_LANE];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    v[i] = (c < D) ? xr[c] : 0.f;
    s += v[i];
  }
  const float mean = warp_sum(s) / (float)D;
  float rstd = 1.f;
  if (rstd_out) {
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAX_PER_LANE; ++i) {
      const int c = lane + i * 32;
      const float d = (c < D) ? v[i] - mean : 0.f;
      q += d * d;
    }
    rstd = rsqrtf(warp_sum(q) / (float)D + eps);
    if (lane == 0) rstd_out[row] = rstd;
  }
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    if (c < D) store_elem(xc, (long long)row * D + c, xc_type, (v[i] - mean) * rstd);
  }
}

// x - mean(x) -> bf16, D a multiple of 128: 16-byte loads, 8-byte stores (the CenterNorm prologue of every
// bf16 field evaluation; the affine and D/(D-1) live in the folded weights)
template <int CH>
__global__ void __launch_bounds__(256) center_rows_bf16_vec_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ xc,
                                                                   int rows, int D) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (long long)row * D);
  const int n4 = D >> 2;
  float4 v[CH];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + i * 32;
    v[i] = (c < n4) ? __ldg(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) / (float)D;
  uint2* out = reinterpret_cast<uint2*>(xc + (long long)row * D);
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + i * 32;
    if (c < n4) {
      const __nv_bfloat162 a = __floats2bfloat162_rn(v[i].x - mean, v[i].y - mean);
      const __nv_bfloat162 b = __floats2bfloat162_rn(v[i].z - mean, v[i].w - mean);
      out[c] = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    }
  }
}

__global__ void __launch_bounds__(256) softmax_rows_kernel(float* p, float* copy_to, long long rows,
                                                           int n) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* pr = p + row * n;
  float v[MAX_PER_LANE];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    v[i] = (c < n) ? pr[c] : -INFINITY;
    mx = fmaxf(mx, v[i]);
  }
  mx = warp_max(mx);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    v[i] = (c < n) ? expf(v[i] - mx) : 0.f;
    s += v[i];
  }
  const float inv = 1.f / warp_sum(s);
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    if (c < n) {
      const float o = v[i] * inv;
      pr[c] = o;
      if (copy_to) copy_to[row * n + c] = o;
    }
  }
}

__global__ void __launch_bounds__(256) softmax_bwd_rows_kernel(const float* __restrict__ p, float* dp,
                                                               const float* __restrict__ dpx,
                                                               long long rows, int n) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* pr = p + row * n;
  float* dr = dp + row * n;
  float pv[MAX_PER_LANE], gv[MAX_PER_LANE];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    pv[i] = 0.f;
    gv[i] = 0.f;
    if (c < n) {
      pv[i] = pr[c];
      gv[i] = dr[c];
      if (dpx) gv[i] += dpx[row * n + c];
    }
    s = fmaf(pv[i], gv[i], s);
  }
  s = warp_sum(s);
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    if (c < n) dr[c] = pv[i] * (gv[i] - s);
  }
}

__global__ void __launch_bounds__(128) colsum_kernel(const void* X, int x_type, long long ld, int rows,
                                                     int cols, int rows_per_block, float* acc) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c >= cols) return;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(rows, r0 + rows_per_block);
  float s = 0.f;
  for (int r = r0; r < r1; ++r) s += load_elem_rw(X, (long long)r * ld + c, x_type);
  atomicAdd(acc + c, s);
}

// bf16 fast path: a warp covers 256 columns with one 16-byte load per lane; the 8 warps of a block take interleaved
// rows of an `rpb`-row panel (8 independent loads in flight per lane) and meet in shared memory; one atomic per column
// and block (cols % 8 == 0, ld % 8 == 0).  Same-address atomics serialise in L2 (~27 cycles each): panels are kept
// tall (few blocks per column) and the memory-level parallelism comes from the unrolled loads instead.
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const __nv_bfloat16* __restrict__ X, long long ld,
                                                          int rows, int cols, int rpb, float* acc) {
  __shared__ float part[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c0 = blockIdx.x * 256 + lane * 8;
  const int r0 = blockIdx.y * rpb;
  const int r1 = min(rows, r0 + rpb);
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c0 < cols) {
    int r = r0 + warp;
    for (; r + 56 < r1; r += 64) {
      uint4 t[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) t[u] = *reinterpret_cast<const uint4*>(X + (long long)(r + 8 * u) * ld + c0);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const uint32_t w[4] = {t[u].x, t[u].y, t[u].z, t[u].w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          s[2 * i] += __uint_as_float(w[i] << 16);
          s[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
        }
      }
    }
    for (; r < r1; r += 8) {
      const uint4 t = *reinterpret_cast<const uint4*>(X + (long long)r * ld + c0);
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        s[2 * i] += __uint_as_float(w[i] << 16);
        s[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) part[warp][lane * 8 + i] = s[i];
  __syncthreads();
  {
    const int c = threadIdx.x;
    const int col = blockIdx.x * 256 + c;
    if (col < cols) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += part[w][c];
      atomicAdd(acc + col, t);
    }
  }
}

__global__ void __launch_bounds__(256) vjp_combine_kernel(CombineArgs a, int rows, int D) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const long long base = (long long)row * D;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    if (c >= D) continue;
    float v = 0.f;
    for (int t = 0; t < a.n_terms; ++t) v = fmaf(a.coef[t], a.term[t][base + c], v);
    if (a.out_f32) a.out_f32[base + c] = v;
    if (a.out_dd) store_elem(a.out_dd, base + c, a.dd_type, a.dd_scale * v);
  }
}

__global__ void __launch_bounds__(256) drop_pair_kernel(const void* x, void* out1, void* out2, int type, Drop d1,
                                                        Drop d2, long long n, int D) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const uint32_t r = (uint32_t)(i / D), c = (uint32_t)(i % D);
    const float v = load_elem_rw(x, i, type);
    store_elem(out1, i, type, d1.thresh ? v * drop_factor(d1, r, c) : v);
    store_elem(out2, i, type, d2.thresh ? v * drop_factor(d2, r, c) : v);
  }
}

// bf16 fast path of drop_pair_kernel: 8 elements (16 bytes) per thread and pass, 64-bit index arithmetic once per 8
// (the element-wise form above moved 2 bytes per access with a 64-bit division per element: 57 us at the bench shape)
__global__ void __launch_bounds__(256) drop_pair_bf16x8_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out1,
                                                               __nv_bfloat16* __restrict__ out2, Drop d1, Drop d2, long long n8, int D) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n8; i += stride) {
    const long long e0 = i * 8;
    const uint32_t r = (uint32_t)(e0 / D), c = (uint32_t)(e0 - (long long)r * D);   // D % 8 == 0: the 8 share a row
    const uint4 t = *reinterpret_cast<const uint4*>(x + e0);
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
    uint32_t o1[4], o2[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float a = __uint_as_float(w[k] << 16), b = __uint_as_float(w[k] & 0xffff0000u);
      const float a1 = d1.thresh ? a * drop_factor(d1, r, c + 2 * k) : a, b1 = d1.thresh ? b * drop_factor(d1, r, c + 2 * k + 1) : b;
      const float a2 = d2.thresh ? a * drop_factor(d2, r, c + 2 * k) : a, b2 = d2.thresh ? b * drop_factor(d2, r, c + 2 * k + 1) : b;
      const __nv_bfloat162 h1 = __floats2bfloat162_rn(a1, b1), h2 = __floats2bfloat162_rn(a2, b2);
      o1[k] = *reinterpret_cast<const uint32_t*>(&h1);
      o2[k] = *reinterpret_cast<const uint32_t*>(&h2);
    }
    *reinterpret_cast<uint4*>(out1 + e0) = make_uint4(o1[0], o1[1], o1[2], o1[3]);
    *reinterpret_cast<uint4*>(out2 + e0) = make_uint4(o2[0], o2[1], o2[2], o2[3]);
  }
}

__global__ void __launch_bounds__(256) drop_rows_inplace_kernel(void* x, int type, Drop d, long long n, int D) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride)
    store_elem(x, i, type, load_elem_rw(x, i, type) * drop_factor(d, (uint32_t)(i / D), (uint32_t)(i % D)));
}

__global__ void resolve_drop_keys_kernel(const uint32_t* __restrict__ seed, uint32_t* __restrict__ table, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) table[i] = drop_site_key(seed[0], seed[1], i / DS_SITES, i % DS_SITES);
}

// state[0] base seed, state[1] step counter, state[2] the seed of the current step (splitmix64 of base + counter)
__global__ void drop_state_advance_kernel(unsigned long long* state) {
  const unsigned long long c = state[1] + 1ull;
  unsigned long long z = state[0] + c * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  state[1] = c;
  state[2] = z ^ (z >> 31);
}

__global__ void __launch_bounds__(256) drop_inplace_kernel(float* p, float* copy_to, Drop d, long long total, int n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const float v = p[i] * drop_factor(d, (uint32_t)(i / n), (uint32_t)(i % n));
    p[i] = v;
    if (copy_to) copy_to[i] = v;
  }
}

__global__ void axpy_kernel(float* y, const float* __restrict__ x, float a, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) y[i] = fmaf(a, x[i], y[i]);
}

// ---- finite-difference curvature of the trajectory ------------------------------------------
// compute_upper_bound_by_fininte_difference (ode_transformer_gpt.py:529-543) forms the second
// difference (s[j+2] - 2 s[j+1] + s[j]) / dt^2 over the whole [T,B,N,D] trajectory, its inf-norm over
// D and the max over time: in PyTorch that is ~6 full-trajectory passes.  Here one warp owns a token
// row (b,n), walks the T rows once with a 3-row register window and emits per_seq[b,n]; every state
// element is read exactly once (algorithmic bytes = T*B*N*D*4).
// out[row] = <P[row, :], G[row, :]>: the part of the softmax VJP's row term that comes from a cotangent on
// the exported attention map (warp per row)
__global__ void __launch_bounds__(256) rowdot_rows_kernel(const float* __restrict__ P, const float* __restrict__ G,
                                                          float* __restrict__ out, long long rows, int n) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* p = P + row * n;
  const float* g = G + row * n;
  float acc = 0.f;
  for (int c = lane; c < n; c += 32) acc = fmaf(p[c], g[c], acc);
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

// JaSMin statistic of exported attention maps (ode_transformer_gpt.py:419-456, detached by the reference):
// one CTA per map slice (evaluation, image, head), 8 warps over its N query rows.  Per row: clamp to
// [1e-12, 1], renormalise by (sum + 1e-12), the k+1 largest entries by repeated warp arg-max over a
// shared-memory copy of the row (one instance removed per round, so ties keep their multiplicity, as in
// the reference's sort), g_j = x_(j) (1 - x_(j) + x_(j+1)), row value log(g_1 / (g_k + 1e-12) + 1e-12)
// (k = 0: log(g_1 + 1e-12)); the CTA writes the maximum over the rows.
__global__ void __launch_bounds__(256) jasmin_rowmax_kernel(const float* __restrict__ P, int N, int k, float* __restrict__ out) {
  extern __shared__ float jas_rows[];
  __shared__ float warp_best[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* row = jas_rows + warp * N;
  const float* base = P + (size_t)blockIdx.x * N * N;
  const int need = (k == 0) ? 2 : k + 1;
  float best = -INFINITY;
  for (int r = warp; r < N; r += 8) {
    const float* src = base + (size_t)r * N;
    float sum = 0.f;
    for (int c = lane; c < N; c += 32) {
      const float v = fminf(fmaxf(src[c], 1e-12f), 1.f);
      row[c] = v;
      sum += v;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float den = sum + 1e-12f;
    __syncwarp();
    float x1 = 0.f, x2 = 0.f, xk = 0.f, xk1 = 0.f;
    for (int t = 1; t <= need && t <= N; ++t) {
      float m = -INFINITY;
      int mi = 0x7fffffff;
      for (int c = lane; c < N; c += 32) {
        const float v = row[c];
        if (v > m) { m = v; mi = c; }
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, m, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
      }
      if (lane == 0) row[mi] = -INFINITY;
      __syncwarp();
      const float x = m / den;
      if (t == 1) x1 = x;
      if (t == 2) x2 = x;
      if (t == k) xk = x;
      if (t == k + 1) xk1 = x;
    }
    const float g1 = x1 * (1.f - x1 + x2);
    float v;
    if (k == 0) v = logf(g1 + 1e-12f);
    else v = logf(g1 / (xk * (1.f - xk + xk1) + 1e-12f) + 1e-12f);
    best = fmaxf(best, v);
    __syncwarp();
  }
  if (lane == 0) warp_best[warp] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    float b = warp_best[0];
    for (int w = 1; w < 8; ++w) b = fmaxf(b, warp_best[w]);
    out[blockIdx.x] = b;
  }
}

template <int CH>  // CH float4 chunks per lane: D <= 128*CH
__global__ void __launch_bounds__(256) fd_curvature_kernel(const float* __restrict__ states, int T, long long rows,
                                                           int D, float dt2, float* __restrict__ per_seq) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const long long stride = rows * D;
  const float* base = states + row * D;
  float4 w[3][CH];
  auto load = [&](float4* dst, int j) {
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      const int c = (lane + i * 32) * 4;
      dst[i] = (c < D) ? __ldcs(reinterpret_cast<const float4*>(base + (long long)j * stride + c))
                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  load(w[0], 0);
  load(w[1], 1);
  float mx = 0.f;
  // the window rotates through the three register rows; unrolled by 3 so the indices stay static
  auto step = [&](float4* a, float4* b, float4* c, int j) {
    load(c, j);
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      // same association as the reference: (s[j+2] - 2*s[j+1]) + s[j]
      mx = fmaxf(mx, fabsf((c[i].x - 2.f * b[i].x) + a[i].x));
      mx = fmaxf(mx, fabsf((c[i].y - 2.f * b[i].y) + a[i].y));
      mx = fmaxf(mx, fabsf((c[i].z - 2.f * b[i].z) + a[i].z));
      mx = fmaxf(mx, fabsf((c[i].w - 2.f * b[i].w) + a[i].w));
    }
  };
  int j = 2;
  for (; j + 2 < T; j += 3) {
    step(w[0], w[1], w[2], j);
    step(w[1], w[2], w[0], j + 1);
    step(w[2], w[0], w[1], j + 2);
  }
  if (j < T) { step(w[0], w[1], w[2], j); ++j; }
  if (j < T) { step(w[1], w[2], w[0], j); ++j; }
  mx = warp_max(mx);
  if (lane == 0) per_seq[row] = mx / dt2;
}

// ---- LayerNorm rows (MACARON) ---------------------------------------------------------------
__global__ void __launch_bounds__(256) ln_rows_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                      const float* __restrict__ b, void* out, int out_type,
                                                      float eps, int rows, int D) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (long long)row * D;
  float v[MAX_PER_LANE];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    v[i] = (c < D) ? xr[c] : 0.f;
    s += v[i];
  }
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    const float d = (c < D) ? v[i] - mean : 0.f;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    if (c < D) store_elem(out, (long long)row * D + c, out_type, (v[i] - mean) * rstd * w[c] + b[c]);
  }
}

// One warp walks rows row0, row0+stride, ...; the per-column sums for dw / db stay in registers and
// meet the other warps of the block in shared memory, then one atomic per column and block.
__global__ void __launch_bounds__(256) ln_bwd_rows_kernel(LnBwdArgs a, int rows, int D) {
  __shared__ float red[8][32 * MAX_PER_LANE];  // 32 KB: per-warp column partials
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float dwp[MAX_PER_LANE], dbp[MAX_PER_LANE];
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) { dwp[i] = 0.f; dbp[i] = 0.f; }
  for (int row = blockIdx.x * 8 + warp; row < rows; row += gridDim.x * 8) {
    const long long base = (long long)row * D;
    float xh[MAX_PER_LANE], dh[MAX_PER_LANE];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAX_PER_LANE; ++i) {
      const int c = lane + i * 32;
      xh[i] = (c < D) ? a.x[base + c] : 0.f;
      s += xh[i];
    }
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAX_PER_LANE; ++i) {
      const int c = lane + i * 32;
      xh[i] = (c < D) ? xh[i] - mean : 0.f;
      q += xh[i] * xh[i];
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)D + a.eps);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < MAX_PER_LANE; ++i) {
      const int c = lane + i * 32;
      xh[i] *= rstd;
      const float dn = (c < D) ? a.dn[base + c] : 0.f;
      dwp[i] = fmaf(dn, xh[i], dwp[i]);
      dbp[i] += dn;
      dh[i] = (c < D) ? dn * a.w[c] : 0.f;
      s1 += dh[i];
      s2 = fmaf(dh[i], xh[i], s2);
    }
    s1 = warp_sum(s1) / (float)D;
    s2 = warp_sum(s2) / (float)D;
#pragma unroll
    for (int i = 0; i < MAX_PER_LANE; ++i) {
      const int c = lane + i * 32;
      if (c >= D) continue;
      float g = rstd * (dh[i] - s1 - xh[i] * s2);
      if (a.g_in) g += a.g_in[base + c];
      if (a.g_out) a.g_out[base + c] = g;
      if (a.dd_out) store_elem(a.dd_out, base + c, a.dd_type, a.dd_coef * g);
    }
  }
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    float* dst = which ? a.db : a.dw;
    if (!dst) continue;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < MAX_PER_LANE; ++i) {
      const int c = lane + i * 32;
      if (c < D) red[warp][c] = which ? dbp[i] : dwp[i];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += 256) {
      float t = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += red[k][c];
      atomicAdd(dst + c, t);
    }
  }
}

template <int EPI>
__global__ void __launch_bounds__(256) rk_apply_kernel(const __grid_constant__ Epi e, const float* __restrict__ v,
                                                       long long n, int D) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) epi_apply<EPI, false>(e, (int)(i / D), (int)(i % D), v[i], 0, 0);
}

// ---- L2 attention pieces ---------------------------------------------------------------------
__global__ void __launch_bounds__(256) head_sqnorm_kernel(const void* qkv, int type, float* sq, int B, int N, int H,
                                                          int D) {
  // one warp per (token row, head, q|k)
  const long long wid = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const long long total = (long long)B * N * H * 2;
  if (wid >= total) return;
  const int which = (int)(wid % 2);
  const int h = (int)((wid / 2) % H);
  const long long row = wid / (2 * H);
  const int d = D / H;
  const long long base = row * 3 * D + (long long)which * D + (long long)h * d;
  float s = 0.f;
  for (int c = lane; c < d; c += 32) {
    const float v = load_elem_rw(qkv, base + c, type);
    s = fmaf(v, v, s);
  }
  s = warp_sum(s);
  if (lane == 0) {
    const long long b = row / N, i = row % N;
    sq[(long long)which * B * H * N + (b * H + h) * N + i] = s;
  }
}

__global__ void __launch_bounds__(256) l2_prob_rows_kernel(float* p, const float* __restrict__ sq, float scale,
                                                           float* copy_to, long long rows, int n) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* pr = p + row * n;
  const float q2 = sq[row];
  const float* k2 = sq + rows + (row / n) * n;  // row = (b*H + h)*N + i
  float v[MAX_PER_LANE];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    v[i] = 0.f;
    if (c < n) {
      const float dist2 = q2 + k2[c] - 2.f * pr[c];
      v[i] = expf(-dist2 * scale);
    }
    s += v[i];
  }
  const float z = warp_sum(s) + 1e-8f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) {
    const int c = lane + i * 32;
    if (c < n) {
      const float o = v[i] / z;
      pr[c] = o;
      if (copy_to) copy_to[row * n + c] = o;
    }
  }
}

// one block per (image, head): row / column sums of ds [N,N] into shared memory, then the rank-one fixes
__global__ void __launch_bounds__(256) l2_vjp_fix_kernel(const float* __restrict__ ds, const void* qkv, int type,
                                                         void* dz, int R, float coef, int N, int H, int D) {
  extern __shared__ float sm[];
  float* rs = sm;
  float* cs = sm + N;
  const int bh = blockIdx.x, b = bh / H, h = bh % H, d = D / H;
  const float* m = ds + (long long)bh * N * N;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = warp; i < N; i += 8) {
    float s = 0.f;
    for (int j = lane; j < N; j += 32) s += m[(long long)i * N + j];
    s = warp_sum(s);
    if (lane == 0) rs[i] = s;
  }
  for (int j = threadIdx.x; j < N; j += 256) {
    float s = 0.f;
    for (int i = 0; i < N; ++i) s += m[(long long)i * N + j];
    cs[j] = s;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < N * d; e += 256) {
    const int i = e / d, c = e % d;
    const long long row = (long long)b * N + i;
    const long long qi = row * 3 * D + (long long)h * d + c;
    const long long zi = row * R + (long long)h * d + c;
    const float q = load_elem_rw(qkv, qi, type), k = load_elem_rw(qkv, qi + D, type);
    store_elem(dz, zi, type, load_elem_rw(dz, zi, type) - coef * rs[i] * q);
    store_elem(dz, zi + D, type, load_elem_rw(dz, zi + D, type) - coef * cs[i] * k);
  }
}

// ---- MACARON gradient assembly ------------------------------------------------------------------
// block = one row i of G2 [D, D+hid]: dWo[i,:] += rs*G2[i,:D], dW2[i,:] += rs*G2[i,D:], biases, and the
// res_scale gradient <Wo,G2a> + <W2,G2b> + <bo,c2> + <b2,c3> (block partial -> one atomic)
__global__ void __launch_bounds__(128) unfold_w2_macaron_kernel(UnfoldArgs a, odevit_weights w, odevit_weight_grads g) {
  const int D = a.D, hid = a.hid, K2 = D + hid;
  const int i = blockIdx.x;
  const float rs = *w.res_scale;
  float dot = 0.f;
  for (int c = threadIdx.x; c < K2; c += 128) {
    const float v = a.G2[(long long)i * K2 + c];
    if (c < D) {
      if (g.out_proj_w) g.out_proj_w[(long long)i * D + c] += rs * v;
      dot = fmaf(w.out_proj_w[(long long)i * D + c], v, dot);
    } else {
      if (g.fc2_w) g.fc2_w[(long long)i * hid + (c - D)] += rs * v;
      dot = fmaf(w.fc2_w[(long long)i * hid + (c - D)], v, dot);
    }
  }
  if (threadIdx.x == 0) {
    if (g.out_proj_b) g.out_proj_b[i] += rs * a.c2[i];
    if (g.fc2_b) g.fc2_b[i] += rs * a.c3[i];
    if (w.out_proj_b) dot = fmaf(w.out_proj_b[i], a.c2[i], dot);
    if (w.fc2_b) dot = fmaf(w.fc2_b[i], a.c3[i], dot);
  }
  __shared__ float red[4];
  dot = warp_sum(dot);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dot;
  __syncthreads();
  if (threadIdx.x == 0 && g.res_scale) atomicAdd(g.res_scale, red[0] + red[1] + red[2] + red[3]);
}

// ---- weight folding (PARALLEL variant) -------------------------------------------------------
// CenterNorm is affine in (x - mean):  n = s*(x-mean)*w + b  with s = D/(D-1)          (:77-83)
//   n_attn @ W_in^T = (x-mean) @ (s * W_in * diag(w_a))^T + W_in @ b_a
// so the packed in-proj and fc1 share ONE left operand xc = x - mean and become ONE GEMM over the
// row-concatenated, column-scaled weight  W1cat = [qs*s*W_in*diag(w_a) ; s*W1*diag(w_m)]  with
// bias  b1cat = [qs*(W_in b_a + b_in) ; W1 b_m + b_fc1]  (qs = 1/sqrt(d) on the Wq rows: the
// q*(1/sqrt(d)) of nn.MultiheadAttention).  out_proj and fc2 concatenate along K:
//   [O | h] @ [Wo | W2]^T.
__global__ void __launch_bounds__(128) fold_w1_kernel(FoldArgs a, odevit_weights w) {
  const int D = a.D;
  const int j = blockIdx.x;
  const bool attn = j < 3 * D;
  const float* Wrow = attn ? w.in_proj_w + (long long)j * D : w.fc1_w + (long long)(j - 3 * D) * D;
  const float* nw = attn ? w.norm_a_w : w.norm_b_w;
  const float* nb = attn ? w.norm_a_b : w.norm_b_b;
  const float* msc = attn ? w.mod_attn_scale : w.mod_mlp_scale;
  const float* msh = attn ? w.mod_attn_shift : w.mod_mlp_shift;
  const float* lb = attn ? w.in_proj_b : w.fc1_b;
  const bool fn = a.fold_norm;
  const float s_cn = fn ? (float)D / ((float)D - 1.f) : 1.f;
  const float qs = (j < D) ? a.q_scale : 1.f;
  float dot = 0.f, fsum = 0.f;
  for (int i = threadIdx.x; i < D; i += 128) {
    float we = fn ? nw[i] : 1.f, be = fn ? nb[i] : 0.f;
    if (fn && msc) { we *= (1.f + msc[i]); be *= (1.f + msc[i]); }
    if (fn && msh) be += msh[i];
    const float wv = Wrow[i];
    const float f = qs * s_cn * wv * we;
    if (!fn) store_elem(a.w1cat, (long long)j * D + i, a.w_type, f);
    fsum += f;
    dot = fmaf(wv, be, dot);
  }
  __shared__ float red[4], red2[4];
  dot = warp_sum(dot);
  fsum = warp_sum(fsum);
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = dot; red2[threadIdx.x >> 5] = fsum; }
  __syncthreads();
  if (fn) {
    // The rows of W1cat are stored CENTRED over D (W1cat (I - 11^T/D)): the product with the left operand then does not
    // change when a constant is added to a row of that operand -- (x - c 1^T)(I - 11^T/D) = x (I - 11^T/D) for ANY c --
    // so the centring of CenterNorm lives in the weights and the operand may be the plain bf16 copy of the state that the
    // previous GEMM's epilogue writes (api.cu: `xc_ready`); an exactly centred operand gives the same product as before.
    const float mean = (red2[0] + red2[1] + red2[2] + red2[3]) / (float)D;
    for (int i = threadIdx.x; i < D; i += 128) {
      float we = nw[i];
      if (msc) we *= (1.f + msc[i]);
      store_elem(a.w1cat, (long long)j * D + i, a.w_type, qs * s_cn * Wrow[i] * we - mean);
    }
  }
  if (threadIdx.x == 0) {
    float t = red[0] + red[1] + red[2] + red[3];
    if (lb) t += lb[j - (attn ? 0 : 3 * D)];
    a.b1cat[j] = qs * t;
    // row mean for the transposed, row-centred copy (fold_w1_transpose_kernel: a thread-per-element store at stride R
    // here scattered 2.4 M two-byte writes and made the fold a 58 us kernel)
    if (a.fmean) a.fmean[j] = fn ? (red2[0] + red2[1] + red2[2] + red2[3]) / (float)D : 0.f;
  }
}

// w1catT[i, j] = f(j, i) - fmean[j] for one 32 x 32 tile of (j, i): rows of W read coalesced, the transposed tile written
// coalesced (32 consecutive j per output row) through shared memory; f is recomputed with fold_w1_kernel's expression.
__global__ void __launch_bounds__(256) fold_w1_transpose_kernel(FoldArgs a, odevit_weights w) {
  const int D = a.D, hid = a.hid, R = 3 * D + hid;
  const int j0 = blockIdx.x * 32, i0 = blockIdx.y * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool fn = a.fold_norm;
  const float s_cn = fn ? (float)D / ((float)D - 1.f) : 1.f;
  __shared__ float tile[32][33];
  for (int r = warp; r < 32; r += 8) {
    const int j = j0 + r, i = i0 + lane;
    float v = 0.f;
    if (j < R && i < D) {
      const bool attn = j < 3 * D;
      const float* Wrow = attn ? w.in_proj_w + (long long)j * D : w.fc1_w + (long long)(j - 3 * D) * D;
      const float* nw = attn ? w.norm_a_w : w.norm_b_w;
      const float* msc = attn ? w.mod_attn_scale : w.mod_mlp_scale;
      float we = fn ? nw[i] : 1.f;
      if (fn && msc) we *= (1.f + msc[i]);
      const float qs = (j < D) ? a.q_scale : 1.f;
      v = qs * s_cn * Wrow[i] * we - a.fmean[j];
    }
    tile[r][lane] = v;
  }
  __syncthreads();
  for (int c = warp; c < 32; c += 8) {
    const int i = i0 + c, j = j0 + lane;
    if (i < D && j < R) store_elem(a.w1catT, (long long)i * R + j, a.w_type, tile[lane][c]);
  }
}

__global__ void __launch_bounds__(128) fold_w2_kernel(FoldArgs a, odevit_weights w) {
  const int D = a.D, hid = a.hid, K2 = D + hid;
  const int i = blockIdx.x;
  for (int c = threadIdx.x; c < K2; c += 128) {
    const float v = (c < D) ? w.out_proj_w[(long long)i * D + c] : w.fc2_w[(long long)i * hid + (c - D)];
    store_elem(a.w2cat, (long long)i * K2 + c, a.w_type, v);
  }
  if (threadIdx.x == 0) {
    float b = 0.f;
    if (w.out_proj_b) b += w.out_proj_b[i];
    if (w.fc2_b) b += w.fc2_b[i];
    a.b2[i] = b;
  }
}

// w2catT[c, i] = [Wo | W2][i, c] through a 32 x 32 shared-memory tile (coalesced reads and writes)
__global__ void __launch_bounds__(256) fold_w2_transpose_kernel(FoldArgs a, odevit_weights w) {
  const int D = a.D, hid = a.hid, K2 = D + hid;
  const int i0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __shared__ float tile[32][33];
  for (int r = warp; r < 32; r += 8) {
    const int i = i0 + r, c = c0 + lane;
    float v = 0.f;
    if (i < D && c < K2) v = (c < D) ? w.out_proj_w[(long long)i * D + c] : w.fc2_w[(long long)i * hid + (c - D)];
    tile[r][lane] = v;
  }
  __syncthreads();
  for (int r = warp; r < 32; r += 8) {
    const int c = c0 + r, i = i0 + lane;
    if (c < K2 && i < D) store_elem(a.w2catT, (long long)c * D + i, a.w_type, tile[lane][r]);
  }
}

// ---- gradient un-folding ---------------------------------------------------------------------
//   G1 = sum dz^T xc,  c1 = colsum dz,  G2 = sum dd^T [O|h],  c2 = colsum dd   (over all f-evals)
//   dW[j,i]  = qs_j * (s*w_eff[i]*G1[j,i] + c1[j]*b_eff[i])
//   dw[i]    = (1+msc[i]) * sum_j qs_j*s*W[j,i]*G1[j,i]
//   db[i]    = (1+msc[i]) * sum_j qs_j*W[j,i]*c1[j]
__global__ void __launch_bounds__(128) unfold_w1_kernel(UnfoldArgs a, odevit_weights w,
                                                        odevit_weight_grads g) {
  const int D = a.D, hid = a.hid;
  const int j = blockIdx.x;
  const bool attn = j < 3 * D;
  const int jr = attn ? j : j - 3 * D;
  float* dW = attn ? g.in_proj_w : g.fc1_w;
  const float* nw = attn ? w.norm_a_w : w.norm_b_w;
  const float* nb = attn ? w.norm_a_b : w.norm_b_b;
  const float* msc = attn ? w.mod_attn_scale : w.mod_mlp_scale;
  const float* msh = attn ? w.mod_attn_shift : w.mod_mlp_shift;
  const bool fn = (a.c3 == nullptr);  // MACARON passes c3 and has no folded norms
  const float s_cn = fn ? (float)D / ((float)D - 1.f) : 1.f;
  const float qs = (j < D) ? a.q_scale : 1.f;
  const float cj = a.c1[j];
  if (fn) {
    // G1 was accumulated against operand rows that carry arbitrary constants (fold_w1_kernel): the gradient of the
    // folded weight is G1 (I - 11^T/D).  Centred IN PLACE: unfold_norm_kernel, launched next, reads the same rows.
    float rs = 0.f;
    for (int i = threadIdx.x; i < D; i += 128) rs += a.G1[(long long)j * D + i];
    __shared__ float red[4];
    rs = warp_sum(rs);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = rs;
    __syncthreads();
    const float mean = (red[0] + red[1] + red[2] + red[3]) / (float)D;
    float* G1w = const_cast<float*>(a.G1);
    for (int i = threadIdx.x; i < D; i += 128) G1w[(long long)j * D + i] -= mean;
    __syncthreads();
  }
  if (dW) {
    for (int i = threadIdx.x; i < D; i += 128) {
      float we = fn ? nw[i] : 1.f, be = fn ? nb[i] : 0.f;
      if (fn && msc) { we *= (1.f + msc[i]); be *= (1.f + msc[i]); }
      if (fn && msh) be += msh[i];
      dW[(long long)jr * D + i] += qs * (s_cn * we * a.G1[(long long)j * D + i] + cj * be);
    }
  }
  if (threadIdx.x == 0) {
    float* db = attn ? g.in_proj_b : g.fc1_b;
    if (db) db[jr] += qs * cj;
  }
  (void)hid;
}

// one block = 128 columns i x a slice of kUnfoldRows rows j of G1; partial sums meet through atomics
constexpr int kUnfoldRows = 16;   // (64 left 288 blocks of 64 dependent row steps each: 38 us of latency for 19 MB)
__global__ void __launch_bounds__(128) unfold_norm_kernel(UnfoldArgs a, odevit_weights w,
                                                          odevit_weight_grads g) {
  const int D = a.D, hid = a.hid;
  const int i = blockIdx.x * 128 + threadIdx.x;
  if (i >= D) return;
  const int j0 = blockIdx.y * kUnfoldRows;
  const int j1 = min(3 * D + hid, j0 + kUnfoldRows);
  const float s_cn = (float)D / ((float)D - 1.f);
  const float q = a.q_scale;
  float dwa = 0.f, dba = 0.f, dwm = 0.f, dbm = 0.f;
#pragma unroll 8
  for (int j = j0; j < j1; ++j) {
    const float g1 = a.G1[(long long)j * D + i], cj = a.c1[j];
    if (j < 3 * D) {
      const float wv = ((j < D) ? q : 1.f) * w.in_proj_w[(long long)j * D + i];
      dwa = fmaf(wv, g1, dwa);
      dba = fmaf(wv, cj, dba);
    } else {
      const float wv = w.fc1_w[(long long)(j - 3 * D) * D + i];
      dwm = fmaf(wv, g1, dwm);
      dbm = fmaf(wv, cj, dbm);
    }
  }
  const float ma = w.mod_attn_scale ? 1.f + w.mod_attn_scale[i] : 1.f;
  const float mm = w.mod_mlp_scale ? 1.f + w.mod_mlp_scale[i] : 1.f;
  if (j0 < 3 * D) {
    if (g.norm_a_w) atomicAdd(g.norm_a_w + i, ma * s_cn * dwa);
    if (g.norm_a_b) atomicAdd(g.norm_a_b + i, ma * dba);
  }
  if (j1 > 3 * D) {
    if (g.norm_b_w) atomicAdd(g.norm_b_w + i, mm * s_cn * dwm);
    if (g.norm_b_b) atomicAdd(g.norm_b_b + i, mm * dbm);
  }
}

__global__ void __launch_bounds__(128) unfold_w2_kernel(UnfoldArgs a, odevit_weight_grads g) {
  const int D = a.D, hid = a.hid, K2 = D + hid;
  const int i = blockIdx.x;
  for (int c = threadIdx.x; c < K2; c += 128) {
    const float v = a.G2[(long long)i * K2 + c];
    if (c < D) { if (g.out_proj_w) g.out_proj_w[(long long)i * D + c] += v; }
    else if (g.fc2_w) g.fc2_w[(long long)i * hid + (c - D)] += v;
  }
  if (threadIdx.x == 0) {
    if (g.out_proj_b) g.out_proj_b[i] += a.c2[i];
    if (g.fc2_b) g.fc2_b[i] += a.c2[i];
  }
}

}  // namespace

int center_rows(const float* x, void* xc, int xc_type, float* rstd_out, float eps, int rows, int D,
                cudaStream_t s) {
  ProfScope prof(KC_CENTER, s);
  if (D > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "center_rows: D=%d > 1024", D);
  if (xc_type == DT_BF16 && !rstd_out && D % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(xc) & 7) == 0) {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(xc);
    const int ch = (D / 4 + 31) / 32;
    if (ch <= 2) center_rows_bf16_vec_kernel<2><<<(rows + 7) / 8, 256, 0, s>>>(x, o, rows, D);
    else if (ch <= 4) center_rows_bf16_vec_kernel<4><<<(rows + 7) / 8, 256, 0, s>>>(x, o, rows, D);
    else if (ch <= 6) center_rows_bf16_vec_kernel<6><<<(rows + 7) / 8, 256, 0, s>>>(x, o, rows, D);
    else center_rows_bf16_vec_kernel<8><<<(rows + 7) / 8, 256, 0, s>>>(x, o, rows, D);
  } else {
    center_rows_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, xc, xc_type, rstd_out, eps, rows, D);
  }
  ODV_LAUNCH_CHECK();
  return 0;
}

int softmax_rows(float* p, float* copy_to, long long rows, int n, cudaStream_t s) {
  ProfScope prof(KC_SOFTMAX, s);
  if (n > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "softmax_rows: N=%d > 1024", n);
  softmax_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(p, copy_to, rows, n);
  ODV_LAUNCH_CHECK();
  return 0;
}

int softmax_bwd_rows(const float* p, float* dp, const float* dpx, long long rows, int n, cudaStream_t s) {
  ProfScope prof(KC_BWD_SOFTMAX, s);
  if (n > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "softmax_bwd_rows: N=%d > 1024", n);
  softmax_bwd_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(p, dp, dpx, rows, n);
  ODV_LAUNCH_CHECK();
  return 0;
}

int colsum_accum(const void* X, int x_type, long long ld, int rows, int cols, float* acc, cudaStream_t s) {
  ProfScope prof(KC_BWD_COLSUM, s);
  if (x_type == DT_BF16 && cols % 8 == 0 && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
    // rows per block: 256 for wide matrices, fewer for narrow ones so that there are at least two blocks per SM
    const int col_blocks = (cols + 255) / 256;
    int rpb = 256;
    while (rpb > 64 && (long long)col_blocks * ((rows + rpb - 1) / rpb) < 296) rpb >>= 1;
    dim3 grid(col_blocks, (rows + rpb - 1) / rpb);
    colsum_bf16_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(X), ld, rows, cols, rpb, acc);
    ODV_LAUNCH_CHECK();
    return 0;
  }
  const int rpb = 256;
  dim3 grid((cols + 127) / 128, (rows + rpb - 1) / rpb);
  colsum_kernel<<<grid, 128, 0, s>>>(X, x_type, ld, rows, cols, rpb, acc);
  ODV_LAUNCH_CHECK();
  return 0;
}

int vjp_combine(const CombineArgs& a, int rows, int D, cudaStream_t s) {
  ProfScope prof(KC_COMBINE, s);
  if (D > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "vjp_combine: D=%d > 1024", D);
  vjp_combine_kernel<<<(rows + 7) / 8, 256, 0, s>>>(a, rows, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

int drop_pair_rows(const void* x, void* out1, void* out2, int type, Drop d1, Drop d2, int rows, int D, cudaStream_t s) {
  ProfScope prof(KC_COMBINE, s);
  const long long n = (long long)rows * D;
  if (type == DT_BF16 && D % 8 == 0 &&
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out1) | reinterpret_cast<uintptr_t>(out2)) & 15) == 0) {
    const long long n8 = n / 8;
    const int blocks8 = (int)((n8 + 255) / 256 < 148 * 16 ? (n8 + 255) / 256 : 148 * 16);
    drop_pair_bf16x8_kernel<<<blocks8 > 0 ? blocks8 : 1, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(x),
                                                                       reinterpret_cast<__nv_bfloat16*>(out1),
                                                                       reinterpret_cast<__nv_bfloat16*>(out2), d1, d2, n8, D);
    ODV_LAUNCH_CHECK();
    return 0;
  }
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  drop_pair_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(x, out1, out2, type, d1, d2, n, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

namespace {
struct SplitPlan {
  int nseg;
  int piece[6];   // which of (hi, mid, lo) goes into segment i
};
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ src, long long ld, int rows, int cols, int concat_rows,
                                                         SplitPlan sp, __nv_bfloat16* __restrict__ dst) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const long long total = (long long)rows * cols;
  if (i >= total) return;
  const int r = (int)(i / cols), c = (int)(i - (long long)r * cols);   // cols % 4 == 0: the 4 elements share a row
  const float4 v = *reinterpret_cast<const float4*>(src + (long long)r * ld + c);
  const float x[4] = {v.x, v.y, v.z, v.w};
  __nv_bfloat16 pc[3][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float rem = x[j];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      pc[q][j] = __float2bfloat16_rn(rem);
      rem -= __bfloat162float(pc[q][j]);
    }
  }
  uint2 P[3];
#pragma unroll
  for (int q = 0; q < 3; ++q) P[q] = make_uint2(*reinterpret_cast<uint32_t*>(&pc[q][0]), *reinterpret_cast<uint32_t*>(&pc[q][2]));
  for (int sg = 0; sg < sp.nseg; ++sg) {
    const uint2 val = sp.piece[sg] == 0 ? P[0] : (sp.piece[sg] == 1 ? P[1] : P[2]);
    if (concat_rows) *reinterpret_cast<uint2*>(dst + (long long)sg * total + (long long)r * cols + c) = val;
    else *reinterpret_cast<uint2*>(dst + (long long)r * sp.nseg * cols + (long long)sg * cols + c) = val;
  }
}
}  // namespace

int split_bf16(const float* src, long long ld, int rows, int cols, int concat_rows, int nseg, const int* piece, void* dst,
               cudaStream_t s) {
  if (cols % 4 || ld % 4 || nseg < 1 || nseg > 6) return set_error(ODEVIT_ERR_UNSUPPORTED, "split_bf16: bad shape");
  ProfScope prof(KC_WEIGHTS, s);
  SplitPlan sp;
  sp.nseg = nseg;
  for (int i = 0; i < 6; ++i) sp.piece[i] = i < nseg ? piece[i] : 0;
  const long long n4 = (long long)rows * cols / 4;
  split_bf16_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(src, ld, rows, cols, concat_rows, sp, reinterpret_cast<__nv_bfloat16*>(dst));
  ODV_LAUNCH_CHECK();
  return 0;
}

int drop_rows_inplace(void* x, int type, Drop d, int rows, int D, cudaStream_t s) {
  ProfScope prof(KC_COMBINE, s);
  const long long n = (long long)rows * D;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  drop_rows_inplace_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(x, type, d, n, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

int resolve_drop_keys(const uint32_t* seed_dev, uint32_t* table, int n, cudaStream_t s) {
  resolve_drop_keys_kernel<<<(n + 255) / 256, 256, 0, s>>>(seed_dev, table, n);
  ODV_LAUNCH_CHECK();
  return 0;
}

int drop_state_advance(unsigned long long* state, cudaStream_t s) {
  drop_state_advance_kernel<<<1, 1, 0, s>>>(state);
  ODV_LAUNCH_CHECK();
  return 0;
}

int drop_inplace_f32(float* p, float* copy_to, Drop d, long long rows, int n, cudaStream_t s) {
  ProfScope prof(KC_SOFTMAX, s);
  const long long total = rows * n;
  const int blocks = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  drop_inplace_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(p, copy_to, d, total, n);
  ODV_LAUNCH_CHECK();
  return 0;
}

namespace {
struct SeedArgs {
  const float* term[4];
  int n_terms;
};
// gy = sum of the injected cotangents; dd = cast(dd_coef * gy): the start of the reverse sweep in ONE pass (float4)
__global__ void __launch_bounds__(256) seed_sweep_kernel(SeedArgs a, float* __restrict__ gy, void* __restrict__ dd, int dd_type,
                                                         float dd_coef, long long n4) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int t = 0; t < 4; ++t)
      if (t < a.n_terms) {
        const float4 x = reinterpret_cast<const float4*>(a.term[t])[i];
        v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
      }
    reinterpret_cast<float4*>(gy)[i] = v;
    if (dd) {
      const float4 d = make_float4(dd_coef * v.x, dd_coef * v.y, dd_coef * v.z, dd_coef * v.w);
      if (dd_type == DT_F32) {
        reinterpret_cast<float4*>(dd)[i] = d;
      } else {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(d.x, d.y), hi = __floats2bfloat162_rn(d.z, d.w);
        reinterpret_cast<uint2*>(dd)[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
      }
    }
  }
}
}  // namespace

// gy[i] = sum_t term[t][i] (n_terms <= 4; 0 terms: zeros);  dd[i] = cast(dd_coef * gy[i]) when dd != null.  n % 4 == 0.
int seed_sweep(const float* const* terms, int n_terms, float* gy, void* dd, int dd_type, float dd_coef, long long n, cudaStream_t s) {
  if (n % 4 || n_terms < 0 || n_terms > 4) return set_error(ODEVIT_ERR_UNSUPPORTED, "seed_sweep: bad arguments");
  ProfScope prof(KC_COMBINE, s);
  SeedArgs a;
  for (int t = 0; t < 4; ++t) a.term[t] = t < n_terms ? terms[t] : nullptr;
  a.n_terms = n_terms;
  const long long n4 = n / 4;
  const int blocks = (int)((n4 + 255) / 256 < 148 * 16 ? (n4 + 255) / 256 : 148 * 16);
  seed_sweep_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(a, gy, dd, dd_type, dd_coef, n4);
  ODV_LAUNCH_CHECK();
  return 0;
}

int axpy_f32(float* y, const float* x, float a, long long n, cudaStream_t s) {
  ProfScope prof(KC_COMBINE, s);
  const int blocks = (int)((n + 1023) / 1024 < 148 * 8 ? (n + 1023) / 1024 : 148 * 8);
  axpy_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(y, x, a, n);
  ODV_LAUNCH_CHECK();
  return 0;
}

int rowdot_rows(const float* P, const float* G, float* out, long long rows, int n, cudaStream_t s) {
  ProfScope prof(KC_BWD_SOFTMAX, s);
  rowdot_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(P, G, out, rows, n);
  ODV_LAUNCH_CHECK();
  return 0;
}

int jasmin_rowmax(const float* P, long long n_slices, int N, int k, float* out, cudaStream_t s) {
  ProfScope prof(KC_FD_BOUND, s);
  if (N < 1 || N > 1024 || k < 0 || k > N)
    return set_error(ODEVIT_ERR_UNSUPPORTED, "jasmin_rowmax: tokens=%d k=%d (need 1 <= tokens <= 1024, 0 <= k <= tokens)", N, k);
  if (n_slices <= 0) return 0;
  jasmin_rowmax_kernel<<<(unsigned)n_slices, 256, (size_t)8 * N * sizeof(float), s>>>(P, N, k, out);
  ODV_LAUNCH_CHECK();
  return 0;
}

int fd_curvature(const float* states, int T, long long rows, int D, float dt2, float* per_seq, cudaStream_t s) {
  ProfScope prof(KC_FD_BOUND, s);
  if (D % 4 || D > 1024) return set_error(ODEVIT_ERR_UNSUPPORTED, "fd_curvature: D=%d (need D %% 4 == 0, D <= 1024)", D);
  const unsigned grid = (unsigned)((rows + 7) / 8);
  const int ch = (D + 127) / 128;
  if (ch <= 2) fd_curvature_kernel<2><<<grid, 256, 0, s>>>(states, T, rows, D, dt2, per_seq);
  else if (ch <= 4) fd_curvature_kernel<4><<<grid, 256, 0, s>>>(states, T, rows, D, dt2, per_seq);
  else if (ch <= 6) fd_curvature_kernel<6><<<grid, 256, 0, s>>>(states, T, rows, D, dt2, per_seq);
  else fd_curvature_kernel<8><<<grid, 256, 0, s>>>(states, T, rows, D, dt2, per_seq);
  ODV_LAUNCH_CHECK();
  return 0;
}

int ln_rows(const float* x, const float* w, const float* b, void* out, int out_type, float eps, int rows, int D,
            cudaStream_t s) {
  ProfScope prof(KC_CENTER, s);
  if (D > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "ln_rows: D=%d > 1024", D);
  ln_rows_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, w, b, out, out_type, eps, rows, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

int ln_bwd_rows(const LnBwdArgs& a, int rows, int D, cudaStream_t s) {
  ProfScope prof(KC_COMBINE, s);
  if (D > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "ln_bwd_rows: D=%d > 1024", D);
  const int blocks = (rows + 7) / 8 < 148 * 4 ? (rows + 7) / 8 : 148 * 4;
  ln_bwd_rows_kernel<<<blocks, 256, 0, s>>>(a, rows, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

int rk_apply_rows(const Epi& e, const float* v, int rows, int D, cudaStream_t s) {
  ProfScope prof(KC_COMBINE, s);
  Epi e2 = e;
  e2.alpha = 1.f; e2.bias = nullptr; e2.dev_scale = nullptr; e2.resid = nullptr; e2.ld_out = D;
  const long long n = (long long)rows * D;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  if (e2.row_dt) {
    if (!e2.y) return set_error(ODEVIT_ERR_INVALID_ARG, "rk_apply_rows: the per-image step combine needs y");
    rk_apply_kernel<EPI_RK | EPI_ROWDT><<<blocks > 0 ? blocks : 1, 256, 0, s>>>(e2, v, n, D);
  } else {
    rk_apply_kernel<EPI_RK><<<blocks > 0 ? blocks : 1, 256, 0, s>>>(e2, v, n, D);
  }
  ODV_LAUNCH_CHECK();
  return 0;
}

int head_sqnorm(const void* qkv, int type, float* sq, int B, int N, int H, int D, cudaStream_t s) {
  ProfScope prof(KC_SOFTMAX, s);
  const long long warps = (long long)B * N * H * 2;
  head_sqnorm_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, s>>>(qkv, type, sq, B, N, H, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

int l2_prob_rows(float* S, const float* sq, float scale, float* copy_to, int B, int H, int N, cudaStream_t s) {
  ProfScope prof(KC_SOFTMAX, s);
  if (N > 32 * MAX_PER_LANE) return set_error(ODEVIT_ERR_UNSUPPORTED, "l2_prob_rows: N=%d > 1024", N);
  const long long rows = (long long)B * H * N;
  l2_prob_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(S, sq, scale, copy_to, rows, N);
  ODV_LAUNCH_CHECK();
  return 0;
}

int l2_vjp_fix(const float* ds, const void* qkv, int type, void* dz, int R, float coef, int B, int N, int H, int D,
               cudaStream_t s) {
  ProfScope prof(KC_BWD_SOFTMAX, s);
  l2_vjp_fix_kernel<<<B * H, 256, 2 * N * sizeof(float), s>>>(ds, qkv, type, dz, R, coef, N, H, D);
  ODV_LAUNCH_CHECK();
  return 0;
}

int unfold_grads_macaron(const UnfoldArgs& a, cudaStream_t s) {
  ProfScope prof(KC_WEIGHTS, s);
  unfold_w1_kernel<<<3 * a.D + a.hid, 128, 0, s>>>(a, *a.w, *a.gw);
  ODV_LAUNCH_CHECK();
  unfold_w2_macaron_kernel<<<a.D, 128, 0, s>>>(a, *a.w, *a.gw);
  ODV_LAUNCH_CHECK();
  return 0;
}

int fold_weights_parallel(const FoldArgs& a, cudaStream_t s) {
  ProfScope prof(KC_WEIGHTS, s);
  const int R = 3 * a.D + a.hid, K2 = a.D + a.hid;
  fold_w1_kernel<<<R, 128, 0, s>>>(a, *a.w);
  ODV_LAUNCH_CHECK();
  fold_w2_kernel<<<a.D, 128, 0, s>>>(a, *a.w);
  ODV_LAUNCH_CHECK();
  if (a.w1catT) {
    fold_w1_transpose_kernel<<<dim3((R + 31) / 32, (a.D + 31) / 32), 256, 0, s>>>(a, *a.w);
    ODV_LAUNCH_CHECK();
  }
  if (a.w2catT) {
    fold_w2_transpose_kernel<<<dim3((a.D + 31) / 32, (K2 + 31) / 32), 256, 0, s>>>(a, *a.w);
    ODV_LAUNCH_CHECK();
  }
  return 0;
}

int unfold_grads_parallel(const UnfoldArgs& a, cudaStream_t s) {
  ProfScope prof(KC_WEIGHTS, s);
  unfold_w1_kernel<<<3 * a.D + a.hid, 128, 0, s>>>(a, *a.w, *a.gw);
  ODV_LAUNCH_CHECK();
  unfold_norm_kernel<<<dim3((a.D + 127) / 128, (3 * a.D + a.hid + kUnfoldRows - 1) / kUnfoldRows), 128, 0, s>>>(a, *a.w, *a.gw);
  ODV_LAUNCH_CHECK();
  unfold_w2_kernel<<<a.D, 128, 0, s>>>(a, *a.gw);
  ODV_LAUNCH_CHECK();
  return 0;
}

}  // namespace odevit
