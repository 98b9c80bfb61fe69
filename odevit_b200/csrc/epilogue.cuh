// Fused GEMM epilogues shared by the FFMA and the tcgen05 GEMM kernels (element-wise form).
//
//   EPI_FWD1  packed in-proj + fc1:  q|k|v store, exact-erf GELU      (ode_transformer_gpt.py:193-200, :228)
//   EPI_RK    out_proj + fc2 + `*scaler` + Runge-Kutta stage combine   (:277, :320 + torchdiffeq step)
//   EPI_BWD3  d[O|h] with GELU' applied to the fc1 half
//   EPI_ACCUM weight-gradient accumulation
#pragma once
#include "internal.h"

namespace odevit {

__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

__device__ __forceinline__ void store_elem(void* p, long long idx, int type, float v) {
  if (type == DT_F32) reinterpret_cast<float*>(p)[idx] = v;
  else reinterpret_cast<__nv_bfloat16*>(p)[idx] = __float2bfloat16_rn(v);
}
__device__ __forceinline__ float load_elem_rw(const void* p, long long idx, int type) {
  if (type == DT_F32) return reinterpret_cast<const float*>(p)[idx];
  return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[idx]);
}

// ---- counter-based dropout masks --------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t drop_mix(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
// key of dropout site `site` of field evaluation `e` under the 64-bit seed (lo, hi) -- one formula for the host path
// (api.cu::make_drop) and the device-seeded path (rows.cu::resolve_drop_keys)
__host__ __device__ __forceinline__ uint32_t drop_site_key(uint32_t lo, uint32_t hi, long long e, int site) {
  return drop_mix(lo ^ drop_mix(hi ^ 0x632BE5ABu) ^ ((uint32_t)(e * DS_SITES + site + 1) * 0x27D4EB2Fu));
}
// multiplier of element (r, c): 0 (dropped) or 1/(1-p)
__device__ __forceinline__ float drop_factor(const Drop& d, uint32_t r, uint32_t c) {
  const uint32_t key = d.key_ptr ? __ldg(d.key_ptr) : d.key;
  return drop_mix((r * 0x9E3779B1U) ^ (c * 0x85EBCA77U) ^ key) >= d.thresh ? d.scale : 0.f;
}

template <int EPI, bool ATOMIC>
__device__ __forceinline__ void epi_apply(const Epi& e, int m, int n, float acc, int zo, int zi) {
  if constexpr ((EPI & 7) == EPI_STORE) {
    float v = e.alpha * acc;
    if (e.dev_scale) v *= *e.dev_scale;
    if (e.bias) v += e.bias[n];
    const long long idx = (long long)zo * e.out_bo + (long long)zi * e.out_bi + (long long)m * e.ld_out + n;
    store_elem(e.out, idx, e.out_type, v);
  } else if constexpr ((EPI & 7) == EPI_FWD1) {
    float v = acc;
    if (e.bias) v += e.bias[n];
    if (n < e.split) {
      store_elem(e.out, (long long)m * e.ld_out + n, e.out_type, v);
    } else {
      const int c = n - e.split;
      if (e.out3) store_elem(e.out3, (long long)m * e.ld_out3 + c, e.aux_type, e.aux_gelu_grad ? gelu_erf_grad(v) : v);
      float gv = gelu_erf(v);
      if constexpr ((EPI & EPI_DROP) != 0) gv *= drop_factor(e.drop, m, c);
      store_elem(e.out2, (long long)m * e.ld_out2 + c, e.aux_type, gv);
    }
  } else if constexpr ((EPI & 7) == EPI_RK) {
    float v = acc;
    if (e.bias) v += e.bias[n];
    v *= e.alpha;
    const long long idx = (long long)m * e.ld_out + n;
    if (e.dev_scale) v *= *e.dev_scale;
    if constexpr ((EPI & EPI_DROP) != 0) v *= drop_factor(e.drop, m, n);
    if (e.resid) v = fmaf(e.resid_coef, e.resid[idx], v);
    if (e.k_store) e.k_store[idx] = v;
    float r = e.c_new * v;
    if constexpr ((EPI & EPI_ROWDT) == 0)
      if (e.y) r = fmaf(e.y_coef, e.y[idx], r);
#pragma unroll
    for (int i = 0; i < Epi::kMaxTerms; ++i)
      if (e.kin[i]) r = fmaf(e.c_k[i], e.kin[i][idx], r);
    if constexpr ((EPI & EPI_ROWDT) != 0) r = fmaf((float)e.row_dt[m / e.rows_per_image], r, e.y_coef * e.y[idx]);
    if (e.out) reinterpret_cast<float*>(e.out)[idx] = r;
    if (e.out2) store_elem(e.out2, idx, e.aux_type, e.out2_scale * r);
    if (e.fd_out)   // (CUDA-core path: one atomic per element; the tcgen05 epilogue reduces over the row first)
      atomicMax(reinterpret_cast<int*>(e.fd_out) + m, __float_as_int(fabsf(r - 2.f * e.y[idx] + e.fd_prev[idx])));
  } else if constexpr ((EPI & 7) == EPI_BWD3) {
    if (n < e.split) {
      store_elem(e.out, (long long)m * e.ld_out + n, e.out_type, acc);
    } else {
      const int c = n - e.split;
      const float hp = load_elem_rw(e.aux, (long long)m * e.ld_aux + c, e.aux_type);
      if (e.dev_scale) acc *= *e.dev_scale;
      if constexpr ((EPI & EPI_DROP) != 0) acc *= drop_factor(e.drop, m, c);
      store_elem(e.out2, (long long)m * e.ld_out2 + c, e.aux_type, acc * (e.aux_gelu_grad ? hp : gelu_erf_grad(hp)));
    }
  } else if constexpr ((EPI & 7) == EPI_TOKENS) {
    const int b = m / e.split, r = m - b * e.split;
    reinterpret_cast<float*>(e.out)[(long long)b * e.out_bo + (long long)(r + e.out_bi) * e.ld_out + n] =
        acc + e.y[(long long)r * e.ld_out + n];
  } else if constexpr ((EPI & 7) == EPI_ACCUM) {
    float* o = reinterpret_cast<float*>(e.out) + (long long)m * e.ld_out + n;
    if constexpr (ATOMIC) atomicAdd(o, e.alpha * acc);
    else *o += e.alpha * acc;
  }
}

// ---- vectorised form for the tcgen05 kernels: one thread holds 16 consecutive columns
// [n, n+16) of row m (n % 16 == 0, all 16 in range; row pointers 16-byte aligned). -------------
__device__ __forceinline__ void store16(void* p, long long idx, int type, const float* v) {
  if (type == DT_F32) {
    float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(p) + idx);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p) + idx);
    o[0] = make_uint4(w[0], w[1], w[2], w[3]);
    o[1] = make_uint4(w[4], w[5], w[6], w[7]);
  }
}
__device__ __forceinline__ void load16(const void* p, long long idx, int type, float* v) {
  if (type == DT_F32) {
    const float4* in = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + idx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 t = in[i];
      v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
  } else {
    const uint4* in = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p) + idx);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint4 t = in[h];
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
        v[8 * h + 2 * i] = __low2float(b);
        v[8 * h + 2 * i + 1] = __high2float(b);
      }
    }
  }
}

template <int EPI, bool ATOMIC>
__device__ __forceinline__ void epi_chunk16(const Epi& e, int m, int n, float* v) {
  if constexpr ((EPI & 7) == EPI_STORE) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = e.alpha * (e.dev_scale ? *e.dev_scale : 1.f) * v[j] + (e.bias ? e.bias[n + j] : 0.f);
    store16(e.out, (long long)m * e.ld_out + n, e.out_type, v);
  } else if constexpr ((EPI & 7) == EPI_FWD1) {
    if (e.bias) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] += e.bias[n + j];
    }
    if (n < e.split) {
      store16(e.out, (long long)m * e.ld_out + n, e.out_type, v);
    } else {
      const int c = n - e.split;
      if (e.out3) {
        if (e.aux_gelu_grad) {
          float gp[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) gp[j] = gelu_erf_grad(v[j]);
          store16(e.out3, (long long)m * e.ld_out3 + c, e.aux_type, gp);
        } else {
          store16(e.out3, (long long)m * e.ld_out3 + c, e.aux_type, v);
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = gelu_erf(v[j]);
      if constexpr ((EPI & EPI_DROP) != 0) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] *= drop_factor(e.drop, m, c + j);
      }
      store16(e.out2, (long long)m * e.ld_out2 + c, e.aux_type, v);
    }
  } else if constexpr ((EPI & 7) == EPI_RK) {
    const long long idx = (long long)m * e.ld_out + n;
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = e.alpha * (v[j] + (e.bias ? e.bias[n + j] : 0.f));
    float r[16], t[16];
    if (e.dev_scale) {
      const float ds = *e.dev_scale;
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] *= ds;
    }
    if constexpr ((EPI & EPI_DROP) != 0) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] *= drop_factor(e.drop, m, n + j);
    }
    if (e.resid) {
      load16(e.resid, idx, DT_F32, t);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = fmaf(e.resid_coef, t[j], v[j]);
    }
    if (e.k_store) store16(e.k_store, idx, DT_F32, v);
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = e.c_new * v[j];
    if constexpr ((EPI & EPI_ROWDT) == 0) {
      if (e.y) {
        load16(e.y, idx, DT_F32, t);
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = fmaf(e.y_coef, t[j], r[j]);
      }
    }
#pragma unroll
    for (int i = 0; i < Epi::kMaxTerms; ++i) {
      if (e.kin[i]) {
        load16(e.kin[i], idx, DT_F32, t);
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = fmaf(e.c_k[i], t[j], r[j]);
      }
    }
    if constexpr ((EPI & EPI_ROWDT) != 0) {
      const float dtb = (float)e.row_dt[m / e.rows_per_image];
      load16(e.y, idx, DT_F32, t);
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] = fmaf(dtb, r[j], e.y_coef * t[j]);
    }
    if (e.out) store16(e.out, idx, DT_F32, r);
    if (e.out2) {
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] *= e.out2_scale;
      store16(e.out2, idx, e.aux_type, r);
    }
  } else if constexpr ((EPI & 7) == EPI_BWD3) {
    if (n < e.split) {
      store16(e.out, (long long)m * e.ld_out + n, e.out_type, v);
    } else {
      const int c = n - e.split;
      float hp[16];
      load16(e.aux, (long long)m * e.ld_aux + c, e.aux_type, hp);
      const float ds = e.dev_scale ? *e.dev_scale : 1.f;
#pragma unroll
      for (int j = 0; j < 16; ++j)
        v[j] *= ds * (e.aux_gelu_grad ? hp[j] : gelu_erf_grad(hp[j])) * ((EPI & EPI_DROP) != 0 ? drop_factor(e.drop, m, c + j) : 1.f);
      store16(e.out2, (long long)m * e.ld_out2 + c, e.aux_type, v);
    }
  } else if constexpr ((EPI & 7) == EPI_ACCUM) {
    float* o = reinterpret_cast<float*>(e.out) + (long long)m * e.ld_out + n;
    if constexpr (ATOMIC) {
#pragma unroll
      for (int j = 0; j < 16; ++j) atomicAdd(o + j, e.alpha * v[j]);
    } else {
      float t[16];
      load16(o, 0, DT_F32, t);
#pragma unroll
      for (int j = 0; j < 16; ++j) t[j] = fmaf(e.alpha, v[j], t[j]);
      store16(o, 0, DT_F32, t);
    }
  }
}


// ---- float4 form for the tcgen05 GEMM's transposed (coalesced) epilogue: a lane holds 4 consecutive
// columns [n, n+4) of row m (n % 4 == 0); 8 consecutive lanes cover 128 contiguous bytes of a row.
__device__ __forceinline__ float4 load4(const void* p, long long idx, int type) {
  if (type == DT_F32) return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + idx);
  const uint2 t = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p) + idx);
  const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&t.x);
  const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&t.y);
  return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
}
__device__ __forceinline__ void store4(void* p, long long idx, int type, float4 v) {
  if (type == DT_F32) {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(p) + idx) = v;
  } else {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 t;
    t.x = *reinterpret_cast<const uint32_t*>(&a);
    t.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p) + idx) = t;
  }
}
__device__ __forceinline__ float4 fma4(float a, float4 x, float4 y) {
  return make_float4(fmaf(a, x.x, y.x), fmaf(a, x.y, y.y), fmaf(a, x.z, y.z), fmaf(a, x.w, y.w));
}
__device__ __forceinline__ float4 scale4(float a, float4 x) { return make_float4(a * x.x, a * x.y, a * x.z, a * x.w); }
__device__ __forceinline__ float4 add4(float4 x, float4 y) { return make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w); }

// Loads the compiler may not sink towards their first use (asm volatile keeps program order among
// themselves): the epilogue issues a whole batch of raw loads, then converts / consumes the batch.
struct Raw4 { uint32_t x, y, z, w; };
__device__ __forceinline__ Raw4 ldg_raw4(const void* p, long long idx, int type) {
  Raw4 r;
  if (type == DT_F32) {
    asm volatile("ld.global.v4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(reinterpret_cast<const float*>(p) + idx));
  } else {
    asm volatile("ld.global.v2.b32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(reinterpret_cast<const __nv_bfloat16*>(p) + idx));
    r.z = 0; r.w = 0;
  }
  return r;
}
__device__ __forceinline__ float4 raw_to_float4(const Raw4& r, int type) {
  if (type == DT_F32) return make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z), __uint_as_float(r.w));
  return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                     __uint_as_float(r.y & 0xffff0000u));
}

// GELU for the bf16 mode's epilogues: GELU(x) = x Phi(x) with the Gaussian cdf in its logistic ("tanh") form
//   Phi(x) ~ sigmoid(2 x (c0 + c1 x^2 + c2 x^4)),
// c fitted to the erf form (x^2 clamped at 49, where the quartic would turn): |GELU error| <= 2.6e-5,
// |GELU' error| <= 1.1e-4 over the reals -- far below the bf16 rounding of the stored values -- at 9 (value) and
// 14 (derivative) instructions with one MUFU.EX2 + one MUFU.RCP, where the Abramowitz-Stegun erf used before
// took ~22 and ~28: the GELU epilogues were issue-bound (more epilogue than main-loop cycles per tile at K = 768).
// The fp32 mode keeps erff (gelu_exact / gelu_grad_exact above).
__device__ __forceinline__ float gelu_phi(float x, float x2) {
  constexpr float K = -2.8853900817779268f;   // -2 log2(e): Phi = 1 / (1 + 2^(K x (c0 + c1 x^2 + c2 x^4)))
  float q = fmaf(K * -0.000351516788525385f, x2, K * 0.037005646025752466f);
  q = fmaf(q, x2, K * 0.7975078842819603f);
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * q));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
  return r;
}
__device__ __forceinline__ float gelu_fast(float x) {
  return x * gelu_phi(x, fminf(x * x, 49.f));
}
// GELU and its derivative from one evaluation of Phi (the forward epilogue stores the derivative for the VJP)
__device__ __forceinline__ void gelu_pair_fast(float x, float& g, float& dg) {
  const float x2 = fminf(x * x, 49.f);
  const float phi = gelu_phi(x, x2);
  float d = fmaf(10.f * -0.000351516788525385f, x2, 6.f * 0.037005646025752466f);
  d = fmaf(d, x2, 2.f * 0.7975078842819603f);
  g = x * phi;
  dg = fmaf(g - g * phi, d, phi);     // x phi (1 - phi) d + phi
}
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float x2 = fminf(x * x, 49.f);
  const float phi = gelu_phi(x, x2);
  float d = fmaf(10.f * -0.000351516788525385f, x2, 6.f * 0.037005646025752466f);   // d/dx of 2 x (c0 + c1 x^2 + c2 x^4)
  d = fmaf(d, x2, 2.f * 0.7975078842819603f);
  return fmaf(x * (phi * (1.f - phi)), d, phi);
}

// ------------------------------------------------------------------------------------------------
// The tcgen05 GEMM's epilogue on one lane's share of a 32 x 32 accumulator chunk: 8 float4s, w[i] holding columns
// [n, n+4) of row m0 + 4*i.  Written for instruction count and latency -- with eight to twelve epilogue warps per SM
// every instruction of this code is paid ~24 times per 128 x 32 accumulator slab, and the first version (per-row
// bounds branches, run-time type switches per store, 64-bit index arithmetic per access: ~520 instructions per
// chunk, measured) made the epilogue, not the main loop, the bound of every fused GEMM:
//   * two phases.  `epi8_issue` starts the chunk's global LOADS (state y / GELU input / accumulator) before the
//     accumulator is even waited for; `epi8_finish` consumes them.  The loads are asm volatile: they stay where they
//     are put.
//   * FULL: the 32-row slab lies inside M (every tile but the last row of tiles) -> no row predicates at all.
//   * element types are tested once per chunk (warp-uniform branch), rows are `base + i * step` off one 64-bit base.
// ------------------------------------------------------------------------------------------------
struct EpiPre {
  Raw4 a[8];
};

template <bool FULL>
__device__ __forceinline__ bool row_in(int m0, int i, int M) {
  if constexpr (FULL) return true;
  else return (m0 + 4 * i) < M;
}

__device__ __forceinline__ Raw4 ldg_f32x4(const float* p) {
  Raw4 r;
  asm volatile("ld.global.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ Raw4 ldg_bf16x4(const __nv_bfloat16* p) {
  Raw4 r;
  asm volatile("ld.global.v2.b32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  r.z = 0; r.w = 0;
  return r;
}
__device__ __forceinline__ float4 raw_f32(const Raw4& r) {
  return make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z), __uint_as_float(r.w));
}
__device__ __forceinline__ float4 raw_bf16(const Raw4& r) {
  return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                     __uint_as_float(r.y & 0xffff0000u));
}
__device__ __forceinline__ void stg_f32x4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void stg_bf16x4(__nv_bfloat16* p, float4 v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 t;
  t.x = *reinterpret_cast<const uint32_t*>(&a);
  t.y = *reinterpret_cast<const uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = t;
}
// 8 rows of one output: row i at element offset i * step from `base` (type tested once)
template <bool FULL>
__device__ __forceinline__ void store_rows8(void* base, int type, long long idx0, int step, int m0, int M,
                                            const float4 (&v)[8]) {
  if (type == DT_F32) {
    float* p = reinterpret_cast<float*>(base) + idx0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (row_in<FULL>(m0, i, M)) stg_f32x4(p + i * step, v[i]);
  } else {
    __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(base) + idx0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (row_in<FULL>(m0, i, M)) stg_bf16x4(p + i * step, v[i]);
  }
}
template <bool FULL>
__device__ __forceinline__ void load_rows8_f32(const float* base, long long idx0, int step, int m0, int M, Raw4 (&t)[8]) {
  const float* p = base + idx0;
  const Raw4 zero = {0u, 0u, 0u, 0u};
#pragma unroll
  for (int i = 0; i < 8; ++i) t[i] = row_in<FULL>(m0, i, M) ? ldg_f32x4(p + i * step) : zero;
}

// ---- phase 1: the chunk's first global operand, issued ahead of the accumulator read-out ----
template <int EPI, bool ATOMIC, bool FULL>
__device__ __forceinline__ void epi8_issue(const Epi& e, int m0, int M, int n, EpiPre& pre) {
  if constexpr ((EPI & 7) == EPI_RK) {
    if (e.y) load_rows8_f32<FULL>(e.y, (long long)m0 * e.ld_out + n, 4 * (int)e.ld_out, m0, M, pre.a);
  } else if constexpr ((EPI & 7) == EPI_BWD3) {
    if (n >= e.split) {
      const long long idx0 = (long long)m0 * e.ld_aux + (n - e.split);
      const int step = 4 * (int)e.ld_aux;
      const Raw4 zero = {0u, 0u, 0u, 0u};
      if (e.aux_type == DT_F32) {
        load_rows8_f32<FULL>(reinterpret_cast<const float*>(e.aux), idx0, step, m0, M, pre.a);
      } else {
        const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(e.aux) + idx0;
#pragma unroll
        for (int i = 0; i < 8; ++i) pre.a[i] = row_in<FULL>(m0, i, M) ? ldg_bf16x4(p + i * step) : zero;
      }
    }
  } else if constexpr ((EPI & 7) == EPI_ACCUM && !ATOMIC) {
    load_rows8_f32<FULL>(reinterpret_cast<const float*>(e.out), (long long)m0 * e.ld_out + n, 4 * (int)e.ld_out, m0, M, pre.a);
  }
}

// column sums of the lane's 8 rows x 4 columns, reduced over the four lanes that hold the same columns (lane, lane ^ 8,
// lane ^ 16, lane ^ 24), one float4 atomic per column group.  Every lane of the warp must call it.
__device__ __forceinline__ void colsum_rows8(float* dst, const float4 (&w)[8]) {
  float4 s = w[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) s = add4(s, w[i]);
#pragma unroll
  for (int o = 8; o <= 16; o <<= 1) {
    s.x += __shfl_xor_sync(0xffffffffu, s.x, o); s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
    s.z += __shfl_xor_sync(0xffffffffu, s.z, o); s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
  }
  if ((threadIdx.x & 31) < 8) atomicAdd(reinterpret_cast<float4*>(dst), s);
}

// ---- phase 2 ----
template <int EPI, bool ATOMIC, bool FULL>
__device__ __forceinline__ void epi8_finish(const Epi& e, int m0, int M, int n, float4 (&w)[8], const EpiPre& pre) {
  float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
  if constexpr ((EPI & 7) == EPI_STORE || (EPI & 7) == EPI_FWD1 || (EPI & 7) == EPI_RK) {
    if (e.bias) bias = *reinterpret_cast<const float4*>(e.bias + n);
  }
  float ds = 1.f;
  if constexpr ((EPI & 7) == EPI_STORE || (EPI & 7) == EPI_RK || (EPI & 7) == EPI_BWD3) {
    if (e.dev_scale) ds = *e.dev_scale;
  }
  if constexpr ((EPI & 7) == EPI_STORE) {
    const float a = e.alpha * ds;
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = fma4(a, w[i], bias);
    store_rows8<FULL>(e.out, e.out_type, (long long)m0 * e.ld_out + n, 4 * (int)e.ld_out, m0, M, w);
  } else if constexpr ((EPI & 7) == EPI_FWD1) {
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = add4(w[i], bias);
    if (n < e.split) {
      store_rows8<FULL>(e.out, e.out_type, (long long)m0 * e.ld_out + n, 4 * (int)e.ld_out, m0, M, w);
    } else {
      const int c = n - e.split;
      const bool want_grad = e.out3 && e.aux_gelu_grad;   // (warp-uniform)
      if (e.out3 && !want_grad) store_rows8<FULL>(e.out3, e.aux_type, (long long)m0 * e.ld_out3 + c, 4 * (int)e.ld_out3, m0, M, w);
      if (want_grad) {
        // GELU'(pre) goes out in two half-batches of 4 rows (16 more live registers, not 32)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float4 dg[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float4& x = w[4 * h + i];
            if constexpr ((EPI & EPI_EXACT) != 0) {
              dg[i] = make_float4(gelu_erf_grad(x.x), gelu_erf_grad(x.y), gelu_erf_grad(x.z), gelu_erf_grad(x.w));
              x = make_float4(gelu_erf(x.x), gelu_erf(x.y), gelu_erf(x.z), gelu_erf(x.w));
            } else {
              gelu_pair_fast(x.x, x.x, dg[i].x); gelu_pair_fast(x.y, x.y, dg[i].y);
              gelu_pair_fast(x.z, x.z, dg[i].z); gelu_pair_fast(x.w, x.w, dg[i].w);
            }
          }
          const long long idx0 = (long long)m0 * e.ld_out3 + c;
          const int step = 4 * (int)e.ld_out3;
          if (e.aux_type == DT_F32) {
            float* p3 = reinterpret_cast<float*>(e.out3) + idx0;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (row_in<FULL>(m0, 4 * h + i, M)) stg_f32x4(p3 + (4 * h + i) * step, dg[i]);
          } else {
            __nv_bfloat16* p3 = reinterpret_cast<__nv_bfloat16*>(e.out3) + idx0;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (row_in<FULL>(m0, 4 * h + i, M)) stg_bf16x4(p3 + (4 * h + i) * step, dg[i]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (!want_grad) {
          if constexpr ((EPI & EPI_EXACT) != 0) w[i] = make_float4(gelu_erf(w[i].x), gelu_erf(w[i].y), gelu_erf(w[i].z), gelu_erf(w[i].w));
          else w[i] = make_float4(gelu_fast(w[i].x), gelu_fast(w[i].y), gelu_fast(w[i].z), gelu_fast(w[i].w));
        }
        if constexpr ((EPI & EPI_DROP) != 0) {
          const uint32_t r = m0 + 4 * i;
          w[i].x *= drop_factor(e.drop, r, c); w[i].y *= drop_factor(e.drop, r, c + 1);
          w[i].z *= drop_factor(e.drop, r, c + 2); w[i].w *= drop_factor(e.drop, r, c + 3);
        }
      }
      store_rows8<FULL>(e.out2, e.aux_type, (long long)m0 * e.ld_out2 + c, 4 * (int)e.ld_out2, m0, M, w);
    }
  } else if constexpr ((EPI & 7) == EPI_RK) {
    // Two half-batches of 4 rows: with 14 warps per CTA a thread has 128 registers, and the prefetched state rows
    // (pre, 32) + the accumulator (w, 32) leave room for 16 + 16 more, not 32 + 32.
    const long long idx0 = (long long)m0 * e.ld_out + n;
    const int step = 4 * (int)e.ld_out;
    const float a = e.alpha * ds;
    const Raw4 zero = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      Raw4 t[4];
      float4 v[4], r[4];
      if (e.resid) {   // (Macaron) batched ahead of the arithmetic
#pragma unroll
        for (int i = 0; i < 4; ++i) t[i] = row_in<FULL>(m0, 4 * h + i, M) ? ldg_f32x4(e.resid + idx0 + (4 * h + i) * step) : zero;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = scale4(a, add4(w[4 * h + i], bias));
      if constexpr ((EPI & EPI_DROP) != 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t rr = m0 + 4 * (4 * h + i);
          v[i].x *= drop_factor(e.drop, rr, n); v[i].y *= drop_factor(e.drop, rr, n + 1);
          v[i].z *= drop_factor(e.drop, rr, n + 2); v[i].w *= drop_factor(e.drop, rr, n + 3);
        }
      }
      if (e.resid) {   // v = drop(alpha*ds*(acc+bias)) + resid_coef*resid
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = fma4(e.resid_coef, raw_f32(t[i]), v[i]);
      }
      if (e.k_store) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (row_in<FULL>(m0, 4 * h + i, M)) stg_f32x4(e.k_store + idx0 + (4 * h + i) * step, v[i]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) r[i] = scale4(e.c_new, v[i]);
      if constexpr ((EPI & EPI_ROWDT) == 0) {
        if (e.y) {
#pragma unroll
          for (int i = 0; i < 4; ++i) r[i] = fma4(e.y_coef, raw_f32(pre.a[4 * h + i]), r[i]);
        }
      }
#pragma unroll 1   // (rolled: ONE operand batch live at a time)
      for (int k = 0; k < Epi::kMaxTerms; ++k) {
        const float* kp = e.kin[k];
        if (kp) {
#pragma unroll
          for (int i = 0; i < 4; ++i) t[i] = row_in<FULL>(m0, 4 * h + i, M) ? ldg_f32x4(kp + idx0 + (4 * h + i) * step) : zero;
          const float ck = e.c_k[k];
#pragma unroll
          for (int i = 0; i < 4; ++i) r[i] = fma4(ck, raw_f32(t[i]), r[i]);
        }
      }
      if constexpr ((EPI & EPI_ROWDT) != 0) {   // r = y_coef*y + dt_b*(c_new*v + sum c_k k); rows past M read image 0
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + 4 * (4 * h + i);
          const float dtb = (float)e.row_dt[row_in<FULL>(m0, 4 * h + i, M) ? m / e.rows_per_image : 0];
          r[i] = fma4(dtb, r[i], scale4(e.y_coef, raw_f32(pre.a[4 * h + i])));
        }
      }
      if constexpr ((EPI & EPI_FD) != 0) {
        // second finite difference of the trajectory at the row y: |r - 2 y + prev|, max over this lane's 4 columns,
        // then over the 8 lanes that share a row, then into fd_out[row]
#pragma unroll
        for (int i = 0; i < 4; ++i) t[i] = row_in<FULL>(m0, 4 * h + i, M) ? ldg_f32x4(e.fd_prev + idx0 + (4 * h + i) * step) : zero;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 yy = raw_f32(pre.a[4 * h + i]), pp = raw_f32(t[i]);
          float mx = fmaxf(fmaxf(fabsf(r[i].x - 2.f * yy.x + pp.x), fabsf(r[i].y - 2.f * yy.y + pp.y)),
                           fmaxf(fabsf(r[i].z - 2.f * yy.z + pp.z), fabsf(r[i].w - 2.f * yy.w + pp.w)));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
          if ((threadIdx.x & 7) == 0 && row_in<FULL>(m0, 4 * h + i, M))
            atomicMax(reinterpret_cast<int*>(e.fd_out) + m0 + 4 * (4 * h + i), __float_as_int(mx));
        }
      }
      if (e.out) {
        float* po = reinterpret_cast<float*>(e.out) + idx0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (row_in<FULL>(m0, 4 * h + i, M)) stg_f32x4(po + (4 * h + i) * step, r[i]);
      }
      if (e.out2) {
        if (e.aux_type == DT_F32) {
          float* po = reinterpret_cast<float*>(e.out2) + idx0;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (row_in<FULL>(m0, 4 * h + i, M)) stg_f32x4(po + (4 * h + i) * step, scale4(e.out2_scale, r[i]));
        } else {
          __nv_bfloat16* po = reinterpret_cast<__nv_bfloat16*>(e.out2) + idx0;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (row_in<FULL>(m0, 4 * h + i, M)) stg_bf16x4(po + (4 * h + i) * step, scale4(e.out2_scale, r[i]));
        }
      }
    }
  } else if constexpr ((EPI & 7) == EPI_BWD3) {
    if (n < e.split) {
      store_rows8<FULL>(e.out, e.out_type, (long long)m0 * e.ld_out + n, 4 * (int)e.ld_out, m0, M, w);
      if (e.colsum_a) colsum_rows8(e.colsum_a + n, w);     // (rows past M hold exact zeros: zero-filled operand rows)
    } else {
      const int c = n - e.split;
      const bool f32 = (e.aux_type == DT_F32);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 hp = f32 ? raw_f32(pre.a[i]) : raw_bf16(pre.a[i]);
        if (e.aux_gelu_grad) {   // the forward stored the derivative itself (warp-uniform branch)
          w[i].x *= ds * hp.x; w[i].y *= ds * hp.y; w[i].z *= ds * hp.z; w[i].w *= ds * hp.w;
        } else if constexpr ((EPI & EPI_EXACT) != 0) {
          w[i].x *= ds * gelu_erf_grad(hp.x); w[i].y *= ds * gelu_erf_grad(hp.y);
          w[i].z *= ds * gelu_erf_grad(hp.z); w[i].w *= ds * gelu_erf_grad(hp.w);
        } else {
          w[i].x *= ds * gelu_grad_fast(hp.x); w[i].y *= ds * gelu_grad_fast(hp.y);
          w[i].z *= ds * gelu_grad_fast(hp.z); w[i].w *= ds * gelu_grad_fast(hp.w);
        }
        if constexpr ((EPI & EPI_DROP) != 0) {
          const uint32_t r = m0 + 4 * i;
          w[i].x *= drop_factor(e.drop, r, c); w[i].y *= drop_factor(e.drop, r, c + 1);
          w[i].z *= drop_factor(e.drop, r, c + 2); w[i].w *= drop_factor(e.drop, r, c + 3);
        }
      }
      store_rows8<FULL>(e.out2, e.aux_type, (long long)m0 * e.ld_out2 + c, 4 * (int)e.ld_out2, m0, M, w);
      if (e.colsum_b) colsum_rows8(e.colsum_b + c, w);
    }
  } else if constexpr ((EPI & 7) == EPI_TOKENS) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (!row_in<FULL>(m0, i, M)) continue;
      const int m = m0 + 4 * i;
      const int b = m / e.split, r = m - b * e.split;
      const float4 add = *reinterpret_cast<const float4*>(e.y + (long long)r * e.ld_out + n);
      stg_f32x4(reinterpret_cast<float*>(e.out) + (long long)b * e.out_bo + (long long)(r + e.out_bi) * e.ld_out + n, add4(w[i], add));
    }
  } else if constexpr ((EPI & 7) == EPI_ACCUM) {
    float* p = reinterpret_cast<float*>(e.out) + (long long)m0 * e.ld_out + n;
    const int step = 4 * (int)e.ld_out;
    if constexpr (ATOMIC) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (row_in<FULL>(m0, i, M)) atomicAdd(reinterpret_cast<float4*>(p + i * step), scale4(e.alpha, w[i]));
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (row_in<FULL>(m0, i, M)) stg_f32x4(p + i * step, fma4(e.alpha, w[i], raw_f32(pre.a[i])));
    }
  }
}

}  // namespace odevit
