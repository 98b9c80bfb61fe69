// CUDA-core (FFMA) GEMM with fused epilogues -- the arithmetic of the fp32 mode (<= 1e-4 of the
// reference) and of the small batched per-head attention products.
//
//   C[m,n] = sum_k A(m,k) * B(n,k),  A(m,k) = A[m*a_rs + k*a_cs],  B(n,k) = B[n*b_rs + k*b_cs]
//
// 64x64x16 tiles, 256 threads, 4x4 outputs per thread, fp32 accumulate.  Operands may be fp32 or
// bf16 and arbitrarily strided (so the same kernel does NT / NN / TN products and the strided
// per-(image, head) batches of attention); tiles are staged through shared memory with the
// thread->element map chosen so that global reads are coalesced along whichever index is
// contiguous.  This replaces the aten::mm / aten::bmm launches of
// models/ode_transformer_gpt.py:193-200, :226-232 in fp32 mode.
#include "epilogue.cuh"
#include "internal.h"

namespace odevit {

namespace {

constexpr int BM = 64, BN = 64, BK = 16, PAD = 4;

__device__ __forceinline__ float load_elem(const void* p, long long idx, int type) {
  if (type == DT_F32) return __ldg(reinterpret_cast<const float*>(p) + idx);
  return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[idx]);
}

template <int EPI>
__global__ void __launch_bounds__(256) gemm_simt_kernel(GemmArgs g) {
  __shared__ __align__(16) float As[BK][BM + PAD];
  __shared__ __align__(16) float Bs[BK][BN + PAD];

  const int z = blockIdx.z;
  const int zo = z / g.batch_inner, zi = z - zo * g.batch_inner;
  const long long a_off = (long long)zo * g.a_bo + (long long)zi * g.a_bi;
  const long long b_off = (long long)zo * g.b_bo + (long long)zi * g.b_bi;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const bool a_kc = (g.a_cs == 1), b_kc = (g.b_cs == 1);

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < g.K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + i * 256;
      int mm, kk;
      if (a_kc) { kk = e & 15; mm = e >> 4; } else { mm = e & 63; kk = e >> 6; }
      float v = 0.f;
      if (m0 + mm < g.M && k0 + kk < g.K)
        v = load_elem(g.A, a_off + (long long)(m0 + mm) * g.a_rs + (long long)(k0 + kk) * g.a_cs, g.a_type);
      As[kk][mm] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + i * 256;
      int nn, kk;
      if (b_kc) { kk = e & 15; nn = e >> 4; } else { nn = e & 63; kk = e >> 6; }
      float v = 0.f;
      if (n0 + nn < g.N && k0 + kk < g.K)
        v = load_elem(g.B, b_off + (long long)(n0 + nn) * g.b_rs + (long long)(k0 + kk) * g.b_cs, g.b_type);
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      epi_apply<EPI, false>(g.epi, m, n, acc[i][j], zo, zi);
    }
  }
}

}  // namespace

int gemm_simt(const GemmArgs& g, cudaStream_t s) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0 || !g.A || !g.B)
    return set_error(ODEVIT_ERR_INVALID_ARG, "gemm_simt: bad problem M=%d N=%d K=%d", g.M, g.N, g.K);
  ProfScope prof(g.kclass, s);
  dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, g.batch_outer * g.batch_inner);
  if (grid.y > 65535 || grid.z > 65535)
    return set_error(ODEVIT_ERR_UNSUPPORTED, "gemm_simt: grid too large");
  switch (g.epi_mode) {
    case EPI_STORE: gemm_simt_kernel<EPI_STORE><<<grid, 256, 0, s>>>(g); break;
    case EPI_FWD1:
      if (g.epi.drop.thresh) gemm_simt_kernel<EPI_FWD1 | EPI_DROP><<<grid, 256, 0, s>>>(g);
      else gemm_simt_kernel<EPI_FWD1><<<grid, 256, 0, s>>>(g);
      break;
    case EPI_RK:
      if (g.epi.row_dt) {
        if (g.epi.drop.thresh || !g.epi.y)
          return set_error(ODEVIT_ERR_INVALID_ARG, "gemm_simt: the per-image step epilogue needs y and no dropout");
        gemm_simt_kernel<EPI_RK | EPI_ROWDT><<<grid, 256, 0, s>>>(g);
      } else if (g.epi.drop.thresh) gemm_simt_kernel<EPI_RK | EPI_DROP><<<grid, 256, 0, s>>>(g);
      else gemm_simt_kernel<EPI_RK><<<grid, 256, 0, s>>>(g);
      break;
    case EPI_BWD3:
      if (g.epi.drop.thresh) gemm_simt_kernel<EPI_BWD3 | EPI_DROP><<<grid, 256, 0, s>>>(g);
      else gemm_simt_kernel<EPI_BWD3><<<grid, 256, 0, s>>>(g);
      break;
    case EPI_ACCUM: gemm_simt_kernel<EPI_ACCUM><<<grid, 256, 0, s>>>(g); break;
    case EPI_TOKENS: gemm_simt_kernel<EPI_TOKENS><<<grid, 256, 0, s>>>(g); break;
    default: return set_error(ODEVIT_ERR_INVALID_ARG, "gemm_simt: bad epilogue %d", g.epi_mode);
  }
  ODV_LAUNCH_CHECK();
  return 0;
}

}  // namespace odevit
