// tcgen05 / TMA GEMM with fused epilogues -- the dense contractions of the bf16 mode.
//
//   C[m,n] = sum_k A(m,k) * B(n,k)       bf16 operands, fp32 accumulation in tensor memory
//
// replaces aten::mm of models/ode_transformer_gpt.py:193-200 (fc1/fc2) and :228 (packed in-proj,
// out_proj), and their autograd counterparts, with the CenterNorm affine / GELU / `*scaler` /
// Runge-Kutta stage combine fused into the epilogues (epilogue.cuh).
//
// Structure: persistent, warp-specialised, 320 threads per CTA; with CG == 2 the two CTAs of a
// 2-cluster (one SM pair) drive ONE 256 x BN tile through tcgen05.mma.cta_group::2, so that every
// byte of A and B fetched from L2 / read from shared memory feeds twice the math of the 1-CTA form.
//   warp 0   TMA producer: 128-byte-swizzled boxes of this CTA's 128 rows of A and its BN/CG rows
//            of B into a STAGES-deep shared-memory ring; completion bytes are credited to the LEADER
//            CTA's `full` mbarrier (cp.async.bulk.tensor ... cta_group::2)
//   warp 1   allocates tensor memory; in the leader CTA one elected thread issues the MMAs
//            (UMMA 128*CG x BN x 16, operands straight from both CTAs' shared memory through
//            matrix descriptors), releases ring slots and publishes accumulators with
//            tcgen05.commit multicast to both CTAs
//   warps 2-9 epilogue (TMEM lane quarter x 2 column groups): tcgen05.ld 32 columns of 32 accumulator rows
//            (thread = row), transpose through a swizzled shared-memory scratch so that 8 consecutive lanes
//            hold 128 contiguous bytes of one output row, apply the fused epilogue on float4s with coalesced
//            global loads / stores (epilogue.cuh: loads issued before the accumulator wait).  Two accumulator
//            buffers in TMEM let the epilogue of tile i overlap the main loop of tile i+1; the peer CTA's epilogue
//            warps release the buffer with a remote arrive on the leader's `acc_empty` barrier.
// Operands may be K-major (row-major [rows, K]) or MN-major (row-major [K, rows], i.e. the
// transposed products of the weight-gradient GEMMs); out-of-range rows / K are zero-filled by TMA.
#include <cuda.h>

#include <cstdlib>
#include <mutex>
#include <type_traits>

#include "epilogue.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace odevit {

namespace {

// -DGEMM_TRACE: CTA 0 prints where its MMA thread and its first epilogue warp spent their cycles (diagnostic build only)
#ifdef GEMM_TRACE
#define GT_DECL() long long gt_acc[3] = {0, 0, 0}, gt_t0 = 0, gt_begin = clock64(); (void)gt_t0
#define GT_T0() gt_t0 = clock64()
#define GT_ADD(i) gt_acc[i] += clock64() - gt_t0
#define GT_REPORT(role, a, b, c, tiles)                                                                              \
  do {                                                                                                               \
    if (blockIdx.x == 0)                                                                                             \
      printf("GT %s EPI %d BN %d tiles %d total %lld | %s %lld | %s %lld | %s %lld\n", role, EPI, BN, (int)(tiles), \
             clock64() - gt_begin, a, gt_acc[0], b, gt_acc[1], c, gt_acc[2]);                                        \
  } while (0)
#else
#define GT_DECL() do { } while (0)
#define GT_T0() do { } while (0)
#define GT_ADD(i) do { } while (0)
#define GT_REPORT(role, a, b, c, tiles) do { } while (0)
#endif

constexpr int BM = 128, BK = 64;
// column groups of epilogue warps (x 4 TMEM lane quarters).  3 groups (14 warps -> 128 registers per thread) were
// measured: no faster for the GELU epilogues and slower for EPI_RK (its operand batches spill).
constexpr int EPI_GROUPS = 2;
constexpr int NUM_EPI_WARPS = 4 * EPI_GROUPS;
constexpr int NUM_THREADS = 64 + NUM_EPI_WARPS * 32;
constexpr int ACC_STRIDE = 256;  // TMEM columns between the two accumulator buffers

template <int CG, int BN>
struct Cfg {
  static constexpr int BROWS = BN / CG;  // rows of B this CTA stages
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // as many stages as fit next to the epilogue scratch: the ring must cover the operand round trip (L2 -> shared memory
  // ~1.6 k cycles under load, tools/ubench/tma_feed.cu) at 64-73 bytes per clock, i.e. well over 100 KB IN FLIGHT
  static constexpr int STAGES = (232448 - 1024 - 256 - NUM_EPI_WARPS * 4096) / STAGE_BYTES;
  static constexpr int TMEM_COLS = (BN <= 128) ? 256 : 512;  // two accumulator buffers, power of two
  static constexpr int ACC2 = (BN <= 128) ? 128 : ACC_STRIDE;
  static constexpr int SCRATCH_BYTES = NUM_EPI_WARPS * 4096;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + SCRATCH_BYTES + 1024 /*align*/ + 256 /*barriers*/;
  static_assert(B_BYTES % 1024 == 0, "B stage must keep 1024-byte alignment");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
};

struct DevArgs {
  int M, N, K;
  int tiles_m, tiles_n, split_k, kb_per_split, num_kb;
  // tiles are dealt in waves of num_units; in wave w unit u takes position (u + tile_skew * w) % num_units of the wave.
  // With skew 0 a unit walks the N tiles with stride num_units % tiles_n: for in-proj + fc1 (12 N tiles, 74 units) the odd
  // units met the two GELU tiles back to back every six tiles and the even units only one -- two long epilogues in a row
  // stall the main loop on its accumulator buffers.  The skew makes that stride coprime with tiles_n (every unit cycles
  // through all N tiles, the expensive ones spread out); the set of tiles in flight per wave is unchanged.
  int tile_skew;
  Epi epi;
  // EPI_DET: split-K partial slabs [split_k][M][N] (fp32, row stride N)
  float* part;
};

// the tile of `unit` in wave w_ (see DevArgs::tile_skew); a unit without a tile in the last wave is done
// (`it` counts the waves: the accumulator-buffer parity every role derives from it)
#define ODV_FOR_TILES(tile, it)                                                                                     \
  for (int tile = unit; it * num_units < total_tiles;                                                               \
       ++it, tile = it * num_units + (unit + g.tile_skew * it) % num_units)                                         \
    if (tile < total_tiles)

// The epilogue warps' role.  (Inlined: as a real call its `g` would be a generic pointer to the kernel parameters and
// every epilogue field a global-path load instead of a constant-bank operand -- measured 20-30 % slower.)
template <int CG, int BN, int EPI>
__device__ __forceinline__ void epilogue_role(const DevArgs& g, float* scratch, uint64_t* acc_full, uint64_t* acc_empty,
                                           uint32_t tmem_base, uint32_t rank, int unit, int num_units, int total_tiles) {
  using C = Cfg<CG, BN>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  {
    // TMEM lane quarter q = warp % 4 (hardware rule) x column group grp; a warp owns the 32-column chunks grp,
    // grp + EPI_GROUPS, ... of its quarter's 32 accumulator rows.
    const int ew = warp - 2;
    const int q = warp & 3;
    const int grp = ew >> 2;
    constexpr int NCHT = BN / 32;                                   // chunks per quarter
    const int my_chunks = (NCHT - grp + EPI_GROUPS - 1) / EPI_GROUPS;
    const uint32_t scr = ptx::smem_u32(scratch + ew * 1024);        // this warp's 32 x 32 fp32 transposition tile
    const uint32_t acc_empty_addr0 = ptx::mapa(&acc_empty[0], 0), acc_empty_addr1 = ptx::mapa(&acc_empty[1], 0);
    const int ch = lane & 7, rsub = lane >> 3;
    // transposition addresses (16-byte chunks XOR-swizzled by row % 8: both phases are bank-conflict free), kept as
    // three registers: store j of lane (= row) at st_base ^ (j << 4); load i (row 4 i + rsub) at ld_base[i & 1] + 512 i
    const uint32_t st_base = (scr + (uint32_t)lane * 128u) | ((uint32_t)(lane & 7) << 4);
    const uint32_t ld_base0 = scr + (uint32_t)rsub * 128u + ((uint32_t)(ch ^ rsub) << 4);
    const uint32_t ld_base1 = scr + (uint32_t)rsub * 128u + ((uint32_t)(ch ^ (rsub + 4)) << 4);
    auto tile_coords = [&](int tile, int& m_base, int& n_tile) {
      const int nt = tile % g.tiles_n;
      const int mt = (tile / g.tiles_n) % g.tiles_m;
      m_base = (mt * CG + (int)rank) * BM + q * 32;
      n_tile = nt * BN;
    };
    constexpr bool IS_ACCUM = (EPI & 7) == EPI_ACCUM;
    const bool atomic = IS_ACCUM && g.split_k > 1;
    GT_DECL();
    int it = 0;
    ODV_FOR_TILES(tile, it) {
      int m_base, n_tile;
      tile_coords(tile, m_base, n_tile);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const uint32_t taddr = tmem_base + acc * C::ACC2 + (static_cast<uint32_t>(q * 32) << 16);
      const int m0 = m_base + rsub;
      // FULL: the 32-row slab lies inside M (no row predicates); ATOMIC: split-K accumulation
      auto chunks = [&](auto full_c, auto atomic_c) {
        constexpr bool FULL = decltype(full_c)::value, ATOMIC = decltype(atomic_c)::value;
#pragma unroll 1
        for (int k = 0; k < my_chunks; ++k) {
          const int c = grp + k * EPI_GROUPS;
          const int n = n_tile + c * 32 + ch * 4;
          const bool live = n < g.N;
          if (k == 0) {
            GT_T0();
            ptx::mbar_wait(&acc_full[acc], acc_phase);
            GT_ADD(0);
            ptx::tc_fence_after();
          }
          GT_T0();
          // the chunk's global operand loads are issued behind the (asynchronous) accumulator load and overlap it and
          // the transposition.  (Issued in FRONT of the accumulator wait they would be spilled at once: tcgen05.ld wants
          // 32 consecutive registers and ptxas evicts whatever sits there to local memory.)
          float v[32];
          ptx::tmem_ld32(taddr + c * 32, v);
          EpiPre pre;
          if (live) epi8_issue<EPI, ATOMIC, FULL>(g.epi, m0, g.M, n, pre);
          ptx::tmem_ld_wait();
          GT_ADD(1);
          GT_T0();
          if (k == my_chunks - 1) {
            // every column of this warp's slice is in registers: hand the accumulator back
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (CG == 2) ptx::mbar_arrive_cluster(acc ? acc_empty_addr1 : acc_empty_addr0);
              else ptx::mbar_arrive(&acc_empty[acc]);
            }
          }
          // transpose: lane = row  ->  (row = i*4 + lane/8, 4 columns at (lane%8)*4)
          float4 w[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) ptx::sts_f32x4(st_base ^ (uint32_t)(j << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) w[i] = ptx::lds_f32x4(((i & 1) ? ld_base1 : ld_base0) + (uint32_t)(512 * i));
          __syncwarp();
          if constexpr ((EPI & EPI_DET) != 0 && ATOMIC) {
            // split-K in the deterministic mode: plain stores into this split's slab; det_sum adds the slabs in order
            if (live) {
              float* pp = g.part + ((long long)(tile / (g.tiles_n * g.tiles_m)) * g.M + m0) * g.N + n;
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (row_in<FULL>(m0, i, g.M)) stg_f32x4(pp + (long long)i * 4 * g.N, scale4(g.epi.alpha, w[i]));
            }
          } else {
            if (live) epi8_finish<EPI, ATOMIC, FULL>(g.epi, m0, g.M, n, w, pre);
          }
          GT_ADD(2);
        }
      };
      const bool full = (m_base + 32 <= g.M);
      if constexpr (IS_ACCUM) {
        if (atomic) { if (full) chunks(std::true_type{}, std::true_type{}); else chunks(std::false_type{}, std::true_type{}); }
        else { if (full) chunks(std::true_type{}, std::false_type{}); else chunks(std::false_type{}, std::false_type{}); }
      } else {
        if (full) chunks(std::true_type{}, std::false_type{}); else chunks(std::false_type{}, std::false_type{});
      }
    }
    if (warp == 2 && lane == 0 && rank == 0) { GT_REPORT("epi", "wait acc_full", "tmem ld + operand issue", "transpose + finish", it); }
  }
}

template <int CG, int BN, int EPI, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ DevArgs g) {
  using C = Cfg<CG, BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* scratch = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES + C::SCRATCH_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* acc_full = bars + 2 * C::STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
  const int unit = blockIdx.x / CG, num_units = gridDim.x / CG;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    for (int i = 0; i < C::STAGES; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&acc_full[i], 1);
      ptx::mbar_init(&acc_empty[i], NUM_EPI_WARPS * CG);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    if constexpr (CG == 2) ptx::tmem_alloc_pair(tmem_slot, C::TMEM_COLS);
    else ptx::tmem_alloc(tmem_slot, C::TMEM_COLS);
  }
  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync();
  else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_tiles = g.tiles_m * g.tiles_n * g.split_k;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      ODV_FOR_TILES(tile, it) {
        const int nt = tile % g.tiles_n;
        const int mt = (tile / g.tiles_n) % g.tiles_m;
        const int ks = tile / (g.tiles_n * g.tiles_m);
        const int kb0 = ks * g.kb_per_split;
        const int kb1 = min(g.num_kb, kb0 + g.kb_per_split);
        const int m0 = (mt * CG + (int)rank) * BM;
        const int n0 = nt * BN + (int)rank * C::BROWS;
        for (int kb = kb0; kb < kb1; ++kb) {
          ptx::mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          if constexpr (CG == 1) {
            ptx::mbar_expect_tx(&full[stage], C::STAGE_BYTES);
            if constexpr (!A_MN) {
              ptx::tma_load_2d(sa, &tmA, &full[stage], kb * BK, m0);
            } else {
#pragma unroll
              for (int i = 0; i < BM / 64; ++i)
                ptx::tma_load_2d(sa + i * (64 * BK * 2), &tmA, &full[stage], m0 + i * 64, kb * BK);
            }
            if constexpr (!B_MN) {
              ptx::tma_load_2d(sb, &tmB, &full[stage], kb * BK, n0);
            } else {
#pragma unroll
              for (int i = 0; i < C::BROWS / 64; ++i)
                ptx::tma_load_2d(sb + i * (64 * BK * 2), &tmB, &full[stage], n0 + i * 64, kb * BK);
            }
          } else {
            // both CTAs' bytes are credited to the leader's barrier, which expects the pair's total
            if (rank == 0) ptx::mbar_expect_tx(&full[stage], 2 * C::STAGE_BYTES);
            const uint32_t bar = ptx::mapa(&full[stage], 0);
            if constexpr (!A_MN) {
              ptx::tma_load_2d_pair(sa, &tmA, bar, kb * BK, m0);
            } else {
#pragma unroll
              for (int i = 0; i < BM / 64; ++i)
                ptx::tma_load_2d_pair(sa + i * (64 * BK * 2), &tmA, bar, m0 + i * 64, kb * BK);
            }
            if constexpr (!B_MN) {
              ptx::tma_load_2d_pair(sb, &tmB, bar, kb * BK, n0);
            } else {
#pragma unroll
              for (int i = 0; i < C::BROWS / 64; ++i)
                ptx::tma_load_2d_pair(sb + i * (64 * BK * 2), &tmB, bar, n0 + i * 64, kb * BK);
            }
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer ======================================
    if (lane == 0 && rank == 0) {
      GT_DECL();
      constexpr uint32_t idesc = ptx::idesc_bf16(BM * CG, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      // K-major: 8-row groups 1024 B apart, one UMMA_K (16 elements) = 32 B along the row.
      // MN-major: 64-wide MN blocks (BK*128 B apart), 8-k-row groups 1024 B apart, UMMA_K = 2 groups.
      constexpr uint32_t A_LBO = A_MN ? BK * 128 : 16, A_SBO = 1024, A_KSTEP = A_MN ? 2048 : 32;
      constexpr uint32_t B_LBO = B_MN ? BK * 128 : 16, B_SBO = 1024, B_KSTEP = B_MN ? 2048 : 32;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      ODV_FOR_TILES(tile, it) {
        const int ks = tile / (g.tiles_n * g.tiles_m);
        const int kb0 = ks * g.kb_per_split;
        const int kb1 = min(g.num_kb, kb0 + g.kb_per_split);
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        GT_T0();
        ptx::mbar_wait(&acc_empty[acc], acc_phase ^ 1);
        GT_ADD(0);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::ACC2;
        for (int kb = kb0; kb < kb1; ++kb) {
          GT_T0();
          ptx::mbar_wait(&full[stage], phase);
          GT_ADD(1);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t sb = sa + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t da = ptx::smem_desc_sw128(sa + k * A_KSTEP, A_LBO, A_SBO);
            const uint64_t db = ptx::smem_desc_sw128(sb + k * B_KSTEP, B_LBO, B_SBO);
            const uint32_t accum = (kb > kb0 || k > 0) ? 1u : 0u;
            if constexpr (CG == 2) ptx::mma_bf16_ss_pair(d_tmem, da, db, idesc, accum);
            else ptx::mma_bf16_ss(d_tmem, da, db, idesc, accum);
          }
          // ring slot reusable (in both CTAs) once these MMAs have read it
          if constexpr (CG == 2) ptx::mma_commit_pair(&empty[stage], 3);
          else ptx::mma_commit(&empty[stage]);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
        if constexpr (CG == 2) ptx::mma_commit_pair(&acc_full[acc], 3);  // accumulator complete
        else ptx::mma_commit(&acc_full[acc]);
      }
      GT_REPORT("mma", "wait acc_empty", "wait full", "-", it);
    }
  } else {
    epilogue_role<CG, BN, EPI>(g, scratch, acc_full, acc_empty, tmem_base, rank, unit, num_units, total_tiles);
  }

  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync();
  else __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if constexpr (CG == 2) ptx::tmem_dealloc_pair(tmem_base, C::TMEM_COLS);
    else ptx::tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                              CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn encode_fn() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  return fn;
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

template <int CG, int BN, int EPI, bool A_MN, bool B_MN>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const DevArgs& d, int units, cudaStream_t s) {
  auto kern = gemm_tc_kernel<CG, BN, EPI, A_MN, B_MN>;
  using C = Cfg<CG, BN>;
  static bool configured = false;
  if (!configured) {
    ODV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    configured = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(units * CG);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ODV_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, d));
  ODV_LAUNCH_CHECK();
  return 0;
}

template <int CG, int BN, int EPI>
int launch_major(bool mn, const CUtensorMap& ta, const CUtensorMap& tb, const DevArgs& d, int units, cudaStream_t s) {
  if (!mn) return launch<CG, BN, EPI, false, false>(ta, tb, d, units, s);
  if constexpr ((EPI == EPI_STORE || EPI == EPI_ACCUM || EPI == (EPI_ACCUM | EPI_DET)) && BN != 192) {
    return launch<CG, BN, EPI, true, true>(ta, tb, d, units, s);
  } else {
    return set_error(ODEVIT_ERR_UNSUPPORTED, "gemm_tc: MN-major operands are built for the store / accumulate epilogues");
  }
}

template <int CG, int BN>
int launch_epi(int epi_mode, bool mn, const CUtensorMap& ta, const CUtensorMap& tb, const DevArgs& d, int units,
               cudaStream_t s) {
  switch (epi_mode) {
    case EPI_STORE: return launch_major<CG, BN, EPI_STORE>(mn, ta, tb, d, units, s);
    case EPI_FWD1:
      if (d.epi.exact_gelu) return launch_major<CG, BN, EPI_FWD1 | EPI_EXACT>(mn, ta, tb, d, units, s);
      if (d.epi.drop.thresh) return launch_major<CG, BN, EPI_FWD1 | EPI_DROP>(mn, ta, tb, d, units, s);
      return launch_major<CG, BN, EPI_FWD1>(mn, ta, tb, d, units, s);
    case EPI_RK:
      if (d.epi.fd_out) {
        if (d.epi.drop.thresh || !d.epi.y || !d.epi.fd_prev || d.N % 32)   // (whole warps reduce over rows: no dead lanes)
          return set_error(ODEVIT_ERR_INVALID_ARG, "gemm_tc: the finite-difference epilogue needs y, fd_prev, N %% 32 == 0 and no dropout");
        return launch_major<CG, BN, EPI_RK | EPI_FD>(mn, ta, tb, d, units, s);
      }
      if (d.epi.row_dt) {
        if (d.epi.drop.thresh || !d.epi.y)
          return set_error(ODEVIT_ERR_INVALID_ARG, "gemm_tc: the per-image step epilogue needs y and no dropout");
        return launch_major<CG, BN, EPI_RK | EPI_ROWDT>(mn, ta, tb, d, units, s);
      }
      if (d.epi.drop.thresh) return launch_major<CG, BN, EPI_RK | EPI_DROP>(mn, ta, tb, d, units, s);
      return launch_major<CG, BN, EPI_RK>(mn, ta, tb, d, units, s);
    case EPI_BWD3:
      if (d.epi.exact_gelu) return launch_major<CG, BN, EPI_BWD3 | EPI_EXACT>(mn, ta, tb, d, units, s);
      if (d.epi.drop.thresh) return launch_major<CG, BN, EPI_BWD3 | EPI_DROP>(mn, ta, tb, d, units, s);
      return launch_major<CG, BN, EPI_BWD3>(mn, ta, tb, d, units, s);
    case EPI_ACCUM:
      if (d.part) return launch_major<CG, BN, EPI_ACCUM | EPI_DET>(mn, ta, tb, d, units, s);
      return launch_major<CG, BN, EPI_ACCUM>(mn, ta, tb, d, units, s);
    case EPI_TOKENS: return launch_major<CG, BN, EPI_TOKENS>(mn, ta, tb, d, units, s);
    default: return set_error(ODEVIT_ERR_INVALID_ARG, "gemm_tc: bad epilogue %d", epi_mode);
  }
}

// Tile shape of one launch: CTA-pair (cg = 2, 256 x bn) unless the problem has a single 128-row
// panel; bn in {128, 192, 256} picked by a wave-count model (the tile that leaves the fewest idle
// SM-pairs in the last wave wins; wider tiles win ties: more math per operand byte).
struct TileChoice {
  int cg, bn, split_k;
};

// no_split: the deterministic mode without partial-slab scratch keeps K whole
TileChoice choose_tile(const GemmArgs& g, bool mn, int sms, bool no_split) {
  const char* env = getenv("ODEVIT_GEMM_TILE");  // "<cg>x<bn>", experiments only
  if (env && !env[0]) env = nullptr;
  const int num_kb = (g.K + BK - 1) / BK;
  TileChoice best = {1, 128, 1};
  double best_cost = 1e30;
  for (int cg = 2; cg >= 1; --cg) {
    for (int bn : {256, 192, 128}) {
      if (cg == 1 && bn != 128) continue;
      if (mn && bn == 192) continue;
      if (env && (env[0] - '0' != cg || atoi(env + 2) != bn)) continue;
      const int units = sms / cg;
      const long long tiles = (long long)((g.M + BM * cg - 1) / (BM * cg)) * ((g.N + bn - 1) / bn);
      int sk = 1;
      if (g.epi_mode == EPI_ACCUM && !no_split) {
        // weight-gradient shapes: few output tiles, very long K -> split K across the idle SMs
        sk = (int)(units / tiles);
        if (sk > num_kb / 8) sk = num_kb / 8;
        if (sk < 1) sk = 1;
      }
      const int kb_per = (num_kb + sk - 1) / sk;
      sk = (num_kb + kb_per - 1) / kb_per;
      const long long waves = (tiles * sk + units - 1) / units;
      // per-tile time ~ bn * (k blocks + epilogue/fill overhead); rows wasted by a half-empty pair count too
      double cost = (double)waves * (bn + 64) * (kb_per + 2.0);
      if (cg == 1) cost *= 1.25;          // half the math per staged byte
      else if (bn == 128) cost *= 1.08;
      if (cg == 2 && g.M <= BM) cost *= 2.0;  // second CTA of every pair would idle
      if (cost < best_cost) { best_cost = cost; best = {cg, bn, sk}; }
    }
  }
  return best;
}

}  // namespace

// dims: inner (contiguous) extent, outer extent, outer stride in elements; box = {box_inner, box_outer}
int make_tmap_2d_bf16(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                      uint32_t box_inner, uint32_t box_outer) {
  EncodeFn fn = encode_fn();
  if (!fn) return set_error(ODEVIT_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(ODEVIT_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return 0;
}

int make_tmap_3d_bf16(CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t ld1_elems,
                      uint64_t ld2_elems, uint32_t b0, uint32_t b1, uint32_t b2) {
  EncodeFn fn = encode_fn();
  if (!fn) return set_error(ODEVIT_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {ld1_elems * 2, ld2_elems * 2};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(ODEVIT_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)r);
  return 0;
}

bool gemm_tc_supports(const GemmArgs& g) {
  if (g.a_type != DT_BF16 || g.b_type != DT_BF16) return false;
  if (g.batch_outer * g.batch_inner != 1) return false;
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return false;
  if (g.N % 16) return false;
  if (g.epi.fd_out && (g.N % 32 || g.epi.drop.thresh)) return false;
  if (g.epi.row_dt && (g.epi.fd_out || g.epi.drop.thresh)) return false;   // (those combinations are not instantiated)
  if (g.epi.exact_gelu && g.epi.drop.thresh) return false;   // (that combination is not instantiated)
  if ((g.epi.colsum_a || g.epi.colsum_b) && (g.epi_mode != EPI_BWD3 || g.N % 32 || g.epi.split % 32)) return false;   // whole warps reduce over rows: no dead lanes
  const bool a_k = (g.a_cs == 1), a_mn = (g.a_rs == 1 && g.a_cs != 1);
  const bool b_k = (g.b_cs == 1), b_mn = (g.b_rs == 1 && g.b_cs != 1);
  if (!(a_k || a_mn) || !(b_k || b_mn)) return false;
  if ((a_k && !a_mn) != (b_k && !b_mn)) return false;  // both K-major or both MN-major
  const bool mn = !a_k;
  if (mn && g.epi_mode != EPI_STORE && g.epi_mode != EPI_ACCUM) return false;
  const long long lda = a_mn ? g.a_cs : g.a_rs, ldb = b_mn ? g.b_cs : g.b_rs;
  if (lda % 8 || ldb % 8) return false;  // TMA: 16-byte global strides
  if ((reinterpret_cast<uintptr_t>(g.A) | reinterpret_cast<uintptr_t>(g.B)) & 15) return false;
  if (a_mn ? (g.M % 8) : (g.K % 8)) return false;
  if (b_mn ? (g.N % 8) : (g.K % 8)) return false;
  switch (g.epi_mode) {
    case EPI_STORE: case EPI_FWD1: case EPI_RK: case EPI_BWD3: case EPI_ACCUM: case EPI_TOKENS: break;
    default: return false;
  }
  if (g.epi_mode == EPI_FWD1 || g.epi_mode == EPI_BWD3) {
    if (g.epi.split % 16 || g.epi.ld_out2 % 8 || (g.epi.out3 && g.epi.ld_out3 % 8)) return false;
  }
  if (g.epi.ld_out % (g.epi.out_type == DT_F32 || g.epi_mode == EPI_RK || g.epi_mode == EPI_ACCUM || g.epi_mode == EPI_TOKENS ? 4 : 8)) return false;
  if (g.epi_mode == EPI_TOKENS && (mn || g.epi.split <= 0 || !g.epi.y || g.epi.out_bo % 4)) return false;
  return true;
}

int gemm_tc(const GemmArgs& g, cudaStream_t s) {
  if (!gemm_tc_supports(g)) return set_error(ODEVIT_ERR_UNSUPPORTED, "gemm_tc: unsupported problem");
  ProfScope prof(g.kclass, s);
  const bool mn = (g.a_cs != 1);
  const int sms = num_sms();
  // deterministic mode: a split-K accumulation goes through partial slabs and det_sum (or, without scratch for them,
  // does not split K); every other GEMM has one writer per output element already
  const bool det = deterministic() && g.epi_mode == EPI_ACCUM;
  TileChoice tc = choose_tile(g, mn, sms, false);
  if (det && tc.split_k > 1 && (!g.det_ws || (size_t)tc.split_k * g.M * g.N * 4 > g.det_ws_bytes))
    tc = choose_tile(g, mn, sms, true);
  const int cg = tc.cg, bn = tc.bn;
  DevArgs d;
  d.M = g.M; d.N = g.N; d.K = g.K;
  d.tiles_m = (g.M + BM * cg - 1) / (BM * cg);
  d.tiles_n = (g.N + bn - 1) / bn;
  d.num_kb = (g.K + BK - 1) / BK;
  d.split_k = tc.split_k;
  d.kb_per_split = (d.num_kb + d.split_k - 1) / d.split_k;
  d.split_k = (d.num_kb + d.kb_per_split - 1) / d.kb_per_split;
  d.epi = g.epi;
  d.tile_skew = 0;
  d.part = (det && d.split_k > 1) ? g.det_ws : nullptr;
  CUtensorMap ta, tb;
  const int brows = bn / cg;
  if (!mn) {
    ODV_TRY(make_tmap_2d_bf16(&ta, g.A, g.K, g.M, g.a_rs, BK, BM));
    ODV_TRY(make_tmap_2d_bf16(&tb, g.B, g.K, g.N, g.b_rs, BK, brows));
  } else {
    ODV_TRY(make_tmap_2d_bf16(&ta, g.A, g.M, g.K, g.a_cs, 64, BK));
    ODV_TRY(make_tmap_2d_bf16(&tb, g.B, g.N, g.K, g.b_cs, 64, BK));
  }
  const int total = d.tiles_m * d.tiles_n * d.split_k;
  const int max_units = sms / cg;
  const int units = total < max_units ? total : max_units;
  if ((g.epi_mode == EPI_FWD1 || g.epi_mode == EPI_BWD3) && d.tiles_n > 2 && total > units) {
    // epilogues whose cost depends on the N tile (GELU / GELU' on the fc1 columns only): see DevArgs::tile_skew
    auto gcd = [](int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; };
    for (int sk = 0; sk < d.tiles_n; ++sk) {
      const int stride = (units + sk) % d.tiles_n;
      if (gcd(stride, d.tiles_n) == 1 && stride != 1 && stride != d.tiles_n - 1) { d.tile_skew = sk; break; }
    }
  }
  if (!d.part) {
    if (cg == 1) return launch_epi<1, 128>(g.epi_mode, mn, ta, tb, d, units, s);
    if (bn == 128) return launch_epi<2, 128>(g.epi_mode, mn, ta, tb, d, units, s);
    if (bn == 192) return launch_epi<2, 192>(g.epi_mode, mn, ta, tb, d, units, s);
    return launch_epi<2, 256>(g.epi_mode, mn, ta, tb, d, units, s);
  }
  if (cg == 1) ODV_TRY((launch_epi<1, 128>(g.epi_mode, mn, ta, tb, d, units, s)));
  else if (bn == 128) ODV_TRY((launch_epi<2, 128>(g.epi_mode, mn, ta, tb, d, units, s)));
  else if (bn == 192) ODV_TRY((launch_epi<2, 192>(g.epi_mode, mn, ta, tb, d, units, s)));
  else ODV_TRY((launch_epi<2, 256>(g.epi_mode, mn, ta, tb, d, units, s)));
  return det_sum(reinterpret_cast<float*>(g.epi.out), g.epi.ld_out, d.part, d.split_k, (long long)g.M * g.N, g.M, g.N, s, false);
}

// split_k * tiles never exceeds the units of one wave (choose_tile), and a tile covers at most 128 * cg x 256 outputs
size_t gemm_tc_det_bytes() { return (size_t)num_sms() * BM * 256 * 4; }

}  // namespace odevit
