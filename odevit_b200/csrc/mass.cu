// The L1-attention-loss front-end (loss_trainer.py:80-117 `extract_mass`) as ONE kernel forward and ONE backward:
//   per (image, head) row a[0..n) of the CLS attention over the patches (n = side^2):
//     (v, idx) = sort(a) ascending;  vn = v / (sum v + 1e-8);  c = cumsum(vn)
//     m = sigmoid((c - (1 - threshold)) * scale)           (smooth)   |   m = [c > 1 - threshold]  (hard)
//     keep[idx[r]] = m[r];   f = a o keep viewed [side, side];   smooth: f = gaussian_blur3x3(f, sigma 0.5, reflect)
//   out_mean[b] = mean over heads of f,  out_heads[b, h] = f,  out_mask[b] = mean over heads of keep (optional).
// The reference runs ~15 small launches (two sorts, cumsum, gather, pad, conv, ...) on a [B, H, 196] tensor.  Here one
// CTA owns an image and walks its heads: bitonic sort of (value, index) pairs in shared memory, block scan, the blur on
// the shared tile, the head mean in registers (deterministic: no atomics).  The backward kernel recomputes the forward
// quantities (nothing saved but the input) and applies the exact adjoints (blur^T, the gather, the sigmoid, the reverse
// scan, the normalisation).  fp32 throughout; ties in the sort are broken by index (torch.sort is not stable either,
// and ties have measure zero on softmax outputs).
#include "internal.h"

namespace odevit {

namespace {

constexpr int MASS_MAX = 1024;

struct MassSmem {
  float v[MASS_MAX];      // sorted values
  int idx[MASS_MAX];      // their original positions
  float scan[MASS_MAX];   // scan scratch / mask in sorted order
  float keep[MASS_MAX];   // mask in original order
  float tile[MASS_MAX];   // a o keep (blur input) / gradient tile
  float red[34];
};

__device__ __forceinline__ float block_sum(float x, float* red, int nthreads) {
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = x;
  __syncthreads();
  if (w == 0) {
    float y = (l < (nthreads + 31) / 32) ? red[l] : 0.f;
    for (int o = 16; o > 0; o >>= 1) y += __shfl_xor_sync(0xffffffffu, y, o);
    if (l == 0) red[32] = y;
  }
  __syncthreads();
  return red[32];
}

// ascending bitonic sort of (v, idx)[0..P), P = blockDim.x (power of two); entries >= n hold +inf
__device__ __forceinline__ void bitonic_sort(float* v, int* idx, int P) {
  const int t = threadIdx.x;
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      const int p = t ^ j;
      if (p > t) {
        const bool up = ((t & k) == 0);
        const float a = v[t], b = v[p];
        const int ia = idx[t], ib = idx[p];
        const bool gt = (a > b) || (a == b && ia > ib);
        if (gt == up) { v[t] = b; v[p] = a; idx[t] = ib; idx[p] = ia; }
      }
    }
  }
  __syncthreads();
}

// inclusive scan of s[0..P) in place (Hillis-Steele through a second buffer-free double step)
__device__ __forceinline__ void inclusive_scan(float* s, int P, bool reverse) {
  const int t = threadIdx.x;
  for (int o = 1; o < P; o <<= 1) {
    __syncthreads();
    float add = 0.f;
    if (!reverse) { if (t >= o) add = s[t - o]; }
    else { if (t + o < P) add = s[t + o]; }
    __syncthreads();
    s[t] += add;
  }
  __syncthreads();
}

__device__ __forceinline__ int reflect(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

struct MassArgs {
  const float* a;       // [B, H, n]
  int B, H, n, side;
  float one_minus_thr, scale;
  int smooth;
  float k0, k1;         // gaussian taps: k0 centre, k1 neighbour (normalised 1-D kernel)
};

// shared forward of one (image, head): leaves v/idx sorted, scan = mask in sorted order, keep, tile = a o keep (pre-blur);
// returns the row sum S
__device__ __forceinline__ float mass_head_forward(const MassArgs& g, const float* row, MassSmem& sm) {
  const int t = threadIdx.x, P = blockDim.x;
  const float x = t < g.n ? row[t] : INFINITY;
  sm.v[t] = x;
  sm.idx[t] = t;
  bitonic_sort(sm.v, sm.idx, P);
  const float S = block_sum(t < g.n ? sm.v[t] : 0.f, sm.red, P);
  sm.scan[t] = t < g.n ? sm.v[t] / (S + 1e-8f) : 0.f;
  inclusive_scan(sm.scan, P, false);
  float m = 0.f;
  if (t < g.n) {
    const float c = sm.scan[t];
    m = g.smooth ? 1.f / (1.f + expf(-(c - g.one_minus_thr) * g.scale)) : (c > g.one_minus_thr ? 1.f : 0.f);
  }
  __syncthreads();
  sm.scan[t] = m;                       // mask, sorted order
  if (t < g.n) sm.keep[sm.idx[t]] = m;
  __syncthreads();
  if (t < g.n) sm.tile[t] = x * sm.keep[t];
  __syncthreads();
  return S;
}

__global__ void mass_fwd_kernel(MassArgs g, float* __restrict__ out_mean, float* __restrict__ out_heads,
                                float* __restrict__ out_mask) {
  __shared__ MassSmem sm;
  const int b = blockIdx.x, t = threadIdx.x;
  const int y = t / g.side, x = t - y * g.side;
  float acc = 0.f, acc_mask = 0.f;
  for (int h = 0; h < g.H; ++h) {
    const float* row = g.a + ((long long)b * g.H + h) * g.n;
    mass_head_forward(g, row, sm);
    float f = 0.f;
    if (t < g.n) {
      if (g.smooth) {
        // separable taps written out as the 3 x 3 product; reflect padding (torchvision gaussian_blur)
        const int ym = reflect(y - 1, g.side), yp = reflect(y + 1, g.side), xm = reflect(x - 1, g.side), xp = reflect(x + 1, g.side);
        const float r0 = g.k1 * sm.tile[ym * g.side + xm] + g.k0 * sm.tile[ym * g.side + x] + g.k1 * sm.tile[ym * g.side + xp];
        const float r1 = g.k1 * sm.tile[y * g.side + xm] + g.k0 * sm.tile[y * g.side + x] + g.k1 * sm.tile[y * g.side + xp];
        const float r2 = g.k1 * sm.tile[yp * g.side + xm] + g.k0 * sm.tile[yp * g.side + x] + g.k1 * sm.tile[yp * g.side + xp];
        f = g.k1 * r0 + g.k0 * r1 + g.k1 * r2;
      } else {
        f = sm.tile[t];
      }
      if (out_heads) out_heads[((long long)b * g.H + h) * g.n + t] = f;
      acc += f;
      acc_mask += sm.keep[t];
    }
    __syncthreads();
  }
  if (t < g.n) {
    out_mean[(long long)b * g.n + t] = acc / g.H;
    if (out_mask) out_mask[(long long)b * g.n + t] = acc_mask / g.H;
  }
}

// g_mean [B, n] and/or g_heads [B, H, n] -> g_a [B, H, n].  DET (deterministic mode): blur^T as a gather with a fixed
// tap order instead of a scatter through shared-memory atomics
template <bool DET>
__global__ void mass_bwd_kernel(MassArgs g, const float* __restrict__ g_mean, const float* __restrict__ g_heads,
                                float* __restrict__ g_a) {
  __shared__ MassSmem sm;
  __shared__ float gt[MASS_MAX];   // gradient wrt the pre-blur tile
  const int b = blockIdx.x, t = threadIdx.x, P = blockDim.x;
  const int y = t / g.side, x = t - y * g.side;
  const float gm = (g_mean && t < g.n) ? g_mean[(long long)b * g.n + t] / g.H : 0.f;
  for (int h = 0; h < g.H; ++h) {
    const long long base = ((long long)b * g.H + h) * g.n;
    const float a_t = t < g.n ? g.a[base + t] : 0.f;
    const float S = mass_head_forward(g, g.a + base, sm);
    float gf = gm;
    if (g_heads && t < g.n) gf += g_heads[base + t];
    // ---- blur^T: scatter the output gradient through the taps ----
    if constexpr (DET) {
      // gather: pixel t collects from the 3 x 3 neighbours whose (reflected) taps land on it.  A neighbour sy reaches y
      // only from {y-1, y, y+1} (reflect(-1) = 1, reflect(side) = side - 2), with weight the sum of its taps that do.
      // (sm.tile, the masked tile, is not read again by the backward: it stages the output gradient)
      if (t < g.n) sm.tile[t] = gf;
      __syncthreads();
      if (t < g.n) {
        if (g.smooth) {
          const float kw[3] = {g.k1, g.k0, g.k1};
          float acc = 0.f;
          for (int sy = y - 1; sy <= y + 1; ++sy) {
            if (sy < 0 || sy >= g.side) continue;
            float wy = 0.f;
#pragma unroll
            for (int i = 0; i < 3; ++i) if (reflect(sy + i - 1, g.side) == y) wy += kw[i];
            for (int sx = x - 1; sx <= x + 1; ++sx) {
              if (sx < 0 || sx >= g.side) continue;
              float wx = 0.f;
#pragma unroll
              for (int j = 0; j < 3; ++j) if (reflect(sx + j - 1, g.side) == x) wx += kw[j];
              acc = fmaf(wy * wx, sm.tile[sy * g.side + sx], acc);
            }
          }
          gt[t] = acc;
        } else {
          gt[t] = gf;
        }
      }
    } else {
    gt[t] = 0.f;
    __syncthreads();
    if (t < g.n) {
      if (g.smooth) {
        const int ys[3] = {reflect(y - 1, g.side), y, reflect(y + 1, g.side)};
        const int xs[3] = {reflect(x - 1, g.side), x, reflect(x + 1, g.side)};
        const float kw[3] = {g.k1, g.k0, g.k1};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) atomicAdd(&gt[ys[i] * g.side + xs[j]], kw[i] * kw[j] * gf);
      } else {
        gt[t] = gf;
      }
    }
    }
    __syncthreads();
    // ---- f = a o keep ----
    float ga = 0.f;
    if (t < g.n) ga = gt[t] * sm.keep[t];
    if (g.smooth) {
      // d keep -> sorted order -> sigmoid -> reverse scan -> normalisation -> back to the original positions
      __syncthreads();
      if (t < g.n) sm.tile[t] = gt[t] * a_t;              // d keep, original order
      __syncthreads();
      float gc = 0.f;
      if (t < g.n) {
        const float m = sm.scan[t];
        gc = sm.tile[sm.idx[t]] * g.scale * m * (1.f - m);
      }
      __syncthreads();
      sm.scan[t] = gc;
      inclusive_scan(sm.scan, P, true);                   // g vn[q] = sum_{r >= q} gc[r]
      const float gvn = t < g.n ? sm.scan[t] : 0.f;
      const float dot = block_sum(t < g.n ? gvn * sm.v[t] : 0.f, sm.red, P);
      const float inv = 1.f / (S + 1e-8f);
      __syncthreads();
      if (t < g.n) sm.tile[sm.idx[t]] = gvn * inv - dot * inv * inv;   // d v scattered to the original positions
      __syncthreads();
      if (t < g.n) ga += sm.tile[t];
    }
    if (t < g.n) g_a[base + t] = ga;
    __syncthreads();
  }
}

int mass_args(MassArgs* g, const float* a, int B, int H, int n, float threshold, int smooth, float scale) {
  int side = 1;
  while (side * side < n) ++side;
  if (side * side != n) return set_error(ODEVIT_ERR_INVALID_ARG, "extract_mass: %d patches are not a square grid", n);
  if (n > MASS_MAX) return set_error(ODEVIT_ERR_UNSUPPORTED, "extract_mass: rows longer than %d are not built", MASS_MAX);
  if (smooth && side < 2) return set_error(ODEVIT_ERR_INVALID_ARG, "extract_mass: the blur needs a grid of at least 2 x 2");
  g->a = a; g->B = B; g->H = H; g->n = n; g->side = side;
  g->one_minus_thr = 1.f - threshold; g->scale = scale; g->smooth = smooth;
  // torchvision _get_gaussian_kernel1d(3, 0.5): pdf(x) = exp(-0.5 (x / sigma)^2) at x = -1, 0, 1, normalised
  const float e = expf(-0.5f * (1.f / 0.5f) * (1.f / 0.5f));
  g->k0 = 1.f / (1.f + 2.f * e);
  g->k1 = e / (1.f + 2.f * e);
  return 0;
}

int mass_threads(int n) {
  int p = 64;
  while (p < n) p <<= 1;
  return p;
}

}  // namespace

int extract_mass_fwd(const float* a, int B, int H, int n, float threshold, int smooth, float scale, float* out_mean,
                     float* out_heads, float* out_mask, cudaStream_t s) {
  MassArgs g;
  ODV_TRY(mass_args(&g, a, B, H, n, threshold, smooth, scale));
  ProfScope prof(KC_OTHER, s);
  mass_fwd_kernel<<<B, mass_threads(n), 0, s>>>(g, out_mean, out_heads, out_mask);
  ODV_LAUNCH_CHECK();
  return 0;
}

int extract_mass_bwd(const float* a, int B, int H, int n, float threshold, int smooth, float scale, const float* g_mean,
                     const float* g_heads, float* g_a, cudaStream_t s) {
  MassArgs g;
  ODV_TRY(mass_args(&g, a, B, H, n, threshold, smooth, scale));
  ProfScope prof(KC_OTHER, s);
  if (deterministic()) mass_bwd_kernel<true><<<B, mass_threads(n), 0, s>>>(g, g_mean, g_heads, g_a);
  else mass_bwd_kernel<false><<<B, mass_threads(n), 0, s>>>(g, g_mean, g_heads, g_a);
  ODV_LAUNCH_CHECK();
  return 0;
}

}  // namespace odevit
