// Codebook gather + straight-through estimator + MSE-loss reduction (forward, ONE pass) and the closed-form
// backward, with the token l2-normalisation of NormalizeCallback/VQKDCallback and the key->index unpack
// fused in.  HBM-bound: per token the forward reads the x row, the codebook row (L2-resident) and the
// 8-byte key, and writes the z row (+ the normalised x row and the int64 index when requested).
//
// Layout: G lanes cooperate on one token row, each lane owns V contiguous elements per step (V = 8:
// 128-bit loads for bf16, 2 x 128-bit for fp32) and keeps its slice of the row in registers, so every
// element is read from memory exactly once although the math needs two passes (norms, then outputs).
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace vqb {

constexpr int kMaxPartials = 4096;

// ---- V-wide row slice load/store -------------------------------------------------------------
template <typename T, int V>
__device__ __forceinline__ void load_slice(const T* __restrict__ p, int d0, int D, float (&v)[V]) {
  if constexpr (V == 8 && sizeof(T) == 4) {
    const float4 a = *reinterpret_cast<const float4*>(p + d0), b = *reinterpret_cast<const float4*>(p + d0 + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else if constexpr (V == 8 && sizeof(T) == 2) {
    const uint4 raw = *reinterpret_cast<const uint4*>(p + d0);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __bfloat1622float2(h[i]);
      v[2 * i] = f.x;
      v[2 * i + 1] = f.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = (d0 + i < D) ? to_f32<T>(p[d0 + i]) : 0.f;
  }
}
template <typename T, int V>
__device__ __forceinline__ void store_slice(T* __restrict__ p, int d0, int D, const float (&v)[V]) {
  if constexpr (V == 8 && sizeof(T) == 4) {
    *reinterpret_cast<float4*>(p + d0) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + d0 + 4) = make_float4(v[4], v[5], v[6], v[7]);
  } else if constexpr (V == 8 && sizeof(T) == 2) {
    uint4 raw;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p + d0) = raw;
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i)
      if (d0 + i < D) p[d0 + i] = from_f32<T>(v[i]);
  }
}

// NCHW addressing of a token-major element (n, d): the caller's `(b h w) c <-> b c h w` rearranges
// (vq/tasks/image_tokenization/models/base.py:124,126-127) folded into the kernels.  For a fixed d consecutive tokens
// are contiguous, so the lanes of a warp (consecutive tokens) still write / read whole 32-byte sectors.
template <typename T, int V>
__device__ __forceinline__ void store_slice_nchw(T* __restrict__ p, int64_t n, int64_t hw, int d0, int D, const float (&v)[V]) {
  const int64_t b = n / hw, s = n - b * hw;
  T* __restrict__ q = p + (b * D + d0) * hw + s;
#pragma unroll
  for (int i = 0; i < V; ++i)
    if (d0 + i < D) q[i * hw] = from_f32<T>(v[i]);
}
template <typename T, int V>
__device__ __forceinline__ void load_slice_nchw(const T* __restrict__ p, int64_t n, int64_t hw, int d0, int D, float (&v)[V]) {
  const int64_t b = n / hw, s = n - b * hw;
  const T* __restrict__ q = p + (b * D + d0) * hw + s;
#pragma unroll
  for (int i = 0; i < V; ++i) v[i] = (d0 + i < D) ? to_f32<T>(q[i * hw]) : 0.f;
}

// block-wide deterministic sum of two values; result valid in thread 0
__device__ __forceinline__ void block_sum2(float& a, float& b, float* sh /* >= 2*8 floats */) {
  a = warp_sum(a);
  b = warp_sum(b);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    sh[w] = a;
    sh[8 + w] = b;
  }
  __syncthreads();
  if (w == 0) {
    a = l < (blockDim.x >> 5) ? sh[l] : 0.f;
    b = l < (blockDim.x >> 5) ? sh[8 + l] : 0.f;
    a = warp_sum(a);
    b = warp_sum(b);
  }
}

__device__ __forceinline__ int64_t row_index(const int64_t* __restrict__ quant,
                                             const unsigned long long* __restrict__ keys, int64_t n,
                                             int64_t key_offset, int64_t K) {
  int64_t q;
  if (quant) {
    q = quant[n];
  } else {
    const unsigned long long k = keys[n];
    q = k == kNoKey ? 0 : (int64_t)key_index(k) - key_offset;   // no finite score (NaN token): 0, like torch.argmin
  }
  return q < 0 ? 0 : (q >= K ? K - 1 : q);  // never read out of bounds on a corrupt index
}

// ---- forward -----------------------------------------------------------------------------------
template <typename TX, int G, int V, int NV>
__global__ void __launch_bounds__(256) quantize_forward_kernel(
    const TX* __restrict__ x, int64_t N, int D, int normalize_x, const float* __restrict__ W, int64_t K,
    const int64_t* __restrict__ quant, const unsigned long long* __restrict__ keys, int64_t key_offset,
    int64_t* __restrict__ quant_out, float* __restrict__ xn_out, float* __restrict__ z_out, int64_t z_hw, int want_norm,
    float* __restrict__ mse4, float* __restrict__ partials, unsigned int* __restrict__ ticket) {
  __shared__ float sh[16];
  pdl_wait();               // keys / codebook come from the preceding launches of the step
  pdl_launch_dependents();
  const int lane = threadIdx.x % G;
  const int64_t rows_per_block = blockDim.x / G;
  float sse = 0.f, sse_n = 0.f;
  for (int64_t base = blockIdx.x * rows_per_block; base < N; base += (int64_t)gridDim.x * rows_per_block) {
    const int64_t n_raw = base + threadIdx.x / G;  // warp-uniform trip count: shuffles need every lane
    const bool valid = n_raw < N;
    const int64_t n = valid ? n_raw : N - 1;
    const int64_t q = row_index(quant, keys, n, key_offset, K);
    const float* __restrict__ wrow = W + q * D;
    const TX* __restrict__ xrow = x + n * D;
    float xr[NV][V], wr[NV][V];
    float sxx = 0.f, sww = 0.f;
#pragma unroll
    for (int it = 0; it < NV; ++it) {
      const int d0 = (it * G + lane) * V;
      if (d0 < D) {
        load_slice<TX, V>(xrow, d0, D, xr[it]);
        load_slice<float, V>(wrow, d0, D, wr[it]);
      } else {
#pragma unroll
        for (int i = 0; i < V; ++i) xr[it][i] = wr[it][i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < V; ++i) {
        sxx = fmaf(xr[it][i], xr[it][i], sxx);
        sww = fmaf(wr[it][i], wr[it][i], sww);
      }
    }
    if (normalize_x) {  // x <- F.normalize(x): the quantizer's view of the token from here on
      sxx = group_sum<G>(sxx);
      const float den = fmaxf(sqrtf(sxx), kNormEps);
      float s2 = 0.f;
#pragma unroll
      for (int it = 0; it < NV; ++it)
#pragma unroll
        for (int i = 0; i < V; ++i) {
          xr[it][i] = __fdiv_rn(xr[it][i], den);
          s2 = fmaf(xr[it][i], xr[it][i], s2);
        }
      sxx = s2;
    }
    float rdx = 1.f, rdw = 1.f;  // reciprocal norms for the norm=True MSE term (1 ulp vs a true division)
    if (want_norm) {
      sxx = group_sum<G>(sxx);
      sww = group_sum<G>(sww);
      rdx = 1.f / fmaxf(sqrtf(sxx), kNormEps);
      rdw = 1.f / fmaxf(sqrtf(sww), kNormEps);
    }
#pragma unroll
    for (int it = 0; it < NV; ++it) {
      const int d0 = (it * G + lane) * V;
      float zr[V];
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const float diff = __fsub_rn(wr[it][i], xr[it][i]);
        zr[i] = __fadd_rn(xr[it][i], diff);  // ste value: x + (z - x)
        if (valid) sse = fmaf(diff, diff, sse);
        if (want_norm) {
          const float dn = wr[it][i] * rdw - xr[it][i] * rdx;
          if (valid) sse_n = fmaf(dn, dn, sse_n);
        }
      }
      if (valid && d0 < D) {
        if (z_hw > 0) store_slice_nchw<float, V>(z_out, n, z_hw, d0, D, zr);   // z straight into the caller's NCHW layout
        else store_slice<float, V>(z_out + n * D, d0, D, zr);
        if (xn_out) store_slice<float, V>(xn_out + n * D, d0, D, xr[it]);
      }
    }
    if (quant_out && valid && lane == 0) quant_out[n] = q;
  }
  block_sum2(sse, sse_n, sh);
  // Only warp 0 stays for the ticket: the other warps retire without waiting for the fence, and the last
  // block's warp 0 alone folds the per-block partials (fixed assignment and tree order -> deterministic).
  if (threadIdx.x >= 32) return;
  unsigned int t = 0;
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = sse;
    partials[kMaxPartials + blockIdx.x] = sse_n;
    __threadfence();
    t = atomicAdd(ticket, 1u);
  }
  t = __shfl_sync(0xffffffffu, t, 0);
  if (t == gridDim.x - 1) {
    __threadfence();
    float a = 0.f, b = 0.f;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) {
      a += __ldcg(partials + i);
      b += __ldcg(partials + kMaxPartials + i);
    }
    a = warp_sum(a);
    b = warp_sum(b);
    if (threadIdx.x == 0) {
      const float inv = 1.f / ((float)N * (float)D);
      mse4[0] = a * inv;
      mse4[1] = a * inv;
      mse4[2] = b * inv;
      mse4[3] = b * inv;
      *ticket = 0u;  // self-reset for the next launch
    }
  }
}

// ---- backward ----------------------------------------------------------------------------------
// With y = F.normalize(x_in) when normalize_x (else y = x_in), z = W[q], u = n(y), v = n(z):
//   g_y = g_zste + c_cm (y - z) + J_n(y)^T [c_cmn (u - v)]         c_* = g4[*] * 2 / (N D)
//   g_z = c_cb (z - y) + J_n(z)^T [c_cbn (v - u)]                   -> atomically added to gW[q]
//   g_x_in = J_n(x_in)^T g_y  when normalize_x, else g_y            J_n(a)^T g = (g - (g.n(a)) n(a)) / |a|
// kRowsOut: store each token's g_z row to gW + n*D ([N, D] rows for the deterministic segment sum) instead of the atomics
template <typename TX, typename TG, int G, int V, int NV, bool kRowsOut = false>
__global__ void __launch_bounds__(256, 4) quantize_backward_kernel(
    const TG* __restrict__ gz, const TX* __restrict__ x, int normalize_x, const float* __restrict__ W, int64_t K,
    const int64_t* __restrict__ quant, int64_t N, int D, const float* __restrict__ g_cb,
    const float* __restrict__ g_cm, const float* __restrict__ g_cbn, const float* __restrict__ g_cmn, int want_norm,
    TX* __restrict__ gx, float* __restrict__ gW, int64_t g_hw) {
  pdl_wait();               // upstream gradients / indices come from the preceding launches
  pdl_launch_dependents();
  const int lane = threadIdx.x % G;
  const int64_t rows_per_block = blockDim.x / G;
  const float scale = 2.f / ((float)N * (float)D);
  const float c_cb = g_cb ? *g_cb * scale : 0.f, c_cm = g_cm ? *g_cm * scale : 0.f;
  const float c_cbn = (want_norm && g_cbn) ? *g_cbn * scale : 0.f, c_cmn = (want_norm && g_cmn) ? *g_cmn * scale : 0.f;
  for (int64_t base = blockIdx.x * rows_per_block; base < N; base += (int64_t)gridDim.x * rows_per_block) {
    const int64_t n_raw = base + threadIdx.x / G;
    const bool valid = n_raw < N;
    const int64_t n = valid ? n_raw : N - 1;
    const int64_t q = row_index(quant, nullptr, n, 0, K);
    const float* __restrict__ wrow = W + q * D;
    const TX* __restrict__ xrow = x + n * D;
    float yr[NV][V], wr[NV][V], gr[NV][V];
    float sxx = 0.f, sww = 0.f;
#pragma unroll
    for (int it = 0; it < NV; ++it) {
      const int d0 = (it * G + lane) * V;
      if (d0 < D) {
        load_slice<TX, V>(xrow, d0, D, yr[it]);
        load_slice<float, V>(wrow, d0, D, wr[it]);
        if (g_hw > 0) load_slice_nchw<TG, V>(gz, n, g_hw, d0, D, gr[it]);   // upstream gradient in the caller's NCHW layout
        else load_slice<TG, V>(gz + n * D, d0, D, gr[it]);
      } else {
#pragma unroll
        for (int i = 0; i < V; ++i) yr[it][i] = wr[it][i] = gr[it][i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < V; ++i) {
        sxx = fmaf(yr[it][i], yr[it][i], sxx);
        sww = fmaf(wr[it][i], wr[it][i], sww);
      }
    }
    float den_in = 1.f;
    bool clamp_in = false;
    if (normalize_x) {
      sxx = group_sum<G>(sxx);
      const float nrm = sqrtf(sxx);
      clamp_in = nrm < kNormEps;
      den_in = fmaxf(nrm, kNormEps);
      const float rin = 1.f / den_in;
      float s2 = 0.f;
#pragma unroll
      for (int it = 0; it < NV; ++it)
#pragma unroll
        for (int i = 0; i < V; ++i) {
          yr[it][i] *= rin;
          s2 = fmaf(yr[it][i], yr[it][i], s2);
        }
      sxx = s2;
    }
    float dy = 1.f, dw = 1.f, uu = 0.f, vv = 0.f, uv = 0.f;
    bool cy = false, cw = false;
    if (want_norm) {
      float syw = 0.f;
#pragma unroll
      for (int it = 0; it < NV; ++it)
#pragma unroll
        for (int i = 0; i < V; ++i) syw = fmaf(yr[it][i], wr[it][i], syw);
      sxx = group_sum<G>(sxx);
      sww = group_sum<G>(sww);
      syw = group_sum<G>(syw);
      const float ny = sqrtf(sxx), nw = sqrtf(sww);
      cy = ny < kNormEps;
      cw = nw < kNormEps;
      dy = 1.f / fmaxf(ny, kNormEps);   // from here on dy, dw hold the RECIPROCAL norms
      dw = 1.f / fmaxf(nw, kNormEps);
      uu = sxx * dy * dy;
      vv = sww * dw * dw;
      uv = syw * dy * dw;
    }
    // g_y (overwrites gr) and the codebook-row gradient
    float gy_dot_y = 0.f;
#pragma unroll
    for (int it = 0; it < NV; ++it) {
      const int d0 = (it * G + lane) * V;
      float gw[V];
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const float yv = yr[it][i], wv = wr[it][i];
        float g_y = gr[it][i] + c_cm * (yv - wv);
        float g_w = c_cb * (wv - yv);
        if (want_norm) {
          const float u = yv * dy, v = wv * dw;
          const float gu = c_cmn * (u - v), gu_dot_u = c_cmn * (uu - uv);
          g_y += (gu - (cy ? 0.f : gu_dot_u * u)) * dy;
          const float gv = c_cbn * (v - u), gv_dot_v = c_cbn * (vv - uv);
          g_w += (gv - (cw ? 0.f : gv_dot_v * v)) * dw;
        }
        gr[it][i] = g_y;
        gy_dot_y = fmaf(g_y, yv, gy_dot_y);
        gw[i] = g_w;
      }
      if constexpr (kRowsOut) {
        if (valid && d0 < D) store_slice<float, V>(gW + n * D, d0, D, gw);
      } else if (gW && valid && d0 < D) {
        float* dst = gW + q * D + d0;
        if constexpr (V == 8) {   // two red.global.add.v4.f32 instead of eight scalar atomics (the slice is 32-byte aligned)
          atomicAdd(reinterpret_cast<float4*>(dst), make_float4(gw[0], gw[1], gw[2], gw[3]));
          atomicAdd(reinterpret_cast<float4*>(dst + 4), make_float4(gw[4], gw[5], gw[6], gw[7]));
        } else {
#pragma unroll
          for (int i = 0; i < V; ++i)
            if (d0 + i < D) atomicAdd(dst + i, gw[i]);
        }
      }
    }
    if (normalize_x) {
      gy_dot_y = group_sum<G>(gy_dot_y);
      const float inv = 1.f / den_in;
      const float proj = clamp_in ? 0.f : gy_dot_y;
#pragma unroll
      for (int it = 0; it < NV; ++it)
#pragma unroll
        for (int i = 0; i < V; ++i) gr[it][i] = (gr[it][i] - proj * yr[it][i]) * inv;
    }
#pragma unroll
    for (int it = 0; it < NV; ++it) {
      const int d0 = (it * G + lane) * V;
      if (valid && d0 < D) {
        if (g_hw > 0) store_slice_nchw<TX, V>(gx, n, g_hw, d0, D, gr[it]);
        else store_slice<TX, V>(gx + n * D, d0, D, gr[it]);
      }
    }
  }
}

__global__ void unpack_keys_kernel(const unsigned long long* __restrict__ keys, int64_t n, int64_t offset,
                                   int64_t* __restrict__ idx, float* __restrict__ score) {
  pdl_wait();               // PDL: inputs come from the preceding launches
  pdl_launch_dependents();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long k = keys[i];
    if (idx) idx[i] = k == kNoKey ? 0 : (int64_t)key_index(k) - offset;   // NaN row: index 0, like torch.argmin
    if (score) score[i] = key_score(k);
  }
}

__global__ void embedding_gather_kernel(const float* __restrict__ W, int64_t K, int D,
                                        const int64_t* __restrict__ quant, int64_t n, float* __restrict__ out) {
  const int64_t total = n * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D;
    const int d = (int)(i - r * D);
    int64_t q = quant[r];
    q = q < 0 ? 0 : (q >= K ? K - 1 : q);
    out[i] = __ldg(W + q * D + d);
  }
}

__global__ void keys_flip_kernel(unsigned long long* __restrict__ keys, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    keys[i] ^= 0x8000000000000000ull;
}

static inline int grid_for(int64_t rows, int rows_per_block) {
  int64_t blocks = (rows + rows_per_block - 1) / rows_per_block;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// row geometry: V elements per lane per step, G lanes per row, NV steps (G*V*NV >= D)
struct RowGeom {
  int V, G, NV;
};
static inline bool row_geom(int D, int64_t N, RowGeom* g) {
  g->V = (D % 8 == 0) ? 8 : 1;
  const int slices = (D + g->V - 1) / g->V;
  g->G = 1;
  while (g->G < 32 && g->G < slices) g->G <<= 1;
  int nv = 1;
  while (nv * g->G < slices) nv <<= 1;
  g->NV = nv;
  // These kernels are one dependent-latency chain per thread: a launch that needs slightly more threads than
  // the GPU holds at once (cfg 2: 65 536 rows x 4 lanes = 1.15 waves) pays the chain twice.  Halving the lanes
  // per row (each lane then owns two slices: more loads in flight per thread) brings it back to one wave.
  const int64_t resident_threads = (int64_t)sm_count() * 1536;
  if (g->V == 8 && g->NV == 1 && g->G >= 2 && g->G <= 16 && N * g->G > resident_threads) {
    g->G >>= 1;
    g->NV = 2;
  }
  return g->NV <= 8;
}

}  // namespace vqb

using namespace vqb;

#define VQB_GEOM_CASE(V_, G_, NV_, ...)                 \
  if (geom.V == V_ && geom.G == G_ && geom.NV == NV_) { \
    constexpr int V = V_, G = G_, NV = NV_;             \
    __VA_ARGS__;                                        \
    launched = true;                                    \
  }
// vector path: D multiple of 8 (<= 2048); scalar path: any D <= 256
#define VQB_DISPATCH_GEOM(...)                                                                                    \
  VQB_GEOM_CASE(8, 1, 1, __VA_ARGS__) VQB_GEOM_CASE(8, 2, 1, __VA_ARGS__) VQB_GEOM_CASE(8, 4, 1, __VA_ARGS__)     \
  VQB_GEOM_CASE(8, 8, 1, __VA_ARGS__) VQB_GEOM_CASE(8, 16, 1, __VA_ARGS__) VQB_GEOM_CASE(8, 32, 1, __VA_ARGS__)   \
  VQB_GEOM_CASE(8, 32, 2, __VA_ARGS__) VQB_GEOM_CASE(8, 32, 4, __VA_ARGS__) VQB_GEOM_CASE(8, 32, 8, __VA_ARGS__)  \
  VQB_GEOM_CASE(8, 1, 2, __VA_ARGS__) VQB_GEOM_CASE(8, 2, 2, __VA_ARGS__) VQB_GEOM_CASE(8, 4, 2, __VA_ARGS__)     \
  VQB_GEOM_CASE(8, 8, 2, __VA_ARGS__)                                                                             \
  VQB_GEOM_CASE(1, 1, 1, __VA_ARGS__) VQB_GEOM_CASE(1, 2, 1, __VA_ARGS__) VQB_GEOM_CASE(1, 4, 1, __VA_ARGS__)     \
  VQB_GEOM_CASE(1, 8, 1, __VA_ARGS__) VQB_GEOM_CASE(1, 16, 1, __VA_ARGS__) VQB_GEOM_CASE(1, 32, 1, __VA_ARGS__)   \
  VQB_GEOM_CASE(1, 32, 2, __VA_ARGS__) VQB_GEOM_CASE(1, 32, 4, __VA_ARGS__) VQB_GEOM_CASE(1, 32, 8, __VA_ARGS__)

extern "C" {

int64_t vqb_loss_partials_count(void) { return 2 * kMaxPartials; }

int vqb_gather_ste_loss(const void* x, int x_dtype, int64_t N, int D, int normalize_x, const float* W, int64_t K,
                        const int64_t* quant, const unsigned long long* keys, int64_t key_index_offset,
                        int64_t* quant_out, float* x_norm_out, float* z_out, int64_t z_hw, int want_norm, float* mse4,
                        float* partials, unsigned int* ticket, void* stream) {
  VQB_REQUIRE(z_hw >= 0 && (z_hw == 0 || N % z_hw == 0), "vqb_gather_ste_loss: z_hw must divide N (tokens = images x h*w)");
  VQB_REQUIRE(x && W && z_out && mse4 && partials && ticket, "vqb_gather_ste_loss: null pointer");
  VQB_REQUIRE((quant != nullptr) != (keys != nullptr), "vqb_gather_ste_loss: pass exactly one of quant / keys");
  VQB_REQUIRE(N >= 1 && D >= 1 && K >= 1, "vqb_gather_ste_loss: bad shape N=%lld D=%d K=%lld", (long long)N, D,
              (long long)K);
  RowGeom geom;
  VQB_REQUIRE(row_geom(D, N, &geom), "vqb_gather_ste_loss: D=%d unsupported (multiple of 8 up to 2048, or any D <= 256)", D);
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = grid_for(N, 256 / geom.G);
  VQB_REQUIRE(blocks <= kMaxPartials, "vqb_gather_ste_loss: grid too large");
  bool launched = false;
  if (x_dtype == VQB_F32) {
    VQB_DISPATCH_GEOM((launch_pdl(quantize_forward_kernel<float, G, V, NV>, blocks, 256, 0, st,
        (const float*)x, N, D, normalize_x, W, K, quant, keys, key_index_offset, quant_out, x_norm_out, z_out, z_hw,
        want_norm, mse4, partials, ticket)))
  } else if (x_dtype == VQB_BF16) {
    VQB_DISPATCH_GEOM((launch_pdl(quantize_forward_kernel<__nv_bfloat16, G, V, NV>, blocks, 256, 0, st,
        (const __nv_bfloat16*)x, N, D, normalize_x, W, K, quant, keys, key_index_offset, quant_out, x_norm_out, z_out,
        z_hw, want_norm, mse4, partials, ticket)))
  }
  VQB_REQUIRE(launched, "vqb_gather_ste_loss: unsupported dtype/geometry");
  VQB_LAUNCH_OK();
  return VQB_OK;
}

}  // extern "C"

// kRowsOut selects the per-token-row variant (gW then points at fp32 [N, D] rows)
template <bool kRowsOut>
static int quantize_backward_launch(const void* gz, int g_dtype, const void* x, int x_dtype, int normalize_x, const float* W,
                                    int64_t K, const int64_t* quant, int64_t N, int D, const float* g_cb, const float* g_cm,
                                    const float* g_cbn, const float* g_cmn, int want_norm, void* gx, float* gW,
                                    int64_t g_hw, void* stream) {
  VQB_REQUIRE(g_hw >= 0 && (g_hw == 0 || N % g_hw == 0), "vqb_quantize_backward: g_hw must divide N");
  VQB_REQUIRE(gz && x && W && quant && gx, "vqb_quantize_backward: null pointer");
  VQB_REQUIRE(!kRowsOut || gW, "vqb_quantize_backward_rows: null gW_rows");
  VQB_REQUIRE(N >= 1 && D >= 1 && K >= 1, "vqb_quantize_backward: bad shape");
  RowGeom geom;
  VQB_REQUIRE(row_geom(D, N, &geom), "vqb_quantize_backward: D=%d unsupported", D);
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = grid_for(N, 256 / geom.G);
  bool launched = false;
  if (x_dtype == VQB_F32 && g_dtype == VQB_F32) {
    VQB_DISPATCH_GEOM((launch_pdl(quantize_backward_kernel<float, float, G, V, NV, kRowsOut>, blocks, 256, 0, st,
        (const float*)gz, (const float*)x, normalize_x, W, K, quant, N, D, g_cb, g_cm, g_cbn, g_cmn, want_norm, (float*)gx, gW, g_hw)))
  } else if (x_dtype == VQB_BF16 && g_dtype == VQB_F32) {
    VQB_DISPATCH_GEOM((launch_pdl(quantize_backward_kernel<__nv_bfloat16, float, G, V, NV, kRowsOut>, blocks, 256, 0, st,
        (const float*)gz, (const __nv_bfloat16*)x, normalize_x, W, K, quant, N, D, g_cb, g_cm, g_cbn, g_cmn, want_norm,
        (__nv_bfloat16*)gx, gW, g_hw)))
  } else if (x_dtype == VQB_BF16 && g_dtype == VQB_BF16) {   // bf16 upstream gradient (autocast training): read as is
    VQB_DISPATCH_GEOM((launch_pdl(quantize_backward_kernel<__nv_bfloat16, __nv_bfloat16, G, V, NV, kRowsOut>, blocks, 256, 0, st,
        (const __nv_bfloat16*)gz, (const __nv_bfloat16*)x, normalize_x, W, K, quant, N, D, g_cb, g_cm, g_cbn, g_cmn,
        want_norm, (__nv_bfloat16*)gx, gW, g_hw)))
  }
  VQB_REQUIRE(launched, "vqb_quantize_backward: unsupported dtype/geometry");
  VQB_LAUNCH_OK();
  return VQB_OK;
}

extern "C" {

int vqb_quantize_backward(const void* gz, int g_dtype, const void* x, int x_dtype, int normalize_x, const float* W, int64_t K,
                          const int64_t* quant, int64_t N, int D, const float* g_cb, const float* g_cm,
                          const float* g_cbn, const float* g_cmn, int want_norm, void* gx, float* gW, int64_t g_hw,
                          void* stream) {
  return quantize_backward_launch<false>(gz, g_dtype, x, x_dtype, normalize_x, W, K, quant, N, D, g_cb, g_cm, g_cbn, g_cmn,
                                         want_norm, gx, gW, g_hw, stream);
}

int vqb_quantize_backward_rows(const void* gz, int g_dtype, const void* x, int x_dtype, int normalize_x, const float* W,
                               int64_t K, const int64_t* quant, int64_t N, int D, const float* g_cb, const float* g_cm,
                               const float* g_cbn, const float* g_cmn, int want_norm, void* gx, float* gW_rows,
                               int64_t g_hw, void* stream) {
  return quantize_backward_launch<true>(gz, g_dtype, x, x_dtype, normalize_x, W, K, quant, N, D, g_cb, g_cm, g_cbn, g_cmn,
                                        want_norm, gx, gW_rows, g_hw, stream);
}

int vqb_unpack_keys(const unsigned long long* keys, int64_t n, int64_t offset, int64_t* idx, float* score,
                    void* stream) {
  VQB_REQUIRE(keys && (idx || score), "vqb_unpack_keys: null pointer");
  if (n <= 0) return VQB_OK;
  int blocks = (int)((n + 255) / 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  launch_pdl(unpack_keys_kernel, blocks, 256, 0, (cudaStream_t)stream, keys, n, offset, idx, score);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

int vqb_embedding_gather(const float* W, int64_t K, int D, const int64_t* quant, int64_t n, float* out,
                         void* stream) {
  VQB_REQUIRE(W && quant && out, "vqb_embedding_gather: null pointer");
  VQB_REQUIRE(K >= 1 && D >= 1, "vqb_embedding_gather: bad shape");
  if (n <= 0) return VQB_OK;
  int64_t blocks64 = (n * D + 255) / 256;
  const int blocks = (int)(blocks64 < (int64_t)sm_count() * 8 ? blocks64 : (int64_t)sm_count() * 8);
  embedding_gather_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(W, K, D, quant, n, out);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

int vqb_keys_flip_sign(unsigned long long* keys, int64_t n, void* stream) {
  VQB_REQUIRE(keys, "vqb_keys_flip_sign: null pointer");
  if (n <= 0) return VQB_OK;
  int blocks = (int)((n + 255) / 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  keys_flip_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(keys, n);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

}  // extern "C"
