// Deterministic per-code reductions (the path taken under torch.use_deterministic_algorithms):
//   1. a stable sort of the tokens by code into CSR form (order, offsets): LSD radix sort, 8-bit digits, every pass
//      three launches (tile histograms, one-block scan, stable scatter ranked with __match_any_sync), no spinning;
//   2. a chunked segment sum of token rows in that order (include/vqb200.h states the association contract).
// No float atomics anywhere; the only atomics are shared-memory integer increments of the tile histograms, whose
// result does not depend on their order.
#include <math.h>

#include "common.cuh"

namespace vqb {

constexpr int kDigitBits = 8;
constexpr int kDigits = 1 << kDigitBits;
constexpr int kSortThreads = 256;
constexpr int kSortRounds = 8;
constexpr int kSortTile = kSortThreads * kSortRounds;   // tokens per tile
constexpr int kScanThreads = 1024;
constexpr int64_t kChunk = VQB_SEGMENT_CHUNK;

__host__ __device__ inline int64_t align_up(int64_t a) { return (a + 255) / 256 * 256; }

// ---- sort -----------------------------------------------------------------------------------------
// bucket of a token: its code in [0, K), K for a code outside that range (sorted after every valid token)
__global__ void code_bucket_kernel(const int64_t* __restrict__ quant, const unsigned long long* __restrict__ keys,
                                   int64_t key_offset, int64_t N, int64_t K, int* __restrict__ bucket) {
  pdl_wait();               // PDL: inputs come from the preceding launches
  pdl_launch_dependents();
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
    int64_t q;
    if (quant) {
      q = quant[n];
    } else {   // packed keys of vqb_assign: no finite score (NaN token) -> index 0, like torch.argmin
      const unsigned long long k = keys[n];
      q = k == kNoKey ? 0 : (int64_t)key_index(k) - key_offset;
    }
    bucket[n] = (q >= 0 && q < K) ? (int)q : (int)K;
  }
}

// hist[digit * tiles + tile] = number of tokens of `tile` whose digit is `digit`
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const int* __restrict__ code, int64_t N, int shift,
                                                                  int* __restrict__ hist, int tiles) {
  __shared__ int h[kDigits];
  pdl_wait();
  pdl_launch_dependents();
  h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kSortTile;
#pragma unroll
  for (int r = 0; r < kSortRounds; ++r) {
    const int64_t i = base + r * kSortThreads + threadIdx.x;
    if (i < N) atomicAdd(&h[(code[i] >> shift) & (kDigits - 1)], 1);
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * tiles + blockIdx.x] = h[threadIdx.x];
}

// in-place exclusive scan of v[0, n) with one block: each thread scans a contiguous run serially
__global__ void __launch_bounds__(kScanThreads) exclusive_scan_kernel(int* __restrict__ v, int64_t n) {
  __shared__ int warp_tot[kScanThreads / 32];
  pdl_wait();
  pdl_launch_dependents();
  const int64_t per = (n + kScanThreads - 1) / kScanThreads;
  const int64_t lo = threadIdx.x * per, hi = lo + per < n ? lo + per : n;
  int sum = 0;
  for (int64_t i = lo; i < hi; ++i) sum += v[i];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_tot[w] = incl;
  __syncthreads();
  if (w == 0) {
    int t = warp_tot[lane];
    int s = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += u;
    }
    warp_tot[lane] = s - t;   // exclusive prefix of the warp totals
  }
  __syncthreads();
  int run = warp_tot[w] + incl - sum;
  for (int64_t i = lo; i < hi; ++i) {
    const int c = v[i];
    v[i] = run;
    run += c;
  }
}

// Stable scatter of one digit pass.  Tokens of a tile are taken in rounds of 256 (one per thread, in index order);
// a token's destination is the digit's running tile offset + the same digit's count in lower warps of the round +
// its rank among the lanes of its own warp that share the digit.  No slot is handed out by an atomic.
__global__ void __launch_bounds__(kSortThreads) radix_scatter_kernel(
    const int* __restrict__ code_in, const int* __restrict__ idx_in, int64_t N, int shift,
    const int* __restrict__ hist, int tiles, int* __restrict__ code_out, int* __restrict__ idx_out) {
  constexpr int kWarps = kSortThreads / 32;
  __shared__ int base[kDigits];
  __shared__ int wc[kWarps][kDigits];
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  base[threadIdx.x] = hist[(int64_t)threadIdx.x * tiles + blockIdx.x];
#pragma unroll
  for (int j = 0; j < kWarps; ++j) wc[j][threadIdx.x] = 0;
  __syncthreads();
  const int64_t tile0 = (int64_t)blockIdx.x * kSortTile;
  for (int r = 0; r < kSortRounds; ++r) {
    const int64_t i = tile0 + r * kSortThreads + threadIdx.x;
    const bool valid = i < N;
    const int c = valid ? code_in[i] : 0;
    const int digit = (c >> shift) & (kDigits - 1);
    const unsigned peers = __match_any_sync(0xffffffffu, valid ? digit : kDigits + lane);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (valid && rank == 0) wc[w][digit] = __popc(peers);
    __syncthreads();
    if (valid) {
      int pos = base[digit] + rank;
      for (int j = 0; j < w; ++j) pos += wc[j][digit];
      code_out[pos] = c;
      idx_out[pos] = idx_in ? idx_in[i] : (int)i;
    }
    __syncthreads();
    int tot = 0;
#pragma unroll
    for (int j = 0; j < kWarps; ++j) {
      tot += wc[j][threadIdx.x];
      wc[j][threadIdx.x] = 0;
    }
    base[threadIdx.x] += tot;
    __syncthreads();
  }
}

// offsets[k] = first position of the sorted buckets holding a value >= k  (k in [0, K])
__global__ void csr_offsets_kernel(const int* __restrict__ sorted, int64_t N, int64_t K, int* __restrict__ offsets) {
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k <= K; k += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = N;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (sorted[mid] < k) lo = mid + 1;
      else hi = mid;
    }
    offsets[k] = (int)lo;
  }
}

struct SortLayout {
  int tiles, passes;
  int64_t code_b, idx_tmp, hist, bytes;   // byte offsets into the scratch (code_a at 0)
};
static inline SortLayout sort_layout(int64_t N, int64_t K) {
  SortLayout l;
  l.tiles = (int)((N + kSortTile - 1) / kSortTile);
  int bits = 0;
  while (bits < 32 && (K >> bits) != 0) ++bits;   // bits of the largest bucket value, K
  l.passes = (bits + kDigitBits - 1) / kDigitBits;
  l.code_b = align_up(N * 4);
  l.idx_tmp = l.code_b + align_up(N * 4);
  l.hist = l.idx_tmp + align_up(N * 4);
  l.bytes = l.hist + align_up((int64_t)kDigits * l.tiles * 4);
  return l;
}

// ---- segment sum --------------------------------------------------------------------------------
// 1 / max(|x_n|, eps) with the lane geometry of scatter_stats_kernel (G, V chosen from D alone): the normalised
// row x_n * inv is then the same fp32 vector the atomic path adds.
template <typename TX, int G, int V>
__global__ void __launch_bounds__(256) row_inv_norm_kernel(const TX* __restrict__ x, int64_t N, int D, float* __restrict__ inv) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x % G;
  const int64_t rows_per_block = blockDim.x / G;
  for (int64_t base = blockIdx.x * rows_per_block; base < N; base += (int64_t)gridDim.x * rows_per_block) {
    const int64_t n_raw = base + threadIdx.x / G;
    const int64_t n = n_raw < N ? n_raw : N - 1;
    const TX* __restrict__ xrow = x + n * D;
    float ss = 0.f;
    for (int d = lane * V; d < D; d += G * V)
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float t = to_f32<TX>(xrow[d + v]);
        ss = fmaf(t, t, ss);
      }
    ss = group_sum<G>(ss);
    if (n_raw < N && lane == 0) inv[n] = 1.f / fmaxf(sqrtf(ss), kNormEps);
  }
}

// Slot of chunk j of code k: offsets[k] / C + k + j.  Strictly increasing in k and never shared between codes;
// at most N / C + K + 1 slots.
__device__ __forceinline__ int64_t slot_base(const int* __restrict__ offsets, int64_t k) {
  return offsets[k] / kChunk + k;
}

// One thread per (slot, 4 consecutive elements): the serial ascending sum of the chunk's rows, from +0.
template <typename TX>
__global__ void __launch_bounds__(256) segment_chunk_kernel(const TX* __restrict__ rows, const float* __restrict__ inv,
                                                            int D, const int* __restrict__ order,
                                                            const int* __restrict__ offsets, int64_t K, int64_t slots,
                                                            float* __restrict__ partials) {
  pdl_wait();
  pdl_launch_dependents();
  const int ds = (D + 3) / 4;
  for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < slots * ds; it += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = it / ds;
    const int d0 = (int)(it - s * ds) * 4;
    int64_t lo = 0, hi = K - 1;   // largest k with slot_base(k) <= s
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (slot_base(offsets, mid) <= s) lo = mid;
      else hi = mid - 1;
    }
    const int64_t first = offsets[lo] + (s - slot_base(offsets, lo)) * kChunk;
    const int64_t end = offsets[lo + 1];
    if (first >= end) continue;
    const int64_t last = first + kChunk < end ? first + kChunk : end;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int64_t p = first; p < last; ++p) {
      const int64_t n = order[p];
      const TX* __restrict__ r = rows + n * D;
      const float sc = inv ? inv[n] : 1.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (d0 + i < D) {
          const float v = inv ? __fmul_rn(to_f32<TX>(r[d0 + i]), sc) : to_f32<TX>(r[d0 + i]);
          acc[i] = __fadd_rn(acc[i], v);
        }
      }
    }
    float* __restrict__ dst = partials + s * D + d0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (d0 + i < D) dst[i] = acc[i];
  }
}

// One thread per (code, element): the chunk sums in chunk order from +0, then ONE read-modify-write of the output.
// Codes without tokens leave their output untouched.
__global__ void __launch_bounds__(256) segment_total_kernel(const float* __restrict__ partials, const int* __restrict__ offsets,
                                                            int64_t K, int D, float* __restrict__ out_sums,
                                                            float* __restrict__ out_counts) {
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < K * D; it += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = it / D;
    const int d = (int)(it - k * D);
    const int64_t cnt = (int64_t)offsets[k + 1] - offsets[k];
    if (cnt == 0) continue;
    const int64_t chunks = (cnt + kChunk - 1) / kChunk;
    const float* __restrict__ p = partials + slot_base(offsets, k) * D + d;
    float total = 0.f;
    for (int64_t j = 0; j < chunks; ++j) total = __fadd_rn(total, p[j * D]);
    out_sums[it] = __fadd_rn(out_sums[it], total);
    if (out_counts && d == 0) out_counts[k] = __fadd_rn(out_counts[k], (float)cnt);
  }
}

static inline int64_t segment_slots(int64_t N, int64_t K) { return N / kChunk + K + 1; }

static inline int grid_items(int64_t items) {
  int64_t blocks = (items + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

static inline int lanes_pow2(int n) {
  int g = 1;
  while (g < 32 && g < n) g <<= 1;
  return g;
}

}  // namespace vqb

using namespace vqb;

#define VQB_SEG_DISPATCH_G(G_, ...)                            \
  switch (G_) {                                                \
    case 1: { constexpr int G = 1; __VA_ARGS__; } break;       \
    case 2: { constexpr int G = 2; __VA_ARGS__; } break;       \
    case 4: { constexpr int G = 4; __VA_ARGS__; } break;       \
    case 8: { constexpr int G = 8; __VA_ARGS__; } break;       \
    case 16: { constexpr int G = 16; __VA_ARGS__; } break;     \
    default: { constexpr int G = 32; __VA_ARGS__; } break;     \
  }

extern "C" {

int64_t vqb_segment_chunk(void) { return kChunk; }

size_t vqb_code_sort_scratch_bytes(int64_t N, int64_t K) {
  if (N < 1 || K < 1) return 0;
  return (size_t)sort_layout(N, K).bytes;
}

int vqb_code_sort(const int64_t* quant, const unsigned long long* keys, int64_t key_index_offset, int64_t N, int64_t K,
                  int* order, int* offsets, void* scratch, size_t scratch_bytes, void* stream) {
  VQB_REQUIRE(order && offsets && scratch, "vqb_code_sort: null pointer");
  VQB_REQUIRE((quant != nullptr) != (keys != nullptr), "vqb_code_sort: pass exactly one of quant / keys");
  VQB_REQUIRE(N >= 1 && K >= 1, "vqb_code_sort: bad shape N=%lld K=%lld", (long long)N, (long long)K);
  VQB_REQUIRE(N < (1ll << 31) && K < (1ll << 31) - 1, "vqb_code_sort: N and K must be below 2^31 (int32 order / offsets)");
  const SortLayout l = sort_layout(N, K);
  VQB_REQUIRE(scratch_bytes >= (size_t)l.bytes, "vqb_code_sort: scratch too small (%zu < %lld bytes)", scratch_bytes,
              (long long)l.bytes);
  cudaStream_t st = (cudaStream_t)stream;
  char* base = static_cast<char*>(scratch);
  int* code_a = reinterpret_cast<int*>(base);
  int* code_b = reinterpret_cast<int*>(base + l.code_b);
  int* idx_tmp = reinterpret_cast<int*>(base + l.idx_tmp);
  int* hist = reinterpret_cast<int*>(base + l.hist);
  VQB_CUDA_OK(launch_pdl(code_bucket_kernel, grid_items(N), 256, 0, st, quant, keys, key_index_offset, N, K, code_a));
  const int* idx_in = nullptr;
  for (int p = 0; p < l.passes; ++p) {
    const int shift = p * kDigitBits;
    int* cin = (p % 2 == 0) ? code_a : code_b;
    int* cout = (p % 2 == 0) ? code_b : code_a;
    int* iout = ((l.passes - 1 - p) % 2 == 0) ? order : idx_tmp;   // the last pass lands in `order`
    VQB_CUDA_OK(launch_pdl(radix_hist_kernel, l.tiles, kSortThreads, 0, st, (const int*)cin, N, shift, hist, l.tiles));
    VQB_CUDA_OK(launch_pdl(exclusive_scan_kernel, 1, kScanThreads, 0, st, hist, (int64_t)kDigits * l.tiles));
    VQB_CUDA_OK(launch_pdl(radix_scatter_kernel, l.tiles, kSortThreads, 0, st, (const int*)cin, idx_in, N, shift,
                           (const int*)hist, l.tiles, cout, iout));
    idx_in = iout;
  }
  const int* sorted = (l.passes % 2 == 1) ? code_b : code_a;
  VQB_CUDA_OK(launch_pdl(csr_offsets_kernel, grid_items(K + 1), 256, 0, st, sorted, N, K, offsets));
  return VQB_OK;
}

size_t vqb_segment_sum_scratch_bytes(int64_t N, int64_t K, int D) {
  if (N < 1 || K < 1 || D < 1) return 0;
  return (size_t)(align_up(segment_slots(N, K) * D * 4) + align_up(N * 4));
}

int vqb_segment_sum_rows(const void* rows, int rows_dtype, int64_t N, int D, int normalize_rows, const int* order,
                         const int* offsets, int64_t K, float* out_sums, float* out_counts, void* scratch,
                         size_t scratch_bytes, void* stream) {
  VQB_REQUIRE(rows && order && offsets && out_sums && scratch, "vqb_segment_sum_rows: null pointer");
  VQB_REQUIRE(N >= 1 && D >= 1 && K >= 1, "vqb_segment_sum_rows: bad shape N=%lld D=%d K=%lld", (long long)N, D,
              (long long)K);
  VQB_REQUIRE(N < (1ll << 31), "vqb_segment_sum_rows: N must be below 2^31");
  VQB_REQUIRE(rows_dtype == VQB_F32 || rows_dtype == VQB_BF16, "vqb_segment_sum_rows: bad dtype");
  VQB_REQUIRE(scratch_bytes >= vqb_segment_sum_scratch_bytes(N, K, D), "vqb_segment_sum_rows: scratch too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t slots = segment_slots(N, K);
  float* partials = static_cast<float*>(scratch);
  float* inv = normalize_rows ? reinterpret_cast<float*>(static_cast<char*>(scratch) + align_up(slots * D * 4)) : nullptr;
  if (normalize_rows) {
    const bool vec = (D % 4 == 0);
    const int g = lanes_pow2(vec ? D / 4 : (D + 3) / 4);
    int64_t blocks = (N + 256 / g - 1) / (256 / g);
    if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
#define LAUNCH(TX)                                                                                                   \
  if (vec) {                                                                                                         \
    VQB_SEG_DISPATCH_G(g, VQB_CUDA_OK(launch_pdl(row_inv_norm_kernel<TX, G, 4>, (int)blocks, 256, 0, st, (const TX*)rows, N, D, inv))); \
  } else {                                                                                                           \
    VQB_SEG_DISPATCH_G(g, VQB_CUDA_OK(launch_pdl(row_inv_norm_kernel<TX, G, 1>, (int)blocks, 256, 0, st, (const TX*)rows, N, D, inv))); \
  }
    if (rows_dtype == VQB_F32) { LAUNCH(float) }
    else { LAUNCH(__nv_bfloat16) }
#undef LAUNCH
  }
  const int64_t items = slots * ((D + 3) / 4);
  if (rows_dtype == VQB_F32)
    VQB_CUDA_OK(launch_pdl(segment_chunk_kernel<float>, grid_items(items), 256, 0, st, (const float*)rows,
                           (const float*)inv, D, order, offsets, K, slots, partials));
  else
    VQB_CUDA_OK(launch_pdl(segment_chunk_kernel<__nv_bfloat16>, grid_items(items), 256, 0, st,
                           (const __nv_bfloat16*)rows, (const float*)inv, D, order, offsets, K, slots, partials));
  VQB_CUDA_OK(launch_pdl(segment_total_kernel, grid_items(K * D), 256, 0, st, (const float*)partials, offsets, K, D,
                         out_sums, out_counts));
  return VQB_OK;
}

}  // extern "C"
