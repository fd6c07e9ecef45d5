// Data formats either side of the quantizer (SURVEY.md §8f items 1 and 3):
//   * the tokenizer model's `b c h w -> (b h w) c` / `(b h w) c -> b c h w` rearranges
//     (vq/tasks/image_tokenization/models/base.py:124,126-127) as one tiled, coalesced batched transpose;
//   * the tokenise-only output: packed assignment keys -> compact token ids (uint16 for K <= 65536, else
//     int32) for the token dumps (runners/callbacks.py:40-53, tools/tokenize_llamagen.py:93-103).
// Both are HBM-bound single passes.
#include "common.cuh"

namespace vqb {

constexpr int kTile = 32;

// src [batch][rows][cols] -> dst [batch][cols][rows]; 32 x 32 tile through padded shared memory, both the
// global read (along cols) and the global write (along rows) are coalesced.
template <typename T>
__global__ void __launch_bounds__(kTile * 8) transpose_last2_kernel(const T* __restrict__ src, int64_t rows,
                                                                    int64_t cols, T* __restrict__ dst) {
  __shared__ T tile[kTile][kTile + 1];
  const int64_t b = blockIdx.z;
  const T* __restrict__ s = src + b * rows * cols;
  T* __restrict__ d = dst + b * rows * cols;
  const int64_t c0 = (int64_t)blockIdx.x * kTile, r0 = (int64_t)blockIdx.y * kTile;
  const int tx = threadIdx.x, ty = threadIdx.y;
#pragma unroll
  for (int i = ty; i < kTile; i += 8) {
    const int64_t r = r0 + i, c = c0 + tx;
    if (r < rows && c < cols) tile[i][tx] = s[r * cols + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < kTile; i += 8) {
    const int64_t c = c0 + i, r = r0 + tx;
    if (r < rows && c < cols) d[c * rows + r] = tile[tx][i];
  }
}

// Vectorised variant (cols and rows multiples of the 16-byte vector): a TR (rows) x TC (cols) tile is read
// with 128-bit loads along cols, transposed through shared memory, and written with 128-bit stores along rows.
template <typename T, int TR, int TC>
__global__ void __launch_bounds__(256) transpose_last2_vec_kernel(const T* __restrict__ src, int64_t rows, int64_t cols,
                                                                  T* __restrict__ dst) {
  constexpr int VE = 16 / sizeof(T);          // elements per 128-bit vector
  constexpr int PITCH = TC + 4 / sizeof(T) + (sizeof(T) == 8 ? 1 : 0);   // +1 bank word: conflict-free column reads
  __shared__ T tile[TR][PITCH];
  const int64_t b = blockIdx.z;
  const T* __restrict__ s = src + b * rows * cols;
  T* __restrict__ d = dst + b * rows * cols;
  const int64_t r0 = (int64_t)blockIdx.y * TR;
  constexpr int VPR = TC / VE;
  constexpr int VPC = TR / VE;
  // a block walks the column tiles of its row band (gridDim.x < number of column tiles when there are plenty of
  // images): a 4-8 KB tile per block left the kernel bound by block scheduling, not by bandwidth
  for (int64_t c0 = (int64_t)blockIdx.x * TC; c0 < cols; c0 += (int64_t)gridDim.x * TC) {
    // load: (TC / VE) vectors per row
    for (int v = threadIdx.x; v < TR * VPR; v += 256) {
      const int r = v / VPR, cv = (v % VPR) * VE;
      if (r0 + r < rows && c0 + cv < cols) {
        const uint4 raw = *reinterpret_cast<const uint4*>(s + (r0 + r) * cols + c0 + cv);
        const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
        for (int i = 0; i < VE; ++i) tile[r][cv + i] = e[i];
      }
    }
    __syncthreads();
    // store: output row = source column c, TR contiguous elements along r -> TR / VE vectors per output row
    for (int v = threadIdx.x; v < TC * VPC; v += 256) {
      // consecutive lanes -> consecutive vectors of ONE output row (then the next row): full 64-128 B segments per
      // row instead of 16-byte pieces strided by the row pitch; the padded pitch keeps the shared reads conflict-free
      // (long output rows, VPC > 8, keep the column-fastest order: their shared reads would conflict 4-way)
      const int rv = (VPC <= 8 ? v % VPC : v / TC) * VE, c = VPC <= 8 ? v / VPC : v % TC;
      if (c0 + c < cols && r0 + rv < rows) {
        uint4 raw;
        T* e = reinterpret_cast<T*>(&raw);
#pragma unroll
        for (int i = 0; i < VE; ++i) e[i] = tile[rv + i][c];
        *reinterpret_cast<uint4*>(d + (c0 + c) * rows + r0 + rv) = raw;
      }
    }
    __syncthreads();
  }
}

// ---- grouped quantization: latents -> one contiguous [N, Dg] token slice per group ---------------------------------
// src [batch][G*Dg][hw] -> dst [G][batch*hw][Dg].  A block takes one band of kTile spatial positions of one image
// (blockIdx.x) and strides over the channel tiles (blockIdx.y, gridDim.y); the loads run along hw, the stores along
// the channels of a token, which are contiguous within a group.
template <typename T>
__global__ void __launch_bounds__(kTile * 8) split_groups_kernel(const T* __restrict__ src, int64_t hw,
                                                                 int64_t bands_per_image, int D, int Dg, int64_t N,
                                                                 T* __restrict__ dst) {
  __shared__ T tile[kTile][kTile + 1];
  const unsigned band = (unsigned)bands_per_image;   // the grid has fewer than 2^31 blocks: 32-bit division
  const int64_t b = blockIdx.x / band;
  const int64_t s0 = (int64_t)(blockIdx.x - (unsigned)b * band) * kTile;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int c0 = blockIdx.y * kTile; c0 < D; c0 += gridDim.y * kTile) {
#pragma unroll
    for (int i = ty; i < kTile; i += 8) {
      const int c = c0 + i;
      const int64_t s = s0 + tx;
      if (c < D && s < hw) tile[i][tx] = src[(b * D + c) * hw + s];
    }
    __syncthreads();
#pragma unroll
    for (int i = ty; i < kTile; i += 8) {
      const int c = c0 + tx;
      const int64_t s = s0 + i;
      if (c < D && s < hw) {
        const int g = c / Dg;
        dst[((int64_t)g * N + b * hw + s) * Dg + (c - g * Dg)] = tile[tx][i];
      }
    }
    __syncthreads();
  }
}

// Token-major src [N][G*Dg] (hw = 1): element (or, with T = uint4, 16-byte vector) i of a row goes to its group's row.
template <typename T>
__global__ void split_groups_rows_kernel(const T* __restrict__ src, int64_t N, int D, int Dg, T* __restrict__ dst) {
  const int64_t total = N * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / D;
    const int c = (int)(i - n * D), g = c / Dg;
    dst[((int64_t)g * N + n) * Dg + (c - g * Dg)] = src[i];
  }
}

// ---- token ids -> NCHW latents (decode_from_quant, vq/tasks/image_reconstruction/models.py:97-108) ----------------
// The transpose above with a different load stage: the "source row" of spatial position s is the codebook row of its
// token id.  A row source provides
//   int64_t code(int64_t n)    the id of token n if it is in [0, size), else -1
//   float4 quad(code, c)       channels c .. c+3 of that code's row (channels >= D: any value; code -1: NaN)
constexpr float kNaN = __builtin_nanf("");

template <typename TI>
__device__ __forceinline__ int64_t checked_id(const TI* __restrict__ ids, int64_t n, int64_t size) {
  const int64_t id = (int64_t)ids[n];
  return id >= 0 && id < size ? id : -1;
}

template <typename TI>
struct VqRowSource {     // nn.Embedding: row = W[id] (fp32 [K, D])
  const TI* __restrict__ ids;
  const float* __restrict__ W;
  int64_t K;
  int D;
  bool vec;              // D % 4 == 0 and W 16-byte aligned: every quad is one 16-byte load
  __device__ __forceinline__ int64_t code(int64_t n) const { return checked_id(ids, n, K); }
  __device__ __forceinline__ float4 quad(int64_t code, int c) const {
    if (code < 0) return make_float4(kNaN, kNaN, kNaN, kNaN);
    const float* row = W + code * D + c;
    if (vec) return __ldg(reinterpret_cast<const float4*>(row));
    float4 q;
    q.x = __ldg(row);
    q.y = c + 1 < D ? __ldg(row + 1) : 0.f;
    q.z = c + 2 < D ? __ldg(row + 2) : 0.f;
    q.w = c + 3 < D ? __ldg(row + 3) : 0.f;
    return q;
  }
};

template <typename TI>
struct FsqRowSource {    // implicit FSQ codebook: digit d of the mixed-radix id, digit / half - 1 (as fsq_decode_kernel)
  const TI* __restrict__ ids;
  vqb_fsq_params p;
  int64_t size;          // prod(levels)
  __device__ __forceinline__ int64_t code(int64_t n) const { return checked_id(ids, n, size); }
  __device__ __forceinline__ float value(int id, int d) const {
    if (d >= p.D) return 0.f;
    const int digit = (id / p.cumprod[d]) % p.levels[d];                 // fsq/quantizers.py:59-63
    return __fsub_rn(__fdiv_rn((float)digit, p.half[d]), 1.f);           // :137
  }
  __device__ __forceinline__ float4 quad(int64_t code, int c) const {
    if (code < 0) return make_float4(kNaN, kNaN, kNaN, kNaN);
    const int id = (int)code;                                              // size < 2^31
    return make_float4(value(id, c), value(id, c + 1), value(id, c + 2), value(id, c + 3));
  }
};

template <typename TI>
struct ResidualRowSource {   // RQ-VAE codes: token n's ids are ids[n*L .. n*L + L); row = sum_l W_l[id_l], level order
  const TI* __restrict__ ids;
  const float* W[VQB_MAX_LEVELS];   // indexed with unrolled constants only: the struct stays in the parameter bank
  int L;
  int64_t K;
  int D;
  bool vec;                  // D % 4 == 0 and every W_l 16-byte aligned
  __device__ __forceinline__ int64_t code(int64_t n) const {   // n when all L ids are in [0, K), else -1
    bool ok = true;
#pragma unroll
    for (int l = 0; l < VQB_MAX_LEVELS; ++l)
      if (l < L) ok = ok && checked_id(ids, n * L + l, K) >= 0;
    return ok ? n : -1;
  }
  __device__ __forceinline__ float4 quad(int64_t code, int c) const {
    if (code < 0) return make_float4(kNaN, kNaN, kNaN, kNaN);
    float4 s;
#pragma unroll
    for (int l = 0; l < VQB_MAX_LEVELS; ++l) {
      if (l < L) {
        const float* row = W[l] + (int64_t)ids[code * L + l] * D + c;
        float4 q;
        if (vec) {
          q = __ldg(reinterpret_cast<const float4*>(row));
        } else {
          q.x = __ldg(row);
          q.y = c + 1 < D ? __ldg(row + 1) : 0.f;
          q.z = c + 2 < D ? __ldg(row + 2) : 0.f;
          q.w = c + 3 < D ? __ldg(row + 3) : 0.f;
        }
        if (l == 0) {
          s = q;
        } else {    // the running sum of vqb_residual_step: one round-to-nearest add per level
          s.x = __fadd_rn(s.x, q.x);
          s.y = __fadd_rn(s.y, q.y);
          s.z = __fadd_rn(s.z, q.z);
          s.w = __fadd_rn(s.w, q.w);
        }
      }
    }
    return s;
  }
};

template <typename TI>
struct GroupRowSource {      // product codes: token n's ids are ids[n*G .. n*G + G); channel g*Dg + d = W_g[id_g][d]
  const TI* __restrict__ ids;
  const float* W[VQB_MAX_LEVELS];   // read through `book` (unrolled constant indices): the struct stays in the parameter bank
  int G;
  int64_t K;
  int Dg;
  int D;                     // G * Dg
  bool vec;                  // Dg % 4 == 0 and every W_g 16-byte aligned: a quad lies inside one group
  __device__ __forceinline__ int64_t code(int64_t n) const {   // n when all G ids are in [0, K), else -1
    bool ok = true;
#pragma unroll
    for (int g = 0; g < VQB_MAX_LEVELS; ++g)
      if (g < G) ok = ok && checked_id(ids, n * G + g, K) >= 0;
    return ok ? n : -1;
  }
  __device__ __forceinline__ const float* book(int g) const {
    const float* w = W[0];
#pragma unroll
    for (int k = 1; k < VQB_MAX_LEVELS; ++k)
      if (k == g) w = W[k];
    return w;
  }
  __device__ __forceinline__ float value(int64_t code, int c) const {   // channel c of the token's row
    if (c >= D) return 0.f;
    const int g = c / Dg;
    return __ldg(book(g) + (int64_t)ids[code * G + g] * Dg + (c - g * Dg));
  }
  __device__ __forceinline__ float4 quad(int64_t code, int c) const {
    if (code < 0) return make_float4(kNaN, kNaN, kNaN, kNaN);
    if (vec) {
      const int g = c / Dg;
      return __ldg(reinterpret_cast<const float4*>(book(g) + (int64_t)ids[code * G + g] * Dg + (c - g * Dg)));
    }
    return make_float4(value(code, c), value(code, c + 1), value(code, c + 2), value(code, c + 3));
  }
};

// z[b][d][s] = row(id[b * hw + s])[d].  Block = one band of TS spatial positions of one image (blockIdx.x) and a
// stride over the channel tiles of TD channels (blockIdx.y, gridDim.y); the rows go through an fp32 shared tile
// and leave as 16-byte stores along hw.  Stores fall back to scalar ones where hw is not a multiple of the vector
// (or z is not 16-byte aligned).  Each block reads its band's ids once; blockIdx.y == 0 counts the bad ones.
template <class Src, typename TO, int TS, int TD>
__global__ void __launch_bounds__(256) decode_tokens_kernel(const Src src, int64_t hw, int64_t bands_per_image, int D,
                                                            TO* __restrict__ z, bool vec_store, int* __restrict__ bad_count) {
  constexpr int VE = 16 / sizeof(TO);          // output elements per 16-byte store
  constexpr int QPR = TD / 4;                  // quads per tile row
  constexpr int VPC = TS / VE;                 // vectors per output row of the tile
  static_assert(TD % 4 == 0 && TS % VE == 0, "tile shape");
  static_assert(TS <= 256, "one id per thread: __syncthreads_count then sums the bad ids");
  __shared__ float tile[TS][TD + 1];           // +1: conflict-free column reads in the store stage
  __shared__ int64_t codes[TS];
  const int64_t b = (int64_t)blockIdx.x / bands_per_image;
  const int64_t s0 = ((int64_t)blockIdx.x - b * bands_per_image) * TS;
  const int ns = (int)min((int64_t)TS, hw - s0);
  int bad = 0;
  for (int r = threadIdx.x; r < TS; r += 256) {
    const int64_t c = r < ns ? src.code(b * hw + s0 + r) : 0;
    codes[r] = c;
    bad += c < 0;
  }
  bad = __syncthreads_count(bad);              // also publishes codes[]
  if (bad && blockIdx.y == 0 && threadIdx.x == 0 && bad_count) atomicAdd(bad_count, bad);
  TO* __restrict__ zb = z + b * D * hw;
  for (int c0 = blockIdx.y * TD; c0 < D; c0 += gridDim.y * TD) {
    for (int v = threadIdx.x; v < TS * QPR; v += 256) {
      const int r = v / QPR, cq = (v % QPR) * 4;
      if (r < ns && c0 + cq < D) {
        const float4 q = src.quad(codes[r], c0 + cq);
        tile[r][cq] = q.x;
        tile[r][cq + 1] = q.y;
        tile[r][cq + 2] = q.z;
        tile[r][cq + 3] = q.w;
      }
    }
    __syncthreads();
    // same store order as transpose_last2_vec_kernel: lanes along one output row when it is short (VPC <= 8)
    for (int v = threadIdx.x; v < TD * VPC; v += 256) {
      const int rv = (VPC <= 8 ? v % VPC : v / TD) * VE, c = VPC <= 8 ? v / VPC : v % TD;
      if (c0 + c < D && rv < ns) {
        TO* out = zb + (int64_t)(c0 + c) * hw + s0 + rv;
        if (vec_store && rv + VE <= ns) {
          uint4 raw;
          TO* e = reinterpret_cast<TO*>(&raw);
#pragma unroll
          for (int i = 0; i < VE; ++i) e[i] = from_f32<TO>(tile[rv + i][c]);
          *reinterpret_cast<uint4*>(out) = raw;
        } else {
          for (int i = 0; i < VE && rv + i < ns; ++i) out[i] = from_f32<TO>(tile[rv + i][c]);
        }
      }
    }
    __syncthreads();
  }
}

template <int TS, int TD, class Src>
static int launch_decode_tokens(const Src& src, int64_t batch, int64_t hw, int D, void* z, int out_dtype, int* bad,
                                cudaStream_t st) {
  const int64_t per_image = (hw + TS - 1) / TS, bands = per_image * batch;
  VQB_REQUIRE(bands <= 0x7fffffff, "decode_tokens: too many tokens (batch * ceil(hw / %d) must be < 2^31)", TS);
  const int64_t ct = (D + TD - 1) / TD;
  int64_t gy = ((int64_t)sm_count() * 16 + bands - 1) / bands;   // enough blocks for ~2 waves, as the transpose
  gy = gy > ct ? ct : (gy < 1 ? 1 : gy);
  const dim3 grid((unsigned)bands, (unsigned)gy);
  const int ve = out_dtype == VQB_F32 ? 4 : 8;
  const bool vec_store = hw % ve == 0 && (uintptr_t)z % 16 == 0;
  if (out_dtype == VQB_F32)
    decode_tokens_kernel<Src, float, TS, TD><<<grid, 256, 0, st>>>(src, hw, per_image, D, (float*)z, vec_store, bad);
  else
    decode_tokens_kernel<Src, __nv_bfloat16, TS, TD><<<grid, 256, 0, st>>>(src, hw, per_image, D, (__nv_bfloat16*)z,
                                                                           vec_store, bad);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

// tile shape follows the row width, as in vqb_transpose_last2: narrow rows (LlamaGen's 8, FSQ's 5-6) get a narrow tile
template <class Src>
static int launch_decode_tokens_for_width(const Src& src, int64_t batch, int64_t hw, int D, void* z, int out_dtype,
                                          int* bad, cudaStream_t st) {
  if (D <= 16) return launch_decode_tokens<128, 16>(src, batch, hw, D, z, out_dtype, bad, st);
  if (D <= 32) return launch_decode_tokens<64, 32>(src, batch, hw, D, z, out_dtype, bad, st);
  return launch_decode_tokens<32, 64>(src, batch, hw, D, z, out_dtype, bad, st);
}

static int check_decode_args(const char* fn, const void* ids, int id_bytes, int64_t batch, int64_t hw, const void* z,
                             int out_dtype) {
  VQB_REQUIRE(ids && z, "%s: null pointer", fn);
  VQB_REQUIRE(id_bytes == 2 || id_bytes == 4 || id_bytes == 8, "%s: id_bytes must be 2 (uint16), 4 (int32) or 8 (int64)", fn);
  VQB_REQUIRE(out_dtype == VQB_F32 || out_dtype == VQB_BF16, "%s: out_dtype must be VQB_F32 or VQB_BF16", fn);
  VQB_REQUIRE(batch >= 0 && hw >= 0, "%s: bad shape", fn);
  return VQB_OK;
}

template <typename TO>
__global__ void compact_tokens_kernel(const unsigned long long* __restrict__ keys, int64_t n, int64_t offset,
                                      TO* __restrict__ out) {
  // 8 keys per thread: four 128-bit loads, 16 (uint16) or 32 (int32) bytes stored contiguously
  const int64_t n8 = n / 8;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    ulonglong2 k[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) k[j] = reinterpret_cast<const ulonglong2*>(keys)[i * 4 + j];
    TO v[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] = (TO)(k[j].x == kNoKey ? 0 : (int64_t)key_index(k[j].x) - offset);
      v[2 * j + 1] = (TO)(k[j].y == kNoKey ? 0 : (int64_t)key_index(k[j].y) - offset);
    }
    if constexpr (sizeof(TO) == 2) {
      reinterpret_cast<uint4*>(out)[i] = *reinterpret_cast<const uint4*>(v);
    } else {
      reinterpret_cast<uint4*>(out)[2 * i] = *reinterpret_cast<const uint4*>(v);
      reinterpret_cast<uint4*>(out)[2 * i + 1] = *reinterpret_cast<const uint4*>(v + 4);
    }
  }
  for (int64_t i = n8 * 8 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long k = keys[i];
    out[i] = (TO)(k == kNoKey ? 0 : (int64_t)key_index(k) - offset);
  }
}

}  // namespace vqb

using namespace vqb;

extern "C" {

int vqb_transpose_last2(const void* src, int elem_bytes, int64_t batch, int64_t rows, int64_t cols, void* dst,
                        void* stream) {
  VQB_REQUIRE(src && dst, "vqb_transpose_last2: null pointer");
  VQB_REQUIRE(src != dst, "vqb_transpose_last2: in-place transpose is not supported");
  VQB_REQUIRE(elem_bytes == 2 || elem_bytes == 4 || elem_bytes == 8, "vqb_transpose_last2: elem_bytes must be 2, 4 or 8");
  VQB_REQUIRE(batch >= 0 && rows >= 0 && cols >= 0, "vqb_transpose_last2: bad shape");
  if (batch == 0 || rows == 0 || cols == 0) return VQB_OK;
  VQB_REQUIRE(batch <= 65535 && (rows + 15) / 16 <= 65535, "vqb_transpose_last2: grid limit (batch, rows/16 <= 65535)");
  cudaStream_t st = (cudaStream_t)stream;
  const int ve = 16 / elem_bytes;
  if (rows % ve == 0 && cols % ve == 0 && (uintptr_t)src % 16 == 0 && (uintptr_t)dst % 16 == 0) {
    // tile shape follows the matrix: a narrow side (channels = 8 or 16) gets a narrow tile
#define VQB_TR_CASE(T_, TR_, TC_)                                                                              \
    do {                                                                                                       \
      const int64_t ct = (cols + TC_ - 1) / TC_, rt = (rows + TR_ - 1) / TR_;                                   \
      int64_t gx = ((int64_t)sm_count() * 16 + rt * batch - 1) / (rt * batch); /* enough blocks for ~2 waves */ \
      if (gx > ct) gx = ct;                                                                                    \
      if (gx < 1) gx = 1;                                                                                      \
      const dim3 vgrid((unsigned)gx, (unsigned)rt, (unsigned)batch);                                           \
      transpose_last2_vec_kernel<T_, TR_, TC_><<<vgrid, 256, 0, st>>>((const T_*)src, rows, cols, (T_*)dst);   \
    } while (0)
#define VQB_TR_SHAPE(T_)                                      \
    do {                                                      \
      if (cols <= 16) VQB_TR_CASE(T_, 128, 16);               \
      else if (rows <= 16) VQB_TR_CASE(T_, 16, 128);          \
      else if (cols <= 32) VQB_TR_CASE(T_, 64, 32);           \
      else VQB_TR_CASE(T_, 32, 64);                           \
    } while (0)
    if (elem_bytes == 2) VQB_TR_SHAPE(uint16_t);
    else if (elem_bytes == 4) VQB_TR_SHAPE(uint32_t);
    else VQB_TR_SHAPE(unsigned long long);
#undef VQB_TR_SHAPE
#undef VQB_TR_CASE
    VQB_LAUNCH_OK();
    return VQB_OK;
  }
  const dim3 grid((unsigned)((cols + kTile - 1) / kTile), (unsigned)((rows + kTile - 1) / kTile), (unsigned)batch);
  const dim3 block(kTile, 8);
  if (elem_bytes == 2)
    transpose_last2_kernel<uint16_t><<<grid, block, 0, st>>>((const uint16_t*)src, rows, cols, (uint16_t*)dst);
  else if (elem_bytes == 4)
    transpose_last2_kernel<uint32_t><<<grid, block, 0, st>>>((const uint32_t*)src, rows, cols, (uint32_t*)dst);
  else
    transpose_last2_kernel<unsigned long long><<<grid, block, 0, st>>>((const unsigned long long*)src, rows, cols,
                                                                        (unsigned long long*)dst);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

int vqb_compact_tokens(const unsigned long long* keys, int64_t n, int64_t index_offset, void* out, int out_bytes,
                       void* stream) {
  VQB_REQUIRE(keys && out, "vqb_compact_tokens: null pointer");
  VQB_REQUIRE(out_bytes == 2 || out_bytes == 4, "vqb_compact_tokens: out_bytes must be 2 (uint16) or 4 (int32)");
  if (n <= 0) return VQB_OK;
  VQB_REQUIRE((uintptr_t)keys % 16 == 0 && (uintptr_t)out % 16 == 0, "vqb_compact_tokens: 16-byte aligned buffers");
  int blocks = (int)((n / 8 + 255) / 256);
  if (blocks < 1) blocks = 1;
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (out_bytes == 2) compact_tokens_kernel<uint16_t><<<blocks, 256, 0, st>>>(keys, n, index_offset, (uint16_t*)out);
  else compact_tokens_kernel<int32_t><<<blocks, 256, 0, st>>>(keys, n, index_offset, (int32_t*)out);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

int vqb_decode_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const float* W, int64_t K, int D,
                      void* z_out, int out_dtype, int* bad_count, void* stream) {
  if (int e = check_decode_args("vqb_decode_tokens", ids, id_bytes, batch, hw, z_out, out_dtype)) return e;
  VQB_REQUIRE(W, "vqb_decode_tokens: null pointer");
  VQB_REQUIRE(K >= 1 && D >= 1, "vqb_decode_tokens: bad codebook shape");
  if (batch == 0 || hw == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = D % 4 == 0 && (uintptr_t)W % 16 == 0;
  if (id_bytes == 2)
    return launch_decode_tokens_for_width(VqRowSource<uint16_t>{(const uint16_t*)ids, W, K, D, vec}, batch, hw, D, z_out,
                                          out_dtype, bad_count, st);
  if (id_bytes == 4)
    return launch_decode_tokens_for_width(VqRowSource<int32_t>{(const int32_t*)ids, W, K, D, vec}, batch, hw, D, z_out,
                                          out_dtype, bad_count, st);
  return launch_decode_tokens_for_width(VqRowSource<int64_t>{(const int64_t*)ids, W, K, D, vec}, batch, hw, D, z_out,
                                        out_dtype, bad_count, st);
}

int vqb_decode_residual_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const vqb_residual_levels* lv,
                               int64_t K, int D, void* z_out, int out_dtype, int* bad_count, void* stream) {
  if (int e = check_decode_args("vqb_decode_residual_tokens", ids, id_bytes, batch, hw, z_out, out_dtype)) return e;
  VQB_REQUIRE(lv, "vqb_decode_residual_tokens: null levels");
  VQB_REQUIRE(lv->L >= 1 && lv->L <= VQB_MAX_LEVELS, "vqb_decode_residual_tokens: L=%d outside [1, %d]", lv->L,
              VQB_MAX_LEVELS);
  VQB_REQUIRE(K >= 1 && D >= 1, "vqb_decode_residual_tokens: bad codebook shape");
  bool aligned = true;
  for (int l = 0; l < lv->L; ++l) {
    VQB_REQUIRE(lv->W[l], "vqb_decode_residual_tokens: null codebook at level %d", l);
    aligned = aligned && (uintptr_t)lv->W[l] % 16 == 0;
  }
  if (batch == 0 || hw == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = D % 4 == 0 && aligned;
#define VQB_RESIDUAL_SRC(TI_) \
  ResidualRowSource<TI_> src{(const TI_*)ids, {}, lv->L, K, D, vec};                                                  \
  for (int l = 0; l < lv->L; ++l) src.W[l] = lv->W[l];                                                               \
  return launch_decode_tokens_for_width(src, batch, hw, D, z_out, out_dtype, bad_count, st);
  if (id_bytes == 2) {
    VQB_RESIDUAL_SRC(uint16_t)
  }
  if (id_bytes == 4) {
    VQB_RESIDUAL_SRC(int32_t)
  }
  VQB_RESIDUAL_SRC(int64_t)
#undef VQB_RESIDUAL_SRC
}

int vqb_decode_group_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const vqb_residual_levels* lv,
                            int64_t K, int Dg, void* z_out, int out_dtype, int* bad_count, void* stream) {
  if (int e = check_decode_args("vqb_decode_group_tokens", ids, id_bytes, batch, hw, z_out, out_dtype)) return e;
  VQB_REQUIRE(lv, "vqb_decode_group_tokens: null groups");
  VQB_REQUIRE(lv->L >= 1 && lv->L <= VQB_MAX_LEVELS, "vqb_decode_group_tokens: G=%d outside [1, %d]", lv->L,
              VQB_MAX_LEVELS);
  VQB_REQUIRE(K >= 1 && Dg >= 1 && (int64_t)Dg * lv->L <= 0x7fffffff, "vqb_decode_group_tokens: bad codebook shape");
  bool aligned = true;
  for (int g = 0; g < lv->L; ++g) {
    VQB_REQUIRE(lv->W[g], "vqb_decode_group_tokens: null codebook of group %d", g);
    aligned = aligned && (uintptr_t)lv->W[g] % 16 == 0;
  }
  if (batch == 0 || hw == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int D = Dg * lv->L;
  const bool vec = Dg % 4 == 0 && aligned;
#define VQB_GROUP_SRC(TI_) \
  GroupRowSource<TI_> src{(const TI_*)ids, {}, lv->L, K, Dg, D, vec};                                               \
  for (int g = 0; g < lv->L; ++g) src.W[g] = lv->W[g];                                                              \
  return launch_decode_tokens_for_width(src, batch, hw, D, z_out, out_dtype, bad_count, st);
  if (id_bytes == 2) {
    VQB_GROUP_SRC(uint16_t)
  }
  if (id_bytes == 4) {
    VQB_GROUP_SRC(int32_t)
  }
  VQB_GROUP_SRC(int64_t)
#undef VQB_GROUP_SRC
}

int vqb_split_groups(const void* src, int dtype, int64_t batch, int G, int Dg, int64_t hw, void* dst, void* stream) {
  VQB_REQUIRE(src && dst, "vqb_split_groups: null pointer");
  VQB_REQUIRE(src != dst, "vqb_split_groups: in-place split is not supported");
  VQB_REQUIRE(dtype == VQB_F32 || dtype == VQB_BF16, "vqb_split_groups: dtype must be VQB_F32 or VQB_BF16");
  VQB_REQUIRE(G >= 1 && G <= VQB_MAX_LEVELS, "vqb_split_groups: G=%d outside [1, %d]", G, VQB_MAX_LEVELS);
  VQB_REQUIRE(Dg >= 1 && (int64_t)Dg * G <= 0x7fffffff && batch >= 0 && hw >= 1, "vqb_split_groups: bad shape");
  if (batch == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int D = G * Dg, eb = dtype == VQB_F32 ? 4 : 2;
  const int64_t N = batch * hw;
  if (hw == 1) {
    const int ve = 16 / eb;
    const bool vec = Dg % ve == 0 && (uintptr_t)src % 16 == 0 && (uintptr_t)dst % 16 == 0;
    const int64_t items = vec ? N * D / ve : N * D;
    int64_t blocks = (items + 255) / 256;
    if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
    if (vec)
      split_groups_rows_kernel<uint4><<<(unsigned)blocks, 256, 0, st>>>((const uint4*)src, N, D / ve, Dg / ve, (uint4*)dst);
    else if (eb == 4)
      split_groups_rows_kernel<uint32_t><<<(unsigned)blocks, 256, 0, st>>>((const uint32_t*)src, N, D, Dg, (uint32_t*)dst);
    else
      split_groups_rows_kernel<uint16_t><<<(unsigned)blocks, 256, 0, st>>>((const uint16_t*)src, N, D, Dg, (uint16_t*)dst);
    VQB_LAUNCH_OK();
    return VQB_OK;
  }
  const int64_t per_image = (hw + kTile - 1) / kTile, bands = per_image * batch;
  VQB_REQUIRE(bands <= 0x7fffffff, "vqb_split_groups: too many tokens (batch * ceil(hw / %d) must be < 2^31)", kTile);
  const int64_t ct = (D + kTile - 1) / kTile;
  int64_t gy = ((int64_t)sm_count() * 16 + bands - 1) / bands;   // enough blocks for ~2 waves, as the transpose
  gy = gy > ct ? ct : (gy < 1 ? 1 : gy);
  const dim3 grid((unsigned)bands, (unsigned)gy), block(kTile, 8);
  if (eb == 4)
    split_groups_kernel<uint32_t><<<grid, block, 0, st>>>((const uint32_t*)src, hw, per_image, D, Dg, N, (uint32_t*)dst);
  else
    split_groups_kernel<uint16_t><<<grid, block, 0, st>>>((const uint16_t*)src, hw, per_image, D, Dg, N, (uint16_t*)dst);
  VQB_LAUNCH_OK();
  return VQB_OK;
}

int vqb_fsq_decode_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const vqb_fsq_params* p_host,
                          void* z_out, int out_dtype, int* bad_count, void* stream) {
  if (int e = check_decode_args("vqb_fsq_decode_tokens", ids, id_bytes, batch, hw, z_out, out_dtype)) return e;
  VQB_REQUIRE(p_host, "vqb_fsq_decode_tokens: null params");
  VQB_REQUIRE(p_host->D >= 1 && p_host->D <= 16, "vqb_fsq_decode_tokens: D must be in 1..16 (got %d)", p_host->D);
  int64_t size = 1;
  for (int d = 0; d < p_host->D && size <= 0x7fffffff; ++d) {
    VQB_REQUIRE(p_host->levels[d] >= 1, "vqb_fsq_decode_tokens: levels must be >= 1");
    size *= p_host->levels[d];
  }
  VQB_REQUIRE(size <= 0x7fffffff, "vqb_fsq_decode_tokens: codebook size must be below 2^31");
  if (batch == 0 || hw == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int D = p_host->D;    // <= 16: one 128 x 16 tile shape
  if (id_bytes == 2)
    return launch_decode_tokens<128, 16>(FsqRowSource<uint16_t>{(const uint16_t*)ids, *p_host, size}, batch, hw, D, z_out,
                                         out_dtype, bad_count, st);
  if (id_bytes == 4)
    return launch_decode_tokens<128, 16>(FsqRowSource<int32_t>{(const int32_t*)ids, *p_host, size}, batch, hw, D, z_out,
                                         out_dtype, bad_count, st);
  return launch_decode_tokens<128, 16>(FsqRowSource<int64_t>{(const int64_t*)ids, *p_host, size}, batch, hw, D, z_out,
                                       out_dtype, bad_count, st);
}

}  // extern "C"
