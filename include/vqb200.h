/*
 * vqb200.h — C-ABI of the B200-native codebook-quantization hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): plain pointers and sizes, no torch
 * types.  The reference (magic-research/vector_quantization) is 100 % Python and
 * has no FFI of its own; every entry point below replaces the ATen/cuBLAS call
 * sequence of one reference function, cited as file:line relative to the
 * reference root.  The Python host layer (`vector_quantization_b200/`) binds these
 * with ctypes; `INTEGRATION.md` shows the stub a reference maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *  - `stream` is a `cudaStream_t` passed as `void*` (0 = legacy default stream);
 *  - the caller allocates everything (outputs and workspaces); nothing is
 *    allocated, freed or synchronised inside the library;
 *  - return value: 0 on success, negative `vqb_status` on error; the message is
 *    available from `vqb_last_error()` (thread-local);
 *  - dtype codes: `VQB_F32` / `VQB_BF16`; all reductions and statistics are fp32;
 *  - there is NO CPU implementation behind any entry point.
 */
#ifndef VQB200_H_
#define VQB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQB200_ABI_VERSION 3 /* 2: fp16 plane formats, vqb_row_inv_norm(f16_rows), vqb_transpose_last2, vqb_compact_tokens; 3: vqb_comm_*, g_dtype of vqb_quantize_backward;
                                3 (additive): vqb_segment_chunk, vqb_code_sort*, vqb_segment_sum_*, vqb_quantize_backward_rows,
                                vqb_decode_tokens, vqb_fsq_decode_tokens */

typedef enum { VQB_OK = 0, VQB_ERR_ARG = -1, VQB_ERR_CUDA = -2, VQB_ERR_UNSUPPORTED = -3 } vqb_status;
typedef enum { VQB_F32 = 0, VQB_BF16 = 1 } vqb_dtype;
typedef enum { VQB_BACKEND_TCGEN05 = 0, VQB_BACKEND_SIMT = 1 } vqb_backend;

/* ---- library ---------------------------------------------------------------------------- */
int vqb_abi_version(void);
const char* vqb_last_error(void);
/* Fills SM count / compute capability of the current device. */
int vqb_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- operand packing -------------------------------------------------------------------- *
 * The distance contraction runs on bf16 tensor cores with fp32 accumulation.  An fp32 matrix
 * is represented EXACTLY as a sum of up to three bf16 "planes" (hi + mid + lo, 3 x 8 mantissa
 * bits); a bf16 matrix is one plane.  `vqb_pack_rows` builds the zero-padded K-major operand
 * buffer  bf16[planes][rows_pad][Dp]  that the TMA descriptors of `vqb_assign` read, and the
 * per-row fp32 side terms.  It also performs the reference's row normalisation:
 *   F.normalize(v) = v / max(||v||, 1e-12)      vq/algorithms/vq/callbacks/normalize.py:24,27
 *                                               vq/algorithms/vq/distances.py:41-42
 * Dp       = vqb_operand_dp(D)        (16, 32 or a multiple of 64)
 * rows_pad = vqb_operand_rows_pad(rows) (multiple of 256)
 *
 * Plane formats (the `planes` / `*_nplanes` arguments):
 *   1..3              bf16 planes hi, mid, lo:  v == hi + mid + lo exactly for 3 planes of an fp32 value.
 *   VQB_PLANES_F16    one IEEE fp16 plane of a bf16 source (`normalize` = 0): exact for 2^-17 <= |v| < 2^15
 *                     (abs. error <= 2^-25 below; a row with a component >= 2^15 is scaled by a power of two,
 *                     which leaves its arg-max unchanged).  The tensor core cannot mix fp16 and bf16 operands,
 *                     so this is how one-plane bf16 tokens meet a VQB_PLANES_F16X2 codebook.
 *   VQB_PLANES_F16X2  two IEEE fp16 planes (hi, lo'):  hi = fp16(v), lo' = fp16((v - hi) * 2^11), so that
 *                     v = hi + lo' * 2^-11 to 22 significant bits (abs. error <= max(2^-22 |v|, 2^-36)).
 *                     Only for l2-normalised rows (|v| <= 1, `normalize` = 1).  `vqb_assign` accumulates the
 *                     lo' term first and folds the 2^-11 into the accumulator with the tensor core's
 *                     scale-input-d, so an fp32 codebook costs TWO MMA terms against one-plane tokens
 *                     instead of three.  The other operand must be VQB_PLANES_F16 or VQB_PLANES_F16X2
 *                     (both operands of one vqb_assign call are bf16 planes, or both are fp16 planes).
 */
#define VQB_PLANES_F16 0x11
#define VQB_PLANES_F16X2 0x12
#define VQB_PLANE_COUNT(p) ((p) & 0xf)
int64_t vqb_operand_dp(int D);
int64_t vqb_operand_rows_pad(int64_t rows);
size_t vqb_operand_bytes(int64_t rows, int D, int planes);
int vqb_pack_rows(const void* src, int src_dtype, int64_t rows, int D,
                  int normalize,            /* 1: pack F.normalize(row) instead of row */
                  int planes,               /* 1..3 bf16 planes, VQB_PLANES_F16 (bf16 source, normalize = 0) or VQB_PLANES_F16X2 (normalize = 1) */
                  void* dst_planes,         /* 16-bit [VQB_PLANE_COUNT(planes)][rows_pad][Dp], fully written (padding zeroed) */
                  float* half_sqnorm,       /* optional [rows_pad]: 0.5*||packed row||^2 (fp32); +inf in padding */
                  float* writeback_f32,     /* optional [rows, D]: the (normalised) fp32 row; may alias src when src is fp32 */
                  unsigned long long* keys_to_reset, int64_t n_keys, /* optional: fill with 0xFF.. (fused memset for vqb_assign) */
                  void* zero_fill, int64_t zero_bytes, /* optional: fused zero-fill (16-byte aligned, multiple of 16 bytes) of the step's statistics buffer */
                  float* lo_norm_max, /* optional, VQB_PLANES_F16X2: *lo_norm_max = max(*lo_norm_max, max_j |row_j - hi_j|_2), the error
                                         bound of a contraction that uses the hi plane only (pre-zeroed DEVICE scalar) */
                  void* stream);

/* ---- nearest-code assignment ------------------------------------------------------------ *
 * Replaces VectorQuantizer._encode = distance + argmin      vq/algorithms/vq/quantizers.py:92-100
 *   L2Distance  torch.cdist                                 vq/algorithms/vq/distances.py:28-32
 *   CosineDistance 1 - normalize(x) normalize(e)^T          vq/algorithms/vq/distances.py:35-46
 * and, with the operands swapped, NearestAnchor's column argmin `d.argmin(0)`
 *                                                           vq/algorithms/cvqvae/anchors.py:83
 * WITHOUT materialising the [a_rows x b_rows] matrix.  For every row i of A it finds
 *      argmax_j  score(i,j) = <A_i, B_j> - b_side[j]   (side_mode 1)   or   <A_i, B_j> * b_side[j]   (side_mode 2)
 * which is argmin_j ||A_i - B_j|| (L2) or argmin_j (1 - cos) when B rows are normalised.
 * Ties resolve to the lowest j (torch.argmin semantics).  The result is min-combined into
 *      keys[i] = (~orderable(score) << 32) | (uint32)(j + b_index_offset)
 * with 64-bit atomicMin, so several launches (codebook shards) and several GPUs (packed
 * min-loc all-reduce) compose.  keys must be initialised to all-ones.
 * `*_plane_rows` is the row stride between planes: 0 = the padded default of vqb_pack_rows; a bf16 [rows, D]
 * tensor with D == vqb_operand_dp(D) is already a valid one-plane operand and can be passed ZERO-COPY with
 * plane_rows = rows (TMA zero-fills the out-of-bounds rows of the last tile).
 * backend VQB_BACKEND_TCGEN05: TMA -> smem -> tcgen05.mma (TMEM accumulators) -> fused argmax
 * epilogue; VQB_BACKEND_SIMT: fp32 CUDA-core kernel with the same contract (cross-check).
 */
int vqb_assign(const void* a_planes, int a_nplanes, int64_t a_rows, int64_t a_plane_rows,
               const void* b_planes, int b_nplanes, int64_t b_rows, int64_t b_plane_rows,
               int D, const float* b_side /* fp32 [vqb_operand_rows_pad(b_rows)] or NULL */,
               int side_mode /* 0 none, 1: score -= b_side[j] (L2, 0.5|b_j|^2), 2: score *= b_side[j] (1/|b_j|) */,
               int64_t b_index_offset,
               unsigned long long* keys, int backend, void* stream);

/* vqb_assign plus the two hooks of the CERTIFIED ONE-TERM pass (D >= 128 is bound by the tensor pipe, and an fp32
 * codebook costs two MMA terms as an fp16 pair):
 *   second_keys  optional [a_rows], all-ones initialised: receives the packed key of the RUNNER-UP score of every row
 *                (index field unspecified).  Run the contraction with the hi plane only (b_nplanes = VQB_PLANES_F16 on a
 *                pair buffer), then vqb_certify: a row whose best - runner-up exceeds twice the operand error bound has
 *                provably the same arg-max as the two-term contraction; the others are re-run exactly.
 *   a_rows_dev   optional DEVICE int: the number of valid A rows is min(a_rows, *a_rows_dev) (the re-run of the
 *                uncertified rows: their count only exists on the device; a_rows is the capacity of the buffer). */
int vqb_assign_ex(const void* a_planes, int a_nplanes, int64_t a_rows, int64_t a_plane_rows,
                  const void* b_planes, int b_nplanes, int64_t b_rows, int64_t b_plane_rows,
                  int D, const float* b_side, int side_mode, int64_t b_index_offset,
                  unsigned long long* keys, unsigned long long* second_keys, const int* a_rows_dev, int backend,
                  void* stream);
/* Lists, in ASCENDING row order (deterministic: every rank of a sharded run builds the same list), the rows r with
 *   score(keys[r]) - score(second_keys[r]) <= 2 * eps_r,   eps_r = (*delta + noise) * s_r,
 * s_r = 1 / row_inv_norm[r] (the token norm: scores are <x_r, e_j>) or 1 when row_inv_norm is NULL (scores already
 * carry the 1/|x| column scale); *delta = max_j |e_j - hi_j| from vqb_pack_rows.  *count receives their number and
 * compact_keys[0 .. count) is reset to all-ones for the exact re-run.  workspace: vqb_certify_workspace_bytes(rows). */
int64_t vqb_certify_workspace_bytes(int64_t rows);
int vqb_certify(const unsigned long long* keys, const unsigned long long* second_keys, int64_t rows,
                const float* row_inv_norm, const float* delta, float noise, int* row_list, int* count,
                unsigned long long* compact_keys, void* workspace, void* stream);
/* CVQ-VAE (cvqvae/quantizer_callback.py:94-102): lists, in ascending order, the codes whose anchor can get a NON-ZERO
 * blend weight this step.  In fp32 the per-code decay 1 - exp(-p*K*10/(1-gamma) - eps) is exactly 1 for every code
 * used at more than ~2 % of the uniform rate, so its anchor is multiplied by exactly 0: only the listed codes need the
 * column arg-min (NearestAnchor) and an anchor row.  Evaluated on a lower bound of the new probability (this rank's
 * counts over the GLOBAL token total): a superset of the truly affected codes on every rank, no exchange needed.
 * Outputs and workspace as vqb_certify (vqb_certify_workspace_bytes(K)). */
int vqb_cvq_needy_codes(const float* prob, const int64_t* counts_local, float total_global, int64_t K, float decay,
                        float one_minus_decay, float eps, int* code_list, int* count,
                        unsigned long long* compact_keys, void* workspace, void* stream);
/* dst[p][i][:] = src[p][row_list[i]][:] for i < *count (16-bit planes, Dp a multiple of 8) */
int vqb_gather_plane_rows(const void* src, int nplanes, int64_t src_plane_rows, int Dp, const int* row_list,
                          const int* count, int64_t cap, void* dst, int64_t dst_plane_rows, void* stream);
/* dst[i] = src[row_list[i]] for i < *count (fp32 side vectors of the gathered rows) */
int vqb_gather_f32(const float* src, const int* row_list, const int* count, int64_t cap, float* dst, void* stream);
/* keys[row_list[i]] = compact_keys[i] for i < *count */
int vqb_scatter_keys(const unsigned long long* compact_keys, const int* row_list, const int* count, int64_t cap,
                     unsigned long long* keys, void* stream);

/* L2 distance (reference: torch.cdist in L2Distance.forward, vq/algorithms/vq/distances.py:28-35) when the operand
 * width leaves VQB_L2_FOLD_COLUMNS spare zero columns (Dp - D >= 6; LlamaGen's D = 8 -> Dp = 16): the -0.5|.|^2 side
 * terms are written INTO the packed exact-bf16 planes, so that the plain contraction over Dp columns already is
 * <x_i, e_j> - 0.5|e_j|^2 - 0.5|x_i|^2 = -0.5 |x_i - e_j|^2 and vqb_assign runs with side_mode 0 (the per-column
 * subtraction of side_mode 1 doubles the instruction count of the D <= 64 epilogue).  Columns D..D+2 carry the codes'
 * term (the codes operand holds the three exact bf16 pieces of -0.5|e|^2, the tokens operand holds 1), columns
 * D+3..D+5 the tokens' term the other way round; an operand with 3 planes keeps its pieces in one column across the
 * planes, an operand with fewer planes spreads them over its three columns of plane 0.
 * role 0: tokens (half_sqnorm may be NULL: the term is constant along the row arg-min), role 1: codes.
 * Call after vqb_pack_rows on the same stream; both operands of a vqb_assign must be folded, with opposite roles. */
#define VQB_L2_FOLD_COLUMNS 6
int vqb_fold_l2_side(void* planes, int n_planes /* 1..3 exact bf16 planes */, int64_t rows, int D,
                     const float* half_sqnorm, int role, void* stream);
/* vqb_pack_rows with the fold fused into the pack launch (no second launch when D is a multiple of 8).
 * fold_role 0: tokens without their own term (row arg-min), 1: codes, 2: tokens with their term (column arg-min). */
int vqb_pack_rows_fold(const void* src, int src_dtype, int64_t rows, int D, int normalize, int planes /* 1..3 */,
                       void* dst_planes, float* half_sqnorm, float* writeback_f32, unsigned long long* keys_to_reset,
                       int64_t n_keys, void* zero_fill, int64_t zero_bytes, int fold_role, void* stream);

/* out[r] = 1 / max(||x_r||, 1e-12), zero in the padding up to vqb_operand_rows_pad(rows): the side_mode-2 column
 * scale that lets the column arg-min of NearestAnchor use RAW (un-normalised, one exact bf16 plane) tokens. */
int vqb_row_inv_norm(const void* x, int x_dtype, int64_t rows, int D,
                     int f16_rows /* 1: the rows are fed as a VQB_PLANES_F16 plane; its power-of-two row scale is folded in */,
                     float* out, void* stream);

/* keys -> int64 indices (and optional fp32 scores); `index_offset` is subtracted. */
int vqb_unpack_keys(const unsigned long long* keys, int64_t n, int64_t index_offset,
                    int64_t* index_out, float* score_out, void* stream);
/* Tokenise-only output (SURVEY.md §8f-3): keys -> compact token ids for the token dumps of
 * vq/tasks/image_tokenization/runners/callbacks.py:40-53 and tools/tokenize_llamagen.py:93-103.
 * out_bytes 2: uint16 (codebooks of at most 65 536 codes), 4: int32. */
int vqb_compact_tokens(const unsigned long long* keys, int64_t n, int64_t index_offset, void* out, int out_bytes,
                       void* stream);
/* Batched transpose of the last two dims, src [batch][rows][cols] -> dst [batch][cols][rows], elem_bytes 2|4|8:
 * the caller's `b c h w -> (b h w) c` (rows = c, cols = h*w) and `(b h w) c -> b c h w` (rows = h*w, cols = c)
 * rearranges around the quantizer, vq/tasks/image_tokenization/models/base.py:124,126-127. */
int vqb_transpose_last2(const void* src, int elem_bytes, int64_t batch, int64_t rows, int64_t cols, void* dst,
                        void* stream);
/* Flip bit 63 so signed-int64 MIN (NCCL/gloo ReduceOp.MIN on torch.int64) orders like unsigned. */
int vqb_keys_flip_sign(unsigned long long* keys, int64_t n, void* stream);

/* ---- codebook gather + straight-through + loss reduction -------------------------------- *
 * Replaces  nn.Embedding gather          vq/algorithms/vq/quantizers.py:102-108
 *           ste: x + (z - x).detach()    vq/tasks/image_tokenization/models/quantizers/utils/ste.py:9-10
 *           CodebookLoss/CommitmentLoss  vq/algorithms/vq/losses.py:41-62 (todd MSELoss, mean; norm=True
 *                                        normalises both arguments first)
 * One pass.  mse4_out = { mean((z-x)^2) [codebook role], same [commitment role],
 *                         mean((n(z)-n(x))^2) [codebook role], same [commitment role] }
 * (the two roles have equal value and different gradient routing).  The reduction is a
 * deterministic two-stage sum: `partials` needs vqb_loss_partials_count() floats x 2 and
 * `ticket` one zero-initialised uint32 (self-resetting).
 */
int64_t vqb_loss_partials_count(void);
int vqb_gather_ste_loss(const void* x, int x_dtype, int64_t N, int D,
                        int normalize_x,               /* 1: the quantizer sees F.normalize(x) (NormalizeCallback, normalize.py:24) */
                        const float* W, int64_t K,
                        const int64_t* quant,          /* [N] indices, or NULL when `keys` is given */
                        const unsigned long long* keys, int64_t key_index_offset, /* packed keys of vqb_assign */
                        int64_t* quant_out,            /* optional [N]: the unpacked indices (memo['quant']) */
                        float* x_norm_out,             /* optional [N,D]: F.normalize(x) (memo['x']) */
                        float* z_ste_out,              /* [N,D] fp32 value x' + (W[q] - x'), x' = (normalised) x */
                        int64_t z_hw,                  /* 0: z token-major [N,D]; h*w > 0: z written as NCHW [N/hw, D, hw] — the caller's
                                                          '(b h w) c -> b c h w' (models/base.py:126-127) fused into the store */
                        int want_norm_mse,
                        float* mse4_out, float* partials, unsigned int* ticket, void* stream);

/* Plain codebook gather out[i] = W[quant[i]] (fp32) — VectorQuantizer._decode on its own, as used by
 * decode_from_quant (vq/tasks/image_reconstruction/models.py:97-108); any index shape, flattened. */
int vqb_embedding_gather(const float* W, int64_t K, int D, const int64_t* quant, int64_t n, float* out,
                         void* stream);

/* Backward of the above (closed form, SURVEY.md App. A.6):
 *   gx = g_zste + g4[1]*2(x-z)/(ND) + J_n(x)^T [ g4[3]*2(n(x)-n(z))/(ND) ]
 *   gW[q] += g4[0]*2(z-x)/(ND) + J_n(z)^T [ g4[2]*2(n(z)-n(x))/(ND) ]     (fp32 atomics; gW pre-zeroed or NULL)
 * g4[i] are the four DEVICE scalars g_codebook, g_commitment, g_codebook_norm, g_commitment_norm (NULL = 0).  With normalize_x the chain through
 * F.normalize is applied as well: gx = J_n(x)^T g_x' (the backward of NormalizeCallback.before_encode). */
int vqb_quantize_backward(const void* g_zste, int g_dtype /* VQB_F32, or VQB_BF16 with bf16 tokens */,
                          const void* x, int x_dtype, int normalize_x,
                          const float* W, int64_t K, const int64_t* quant, int64_t N, int D,
                          const float* g_codebook, const float* g_commitment,           /* DEVICE scalars, NULL = 0 */
                          const float* g_codebook_norm, const float* g_commitment_norm,
                          int want_norm_mse,
                          void* gx_out /* x dtype */, float* gW_accum,
                          int64_t g_hw /* 0: g_zste and gx token-major; h*w > 0: both NCHW [N/hw, D, hw] (x stays token-major) */,
                          void* stream);
/* The same backward with each token's codebook-gradient row STORED to gW_rows fp32 [N, D] instead of atomically added
 * into gW (gx bit-identical to vqb_quantize_backward).  vqb_segment_sum_rows over those rows gives a deterministic gW. */
int vqb_quantize_backward_rows(const void* g_zste, int g_dtype, const void* x, int x_dtype, int normalize_x,
                               const float* W, int64_t K, const int64_t* quant, int64_t N, int D,
                               const float* g_codebook, const float* g_commitment,
                               const float* g_codebook_norm, const float* g_commitment_norm,
                               int want_norm_mse, void* gx_out, float* gW_rows, int64_t g_hw, void* stream);
/* The rotation trick (Fifty et al., arXiv:2410.06424): vqb_quantize_backward / _rows with each token's g_zste first
 * replaced by  g' = lambda R^T g_zste,  R the rotation taking y/|y| to e/|e| (y the token as quantized, e = W[q]),
 * lambda = |e|/|y|;  a token with |y| or |e| below 1e-12 keeps g_zste.  gW is bit-identical to the unrotated entry
 * points; only gx differs (DESIGN.md §4.9). */
int vqb_quantize_backward_rotated(const void* g_zste, int g_dtype, const void* x, int x_dtype, int normalize_x,
                                  const float* W, int64_t K, const int64_t* quant, int64_t N, int D,
                                  const float* g_codebook, const float* g_commitment,
                                  const float* g_codebook_norm, const float* g_commitment_norm,
                                  int want_norm_mse, void* gx_out, float* gW_accum, int64_t g_hw, void* stream);
int vqb_quantize_backward_rotated_rows(const void* g_zste, int g_dtype, const void* x, int x_dtype, int normalize_x,
                                       const float* W, int64_t K, const int64_t* quant, int64_t N, int D,
                                       const float* g_codebook, const float* g_commitment,
                                       const float* g_codebook_norm, const float* g_commitment_norm,
                                       int want_norm_mse, void* gx_out, float* gW_rows, int64_t g_hw, void* stream);

/* ---- residual quantization (RQ-VAE: L codebooks, level l quantizes what levels 1..l-1 left over) ------------ *
 *   r_0 = x;  e_l = W_l[q_l];  zhat_1 = e_1, zhat_l = zhat_{l-1} + e_l;  r_l = r_{l-1} - e_l   (fp32 add / subtract,
 *   never fused into an FMA);  z = x + (zhat_L - x) (straight-through to x over the whole depth).
 * Level l's four MSE terms compare e_l with r_{l-1} exactly as vqb_gather_ste_loss compares W[q] with x, so L = 1
 * gives bit for bit the results of vqb_gather_ste_loss / vqb_quantize_backward.  The per-level pointers travel BY
 * VALUE (the struct is copied into the kernel parameters): no device pointer table, no host-to-device copy. */
#define VQB_MAX_LEVELS 16
typedef struct {
  int L;                                   /* 1 .. VQB_MAX_LEVELS */
  const float* W[VQB_MAX_LEVELS];          /* level codebooks, fp32 [K, D] each (the same K and D at every level) */
  float* gW[VQB_MAX_LEVELS];               /* backward: gW_l accumulators (pre-zeroed; NULL = not wanted), or the
                                              level's fp32 [N, D] rows of the _rows variant */
  const float* g[VQB_MAX_LEVELS][4];       /* backward: DEVICE scalars g_codebook, g_commitment, g_codebook_norm,
                                              g_commitment_norm of level l (NULL = 0) */
} vqb_residual_levels;
/* One level: reads r_{l-1} (r_dtype: x's dtype at level 0, VQB_F32 after), the level's keys or indices and W_l[q];
 * writes quant_out[n*L + level] (optional; the [N, L] code layout), and
 *   level < L-1 (r_out != NULL): zhat (fp32 [N, D], written at level 0, updated in place after) and r_out = r_l;
 *   level = L-1 (r_out == NULL): z_out = x + (zhat_L - x) (optional; token-major, or NCHW with z_hw > 0 as in
 *                                vqb_gather_ste_loss); zhat is read, not written.
 * mse4_out: this level's four terms (deterministic two-stage sum; partials / ticket as for vqb_gather_ste_loss). */
int vqb_residual_step(const void* r_in, int r_dtype, const void* x, int x_dtype, int64_t N, int D,
                      const float* W, int64_t K, const int64_t* quant, const unsigned long long* keys,
                      int64_t key_index_offset, int64_t* quant_out, int L, int level, float* zhat, float* r_out,
                      float* z_out, int64_t z_hw, int want_norm_mse, float* mse4_out, float* partials,
                      unsigned int* ticket, void* stream);
/* The whole depth's backward in ONE launch.  Per token r_{l-1} is recomputed with the forward's operations (bit
 * identical), then  gx = g_z + sum_l [commitment-role terms of level l]  (x dtype) and  gW_l[q_l] += [codebook-role
 * row of level l]  (fp32 vector atomics), each term as in vqb_quantize_backward with (x, W) = (r_{l-1}, W_l).
 * quant: int64 [N, L].  g_hw as in vqb_quantize_backward. */
int vqb_residual_backward(const void* g_z, int g_dtype, const void* x, int x_dtype, const vqb_residual_levels* levels,
                          int64_t K, const int64_t* quant, int64_t N, int D, int want_norm_mse, void* gx_out,
                          int64_t g_hw, void* stream);
/* The same with level l's codebook-gradient rows STORED to levels->gW[l] (fp32 [N, D] each; gx identical): their
 * vqb_segment_sum_rows, level by level, is a deterministic gW_l. */
int vqb_residual_backward_rows(const void* g_z, int g_dtype, const void* x, int x_dtype,
                               const vqb_residual_levels* levels, int64_t K, const int64_t* quant, int64_t N, int D,
                               int want_norm_mse, void* gx_out, int64_t g_hw, void* stream);
/* vqb_residual_backward / _rows with the rotation trick of vqb_quantize_backward_rotated over the whole depth, the
 * stack's one straight-through estimator (DESIGN.md §4.7, §4.9).  Per token, in fp32 (bf16 tokens up-cast):
 *   zhat_L = W_0[q_0] + W_1[q_1] + ... + W_{L-1}[q_{L-1}]   (round-to-nearest adds in level order: the forward's zhat)
 *   g' = rotate(x, zhat_L, g_z)   (|x| or |zhat_L| below 1e-12: g' = g_z)
 *   gx = g' + sum_l [commitment-role terms of level l]   (unchanged, level order)
 * gW_l is bit-identical to the unrotated entry points; only gx differs. */
int vqb_residual_backward_rotated(const void* g_z, int g_dtype, const void* x, int x_dtype,
                                  const vqb_residual_levels* levels, int64_t K, const int64_t* quant, int64_t N, int D,
                                  int want_norm_mse, void* gx_out, int64_t g_hw, void* stream);
int vqb_residual_backward_rotated_rows(const void* g_z, int g_dtype, const void* x, int x_dtype,
                                       const vqb_residual_levels* levels, int64_t K, const int64_t* quant, int64_t N,
                                       int D, int want_norm_mse, void* gx_out, int64_t g_hw, void* stream);
/* Quantizer dropout (DESIGN.md §4.10): the entry points above with a per-token depth.  Token n is coded by its first
 * d_n = depth[n / depth_hw] levels (int32; depth_hw = h*w for one depth per image, 1 for one per token; values outside
 * [1, L] are clamped to it, there is no host check).  Assignment is unchanged: q_l and r_l exist at every level.
 *   step:      zhat adds e_l, and the level's mse4 sums take the token, only when level < d_n (mse4 keeps the 1/(N*D)
 *              denominator); z = x + (zhat_{d_n} - x).
 *   backward:  levels l >= d_n add nothing to gx and nothing to gW_l (the _rows variants store zero rows for them);
 *              the _rotated variants rotate towards zhat_{d_n}.
 * With every depth = L the results are bit for bit those of the entry points without _depth. */
int vqb_residual_step_depth(const void* r_in, int r_dtype, const void* x, int x_dtype, int64_t N, int D,
                            const float* W, int64_t K, const int64_t* quant, const unsigned long long* keys,
                            int64_t key_index_offset, int64_t* quant_out, int L, int level, float* zhat, float* r_out,
                            float* z_out, int64_t z_hw, int want_norm_mse, float* mse4_out, float* partials,
                            unsigned int* ticket, const int32_t* depth, int64_t depth_hw, void* stream);
int vqb_residual_backward_depth(const void* g_z, int g_dtype, const void* x, int x_dtype,
                                const vqb_residual_levels* levels, int64_t K, const int64_t* quant, int64_t N, int D,
                                int want_norm_mse, void* gx_out, int64_t g_hw, const int32_t* depth, int64_t depth_hw,
                                void* stream);
int vqb_residual_backward_depth_rows(const void* g_z, int g_dtype, const void* x, int x_dtype,
                                     const vqb_residual_levels* levels, int64_t K, const int64_t* quant, int64_t N,
                                     int D, int want_norm_mse, void* gx_out, int64_t g_hw, const int32_t* depth,
                                     int64_t depth_hw, void* stream);
int vqb_residual_backward_depth_rotated(const void* g_z, int g_dtype, const void* x, int x_dtype,
                                        const vqb_residual_levels* levels, int64_t K, const int64_t* quant, int64_t N,
                                        int D, int want_norm_mse, void* gx_out, int64_t g_hw, const int32_t* depth,
                                        int64_t depth_hw, void* stream);
int vqb_residual_backward_depth_rotated_rows(const void* g_z, int g_dtype, const void* x, int x_dtype,
                                             const vqb_residual_levels* levels, int64_t K, const int64_t* quant,
                                             int64_t N, int D, int want_norm_mse, void* gx_out, int64_t g_hw,
                                             const int32_t* depth, int64_t depth_hw, void* stream);

/* ---- grouped (product) quantization: G codebooks, group g quantizes channels [g*Dg, (g+1)*Dg) of every token ---- *
 * Group g behaves exactly like its own vqb_gather_ste_loss / vqb_quantize_backward on the contiguous [N, Dg] slice
 * x_g (same row geometry, same grid, its own partials and ticket), so every per-group result is bit for bit that of
 * a standalone quantizer on x_g.  The per-group pointers travel BY VALUE in a vqb_residual_levels with L = G
 * (W[g], gW[g], g[g][4]).
 * Split: src [batch, G*Dg, hw] (NCHW latents; hw = 1 is token-major [N, D]) -> dst [G, batch*hw, Dg], the group-major
 * copy whose group g is the contiguous x_g.  dtype VQB_F32 or VQB_BF16 (copied as is). */
int vqb_split_groups(const void* src, int dtype, int64_t batch, int G, int Dg, int64_t hw, void* dst, void* stream);
/* Every group's gather + straight-through + MSE terms in ONE launch (grid y = group).  xs: the split [G, N, Dg];
 * quant / keys: group-major [G, N] (exactly one); writes quant_out[n*G + g] (optional; the [N, G] code layout),
 * z = x_g + (W_g[q_g] - x_g) into channels [g*Dg, (g+1)*Dg) of z_out (token-major [N, G*Dg], or NCHW with z_hw > 0
 * as in vqb_gather_ste_loss) and group g's four terms to mse4_out[4*g .. 4*g+4).  partials: G x
 * vqb_loss_partials_count() floats, tickets: G zero-initialised (self-resetting) uint32. */
int vqb_group_gather_ste_loss(const void* xs, int x_dtype, int64_t N, int Dg, const vqb_residual_levels* groups,
                              int64_t K, const int64_t* quant, const unsigned long long* keys, int64_t* quant_out,
                              float* z_out, int64_t z_hw, int want_norm_mse, float* mse4_out, float* partials,
                              unsigned int* tickets, void* stream);
/* Every group's backward in ONE launch: the closed form of vqb_quantize_backward per group with (x, W, quant) =
 * (x_g, W_g, quant[:, g]).  gx channels [g*Dg, (g+1)*Dg) = g_z's + group g's commitment-role terms (x dtype; token-major
 * [N, G*Dg], or NCHW for both g_z and gx with g_hw > 0); gW_g[q_g] += the codebook-role row (fp32 vector atomics).
 * xs: the split [G, N, Dg] of the forward; quant: int64 [N, G]. */
int vqb_group_backward(const void* g_z, int g_dtype, const void* xs, int x_dtype, const vqb_residual_levels* groups,
                       int64_t K, const int64_t* quant, int64_t N, int Dg, int want_norm_mse, void* gx_out, int64_t g_hw,
                       void* stream);
/* The same with group g's codebook-gradient rows STORED to groups->gW[g] (fp32 [N, Dg] each; gx identical): their
 * vqb_segment_sum_rows, group by group, is a deterministic gW_g. */
int vqb_group_backward_rows(const void* g_z, int g_dtype, const void* xs, int x_dtype, const vqb_residual_levels* groups,
                            int64_t K, const int64_t* quant, int64_t N, int Dg, int want_norm_mse, void* gx_out,
                            int64_t g_hw, void* stream);
/* vqb_group_backward / _rows with the rotation trick of vqb_quantize_backward_rotated, per group on (x_g, W_g[q_g]). */
int vqb_group_backward_rotated(const void* g_z, int g_dtype, const void* xs, int x_dtype,
                               const vqb_residual_levels* groups, int64_t K, const int64_t* quant, int64_t N, int Dg,
                               int want_norm_mse, void* gx_out, int64_t g_hw, void* stream);
int vqb_group_backward_rotated_rows(const void* g_z, int g_dtype, const void* xs, int x_dtype,
                                    const vqb_residual_levels* groups, int64_t K, const int64_t* quant, int64_t N,
                                    int Dg, int want_norm_mse, void* gx_out, int64_t g_hw, void* stream);

/* ---- row l2-normalisation (NormalizeCallback.before_encode on x) ------------------------ *
 * vq/algorithms/vq/callbacks/normalize.py:24  — forward y = x / max(||x||, 1e-12); backward
 * gx = (gy - (gy.y) y) / max(||x||, 1e-12). */
int vqb_l2norm_forward(const void* x, int x_dtype, int64_t rows, int D, void* y, int y_dtype, void* stream);
int vqb_l2norm_backward(const void* gy, int g_dtype, const void* x, int x_dtype, int64_t rows, int D,
                        void* gx, int gx_dtype, void* stream);

/* ---- usage / EMA statistics -------------------------------------------------------------- *
 * Replaces QuantStatistics.bin_count                vq/algorithms/vq/utils.py:40-43
 *          VQKDCallback._kmeans scatter_add_        vq/algorithms/vqkd/quantizers/callbacks.py:60-62
 * stats = fp32 [K*D sums | K counts] in ONE buffer (one all-reduce), pre-zeroed by the caller.
 * normalize_x: accumulate F.normalize(x) rows (callbacks.py:124). */
int vqb_scatter_stats(const void* x, int x_dtype, int64_t N, int D, int normalize_x,
                      const int64_t* quant,          /* [N] indices, or NULL when `keys` is given */
                      const unsigned long long* keys, int64_t key_index_offset, /* packed keys of vqb_assign */
                      float* stats, int64_t K, void* stream);
/* int64 histogram accumulate — CodebookMixin.forward, vq/tasks/image_tokenization/runners/metrics.py:37-45 */
int vqb_bincount_accumulate(const int64_t* quant, int64_t n, int64_t* counts, int64_t K,
                            int add_total, /* 1: counts[K] += n (numel slot of the fused [K | 1] all-reduce buffer) */
                            void* stream);

/* ---- deterministic per-code reductions (torch.use_deterministic_algorithms) --------------- *
 * The atomic scatters above (vqb_scatter_stats, the gW of vqb_quantize_backward) are order-dependent in the last
 * bits.  These entry points give the same sums with a fixed association:
 *   for code k with tokens t_1 < ... < t_m (tokens whose code is outside [0, K) are skipped; packed keys resolve
 *   as in vqb_scatter_stats), cut the list into consecutive chunks of VQB_SEGMENT_CHUNK tokens; sum each chunk
 *   serially in ascending token order from +0.0f, add the chunk sums serially in chunk order from +0.0f, and add
 *   that total ONCE to the output element (a plain read-modify-write: a zero-filled output keeps the accumulate
 *   semantics of vqb_scatter_stats).  Codes without tokens leave their output untouched.
 * VQB_SEGMENT_CHUNK = 256: the longest serial chain is max(C, m / C) additions, so a collapsed codebook (all N tokens
 * on one code) costs ~2 sqrt(N) dependent additions at N = 65 536 instead of N; a smaller C mostly adds chunk
 * partials (scratch traffic) for codes of a few tokens, the common case. */
#define VQB_SEGMENT_CHUNK 256
int64_t vqb_segment_chunk(void);
/* Stable sort of the tokens by code (LSD radix, 8-bit digits: ceil(bits(K) / 8) passes of 3 launches + 2 launches; no
 * host synchronisation, no spinning).  order: int32 [N] token indices grouped by code, ascending within a code, the
 * tokens with an out-of-range code last; offsets: int32 [K+1], code k owns order[offsets[k] .. offsets[k+1]).
 * N < 2^31.  `scratch` needs vqb_code_sort_scratch_bytes(N, K) bytes. */
size_t vqb_code_sort_scratch_bytes(int64_t N, int64_t K);
int vqb_code_sort(const int64_t* quant,                /* [N] indices, or NULL when `keys` is given */
                  const unsigned long long* keys, int64_t key_index_offset, int64_t N, int64_t K,
                  int32_t* order, int32_t* offsets, void* scratch, size_t scratch_bytes, void* stream);
/* out_sums fp32 [K, D] (+)= the contract sums of rows (fp32 or bf16 [N, D]; normalize_rows: F.normalize of each row,
 * its norm computed with the lane geometry of vqb_scatter_stats, so each row's value depends on that row alone);
 * out_counts (optional) fp32 [K] (+)= offsets[k+1] - offsets[k].  (order, offsets) from vqb_code_sort.  No float
 * atomics.  `scratch` needs vqb_segment_sum_scratch_bytes(N, K, D) bytes (chunk partials, N / C + K + 1 rows). */
size_t vqb_segment_sum_scratch_bytes(int64_t N, int64_t K, int D);
int vqb_segment_sum_rows(const void* rows, int rows_dtype, int64_t N, int D, int normalize_rows,
                         const int32_t* order, const int32_t* offsets, int64_t K,
                         float* out_sums, float* out_counts, void* scratch, size_t scratch_bytes, void* stream);

/* VQKDCallback._kmeans tail + after_encode:  callbacks.py:66-71,126-128,73-75
 *   C = cnt>0 ? S/max(cnt,1) : E ;  W <- normalize( E*decay + normalize(C)*(1-decay) )   (in place) */
int vqb_kmeans_ema_update(const float* stats, float* W, int64_t K, int D, float decay, float one_minus_decay,
                          void* stream);

/* rows_out[k] = x[idx(keys[k])]  (fp32)  — NearestAnchor `x[indices]`, cvqvae/anchors.py:84.
 * Keys whose index falls outside [index_offset, index_offset+N) produce zero rows (their owner
 * rank supplies them; the caller sums over ranks). */
int vqb_gather_rows_by_key(const void* x, int x_dtype, int64_t N, int D,
                           const unsigned long long* keys, int64_t K, int64_t index_offset,
                           float* rows_out, void* stream);

/* CVQVAECallback.after_encode tail:  vq/algorithms/cvqvae/quantizer_callback.py:93-103
 *   p <- p*decay + (cnt/total)*(1-decay)
 *   dec = 1 - exp(-p*K*10/(1-decay) - eps) ;  W <- W*dec + anchors*anchor_scale*(1-dec)   (in place)
 * counts = int64 [K] (all-reduced bincount), total = DEVICE pointer to the all-reduced int64 token count
 * (QuantStatistics.frequency, vq/algorithms/vq/utils.py:48-52: int64 / int64 -> fp32). */
int vqb_cvq_update(float* W, const float* anchors, float anchor_scale, float* prob, const int64_t* counts,
                   const int64_t* total, int64_t K, int D, float decay, float one_minus_decay, float eps,
                   void* stream);

/* ---- finite scalar quantisation ---------------------------------------------------------- *
 * FiniteScalarQuantizer._encode / _decode           vq/algorithms/fsq/quantizers.py:108-137
 * Per-channel constants are computed by the host exactly as torch computes them and passed by
 * value: max_[d], odd[d], shift[d] = atanh(odd/max_), half[d] = L//2, cumprod[d], levels[d]. D <= 16. */
typedef struct {
  int D;
  float max_[16];
  float odd[16];
  float shift[16];
  float half[16];
  int cumprod[16];
  int levels[16];
} vqb_fsq_params;
int vqb_fsq_forward(const void* x, int x_dtype, int64_t N, const vqb_fsq_params* p_host,
                    void* zq_out, int out_dtype, int32_t* index_out, void* stream);
int vqb_fsq_backward(const void* gz, int g_dtype, const void* x, int x_dtype, int64_t N,
                     const vqb_fsq_params* p_host, void* gx, int gx_dtype, void* stream);
int vqb_fsq_decode(const int32_t* index, int64_t N, const vqb_fsq_params* p_host, float* z_out, void* stream);

/* ---- token ids -> NCHW latents ---------------------------------------------------------------- *
 * Decode-only path of the tokenizer (decode_from_quant, vq/tasks/image_reconstruction/models.py:97-108):
 * z[b][d][s] = W[id[b*hw + s]][d], written straight into the caller's NCHW layout ('b h w c -> b c h w' fused).
 * ids: [batch * hw], id_bytes 2 (uint16), 4 (int32) or 8 (int64).  out_dtype VQB_F32 or VQB_BF16 (round to nearest even).
 * An id outside [0, K) gives a NaN row (every channel); if bad_count is given (a device int, zeroed by the caller),
 * it is incremented by the number of such tokens.  No fault, no clamping.  (vqb_embedding_gather and vqb_fsq_decode
 * keep their clamp / wrap behaviour.) */
int vqb_decode_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const float* W, int64_t K, int D,
                      void* z_out, int out_dtype, int* bad_count, void* stream);
/* The same for FSQ's implicit codebook (fsq/quantizers.py:59-63,136-137): digits of the mixed-radix id, value
 * digit / half - 1 evaluated exactly as vqb_fsq_decode does; valid ids are [0, prod(levels)). */
int vqb_fsq_decode_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const vqb_fsq_params* p_host,
                          void* z_out, int out_dtype, int* bad_count, void* stream);
/* The same for residual codes: ids [batch * hw, L] (a token's L ids contiguous), z[b][d][s] = sum_l W_l[id_l][d]
 * with the fp32 adds of zhat in vqb_residual_step (level order).  An id outside [0, K) at ANY level gives a NaN row
 * and counts the token once.  Only levels->L and levels->W are read. */
int vqb_decode_residual_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw,
                               const vqb_residual_levels* levels, int64_t K, int D, void* z_out, int out_dtype,
                               int* bad_count, void* stream);
/* The same for grouped codes: ids [batch * hw, G] (a token's G ids contiguous), z[b][g*Dg + d][s] = W_g[id_g][d].
 * An id outside [0, K) in ANY group gives a NaN row (every channel) and counts the token once.  G = groups->L; only
 * groups->L and groups->W are read. */
int vqb_decode_group_tokens(const void* ids, int id_bytes, int64_t batch, int64_t hw, const vqb_residual_levels* groups,
                            int64_t K, int Dg, void* z_out, int out_dtype, int* bad_count, void* stream);

/* ---- compatibility mode: the materialised distance matrix ---------------------------------- *
 * out[n, k] = torch.cdist(x, W)[n, k]  (cosine = 0)         vq/algorithms/vq/distances.py:28-32
 *           = 1 - <x_n/|x_n|, W_k/|W_k|>  (cosine = 1)       vq/algorithms/vq/distances.py:35-46
 * i.e. `memo['encode']['distance']` of VectorQuantizer._encode (vq/algorithms/vq/quantizers.py:97-98), which the
 * hot path never builds.  Produced on demand for its consumers (EntropyLoss, MultinomialAnchor, user callbacks,
 * the `materialize_distance` debug switch); fp32 CUDA-core kernel, exact fp32 products. */
int vqb_distance_matrix(const void* x, int x_dtype, int64_t N, int D, const float* W, int64_t K, int cosine,
                        float* out /* fp32 [N, K] */, void* stream);

/* ---- multi-GPU exchange over NVLink peer memory, fused with the codebook update ------------ *
 * One process per GPU (the reference's DDP model).  Replaces the statistics collectives of the path
 *   QuantStatistics all_reduce x2                       vq/algorithms/vq/utils.py:35
 *   VQ-KD centroid all_reduce                           vq/algorithms/vqkd/quantizers/callbacks.py:63-64
 *   CVQ-VAE anchors all_reduce / all_gather             vq/algorithms/cvqvae/anchors.py:50-57,64-67
 * Every rank allocates one REGION of the same size with vqb_comm_alloc (cudaMalloc + CUDA IPC handle), the host
 * layer exchanges the 64-byte handles (any out-of-band channel: torch.distributed here), maps the peers with
 * vqb_comm_open and publishes the table of mapped base pointers with vqb_comm_bind.  The first
 * VQB_COMM_HEADER_BYTES of a region are the library's control block (epoch flags + peer table); everything
 * behind it is laid out by the caller, IDENTICALLY on every rank, and addressed by byte offsets.
 * The exchange kernels are two-shot: rank r reduces the slice [r*n/w, (r+1)*n/w) of every peer's buffer in fixed
 * rank order (all replicas get bit-identical results), applies the update, and stores the result into every
 * peer's region.  Collective semantics: all ranks must issue the same sequence of vqb_comm_* launches.
 * Waits are bounded (~2 s, then the kernel traps): a missing peer is an error code, not a hang. */
#define VQB_COMM_HEADER_BYTES 512
#define VQB_COMM_MAX_WORLD 16
#define VQB_IPC_HANDLE_BYTES 64
int vqb_comm_alloc(size_t bytes, void** region, unsigned char* handle_out /* [VQB_IPC_HANDLE_BYTES] */);
int vqb_comm_open(const unsigned char* handle, void** peer_region);
int vqb_comm_close(void* peer_region);
int vqb_comm_free(void* region);
int vqb_comm_bind(void* region, const void* const* peer_regions_host /* [world], [rank] == region */, int rank, int world);
/* stats_off: fp32 [K*D sums | K counts] (per-rank partials of vqb_scatter_stats); w_off: fp32 [K, D] codebook.
 * = all_reduce(SUM) + vqb_kmeans_ema_update in one launch; afterwards every rank's codebook holds the same rows. */
/* ll_in_off / ll_out_off: (size_t)-1 selects the barrier protocol (six NVLink hops).  Otherwise the LOW-LATENCY
 * protocol: every fp32 word is its own flag (its mantissa LSB carries the parity of the exchange counter), so the
 * exchange needs no barrier or fence (two one-way hops) at 1x wire bytes; transmitted values lose their LSB (<= 1 ulp)
 * and every replica stores the same truncated rows.  ll_in_off: uint32 [world][ceil(K/world)][D+1] staging for the
 * partial sums pushed to this rank; ll_out_off: uint32 [K][D] staging for the updated rows pushed to this rank.  Both
 * zero-initialised once, never reset. */
int vqb_comm_kmeans_ema_update(void* region, int rank, int world, size_t stats_off, size_t w_off, size_t ll_in_off,
                               size_t ll_out_off, int64_t K, int D, float decay, float one_minus_decay, void* stream);
/* counts_off: int64 [K counts | numel] per-rank partials; anchors_off: fp32 [K, D] per-rank nearest-token rows;
 * keys_off: (size_t)-1 for sync=False anchors (mean over ranks), else uint64 [K] per-rank packed
 * (distance, global token index) keys: the minimum key wins and its row is taken from the rank that holds it;
 * w_off / prob_off: the codebook and the `_probability` buffer.  = the two all-reduces + vqb_cvq_update. */
int vqb_comm_cvq_update(void* region, int rank, int world, size_t counts_off, size_t anchors_off, size_t keys_off,
                        size_t w_off, size_t prob_off, int64_t K, int D, float decay, float one_minus_decay,
                        float eps, void* stream);
/* packed (score, index) min-loc all-reduce over uint64 [n] (codebook shards; no sign flip needed) */
int vqb_comm_allreduce_min_keys(void* region, int rank, int world, size_t keys_off, int64_t n, void* stream);
/* fp32 SUM all-reduce over [n] (buffer padded to a multiple of 4 floats) */
int vqb_comm_allreduce_sum_f32(void* region, int rank, int world, size_t off, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VQB200_H_ */
