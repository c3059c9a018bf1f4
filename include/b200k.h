/* b200k.h — the C ABI of libb200k.so: B200-native (sm_100a) replacements for the hot paths of
 * DefTruth/CUDA-Learn-Notes.  Plain C: raw device pointers, sizes, a CUDA stream handle.  No torch types.
 *
 * Every entry point
 *   - takes DEVICE pointers owned by the caller (never allocates, keeps no state between calls),
 *   - enqueues its kernels on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream, which is
 *     what the reference launches on) and returns without synchronising,
 *   - returns B200K_OK or a negative B200K_E* code; b200k_last_error() gives the message for the calling thread.
 *
 * Each declaration cites the reference interface it replaces (paths relative to the reference repo root).
 * The Python side (cuda-learn-notes_b200/b200k/_loader.py) binds exactly these symbols with ctypes; the
 * reference-side stubs a maintainer would add are shown in INTEGRATION.md.
 */
#ifndef B200K_H_
#define B200K_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200K_OK 0
#define B200K_EDTYPE (-1)   /* unsupported dtype / pack enum                         */
#define B200K_ESHAPE (-2)   /* shape not supported (see each function)               */
#define B200K_EALIGN (-3)   /* pointer or row pitch not 16-byte aligned              */
#define B200K_EHEADDIM (-4) /* head dim not supported ("headdim not support!")       */
#define B200K_ECUDA (-5)    /* a CUDA runtime / driver call failed                   */
#define B200K_EARCH (-6)    /* current device is not compute capability 10.x (B200)  */
#define B200K_EARG (-7)     /* bad enum / null pointer                               */

#define B200K_ABI_VERSION 1

int b200k_abi_version(void);
const char* b200k_last_error(void);
/* Fills sm count and compute capability of the current device; B200K_EARCH if it is not sm_100. */
int b200k_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------------ HGEMM
 * C[M,N] = A[M,K] * B, fp16 in / fp16 out, fp32 accumulation in tensor memory (tcgen05.mma kind::f16).
 *   b_is_nk = 0 ("NN"): B is [K,N] row-major           — replaces every NN entry point of
 *       kernels/hgemm/pybind/hgemm.cc:L58-107, flagship kernels/hgemm/mma/basic/hgemm_mma_stage.cu:L2380-2454
 *       (hgemm_mma_m16n8k16_mma2x4_warp4x4x2_stages_dsmem)
 *   b_is_nk = 1 ("TN"): B storage is B^T = [N,K] row-major — replaces
 *       kernels/hgemm/mma/basic/hgemm_mma_stage_tn.cu:L517 (…_dsmem_tn),
 *       kernels/hgemm/mma/swizzle/hgemm_mma_stage_tn_swizzle_x4.cu:L860, kernels/hgemm/cutlass/hgemm_mma_stage_tn_cute.cu:L522,
 *       kernels/hgemm/cublas/hgemm_cublas.cu:L63-84 (hgemm_cublas_tensor_op_tn)
 * All matrices contiguous row-major; M,N,K >= 1; K % 8 == 0 and N % 8 == 0 (16-byte row pitch for TMA).
 * Ragged M/N/K (not multiples of the tile) are handled by TMA zero-fill / store clipping.
 * variant (low 8 bits): 0 = auto; 1 = 1-CTA 128x256 tiles; 2 = 2-CTA (cta_group::2) 256x256 tiles, two accumulator buffers,
 *   stream-K remainder round; 3 = 2-CTA 256x128 tiles; 4 = 2-CTA 512x256 tiles (auto picks it from ~3 rounds of them).
 *   Higher bits are measurement switches (GROUP_M, L2 hints, bit 20 stream-K off, bit 21 keep 256x256), see hgemm_tcgen05.cu.
 * Workspace: the stream-K round keeps one device workspace per (device, stream), cudaMalloc'ed on first use.
 */
#define B200K_HGEMM_AUTO 0
#define B200K_HGEMM_1CTA_128x256 1
#define B200K_HGEMM_2CTA_256x256 2
#define B200K_HGEMM_2CTA_256x128 3
#define B200K_HGEMM_2CTA_512x256 4 /* 256 x 256 per CTA: both accumulators of a tile fill TMEM, 25 % less L2 -> SM traffic per flop */
int b200k_hgemm_f16(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int b_is_nk,
                    int variant, void* stream);

/* Same kernel for other operand types (SURVEY.md section 8f-4): dtype B200K_F16 (identical to b200k_hgemm_f16),
 * B200K_BF16 (bf16 in / bf16 out, fp32 accumulation), or B200K_F32 = TF32 tensor-core product of fp32 matrices with
 * fp32 output (tcgen05.mma kind::tf32: the operands' low 13 mantissa bits are ignored by the tensor core, fp32
 * accumulation) - the B200 counterpart of kernels/sgemm/sgemm_wmma_tf32_stage.cu:L25-420 (sgemm_wmma_m16n16k8_*).
 * K and N must be multiples of 8 (16-bit types) or 4 (fp32).  An fp32 [K,N] B is read as an MN-major operand through the
 * "128B swizzle with 32-byte atoms" shared-memory layout (TMA SWIZZLE_128B_ATOM_32B, UMMA layout type 1). */
int b200k_gemm(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int b_is_nk, int dtype, int variant,
               void* stream);
/* All four storage cases (SURVEY.md 8(f)-4 "TN/NT"): a_is_km != 0 means A is stored transposed, [K,M] row-major (the BLAS
 * "NT" / "TT" cases; f16 and bf16; M % 8 == 0); b_is_nk as above.  Operands are consumed in place (MN-major UMMA
 * descriptors), no transpose pass.  b200k_gemm(...) == b200k_gemm_ex(..., a_is_km = 0, ...). */
int b200k_gemm_ex(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int a_is_km, int b_is_nk, int dtype,
                  int variant, void* stream);

/* ------------------------------------------------------------------------------------------------ attention
 * O = softmax(Q K^T * scale) V, non-causal, Q/K/V/O [B,H,N,D] fp16 contiguous (V optionally [B,H,D,N]).
 *
 * b200k_fa2_fwd_f16 — FlashAttention-2 forward, D in {32, 64, 96, 128}; N % 128 == 0 is NOT required (ragged N
 *   is masked), N >= 1.  Replaces the 25(+3) entry points flash_attn_mma_stages_* of
 *   kernels/flash-attn/pybind/flash_attn.cc:L182-216, flagship
 *   kernels/flash-attn/mma/basic/flash_attn_mma_share_qkv.cu:L833-886 (…_split_q_shared_qkv).
 *   v_is_dn = 1: V is passed transposed as [B,H,D,N] (the *_swizzle_qkv entry points, flash_attn_mma.py:L378).
 *
 * b200k_ffpa_fwd_f16 — large-headdim forward (FFPA L1), D in {160 .. 1024 step 32} (and the small D above); the
 *   D % 64 == 32 rungs are the reference's ENABLE_FFPA_ALL_HEADDIM set (launch_templates.cuh:L483-552).
 *   Replaces ffpa_mma_acc_f16_L1 / ffpa_mma_acc_f32_L1, ffpa-attn-mma/csrc/pybind/ffpa_attn_api.cc:L8-17,
 *   launcher ffpa-attn-mma/csrc/cuffpa/launch_templates.cuh:L261-449.
 * scale <= 0 means 1/sqrt(D) (what both references hard-code).
 * variant: 0 = the shipped configuration.  Other values select experiment / fallback builds of the same math (piece
 *   counts, polynomial exp2 fraction, TMEM layout, 1-CTA vs CTA-pair FFPA, cycle trace); the bits are listed next to
 *   the dispatchers in csrc/fa2_fwd_tcgen05.cu and csrc/ffpa_fwd_tcgen05.cu.  Every build is parity-tested.
 *   FFPA kernel selection: D = 512 runs the O^T kernel (csrc/ffpa3_fwd_tcgen05.cu: one pass over Q K^T per KV tile, like
 *   the reference's ffpa_attn_templates_L1.cuh:L219-368); bit 0x400 keeps the D-sliced CTA-pair kernel there, bit 0x200
 *   selects the O^T kernel at D = 256; every other D runs the D-sliced kernels (S recomputed per 256-column slice of O).
 */
int b200k_fa2_fwd_f16(const void* Q, const void* K, const void* V, void* O, int64_t B, int64_t H, int64_t N,
                      int64_t D, float scale, int v_is_dn, int variant, void* stream);
int b200k_ffpa_fwd_f16(const void* Q, const void* K, const void* V, void* O, int64_t B, int64_t H, int64_t N,
                       int64_t D, float scale, int variant, void* stream);
/* b200k_fa2_fwd — the same FA-2 kernel with the caller-facing options the reference lacks (SURVEY.md 8(f)-4):
 *   dtype      B200K_F16 or B200K_BF16 (Q, K, V, O and the P operand; statistics and accumulators stay fp32)
 *   causal     != 0: query row r attends keys <= r; KV tiles above the diagonal are skipped, not masked
 *   seqlens_k  NULL, or int32 device array [B]: keys >= seqlens_k[b] are masked for batch b (key-padding mask of the
 *              padded [B,H,N,D] layout; 1 <= seqlens_k[b] <= N; every query row is still computed).  K and V past
 *              seqlens_k[b] are never used and may be uninitialised.
 * b200k_fa2_fwd_f16(...) == b200k_fa2_fwd(..., B200K_F16, 0, NULL, ...). */
int b200k_fa2_fwd(const void* Q, const void* K, const void* V, void* O, int64_t B, int64_t H, int64_t N, int64_t D,
                  float scale, int v_is_dn, int dtype, int causal, const int* seqlens_k, int variant, void* stream);

/* ------------------------------------------------------------------------------------------------ support kernels
 * HBM-roofline kernels (128-bit vectorised, warp-shuffle reductions, no tensor cores).  dtype enums: */
#define B200K_F32 0
#define B200K_F16 1
#define B200K_BF16 2
#define B200K_I8 3
#define B200K_FP8_E4M3 4
#define B200K_FP8_E5M2 5
#define B200K_I32 6

/* c = a + b, n elements.  kernels/elementwise/elementwise.cu:L24-168 (elementwise_add_{f32,f32x4,f16,f16x2,f16x8,f16x8_pack}). */
int b200k_elementwise_add(const void* a, const void* b, void* c, int64_t n, int dtype, void* stream);

/* out[0] = sum(x[0..n)).  `out` is a 1-element device buffer (f32, or i32 when dtype == B200K_I8) that this call
 * overwrites.  acc_f16 = 1 reproduces the reference's half-precision per-thread partial sums.
 * kernels/reduce/block_all_reduce.cu:L42-686, bindings L734-790 (block_all_reduce_sum_*).
 * Deterministic (fixed two-pass order) where the reference uses atomicAdd. `workspace`: >= b200k_reduce_workspace_bytes(). */
size_t b200k_reduce_workspace_bytes(void);
int b200k_block_all_reduce_sum(const void* x, void* out, int64_t n, int dtype, int acc_f16, void* workspace,
                               void* stream);

/* Row softmax over the last dim of x[S,H] -> y[S,H].  kernels/softmax/softmax.cu:L102-391, bindings L778-884.
 * mode 0: softmax over the WHOLE tensor (softmax_f32 / softmax_f32x4: one global sum, grid fence),
 * mode 1: per-token (per-row) softmax without max subtraction, mode 2: per-token safe softmax,
 * mode 3: per-token online safe softmax (same result as 2).  dtype F32 or F16 (f16 I/O, f32 math).
 * `workspace` (mode 0 only): >= b200k_reduce_workspace_bytes(). */
int b200k_softmax(const void* x, void* y, int64_t S, int64_t H, int dtype, int mode, void* workspace, void* stream);

/* y = x * rsqrt(mean(x^2) + eps) * g for each row of x[N,K]; scalar g.  kernels/rms-norm/rms_norm.cu:L53-366, L457-800.
 * eps_inside_k = 1 reproduces the reference's f16-input kernels, which compute rsqrt(sum/(K + eps)) (L164 etc.).
 * acc_f16 = 1: squares summed in half like the *_f16 variants. */
int b200k_rms_norm(const void* x, void* y, int64_t N, int64_t K, float g, float eps, int dtype, int acc_f16,
                   int eps_inside_k, void* stream);

/* Interleaved-pair rotary embedding on x[seq_len, hidden] f32, theta = 10000.  kernels/rope/rope.cu:L20-113.
 * ref_quirk = 1 reproduces the reference kernels' integer-division exponent (every pair rotates with frequency 1.0,
 * see SURVEY.md §8 a9); ref_quirk = 0 is the textbook formula of the script's naive_rope (rope.py:L71-91). */
int b200k_rope_f32(const void* x, void* out, int64_t seq_len, int64_t hidden, int ref_quirk, void* stream);

/* hist[v] += 1 for v in a[0..n) (int32 values in [0, nbins)); `hist` (int32[nbins]) is zeroed by this call.
 * kernels/histogram/histogram.cu:L18-72.  b200k_max_i32 gives max(a) (the reference sizes its output as max+1
 * through a host sync, L57-60); `out_max` is a 1-element int32 device buffer. */
int b200k_max_i32(const void* a, int64_t n, void* out_max, void* stream);
int b200k_histogram_i32(const void* a, int64_t n, void* hist, int64_t nbins, void* stream);

/* out[i,:] = weight[idx[i],:], idx int32[n], weight [rows, emb] f32 or f16.  kernels/embedding/embedding.cu:L16-119. */
int b200k_embedding(const void* idx, const void* weight, void* out, int64_t n, int64_t rows, int64_t emb, int dtype,
                    void* stream);

/* ------------------------------------------------------------------------------------------------ support kernels, set 2
 * (SURVEY.md section 8f-3: the remaining bandwidth kernels of the reference, same recipe as above.)
 *
 * y = f(x) elementwise over n values, dtype B200K_F32 or B200K_F16 (f16 I/O, f32 math).
 *   kernels/relu/relu.cu:L21-97, sigmoid/sigmoid.cu:L24-136, gelu/gelu.cu:L38-163 (tanh approximation), swish/swish.cu:L20-97,
 *   elu/elu.cu:L35-120 (alpha = 1), hardswish/hardswish.cu:L36-140, hardshrink/hardshrink.cu:L33-135 (lambda = 0.5); each
 *   family's six entry points (f32, f32x4, f16, f16x2, f16x8, f16x8_pack) map here.
 * ref_clamp = 1 reproduces the input clamp of the reference's sigmoid / gelu kernels: x limited to +-88.3762626647949
 *   (f32 kernels) or to [-9.703125, 11.09375] (f16 kernels: MIN_EXP_F16 / MAX_EXP_F16 as rounded to half) BEFORE the
 *   function, so the f16 gelu saturates at 11.09375 for large x.  ref_clamp = 0 is the plain function. */
#define B200K_ACT_RELU 0
#define B200K_ACT_SIGMOID 1
#define B200K_ACT_GELU 2
#define B200K_ACT_SWISH 3
#define B200K_ACT_ELU 4
#define B200K_ACT_HARDSWISH 5
#define B200K_ACT_HARDSHRINK 6
int b200k_activation(const void* x, void* y, int64_t n, int dtype, int op, int ref_clamp, void* stream);

/* y = (x - mean(x)) * rsqrt(v) * g + b for each row of x[N,K]; scalar g, b; dtype F32 or F16 (f32 math).
 * kernels/layer-norm/layer_norm.cu:L48-419, bindings L732-812.  eps_inside_k = 1 reproduces the reference:
 * v = sum((x-mean)^2) / (K + eps) (L69, L103, L187 ...); eps_inside_k = 0 is the textbook v = sum(..)/K + eps. */
int b200k_layer_norm(const void* x, void* y, int64_t N, int64_t K, float g, float b, float eps, int dtype,
                     int eps_inside_k, void* stream);

/* out[0] = sum_i a[i] * b[i] (f32 result, f32 accumulation; dtype F32 or F16).  kernels/dot-product/dot_product.cu:L20-184,
 * bindings L233-283.  Deterministic (fixed two-pass order) where the reference uses atomicAdd.  `out`: 1-element f32
 * device buffer; `workspace`: >= b200k_reduce_workspace_bytes(). */
int b200k_dot_prod(const void* a, const void* b, void* out, int64_t n, int dtype, void* workspace, void* stream);

/* y[N,M] = transpose(x[M,N]), fp32.  kernels/mat-transpose/mat_transpose.cu:L20-278 (13 entry points, L296-359). */
int b200k_mat_transpose_f32(const void* x, void* y, int64_t M, int64_t N, void* stream);

/* y[M] = A[M,K] x[K], dtype F32 or F16 (f32 accumulation; the reference's hgemv accumulates in half).
 * kernels/sgemv/sgemv.cu:L20-104 (sgemv_k32_f32, sgemv_k128_f32x4, sgemv_k16_f32), kernels/hgemv/hgemv.cu:L24-108. */
int b200k_gemv(const void* a, const void* x, void* y, int64_t M, int64_t K, int dtype, void* stream);
/* y[b][N,M] = x[b][M,N]^T for 16-bit elements (f16 / bf16), `batch` matrices back to back; exact.  Used by the drop-in
 * flash_attn_mma_stages_*_swizzle_qkv entry points for head dims above 128 (V arrives as [B,H,D,N], flash_attn.cc:L128-159). */
int b200k_transpose_u16_batched(const void* x, void* y, int64_t batch, int64_t M, int64_t N, void* stream);

/* Debug hook, not part of the drop-in surface: device buffer of 3*32*8 uint64 that the next traced FA-2 launch
 * (variant | 0x100, D = 64 or 128) fills with clock64() stamps of CTA (0,0); see tools/gpu_trace_fa2.py. */
int b200k_debug_set_trace(void* dev_u64_buffer);
/* Debug hook of the GEMM kernel: 128 uint64 %globaltimer stamps per cluster (see hgemm_tcgen05.cu); NULL switches it off. */
int b200k_debug_set_hgemm_trace(void* dev_u64_buffer);
/* Debug hook, host only (runs without a GPU): the stream-K work-item schedule of the 256 x 256 pair GEMM for `num_tiles`
 * tiles of `num_kb` k-blocks on `clusters` CTA pairs, as rows of 7 int32 {cluster, item, tile, kb0, kb1, kind, last_writer}
 * (kind 0 = whole tile, 1 = writer of partial sums, 2 = finisher); returns the row count.  tests/test_abi.py checks coverage
 * and the wait-for order with it. */
int64_t b200k_debug_hgemm_schedule(int64_t num_tiles, int num_kb, int clusters, int tune, int32_t* rows, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* B200K_H_ */
