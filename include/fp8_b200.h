/*
 * fp8_b200.h -- C ABI of libfp8_b200.so: the B200 (sm_100a) implementation of the
 * fp8-mps-metal FP8 (e4m3fn) hot path.
 *
 * This is the drop-in boundary.  Every entry point replaces one kernel-dispatch site of the
 * reference (audiohacking/fp8-mps-metal); the reference's closest analogue of this ABI is the
 * buffer-index / setBytes contract of its C++ bridge (fp8_bridge.cpp:209-240) and the
 * torch.mps.compile_shader call sites in fp8_mps_native.py.
 *
 * Conventions (all entry points):
 *   - plain C: raw DEVICE pointers, extents, dtype enums, a CUDA stream handle (cudaStream_t
 *     passed as void*; NULL = legacy default stream).  No torch types.
 *   - no allocation, no host synchronisation, no ownership transfer.  The call enqueues work on
 *     `stream` and returns.  Re-entrant and thread-safe: any host thread may call any entry point on
 *     any stream, including its first call of the process or of the thread (a thread without a current
 *     CUDA context is given the current device's primary context).  Every entry point may be called
 *     while the stream is being captured into a CUDA graph, global capture mode included, first call
 *     included; a replay runs the captured kernels only.
 *   - optional arguments are NULL pointers (absent), never sentinel values.
 *   - return value: FP8B_OK (0) or a negative fp8b_status.  There is NO silent fallback: an
 *     unsupported shape/alignment returns FP8B_ERR_UNSUPPORTED and does nothing; there is no CPU
 *     path anywhere in this library.
 *   - the FP8 format is e4m3fn stored as uint8 with the REFERENCE's codec semantics
 *     (fp8_matmul.metal:19-92): decode maps 0x7F/0xFF to +0.0; encode saturates at +-448 (0x7E),
 *     flushes |v| < 2^-9 to signed zero (-0.0 -> 0x00), rounds the 3-bit mantissa to nearest-even
 *     WITHOUT carrying into the exponent.  NaN inputs to encode (undefined in the reference)
 *     give 0x7F.
 */
#ifndef FP8_B200_H
#define FP8_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FP8B_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define FP8B_API __attribute__((visibility("default")))
#else
#define FP8B_API
#endif

typedef enum fp8b_status {
    FP8B_OK = 0,
    FP8B_ERR_INVALID = -1,     /* bad argument (null pointer, negative extent, bad enum, bad scale length) */
    FP8B_ERR_UNSUPPORTED = -2, /* valid request this entry point cannot serve (alignment, M range, workspace) */
    FP8B_ERR_CUDA = -3,        /* a CUDA runtime/driver call failed; see fp8b_last_cuda_error() */
    FP8B_ERR_NO_DEVICE = -4    /* current device is not compute capability 10.x */
} fp8b_status;

/* Element types.  FP8B_OUT_E4M3FN is an OUTPUT type of the matmul entry points only (1-byte elements, the reference
 * codec's bytes of the fp32 epilogue value, exactly fp8b_encode with no prescale); every cast entry point, every
 * bias_dtype and the x_dtype of fp8b_linear_dynamic reject it with FP8B_ERR_INVALID. */
typedef enum fp8b_dtype {
    FP8B_F32 = 0,
    FP8B_F16 = 1,
    FP8B_BF16 = 2,
    FP8B_OUT_E4M3FN = 3
} fp8b_dtype;

/* Which matmul kernel fp8b_scaled_mm() picked / should pick. */
typedef enum fp8b_mm_algo {
    FP8B_MM_AUTO = 0,    /* M <= 16 -> GEMV; else tcgen05 when its alignment rules hold, else SIMT */
    FP8B_MM_GEMV = 1,    /* split-K streaming GEMV, M in [1,16]   (replaces fp8_scaled_vecmat_kernel) */
    FP8B_MM_TCGEN05 = 2, /* tcgen05/TMEM/TMA GEMM                 (replaces fp8_scaled_matmul_kernel / fp8_scaled_mm_fast) */
    FP8B_MM_SIMT = 3     /* CUDA-core tiled GEMM, any shape/alignment (the no-TMA device path) */
} fp8b_mm_algo;

/* ---- library / diagnostics ------------------------------------------------------------- */

FP8B_API int fp8b_version(void);
FP8B_API const char* fp8b_status_string(int status);
/* cudaError_t of the most recent failing CUDA call on this thread, or the CUresult of a failing tensor-map encode
 * (0 if none). */
FP8B_API int fp8b_last_cuda_error(void);
/* Number of kernel launches this library has enqueued since load (all threads).  bench.py
 * reads it before/after the timed region to report `gpu_launches`. */
FP8B_API uint64_t fp8b_launch_count(void);

/*
 * Library options (process-wide, may be changed between calls).
 *   FP8B_OPT_PDL             1 (default): the GEMV and cast kernels are launched with programmatic dependent launch:
 *                            they become resident while their predecessor on the stream drains and wait
 *                            (griddepcontrol.wait) before their first global access, so results never depend on
 *                            it.  0: plain stream order always.
 *   FP8B_OPT_STATIC_WEIGHTS  0 (default).  1: the caller promises that the B operand (the weight matrix) of
 *                            fp8b_scaled_mm is never written by work still in flight on the stream.  The GEMV
 *                            kernels then start streaming B BEFORE waiting for the predecessor (only A, the
 *                            scales and the bias are read after the wait), which overlaps the ramp-up of one
 *                            call with the drain of the previous one in a chain of decode GEMVs.
 *   FP8B_OPT_TUNE_*          developer knobs that pick between RESULT-IDENTICAL kernel variants (tests and profiling
 *                            scripts A/B them); -1 = built-in rule.  Each starts from the environment variable of the
 *                            same name without the OPT_TUNE_ part (FP8B_GEMM_CFG, ...), read once at load time.
 *                              GEMM_CFG      tcgen05 tile: 1 = 128x256, 2 = 128x128 (one CTA); 3 = 256x256, 4 = 256x128,
 *                                            5 = 256x192 (CTA pairs)
 *                              GEMV_IMPL     1 = FHFMA warp-per-row, 2 = warp-MMA (other values: the built-in rule)
 *                              DYNAMIC_PLAN  fp8b_linear_dynamic: 1 = single kernel, 2 = quantise + chained GEMV
 *                              CAST_SHAPE    cast launch shape: 1 = small tiles, 2 = big tiles
 *                              GEMM_STORE    tcgen05 epilogue: 1 = st.global from the epilogue warps, 2 = TMA store
 *                              GEMV_UNROLL / GEMV_BATCH / AMAX_CAP   load batching of the GEMV kernels / amax grid cap
 *                              GEMM_RASTER   tcgen05 tile order: 1 = M fastest, 2 = N fastest (whole output rows complete together),
 *                                            3 = N fastest inside bands of 8 M-blocks (L2 reuse when both operands are large)
 *                              GEMM_SPLITK   split-K plan for problems with few tiles: 1 = never, 2 / 4 = that many CTAs per tile.
 *                                            (The one knob that is not bit-neutral: partial sums over K ranges are added in
 *                                            rank order, so results are deterministic but rounded differently from the
 *                                            one-CTA-per-tile plans; both are within the stated tolerances of the oracle.)
 */
typedef enum fp8b_option {
    FP8B_OPT_PDL = 0,
    FP8B_OPT_STATIC_WEIGHTS = 1,
    FP8B_OPT_TUNE_GEMM_CFG = 16,
    FP8B_OPT_TUNE_GEMV_IMPL = 17,
    FP8B_OPT_TUNE_DYNAMIC_PLAN = 18,
    FP8B_OPT_TUNE_CAST_SHAPE = 19,
    FP8B_OPT_TUNE_GEMM_STORE = 20,
    FP8B_OPT_TUNE_GEMV_UNROLL = 21,
    FP8B_OPT_TUNE_GEMV_BATCH = 22,
    FP8B_OPT_TUNE_AMAX_CAP = 23,
    FP8B_OPT_TUNE_GEMM_RASTER = 24,
    FP8B_OPT_TUNE_GEMM_SPLITK = 25
} fp8b_option;
FP8B_API int fp8b_set_option(int option, int value);
FP8B_API int fp8b_get_option(int option);

/* ---- casts ------------------------------------------------------------------------------ */

/*
 * FP8 -> fp16 dequantise.  Replaces fp8_to_half_kernel (fp8_matmul.metal:215-223) together with
 * the host-side scale pass of fp8_dequantize (fp8_mps_native.py:98-124; bridge fp8_bridge.cpp:265-306):
 *     out[i] = RN16( half(dec(in[i])) * RN16(scale[0]) )        (fp16 multiply, native.py:121-122)
 * scale: device pointer to one float, or NULL for the bare kernel (out = half(dec(in))).
 */
FP8B_API int fp8b_dequant_f16(const uint8_t* in, void* out_f16, size_t n, const float* scale, void* stream);

/*
 * FP8 -> {f32,f16,bf16} exact cast (every e4m3 value is representable in all three).  This is
 * the `.to(dtype)` route of the patch (fp8_mps_patch.py:200-223: dequantise with scale 1, then
 * .to(dtype)) done in one pass.
 */
FP8B_API int fp8b_dequant(const uint8_t* in, void* out, int out_dtype, size_t n, void* stream);

/*
 * FP8 operand formats.  Every entry point without a format argument takes e4m3fn, the only format the reference has
 * kernels for.  The reference's patch also ACCEPTS float8_e5m2 tensors (fp8_mps_patch.py:48-49,65) but decodes
 * them with the e4m3fn codec, i.e. wrongly; the *_fmt entry points decode e5m2 by its own definition (the upper
 * byte of an IEEE binary16: exact, +-inf and NaN preserved -- PyTorch's cast).  Decode only: there is no e5m2 encoder.
 */
enum fp8b_format {
    FP8B_E4M3FN = 0,
    FP8B_E5M2 = 1
};

/* fp8b_dequant / fp8b_dequant_f16 for either format.  scale (nullable) is allowed for FP8B_F16 output only. */
FP8B_API int fp8b_dequant_fmt(const uint8_t* in, int in_format, void* out, int out_dtype, size_t n, const float* scale,
                     void* stream);

/*
 * {f32,f16,bf16} -> FP8 encode.  Replaces float_to_fp8_kernel (fp8_matmul.metal:228-236) and the
 * host-side fp32 up-conversion / pre-scale passes of fp8_encode and fp8_quantize
 * (fp8_mps_native.py:127-155, :170-187):
 *     out[i] = enc( f32(in[i]) * prescale[0] )      (fp32 multiply; prescale NULL = no multiply)
 * The input is read in its native dtype (widening to fp32 is exact, native.py:142).
 */
FP8B_API int fp8b_encode(const void* in, int in_dtype, uint8_t* out, size_t n, const float* prescale, void* stream);

/*
 * Batched casts: many tensors, ONE launch (per 512 tensors).  Converting a checkpoint with the reference is one
 * Tensor.to() per weight (fp8_mps_patch.py:143-230 -> fp8_mps_native.py:127-155 / :98-124), i.e. one kernel launch
 * per tensor; on a B200 the ramp-up and drain of a launch cost ~15 % of a FLUX-sized tensor's streaming time.
 * These entry points take a HOST array of (in, out, n) device spans and stream them as one tile list.
 *   fp8b_encode_batch : span.in = in_dtype elements, span.out = uint8     (== fp8b_encode with prescale NULL, per span)
 *   fp8b_dequant_batch: span.in = uint8,             span.out = out_dtype (== fp8b_dequant, per span)
 * Spans may have any length (0 allowed) and any alignment (unaligned ones take the single-tensor path); they must
 * not overlap.  The span table is passed in the kernel parameters: nothing is copied, nothing is allocated.
 */
typedef struct fp8b_span {
    const void* in;
    void* out;
    size_t n;          /* elements */
} fp8b_span;
FP8B_API int fp8b_encode_batch(const fp8b_span* spans, int count, int in_dtype, void* stream);
FP8B_API int fp8b_dequant_batch(const fp8b_span* spans, int count, int out_dtype, void* stream);

/*
 * amax -> scale, on the device, without the reference's .item() host sync (fp8_mps_native.py:174-176,:189):
 *     amax      = max_i |f32(in[i])|
 *     scale_d   = amax > 0 ? 448.0 / (double)amax : 1.0        (Python-double arithmetic)
 *     scale_out[0]     = (float)scale_d                         (what fp8b_encode takes as prescale)
 *     inv_scale_out[0] = (float)(1.0 / scale_d)                 (what fp8_quantize returns)
 * scratch: device pointer to one uint32 the call may clobber (it is reset by the call itself).
 * Special amax values give (here, in fp8b_quantize_rows and in fp8b_linear_dynamic, per row):
 *     n == 0 or amax == 0       : scale 1, inv 1
 *     amax NaN (a NaN input)    : amax > 0 fails, so scale 1, inv 1; NaN inputs encode to 0x7F
 *     amax +inf (an inf input)  : scale 0, inv = (float)(1.0/0.0) = +inf (the reference raises ZeroDivisionError);
 *                                 finite inputs encode to 0x00, +-inf to 0x7F (inf * 0 = NaN)
 *     amax < A* ~= 1.3166e-36   : (float)scale_d overflows to +inf, inv is a subnormal or 0; zeros encode to 0x7F
 *                                 (0 * inf = NaN), nonzeros to 0x7E / 0xFE
 */
FP8B_API int fp8b_amax_scale(const void* in, int in_dtype, size_t n, float* scale_out, float* inv_scale_out,
                    uint32_t* scratch, void* stream);

/*
 * Row-wise (per-channel) quantise: the fp8_quantize arithmetic (fp8_mps_native.py:158-190) applied to each
 * row of a contiguous (rows, cols) matrix in one launch:
 *     amax_r = max_j |f32(in[r,j])|;  scale_r = amax_r > 0 ? 448.0/amax_r : 1.0 (double)
 *     out[r,j] = enc( f32(in[r,j]) * (float)scale_r );   inv_scale_out[r] = (float)(1.0/scale_r)
 * inv_scale_out (device float[rows]) is what fp8b_scaled_mm takes as a per-row scale_a / scale_b.
 * NaN, inf and tiny amax values give the results listed at fp8b_amax_scale, row by row.
 * (The reference only quantises per tensor; its kernels accept per-row scales, fp8_matmul.metal:144-145.)
 */
FP8B_API int fp8b_quantize_rows(const void* in, int in_dtype, int rows, size_t cols, uint8_t* out,
                       float* inv_scale_out, void* stream);

/* ---- scaled matmul ---------------------------------------------------------------------- */

/*
 * C[m,n] = cast_out( (((sum_k dec(A[m,k]) * dec(B[n,k])) * sa) * sb [+ bias[n]]) [* scale_result[0]] )
 *
 * Replaces fp8_scaled_matmul_kernel (fp8_matmul.metal:99-147), fp8_scaled_vecmat_kernel (:155-210),
 * fp8_scaled_mm_fast (fp8_mps_native.py:213-267) and the patch's separate bias / scale_result / cast
 * passes (fp8_mps_patch.py:95-104), in one kernel.
 *
 *   A            (M,K) uint8 row-major, contiguous (lda = K)
 *   B            (N,K) uint8 row-major, contiguous -- the reference's "pre-transposed" weight layout
 *   C            (M,N) out_dtype, row stride ldc elements (ldc >= N); ldc lets a rank write its column
 *                shard straight into a wider matrix.  out_dtype FP8B_OUT_E4M3FN: C[m,n] = enc(v) where v is the
 *                fp32 value the same call computes for FP8B_F32 and enc is fp8b_encode's codec (saturate at
 *                +-448, inf included; flush |v| < 2^-9; no carry into the exponent; -0.0 -> 0x00; NaN -> 0x7F).
 *                Elements are 1 byte, so ldc counts bytes and every 16-byte rule below counts bytes.  The
 *                kernel choice does not depend on out_dtype.  (float8_e5m2 output is not offered.)
 *   scale_a      device float[scale_a_len], scale_a_len in {1, M}   (independently of scale_b: fixes the
 *   scale_b      device float[scale_b_len], scale_b_len in {1, N}    reference's all-or-nothing scale_mode)
 *   bias         device [N] of bias_dtype, or NULL
 *   scale_result device float[1], or NULL
 *   workspace    device scratch of at least fp8b_scaled_mm_workspace_bytes(M,N,K) bytes (may be NULL
 *                when that is 0).  Contents are don't-care on entry and exit.
 *   algo         fp8b_mm_algo; a non-AUTO choice that cannot serve the shape returns
 *                FP8B_ERR_UNSUPPORTED (no re-dispatch).
 *
 * NaN bytes (0x7F/0xFF) in A or B contribute 0, as in the reference (fp8_matmul.metal:21).
 *
 * Degenerate extents: M == 0 or N == 0 returns FP8B_OK and launches nothing.  K == 0 is a valid problem whose sum
 * is 0, so C = cast_out(((0 * sa) * sb [+ bias]) [* scale_result]); AUTO, GEMV (M <= 16) and SIMT serve it,
 * TCGEN05 needs K >= 16 and returns FP8B_ERR_UNSUPPORTED without touching C.
 */
FP8B_API int fp8b_scaled_mm(const uint8_t* A, const uint8_t* B, void* C, int out_dtype,
                   int M, int N, int K, int64_t ldc,
                   const float* scale_a, int scale_a_len,
                   const float* scale_b, int scale_b_len,
                   const void* bias, int bias_dtype,
                   const float* scale_result,
                   void* workspace, size_t workspace_bytes,
                   int algo, void* stream);

/*
 * Several independent M = 1 GEMVs in ONE launch (per 16 items):  y_i = _scaled_mm(x_i (1,K), W_i (N_i,K)^T) with
 * per-tensor scale_x, per-tensor or per-row scale_w, optional bias, all of one K, one out_dtype and one bias_dtype.
 * The reference issues one fp8_scaled_vecmat_kernel per projection (fp8_mps_native.py:78-86); on a B200 a third of a
 * decode GEMV's time is launch ramp-up and drain, which the projections of a layer that are independent of each
 * other (Q/K/V, gate/up; the x_i may be the same pointer) can pay once.  `items` is a HOST array; results are those
 * of fp8b_scaled_mm's M = 1 kernel.  Needs K % 16 == 0, 16 <= K <= 49152 and 16-byte aligned x_i / W_i, else
 * FP8B_ERR_UNSUPPORTED.  N_i == 0 items are skipped.
 */
typedef struct fp8b_gemv_item {
    const uint8_t* x;          /* (K,)   e4m3fn bytes */
    const uint8_t* W;          /* (N,K)  e4m3fn bytes, row-major */
    void* y;                   /* (N,)   out_dtype */
    int N;
    const float* scale_x;      /* [1] */
    const float* scale_w;      /* [1] or [N] */
    int scale_w_len;
    const void* bias;          /* [N] of bias_dtype, or NULL */
} fp8b_gemv_item;
FP8B_API int fp8b_gemv_batch(const fp8b_gemv_item* items, int count, int K, int out_dtype, int bias_dtype, void* stream);

/*
 * fp8b_scaled_mm with per-operand formats.  e4m3fn NaN bytes contribute 0 (the reference kernels' rule); e5m2
 * operands follow IEEE arithmetic (inf and NaN propagate into the fp32 sum).  M <= 16 runs the warp-MMA GEMV
 * (all four type pairs), larger M the tcgen05 GEMM (formats are two bits of the instruction descriptor).
 */
FP8B_API int fp8b_scaled_mm_fmt(const uint8_t* A, int a_format, const uint8_t* B, int b_format, void* C, int out_dtype,
                       int M, int N, int K, int64_t ldc,
                       const float* scale_a, int scale_a_len,
                       const float* scale_b, int scale_b_len,
                       const void* bias, int bias_dtype,
                       const float* scale_result,
                       int algo, void* stream);

/*
 * Linear layer with DYNAMIC per-row activation quantisation: fp8_quantize (per row) -> _scaled_mm in one call,
 * no host synchronisation (the reference's fp8_quantize reads amax back with .item(), fp8_mps_native.py:174):
 *     q[m,:], inv_m = fp8_quantize(X[m,:])          (amax, 448/amax in double, encode; fp8_mps_native.py:158-190)
 *     C[m,n] = cast_out( (((sum_k dec(q[m,k]) * dec(B[n,k])) * inv_m) * sb [+ bias[n]]) [* scale_result[0]] )
 * X is (M,K) float32 / float16 / bfloat16, contiguous.  For M == 1 this is exactly the reference composition
 * fp8_quantize(x) then torch._scaled_mm(x8, w8.t(), scale_a=inv, ...); for M > 1 each row gets its own scale
 * (= fp8b_quantize_rows).  inv_scale_a_out (device float[M], nullable) receives the row scales.
 * Special rows follow fp8b_amax_scale: a NaN amax gives inv_m = 1; an infinite amax gives inv_m = +inf, so that row of C
 * is NaN (every q is 0x00 or 0x7F, which decodes to 0, and 0 * inf = NaN); an amax below A* gives q = 0x7E / 0xFE
 * (zeros 0x7F) and a subnormal or zero inv_m.
 *
 * workspace: device, 16-byte aligned, >= fp8b_linear_dynamic_workspace_bytes(M,K).
 *   M <= 16, workspace given : rows quantised once by a one-CTA-per-row kernel, the GEMV chained behind it with
 *                              programmatic dependent launch (two launches).  The default plan of the bindings.
 *   M <= 16, workspace NULL  : ONE kernel, every CTA quantises the rows itself -- no scratch memory, but the encode
 *                              is repeated per CTA, so it only pays for small N.  Needs K % 16 == 0 and 16-byte
 *                              aligned X and B, else FP8B_ERR_UNSUPPORTED.  Same result bits as the chained plan.
 *   M  > 16                  : workspace required (FP8B_ERR_UNSUPPORTED without); quantise kernel, then the GEMM
 *                              fp8b_scaled_mm would pick, with per-row scale_a.
 * K == 0: the workspace plans serve it (every row has amax 0, so its scale is 1.0 and its sum 0); without a workspace
 * it is FP8B_ERR_UNSUPPORTED.
 */
FP8B_API int fp8b_linear_dynamic(const void* X, int x_dtype, const uint8_t* B, void* C, int out_dtype,
                      int M, int N, int K, int64_t ldc,
                      const float* scale_b, int scale_b_len,
                      const void* bias, int bias_dtype, const float* scale_result,
                      float* inv_scale_a_out, void* workspace, size_t workspace_bytes, void* stream);
FP8B_API size_t fp8b_linear_dynamic_workspace_bytes(int M, int K);

FP8B_API size_t fp8b_scaled_mm_workspace_bytes(int M, int N, int K);

/*
 * fp8b_scaled_mm (tcgen05 kernel) whose output pointer is an NVSwitch MULTICAST address -- the
 * fused compute + exchange step of an N-sharded linear (no reference counterpart; the reference is
 * single-device).  C_multicast addresses element (0,0) of this rank's column block inside a
 * multicast mapping (cuMulticast* / torch symmetric memory `multicast_ptr`) of a row-major (M, ldc)
 * matrix that exists on every GPU of the group: the epilogue stores each tile with multimem.st, so
 * the switch replicates it into every GPU's copy while the next tile is being computed.
 * The caller orders ranks around the call (a barrier before reuse of the buffer and one after).
 * Requires N % 32 == 0, 16-byte aligned C_multicast / ldc / scale_b / bias, and the TMA alignment
 * rules of the tcgen05 kernel; otherwise FP8B_ERR_UNSUPPORTED.  out_dtype FP8B_OUT_E4M3FN is FP8B_ERR_UNSUPPORTED
 * here: the multicast store path can only be exercised on an NVSwitch group, so no byte output is offered on it.
 */
FP8B_API int fp8b_scaled_mm_multicast(const uint8_t* A, const uint8_t* B, void* C_multicast, int out_dtype,
                             int M, int N, int K, int64_t ldc,
                             const float* scale_a, int scale_a_len,
                             const float* scale_b, int scale_b_len,
                             const void* bias, int bias_dtype,
                             const float* scale_result, void* stream);

/*
 * The same N-sharded linear with PEER STORES instead of the multicast mapping: the epilogue writes every 16-byte
 * piece of the output tile into this rank's (M,N) buffer and, as plain stores over NVLink, into the same offset of
 * each peer's buffer.  peer_deltas: DEVICE array of `world` (2..8) byte offsets, delta[r] = (address of rank r's
 * buffer as mapped in this process) - (address of the local buffer); the entry of the calling rank is 0.
 * C_local points at this rank's shard column inside its own buffer (ldc = full N).  Against the multicast mode a
 * rank's own shard does not travel to the switch and back, so each GPU receives (world-1)/world of the output
 * instead of all of it: the better plan for small worlds.  Same 16-byte-path requirements as the multicast mode
 * (N % 32 == 0; 16-byte aligned C_local, ldc * sizeof(out), per-row scale_b and bias; K % 16 == 0, K > 0).  Runs on
 * the CTA-pair tile configurations only: the built-in tile rule picks one when M > 128 and N > 128, a forced
 * FP8B_OPT_TUNE_GEMM_CFG 3 / 4 / 5 serves any M and N, and a forced one-CTA configuration (1 / 2) is refused.  Every
 * unmet requirement returns FP8B_ERR_UNSUPPORTED with nothing launched; world outside 2..8 or a NULL peer_deltas returns
 * FP8B_ERR_INVALID.  M == 0 or N == 0: FP8B_OK, nothing launched.
 */
FP8B_API int fp8b_scaled_mm_peers(const uint8_t* A, const uint8_t* B, void* C_local, const int64_t* peer_deltas, int world,
                         int out_dtype, int M, int N, int K, int64_t ldc,
                         const float* scale_a, int scale_a_len,
                         const float* scale_b, int scale_b_len,
                         const void* bias, int bias_dtype,
                         const float* scale_result, void* stream);

/*
 * The N-sharded linear as ONE kernel that computes and exchanges: the tcgen05 GEMM with a TMA-store epilogue that
 * pushes every finished 128-row x 128-byte box of the output to n_dst destinations -- this rank's (M, ldc) buffer and
 * the same place in each peer's buffer, mapped into this process (torch symmetric memory `buffer_ptrs`, cuMemMap of
 * a fabric / POSIX handle, or cudaIpcOpenMemHandle).  No reference counterpart (the reference is single-device,
 * fp8_bridge.cpp:67); it replaces "GEMM, then ncclAllGather, then a re-layout pass" of BASELINE.json's C4 config.
 *   C_dsts   HOST array of n_dst (1..8) device pointers.  C_dsts[d] addresses element (0,0) of THIS rank's column
 *            block inside destination d's row-major (M, ldc) matrix; C_dsts[0] is normally the local buffer.  With
 *            n_dst == 1 this is fp8b_scaled_mm's tcgen05 kernel with a TMA-store epilogue.
 * The epilogue warps only fill a shared-memory ring; a dedicated warp issues cp.async.bulk.tensor stores, several
 * in flight, so the tensor-memory accumulator is released as soon as it is drained and NVLink writes overlap the
 * next tile's MMAs.  Each GPU receives (world-1)/world of the output.  The caller orders ranks around the call (a
 * barrier before a buffer is reused and one after).  Needs 16-byte aligned A / B / every C_dsts[d], K % 16 == 0,
 * ldc * sizeof(out) % 16 == 0 and N * sizeof(out) % 16 == 0 (TMA stores move 16-byte units); otherwise any M, N -- TMA
 * clips the tile edges (fp8b_scaled_mm_push_supported).  Else FP8B_ERR_UNSUPPORTED.  With FP8B_OUT_E4M3FN (1-byte
 * elements: N % 16 == 0 and ldc % 16 == 0) a tile must also be a whole number of 128-column boxes, so the built-in tile
 * rule never picks 256 x 192 for it and a forced FP8B_OPT_TUNE_GEMM_CFG 5 returns FP8B_ERR_UNSUPPORTED.
 */
FP8B_API int fp8b_scaled_mm_push(const uint8_t* A, const uint8_t* B, void* const* C_dsts, int n_dst,
                        int out_dtype, int M, int N, int K, int64_t ldc,
                        const float* scale_a, int scale_a_len,
                        const float* scale_b, int scale_b_len,
                        const void* bias, int bias_dtype,
                        const float* scale_result, void* stream);
/*
 * fp8b_scaled_mm_push with the closing barrier's SEND side fused into the kernel: when the last CTA of the grid has
 * pushed its last box it stores `epoch` (release, system scope) into signal_flags[d] for every destination d --
 * a 64-bit word in destination d's memory (its slot for this rank in a symmetric flag array; NULL for this rank
 * itself).  cta_counter: a device uint32 that is zero between launches.  Epochs must increase from call to call.
 * The RECEIVE side is fp8b_peer_wait: a one-warp kernel, launched with programmatic dependent launch so that it is
 * resident and polling while the push kernel still runs; it completes when flags[r] >= epoch for every r != rank
 * (every peer's boxes have landed here) and this rank's own push kernel has completed.  Together they replace the
 * separate barrier kernel after the exchange (8 us at w = 2) by ~one NVLink round trip.  A peer that never signals
 * trips a 20 s watchdog (the kernel traps) instead of hanging the GPU.
 */
FP8B_API int fp8b_scaled_mm_push_signal(const uint8_t* A, const uint8_t* B, void* const* C_dsts, int n_dst,
                               int out_dtype, int M, int N, int K, int64_t ldc,
                               const float* scale_a, int scale_a_len,
                               const float* scale_b, int scale_b_len,
                               const void* bias, int bias_dtype, const float* scale_result,
                               uint64_t* const* signal_flags, uint32_t* cta_counter, uint64_t epoch, void* stream);
FP8B_API int fp8b_peer_wait(const uint64_t* flags, int world, int rank, uint64_t epoch, void* stream);

/* 1 when fp8b_scaled_mm_push can serve this shape and alignment (a pure function: every rank of a group can
 * evaluate it for every other rank's shard before anyone launches). */
FP8B_API int fp8b_scaled_mm_push_supported(int out_dtype, int M, int N, int K, int64_t ldc, const void* A, const void* B,
                                  const void* C);

/* The algorithm FP8B_MM_AUTO resolves to for this problem (pointers supply the alignment). */
FP8B_API int fp8b_scaled_mm_select(const uint8_t* A, const uint8_t* B, const void* C, int out_dtype,
                          int M, int N, int K, int64_t ldc);

#ifdef __cplusplus
}
#endif
#endif /* FP8_B200_H */
