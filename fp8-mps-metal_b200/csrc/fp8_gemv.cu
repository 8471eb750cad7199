// FP8 GEMV for M = 1..16:  C[m,n] = epi( sum_k dec(A[m,k]) * dec(B[n,k]) ).
//
// Replaces fp8_scaled_vecmat_kernel (fp8_matmul.metal:155-210; one 32-lane simdgroup per output
// row, 4 bytes per lane per step, exp2() decode, simd_sum) and the M = 2..16 use of
// fp8_scaled_matmul_kernel (:99-147, dispatch rule fp8_mps_native.py:208).
//
// HBM-bound: the weight matrix B (N*K bytes) is streamed exactly once.
//   * one warp per weight row, 8 rows per CTA; each lane issues UNROLL independent 16-byte
//     ld.global.L1::no_allocate loads (512 contiguous bytes per warp per load) before consuming any
//     of them.  Coherent loads, not .nc: every launch uses programmatic dependent launch and ptxas
//     moves non-coherent loads above griddepcontrol.wait (see ld_x_v4 / ldg_w_v4);
//   * x (the A rows) is decoded once per CTA into shared memory as fp16 (every e4m3 value is
//     exact in fp16), split in two 16-byte planes so the per-lane LDS.128 are conflict-free;
//   * weights are decoded in registers with cvt.rn.f16x2.e4m3x2 (2 elements / instruction) and
//     accumulated with the sm_100 mixed-precision FMA fma.rn.f32.f16 (SASS FHFMA): the fp16 x fp16
//     product is formed exactly and added into an fp32 accumulator -- the reference's fp32
//     accumulation (metal:192) without ever widening the operands;
//   * lanes are reduced with warp shuffles (the simd_sum of metal:202);
//   * split-K: when N alone cannot fill the GPU the K range is split over a thread-block cluster
//     (1 x S x 1) and the S partial sums are reduced through distributed shared memory by the
//     rank-0 CTA, in rank order (deterministic, no workspace, no atomics);
//   * scales, bias, scale_result and the output cast are fused into the epilogue.
//   * fp8_gemv_xq_kernel: the same kernel fed with UN-quantised activations (fused per-row
//     fp8_quantize, fp8b_linear_dynamic without a workspace);
//   * NaN bytes: the hardware decode yields NaN where the reference decodes 0 (metal:21).  A NaN
//     accumulator can only come from such a byte, so it is detected after the reduction and that
//     output alone is recomputed with the masked scalar loop.
#include <cooperative_groups.h>
#include "fp8_mm.cuh"

namespace cg = cooperative_groups;

namespace fp8b {

constexpr int kGemvThreads = 256;
constexpr int kGemvWarps = kGemvThreads / 32;
constexpr int kGemvMaxMT = 4;
constexpr int kGemvMaxSplit = 8;
constexpr int kGemvMaxSmem = 96 * 1024;

struct GemvParams {
    const uint8_t* A;      // already offset to the first row handled by this launch
    const uint8_t* B;
    int m0;                // global row index of A row 0 (for scales / output)
    int N, K;
    int k_per_split;       // multiple of 16
    int k_panel;           // multiple of 16; smem holds MT * k_panel fp16
    int static_b;          // FP8B_OPT_STATIC_WEIGHTS: B may be read before the predecessor kernel completes
    Epi epi;
};

// fused dynamic-quantisation kernel: GemvParams (A unused) + the un-quantised activations
struct GemvXqParams {
    GemvParams g;
    const void* X;         // (M,K) of x_dtype, row m0 first
    int x_dtype;
    float* inv_scale_out;  // optional [M] output of the per-row inverse scales (may be null)
};

__device__ __forceinline__ uint4 ldg_w_v4(const uint8_t* p) {
    uint4 r;
    // coherent (no .nc): every launch uses programmatic dependent launch, and ptxas hoists non-coherent loads above
    // griddepcontrol.wait -- B may have been written by the kernel just before (an encode, a transfer)
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// Activations: coherent load.  x is typically written by the predecessor kernel; ptxas hoists non-coherent
// (.nc / __ldg) loads above griddepcontrol.wait, so those must never be used for it.
__device__ __forceinline__ uint4 ld_x_v4(const uint8_t* p) {
    uint4 r;
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// acc += w.lo*x.lo + w.hi*x.hi with exact fp16 products and fp32 accumulation (FHFMA).
__device__ __forceinline__ void fhfma2(float& acc, uint32_t w2, uint32_t x2) {
    asm("{\n\t.reg .b16 a0, a1, b0, b1;\n\t"
        "mov.b32 {a0, a1}, %1;\n\tmov.b32 {b0, b1}, %2;\n\t"
        "fma.rn.f32.f16 %0, a0, b0, %0;\n\tfma.rn.f32.f16 %0, a1, b1, %0;\n\t}"
        : "+f"(acc) : "r"(w2), "r"(x2));
}

__device__ __forceinline__ float gemv_load_x(const void* x, int dtype, size_t i) {
    if (dtype == FP8B_F32) return reinterpret_cast<const float*>(x)[i];
    if (dtype == FP8B_F16) return __half2float(reinterpret_cast<const __half*>(x)[i]);
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(x)[i]);
}

// 16 consecutive activations as fp32 (16-byte loads; i is a multiple of 16 and X is 16-byte aligned)
__device__ __forceinline__ void xq_load16(const void* x, int dtype, size_t i, float (&f)[16]) {
    if (dtype == FP8B_F32) {
        const float4* v = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + i);
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float4 q = v[j]; f[4 * j] = q.x; f[4 * j + 1] = q.y; f[4 * j + 2] = q.z; f[4 * j + 3] = q.w; }
    } else {
        const uint4* v = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(x) + i);
        uint32_t w[8];
        { const uint4 q0 = v[0], q1 = v[1]; w[0] = q0.x; w[1] = q0.y; w[2] = q0.z; w[3] = q0.w; w[4] = q1.x; w[5] = q1.y; w[6] = q1.z; w[7] = q1.w; }
        if (dtype == FP8B_F16) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
                f[2 * j] = t.x; f[2 * j + 1] = t.y;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) { f[2 * j] = __uint_as_float(w[j] << 16); f[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u); }
        }
    }
}

// quantised value of one activation, as the reference composition fp8_quantize -> kernel decode sees it
__device__ __forceinline__ float gemv_xq_value(const void* x, int dtype, size_t i, float scale) {
    return dec1_f32(enc1_f32(__fmul_rn(gemv_load_x(x, dtype, i), scale)));
}

// masked reference dot product for the XQ kernels (NaN weight bytes contribute 0, fp8_matmul.metal:21)
static __device__ __noinline__ float slow_dot_masked_xq(const void* x, int dtype, size_t x_off, float scale,
                                                        const uint8_t* __restrict__ b, int K) {
    float s = 0.0f;
    for (int k = 0; k < K; ++k) s = __fmaf_rn(gemv_xq_value(x, dtype, x_off + k, scale), dec1_f32(b[k]), s);
    return s;
}

template <int MT>
__device__ __forceinline__ void gemv_consume(const uint4& w, const uint4* __restrict__ xs, int nvec_panel, int v,
                                             float (&acc0)[MT], float (&acc1)[MT])
{
    uint32_t w0l, w0h, w1l, w1h, w2l, w2h, w3l, w3h;
    dec4_f16x2_raw(w.x, w0l, w0h);
    dec4_f16x2_raw(w.y, w1l, w1h);
    dec4_f16x2_raw(w.z, w2l, w2h);
    dec4_f16x2_raw(w.w, w3l, w3h);
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        const uint4 xa = xs[(m * 2 + 0) * nvec_panel + v];     // elements 0..7 of the vector
        const uint4 xb = xs[(m * 2 + 1) * nvec_panel + v];     // elements 8..15
        fhfma2(acc0[m], w0l, xa.x); fhfma2(acc1[m], w0h, xa.y);
        fhfma2(acc0[m], w1l, xa.z); fhfma2(acc1[m], w1h, xa.w);
        fhfma2(acc0[m], w2l, xb.x); fhfma2(acc1[m], w2h, xb.y);
        fhfma2(acc0[m], w3l, xb.z); fhfma2(acc1[m], w3h, xb.w);
    }
}

template <int MT, int U>
__global__ void __launch_bounds__(kGemvThreads)
fp8_gemv_kernel(const GemvParams p)
{
    extern __shared__ __align__(16) uint8_t gemv_smem[];
    uint4* xs = reinterpret_cast<uint4*>(gemv_smem);
    __shared__ float part[kGemvWarps][kGemvMaxMT];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * kGemvWarps + warp;
    const bool row_ok = row < p.N;
    const int K = p.K;
    const int k_begin = blockIdx.y * p.k_per_split;
    const int k_end = min(K, k_begin + p.k_per_split);
    const uint8_t* wrow = p.B + (size_t)(row_ok ? row : 0) * K;

    float acc0[MT], acc1[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) { acc0[m] = 0.0f; acc1[m] = 0.0f; }

    // Programmatic dependent launch (see fp8_b200.h, FP8B_OPT_STATIC_WEIGHTS): the next kernel may start
    // scheduling now; we wait for our predecessor before reading anything it may have written -- all
    // inputs by default, everything except the weights when they are declared static.
    pdl_launch_dependents();
    bool need_wait = p.static_b != 0;
    if (!need_wait) pdl_wait();

    for (int kp = k_begin; kp < k_end; kp += p.k_panel) {
        const int len = min(k_end - kp, p.k_panel);
        const int nvec = len >> 4;
        const int nvec_panel = p.k_panel >> 4;
        const uint8_t* wp = wrow + kp;
        // first batch of weight vectors goes in flight BEFORE x is staged, so the prologue
        // (x load + decode + barrier) overlaps the first HBM round trip
        uint4 cur[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int vv = lane + 32 * u;
            cur[u] = (row_ok && vv < nvec) ? ldg_w_v4(wp + (size_t)vv * 16) : make_uint4(0u, 0u, 0u, 0u);
        }
        if (need_wait) { pdl_wait(); need_wait = false; }
        if (kp != k_begin) __syncthreads();
        // stage x[:, kp : kp+len] as fp16 (raw hardware decode; NaN bytes stay NaN on purpose)
        for (int i = threadIdx.x; i < MT * nvec; i += kGemvThreads) {
            const int m = i / nvec, v = i - m * nvec;
            const uint4 xb = ld_x_v4(p.A + (size_t)m * K + kp + (size_t)v * 16);
            uint4 lo, hi;
            dec4_f16x2_raw(xb.x, lo.x, lo.y);
            dec4_f16x2_raw(xb.y, lo.z, lo.w);
            dec4_f16x2_raw(xb.z, hi.x, hi.y);
            dec4_f16x2_raw(xb.w, hi.z, hi.w);
            xs[(m * 2 + 0) * nvec_panel + v] = lo;
            xs[(m * 2 + 1) * nvec_panel + v] = hi;
        }
        __syncthreads();
        if (row_ok) {
            for (int v = lane; v < nvec; v += 32 * U) {
                uint4 nxt[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {                       // next batch in flight while this one is consumed
                    const int vv = v + 32 * (U + u);
                    nxt[u] = vv < nvec ? ldg_w_v4(wp + (size_t)vv * 16) : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int vv = v + 32 * u;
                    if (vv < nvec) gemv_consume<MT>(cur[u], xs, nvec_panel, vv, acc0, acc1);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) cur[u] = nxt[u];
            }
        }
    }

    if (need_wait) pdl_wait();                       // empty K range: still order the stores below
    float s[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        float t = acc0[m] + acc1[m];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, o);
        s[m] = t;
    }

    const int S = gridDim.y;
    if (S == 1) {
        if (row_ok && lane < MT) {
            float v = 0.0f;
#pragma unroll
            for (int m = 0; m < MT; ++m) if (lane == m) v = s[m];
            if (v != v) v = slow_dot_masked(p.A + (size_t)lane * K, wrow, K);
            const int gm = p.m0 + lane;
            epi_store(p.epi, gm, row, epi_apply(p.epi, v, gm, row));
        }
        return;
    }

    // split-K: reduce the S partial sums through distributed shared memory, in rank order
    cg::cluster_group cluster = cg::this_cluster();
    if (lane == 0) {
#pragma unroll
        for (int m = 0; m < MT; ++m) part[warp][m] = s[m];
    }
    cluster.sync();
    if (cluster.block_rank() == 0 && row_ok && lane < MT) {
        float v = 0.0f;
        for (int r = 0; r < S; ++r) {
            const float* rp = cluster.map_shared_rank(&part[0][0], r);
            v += rp[warp * kGemvMaxMT + lane];
        }
        if (v != v) v = slow_dot_masked(p.A + (size_t)lane * K, wrow, K);
        const int gm = p.m0 + lane;
        epi_store(p.epi, gm, row, epi_apply(p.epi, v, gm, row));
    }
    cluster.sync();
}

// Fused dynamic quantisation: the activations arrive UN-quantised (f32/f16/bf16).  Every CTA computes each row's amax, the
// reference's double-precision scale 448/amax (fp8_mps_native.py:174-176) and stages enc(x*scale) decoded to
// fp16 -- the composition fp8_quantize(x) -> _scaled_mm in ONE launch, bit-identical in the quantised values,
// with the inverse scale applied in the epilogue as scale_a.
template <int MT, int U>
__global__ void __launch_bounds__(kGemvThreads)
fp8_gemv_xq_kernel(const GemvXqParams xp)
{
    const GemvParams& p = xp.g;
    constexpr bool XQ = true;      // (the body keeps the structure of fp8_gemv_kernel; a shared template cost that kernel 2 %)
    extern __shared__ __align__(16) uint8_t gemv_smem[];
    uint4* xs = reinterpret_cast<uint4*>(gemv_smem);
    __shared__ float part[kGemvWarps][kGemvMaxMT];
    __shared__ float xq_scale[kGemvMaxMT], xq_inv[kGemvMaxMT];
    __shared__ uint32_t xq_red[kGemvWarps];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * kGemvWarps + warp;
    const bool row_ok = row < p.N;
    const int K = p.K;
    const int k_begin = blockIdx.y * p.k_per_split;
    const int k_end = min(K, k_begin + p.k_per_split);
    const uint8_t* wrow = p.B + (size_t)(row_ok ? row : 0) * K;

    float acc0[MT], acc1[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) { acc0[m] = 0.0f; acc1[m] = 0.0f; }

    // Programmatic dependent launch (see fp8_b200.h, FP8B_OPT_STATIC_WEIGHTS): the next kernel may start
    // scheduling now; we wait for our predecessor before reading anything it may have written -- all
    // inputs by default, everything except the weights when they are declared static.
    pdl_launch_dependents();
    bool need_wait = p.static_b != 0;
    if (!need_wait) pdl_wait();

    if (XQ) {
        // per-row amax over the FULL K range (every CTA recomputes it: x is tiny next to its weight rows and
        // L2-resident after the first CTA).  16-byte loads; |x| compared on the bit patterns.
        if (need_wait) { pdl_wait(); need_wait = false; }
        for (int m = 0; m < MT; ++m) {
            uint32_t mx = 0;
            if (xp.x_dtype == FP8B_F32) {
                const uint4* xv = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(xp.X) + (size_t)m * K);
                for (int i = threadIdx.x; i < (K >> 2); i += kGemvThreads) {
                    const uint4 q = xv[i];
                    mx = max(max(mx, q.x & 0x7FFFFFFFu), max(q.y & 0x7FFFFFFFu, max(q.z & 0x7FFFFFFFu, q.w & 0x7FFFFFFFu)));
                }
            } else {
                const uint4* xv = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(xp.X) + (size_t)m * K);
                uint32_t m2 = 0;                                    // two u16 maxima side by side
                for (int i = threadIdx.x; i < (K >> 3); i += kGemvThreads) {
                    const uint4 q = xv[i];
                    m2 = __vmaxu2(__vmaxu2(m2, q.x & 0x7FFF7FFFu),
                                  __vmaxu2(__vmaxu2(q.y & 0x7FFF7FFFu, q.z & 0x7FFF7FFFu), q.w & 0x7FFF7FFFu));
                }
                const uint32_t h = max(m2 & 0xFFFFu, m2 >> 16);
                mx = xp.x_dtype == FP8B_F16 ? __float_as_uint(__half2float(__ushort_as_half((unsigned short)h))) : (h << 16);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
            if (lane == 0) xq_red[warp] = mx;
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t mm = 0;
                for (int w = 0; w < kGemvWarps; ++w) mm = max(mm, xq_red[w]);
                const float amax = __uint_as_float(mm);
                const double sc = (amax > 0.0f) ? 448.0 / (double)amax : 1.0;      // fp8_mps_native.py:175-176
                xq_scale[m] = (float)sc;
                xq_inv[m] = (float)(1.0 / sc);                                      // :189
                if (xp.inv_scale_out && blockIdx.x == 0 && blockIdx.y == 0) xp.inv_scale_out[m] = (float)(1.0 / sc);
            }
            __syncthreads();
        }
    }

    for (int kp = k_begin; kp < k_end; kp += p.k_panel) {
        const int len = min(k_end - kp, p.k_panel);
        const int nvec = len >> 4;
        const int nvec_panel = p.k_panel >> 4;
        const uint8_t* wp = wrow + kp;
        // first batch of weight vectors goes in flight BEFORE x is staged, so the prologue
        // (x load + decode + barrier) overlaps the first HBM round trip
        uint4 cur[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int vv = lane + 32 * u;
            cur[u] = (row_ok && vv < nvec) ? ldg_w_v4(wp + (size_t)vv * 16) : make_uint4(0u, 0u, 0u, 0u);
        }
        if (need_wait) { pdl_wait(); need_wait = false; }
        if (kp != k_begin) __syncthreads();
        // stage x[:, kp : kp+len] as fp16 (raw hardware decode; NaN bytes stay NaN on purpose)
        for (int i = threadIdx.x; i < MT * nvec; i += kGemvThreads) {
            const int m = i / nvec, v = i - m * nvec;
            uint4 xb;
            if (XQ) {
                const size_t base = (size_t)m * K + kp + (size_t)v * 16;
                const float sc = xq_scale[m];
                float f[16];
                xq_load16(xp.X, xp.x_dtype, base, f);
#pragma unroll
                for (int j = 0; j < 16; ++j) f[j] = __fmul_rn(f[j], sc);                                    // native.py:179
                xb.x = enc4_f32(f[0], f[1], f[2], f[3]);
                xb.y = enc4_f32(f[4], f[5], f[6], f[7]);
                xb.z = enc4_f32(f[8], f[9], f[10], f[11]);
                xb.w = enc4_f32(f[12], f[13], f[14], f[15]);
            } else {
                xb = ld_x_v4(p.A + (size_t)m * K + kp + (size_t)v * 16);
            }
            uint4 lo, hi;
            dec4_f16x2_raw(xb.x, lo.x, lo.y);
            dec4_f16x2_raw(xb.y, lo.z, lo.w);
            dec4_f16x2_raw(xb.z, hi.x, hi.y);
            dec4_f16x2_raw(xb.w, hi.z, hi.w);
            xs[(m * 2 + 0) * nvec_panel + v] = lo;
            xs[(m * 2 + 1) * nvec_panel + v] = hi;
        }
        __syncthreads();
        if (row_ok) {
            for (int v = lane; v < nvec; v += 32 * U) {
                uint4 nxt[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {                       // next batch in flight while this one is consumed
                    const int vv = v + 32 * (U + u);
                    nxt[u] = vv < nvec ? ldg_w_v4(wp + (size_t)vv * 16) : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int vv = v + 32 * u;
                    if (vv < nvec) gemv_consume<MT>(cur[u], xs, nvec_panel, vv, acc0, acc1);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) cur[u] = nxt[u];
            }
        }
    }

    if (need_wait) pdl_wait();                       // empty K range: still order the stores below
    float s[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        float t = acc0[m] + acc1[m];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, o);
        s[m] = t;
    }

    const int S = gridDim.y;
    if (S == 1) {
        if (row_ok && lane < MT) {
            float v = 0.0f;
#pragma unroll
            for (int m = 0; m < MT; ++m) if (lane == m) v = s[m];
            const int gm = p.m0 + lane;
            if (XQ) {
                if (v != v) v = slow_dot_masked_xq(xp.X, xp.x_dtype, (size_t)lane * K, xq_scale[lane], wrow, K);
                epi_store(p.epi, gm, row, epi_apply_sa(p.epi, v, xq_inv[lane], row));
            } else {
                if (v != v) v = slow_dot_masked(p.A + (size_t)lane * K, wrow, K);
                epi_store(p.epi, gm, row, epi_apply(p.epi, v, gm, row));
            }
        }
        return;
    }

    // split-K: reduce the S partial sums through distributed shared memory, in rank order
    cg::cluster_group cluster = cg::this_cluster();
    if (lane == 0) {
#pragma unroll
        for (int m = 0; m < MT; ++m) part[warp][m] = s[m];
    }
    cluster.sync();
    if (cluster.block_rank() == 0 && row_ok && lane < MT) {
        float v = 0.0f;
        for (int r = 0; r < S; ++r) {
            const float* rp = cluster.map_shared_rank(&part[0][0], r);
            v += rp[warp * kGemvMaxMT + lane];
        }
        const int gm = p.m0 + lane;
        if (XQ) {
            if (v != v) v = slow_dot_masked_xq(xp.X, xp.x_dtype, (size_t)lane * K, xq_scale[lane], wrow, K);
            epi_store(p.epi, gm, row, epi_apply_sa(p.epi, v, xq_inv[lane], row));
        } else {
            if (v != v) v = slow_dot_masked(p.A + (size_t)lane * K, wrow, K);
            epi_store(p.epi, gm, row, epi_apply(p.epi, v, gm, row));
        }
    }
    cluster.sync();
}

// Any K / any alignment: byte loads, masked scalar decode, fp32 FMA.  Correct, not fast.
__global__ void __launch_bounds__(kGemvThreads)
fp8_gemv_generic_kernel(const uint8_t* __restrict__ A, const uint8_t* __restrict__ B, int M, int N, int K, const Epi epi,
                        int a_fmt, int b_fmt)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * kGemvWarps + warp;
    if (row >= N) return;
    const uint8_t* wrow = B + (size_t)row * K;
    for (int m = 0; m < M; ++m) {
        const uint8_t* x = A + (size_t)m * K;
        float acc = 0.0f;
        for (int k = lane; k < K; k += 32) acc = __fmaf_rn(dec1_fmt_f32(x[k], a_fmt), dec1_fmt_f32(wrow[k], b_fmt), acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
        if (lane == 0) epi_store(epi, m, row, epi_apply(epi, acc, m, row));
    }
}

bool gemv_supported(const MMArgs& a) { return a.M >= 1 && a.M <= 16; }

template <int MT, int U>
static int launch_gemv_mt(const GemvParams& p, int S, size_t smem, cudaStream_t st)
{
    static std::atomic<int> attr_done[64];
    if (int rc = ensure_max_smem(fp8_gemv_kernel<MT, U>, kGemvMaxSmem, attr_done)) return rc;
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;   // always: resident while the predecessor drains
    return launch_ex(fp8_gemv_kernel<MT, U>, dim3((p.N + kGemvWarps - 1) / kGemvWarps, S, 1), dim3(kGemvThreads, 1, 1),
                     smem, st, 1, S, pdl, p);
}

template <int MT, int U>
static int launch_gemv_xq_mt(const GemvXqParams& xp, int S, size_t smem, cudaStream_t st)
{
    static std::atomic<int> attr_done[64];
    if (int rc = ensure_max_smem(fp8_gemv_xq_kernel<MT, U>, kGemvMaxSmem, attr_done)) return rc;
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;
    return launch_ex(fp8_gemv_xq_kernel<MT, U>, dim3((xp.g.N + kGemvWarps - 1) / kGemvWarps, S, 1), dim3(kGemvThreads, 1, 1),
                     smem, st, 1, S, pdl, xp);
}

int launch_gemv_fhfma(const MMArgs& a, const Epi& epi, const void* X, int x_dtype, float* inv_scale_out);

int launch_gemv(const MMArgs& a)
{
    if (!gemv_supported(a)) return FP8B_ERR_UNSUPPORTED;
    // kernel choice: M == 1 -> CUDA-core FHFMA kernel (exact fp32 accumulation order per lane);
    // M >= 2 -> warp-level tensor-core kernel (weights streamed once for all M rows).
    // FP8B_GEMV_IMPL=1 / 2 forces the first / second (profiling knob); any other value takes this rule.
    const int impl = tune(kTuneGemvImpl, 0);
    if (a.a_fmt | a.b_fmt) {        // an e5m2 operand: the warp-MMA kernel has all four type pairs; else the generic kernel
        if (gemv_mma_supported(a)) return launch_gemv_mma(a);
        fp8_gemv_generic_kernel<<<(a.N + kGemvWarps - 1) / kGemvWarps, kGemvThreads, 0, a.st>>>(a.A, a.B, a.M, a.N, a.K, make_epi(a),
                                                                                             a.a_fmt, a.b_fmt);
        return after_launch();
    }
    if (gemv_mma_supported(a) && (impl == 2 || (impl != 1 && a.M >= 2))) return launch_gemv_mma(a);
    const Epi epi = make_epi(a);
    const bool fast = (a.K % 16 == 0) && a.K >= 16 && aligned(a.A, 16) && aligned(a.B, 16);
    if (!fast) {
        fp8_gemv_generic_kernel<<<(a.N + kGemvWarps - 1) / kGemvWarps, kGemvThreads, 0, a.st>>>(a.A, a.B, a.M, a.N, a.K, epi, 0, 0);
        return after_launch();
    }
    return launch_gemv_fhfma(a, epi, nullptr, 0, nullptr);
}

// Shared launch planning for the FHFMA kernel: A = fp8 bytes (X == nullptr) or X = un-quantised activations.
int launch_gemv_fhfma(const MMArgs& a, const Epi& epi, const void* X, int x_dtype, float* inv_scale_out)
{
    const DeviceInfo& di = device_info();
    const int row_blocks = (a.N + kGemvWarps - 1) / kGemvWarps;
    const size_t x_esz = X ? dtype_size(x_dtype) : 1;
    for (int m0 = 0; m0 < a.M; m0 += kGemvMaxMT) {
        const int mt = a.M - m0 < kGemvMaxMT ? a.M - m0 : kGemvMaxMT;
        // split K over a cluster until the grid covers the GPU about twice (each CTA keeps >= 2 KB of K)
        int S = 1;
        while (S < kGemvMaxSplit && row_blocks * S < 2 * di.sm_count && a.K / (S * 2) >= 2048) S *= 2;
        int kps = ((a.K + S - 1) / S + 15) & ~15;
        // shrink S if the rounding left trailing ranks without work
        while (S > 1 && (size_t)kps * (S - 1) >= (size_t)a.K) { S /= 2; kps = ((a.K + S - 1) / S + 15) & ~15; }
        int panel = kps;
        const int max_panel = (kGemvMaxSmem / (2 * mt)) & ~15;
        if (panel > max_panel) panel = max_panel;
        GemvParams p;
        p.A = X ? nullptr : a.A + (size_t)m0 * a.K; p.B = a.B; p.m0 = m0; p.N = a.N; p.K = a.K;
        p.k_per_split = kps; p.k_panel = panel; p.epi = epi;
        p.static_b = (g_opt_pdl.load(std::memory_order_relaxed) && (a.chain_pdl || g_opt_static_weights.load(std::memory_order_relaxed))) ? 1 : 0;
        const size_t smem = (size_t)mt * panel * 2;
        int rc;
        if (X) {
            GemvXqParams xp;
            xp.g = p;
            xp.X = static_cast<const uint8_t*>(X) + (size_t)m0 * a.K * x_esz;
            xp.x_dtype = x_dtype;
            xp.inv_scale_out = inv_scale_out ? inv_scale_out + m0 : nullptr;
            switch (mt) {
                case 1: rc = launch_gemv_xq_mt<1, 4>(xp, S, smem, a.st); break;
                case 2: rc = launch_gemv_xq_mt<2, 4>(xp, S, smem, a.st); break;
                case 3: rc = launch_gemv_xq_mt<3, 4>(xp, S, smem, a.st); break;
                default: rc = launch_gemv_xq_mt<4, 4>(xp, S, smem, a.st); break;
            }
        } else {
            const int unroll = tune(kTuneGemvUnroll, 4);
            switch (mt) {
                case 1: rc = unroll == 2 ? launch_gemv_mt<1, 2>(p, S, smem, a.st)
                           : unroll == 8 ? launch_gemv_mt<1, 8>(p, S, smem, a.st) : launch_gemv_mt<1, 4>(p, S, smem, a.st); break;
                case 2: rc = launch_gemv_mt<2, 4>(p, S, smem, a.st); break;
                case 3: rc = launch_gemv_mt<3, 4>(p, S, smem, a.st); break;
                default: rc = launch_gemv_mt<4, 4>(p, S, smem, a.st); break;
            }
        }
        if (rc != FP8B_OK) return rc;
    }
    return FP8B_OK;
}

}  // namespace fp8b
