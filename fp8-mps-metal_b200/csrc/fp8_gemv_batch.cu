// Several independent M = 1 GEMVs in ONE launch:  y_i[n] = epi_i( sum_k dec(x_i[k]) * dec(W_i[n,k]) ),  i < count.
//
// No counterpart in the reference, where every projection of a decode step is its own fp8_scaled_vecmat_kernel
// dispatch (fp8_mps_native.py:78-86).  On a B200 a C2-sized GEMV is at the single-launch floor: about 4.3 us of
// its 11.9 us is ramp-up and drain (profiles/tools/membw.cu).  The projections of one layer that share their
// input (Q/K/V, gate/up) are independent, so they can share one launch and pay that once: the grid is the
// concatenation of the problems' 8-row blocks, the problem table travels in the kernel parameters.
//
// The arithmetic per output is that of fp8_gemv_kernel<1, 4> (fp8_gemv.cu): x decoded once per CTA into shared
// memory as fp16, weights streamed with 16-byte coherent loads, decoded in registers, exact fp16 products
// accumulated in fp32 (FHFMA), lane sums by warp shuffle, NaN accumulators recomputed with the masked scalar
// loop, fused scale / bias / output cast.  The helpers below are copies of the ones in fp8_gemv.cu on purpose:
// that file's kernel is tuned to its exact instruction schedule and is not touched for this addition.
#include "fp8_mm.cuh"

namespace fp8b {

constexpr int kGbThreads = 256;
constexpr int kGbWarps = kGbThreads / 32;
constexpr int kGbMaxItems = 16;
constexpr int kGbMaxSmem = 96 * 1024;
constexpr int kGbUnroll = 4;

struct GemvBatchParams {
    int count, K, out_dtype, bias_dtype;
    int block_end[kGbMaxItems];              // running total of 8-row blocks up to and including item i
    int N[kGbMaxItems];
    int sb_stride[kGbMaxItems];
    const uint8_t* x[kGbMaxItems];
    const uint8_t* W[kGbMaxItems];
    void* y[kGbMaxItems];
    const float* sx[kGbMaxItems];
    const float* sw[kGbMaxItems];
    const void* bias[kGbMaxItems];
};

__device__ __forceinline__ uint4 gb_ldg_w(const uint8_t* p) {
    uint4 r;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 gb_ld_x(const uint8_t* p) {
    uint4 r;
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void gb_fhfma2(float& acc, uint32_t w2, uint32_t x2) {
    asm("{\n\t.reg .b16 a0, a1, b0, b1;\n\t"
        "mov.b32 {a0, a1}, %1;\n\tmov.b32 {b0, b1}, %2;\n\t"
        "fma.rn.f32.f16 %0, a0, b0, %0;\n\tfma.rn.f32.f16 %0, a1, b1, %0;\n\t}"
        : "+f"(acc) : "r"(w2), "r"(x2));
}
__device__ __forceinline__ void gb_consume(const uint4& w, const uint4* __restrict__ xs, int nvec, int v, float& acc0, float& acc1)
{
    uint32_t w0l, w0h, w1l, w1h, w2l, w2h, w3l, w3h;
    dec4_f16x2_raw(w.x, w0l, w0h);
    dec4_f16x2_raw(w.y, w1l, w1h);
    dec4_f16x2_raw(w.z, w2l, w2h);
    dec4_f16x2_raw(w.w, w3l, w3h);
    const uint4 xa = xs[v];                  // elements 0..7 of the vector
    const uint4 xb = xs[nvec + v];           // elements 8..15
    gb_fhfma2(acc0, w0l, xa.x); gb_fhfma2(acc1, w0h, xa.y);
    gb_fhfma2(acc0, w1l, xa.z); gb_fhfma2(acc1, w1h, xa.w);
    gb_fhfma2(acc0, w2l, xb.x); gb_fhfma2(acc1, w2h, xb.y);
    gb_fhfma2(acc0, w3l, xb.z); gb_fhfma2(acc1, w3h, xb.w);
}

__global__ void __launch_bounds__(kGbThreads)
fp8_gemv_batch_kernel(const __grid_constant__ GemvBatchParams p)
{
    extern __shared__ __align__(16) uint8_t gb_smem[];
    uint4* xs = reinterpret_cast<uint4*>(gb_smem);
    constexpr int U = kGbUnroll;

    int it = 0;
    while ((int)blockIdx.x >= p.block_end[it]) ++it;          // host guarantees blockIdx.x < block_end[count - 1]
    const int first_block = it ? p.block_end[it - 1] : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int N = p.N[it], K = p.K;
    const int row = ((int)blockIdx.x - first_block) * kGbWarps + warp;
    const bool row_ok = row < N;
    const uint8_t* x = p.x[it];
    const uint8_t* wrow = p.W[it] + (size_t)(row_ok ? row : 0) * K;
    const int nvec = K >> 4;

    pdl_launch_dependents();
    pdl_wait();                                               // nothing global is read before this

    uint4 cur[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {                             // first weight batch in flight while x is staged
        const int vv = lane + 32 * u;
        cur[u] = (row_ok && vv < nvec) ? gb_ldg_w(wrow + (size_t)vv * 16) : make_uint4(0u, 0u, 0u, 0u);
    }
    for (int v = threadIdx.x; v < nvec; v += kGbThreads) {    // x as fp16 (raw decode: NaN bytes stay NaN on purpose)
        const uint4 xb = gb_ld_x(x + (size_t)v * 16);
        uint4 lo, hi;
        dec4_f16x2_raw(xb.x, lo.x, lo.y);
        dec4_f16x2_raw(xb.y, lo.z, lo.w);
        dec4_f16x2_raw(xb.z, hi.x, hi.y);
        dec4_f16x2_raw(xb.w, hi.z, hi.w);
        xs[v] = lo;
        xs[nvec + v] = hi;
    }
    __syncthreads();

    float acc0 = 0.0f, acc1 = 0.0f;
    if (row_ok) {
        for (int v = lane; v < nvec; v += 32 * U) {
            uint4 nxt[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {                     // next batch in flight while this one is consumed
                const int vv = v + 32 * (U + u);
                nxt[u] = vv < nvec ? gb_ldg_w(wrow + (size_t)vv * 16) : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int vv = v + 32 * u;
                if (vv < nvec) gb_consume(cur[u], xs, nvec, vv, acc0, acc1);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) cur[u] = nxt[u];
        }
    }
    float t = acc0 + acc1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, o);

    if (row_ok && lane == 0) {
        if (t != t) t = slow_dot_masked(x, wrow, K);          // a NaN byte somewhere: the reference decodes it as 0
        Epi e;
        e.sa = p.sx[it]; e.sa_stride = 0;
        e.sb = p.sw[it]; e.sb_stride = p.sb_stride[it];
        e.bias = p.bias[it]; e.bias_dtype = p.bias_dtype; e.sr = nullptr;
        e.C = p.y[it]; e.ldc = N; e.out_dtype = p.out_dtype;
        epi_store(e, 0, row, epi_apply(e, t, 0, row));
    }
}

}  // namespace fp8b

using namespace fp8b;

extern "C" int fp8b_gemv_batch(const fp8b_gemv_item* items, int count, int K, int out_dtype, int bias_dtype, void* stream)
{
    if (count < 0 || (count > 0 && !items) || K < 0) return FP8B_ERR_INVALID;
    if (!valid_out_dtype(out_dtype)) return FP8B_ERR_INVALID;
    if (count == 0) return FP8B_OK;
    bool any_bias = false;
    for (int i = 0; i < count; ++i) {
        const fp8b_gemv_item& q = items[i];
        if (q.N < 0) return FP8B_ERR_INVALID;
        if (q.N == 0) continue;
        if (!q.x || !q.W || !q.y || !q.scale_x || !q.scale_w) return FP8B_ERR_INVALID;
        if (!(q.scale_w_len == 1 || q.scale_w_len == q.N)) return FP8B_ERR_INVALID;
        any_bias = any_bias || q.bias != nullptr;
    }
    if (any_bias && (bias_dtype < FP8B_F32 || bias_dtype > FP8B_BF16)) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    if (K < 16 || (K % 16) != 0 || (size_t)K * 2 > (size_t)kGbMaxSmem) return FP8B_ERR_UNSUPPORTED;
    for (int i = 0; i < count; ++i)
        if (items[i].N > 0 && (!aligned(items[i].x, 16) || !aligned(items[i].W, 16))) return FP8B_ERR_UNSUPPORTED;

    static std::atomic<int> attr_done[64];
    if (int rc = ensure_max_smem(fp8_gemv_batch_kernel, kGbMaxSmem, attr_done)) return rc;
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;
    cudaStream_t st = (cudaStream_t)stream;

    GemvBatchParams p;
    int n = 0, blocks = 0;
    auto flush = [&]() -> int {
        if (n == 0) return FP8B_OK;
        p.count = n; p.K = K; p.out_dtype = out_dtype; p.bias_dtype = bias_dtype;
        for (int j = n; j < kGbMaxItems; ++j) {               // keep the unused slots defined
            p.block_end[j] = blocks; p.N[j] = 0; p.sb_stride[j] = 0;
            p.x[j] = nullptr; p.W[j] = nullptr; p.y[j] = nullptr; p.sx[j] = nullptr; p.sw[j] = nullptr; p.bias[j] = nullptr;
        }
        const int rc = launch_ex(fp8_gemv_batch_kernel, dim3(blocks), dim3(kGbThreads), (size_t)K * 2, st, 1, 1, pdl, p);
        n = 0; blocks = 0;
        return rc;
    };
    for (int i = 0; i < count; ++i) {
        const fp8b_gemv_item& q = items[i];
        if (q.N == 0) continue;
        if (n == kGbMaxItems) { if (int rc = flush()) return rc; }
        blocks += (q.N + kGbWarps - 1) / kGbWarps;
        p.block_end[n] = blocks; p.N[n] = q.N; p.sb_stride[n] = q.scale_w_len == 1 ? 0 : 1;
        p.x[n] = q.x; p.W[n] = q.W; p.y[n] = q.y; p.sx[n] = q.scale_x; p.sw[n] = q.scale_w; p.bias[n] = q.bias;
        ++n;
    }
    return flush();
}
