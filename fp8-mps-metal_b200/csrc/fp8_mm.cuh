// Internal interface between the C-ABI dispatcher (fp8_capi.cu) and the three matmul kernels,
// plus the fused epilogue they share.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "fp8_codec.cuh"
#include "fp8_common.cuh"

namespace fp8b {

// optional completion signal of the push kernel (fp8b_scaled_mm_push_signal)
struct PushSignal {
    uint64_t* flags[8];            // flags[d]: the word in destination d's memory to set (null for this rank itself)
    unsigned int* cta_counter;     // local device counter, zero between launches
    uint64_t epoch;
};

// Where the tcgen05 GEMM stores the tile; every other kernel stores to C only (Local).
enum class Store {
    Local,        // C
    Multicast,    // C is an NVSwitch multicast address (multimem.st)
    Peers,        // C and, at C + peer_deltas[r], every rank's buffer (st.global)
    Push          // TMA stores to the n_dst buffers dsts[]
};

struct MMArgs {
    const uint8_t* A;      // (M,K) row-major
    const uint8_t* B;      // (N,K) row-major
    void* C;               // (M,N), row stride ldc elements
    int out_dtype;
    int M, N, K;
    int64_t ldc;
    const float* sa; int sa_len;
    const float* sb; int sb_len;
    const void* bias; int bias_dtype;
    const float* sr;
    cudaStream_t st;
    int a_fmt = 0, b_fmt = 0;   // operand formats (FP8B_E4M3FN / FP8B_E5M2); host-side routing only
    Store store = Store::Local;
    int n_dst = 1;                          // Peers: world size; Push: number of destinations
    const int64_t* peer_deltas = nullptr;   // Peers: DEVICE table of n_dst byte offsets from C (0 for this rank)
    void* const* dsts = nullptr;            // Push: HOST array of n_dst destination buffers
    const PushSignal* sig = nullptr;   // push kernel only
    int chain_pdl = 0;     // GEMV only: the predecessor on the stream is our own quantise kernel (never writes B),
                           // so launch with PDL and prefetch B before griddepcontrol.wait
};

bool gemv_supported(const MMArgs& a);
bool tcgen05_supported(const MMArgs& a);
int launch_gemv(const MMArgs& a);
bool gemv_mma_supported(const MMArgs& a);
int launch_gemv_mma(const MMArgs& a);
int launch_gemm_simt(const MMArgs& a);
int launch_gemm_tcgen05(const MMArgs& a);
int launch_peer_wait(const uint64_t* flags, int world, int rank, uint64_t epoch, cudaStream_t st);

// ---- fused epilogue -----------------------------------------------------------------------
// out = cast( (((acc * sa) * sb) [+ bias]) [* scale_result] ), every step a separately rounded
// fp32 operation in the reference's order (fp8_matmul.metal:146, fp8_mps_patch.py:95-104).
struct Epi {
    const float* sa; int sa_stride;     // stride 0 = per-tensor, 1 = per-row
    const float* sb; int sb_stride;
    const void* bias; int bias_dtype;
    const float* sr;
    void* C; int64_t ldc; int out_dtype;
};

inline Epi make_epi(const MMArgs& a) {
    Epi e;
    e.sa = a.sa; e.sa_stride = a.sa_len == 1 ? 0 : 1;
    e.sb = a.sb; e.sb_stride = a.sb_len == 1 ? 0 : 1;
    e.bias = a.bias; e.bias_dtype = a.bias_dtype; e.sr = a.sr;
    e.C = a.C; e.ldc = a.ldc; e.out_dtype = a.out_dtype;
    return e;
}

// FHFMA GEMV planner shared by the pre-quantised path (X == nullptr) and the fused dynamic-quantise path.
int launch_gemv_fhfma(const MMArgs& a, const Epi& epi, const void* X, int x_dtype, float* inv_scale_out);

// NOTE: plain loads, not __ldg(): nvcc treats ld.global.nc as speculatable and hoisted a guarded
// `__ldg(bias + n)` above its `if (bias)` check (observed in SASS; a null bias then faults).
__device__ __forceinline__ float epi_bias(const Epi& e, int n) {
    if (e.bias_dtype == FP8B_F32) return reinterpret_cast<const float*>(e.bias)[n];
    if (e.bias_dtype == FP8B_F16) return __half2float(reinterpret_cast<const __half*>(e.bias)[n]);
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(e.bias)[n]);
}

__device__ __forceinline__ float epi_apply(const Epi& e, float acc, int m, int n) {
    float v = __fmul_rn(acc, e.sa[(size_t)m * e.sa_stride]);
    v = __fmul_rn(v, e.sb[(size_t)n * e.sb_stride]);
    if (e.bias) v = __fadd_rn(v, epi_bias(e, n));
    if (e.sr) v = __fmul_rn(v, *e.sr);
    return v;
}

// same with the row scale supplied by the caller (kernels that quantise the activations themselves)
__device__ __forceinline__ float epi_apply_sa(const Epi& e, float acc, float sa, int n) {
    float v = __fmul_rn(acc, sa);
    v = __fmul_rn(v, e.sb[(size_t)n * e.sb_stride]);
    if (e.bias) v = __fadd_rn(v, epi_bias(e, n));
    if (e.sr) v = __fmul_rn(v, *e.sr);
    return v;
}

__device__ __forceinline__ void epi_store(const Epi& e, int m, int n, float v) {
    const size_t idx = (size_t)m * e.ldc + n;
    if (e.out_dtype == FP8B_F32) reinterpret_cast<float*>(e.C)[idx] = v;
    else if (e.out_dtype == FP8B_F16) reinterpret_cast<__half*>(e.C)[idx] = __float2half_rn(v);
    else if (e.out_dtype == FP8B_OUT_E4M3FN) reinterpret_cast<uint8_t*>(e.C)[idx] = enc1_f32(v);
    else reinterpret_cast<__nv_bfloat16*>(e.C)[idx] = __float2bfloat16_rn(v);
}

// Exact reference dot product for one output element, NaN bytes contributing 0
// (fp8_matmul.metal:21).  Used by the fast kernels only to repair an accumulator that the
// hardware decode turned into NaN; see "NaN-byte fix-up" in DESIGN.md.
static __device__ __noinline__ float slow_dot_masked(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, int K) {
    float s = 0.0f;
    for (int k = 0; k < K; ++k) s = __fmaf_rn(dec1_f32(a[k]), dec1_f32(b[k]), s);
    return s;
}

// Same for any operand formats: e4m3fn NaN bytes contribute 0, e5m2 inf / NaN propagate (IEEE).  With an e5m2
// operand a NaN accumulator may be the right answer; this loop then simply reproduces it.
static __device__ __noinline__ float slow_dot_fmt(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, int K,
                                                  int a_fmt, int b_fmt) {
    float s = 0.0f;
    for (int k = 0; k < K; ++k) s = __fmaf_rn(dec1_fmt_f32(a[k], a_fmt), dec1_fmt_f32(b[k], b_fmt), s);
    return s;
}

}  // namespace fp8b
