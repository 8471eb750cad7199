// Streaming cast kernels: FP8 -> {f16,bf16,f32} and {f32,f16,bf16} -> FP8, plus the on-device
// amax -> scale step of fp8_quantize.
//
// Reference: fp8_to_half_kernel (fp8_matmul.metal:215-223) and float_to_fp8_kernel (:228-236), one
// element per thread, with the scale / up-conversion / pre-scale done as separate torch passes
// on the host side (fp8_mps_native.py:121-122, :142, :170-179).  Here each is ONE pass over HBM:
// every thread-iteration moves one 16- (or 32-) byte vector on the wide side (the f16/bf16/f32 side)
// and the matching vector on the FP8 side, so both sides are fully coalesced; the work is cut into
// tiles of THREADS x UNROLL vectors (see "Tiles" below for the measured launch shapes).  HBM-bound:
// 3 B/element (16-bit side) or 5 B/element (f32 side) of algorithmic traffic.
//
// In this file: tile kernels (single tensor), batched kernels (many tensors, one launch, span table in
// the kernel parameters), the amax / finalize kernels of fp8_quantize, the row-wise quantise kernels
// (two-pass and register-resident), float8_e5m2 decode (FMT template parameter), and the C entry points.
// The tile kernels run under programmatic dependent launch: coherent loads only.
#include "fp8_codec.cuh"
#include "fp8_common.cuh"

namespace fp8b {

constexpr int kCastThreads = 256;

// Streaming loads.  Deliberately NOT .nc: the tile kernels run under programmatic dependent launch (resident before
// their predecessor has finished), and ptxas moves non-coherent loads above griddepcontrol.wait (seen in the
// GEMV kernels' SASS); a coherent load stays behind it.
__device__ __forceinline__ uint4 ldg_stream_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
// 256-bit load (sm_100: LDG.E.256).  For the read+write streams of wide -> fp8, 32-byte loads with 4 per thread
// in flight measured 6.85 TB/s against 6.0 TB/s for the same bytes in flight as 16-byte loads
// (profiles/tools/castbw.cu); 256-bit STORES made no difference for fp8 -> wide.
__device__ __forceinline__ void ldg_stream_v8(const void* p, uint4& lo, uint4& hi) {
    asm volatile("ld.global.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w) : "l"(p));
}
__device__ __forceinline__ uint2 ldg_stream_v2(const void* p) {
    uint2 r;
    asm volatile("ld.global.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream_u32(const void* p) {
    uint32_t r;
    asm volatile("ld.global.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_v4(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void stg_stream_v2(void* p, uint2 v) {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void stg_stream_u32(void* p, uint32_t v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// the optional scale / prescale scalar is typically written by the kernel just before (amax_finalize_kernel)
__device__ __forceinline__ float ld_scalar_f32(const float* p) {
    float r;
    asm volatile("ld.global.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t f16x2_to_bf16x2(uint32_t v) {
    float2 f = __half22float2(*reinterpret_cast<__half2*>(&v));
    __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);       // exact: e4m3 values fit bf16
    return *reinterpret_cast<uint32_t*>(&b);
}

// ------------------------------------------------------------------------------------------
// Tiles.  A tile is THREADS * UNROLL consecutive 16-byte vectors of the wide side (f16/bf16: 8 elements each,
// f32: 4) and the matching 8- / 4-byte vectors of the FP8 side; one CTA converts one tile per iteration, every
// thread keeping UNROLL independent loads in flight (stride THREADS vectors, so a warp touches 512 contiguous
// bytes per load).  Launch shapes are chosen on the host (cast_shape below): measured on B200, copy-like
// kernels peak with ~4096 wide vectors (64 KB) in flight per SM and LOSE bandwidth beyond that.

// How one CTA of a single-tensor launch walks its tensor: `rounds` full rounds of gridDim.x tiles (CTA b takes tile
// r * gridDim.x + b), then the remaining < gridDim.x tiles' worth of vectors is cut into gridDim.x equal
// contiguous shares (512-byte granules), so every CTA finishes at the same time instead of a third of the SMs
// idling through a last partial round.
template <int TILE>
struct TileWalk {
    size_t rounds, rem_begin, rem_end;
    __device__ __forceinline__ explicit TileWalk(size_t nvec) {
        const size_t per_round = (size_t)gridDim.x * TILE;
        rounds = nvec / per_round;
        const size_t base = rounds * per_round;
        const size_t granules = (nvec - base + 31) / 32;
        const size_t share = (granules + gridDim.x - 1) / gridDim.x * 32;      // <= TILE because nvec - base < per_round
        rem_begin = base + blockIdx.x * share;
        rem_end = rem_begin + share < nvec ? rem_begin + share : nvec;
    }
};

// FP8 -> wide.  OUT: FP8B_F16 / FP8B_BF16 / FP8B_F32.  SCALED (f16 only): fp16 multiply by RN16(scale).
template <int OUT, bool SCALED, int THREADS, int UNROLL, int FMT = 0>
__device__ __forceinline__ void decode_tile(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, size_t vbegin,
                                            size_t nvec, uint32_t s2)
{
    const size_t v0 = vbegin + threadIdx.x;                    // converts vectors [vbegin, min(vbegin + tile, nvec))
    uint2 w[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const size_t v = v0 + (size_t)u * THREADS;
        if (OUT == FP8B_F32) w[u] = make_uint2(v < nvec ? ldg_stream_u32(in + v * 4) : 0u, 0u);
        else w[u] = v < nvec ? ldg_stream_v2(in + v * 8) : make_uint2(0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const size_t v = v0 + (size_t)u * THREADS;
        if (v < nvec) {
            uint4 o;
            if (OUT == FP8B_F32) {
                uint32_t lo, hi;
                dec4_fmt_f16x2<FMT>(w[u].x, lo, hi);
                const float2 a = __half22float2(*reinterpret_cast<__half2*>(&lo));
                const float2 c = __half22float2(*reinterpret_cast<__half2*>(&hi));
                o = make_uint4(__float_as_uint(a.x), __float_as_uint(a.y), __float_as_uint(c.x), __float_as_uint(c.y));
            } else {
                dec4_fmt_f16x2<FMT>(w[u].x, o.x, o.y);
                dec4_fmt_f16x2<FMT>(w[u].y, o.z, o.w);
                if (SCALED) {                                   // fp16 multiply, native.py:122
                    const __half2 sc = *reinterpret_cast<const __half2*>(&s2);
                    uint32_t* q = &o.x;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        __half2 r = __hmul2(*reinterpret_cast<__half2*>(&q[j]), sc);
                        q[j] = *reinterpret_cast<uint32_t*>(&r);
                    }
                }
                if (OUT == FP8B_BF16) {
                    o.x = f16x2_to_bf16x2(o.x); o.y = f16x2_to_bf16x2(o.y);
                    o.z = f16x2_to_bf16x2(o.z); o.w = f16x2_to_bf16x2(o.w);
                }
            }
            stg_stream_v4(out + v * 16, o);
        }
    }
}

// ragged tail (< one vector) of a tensor, one thread
template <int OUT, bool SCALED, int FMT = 0>
__device__ __forceinline__ void decode_tail(const uint8_t* in, void* out, size_t from, size_t n, const float* scale)
{
    for (size_t i = from; i < n; ++i) {
        const float f = dec1_fmt_f32(in[i], FMT);
        if (OUT == FP8B_F32) reinterpret_cast<float*>(out)[i] = f;
        else if (OUT == FP8B_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(f);
        else {
            __half h = __float2half_rn(f);
            if (SCALED) h = __hmul(h, __float2half_rn(ld_scalar_f32(scale)));
            reinterpret_cast<__half*>(out)[i] = h;
        }
    }
}

template <int OUT, bool SCALED, int THREADS, int UNROLL, int FMT = 0>
__global__ void __launch_bounds__(THREADS)
fp8_to_wide_kernel(const uint8_t* __restrict__ in, void* __restrict__ out, size_t n,
                   const float* __restrict__ scale)
{
    constexpr int EPV = (OUT == FP8B_F32) ? 4 : 8;            // elements per 16-byte vector
    const size_t nvec = n / EPV;
    pdl_launch_dependents();          // resident early, idle until the predecessor has completed and flushed
    pdl_wait();
    uint32_t s2 = 0;
    if (SCALED) {
        __half2 s = __float2half2_rn(ld_scalar_f32(scale));   // RN16(scale), native.py:121
        s2 = *reinterpret_cast<uint32_t*>(&s);
    }
    uint8_t* o8 = reinterpret_cast<uint8_t*>(out);
    TileWalk<THREADS * UNROLL> walk(nvec);
    for (size_t r = 0; r < walk.rounds; ++r)
        decode_tile<OUT, SCALED, THREADS, UNROLL, FMT>(in, o8, (r * gridDim.x + blockIdx.x) * (size_t)(THREADS * UNROLL), nvec, s2);
    if (walk.rem_begin < walk.rem_end) decode_tile<OUT, SCALED, THREADS, UNROLL, FMT>(in, o8, walk.rem_begin, walk.rem_end, s2);
    if (blockIdx.x == 0 && threadIdx.x == 0) decode_tail<OUT, SCALED, FMT>(in, out, nvec * EPV, n, scale);
}

template <int OUT, bool SCALED, int FMT = 0>
__global__ void __launch_bounds__(kCastThreads)
fp8_to_wide_scalar_kernel(const uint8_t* __restrict__ in, void* __restrict__ out, size_t n,
                          const float* __restrict__ scale)
{
    const size_t stride = (size_t)gridDim.x * kCastThreads;
    for (size_t i = (size_t)blockIdx.x * kCastThreads + threadIdx.x; i < n; i += stride) {
        float f = dec1_fmt_f32(in[i], FMT);
        if (OUT == FP8B_F32) reinterpret_cast<float*>(out)[i] = f;
        else if (OUT == FP8B_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(f);
        else {
            __half h = __float2half_rn(f);
            if (SCALED) h = __hmul(h, __float2half_rn(__ldg(scale)));
            reinterpret_cast<__half*>(out)[i] = h;
        }
    }
}

// ------------------------------------------------------------------------------------------
// wide -> FP8.  IN: f32 (16-byte load = 4 elements, 4-byte store) or f16/bf16 (8 elements, 8-byte
// store).  PRESCALE: out = enc(f32(in) * prescale[0]) with the multiply in fp32 (native.py:179).
template <int IN, bool PRESCALE>
__device__ __forceinline__ void encode_vec(const uint4& w, float s, uint32_t& o0, uint32_t& o1) {
    if (IN == FP8B_F32) {
        float a = __uint_as_float(w.x), b = __uint_as_float(w.y), c = __uint_as_float(w.z), d = __uint_as_float(w.w);
        if (PRESCALE) { a = __fmul_rn(a, s); b = __fmul_rn(b, s); c = __fmul_rn(c, s); d = __fmul_rn(d, s); }
        o0 = enc4_f32(a, b, c, d);
        o1 = 0;
    } else if (PRESCALE) {
        const uint32_t* p = &w.x;
        float f[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (IN == FP8B_F16) {
                float2 t = __half22float2(*reinterpret_cast<const __half2*>(&p[j]));
                f[2 * j] = t.x; f[2 * j + 1] = t.y;
            } else {
                f[2 * j] = __uint_as_float(p[j] << 16); f[2 * j + 1] = __uint_as_float(p[j] & 0xFFFF0000u);
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = __fmul_rn(f[j], s);
        o0 = enc4_f32(f[0], f[1], f[2], f[3]);
        o1 = enc4_f32(f[4], f[5], f[6], f[7]);
    } else if (IN == FP8B_F16) {
        o0 = (uint32_t)enc2_f16x2(w.x) | ((uint32_t)enc2_f16x2(w.y) << 16);
        o1 = (uint32_t)enc2_f16x2(w.z) | ((uint32_t)enc2_f16x2(w.w) << 16);
    } else {
        o0 = (uint32_t)enc2_bf16x2(w.x) | ((uint32_t)enc2_bf16x2(w.y) << 16);
        o1 = (uint32_t)enc2_bf16x2(w.z) | ((uint32_t)enc2_bf16x2(w.w) << 16);
    }
}

template <int IN>
__device__ __forceinline__ float load_wide_scalar(const void* in, size_t i) {
    if (IN == FP8B_F32) return reinterpret_cast<const float*>(in)[i];
    if (IN == FP8B_F16) return __half2float(reinterpret_cast<const __half*>(in)[i]);
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(in)[i]);
}

// VB = bytes per wide-side vector: 16 (any 16-byte aligned tensor) or 32 (256-bit loads, 32-byte aligned tensors).
template <int IN, bool PRESCALE, int THREADS, int UNROLL, int VB = 16>
__device__ __forceinline__ void encode_tile(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, size_t vbegin,
                                            size_t nvec, float s)
{
    const size_t v0 = vbegin + threadIdx.x;                    // converts vectors [vbegin, min(vbegin + tile, nvec))
    if (VB == 16) {
        uint4 w[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const size_t v = v0 + (size_t)u * THREADS;
            w[u] = v < nvec ? ldg_stream_v4(in + v * 16) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const size_t v = v0 + (size_t)u * THREADS;
            if (v < nvec) {
                uint32_t o0, o1;
                encode_vec<IN, PRESCALE>(w[u], s, o0, o1);
                if (IN == FP8B_F32) stg_stream_u32(out + v * 4, o0);
                else stg_stream_v2(out + v * 8, make_uint2(o0, o1));
            }
        }
    } else {
        uint4 lo[UNROLL], hi[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const size_t v = v0 + (size_t)u * THREADS;
            lo[u] = hi[u] = make_uint4(0, 0, 0, 0);
            if (v < nvec) ldg_stream_v8(in + v * 32, lo[u], hi[u]);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const size_t v = v0 + (size_t)u * THREADS;
            if (v < nvec) {
                uint32_t o0, o1, o2, o3;
                encode_vec<IN, PRESCALE>(lo[u], s, o0, o1);
                encode_vec<IN, PRESCALE>(hi[u], s, o2, o3);
                if (IN == FP8B_F32) stg_stream_v2(out + v * 8, make_uint2(o0, o2));
                else stg_stream_v4(out + v * 16, make_uint4(o0, o1, o2, o3));
            }
        }
    }
}

template <int IN, bool PRESCALE, int THREADS, int UNROLL, int VB = 16>
__global__ void __launch_bounds__(THREADS)
wide_to_fp8_kernel(const void* __restrict__ in, uint8_t* __restrict__ out, size_t n,
                   const float* __restrict__ prescale)
{
    constexpr int EPV = ((IN == FP8B_F32) ? 4 : 8) * (VB / 16);
    const size_t nvec = n / EPV;
    pdl_launch_dependents();
    pdl_wait();
    const float s = PRESCALE ? ld_scalar_f32(prescale) : 1.0f;
    const uint8_t* i8 = reinterpret_cast<const uint8_t*>(in);
    TileWalk<THREADS * UNROLL> walk(nvec);
    for (size_t r = 0; r < walk.rounds; ++r)
        encode_tile<IN, PRESCALE, THREADS, UNROLL, VB>(i8, out, (r * gridDim.x + blockIdx.x) * (size_t)(THREADS * UNROLL), nvec, s);
    if (walk.rem_begin < walk.rem_end) encode_tile<IN, PRESCALE, THREADS, UNROLL, VB>(i8, out, walk.rem_begin, walk.rem_end, s);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (size_t i = nvec * EPV; i < n; ++i) {
            float f = load_wide_scalar<IN>(in, i);
            if (PRESCALE) f = __fmul_rn(f, s);
            out[i] = enc1_f32(f);
        }
    }
}

template <int IN, bool PRESCALE>
__global__ void __launch_bounds__(kCastThreads)
wide_to_fp8_scalar_kernel(const void* __restrict__ in, uint8_t* __restrict__ out, size_t n,
                          const float* __restrict__ prescale)
{
    const size_t stride = (size_t)gridDim.x * kCastThreads;
    const float s = PRESCALE ? __ldg(prescale) : 1.0f;
    for (size_t i = (size_t)blockIdx.x * kCastThreads + threadIdx.x; i < n; i += stride) {
        float f = load_wide_scalar<IN>(in, i);
        if (PRESCALE) f = __fmul_rn(f, s);
        out[i] = enc1_f32(f);
    }
}

// ------------------------------------------------------------------------------------------
// amax over |f32(in)| -> atomicMax on the float bit pattern (non-negative floats order like
// unsigned ints; NaN bit patterns sort above inf, so a NaN input yields a NaN amax exactly like
// torch's abs().max(), fp8_mps_native.py:174).
template <int IN>
__global__ void __launch_bounds__(kCastThreads)
amax_kernel(const void* __restrict__ in, size_t n, uint32_t* __restrict__ amax_bits)
{
    constexpr int EPV = (IN == FP8B_F32) ? 4 : 8;
    const size_t nvec = n / EPV;
    constexpr int UNROLL = 4;                                  // independent 16-byte loads in flight per thread
    const size_t stride = (size_t)gridDim.x * kCastThreads;
    uint32_t m = 0;
    for (size_t v0 = (size_t)blockIdx.x * kCastThreads + threadIdx.x; v0 < nvec; v0 += stride * UNROLL) {
        uint4 w[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const size_t v = v0 + (size_t)u * stride;
            w[u] = v < nvec ? ldg_stream_v4(reinterpret_cast<const uint8_t*>(in) + v * 16) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint32_t* p = &w[u].x;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (IN == FP8B_F32) m = max(m, p[j] & 0x7FFFFFFFu);
                else if (IN == FP8B_BF16) { m = max(m, (p[j] << 16) & 0x7FFFFFFFu); m = max(m, p[j] & 0x7FFF0000u); }
                else {
                    float2 t = __half22float2(*reinterpret_cast<const __half2*>(&p[j]));
                    m = max(m, __float_as_uint(t.x) & 0x7FFFFFFFu);
                    m = max(m, __float_as_uint(t.y) & 0x7FFFFFFFu);
                }
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (size_t i = nvec * EPV; i < n; ++i) m = max(m, __float_as_uint(load_wide_scalar<IN>(in, i)) & 0x7FFFFFFFu);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    __shared__ uint32_t sm[kCastThreads / 32];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < kCastThreads / 32 ? sm[threadIdx.x] : 0u;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
        if (threadIdx.x == 0) atomicMax(amax_bits, m);
    }
}

template <int IN>
__global__ void __launch_bounds__(kCastThreads)
amax_scalar_kernel(const void* __restrict__ in, size_t n, uint32_t* __restrict__ amax_bits)
{
    const size_t stride = (size_t)gridDim.x * kCastThreads;
    uint32_t m = 0;
    for (size_t i = (size_t)blockIdx.x * kCastThreads + threadIdx.x; i < n; i += stride)
        m = max(m, __float_as_uint(load_wide_scalar<IN>(in, i)) & 0x7FFFFFFFu);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(amax_bits, m);
}

// scale = 448.0/amax in double, as the reference's Python does (fp8_mps_native.py:175-176,:189);
// resets the scratch word for the next call.
__global__ void amax_finalize_kernel(uint32_t* amax_bits, float* scale_out, float* inv_scale_out)
{
    float amax = __uint_as_float(*amax_bits);
    double scale = (amax > 0.0f) ? 448.0 / (double)amax : 1.0;
    if (scale_out) *scale_out = (float)scale;
    if (inv_scale_out) *inv_scale_out = (float)(1.0 / scale);
    *amax_bits = 0u;
}

// ------------------------------------------------------------------------------------------
// Row-wise (per-channel) quantise: fp8_quantize (fp8_mps_native.py:158-190) applied to every row of a
// (rows, cols) matrix in ONE launch -- amax, double-precision scale and fused multiply+encode per row --
// producing the per-row inverse scales that `_scaled_mm` takes as a length-M / length-N scale.
// One CTA per row; the second pass re-reads the row from L2.
template <int IN>
__global__ void __launch_bounds__(kCastThreads)
quantize_rows_kernel(const void* __restrict__ in, uint8_t* __restrict__ out, float* __restrict__ inv_scale,
                     size_t cols, int vec_ok)
{
    constexpr int EPV = (IN == FP8B_F32) ? 4 : 8;
    constexpr int ESZ = (IN == FP8B_F32) ? 4 : 2;
    pdl_launch_dependents();             // fp8b_linear_dynamic chains a GEMV behind this kernel (it waits before reading out)
    const size_t row = blockIdx.x;
    const uint8_t* rin = reinterpret_cast<const uint8_t*>(in) + row * cols * ESZ;
    uint8_t* rout = out + row * cols;
    const size_t nvec = vec_ok ? cols / EPV : 0;
    uint32_t m = 0;
    for (size_t v = threadIdx.x; v < nvec; v += kCastThreads) {
        const uint4 w = *reinterpret_cast<const uint4*>(rin + v * 16);
        const uint32_t* p = &w.x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (IN == FP8B_F32) m = max(m, p[j] & 0x7FFFFFFFu);
            else if (IN == FP8B_BF16) { m = max(m, (p[j] << 16) & 0x7FFFFFFFu); m = max(m, p[j] & 0x7FFF0000u); }
            else {
                float2 t = __half22float2(*reinterpret_cast<const __half2*>(&p[j]));
                m = max(m, __float_as_uint(t.x) & 0x7FFFFFFFu);
                m = max(m, __float_as_uint(t.y) & 0x7FFFFFFFu);
            }
        }
    }
    for (size_t i = nvec * EPV + threadIdx.x; i < cols; i += kCastThreads)
        m = max(m, __float_as_uint(load_wide_scalar<IN>(rin, i)) & 0x7FFFFFFFu);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    __shared__ uint32_t sm[kCastThreads / 32];
    __shared__ float s_scale;
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t mm = 0;
        for (int i = 0; i < kCastThreads / 32; ++i) mm = max(mm, sm[i]);
        const float amax = __uint_as_float(mm);
        const double scale = (amax > 0.0f) ? 448.0 / (double)amax : 1.0;     // native.py:175-176, in double
        s_scale = (float)scale;
        inv_scale[row] = (float)(1.0 / scale);                                 // native.py:189
    }
    __syncthreads();
    const float s = s_scale;
    for (size_t v = threadIdx.x; v < nvec; v += kCastThreads) {
        const uint4 w = *reinterpret_cast<const uint4*>(rin + v * 16);
        uint32_t o0, o1;
        encode_vec<IN, true>(w, s, o0, o1);
        if (IN == FP8B_F32) *reinterpret_cast<uint32_t*>(rout + v * 4) = o0;
        else *reinterpret_cast<uint2*>(rout + v * 8) = make_uint2(o0, o1);
    }
    for (size_t i = nvec * EPV + threadIdx.x; i < cols; i += kCastThreads)
        rout[i] = enc1_f32(__fmul_rn(load_wide_scalar<IN>(rin, i), s));
}

// Register-resident variant for rows that fit in registers: TPR threads per row (32: a warp per row, 8 rows per
// CTA, no barrier at all; ... 256: a CTA per row), each thread holding V 16-byte vectors.  The row is read from HBM
// ONCE -- amax, scale and encode all work on the registers -- and every thread has V independent loads in flight.
// Same arithmetic as quantize_rows_kernel, so the bytes and scales are identical.
template <int IN, int V, int TPR>
__global__ void __launch_bounds__(kCastThreads)
quantize_rows_reg_kernel(const void* __restrict__ in, uint8_t* __restrict__ out, float* __restrict__ inv_scale,
                         int rows, int nvec)
{
    constexpr int EPV = (IN == FP8B_F32) ? 4 : 8;
    constexpr int ESZ = (IN == FP8B_F32) ? 4 : 2;
    constexpr int RPC = kCastThreads / TPR;                  // rows per CTA
    pdl_launch_dependents();
    const int t = threadIdx.x % TPR;
    const int row = blockIdx.x * RPC + threadIdx.x / TPR;
    const bool row_ok = row < rows;
    const size_t cols = (size_t)nvec * EPV;
    const uint8_t* rin = reinterpret_cast<const uint8_t*>(in) + (size_t)(row_ok ? row : 0) * cols * ESZ;
    uint4 w[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int v = t + j * TPR;
        w[j] = (row_ok && v < nvec) ? ldg_stream_v4(rin + (size_t)v * 16) : make_uint4(0, 0, 0, 0);
    }
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const uint32_t* p = &w[j].x;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (IN == FP8B_F32) m = max(m, p[i] & 0x7FFFFFFFu);
            else if (IN == FP8B_BF16) { m = max(m, (p[i] << 16) & 0x7FFFFFFFu); m = max(m, p[i] & 0x7FFF0000u); }
            else {
                float2 f = __half22float2(*reinterpret_cast<const __half2*>(&p[i]));
                m = max(m, __float_as_uint(f.x) & 0x7FFFFFFFu);
                m = max(m, __float_as_uint(f.y) & 0x7FFFFFFFu);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if (TPR > 32) {                                           // TPR / 32 warps share a row: combine them
        constexpr int WPR = TPR / 32;
        __shared__ uint32_t sm[kCastThreads / 32];
        if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
        __syncthreads();
        const int w0 = (threadIdx.x / TPR) * WPR;
        m = 0;
#pragma unroll
        for (int i = 0; i < WPR; ++i) m = max(m, sm[w0 + i]);
    }
    float s = 1.0f;
    if ((threadIdx.x & 31) == 0) {                            // one double division per warp, broadcast below
        const float amax = __uint_as_float(m);
        const double scale = (amax > 0.0f) ? 448.0 / (double)amax : 1.0;     // native.py:175-176, in double
        s = (float)scale;
        if (row_ok && t == 0) inv_scale[row] = (float)(1.0 / scale);          // native.py:189
    }
    s = __shfl_sync(0xFFFFFFFFu, s, 0);
    uint8_t* rout = out + (size_t)(row_ok ? row : 0) * cols;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int v = t + j * TPR;
        if (row_ok && v < nvec) {
            uint32_t o0, o1;
            encode_vec<IN, true>(w[j], s, o0, o1);
            if (IN == FP8B_F32) *reinterpret_cast<uint32_t*>(rout + (size_t)v * 4) = o0;
            else *reinterpret_cast<uint2*>(rout + (size_t)v * 8) = make_uint2(o0, o1);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Batched casts: MANY tensors in ONE launch (a whole checkpoint's weights; the reference converts them one
// .to() at a time, fp8_mps_patch.py:143-230).  A per-tensor launch pays ~3 us of ramp + drain on a ~18 us
// tensor; here the tensors are cut into tiles (see "Tiles" above) and one persistent grid walks
// the concatenated tile list, so HBM stays saturated across tensor boundaries.  The span table travels in
// the kernel parameters (constant bank): no device-side descriptor buffer, no host->device copy.
constexpr int kBatchMaxSpans = 512;

struct CastBatch {
    int count;
    uint32_t tile_end[kBatchMaxSpans];      // running total of tiles up to and including span i
    const void* in[kBatchMaxSpans];
    void* out[kBatchMaxSpans];
    size_t n[kBatchMaxSpans];
};

template <int IN, int THREADS, int UNROLL, int VB = 16>
__global__ void __launch_bounds__(THREADS)
wide_to_fp8_batch_kernel(const __grid_constant__ CastBatch b)
{
    pdl_launch_dependents();
    pdl_wait();
    constexpr int EPV = ((IN == FP8B_F32) ? 4 : 8) * (VB / 16);
    const uint32_t total = b.tile_end[b.count - 1];
    int span = 0;
    for (uint32_t t = blockIdx.x; t < total; t += gridDim.x) {
        while (t >= b.tile_end[span]) ++span;                 // tiles are visited in increasing order
        const uint32_t t0 = span ? b.tile_end[span - 1] : 0u;
        const size_t n = b.n[span];
        const uint8_t* in = reinterpret_cast<const uint8_t*>(b.in[span]);
        uint8_t* out = reinterpret_cast<uint8_t*>(b.out[span]);
        encode_tile<IN, false, THREADS, UNROLL, VB>(in, out, (size_t)(t - t0) * (THREADS * UNROLL), n / EPV, 1.0f);
        if (t + 1 == b.tile_end[span] && threadIdx.x == 0)    // ragged tail of this tensor (< EPV elements)
            for (size_t i = n / EPV * EPV; i < n; ++i) out[i] = enc1_f32(load_wide_scalar<IN>(in, i));
    }
}

template <int OUT, int THREADS, int UNROLL>
__global__ void __launch_bounds__(THREADS)
fp8_to_wide_batch_kernel(const __grid_constant__ CastBatch b)
{
    pdl_launch_dependents();
    pdl_wait();
    constexpr int EPV = (OUT == FP8B_F32) ? 4 : 8;
    const uint32_t total = b.tile_end[b.count - 1];
    int span = 0;
    for (uint32_t t = blockIdx.x; t < total; t += gridDim.x) {
        while (t >= b.tile_end[span]) ++span;
        const uint32_t t0 = span ? b.tile_end[span - 1] : 0u;
        const size_t n = b.n[span];
        const uint8_t* in = reinterpret_cast<const uint8_t*>(b.in[span]);
        uint8_t* out = reinterpret_cast<uint8_t*>(b.out[span]);
        decode_tile<OUT, false, THREADS, UNROLL>(in, out, (size_t)(t - t0) * (THREADS * UNROLL), n / EPV, 0u);
        if (t + 1 == b.tile_end[span] && threadIdx.x == 0) decode_tail<OUT, false>(in, out, n / EPV * EPV, n, nullptr);
    }
}

// Launch shape for `nvec` wide-side vectors.  Measured on B200 (profiles/tools/cast_exp.py, 12.9 GB per sweep):
// bandwidth peaks at ~4096 vectors in flight per SM -- wide->fp8 with one 1024-thread CTA x 4 loads per thread
// (6.36 TB/s; 8 CTAs x 256 x 4 gives 5.7), fp8->wide with one 512-thread CTA x 8 (6.11 TB/s).  Tensors too small
// to give every SM a big tile use 256-thread x 4 tiles, at most 4 CTAs per SM (same amount in flight).
struct CastShape { int big; int grid; };
static CastShape cast_shape(size_t nvec) {
    const DeviceInfo& di = device_info();
    CastShape c;
    const int mode = tune(kTuneCastShape, 0);          // profiling knob: 1 = always small tiles, 2 = always big
    c.big = mode == 2 || (mode == 0 && nvec >= (size_t)di.sm_count * 4096);
    const size_t tile = c.big ? 4096 : 1024;
    size_t tiles = (nvec + tile - 1) / tile;
    if (tiles < 1) tiles = 1;
    const size_t cap = (size_t)di.sm_count * (c.big ? 1 : 4);
    c.grid = (int)(tiles < cap ? tiles : cap);
    return c;
}

static int cast_grid(size_t work_items) {
    const DeviceInfo& di = device_info();
    size_t want = (work_items + kCastThreads - 1) / kCastThreads;
    size_t cap = (size_t)di.sm_count * 8;                     // 8 x 256 threads = full occupancy
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

}  // namespace fp8b

using namespace fp8b;

// fp8 -> wide launch: big tiles = 512 threads x 8, small = 256 x 4
template <int OUT, bool SCALED, int FMT = 0>
static int launch_decode_vec(const uint8_t* in, void* out, size_t n, const float* scale, cudaStream_t st)
{
    constexpr int EPV = (OUT == FP8B_F32) ? 4 : 8;
    const CastShape c = cast_shape(n / EPV);
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;
#ifdef FP8B_PROFILE
    // launch-shape sweep for the write-heavy direction (profiling builds only): CAST_SHAPE 11.. = threads x unroll x CTAs/SM
    if constexpr (OUT == FP8B_F16 && !SCALED && FMT == 0) {
        const int sms = device_info().sm_count;
        switch (tune(kTuneCastShape, 0)) {
            case 11: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 256, 8, FMT>, dim3(sms * 2), dim3(256), 0, st, 1, 1, pdl, in, out, n, scale);
            case 12: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 256, 8, FMT>, dim3(sms * 4), dim3(256), 0, st, 1, 1, pdl, in, out, n, scale);
            case 13: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 512, 4, FMT>, dim3(sms * 2), dim3(512), 0, st, 1, 1, pdl, in, out, n, scale);
            case 14: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 1024, 4, FMT>, dim3(sms), dim3(1024), 0, st, 1, 1, pdl, in, out, n, scale);
            case 15: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 512, 16, FMT>, dim3(sms), dim3(512), 0, st, 1, 1, pdl, in, out, n, scale);
            case 16: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 512, 8, FMT>, dim3(sms * 2), dim3(512), 0, st, 1, 1, pdl, in, out, n, scale);
            case 17: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 256, 4, FMT>, dim3(sms * 8), dim3(256), 0, st, 1, 1, pdl, in, out, n, scale);
            case 18: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 128, 8, FMT>, dim3(sms * 8), dim3(128), 0, st, 1, 1, pdl, in, out, n, scale);
            case 19: return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 1024, 8, FMT>, dim3(sms), dim3(1024), 0, st, 1, 1, pdl, in, out, n, scale);
            default: break;
        }
    }
#endif
    if (c.big) return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 512, 8, FMT>, dim3(c.grid), dim3(512), 0, st, 1, 1, pdl, in, out, n, scale);
    return launch_ex(fp8_to_wide_kernel<OUT, SCALED, 256, 4, FMT>, dim3(c.grid), dim3(256), 0, st, 1, 1, pdl, in, out, n, scale);
}

extern "C" int fp8b_dequant_f16(const uint8_t* in, void* out, size_t n, const float* scale, void* stream)
{
    if (n == 0) return FP8B_OK;
    if (!in || !out) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    if (aligned(in, 8) && aligned(out, 16))
        return scale ? launch_decode_vec<FP8B_F16, true>(in, out, n, scale, st)
                     : launch_decode_vec<FP8B_F16, false>(in, out, n, nullptr, st);
    const int g = cast_grid(n);
    if (scale) fp8_to_wide_scalar_kernel<FP8B_F16, true><<<g, kCastThreads, 0, st>>>(in, out, n, scale);
    else fp8_to_wide_scalar_kernel<FP8B_F16, false><<<g, kCastThreads, 0, st>>>(in, out, n, nullptr);
    return after_launch();
}

extern "C" int fp8b_dequant(const uint8_t* in, void* out, int out_dtype, size_t n, void* stream)
{
    if (!valid_dtype(out_dtype)) return FP8B_ERR_INVALID;
    if (out_dtype == FP8B_F16) return fp8b_dequant_f16(in, out, n, nullptr, stream);
    if (n == 0) return FP8B_OK;
    if (!in || !out) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    if (out_dtype == FP8B_BF16) {
        if (aligned(in, 8) && aligned(out, 16)) return launch_decode_vec<FP8B_BF16, false>(in, out, n, nullptr, st);
        fp8_to_wide_scalar_kernel<FP8B_BF16, false><<<cast_grid(n), kCastThreads, 0, st>>>(in, out, n, nullptr);
    } else {
        if (aligned(in, 4) && aligned(out, 16)) return launch_decode_vec<FP8B_F32, false>(in, out, n, nullptr, st);
        fp8_to_wide_scalar_kernel<FP8B_F32, false><<<cast_grid(n), kCastThreads, 0, st>>>(in, out, n, nullptr);
    }
    return after_launch();
}

// float8_e5m2 -> wide (decode only; see fp8_codec.cuh).  scale: optional, fp16 output only, applied like fp8b_dequant_f16.
template <int OUT, bool SCALED>
static int launch_decode_e5m2(const uint8_t* in, void* out, size_t n, const float* scale, cudaStream_t st)
{
    constexpr int EPV = (OUT == FP8B_F32) ? 4 : 8;
    if (aligned(in, EPV) && aligned(out, 16)) return launch_decode_vec<OUT, SCALED, 1>(in, out, n, scale, st);
    fp8_to_wide_scalar_kernel<OUT, SCALED, 1><<<cast_grid(n), kCastThreads, 0, st>>>(in, out, n, scale);
    return after_launch();
}

extern "C" int fp8b_dequant_fmt(const uint8_t* in, int in_format, void* out, int out_dtype, size_t n, const float* scale,
                                void* stream)
{
    if (!valid_dtype(out_dtype) || (in_format != FP8B_E4M3FN && in_format != FP8B_E5M2)) return FP8B_ERR_INVALID;
    if (scale && out_dtype != FP8B_F16) return FP8B_ERR_INVALID;
    if (in_format == FP8B_E4M3FN)
        return out_dtype == FP8B_F16 ? fp8b_dequant_f16(in, out, n, scale, stream) : fp8b_dequant(in, out, out_dtype, n, stream);
    if (n == 0) return FP8B_OK;
    if (!in || !out) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    if (out_dtype == FP8B_F32) return launch_decode_e5m2<FP8B_F32, false>(in, out, n, nullptr, st);
    if (out_dtype == FP8B_BF16) return launch_decode_e5m2<FP8B_BF16, false>(in, out, n, nullptr, st);
    return scale ? launch_decode_e5m2<FP8B_F16, true>(in, out, n, scale, st)
                 : launch_decode_e5m2<FP8B_F16, false>(in, out, n, nullptr, st);
}

// wide -> fp8 launch: big tiles = 512 threads x 4 x 32 B (or 1024 x 4 x 16 B), small = 256 x 4 x 16 B
template <int IN, bool PRESCALE>
static int launch_encode_vec(const void* in, uint8_t* out, size_t n, const float* prescale, cudaStream_t st)
{
    constexpr int EPV = (IN == FP8B_F32) ? 4 : 8;
    const CastShape c = cast_shape(n / EPV);
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;
    // big tiles: 512 threads x 4 x 32-byte loads when the tensor allows 256-bit access, else 1024 x 4 x 16 bytes
    // (256-bit loads pay from ~2^26 elements: +3 % at 2^28, +10 % at 2^32, but -20 % at 2^24 where the kernel is
    // mostly ramp and the 512-thread CTAs expose less parallelism -- profiles/tools/cast_exp.py)
    if (c.big && n / EPV >= ((size_t)1 << 23) && aligned(in, 32) && aligned(out, 2 * EPV))
        return launch_ex(wide_to_fp8_kernel<IN, PRESCALE, 512, 4, 32>, dim3(c.grid), dim3(512), 0, st, 1, 1, pdl, in, out, n, prescale);
    if (c.big) return launch_ex(wide_to_fp8_kernel<IN, PRESCALE, 1024, 4>, dim3(c.grid), dim3(1024), 0, st, 1, 1, pdl, in, out, n, prescale);
    return launch_ex(wide_to_fp8_kernel<IN, PRESCALE, 256, 4>, dim3(c.grid), dim3(256), 0, st, 1, 1, pdl, in, out, n, prescale);
}

template <int IN>
static int launch_encode(const void* in, uint8_t* out, size_t n, const float* prescale, cudaStream_t st)
{
    constexpr int EPV = (IN == FP8B_F32) ? 4 : 8;
    if (aligned(in, 16) && aligned(out, EPV))
        return prescale ? launch_encode_vec<IN, true>(in, out, n, prescale, st)
                        : launch_encode_vec<IN, false>(in, out, n, nullptr, st);
    const int g = cast_grid(n);
    if (prescale) wide_to_fp8_scalar_kernel<IN, true><<<g, kCastThreads, 0, st>>>(in, out, n, prescale);
    else wide_to_fp8_scalar_kernel<IN, false><<<g, kCastThreads, 0, st>>>(in, out, n, nullptr);
    return after_launch();
}

extern "C" int fp8b_encode(const void* in, int in_dtype, uint8_t* out, size_t n, const float* prescale, void* stream)
{
    if (!valid_dtype(in_dtype)) return FP8B_ERR_INVALID;
    if (n == 0) return FP8B_OK;
    if (!in || !out) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    if (in_dtype == FP8B_F32) return launch_encode<FP8B_F32>(in, out, n, prescale, st);
    if (in_dtype == FP8B_F16) return launch_encode<FP8B_F16>(in, out, n, prescale, st);
    return launch_encode<FP8B_BF16>(in, out, n, prescale, st);
}

template <int IN>
static int launch_amax(const void* in, size_t n, uint32_t* scratch, cudaStream_t st)
{
    constexpr int EPV = (IN == FP8B_F32) ? 4 : 8;
    if (aligned(in, 16)) {
        const size_t cap = (size_t)device_info().sm_count * tune(kTuneAmaxCap, 8);
        const size_t want = (n / EPV + kCastThreads * 4 - 1) / (kCastThreads * 4) + 1;
        amax_kernel<IN><<<(int)(want < cap ? want : cap), kCastThreads, 0, st>>>(in, n, scratch);
    }
    else amax_scalar_kernel<IN><<<cast_grid(n), kCastThreads, 0, st>>>(in, n, scratch);
    return after_launch();
}

// ---- batched entry points ------------------------------------------------------------------
namespace {

// Collects aligned, non-empty spans into CastBatch tables and launches one persistent grid per table.
// epv: elements per wide-side vector; fp8_in: true for fp8 -> wide.  launch(table, grid, big).
template <typename LaunchFn, typename SingleFn>
int run_batch(const fp8b_span* spans, int count, int epv, bool fp8_in, int big_align_mult, LaunchFn launch, SingleFn single)
{
    if (count < 0 || (count > 0 && !spans)) return FP8B_ERR_INVALID;
    for (int i = 0; i < count; ++i)
        if (spans[i].n != 0 && (!spans[i].in || !spans[i].out)) return FP8B_ERR_INVALID;
    if (count == 0) return FP8B_OK;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    auto vec_ok = [&](const fp8b_span& sp) {
        return aligned(fp8_in ? sp.out : sp.in, 16) && aligned(fp8_in ? sp.in : sp.out, epv);
    };
    // tile size for the whole call, from the total amount of vector work (cast_shape)
    uint64_t total_vecs = 0;
    for (int i = 0; i < count; ++i) if (spans[i].n && vec_ok(spans[i])) total_vecs += spans[i].n / epv;
    const CastShape shape = cast_shape((size_t)total_vecs);
    // the big-tile kernel of this direction may need wider alignment (256-bit loads): such spans still convert,
    // through the single-tensor entry point
    const bool wide_loads = shape.big && big_align_mult > 1 && total_vecs >= (1ull << 23);
    const int mult = wide_loads ? big_align_mult : 1;
    auto table_ok = [&](const fp8b_span& sp) {
        return aligned(fp8_in ? sp.out : sp.in, 16 * mult) && aligned(fp8_in ? sp.in : sp.out, epv * mult);
    };
    const uint64_t tile_vecs = shape.big ? 4096 : 1024;
    const uint64_t cap = (uint64_t)device_info().sm_count * (shape.big ? 1 : 4);
    CastBatch b;
    b.count = 0;
    uint64_t tiles = 0;
    auto flush = [&]() -> int {
        if (b.count == 0) return FP8B_OK;
        const int rc = launch(b, (int)(tiles < cap ? tiles : cap), shape.big ? (wide_loads ? 2 : 1) : 0);
        b.count = 0; tiles = 0;
        return rc;
    };
    for (int i = 0; i < count; ++i) {
        const fp8b_span& sp = spans[i];
        if (sp.n == 0) continue;
        if (!table_ok(sp)) {                                           // rare: single-tensor path (scalar or 16-byte kernels)
            if (int rc = single(sp)) return rc;
            continue;
        }
        const uint64_t nvec = sp.n / epv;
        uint64_t t = (nvec + tile_vecs - 1) / tile_vecs;
        if (t == 0) t = 1;                                             // n < epv: one tile for the scalar tail
        if (t > 0xFFFFFFFFull) { if (int rc = single(sp)) return rc; continue; }
        if (b.count == kBatchMaxSpans || tiles + t > 0xFFFFFFFFull) { if (int rc = flush()) return rc; }
        tiles += t;
        b.tile_end[b.count] = (uint32_t)tiles;
        b.in[b.count] = sp.in; b.out[b.count] = sp.out; b.n[b.count] = sp.n;
        ++b.count;
    }
    return flush();
}

template <int IN>
int launch_encode_batch(const CastBatch& b, int grid, int big, cudaStream_t st)
{
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;
    if (big == 2) return launch_ex(wide_to_fp8_batch_kernel<IN, 512, 4, 32>, dim3(grid), dim3(512), 0, st, 1, 1, pdl, b);
    if (big) return launch_ex(wide_to_fp8_batch_kernel<IN, 1024, 4>, dim3(grid), dim3(1024), 0, st, 1, 1, pdl, b);
    return launch_ex(wide_to_fp8_batch_kernel<IN, 256, 4>, dim3(grid), dim3(256), 0, st, 1, 1, pdl, b);
}

template <int OUT>
int launch_decode_batch(const CastBatch& b, int grid, int big, cudaStream_t st)
{
    const bool pdl = g_opt_pdl.load(std::memory_order_relaxed) != 0;
    if (big) return launch_ex(fp8_to_wide_batch_kernel<OUT, 512, 8>, dim3(grid), dim3(512), 0, st, 1, 1, pdl, b);
    return launch_ex(fp8_to_wide_batch_kernel<OUT, 256, 4>, dim3(grid), dim3(256), 0, st, 1, 1, pdl, b);
}

}  // namespace

extern "C" int fp8b_encode_batch(const fp8b_span* spans, int count, int in_dtype, void* stream)
{
    if (!valid_dtype(in_dtype)) return FP8B_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    auto launch = [&](const CastBatch& b, int grid, int big) -> int {
        if (in_dtype == FP8B_F32) return launch_encode_batch<FP8B_F32>(b, grid, big, st);
        if (in_dtype == FP8B_F16) return launch_encode_batch<FP8B_F16>(b, grid, big, st);
        return launch_encode_batch<FP8B_BF16>(b, grid, big, st);
    };
    auto single = [&](const fp8b_span& sp) -> int {
        return fp8b_encode(sp.in, in_dtype, static_cast<uint8_t*>(sp.out), sp.n, nullptr, stream);
    };
    return run_batch(spans, count, in_dtype == FP8B_F32 ? 4 : 8, false, 2, launch, single);
}

extern "C" int fp8b_dequant_batch(const fp8b_span* spans, int count, int out_dtype, void* stream)
{
    if (!valid_dtype(out_dtype)) return FP8B_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    auto launch = [&](const CastBatch& b, int grid, int big) -> int {
        if (out_dtype == FP8B_F32) return launch_decode_batch<FP8B_F32>(b, grid, big, st);
        if (out_dtype == FP8B_F16) return launch_decode_batch<FP8B_F16>(b, grid, big, st);
        return launch_decode_batch<FP8B_BF16>(b, grid, big, st);
    };
    auto single = [&](const fp8b_span& sp) -> int {
        return fp8b_dequant(static_cast<const uint8_t*>(sp.in), sp.out, out_dtype, sp.n, stream);
    };
    return run_batch(spans, count, out_dtype == FP8B_F32 ? 4 : 8, true, 1, launch, single);
}

extern "C" int fp8b_amax_scale(const void* in, int in_dtype, size_t n, float* scale_out, float* inv_scale_out,
                               uint32_t* scratch, void* stream)
{
    if (!valid_dtype(in_dtype) || !scratch || (!scale_out && !inv_scale_out)) return FP8B_ERR_INVALID;
    if (n != 0 && !in) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(scratch, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess) return cuda_fail(e);
    int rc = FP8B_OK;
    if (n) {
        if (in_dtype == FP8B_F32) rc = launch_amax<FP8B_F32>(in, n, scratch, st);
        else if (in_dtype == FP8B_F16) rc = launch_amax<FP8B_F16>(in, n, scratch, st);
        else rc = launch_amax<FP8B_BF16>(in, n, scratch, st);
        if (rc != FP8B_OK) return rc;
    }
    amax_finalize_kernel<<<1, 1, 0, st>>>(scratch, scale_out, inv_scale_out);
    return after_launch();
}

extern "C" int fp8b_quantize_rows(const void* in, int in_dtype, int rows, size_t cols, uint8_t* out,
                                  float* inv_scale_out, void* stream)
{
    if (!valid_dtype(in_dtype) || rows < 0) return FP8B_ERR_INVALID;
    if (rows == 0) return FP8B_OK;
    if (!inv_scale_out || (cols != 0 && (!in || !out))) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t esz = dtype_size(in_dtype);
    const size_t epv = 16 / esz;
    // vector path: every row start 16-byte aligned on the wide side and epv-byte aligned on the fp8 side
    const int vec_ok = aligned(in, 16) && aligned(out, epv) && ((cols * esz) % 16 == 0) ? 1 : 0;
    // rows that fit in registers: one HBM read, no second pass (quantize_rows_reg_kernel)
    if (vec_ok && cols % epv == 0 && cols / epv <= 256 * 8 && cols > 0) {
        const int nvec = (int)(cols / epv);
        int rc = FP8B_OK;
#define FP8B_ROWS_REG(IN, V, TPR) \
        quantize_rows_reg_kernel<IN, V, TPR><<<(rows + (kCastThreads / TPR) - 1) / (kCastThreads / TPR), kCastThreads, 0, st>>>( \
            in, out, inv_scale_out, rows, nvec)
        // Few vectors per thread (V <= 4: registers stay low, many warps resident) and as many threads per row as
        // that needs; when there are too few rows to fill the GPU with warps, a whole CTA per row instead.
        const bool few_rows = (size_t)rows * 64 < (size_t)device_info().sm_count * 2048;
#define FP8B_ROWS_PICK(IN) \
        do { \
            if (few_rows || nvec > 128 * 4) { \
                if (nvec <= 256) FP8B_ROWS_REG(IN, 1, 256); \
                else if (nvec <= 512) FP8B_ROWS_REG(IN, 2, 256); \
                else if (nvec <= 1024) FP8B_ROWS_REG(IN, 4, 256); \
                else FP8B_ROWS_REG(IN, 8, 256); \
            } \
            else if (nvec <= 32 * 2) FP8B_ROWS_REG(IN, 2, 32); \
            else if (nvec <= 32 * 4) FP8B_ROWS_REG(IN, 4, 32); \
            else if (nvec <= 64 * 4) FP8B_ROWS_REG(IN, 4, 64); \
            else FP8B_ROWS_REG(IN, 4, 128); \
        } while (0)
        if (in_dtype == FP8B_F32) FP8B_ROWS_PICK(FP8B_F32);
        else if (in_dtype == FP8B_F16) FP8B_ROWS_PICK(FP8B_F16);
        else FP8B_ROWS_PICK(FP8B_BF16);
#undef FP8B_ROWS_PICK
#undef FP8B_ROWS_REG
        (void)rc;
        return after_launch();
    }
    if (in_dtype == FP8B_F32) quantize_rows_kernel<FP8B_F32><<<rows, kCastThreads, 0, st>>>(in, out, inv_scale_out, cols, vec_ok);
    else if (in_dtype == FP8B_F16) quantize_rows_kernel<FP8B_F16><<<rows, kCastThreads, 0, st>>>(in, out, inv_scale_out, cols, vec_ok);
    else quantize_rows_kernel<FP8B_BF16><<<rows, kCastThreads, 0, st>>>(in, out, inv_scale_out, cols, vec_ok);
    return after_launch();
}
