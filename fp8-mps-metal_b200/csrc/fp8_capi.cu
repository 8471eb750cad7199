// C-ABI surface of libfp8_b200.so that is not a kernel file's own: library info, device facts, and
// the scaled-matmul dispatcher (the analogue of the M-based selection in
// fp8_mps_native.fp8_scaled_mm / fp8_scaled_mm_auto, fp8_mps_native.py:78-93, :193-210).
#include <cstdlib>
#include <mutex>
#include "fp8_mm.cuh"

namespace fp8b {

std::atomic<uint64_t> g_launches{0};
std::atomic<int> g_opt_pdl{1};
std::atomic<int> g_opt_static_weights{0};
thread_local int t_last_cuda_error = 0;

const DeviceInfo& device_info()
{
    // One entry per device ordinal, filled on first use (the analogue of the reference bridge's
    // call_once context, fp8_bridge.cpp:63-71).
    static DeviceInfo info[64];
    static std::once_flag once[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
        static DeviceInfo bad = {0, 0, 0, 0};
        return bad;
    }
    std::call_once(once[dev], [dev] {
        DeviceInfo d = {0, 0, 0, 0};
        cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev);
        cudaDeviceGetAttribute(&d.cc_minor, cudaDevAttrComputeCapabilityMinor, dev);
        d.ok = (d.cc_major == 10 && d.sm_count > 0) ? 1 : 0;   // the fatbin holds sm_100a code only
        info[dev] = d;
    });
    return info[dev];
}

static int env_int(const char* name, int dflt)
{
    const char* v = std::getenv(name);
    return (v && *v) ? std::atoi(v) : dflt;
}
#ifdef FP8B_PROFILE
int tune_int(const char* name, int dflt) { return env_int(name, dflt); }
#endif

std::atomic<int> g_tune[kTuneCount];
namespace {
const char* const kTuneEnv[kTuneCount] = {"FP8B_GEMM_CFG", "FP8B_GEMV_IMPL", "FP8B_DYNAMIC_PLAN", "FP8B_CAST_SHAPE",
                                          "FP8B_GEMM_STORE", "FP8B_GEMV_UNROLL", "FP8B_GEMV_BATCH", "FP8B_AMAX_CAP",
                                          "FP8B_GEMM_RASTER", "FP8B_GEMM_SPLITK"};
struct TuneInit {
    TuneInit() { for (int k = 0; k < kTuneCount; ++k) g_tune[k].store(env_int(kTuneEnv[k], -1)); }
} g_tune_init;
}  // namespace

static int validate(const MMArgs& a)
{
    if (a.M < 0 || a.N < 0 || a.K < 0) return FP8B_ERR_INVALID;
    if (a.M == 0 || a.N == 0) return FP8B_OK;
    if (!a.C || !a.sa || !a.sb) return FP8B_ERR_INVALID;
    if (a.K > 0 && (!a.A || !a.B)) return FP8B_ERR_INVALID;
    if (!valid_out_dtype(a.out_dtype)) return FP8B_ERR_INVALID;
    if (a.bias && !valid_dtype(a.bias_dtype)) return FP8B_ERR_INVALID;
    if (a.ldc < a.N) return FP8B_ERR_INVALID;
    if (!(a.sa_len == 1 || a.sa_len == a.M)) return FP8B_ERR_INVALID;
    if (!(a.sb_len == 1 || a.sb_len == a.N)) return FP8B_ERR_INVALID;
    return FP8B_OK;
}

static int select_algo(const MMArgs& a)
{
    if (gemv_supported(a)) return FP8B_MM_GEMV;                 // M <= 16, fp8_mps_native.py:208
    if (tcgen05_supported(a)) return FP8B_MM_TCGEN05;
    return FP8B_MM_SIMT;
}

static int launch_algo(const MMArgs& a, int algo)
{
    switch (algo == FP8B_MM_AUTO ? select_algo(a) : algo) {
        case FP8B_MM_GEMV: return launch_gemv(a);
        case FP8B_MM_TCGEN05: return launch_gemm_tcgen05(a);
        case FP8B_MM_SIMT: return launch_gemm_simt(a);
        default: return FP8B_ERR_INVALID;
    }
}

// The arguments every scaled-matmul entry point shares; the result stores to C (Store::Local).
static MMArgs mm_args(const uint8_t* A, const uint8_t* B, void* C, int out_dtype, int M, int N, int K, int64_t ldc,
                      const float* scale_a, int scale_a_len, const float* scale_b, int scale_b_len,
                      const void* bias, int bias_dtype, const float* scale_result, void* stream)
{
    MMArgs a;
    a.A = A; a.B = B; a.C = C; a.out_dtype = out_dtype; a.M = M; a.N = N; a.K = K; a.ldc = ldc;
    a.sa = scale_a; a.sa_len = scale_a_len; a.sb = scale_b; a.sb_len = scale_b_len;
    a.bias = bias; a.bias_dtype = bias_dtype; a.sr = scale_result;
    a.st = (cudaStream_t)stream;
    return a;
}

// The exchange entry points (multicast, peers, push): tcgen05 only, no fallback.  `empty` is the status of an
// empty shard (M == 0 or N == 0).
static int launch_exchange(const MMArgs& a, int empty)
{
    int rc = validate(a);
    if (rc != FP8B_OK) return rc;
    if (a.M == 0 || a.N == 0) return empty;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    return launch_gemm_tcgen05(a);          // FP8B_ERR_UNSUPPORTED unless tcgen05_supported(a)
}

static bool valid_dsts(void* const* dsts, int n_dst)
{
    if (n_dst < 1 || n_dst > 8 || !dsts) return false;
    for (int d = 0; d < n_dst; ++d)
        if (!dsts[d]) return false;
    return true;
}

}  // namespace fp8b

using namespace fp8b;

extern "C" int fp8b_version(void) { return FP8B_VERSION; }

extern "C" const char* fp8b_status_string(int status)
{
    switch (status) {
        case FP8B_OK: return "ok";
        case FP8B_ERR_INVALID: return "invalid argument";
        case FP8B_ERR_UNSUPPORTED: return "unsupported by the requested entry point (no fallback taken)";
        case FP8B_ERR_CUDA: return "CUDA call failed (see fp8b_last_cuda_error)";
        case FP8B_ERR_NO_DEVICE: return "current device is not an sm_100 (B200-class) GPU";
        default: return "unknown status";
    }
}

extern "C" int fp8b_set_option(int option, int value)
{
    switch (option) {
        case FP8B_OPT_PDL: g_opt_pdl.store(value ? 1 : 0); return FP8B_OK;
        case FP8B_OPT_STATIC_WEIGHTS: g_opt_static_weights.store(value ? 1 : 0); return FP8B_OK;
        default:
            if (option >= FP8B_OPT_TUNE_GEMM_CFG && option < FP8B_OPT_TUNE_GEMM_CFG + kTuneCount) {
                g_tune[option - FP8B_OPT_TUNE_GEMM_CFG].store(value < 0 ? -1 : value);
                return FP8B_OK;
            }
            return FP8B_ERR_INVALID;
    }
}

extern "C" int fp8b_get_option(int option)
{
    switch (option) {
        case FP8B_OPT_PDL: return g_opt_pdl.load();
        case FP8B_OPT_STATIC_WEIGHTS: return g_opt_static_weights.load();
        default:
            if (option >= FP8B_OPT_TUNE_GEMM_CFG && option < FP8B_OPT_TUNE_GEMM_CFG + kTuneCount)
                return g_tune[option - FP8B_OPT_TUNE_GEMM_CFG].load();
            return FP8B_ERR_INVALID;
    }
}

extern "C" int fp8b_last_cuda_error(void) { return t_last_cuda_error; }
extern "C" uint64_t fp8b_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" size_t fp8b_scaled_mm_workspace_bytes(int, int, int) { return 0; }   // split-K reduces through DSMEM

extern "C" int fp8b_scaled_mm_select(const uint8_t* A, const uint8_t* B, const void* C, int out_dtype,
                                     int M, int N, int K, int64_t ldc)
{
    MMArgs a = {};
    a.A = A; a.B = B; a.C = const_cast<void*>(C); a.out_dtype = out_dtype; a.M = M; a.N = N; a.K = K; a.ldc = ldc;
    return select_algo(a);
}

static int scaled_mm_impl(const MMArgs& a, int algo)
{
    int rc = validate(a);
    if (rc != FP8B_OK) return rc;
    if (a.M == 0 || a.N == 0) return FP8B_OK;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    return launch_algo(a, algo);
}

extern "C" int fp8b_scaled_mm(const uint8_t* A, const uint8_t* B, void* C, int out_dtype,
                              int M, int N, int K, int64_t ldc,
                              const float* scale_a, int scale_a_len,
                              const float* scale_b, int scale_b_len,
                              const void* bias, int bias_dtype,
                              const float* scale_result,
                              void* /*workspace*/, size_t /*workspace_bytes*/,     // no kernel needs one
                              int algo, void* stream)
{
    return scaled_mm_impl(mm_args(A, B, C, out_dtype, M, N, K, ldc, scale_a, scale_a_len, scale_b, scale_b_len,
                                  bias, bias_dtype, scale_result, stream), algo);
}

extern "C" int fp8b_scaled_mm_fmt(const uint8_t* A, int a_format, const uint8_t* B, int b_format, void* C, int out_dtype,
                                  int M, int N, int K, int64_t ldc,
                                  const float* scale_a, int scale_a_len,
                                  const float* scale_b, int scale_b_len,
                                  const void* bias, int bias_dtype,
                                  const float* scale_result,
                                  int algo, void* stream)
{
    if ((a_format != FP8B_E4M3FN && a_format != FP8B_E5M2) || (b_format != FP8B_E4M3FN && b_format != FP8B_E5M2))
        return FP8B_ERR_INVALID;
    MMArgs a = mm_args(A, B, C, out_dtype, M, N, K, ldc, scale_a, scale_a_len, scale_b, scale_b_len, bias, bias_dtype,
                       scale_result, stream);
    a.a_fmt = a_format; a.b_fmt = b_format;
    return scaled_mm_impl(a, algo);
}

extern "C" int fp8b_scaled_mm_multicast(const uint8_t* A, const uint8_t* B, void* C_multicast, int out_dtype,
                                        int M, int N, int K, int64_t ldc,
                                        const float* scale_a, int scale_a_len,
                                        const float* scale_b, int scale_b_len,
                                        const void* bias, int bias_dtype,
                                        const float* scale_result, void* stream)
{
    MMArgs a = mm_args(A, B, C_multicast, out_dtype, M, N, K, ldc, scale_a, scale_a_len, scale_b, scale_b_len, bias,
                       bias_dtype, scale_result, stream);
    a.store = Store::Multicast;
    // no byte output through the multicast mapping
    if (out_dtype == FP8B_OUT_E4M3FN && validate(a) == FP8B_OK) return FP8B_ERR_UNSUPPORTED;
    return launch_exchange(a, FP8B_OK);
}

static size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

extern "C" size_t fp8b_linear_dynamic_workspace_bytes(int M, int K)
{
    if (M <= 0 || K <= 0) return 0;
    return align16((size_t)M * (size_t)K) + align16((size_t)M * sizeof(float));
}

extern "C" int fp8b_linear_dynamic(const void* X, int x_dtype, const uint8_t* B, void* C, int out_dtype,
                                 int M, int N, int K, int64_t ldc,
                                 const float* scale_b, int scale_b_len,
                                 const void* bias, int bias_dtype, const float* scale_result,
                                 float* inv_scale_a_out, void* workspace, size_t workspace_bytes, void* stream)
{
    if (M < 0 || N < 0 || K < 0) return FP8B_ERR_INVALID;
    if (M == 0 || N == 0) return FP8B_OK;
    if (!X || !B || !C || !scale_b || !valid_dtype(x_dtype) || !valid_out_dtype(out_dtype)) return FP8B_ERR_INVALID;
    if (bias && !valid_dtype(bias_dtype)) return FP8B_ERR_INVALID;
    if (ldc < N || !(scale_b_len == 1 || scale_b_len == N)) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    const size_t need = fp8b_linear_dynamic_workspace_bytes(M, K);
    const bool have_ws = workspace && workspace_bytes >= need && aligned(workspace, 16);
    // the single-kernel plan reads X and B with 16-byte vectors; the workspace plan (quantise rows, then the GEMV
    // dispatcher) takes any K and alignment through their scalar / generic kernels
    const bool vec_ok = K >= 16 && (K % 16) == 0 && aligned(B, 16) && aligned(X, 16);
    if (M <= 16 && !have_ws && !vec_ok) return FP8B_ERR_UNSUPPORTED;
    if (M > 16 && !have_ws) return FP8B_ERR_UNSUPPORTED;         // the GEMM path always quantises into the workspace
    // A and scale_a: set below (workspace plans) / unused (single-kernel plan)
    MMArgs a = mm_args(nullptr, B, C, out_dtype, M, N, K, ldc, scale_b, 1, scale_b, scale_b_len, bias, bias_dtype,
                       scale_result, stream);

    // Two plans.  With a workspace: quantise once (one CTA per row) and chain the GEMV behind it with
    // programmatic dependent launch -- the GEMV is resident and already streaming its first weight vectors
    // while the rows are quantised.  Without: one kernel in which every CTA quantises the rows it needs
    // (cheaper only when the grid is small; it repeats the encode per CTA).
    // M > 16: the same quantise kernel, then the shape-selected GEMM (tcgen05 when TMA-able) with per-row
    // scale_a.  Converting inside the GEMM's producer stage instead would redo the encode once per N-tile
    // column (48x for C4) on data that is read from L2 anyway; one 6 us pass over A is cheaper.
    const int plan = tune(kTuneDynamicPlan, 0);         // 1 = force single kernel, 2 = force chain
    if (have_ws && (plan != 1 || M > 16 || !vec_ok)) {
        uint8_t* q = static_cast<uint8_t*>(workspace);
        float* inv = inv_scale_a_out ? inv_scale_a_out
                                     : reinterpret_cast<float*>(q + align16((size_t)M * (size_t)K));
        int rc = fp8b_quantize_rows(X, x_dtype, M, (size_t)K, q, inv, stream);
        if (rc != FP8B_OK) return rc;
        a.A = q; a.sa = inv; a.sa_len = M;
        if (M > 16) return launch_algo(a, FP8B_MM_AUTO);
        a.chain_pdl = 1;
        return launch_gemv(a);
    }
    if (plan == 2) return FP8B_ERR_INVALID;
    return launch_gemv_fhfma(a, make_epi(a), X, x_dtype, inv_scale_a_out);
}

extern "C" int fp8b_scaled_mm_peers(const uint8_t* A, const uint8_t* B, void* C_local, const int64_t* peer_deltas, int world,
                                    int out_dtype, int M, int N, int K, int64_t ldc,
                                    const float* scale_a, int scale_a_len,
                                    const float* scale_b, int scale_b_len,
                                    const void* bias, int bias_dtype,
                                    const float* scale_result, void* stream)
{
    if (world < 2 || world > 8 || !peer_deltas) return FP8B_ERR_INVALID;
    MMArgs a = mm_args(A, B, C_local, out_dtype, M, N, K, ldc, scale_a, scale_a_len, scale_b, scale_b_len, bias,
                       bias_dtype, scale_result, stream);
    a.store = Store::Peers; a.n_dst = world; a.peer_deltas = peer_deltas;
    return launch_exchange(a, FP8B_OK);
}

// N-sharded linear, fused compute + exchange with TMA stores: see include/fp8_b200.h.
extern "C" int fp8b_scaled_mm_push(const uint8_t* A, const uint8_t* B, void* const* C_dsts, int n_dst,
                                   int out_dtype, int M, int N, int K, int64_t ldc,
                                   const float* scale_a, int scale_a_len,
                                   const float* scale_b, int scale_b_len,
                                   const void* bias, int bias_dtype,
                                   const float* scale_result, void* stream)
{
    if (!valid_dsts(C_dsts, n_dst)) return FP8B_ERR_INVALID;
    MMArgs a = mm_args(A, B, C_dsts[0], out_dtype, M, N, K, ldc, scale_a, scale_a_len, scale_b, scale_b_len, bias,
                       bias_dtype, scale_result, stream);
    a.store = Store::Push; a.n_dst = n_dst; a.dsts = C_dsts;
    return launch_exchange(a, FP8B_OK);
}

extern "C" int fp8b_scaled_mm_push_signal(const uint8_t* A, const uint8_t* B, void* const* C_dsts, int n_dst,
                                          int out_dtype, int M, int N, int K, int64_t ldc,
                                          const float* scale_a, int scale_a_len,
                                          const float* scale_b, int scale_b_len,
                                          const void* bias, int bias_dtype, const float* scale_result,
                                          uint64_t* const* signal_flags, uint32_t* cta_counter, uint64_t epoch, void* stream)
{
    if (!valid_dsts(C_dsts, n_dst) || !signal_flags || !cta_counter) return FP8B_ERR_INVALID;
    PushSignal sig;
    for (int d = 0; d < 8; ++d) sig.flags[d] = d < n_dst ? signal_flags[d] : nullptr;
    sig.cta_counter = cta_counter;
    sig.epoch = epoch;
    MMArgs a = mm_args(A, B, C_dsts[0], out_dtype, M, N, K, ldc, scale_a, scale_a_len, scale_b, scale_b_len, bias,
                       bias_dtype, scale_result, stream);
    a.store = Store::Push; a.n_dst = n_dst; a.dsts = C_dsts;
    a.sig = &sig;
    // an empty shard cannot signal: the caller uses fp8b_peer_signal
    return launch_exchange(a, FP8B_ERR_UNSUPPORTED);
}

extern "C" int fp8b_peer_wait(const uint64_t* flags, int world, int rank, uint64_t epoch, void* stream)
{
    if (!flags || world < 2 || world > 8 || rank < 0 || rank >= world) return FP8B_ERR_INVALID;
    if (!device_info().ok) return FP8B_ERR_NO_DEVICE;
    return launch_peer_wait(flags, world, rank, epoch, (cudaStream_t)stream);
}

extern "C" int fp8b_scaled_mm_push_supported(int out_dtype, int M, int N, int K, int64_t ldc, const void* A, const void* B,
                                             const void* C)
{
    if (M < 1 || N < 1 || K < 16 || (K % 16) != 0 || !valid_out_dtype(out_dtype) || ldc < N) return 0;
    if (!aligned(A, 16) || !aligned(B, 16) || !aligned(C, 16)) return 0;
    return (((size_t)ldc * dtype_size(out_dtype)) % 16 == 0 && ((size_t)N * dtype_size(out_dtype)) % 16 == 0) ? 1 : 0;
}
