// Shared host-side helpers for libfp8_b200 (launch bookkeeping, status plumbing).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <utility>
#include "../../include/fp8_b200.h"

namespace fp8b {

extern std::atomic<uint64_t> g_launches;       // fp8b_launch_count()
extern thread_local int t_last_cuda_error;     // fp8b_last_cuda_error()

inline int cuda_fail(cudaError_t e) { t_last_cuda_error = (int)e; return FP8B_ERR_CUDA; }

// Call after every <<<>>> launch: counts it and converts a launch error into a status.
inline int after_launch() {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) { (void)cudaGetLastError(); return cuda_fail(e); }
    return FP8B_OK;
}

// One-time device facts (SM count, compute capability) for the current device.
struct DeviceInfo { int sm_count; int cc_major; int cc_minor; int ok; };
const DeviceInfo& device_info();

// Developer tuning knobs (fp8b_set_option, option ids FP8B_OPT_TUNE_*): choose between result-identical kernel
// variants so that tests and profiling scripts can A/B them without rebuilding.  Each starts from the environment
// variable of the same name (FP8B_GEMM_CFG, ...) read ONCE when the library is loaded -- never per call -- and none
// of them can change a result.  -1 = unset (use the built-in rule).
enum TuneKnob { kTuneGemmCfg = 0, kTuneGemvImpl, kTuneDynamicPlan, kTuneCastShape, kTuneGemmStore, kTuneGemvUnroll,
                kTuneGemvBatch, kTuneAmaxCap, kTuneGemmRaster, kTuneGemmSplitK, kTuneCount };
extern std::atomic<int> g_tune[kTuneCount];
inline int tune(TuneKnob k, int dflt) { const int v = g_tune[k].load(std::memory_order_relaxed); return v < 0 ? dflt : v; }
#ifdef FP8B_PROFILE
int tune_int(const char* name, int dflt);      // profiling builds only: environment, read per call
#endif

// Library options (fp8b_set_option)
extern std::atomic<int> g_opt_pdl;
extern std::atomic<int> g_opt_static_weights;

// Launch with optional cluster dimensions and programmatic dependent launch.
template <typename... KArgs, typename... Args>
inline int launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                     int cluster_x, int cluster_y, bool pdl, Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (cluster_x * cluster_y > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster_x; attr[n].val.clusterDim.y = cluster_y; attr[n].val.clusterDim.z = 1;
        ++n;
    }
    if (pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    cfg.attrs = attr; cfg.numAttrs = n;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
    if (e != cudaSuccess) return cuda_fail(e);
    return after_launch();
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: remember it per (kernel instantiation, device).
// `flags` is a function-local static array of 64 atomics owned by the caller.
template <typename K>
inline int ensure_max_smem(K kernel, int bytes, std::atomic<int>* flags)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return FP8B_ERR_NO_DEVICE;
    if (flags[dev].load(std::memory_order_acquire)) return FP8B_OK;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return cuda_fail(e);
    flags[dev].store(1, std::memory_order_release);      // idempotent if two threads race
    return FP8B_OK;
}

#ifdef __CUDACC__
// Programmatic dependent launch, device side.  Both are no-ops when the kernel was not launched with
// the PDL attribute (or has no predecessor).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }
inline size_t dtype_size(int dt) { return dt == FP8B_F32 ? 4 : dt == FP8B_OUT_E4M3FN ? 1 : 2; }
// input types (casts, bias, X of fp8b_linear_dynamic)
inline bool valid_dtype(int dt) { return dt == FP8B_F32 || dt == FP8B_F16 || dt == FP8B_BF16; }
// output types of the matmul entry points: the inputs plus e4m3fn bytes
inline bool valid_out_dtype(int dt) { return valid_dtype(dt) || dt == FP8B_OUT_E4M3FN; }

}  // namespace fp8b
