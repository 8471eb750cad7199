// fp8_metal -- the torch extension of the B200 build: a thin binding from torch tensors to the
// C ABI of libfp8_b200.so (include/fp8_b200.h).
//
// It is the analogue of the reference's fp8_bridge.cpp (module `fp8_metal`,
// fp8_bridge.cpp:361-371) and keeps its three ops with the same names, argument order and
// TORCH_CHECK behaviour (fp8_bridge.cpp:174-177,191,269):
//     fp8_scaled_mm(A, B, scale_a, scale_b) -> (M,N) float32
//     fp8_dequantize(input, scale)          -> float16, same shape
//     fp8_quantize(input)                   -> (uint8, inv_scale float32[1])
// Where the reference bridge copies every tensor MPS->CPU->MTLBuffer and blocks on
// waitUntilCompleted (fp8_bridge.cpp:180-185,244-245), this one passes device pointers and the
// caller's current CUDA stream and returns without synchronising.  No CUDA kernel lives here and
// nothing falls back to ATen math: every op is one or two calls into the C ABI.
#include <mutex>
#include <stdexcept>
#include <string>
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>

#include <tuple>

#include "../../include/fp8_b200.h"

namespace {

int to_fp8b_dtype(at::ScalarType t)
{
    switch (t) {
        case at::kFloat: return FP8B_F32;
        case at::kHalf: return FP8B_F16;
        case at::kBFloat16: return FP8B_BF16;
        default: throw std::runtime_error(std::string("fp8_metal: unsupported dtype ") + c10::toString(t) +
                                          " (need float32, float16 or bfloat16)");
    }
    return -1;
}

// Output dtype of the matmul ops: the three above plus float8_e4m3fn, whose bytes are the reference encoder's bytes of the
// fp32 epilogue value (what the reference's `_scaled_mm(...).to(float8_e4m3fn)` produces).  Inputs and biases stay with
// to_fp8b_dtype; float8_e5m2 is never an output.
int to_fp8b_out_dtype(at::ScalarType t)
{
    if (t == at::kFloat8_e4m3fn) return FP8B_OUT_E4M3FN;
    if (t == at::kFloat || t == at::kHalf || t == at::kBFloat16) return to_fp8b_dtype(t);
    throw std::runtime_error(std::string("fp8_metal: unsupported output dtype ") + c10::toString(t) +
                             " (need float32, float16, bfloat16 or float8_e4m3fn)");
}

// The reference raises std::runtime_error for launch failures (fp8_bridge.cpp:96-101); so does this.
void check_status(int rc, const char* what)
{
    if (rc == FP8B_OK) return;
    std::string msg = std::string("fp8_metal: ") + what + " failed: " + fp8b_status_string(rc) + " (status " +
                      std::to_string(rc) + ", cuda error " + std::to_string(fp8b_last_cuda_error()) + ")";
    throw std::runtime_error(msg);
}

void* current_stream() { return static_cast<void*>(at::cuda::getCurrentCUDAStream().stream()); }

const uint8_t* u8_ptr(const torch::Tensor& t) { return static_cast<const uint8_t*>(t.data_ptr()); }

// ---- argument preparation shared by the bindings ----------------------------------------------
// Each rule below exists once; the bindings only name which ones apply to them.

// A float tensor as the kernels read it: contiguous, float32/float16/bfloat16 as they are, anything else widened to
// float32 (fp8_mps_native.py:142).  Inputs of the casts and biases of the matmuls follow the same rule.
torch::Tensor float_input(const torch::Tensor& t)
{
    torch::Tensor in = t.contiguous();
    const auto st = in.scalar_type();
    return (st == at::kFloat || st == at::kHalf || st == at::kBFloat16) ? in : in.to(torch::kFloat32);
}

// FP8-encoded matmul operand: uint8, on the GPU, row-major.
void check_fp8_operand(const torch::Tensor& t, const char* name)
{
    TORCH_CHECK(t.dtype() == torch::kUInt8, name, " must be uint8 (FP8 encoded)");
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
    TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}

// A (M,K) and B (N,K) of one matmul.
void check_fp8_pair(const torch::Tensor& A, const torch::Tensor& B)
{
    check_fp8_operand(A, "A");
    check_fp8_operand(B, "B");
    TORCH_CHECK(A.dim() == 2 && B.dim() == 2, "A must be (M,K) and B must be (N,K)");
    TORCH_CHECK(B.size(1) == A.size(1), "K dimension mismatch between A and B");
    TORCH_CHECK(A.device() == B.device(), "A and B must be on the same device");
    TORCH_CHECK(A.size(0) < (1LL << 31) && B.size(0) < (1LL << 31) && A.size(1) < (1LL << 31), "extent too large");
}

struct Scale {
    torch::Tensor keep;                 // holds a converted scale alive until the call
    const float* ptr = nullptr;
    int len = 0;
};

// The default scale 1.0 of one device: a float of its own cudaMalloc memory, written once and kept for the life of the
// process, so that no call allocates or launches anything for it.  It is written by a blocking copy on a private stream,
// never on the caller's stream: a first call inside a graph capture would otherwise capture the fill instead of running
// it (every eager call before the first replay would read unwritten memory), and a first call on a busy stream would
// let a call on another stream read the scale before the fill had run.  Relaxed capture mode lets the allocation and
// the blocking copy run while this or another thread is capturing.
const float* default_scale(int device)
{
    static std::mutex mu;
    static float* ones[64] = {};
    TORCH_CHECK(device >= 0 && device < 64, "fp8_metal: device ordinal out of range");
    std::lock_guard<std::mutex> lock(mu);
    if (ones[device]) return ones[device];
    static const float one = 1.0f;
    cudaStreamCaptureMode mode = cudaStreamCaptureModeRelaxed;
    cudaThreadExchangeStreamCaptureMode(&mode);
    float* ptr = nullptr;
    cudaStream_t st = nullptr;
    cudaError_t e = cudaMalloc(&ptr, sizeof(float));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ptr, &one, sizeof(float), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (st) cudaStreamDestroy(st);
    if (e != cudaSuccess && ptr) cudaFree(ptr);
    cudaThreadExchangeStreamCaptureMode(&mode);
    TORCH_CHECK(e == cudaSuccess, "fp8_metal: could not set up the default scale: ", cudaGetErrorString(e));
    ones[device] = ptr;
    return ptr;
}

// A scale as a float32 device pointer of 1 or n elements (`msg` when it has neither).  A tensor that already is one is
// used as it is, any other is converted; None is the default scale 1.0 (fp8_mps_patch.py:87-90).
Scale scale_arg(const c10::optional<torch::Tensor>& s, const torch::Device& dev, int64_t n, const char* msg)
{
    Scale r;
    if (!s.has_value() || !s->defined()) {
        r.ptr = default_scale(dev.has_index() ? dev.index() : c10::cuda::current_device());
        r.len = 1;
        return r;
    } else if (s->device() == dev && s->scalar_type() == at::kFloat && s->is_contiguous()) {
        r.keep = *s;
    } else {
        r.keep = s->to(dev, torch::kFloat32).contiguous();
    }
    const int64_t len = r.keep.numel();
    TORCH_CHECK(len == 1 || len == n, msg);
    r.ptr = r.keep.data_ptr<float>();
    r.len = (int)len;
    return r;
}

// scale_result: nullptr when absent, else one element.
Scale scale_result_arg(const c10::optional<torch::Tensor>& s, const torch::Device& dev)
{
    if (!s.has_value() || !s->defined()) return Scale();
    return scale_arg(s, dev, 1, "scale_result must have 1 element");
}

struct Bias {
    torch::Tensor keep;
    const void* ptr = nullptr;
    int dtype = FP8B_F32;
};

// An N-element bias on `dev` as (pointer, FP8B dtype); none when undefined.  A contiguous tensor on `dev` in a bias
// dtype is passed as it is.
Bias bias_arg(const c10::optional<torch::Tensor>& bias, const torch::Device& dev, int64_t N)
{
    Bias r;
    if (!bias.has_value() || !bias->defined()) return r;
    r.keep = float_input(bias->device() == dev ? *bias : bias->to(dev));
    TORCH_CHECK(r.keep.numel() == N, "bias must have N elements");
    r.ptr = r.keep.data_ptr();
    r.dtype = to_fp8b_dtype(r.keep.scalar_type());
    return r;
}

// Exchange bindings: the N-column block at n0 of a row-major (M, full_N) buffer at `base` must lie inside it; returns
// the address of its first element.
void* column_block(uintptr_t base, int64_t n0, int64_t N, int64_t full_N, size_t elem_size)
{
    TORCH_CHECK(n0 >= 0 && n0 + N <= full_N, "column block outside the full matrix");
    return reinterpret_cast<void*>(base + static_cast<uintptr_t>(n0) * elem_size);
}

// ---- fused scaled matmul: everything torch._scaled_mm can ask for, in one kernel -------------
torch::Tensor fp8_scaled_mm_fused(torch::Tensor A, torch::Tensor B, torch::Tensor scale_a, torch::Tensor scale_b,
                                  c10::optional<torch::Tensor> bias, c10::optional<torch::Tensor> scale_result,
                                  c10::optional<at::ScalarType> out_dtype, int64_t algo,
                                  c10::optional<torch::Tensor> out, int64_t a_format, int64_t b_format)
{
    check_fp8_pair(A, B);
    const int64_t M = A.size(0), K = A.size(1), N = B.size(0);
    const auto dev = A.device();
    c10::cuda::CUDAGuard guard(dev);
    const Scale sa = scale_arg(scale_a, dev, M, "scale_a must have 1 or M elements");
    const Scale sb = scale_arg(scale_b, dev, N, "scale_b must have 1 or N elements");

    const at::ScalarType odt = out_dtype.value_or(at::kFloat);          // out_dtype=None -> fp32 (fp8_mps_patch.py:103)
    torch::Tensor C;
    int64_t ldc = N;
    if (out.has_value()) {
        C = *out;
        TORCH_CHECK(C.is_cuda() && C.device() == dev && C.dim() == 2 && C.size(0) == M && C.size(1) == N,
                    "out must be a (M,N) CUDA tensor on A's device");
        TORCH_CHECK(C.scalar_type() == odt, "out dtype mismatch");
        TORCH_CHECK(C.stride(1) == 1 && C.stride(0) >= N, "out must be row-major with unit column stride");
        ldc = C.stride(0);
    } else {
        C = torch::empty({M, N}, torch::TensorOptions().dtype(odt).device(dev));
    }
    const Bias b = bias_arg(bias, dev, N);
    const Scale sr = scale_result_arg(scale_result, dev);

    if (M == 0 || N == 0) return C;
    check_status(fp8b_scaled_mm_fmt(u8_ptr(A), (int)a_format, u8_ptr(B), (int)b_format, C.data_ptr(), to_fp8b_out_dtype(odt),
                                    (int)M, (int)N, (int)K, ldc, sa.ptr, sa.len, sb.ptr, sb.len, b.ptr, b.dtype, sr.ptr,
                                    (int)algo, current_stream()),
                 "fp8b_scaled_mm");
    return C;
}

// ---- torch._scaled_mm as the patch sees it, in one C++ call --------------------------------------
// fp8_mps_patch._metal_scaled_mm used to do the dtype views, the transpose check and the scale conversions as
// separate Python-level tensor ops (~6 us of host time per call, more than a decode GEMV's kernel time); this does
// the same on raw strides and pointers.  input: (M,K) uint8 / float8_e4m3fn / float8_e5m2; other: (K,N), normally
// column-major so that its memory IS the (N,K) row-major weight (fp8_mps_patch.py:82-84).
int format_of(const torch::Tensor& t)
{
    return t.scalar_type() == at::kFloat8_e5m2 ? FP8B_E5M2 : FP8B_E4M3FN;     // uint8 is taken as e4m3fn (reference)
}

bool is_fp8_like(const torch::Tensor& t)
{
    const auto st = t.scalar_type();
    return st == at::kByte || st == at::kFloat8_e4m3fn || st == at::kFloat8_e5m2;
}

torch::Tensor scaled_mm_patch(torch::Tensor input, torch::Tensor other, c10::optional<torch::Tensor> scale_a,
                              c10::optional<torch::Tensor> scale_b, c10::optional<torch::Tensor> bias,
                              c10::optional<torch::Tensor> scale_result, c10::optional<at::ScalarType> out_dtype)
{
    TORCH_CHECK(is_fp8_like(input) && is_fp8_like(other), "operands must be uint8 / float8_e4m3fn / float8_e5m2");
    TORCH_CHECK(input.is_cuda() && other.is_cuda() && input.device() == other.device(), "operands must be CUDA tensors on one device");
    TORCH_CHECK(input.dim() == 2 && other.dim() == 2 && input.size(1) == other.size(0), "K dimension mismatch between A and B");
    const int64_t M = input.size(0), K = input.size(1), N = other.size(1);
    TORCH_CHECK(M < (1LL << 31) && N < (1LL << 31) && K < (1LL << 31), "extent too large");
    const auto dev = input.device();
    c10::cuda::CUDAGuard guard(dev);

    torch::Tensor a = input.is_contiguous() ? input : input.contiguous();
    // (N,K) row-major view of `other`: free when other is column-major, one copy otherwise (fp8_mps_patch.py:84)
    torch::Tensor b = (other.stride(0) == 1 && (other.stride(1) == K || N == 1)) ? other : other.t().contiguous();

    const Scale sa = scale_arg(scale_a, dev, M, "scale_a must have 1 or M elements");
    const Scale sb = scale_arg(scale_b, dev, N, "scale_b must have 1 or N elements");
    const Bias bi = bias_arg(bias, dev, N);
    const Scale sr = scale_result_arg(scale_result, dev);
    const at::ScalarType odt = out_dtype.value_or(at::kFloat);          // out_dtype=None -> fp32 (fp8_mps_patch.py:103)
    torch::Tensor C = torch::empty({M, N}, torch::TensorOptions().dtype(odt).device(dev));
    if (M == 0 || N == 0) return C;
    check_status(fp8b_scaled_mm_fmt(u8_ptr(a), format_of(input), u8_ptr(b), format_of(other), C.data_ptr(),
                                    to_fp8b_out_dtype(odt), (int)M, (int)N, (int)K, N, sa.ptr, sa.len, sb.ptr, sb.len,
                                    bi.ptr, bi.dtype, sr.ptr, FP8B_MM_AUTO, current_stream()),
                 "fp8b_scaled_mm");
    return C;
}

// ---- the reference bridge's three ops (fp8_bridge.cpp:165, :265, :312) ------------------------
torch::Tensor fp8_scaled_mm(torch::Tensor A, torch::Tensor B, torch::Tensor scale_a, torch::Tensor scale_b)
{
    return fp8_scaled_mm_fused(A, B, scale_a, scale_b, c10::nullopt, c10::nullopt, c10::nullopt, FP8B_MM_AUTO, c10::nullopt,
                               FP8B_E4M3FN, FP8B_E4M3FN);
}

torch::Tensor fp8_dequantize(torch::Tensor input, torch::Tensor scale)
{
    TORCH_CHECK(input.dtype() == torch::kUInt8, "input must be uint8");
    TORCH_CHECK(input.is_cuda(), "input must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(input.device());
    torch::Tensor in = input.contiguous();
    const Scale sc = scale_arg(scale, input.device(), 1, "scale must be a scalar tensor");
    torch::Tensor out = torch::empty(in.sizes(), torch::TensorOptions().dtype(torch::kFloat16).device(in.device()));
    check_status(fp8b_dequant_f16(u8_ptr(in), out.data_ptr(), (size_t)in.numel(), sc.ptr, current_stream()),
                 "fp8b_dequant_f16");
    return out;
}

// FP8 -> dtype exact cast (no scale): the `.to(dtype)` route of the patch in one pass.
torch::Tensor fp8_dequantize_to(torch::Tensor input, at::ScalarType dtype, int64_t format)
{
    TORCH_CHECK(input.dtype() == torch::kUInt8, "input must be uint8");
    TORCH_CHECK(input.is_cuda(), "input must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(input.device());
    torch::Tensor in = input.contiguous();
    torch::Tensor out = torch::empty(in.sizes(), torch::TensorOptions().dtype(dtype).device(in.device()));
    check_status(fp8b_dequant_fmt(u8_ptr(in), (int)format, out.data_ptr(), to_fp8b_dtype(dtype), (size_t)in.numel(), nullptr,
                                  current_stream()),
                 "fp8b_dequant_fmt");
    return out;
}

// float -> FP8 without scaling (fp8_mps_native.fp8_encode); reads f32/f16/bf16 natively.
torch::Tensor fp8_encode(torch::Tensor input)
{
    TORCH_CHECK(input.is_cuda(), "input must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(input.device());
    torch::Tensor in = float_input(input);
    torch::Tensor out = torch::empty(in.sizes(), torch::TensorOptions().dtype(torch::kUInt8).device(in.device()));
    check_status(fp8b_encode(in.data_ptr(), to_fp8b_dtype(in.scalar_type()), static_cast<uint8_t*>(out.data_ptr()),
                             (size_t)in.numel(), nullptr, current_stream()),
                 "fp8b_encode");
    return out;
}

// Many tensors, one launch per dtype group (fp8b_encode_batch): the checkpoint-conversion path.
std::vector<torch::Tensor> fp8_encode_many(std::vector<torch::Tensor> inputs)
{
    std::vector<torch::Tensor> ins(inputs.size()), outs(inputs.size());
    if (inputs.empty()) return outs;
    const auto dev = inputs[0].device();
    TORCH_CHECK(dev.is_cuda(), "inputs must be CUDA tensors");
    c10::cuda::CUDAGuard guard(dev);
    for (size_t i = 0; i < inputs.size(); ++i) {
        TORCH_CHECK(inputs[i].device() == dev, "all inputs must be on one device");
        ins[i] = float_input(inputs[i]);
        outs[i] = torch::empty(ins[i].sizes(), torch::TensorOptions().dtype(torch::kUInt8).device(dev));
    }
    for (at::ScalarType dt : {at::kFloat, at::kHalf, at::kBFloat16}) {
        std::vector<fp8b_span> spans;
        for (size_t i = 0; i < ins.size(); ++i)
            if (ins[i].scalar_type() == dt) spans.push_back({ins[i].data_ptr(), outs[i].data_ptr(), (size_t)ins[i].numel()});
        if (!spans.empty())
            check_status(fp8b_encode_batch(spans.data(), (int)spans.size(), to_fp8b_dtype(dt), current_stream()),
                         "fp8b_encode_batch");
    }
    return outs;
}

std::vector<torch::Tensor> fp8_dequantize_many(std::vector<torch::Tensor> inputs, at::ScalarType dtype)
{
    std::vector<torch::Tensor> ins(inputs.size()), outs(inputs.size());
    if (inputs.empty()) return outs;
    const auto dev = inputs[0].device();
    TORCH_CHECK(dev.is_cuda(), "inputs must be CUDA tensors");
    c10::cuda::CUDAGuard guard(dev);
    std::vector<fp8b_span> spans;
    for (size_t i = 0; i < inputs.size(); ++i) {
        TORCH_CHECK(inputs[i].dtype() == torch::kUInt8, "inputs must be uint8");
        TORCH_CHECK(inputs[i].device() == dev, "all inputs must be on one device");
        ins[i] = inputs[i].contiguous();
        outs[i] = torch::empty(ins[i].sizes(), torch::TensorOptions().dtype(dtype).device(dev));
        spans.push_back({ins[i].data_ptr(), outs[i].data_ptr(), (size_t)ins[i].numel()});
    }
    check_status(fp8b_dequant_batch(spans.data(), (int)spans.size(), to_fp8b_dtype(dtype), current_stream()),
                 "fp8b_dequant_batch");
    return outs;
}

std::tuple<torch::Tensor, torch::Tensor> fp8_quantize(torch::Tensor input)
{
    TORCH_CHECK(input.is_cuda(), "input must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(input.device());
    torch::Tensor in = float_input(input);
    auto f32 = torch::TensorOptions().dtype(torch::kFloat32).device(in.device());
    torch::Tensor scales = torch::empty({2}, f32);                    // [scale, inv_scale]
    torch::Tensor scratch = torch::empty({1}, torch::TensorOptions().dtype(torch::kInt32).device(in.device()));
    torch::Tensor out = torch::empty(in.sizes(), torch::TensorOptions().dtype(torch::kUInt8).device(in.device()));
    float* sp = scales.data_ptr<float>();
    const int dt = to_fp8b_dtype(in.scalar_type());
    check_status(fp8b_amax_scale(in.data_ptr(), dt, (size_t)in.numel(), sp, sp + 1,
                                 reinterpret_cast<uint32_t*>(scratch.data_ptr()), current_stream()),
                 "fp8b_amax_scale");
    check_status(fp8b_encode(in.data_ptr(), dt, static_cast<uint8_t*>(out.data_ptr()), (size_t)in.numel(), sp,
                             current_stream()),
                 "fp8b_encode");
    return std::make_tuple(out, scales.slice(0, 1, 2));
}

// Fused compute + exchange for the N-sharded linear: this rank's (M, N_local) block is stored through
// the NVSwitch multicast address `mc_ptr` (element (0,0) of the full row-major (M, full_N) matrix) at
// column offset n0, so it lands in every rank's copy.
void fp8_scaled_mm_multicast(torch::Tensor A, torch::Tensor B, torch::Tensor scale_a, torch::Tensor scale_b,
                             c10::optional<torch::Tensor> bias, at::ScalarType out_dtype,
                             int64_t mc_ptr, int64_t full_N, int64_t n0)
{
    check_fp8_pair(A, B);
    const int64_t M = A.size(0), K = A.size(1), N = B.size(0);
    const int odt = to_fp8b_dtype(out_dtype);                 // no float8_e4m3fn output through the multicast mapping
    void* c_mc = column_block(static_cast<uintptr_t>(mc_ptr), n0, N, full_N, c10::elementSize(out_dtype));
    const auto dev = A.device();
    c10::cuda::CUDAGuard guard(dev);
    const Scale sa = scale_arg(scale_a, dev, M, "scale_a must have 1 or M elements");
    const Scale sb = scale_arg(scale_b, dev, N, "scale_b must have 1 or N elements");
    const Bias b = bias_arg(bias, dev, N);
    check_status(fp8b_scaled_mm_multicast(u8_ptr(A), u8_ptr(B), c_mc, odt, (int)M, (int)N, (int)K, full_N, sa.ptr, sa.len,
                                          sb.ptr, sb.len, b.ptr, b.dtype, nullptr, current_stream()),
                 "fp8b_scaled_mm_multicast");
}

// Several independent M = 1 GEMVs (same K, same out dtype) in one launch: fp8b_gemv_batch.
std::vector<torch::Tensor> fp8_scaled_mm_many(std::vector<torch::Tensor> xs, std::vector<torch::Tensor> Ws,
                                              std::vector<torch::Tensor> scale_xs, std::vector<torch::Tensor> scale_ws,
                                              c10::optional<std::vector<torch::Tensor>> biases,
                                              c10::optional<at::ScalarType> out_dtype)
{
    const size_t n = Ws.size();
    TORCH_CHECK(xs.size() == n && scale_xs.size() == n && scale_ws.size() == n, "xs, Ws and the scale lists must have equal length");
    TORCH_CHECK(!biases.has_value() || biases->size() == n, "biases must have one entry per problem");
    std::vector<torch::Tensor> outs(n);
    if (n == 0) return outs;
    const auto dev = Ws[0].device();
    TORCH_CHECK(dev.is_cuda(), "operands must be CUDA tensors");
    c10::cuda::CUDAGuard guard(dev);
    const at::ScalarType odt = out_dtype.value_or(at::kFloat);
    const int64_t K = Ws[0].size(1);
    std::vector<torch::Tensor> keep;                              // converted scales / biases stay alive until the launch
    std::vector<fp8b_gemv_item> items(n);
    int bias_dt = FP8B_F32;
    bool bias_seen = false;
    for (size_t i = 0; i < n; ++i) {
        const torch::Tensor& x = xs[i];
        const torch::Tensor& W = Ws[i];
        check_fp8_operand(x, "x");
        check_fp8_operand(W, "W");
        TORCH_CHECK(x.device() == dev && W.device() == dev, "all operands must be on one device");
        TORCH_CHECK(W.dim() == 2 && W.size(1) == K && x.numel() == K, "every problem must have M = 1 and the same K");
        const int64_t N = W.size(0);
        const Scale sx = scale_arg(scale_xs[i], dev, 1, "scale_x must have 1 element");
        const Scale sw = scale_arg(scale_ws[i], dev, N, "scale_w must have 1 or N elements");
        // fp8_mps_native passes an empty tensor for a problem without bias
        const bool has_bias = biases.has_value() && (*biases)[i].defined() && (*biases)[i].numel() > 0;
        const Bias b = bias_arg(has_bias ? c10::optional<torch::Tensor>((*biases)[i]) : c10::nullopt, dev, N);
        if (b.ptr) {
            TORCH_CHECK(!bias_seen || b.dtype == bias_dt, "all biases must share one dtype");
            bias_dt = b.dtype; bias_seen = true;
        }
        keep.insert(keep.end(), {sx.keep, sw.keep, b.keep});
        outs[i] = torch::empty({1, N}, torch::TensorOptions().dtype(odt).device(dev));
        fp8b_gemv_item& q = items[i];
        q.x = u8_ptr(x); q.W = u8_ptr(W); q.y = outs[i].data_ptr(); q.N = (int)N;
        q.scale_x = sx.ptr; q.scale_w = sw.ptr; q.scale_w_len = sw.len;
        q.bias = b.ptr;
    }
    check_status(fp8b_gemv_batch(items.data(), (int)n, (int)K, to_fp8b_out_dtype(odt), bias_dt, current_stream()), "fp8b_gemv_batch");
    return outs;
}

// N-sharded linear with peer stores: `out` is this rank's full (M, full_N) symmetric buffer, `peer_deltas` a device
// int64[world] tensor of byte offsets from it to every rank's buffer (0 for this rank).
void fp8_scaled_mm_peers(torch::Tensor A, torch::Tensor B, torch::Tensor scale_a, torch::Tensor scale_b,
                         c10::optional<torch::Tensor> bias, torch::Tensor out, torch::Tensor peer_deltas, int64_t n0)
{
    check_fp8_pair(A, B);
    TORCH_CHECK(out.is_cuda() && out.dim() == 2 && out.is_contiguous() && out.size(0) == A.size(0), "out must be (M, full_N) contiguous");
    TORCH_CHECK(peer_deltas.is_cuda() && peer_deltas.scalar_type() == at::kLong && peer_deltas.is_contiguous(),
                "peer_deltas must be a contiguous CUDA int64 tensor");
    const int64_t M = A.size(0), K = A.size(1), N = B.size(0), full_N = out.size(1);
    void* c_local = column_block(reinterpret_cast<uintptr_t>(out.data_ptr()), n0, N, full_N, out.element_size());
    const auto dev = A.device();
    c10::cuda::CUDAGuard guard(dev);
    const Scale sa = scale_arg(scale_a, dev, M, "scale_a must have 1 or M elements");
    const Scale sb = scale_arg(scale_b, dev, N, "scale_b must have 1 or N elements");
    const Bias b = bias_arg(bias, dev, N);
    check_status(fp8b_scaled_mm_peers(u8_ptr(A), u8_ptr(B), c_local, peer_deltas.data_ptr<int64_t>(), (int)peer_deltas.numel(),
                                      to_fp8b_out_dtype(out.scalar_type()), (int)M, (int)N, (int)K, full_N, sa.ptr, sa.len,
                                      sb.ptr, sb.len, b.ptr, b.dtype, nullptr, current_stream()),
                 "fp8b_scaled_mm_peers");
}

// N-sharded linear, fused compute + exchange with TMA stores (fp8b_scaled_mm_push).  `out` is this rank's (M, full_N)
// buffer; `dst_ptrs` are the base addresses of the 1..8 destination buffers of that same geometry as mapped into this
// process (torch symmetric memory `buffer_ptrs`; this rank's own buffer among them), in the order they should be
// written.  The column block [n0, n0 + N) of every destination is written.
void fp8_scaled_mm_push(torch::Tensor A, torch::Tensor B, torch::Tensor scale_a, torch::Tensor scale_b,
                        c10::optional<torch::Tensor> bias, torch::Tensor out, std::vector<int64_t> dst_ptrs, int64_t n0,
                        std::vector<int64_t> signal_ptrs, c10::optional<torch::Tensor> cta_counter, int64_t epoch,
                        c10::optional<torch::Tensor> wait_flags, int64_t rank)
{
    check_fp8_pair(A, B);
    TORCH_CHECK(out.is_cuda() && out.dim() == 2 && out.is_contiguous() && out.size(0) == A.size(0), "out must be (M, full_N) contiguous");
    TORCH_CHECK(!dst_ptrs.empty() && dst_ptrs.size() <= 8, "need 1..8 destination buffers");
    const int64_t M = A.size(0), K = A.size(1), N = B.size(0), full_N = out.size(1);
    void* dsts[8];
    for (size_t d = 0; d < dst_ptrs.size(); ++d)
        dsts[d] = column_block(static_cast<uintptr_t>(dst_ptrs[d]), n0, N, full_N, out.element_size());
    const auto dev = A.device();
    c10::cuda::CUDAGuard guard(dev);
    const Scale sa = scale_arg(scale_a, dev, M, "scale_a must have 1 or M elements");
    const Scale sb = scale_arg(scale_b, dev, N, "scale_b must have 1 or N elements");
    const Bias b = bias_arg(bias, dev, N);
    const int n_dst = (int)dst_ptrs.size();
    const int odt = to_fp8b_out_dtype(out.scalar_type());
    if (signal_ptrs.empty()) {
        check_status(fp8b_scaled_mm_push(u8_ptr(A), u8_ptr(B), dsts, n_dst, odt, (int)M, (int)N, (int)K, full_N, sa.ptr, sa.len,
                                         sb.ptr, sb.len, b.ptr, b.dtype, nullptr, current_stream()),
                     "fp8b_scaled_mm_push");
        return;
    }
    // fused closing barrier: the kernel signals every peer when its last box has landed; fp8b_peer_wait (PDL) follows
    TORCH_CHECK(signal_ptrs.size() == dst_ptrs.size(), "one signal pointer per destination (0 for this rank)");
    TORCH_CHECK(cta_counter.has_value() && cta_counter->is_cuda() && cta_counter->scalar_type() == at::kInt, "cta_counter: CUDA int32[1]");
    TORCH_CHECK(wait_flags.has_value() && wait_flags->is_cuda() && wait_flags->scalar_type() == at::kLong, "wait_flags: CUDA int64");
    uint64_t* sig[8];
    for (int d = 0; d < n_dst; ++d) sig[d] = reinterpret_cast<uint64_t*>(static_cast<uintptr_t>(signal_ptrs[d]));
    check_status(fp8b_scaled_mm_push_signal(u8_ptr(A), u8_ptr(B), dsts, n_dst, odt, (int)M, (int)N, (int)K, full_N, sa.ptr, sa.len,
                                            sb.ptr, sb.len, b.ptr, b.dtype, nullptr, sig,
                                            reinterpret_cast<uint32_t*>(cta_counter->data_ptr()), (uint64_t)epoch, current_stream()),
                 "fp8b_scaled_mm_push_signal");
    check_status(fp8b_peer_wait(reinterpret_cast<const uint64_t*>(wait_flags->data_ptr()), n_dst, (int)rank, (uint64_t)epoch,
                                current_stream()),
                 "fp8b_peer_wait");
}

// per-row fp8_quantize of a 2-D tensor: returns (uint8 (rows, cols), inv_scale float32 [rows])
std::tuple<torch::Tensor, torch::Tensor> fp8_quantize_rowwise(torch::Tensor input)
{
    TORCH_CHECK(input.is_cuda(), "input must be a CUDA tensor");
    TORCH_CHECK(input.dim() == 2, "input must be 2-D (rows, cols)");
    c10::cuda::CUDAGuard guard(input.device());
    torch::Tensor in = float_input(input);
    torch::Tensor out = torch::empty(in.sizes(), torch::TensorOptions().dtype(torch::kUInt8).device(in.device()));
    torch::Tensor inv = torch::empty({in.size(0)}, torch::TensorOptions().dtype(torch::kFloat32).device(in.device()));
    check_status(fp8b_quantize_rows(in.data_ptr(), to_fp8b_dtype(in.scalar_type()), (int)in.size(0), (size_t)in.size(1),
                                    static_cast<uint8_t*>(out.data_ptr()), inv.data_ptr<float>(), current_stream()),
                 "fp8b_quantize_rows");
    return std::make_tuple(out, inv);
}

// Per-row fp8_quantize(x) -> scaled matmul in one library call (any M): x is float, B is uint8 (N,K).
// Returns (C, inv_scale_a[M]).
std::tuple<torch::Tensor, torch::Tensor> fp8_linear_dynamic(torch::Tensor x, torch::Tensor B, torch::Tensor scale_b,
                                                            c10::optional<torch::Tensor> bias,
                                                            c10::optional<at::ScalarType> out_dtype, bool single_kernel)
{
    check_fp8_operand(B, "B");
    TORCH_CHECK(x.is_cuda() && x.device() == B.device(), "x and B must be CUDA tensors on one device");
    TORCH_CHECK(x.dim() == 2 && B.dim() == 2 && x.size(1) == B.size(1), "K dimension mismatch between x and B");
    const auto dev = x.device();
    c10::cuda::CUDAGuard guard(dev);
    torch::Tensor xin = float_input(x);
    const int64_t M = xin.size(0), K = xin.size(1), N = B.size(0);
    const Scale sb = scale_arg(scale_b, dev, N, "scale_b must have 1 or N elements");
    const Bias b = bias_arg(bias, dev, N);
    const at::ScalarType odt = out_dtype.value_or(at::kFloat);
    torch::Tensor C = torch::empty({M, N}, torch::TensorOptions().dtype(odt).device(dev));
    torch::Tensor inv = torch::empty({M}, torch::TensorOptions().dtype(torch::kFloat32).device(dev));
    if (M == 0 || N == 0) return std::make_tuple(C, inv);
    torch::Tensor ws;
    void* ws_ptr = nullptr;
    size_t workspace_bytes = 0;
    if (!single_kernel) {
        workspace_bytes = fp8b_linear_dynamic_workspace_bytes((int)M, (int)K);
        ws = torch::empty({(int64_t)workspace_bytes}, torch::TensorOptions().dtype(torch::kUInt8).device(dev));
        ws_ptr = ws.data_ptr();
    }
    int rc = fp8b_linear_dynamic(xin.data_ptr(), to_fp8b_dtype(xin.scalar_type()), u8_ptr(B), C.data_ptr(), to_fp8b_out_dtype(odt),
                               (int)M, (int)N, (int)K, N, sb.ptr, sb.len, b.ptr, b.dtype, nullptr,
                               inv.data_ptr<float>(), ws_ptr, workspace_bytes, current_stream());
    check_status(rc, "fp8b_linear_dynamic");
    return std::make_tuple(C, inv);
}

int64_t select_algo(torch::Tensor A, torch::Tensor B, at::ScalarType out_dtype)
{
    return fp8b_scaled_mm_select(u8_ptr(A), u8_ptr(B), nullptr, to_fp8b_out_dtype(out_dtype), (int)A.size(0), (int)B.size(0),
                                 (int)A.size(1), B.size(0));
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m)
{
    m.doc() = "fp8_metal: B200 (sm_100a) kernels behind the fp8-mps-metal extension API";
    m.def("fp8_scaled_mm", &fp8_scaled_mm, "FP8 scaled matrix multiplication on the GPU",
          py::arg("A"), py::arg("B"), py::arg("scale_a"), py::arg("scale_b"));
    m.def("fp8_dequantize", &fp8_dequantize, "FP8 to float16 dequantization on the GPU",
          py::arg("input"), py::arg("scale"));
    m.def("fp8_quantize", &fp8_quantize, "Float to FP8 quantization on the GPU", py::arg("input"));
    m.def("fp8_linear_dynamic", &fp8_linear_dynamic, "Per-row dynamic quantize + FP8 matmul in one call",
          py::arg("x"), py::arg("B"), py::arg("scale_b"), py::arg("bias") = py::none(), py::arg("out_dtype") = py::none(),
          py::arg("single_kernel") = false);
    m.def("fp8_quantize_rowwise", &fp8_quantize_rowwise, "Per-row float to FP8 quantization", py::arg("input"));
    m.def("fp8_encode", &fp8_encode, "Float to FP8 encoding without scaling", py::arg("input"));
    m.def("fp8_encode_many", &fp8_encode_many, "Float to FP8 encoding of a list of tensors in one launch", py::arg("inputs"));
    m.def("fp8_dequantize_many", &fp8_dequantize_many, "FP8 to float cast of a list of tensors in one launch",
          py::arg("inputs"), py::arg("dtype"));
    m.def("fp8_dequantize_to", &fp8_dequantize_to, "FP8 (e4m3fn or e5m2) to float32/float16/bfloat16 exact cast",
          py::arg("input"), py::arg("dtype"), py::arg("format") = 0);
    m.def("fp8_scaled_mm_fused", &fp8_scaled_mm_fused,
          "FP8 scaled matmul with fused scales, bias, scale_result and output cast",
          py::arg("A"), py::arg("B"), py::arg("scale_a"), py::arg("scale_b"), py::arg("bias") = py::none(),
          py::arg("scale_result") = py::none(), py::arg("out_dtype") = py::none(), py::arg("algo") = 0,
          py::arg("out") = py::none(), py::arg("a_format") = 0, py::arg("b_format") = 0);
    m.def("scaled_mm_patch", &scaled_mm_patch, "torch._scaled_mm(input, other, ...) for FP8 operands, whole wrapper in C++",
          py::arg("input"), py::arg("other"), py::arg("scale_a") = py::none(), py::arg("scale_b") = py::none(),
          py::arg("bias") = py::none(), py::arg("scale_result") = py::none(), py::arg("out_dtype") = py::none());
    m.def("fp8_scaled_mm_multicast", &fp8_scaled_mm_multicast,
          "FP8 scaled matmul storing through an NVSwitch multicast address (N-sharded linear)",
          py::arg("A"), py::arg("B"), py::arg("scale_a"), py::arg("scale_b"), py::arg("bias"), py::arg("out_dtype"),
          py::arg("mc_ptr"), py::arg("full_N"), py::arg("n0"));
    m.def("fp8_scaled_mm_many", &fp8_scaled_mm_many, "Several independent M = 1 FP8 GEMVs of one K in one launch",
          py::arg("xs"), py::arg("Ws"), py::arg("scale_xs"), py::arg("scale_ws"), py::arg("biases") = py::none(),
          py::arg("out_dtype") = py::none());
    m.def("fp8_scaled_mm_peers", &fp8_scaled_mm_peers,
          "FP8 scaled matmul storing its tiles into every rank's symmetric buffer with peer stores (N-sharded linear)",
          py::arg("A"), py::arg("B"), py::arg("scale_a"), py::arg("scale_b"), py::arg("bias"), py::arg("out"),
          py::arg("peer_deltas"), py::arg("n0"));
    m.def("fp8_scaled_mm_push", &fp8_scaled_mm_push,
          "N-sharded linear: tcgen05 GEMM whose TMA-store epilogue pushes each tile into every destination buffer",
          py::arg("A"), py::arg("B"), py::arg("scale_a"), py::arg("scale_b"), py::arg("bias"), py::arg("out"),
          py::arg("dst_ptrs"), py::arg("n0"), py::arg("signal_ptrs") = std::vector<int64_t>(), py::arg("cta_counter") = py::none(),
          py::arg("epoch") = 0, py::arg("wait_flags") = py::none(), py::arg("rank") = 0);
    m.def("push_supported", [](int64_t M, int64_t N, int64_t K, int64_t ldc, at::ScalarType dt) {
        // alignment of torch allocations (>= 256 B) is assumed; this answers the shape part
        return fp8b_scaled_mm_push_supported(to_fp8b_out_dtype(dt), (int)M, (int)N, (int)K, ldc, nullptr, nullptr, nullptr) != 0;
    });
    m.def("select_algo", &select_algo, py::arg("A"), py::arg("B"), py::arg("out_dtype"));
    m.def("launch_count", []() { return (uint64_t)fp8b_launch_count(); });
    m.def("set_option", [](int option, int value) { check_status(fp8b_set_option(option, value), "fp8b_set_option"); });
    m.def("get_option", [](int option) { return fp8b_get_option(option); });
    m.attr("OPT_PDL") = (int)FP8B_OPT_PDL;
    m.attr("OPT_STATIC_WEIGHTS") = (int)FP8B_OPT_STATIC_WEIGHTS;
    m.def("version", []() { return fp8b_version(); });
    m.attr("FMT_E4M3FN") = (int)FP8B_E4M3FN;
    m.attr("FMT_E5M2") = (int)FP8B_E5M2;
    m.attr("ALGO_AUTO") = (int)FP8B_MM_AUTO;
    m.attr("ALGO_GEMV") = (int)FP8B_MM_GEMV;
    m.attr("ALGO_TCGEN05") = (int)FP8B_MM_TCGEN05;
    m.attr("ALGO_SIMT") = (int)FP8B_MM_SIMT;
}
