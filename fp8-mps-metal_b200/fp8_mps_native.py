"""
FP8 kernels behind the fp8-mps-metal kernel API, on B200 (sm_100a).

Same six entry points as the reference's ``fp8_mps_native`` module (fp8_mps_native.py:41,98,127,
158,193,213) with the same argument meaning, asserts and "inputs are moved to the accelerator"
behaviour.  Where the reference compiles a Metal shader with ``torch.mps.compile_shader`` and
launches it zero-copy on MPS buffers (fp8_mps_native.py:30-38), this module hands the tensors to
the ``fp8_metal`` torch extension (csrc/fp8_bridge.cpp), a thin binding to the C ABI of
``libfp8_b200.so`` (include/fp8_b200.h): hand-written CUDA for sm_100a, launched on the caller's
current stream with no host synchronisation.

There is no CPU fallback and no other backend: if the extension is not built, importing the
first kernel raises.  Build with ``python fp8-mps-metal_b200/build.py``.
"""

import os
import sys

import torch

_lib = None
_HERE = os.path.dirname(os.path.abspath(__file__))

#: device every entry point computes on (the reference hard-codes "mps")
DEVICE_TYPE = "cuda"


def _get_lib():
    """Get the compiled kernel library (singleton) -- the analogue of fp8_mps_native.py:30-38."""
    global _lib
    if _lib is not None:
        return _lib
    if _HERE not in sys.path:
        sys.path.insert(0, _HERE)
    try:
        import fp8_metal  # noqa: WPS433  (the in-tree extension, csrc/fp8_bridge.cpp)
    except ImportError as e:  # fail loudly: there is nothing to fall back to
        raise ImportError(
            "fp8_metal extension (B200 CUDA kernels) is not built or failed to load: "
            f"{e}.  Run `python {os.path.join(_HERE, 'build.py')}`."
        ) from e
    _lib = fp8_metal
    return _lib


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError("fp8_mps_native (B200 build) needs a CUDA device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _to_device(t: torch.Tensor) -> torch.Tensor:
    return t if t.device.type == DEVICE_TYPE else t.to(_device())


def set_static_weights(flag: bool) -> None:
    """Promise (or withdraw the promise) that weight matrices passed as B are never written by work still
    in flight on the stream.  The GEMV kernels then start streaming B before the preceding kernel has
    finished (programmatic dependent launch), which overlaps consecutive decode GEMVs.  Off by default;
    no reference counterpart."""
    lib = _get_lib()
    lib.set_option(lib.OPT_STATIC_WEIGHTS, 1 if flag else 0)


def fp8_scaled_mm(A: torch.Tensor, B: torch.Tensor,
                  scale_a: torch.Tensor, scale_b: torch.Tensor) -> torch.Tensor:
    """
    FP8 scaled matrix multiplication (reference: fp8_mps_native.py:41-95).

    A: (M, K) uint8 -- FP8 e4m3fn encoded, row-major
    B: (N, K) uint8 -- FP8 e4m3fn encoded, row-major (B is pre-transposed)
    scale_a: per-tensor [1] or per-row [M] float32
    scale_b: per-tensor [1] or per-row [N] float32

    Returns: (M, N) float32 on the GPU.  M <= 16 runs the streaming GEMV, larger M the tcgen05
    GEMM (the reference splits at M == 1, :78); scale lengths are independent (the reference's
    single scale_mode flag, :73, is not).
    """
    lib = _get_lib()

    assert A.dtype == torch.uint8 and B.dtype == torch.uint8
    assert A.is_contiguous() and B.is_contiguous()

    M, K = A.shape
    N = B.shape[0]
    assert B.shape[1] == K

    A = _to_device(A)
    B = _to_device(B)
    return lib.fp8_scaled_mm(A, B, scale_a, scale_b)


_FORMATS = {"e4m3fn": 0, "e5m2": 1, 0: 0, 1: 1, None: 0,
            getattr(torch, "float8_e4m3fn", "e4m3fn"): 0, getattr(torch, "float8_e5m2", "e5m2"): 1}


def fp8_scaled_mm_fused(A, B, scale_a, scale_b, bias=None, scale_result=None, out_dtype=None,
                        algo=0, out=None, a_format="e4m3fn", b_format="e4m3fn") -> torch.Tensor:
    """`fp8_scaled_mm` with the epilogue the patch applies as separate torch ops
    (fp8_mps_patch.py:95-104: + bias, * scale_result, .to(out_dtype)) fused into the kernel.
    ``out`` may be a row-major (M,N) view with a wider row stride (a column shard of a bigger
    matrix).  ``out_dtype=torch.float8_e4m3fn`` returns the reference encoder's bytes of the fp32 result, encoded in
    the same kernel (what ``fp8_encode`` of the float32 output gives, at a quarter of its output traffic); float8_e5m2
    is not an output dtype.  ``a_format`` / ``b_format``: "e4m3fn" (default; the reference codec, NaN bytes count as 0) or
    "e5m2" (decoded as e5m2 -- the reference mis-decodes such tensors as e4m3fn -- with IEEE inf/NaN)."""
    lib = _get_lib()
    assert A.dtype == torch.uint8 and B.dtype == torch.uint8
    assert A.is_contiguous() and B.is_contiguous()
    assert B.shape[1] == A.shape[1]
    return lib.fp8_scaled_mm_fused(_to_device(A), _to_device(B), scale_a, scale_b, bias, scale_result,
                                   out_dtype, algo, out, _FORMATS[a_format], _FORMATS[b_format])


def scaled_mm_patch(input, other, scale_a=None, scale_b=None, bias=None, scale_result=None, out_dtype=None):
    """`torch._scaled_mm(input, other, ...)` for FP8 operands on the GPU, the whole wrapper in one extension call
    (what fp8_mps_patch._metal_scaled_mm dispatches to).  input (M,K), other (K,N) uint8 / float8_e4m3fn /
    float8_e5m2; scales default to 1 (fp8_mps_patch.py:87-90); out_dtype None -> float32 (:103-104)."""
    return _get_lib().scaled_mm_patch(input, other, scale_a, scale_b, bias, scale_result, out_dtype)


def fp8_scaled_mm_many(xs, Ws, scale_xs, scale_ws, biases=None, out_dtype=None):
    """Several independent decode GEMVs in ONE launch: ``[fp8_scaled_mm_fused(x, W, sx, sw, bias, None, out_dtype)
    for ...]`` for M = 1 problems that share K (the Q/K/V or gate/up projections of a layer; the x may be the same
    tensor).  A C2-sized GEMV spends a third of its time in launch ramp-up and drain; sharing the launch pays that
    once.  xs: list of (1,K) uint8; Ws: list of (N_i,K) uint8; scale_xs: list of 1-element tensors; scale_ws: list of
    1- or N_i-element tensors; biases: optional list (entries may be None).  Returns a list of (1,N_i) tensors."""
    lib = _get_lib()
    if biases is not None:
        biases = [b if b is not None else torch.empty(0) for b in biases]
    return lib.fp8_scaled_mm_many([_to_device(x) for x in xs], [_to_device(W) for W in Ws], list(scale_xs), list(scale_ws),
                                  biases, out_dtype)


def fp8_dequantize(input: torch.Tensor, scale: torch.Tensor) -> torch.Tensor:
    """
    FP8 -> half dequantization (reference: fp8_mps_native.py:98-124).

    input: uint8 tensor (FP8 e4m3fn encoded)
    scale: scalar float32 tensor
    Returns: float16 tensor on the GPU, scaled: RN16(half(dec(b)) * RN16(scale)), one pass.
    """
    lib = _get_lib()
    input = _to_device(input)
    return lib.fp8_dequantize(input, scale)


def fp8_dequantize_to(input: torch.Tensor, dtype: torch.dtype, format="e4m3fn") -> torch.Tensor:
    """FP8 -> float32/float16/bfloat16 exact cast in one pass (what the patch's scenario 3 does
    in two, fp8_mps_patch.py:213-221).  ``format="e5m2"`` decodes float8_e5m2 bytes (exact, inf/NaN kept)."""
    lib = _get_lib()
    return lib.fp8_dequantize_to(_to_device(input), dtype, _FORMATS[format])


def fp8_encode(input: torch.Tensor):
    """
    Float -> FP8 encoding without scaling (reference: fp8_mps_native.py:127-155).

    Values are clamped to [-448, 448] but NOT scaled.  float32/float16/bfloat16 inputs are read
    in their own dtype (the reference converts to float32 in a separate pass, :142).
    Returns: uint8 tensor on the GPU (FP8 encoded), bit-identical to the reference's shader.
    """
    lib = _get_lib()
    inp = _to_device(input)
    return lib.fp8_encode(inp)


def fp8_encode_many(inputs):
    """`fp8_encode` of a list of tensors (a checkpoint's weights) in ONE launch per input dtype instead of one
    launch per tensor: the tensors are streamed as a single tile list, so HBM stays saturated across tensor
    boundaries.  Returns a list of uint8 tensors, bit-identical to ``[fp8_encode(t) for t in inputs]``."""
    lib = _get_lib()
    return lib.fp8_encode_many([_to_device(t) for t in inputs])


def fp8_dequantize_many(inputs, dtype: torch.dtype = torch.float16):
    """`fp8_dequantize_to` of a list of uint8 tensors in one launch (unscaled exact cast)."""
    lib = _get_lib()
    return lib.fp8_dequantize_many([_to_device(t) for t in inputs], dtype)


def fp8_quantize(input: torch.Tensor):
    """
    Float -> FP8 quantization with automatic scaling (reference: fp8_mps_native.py:158-190).

    scale = 448/amax is computed ON THE DEVICE in double precision (the reference syncs the
    host with .item(), :174); the multiply and encode are fused into one pass.
    Returns: (uint8 tensor, inverse_scale float32[1]) on the GPU.
    """
    lib = _get_lib()
    inp = _to_device(input)
    return lib.fp8_quantize(inp)


def fp8_quantize_rowwise(input: torch.Tensor):
    """
    Per-row (per-channel) `fp8_quantize`: the reference's amax -> 448/amax -> encode arithmetic
    (fp8_mps_native.py:158-190) applied to each row of a 2-D tensor in one launch.

    Returns: (uint8 (rows, cols), inverse scales float32 [rows]) -- the second is directly usable as a
    per-row ``scale_a`` / ``scale_b`` of ``fp8_scaled_mm`` (the reference kernels' scale_mode 1,
    fp8_matmul.metal:144-145, which the reference itself never feeds).
    """
    lib = _get_lib()
    return lib.fp8_quantize_rowwise(_to_device(input))


def fp8_linear_dynamic(x: torch.Tensor, B: torch.Tensor, scale_b: torch.Tensor, bias=None, out_dtype=None,
                       single_kernel: bool = False):
    """
    Linear layer with dynamic per-row activation quantisation in one library call, no host sync (any M):

        q, inv = fp8_quantize(x[m])  per row        (fp8_mps_native.py:158-190)
        y = ((dec(q) @ dec(B).T) * inv) * scale_b (+ bias) -> out_dtype

    i.e. what a caller of the reference writes as ``q, s = fp8_quantize(x); torch._scaled_mm(q8, w8.t(),
    scale_a=s, scale_b=...)`` -- five launches and a host sync there.  x: (M,K) float32/float16/bfloat16;
    B: (N,K) uint8.  Returns (y, inv_scale_a[M]).

    Default plan: a one-CTA-per-row quantise kernel, then the GEMV (M <= 16, chained by programmatic dependent
    launch) or the tcgen05 GEMM (M > 16) with per-row scale_a.  ``single_kernel=True`` (M <= 16 only) quantises
    inside every GEMV CTA instead: no scratch buffer, worthwhile for small N only.  Same result bits.
    """
    lib = _get_lib()
    assert B.dtype == torch.uint8 and B.is_contiguous() and x.shape[1] == B.shape[1]
    return lib.fp8_linear_dynamic(_to_device(x), _to_device(B), scale_b, bias, out_dtype, single_kernel)


def fp8_scaled_mm_auto(A: torch.Tensor, B: torch.Tensor,
                       scale_a: torch.Tensor, scale_b: torch.Tensor) -> torch.Tensor:
    """Auto-select the matmul kernel from the shape (reference: fp8_mps_native.py:193-210):
    M <= 16 -> GEMV, else the tcgen05 GEMM (SIMT kernel when TMA alignment rules fail)."""
    return fp8_scaled_mm(A, B, scale_a, scale_b)


def fp8_scaled_mm_fast(A: torch.Tensor, B: torch.Tensor,
                       scale_a: torch.Tensor, scale_b: torch.Tensor) -> torch.Tensor:
    """The reference's large-M route (fp8_mps_native.py:213-267: dequantise to fp16 + fp16 GEMM).
    Here it forces the tensor-core kernel for any M; scales are applied in fp32 in the epilogue,
    so per-row scales work (the reference's fp16 pre-scaling mis-broadcasts them, :258-261)."""
    lib = _get_lib()
    assert A.dtype == torch.uint8 and B.dtype == torch.uint8
    A = _to_device(A).contiguous()
    B = _to_device(B).contiguous()
    algo = lib.select_algo(A, B, torch.float32)
    if algo == lib.ALGO_GEMV:                      # M <= 16: still honour "fast" = tensor cores if TMA-able
        A16 = (A.shape[1] % 16 == 0) and A.data_ptr() % 16 == 0 and B.data_ptr() % 16 == 0
        algo = lib.ALGO_TCGEN05 if A16 else lib.ALGO_GEMV
    return lib.fp8_scaled_mm_fused(A, B, scale_a, scale_b, None, None, None, algo, None, 0, 0)
