"""
Interception layer: route FP8 work on the accelerator through the B200 kernels.

Same public surface as the reference's ``fp8_mps_patch`` (fp8_mps_patch.py:443-497):

    import fp8_mps_patch
    fp8_mps_patch.install()     # swaps torch._scaled_mm, Tensor.to, Tensor.copy_
    fp8_mps_patch.uninstall()   # restores them
    fp8_mps_patch.is_installed()

and the same module-level names the reference's tests read: ``_original_scaled_mm``,
``_original_tensor_to``, ``_original_tensor_copy`` (test_fp8_metal.py:337-341, :558-563),
``_metal_scaled_mm``, ``_metal_tensor_to``, ``_metal_tensor_copy``,
``patch_vae_decode_for_mps_limits`` (test_mps_limits_patch.py:135-143).  The wrappers keep the
reference's decision structure -- "is this FP8 on the accelerator?  route to the kernels : call the
original" -- with the accelerator being CUDA (sm_100a) instead of MPS.

Deliberate differences from the reference (SURVEY Appendix B):
  * ``_metal_scaled_mm`` accepts scales positionally (the real aten schema) as well as by keyword
    (reference: keyword-only, fp8_mps_patch.py:53);
  * bias, scale_result and out_dtype are fused into the matmul kernel instead of three extra
    elementwise passes (fp8_mps_patch.py:95-104); out_dtype=float8_e4m3fn gives the bytes the reference's
    ``result.to(float8_e4m3fn)`` gives, encoded in the same kernel (float8_e5m2 output raises);
  * float8_e5m2 operands are decoded AS e5m2 (the reference sends them to its e4m3fn kernels and
    mis-decodes them, fp8_mps_patch.py:48-49,65); only decode exists: float -> e5m2 stays with torch;
  * FP8 -> float32/bfloat16 is one exact pass, not dequantise-to-fp16 then .to();
  * the VAE-decode tiling (fp8_mps_patch.py:305-440) works around an MPSGraph tensor-size limit
    that CUDA does not have; the symbol is kept and is a no-op.
"""

import os

import torch

try:  # ComfyUI is optional (fp8_mps_patch.py:19-23)
    import comfy.sd  # noqa: F401
    _COMFY_AVAILABLE = True
except ImportError:
    _COMFY_AVAILABLE = False

# Kept for API compatibility with the reference (fp8_mps_patch.py:32,36); unused on CUDA.
MPS_TENSOR_SIZE_THRESHOLD = 15_000_000
VAE_UPSCALE_FACTOR = 64

#: device type the wrappers intercept (the reference: "mps")
ACCEL = "cuda"

_original_scaled_mm = None
_original_tensor_to = None
_original_tensor_copy = None
_installed = False

_E4M3 = getattr(torch, "float8_e4m3fn", None)
_E5M2 = getattr(torch, "float8_e5m2", None)


def _is_fp8_dtype(dtype):
    """True for either torch FP8 dtype (fp8_mps_patch.py:44-50)."""
    return dtype is not None and (dtype == _E4M3 or dtype == _E5M2)


def _kernels():
    import fp8_mps_native  # lazy, like the reference (fp8_mps_patch.py:74)
    return fp8_mps_native


def _device_type(device):
    if device is None:
        return None
    if isinstance(device, torch.device):
        return device.type
    if isinstance(device, str):
        return device.split(":", 1)[0]
    if isinstance(device, int) and not isinstance(device, bool):
        return ACCEL                                   # a bare ordinal names an accelerator device, as in torch
    return None


def _as_device(device):
    """str / int / torch.device -> torch.device (the reference only ever saw the single "mps" device)."""
    if isinstance(device, int) and not isinstance(device, bool):
        return torch.device(ACCEL, device)
    return torch.device(device)


def _same_accel_device(tensor, device):
    """`device` (None, str or torch.device) names the accelerator device `tensor` already lives on."""
    if device is None:
        return True
    d = _as_device(device)
    if d.type != tensor.device.type:
        return False
    index = d.index if d.index is not None else torch.cuda.current_device()
    return index == tensor.device.index


# --------------------------------------------------------------------------- _scaled_mm

_SCALED_MM_POSITIONAL = ("scale_a", "scale_b", "bias", "scale_result", "out_dtype", "use_fast_accum")
_FP8_DTYPES = frozenset(d for d in (_E4M3, _E5M2) if d is not None)
_FP8_LIKE = frozenset(d for d in (torch.uint8, _E4M3, _E5M2) if d is not None)     # fp8_mps_patch.py:64-65
_scaled_mm_patch_fn = None


def _bind_kernel():
    """Resolve the extension's scaled_mm_patch once (the import is lazy, like the reference's, fp8_mps_patch.py:74)."""
    global _scaled_mm_patch_fn
    _scaled_mm_patch_fn = _kernels()._get_lib().scaled_mm_patch       # the extension function itself, no Python layer between
    return _scaled_mm_patch_fn


def _metal_scaled_mm(input, other, *args, out_dtype=None, scale_a=None, scale_b=None, bias=None,
                     scale_result=None, use_fast_accum=False):
    """
    Drop-in replacement for torch._scaled_mm for FP8 operands on the GPU.

    input: (M, K) activation, uint8 / float8_e4m3fn / float8_e5m2
    other: (K, N) weight, normally column-major so that other.t() is the (N, K) row-major
           layout the kernels take (fp8_mps_patch.py:82-84)
    Result: ((sum_k a*b) * scale_a) * scale_b [+ bias] [* scale_result], cast to out_dtype
            (float32 when out_dtype is None, fp8_mps_patch.py:103-104).
    """
    # Hot path first, with as little Python as possible (a decode GEMV runs 5-12 us on the GPU; this wrapper is
    # called once per linear layer): FP8 operands on the accelerator go straight to ONE extension call.
    if input.is_cuda and input.dtype in _FP8_LIKE and other.dtype in _FP8_LIKE:
        n = len(args)
        if n:                                          # aten schema order: scale_a, scale_b, bias, scale_result, out_dtype
            if n > len(_SCALED_MM_POSITIONAL):
                raise TypeError(f"_scaled_mm() takes at most {2 + len(_SCALED_MM_POSITIONAL)} positional arguments")
            scale_a = args[0]
            if n > 1:
                scale_b = args[1]
                if n > 2:
                    bias = args[2]
                    if n > 3:
                        scale_result = args[3]
                        if n > 4:
                            out_dtype = args[4]
        # dtype views, the (N,K) view of `other`, default scales (fp8_mps_patch.py:82-90) and the fused epilogue
        # (:95-104) all happen inside that call.  float8_e5m2 operands are decoded as e5m2; uint8 is taken as e4m3fn.
        return (_scaled_mm_patch_fn or _bind_kernel())(input, other, scale_a, scale_b, bias, scale_result, out_dtype)

    kw = dict(out_dtype=out_dtype, scale_a=scale_a, scale_b=scale_b, bias=bias,
              scale_result=scale_result, use_fast_accum=use_fast_accum)
    if len(args) > len(_SCALED_MM_POSITIONAL):
        raise TypeError(f"_scaled_mm() takes at most {2 + len(_SCALED_MM_POSITIONAL)} positional arguments")
    for name, value in zip(_SCALED_MM_POSITIONAL, args):      # aten schema order
        kw[name] = value
    return _original_scaled_mm(input, other, **kw)             # not FP8-on-accelerator: the reference's predicate (:64-65)


# --------------------------------------------------------------------------- Tensor.to

def _parse_to_args(args, kwargs):
    """dtype / device out of the many call forms of Tensor.to (fp8_mps_patch.py:119-133)."""
    dtype = kwargs.get("dtype")
    device = kwargs.get("device")
    for pos, arg in enumerate(args):
        if isinstance(arg, torch.dtype):
            if dtype is None:
                dtype = arg
        elif isinstance(arg, (torch.device, str)):
            if device is None:
                device = arg
        elif pos == 0 and isinstance(arg, int) and not isinstance(arg, bool):
            if device is None:
                device = arg                               # to(0, dtype): a device ordinal (later ints are non_blocking / copy)
        elif isinstance(arg, torch.Tensor) and dtype is None and device is None:
            dtype, device = arg.dtype, arg.device          # to(other_tensor)
    return dtype, device


def _metal_tensor_to(self, *args, **kwargs):
    """
    Drop-in replacement for Tensor.to() handling FP8 on the GPU (fp8_mps_patch.py:109-226):

    1. FP8 tensor elsewhere -> GPU: raw byte transfer, dtype preserved;
    2. float tensor -> FP8 on the GPU: encode with the reference codec (no scaling);
    3. FP8 tensor on the GPU: no-op, FP8<->FP8 reinterpretation, or exact dequantise.
    Everything else goes to the original method untouched.
    """
    # Fast exit for the overwhelmingly common call that involves no FP8 at all: this wrapper sits on EVERY Tensor.to()
    # in the process (a10 in SURVEY 8a), so the non-FP8 path must cost next to nothing.
    if self.dtype not in _FP8_DTYPES and kwargs.get("dtype") is not _E4M3:
        for a in args:
            if a is _E4M3:
                break
            if isinstance(a, torch.Tensor) and a.dtype is _E4M3:
                break
        else:
            return _original_tensor_to(self, *args, **kwargs)
    dtype, device = _parse_to_args(args, kwargs)
    src_fp8 = _is_fp8_dtype(self.dtype)
    dst_fp8 = _is_fp8_dtype(dtype)
    dst_type = _device_type(device)
    target_on_accel = (dst_type == ACCEL) if device is not None else (self.device.type == ACCEL)
    passthrough = {k: v for k, v in kwargs.items() if k not in ("device", "dtype")}

    # 1. FP8 bytes moving onto the accelerator
    if src_fp8 and device is not None and target_on_accel and self.device.type != ACCEL:
        moved = _original_tensor_to(self.view(torch.uint8), _as_device(device), **passthrough).view(self.dtype)
        if dtype is not None and dtype != self.dtype:
            if dst_fp8:
                return moved.view(torch.uint8).view(dtype)
            return _metal_tensor_to(moved, dtype)
        return moved

    # 2. float -> FP8 on the accelerator (only e4m3fn has kernels; e5m2 stays with torch).  The tensor is first
    #    moved to the REQUESTED device -- which may be another GPU than the one it lives on -- then encoded there.
    if target_on_accel and dtype is not None and dtype == _E4M3 and not src_fp8:
        if self.device.type == ACCEL and _same_accel_device(self, device):
            on_dev = self
        else:
            on_dev = _original_tensor_to(self, _as_device(device) if device is not None else ACCEL, **passthrough)
        return _kernels().fp8_encode(on_dev).view(dtype)

    # 3. FP8 already on the accelerator
    if src_fp8 and self.device.type == ACCEL and (device is None or target_on_accel):
        if _same_accel_device(self, device):
            if dtype is None or dtype == self.dtype:
                return self
            if dst_fp8:
                return self.view(torch.uint8).view(dtype)
            if dtype in (torch.float32, torch.float16, torch.bfloat16):
                return _kernels().fp8_dequantize_to(self.view(torch.uint8), dtype,
                                                    format="e5m2" if self.dtype == _E5M2 else "e4m3fn")

    return _original_tensor_to(self, *args, **kwargs)


# --------------------------------------------------------------------------- Tensor.copy_

def _metal_tensor_copy(self, src, non_blocking=False):
    """
    Drop-in replacement for Tensor.copy_() for FP8 destinations on the GPU
    (fp8_mps_patch.py:229-302): FP8 -> FP8 is a byte copy, also between the two FP8 dtypes (:245-264); any
    non-FP8 source -> float8_e4m3fn encodes with the reference codec (:266-290; non-float sources go through
    float32 first like fp8_encode, fp8_mps_native.py:142).  A float8_e5m2 destination with a non-FP8 source stays
    with torch's own cast (the reference would store e4m3fn codes in it; DESIGN.md section 5).  Everything else goes
    to the original method.
    """
    # fast exit: only FP8 destinations on the accelerator are intercepted (this wrapper sits on every copy_())
    if self.dtype not in _FP8_DTYPES or not self.is_cuda or not hasattr(src, "dtype"):
        return _original_tensor_copy(self, src, non_blocking=non_blocking)
    src_fp8 = _is_fp8_dtype(src.dtype)

    if src_fp8:
        _original_tensor_copy(self.view(torch.uint8), src.contiguous().view(torch.uint8), non_blocking=non_blocking)
        return self

    if self.dtype == _E4M3:
        on_dev = src if src.device == self.device else _original_tensor_to(src, self.device)
        encoded = _kernels().fp8_encode(on_dev)
        _original_tensor_copy(self.view(torch.uint8), encoded, non_blocking=non_blocking)
        return self

    return _original_tensor_copy(self, src, non_blocking=non_blocking)


# --------------------------------------------------------------------------- VAE decode (stub)

def patch_vae_decode_for_mps_limits():
    """The reference tiles huge VAE decodes to stay under MPSGraph's INT_MAX tensor limit
    (fp8_mps_patch.py:362-440).  CUDA has no such limit, so nothing is patched."""
    if not _COMFY_AVAILABLE:
        print("[fp8-mps-metal] ComfyUI not available, skipping VAE decode patch")
        return
    print("[fp8-mps-metal] CUDA backend: VAE decode needs no tensor-size tiling, nothing patched")


# --------------------------------------------------------------------------- install / uninstall

def install():
    """Monkey-patch torch._scaled_mm, Tensor.to() and Tensor.copy_() (fp8_mps_patch.py:443-471)."""
    global _original_scaled_mm, _original_tensor_to, _original_tensor_copy, _installed
    if _installed:
        return

    # The reference sets this for MPS (fp8_mps_patch.py:451) and its tests assert it
    # (test_mps_limits_patch.py:50-56); it is inert on CUDA.
    os.environ["PYTORCH_ENABLE_MPS_FALLBACK"] = "1"

    if not hasattr(torch, "_scaled_mm"):
        raise RuntimeError("torch._scaled_mm not found — requires PyTorch 2.4+")
    _original_scaled_mm = torch._scaled_mm
    torch._scaled_mm = _metal_scaled_mm

    _original_tensor_to = torch.Tensor.to
    torch.Tensor.to = _metal_tensor_to

    _original_tensor_copy = torch.Tensor.copy_
    torch.Tensor.copy_ = _metal_tensor_copy

    patch_vae_decode_for_mps_limits()
    _installed = True


def uninstall():
    """Restore the three originals (fp8_mps_patch.py:474-492)."""
    global _original_scaled_mm, _original_tensor_to, _original_tensor_copy, _installed
    if not _installed:
        return
    if _original_scaled_mm is not None:
        torch._scaled_mm = _original_scaled_mm
        _original_scaled_mm = None
    if _original_tensor_to is not None:
        torch.Tensor.to = _original_tensor_to
        _original_tensor_to = None
    if _original_tensor_copy is not None:
        torch.Tensor.copy_ = _original_tensor_copy
        _original_tensor_copy = None
    _installed = False


def is_installed():
    """Whether the monkey-patch is active (fp8_mps_patch.py:495-497)."""
    return _installed
