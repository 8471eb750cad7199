"""Shared helpers for the tests: ctypes view of the C ABI, torch<->numpy glue."""
import ctypes
import os
import re

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "fp8-mps-metal_b200")
LIB_PATH = os.environ.get("FP8B_LIB") or os.path.join(PKG, "libfp8_b200.so")    # FP8B_LIB: A/B a differently built library
HEADER = os.path.join(ROOT, "include", "fp8_b200.h")

F32, F16, BF16 = 0, 1, 2
ALGO_AUTO, ALGO_GEMV, ALGO_TCGEN05, ALGO_SIMT = 0, 1, 2, 3

_lib = None

DEV = "cuda"
GUARD_ROWS = 3
SENT = {torch.float32: 0x7FA5A5A5, torch.float16: 0x7DA5, torch.bfloat16: 0x7FA5}    # NaN payloads no kernel writes
_INT = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}
BIG_SCALE = 1024.0                                    # what sits behind per-row scales


def declared_symbols():
    """Every function include/fp8_b200.h declares (the FP8B_API lines)."""
    src = open(HEADER).read()
    return re.findall(r"FP8B_API\s+[\w\s\*]+?\b(fp8b_\w+)\s*\(", src)


def capi():
    """libfp8_b200.so through ctypes, with argument types set."""
    global _lib
    if _lib is not None:
        return _lib
    L = ctypes.CDLL(LIB_PATH)
    vp, sz, i32, i64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int64
    L.fp8b_version.restype = i32
    L.fp8b_status_string.restype = ctypes.c_char_p
    L.fp8b_status_string.argtypes = [i32]
    L.fp8b_last_cuda_error.restype = i32
    L.fp8b_launch_count.restype = ctypes.c_uint64
    L.fp8b_set_option.restype = i32
    L.fp8b_set_option.argtypes = [i32, i32]
    L.fp8b_get_option.restype = i32
    L.fp8b_get_option.argtypes = [i32]
    L.fp8b_dequant_f16.restype = i32
    L.fp8b_dequant_f16.argtypes = [vp, vp, sz, vp, vp]
    L.fp8b_dequant.restype = i32
    L.fp8b_dequant.argtypes = [vp, vp, i32, sz, vp]
    L.fp8b_encode.restype = i32
    L.fp8b_encode.argtypes = [vp, i32, vp, sz, vp, vp]
    L.fp8b_amax_scale.restype = i32
    L.fp8b_amax_scale.argtypes = [vp, i32, sz, vp, vp, vp, vp]
    L.fp8b_quantize_rows.restype = i32
    L.fp8b_quantize_rows.argtypes = [vp, i32, i32, sz, vp, vp, vp]
    L.fp8b_scaled_mm.restype = i32
    L.fp8b_scaled_mm.argtypes = [vp, vp, vp, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, i32, vp, vp, sz, i32, vp]
    L.fp8b_scaled_mm_multicast.restype = i32
    L.fp8b_scaled_mm_multicast.argtypes = [vp, vp, vp, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, i32, vp, vp]
    L.fp8b_scaled_mm_workspace_bytes.restype = sz
    L.fp8b_scaled_mm_workspace_bytes.argtypes = [i32, i32, i32]
    L.fp8b_scaled_mm_select.restype = i32
    L.fp8b_scaled_mm_select.argtypes = [vp, vp, vp, i32, i32, i32, i32, i64]
    if hasattr(L, "fp8b_gemv_batch") or not os.environ.get("FP8B_LIB"):
        L.fp8b_gemv_batch.restype = i32
        L.fp8b_gemv_batch.argtypes = [vp, i32, i32, i32, i32, vp]
    if hasattr(L, "fp8b_scaled_mm_fmt") or not os.environ.get("FP8B_LIB"):
        L.fp8b_scaled_mm_fmt.restype = i32
        L.fp8b_scaled_mm_fmt.argtypes = [vp, i32, vp, i32, vp, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, i32, vp, i32, vp]
        L.fp8b_dequant_fmt.restype = i32
        L.fp8b_dequant_fmt.argtypes = [vp, i32, vp, i32, sz, vp, vp]
    if hasattr(L, "fp8b_encode_batch") or not os.environ.get("FP8B_LIB"):
        L.fp8b_encode_batch.restype = i32
        L.fp8b_encode_batch.argtypes = [vp, i32, i32, vp]
        L.fp8b_dequant_batch.restype = i32
        L.fp8b_dequant_batch.argtypes = [vp, i32, i32, vp]
    if hasattr(L, "fp8b_linear_dynamic") or not os.environ.get("FP8B_LIB"):   # (an older A/B build may lack it)
        L.fp8b_linear_dynamic.restype = i32
        L.fp8b_linear_dynamic.argtypes = [vp, i32, vp, vp, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, vp, vp, sz, vp]
        L.fp8b_linear_dynamic_workspace_bytes.restype = sz
        L.fp8b_linear_dynamic_workspace_bytes.argtypes = [i32, i32]
    if hasattr(L, "fp8b_scaled_mm_push") or not os.environ.get("FP8B_LIB"):
        L.fp8b_scaled_mm_peers.restype = i32
        L.fp8b_scaled_mm_peers.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, i32, vp, vp]
        L.fp8b_scaled_mm_push.restype = i32
        L.fp8b_scaled_mm_push.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, i32,
                                          vp, vp]
        L.fp8b_scaled_mm_push_signal.restype = i32
        L.fp8b_scaled_mm_push_signal.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i64, vp, i32, vp, i32, vp, i32, vp,
                                                 vp, vp, i64, vp]
        L.fp8b_peer_wait.restype = i32
        L.fp8b_peer_wait.argtypes = [vp, i32, i32, i64, vp]
        L.fp8b_scaled_mm_push_supported.restype = i32
        L.fp8b_scaled_mm_push_supported.argtypes = [i32, i32, i32, i32, i64, vp, vp, vp]
    _lib = L
    return L


class Span(ctypes.Structure):
    """fp8b_span (include/fp8_b200.h)"""
    _fields_ = [("inp", ctypes.c_void_p), ("out", ctypes.c_void_p), ("n", ctypes.c_size_t)]


class GemvItem(ctypes.Structure):
    """fp8b_gemv_item (include/fp8_b200.h)"""
    _fields_ = [("x", ctypes.c_void_p), ("W", ctypes.c_void_p), ("y", ctypes.c_void_p), ("N", ctypes.c_int),
                ("scale_x", ctypes.c_void_p), ("scale_w", ctypes.c_void_p), ("scale_w_len", ctypes.c_int),
                ("bias", ctypes.c_void_p)]


def make_spans(triples):
    arr = (Span * max(1, len(triples)))()
    for i, (a, b, n) in enumerate(triples):
        arr[i].inp, arr[i].out, arr[i].n = a, b, n
    return arr


def dt_code(torch_dtype):
    import torch
    return {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}[torch_dtype]


def dt_name(torch_dtype):
    import torch
    return {torch.float32: "f32", torch.float16: "f16", torch.bfloat16: "bf16", None: "f32"}[torch_dtype]


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def p(t):
    """device pointer of a torch tensor (or None)."""
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def mm_capi(A, B, sa, sb, bias=None, sr=None, out_dtype=None, algo=ALGO_AUTO, out=None):
    """fp8b_scaled_mm through the raw C ABI on torch CUDA tensors."""
    import torch
    L = capi()
    M, K = A.shape
    N = B.shape[0]
    odt = out_dtype or torch.float32
    C = out if out is not None else torch.empty(M, N, dtype=odt, device=A.device)
    ldc = C.stride(0) if C.dim() == 2 and M > 0 else N
    sa = sa.to(device=A.device, dtype=torch.float32).contiguous().reshape(-1)
    sb = sb.to(device=A.device, dtype=torch.float32).contiguous().reshape(-1)
    rc = L.fp8b_scaled_mm(p(A), p(B), p(C), dt_code(odt), M, N, K, ldc, p(sa), sa.numel(), p(sb), sb.numel(),
                          p(bias), dt_code(bias.dtype) if bias is not None else 0, p(sr), None, 0, algo, stream_ptr())
    return rc, C


def mm_push_capi(A, B, sa, sb, dsts, n0=0, bias=None, sr=None):
    """fp8b_scaled_mm_push through the raw C ABI: `dsts` are (M, ldc) torch tensors of one dtype and geometry; this
    call writes the column block [n0, n0 + N) of each."""
    import torch
    L = capi()
    M, K = A.shape
    N = B.shape[0]
    odt = dsts[0].dtype
    ldc = dsts[0].stride(0)
    esz = dsts[0].element_size()
    arr = (ctypes.c_void_p * len(dsts))(*[d.data_ptr() + n0 * esz for d in dsts])
    sa = sa.to(device=A.device, dtype=torch.float32).contiguous().reshape(-1)
    sb = sb.to(device=A.device, dtype=torch.float32).contiguous().reshape(-1)
    return L.fp8b_scaled_mm_push(p(A), p(B), arr, len(dsts), dt_code(odt), M, N, K, ldc, p(sa), sa.numel(), p(sb), sb.numel(),
                                 p(bias), dt_code(bias.dtype) if bias is not None else 0, p(sr), stream_ptr())


def to_np(t):
    """torch tensor (any float dtype, any device) -> float32 numpy, exactly."""
    return t.detach().float().cpu().numpy()


def u8_np(t):
    import torch
    return t.detach().view(torch.uint8).cpu().numpy()


# ------------------------------------------------------------------ device buffers with guard bands

class Out:
    """C as an interior view of a sentinel-filled buffer: GUARD_ROWS rows above and below, `cl` columns left and at
    least 8 right.  aligned=True keeps the view 16-byte aligned with ldc * esz % 16 == 0 (the vector / TMA store
    paths); False shifts it by one element and makes ldc odd (the scalar store paths)."""

    def __init__(self, M, N, dtype, aligned=True, cl=None):
        esz = torch.empty(0, dtype=dtype).element_size()
        self.dtype, self.M, self.N = dtype, M, N
        self.cl = (16 // esz if aligned else 1) if cl is None else cl
        ldc = self.cl + N + 8
        if aligned:
            ldc += (-ldc * esz) % 16 // esz
        elif ldc % 2 == 0:
            ldc += 1
        self.ldc = ldc
        self.buf = torch.full((M + 2 * GUARD_ROWS, ldc), SENT[dtype], dtype=_INT[dtype], device=DEV).view(dtype)
        self.view = self.buf[GUARD_ROWS:GUARD_ROWS + M, self.cl:self.cl + N]

    @property
    def ptr(self):
        return self.buf.data_ptr() + (GUARD_ROWS * self.ldc + self.cl) * self.buf.element_size()

    def check_guard(self, what, interior_written=True):
        raw = self.buf.view(_INT[self.dtype]).clone()
        if interior_written:
            raw[GUARD_ROWS:GUARD_ROWS + self.M, self.cl:self.cl + self.N] = SENT[self.dtype]
        bad = (raw != SENT[self.dtype]).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.shape[0]} elements written outside C, first at buffer {bad[0].tolist()} " \
                                 f"(C = rows [{GUARD_ROWS}, {GUARD_ROWS + self.M}), cols [{self.cl}, {self.cl + self.N}))"


def dev_f32(v, big=BIG_SCALE, extra=8):
    v = np.asarray(v, np.float32).reshape(-1)
    return torch.from_numpy(np.concatenate([v, np.full(extra, big, np.float32)])).to(DEV)


# ------------------------------------------------------------------ exact comparison

def assert_bits_equal(got, ref, what, any_nan=False):
    """float32 arrays holding values of the output dtype: equal bit patterns, with +0 == -0.  any_nan: a NaN matches
    a NaN of any sign and payload."""
    g = (np.asarray(got, np.float32) + np.float32(0.0)).view(np.uint32)
    r = (np.asarray(ref, np.float32) + np.float32(0.0)).view(np.uint32)
    assert g.shape == r.shape
    if any_nan:
        nan = np.isnan(np.asarray(ref, np.float32))
        g, r = np.where(nan & np.isnan(np.asarray(got, np.float32)), 0x7FC00000, g), np.where(nan, 0x7FC00000, r)
    if not np.array_equal(g, r):
        bad = np.argwhere(g != r)
        i = tuple(bad[0])
        raise AssertionError(f"{what}: {len(bad)} of {g.size} outputs differ from the exact result; first at {list(i)}: "
                             f"got {got[i]!r} want {ref[i]!r}")
