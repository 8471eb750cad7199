"""Shared helpers for the tests: ctypes view of the C ABI, torch<->numpy glue."""
import ctypes
import os
import re
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "fp8-mps-metal_b200")
LIB_PATH = os.environ.get("FP8B_LIB") or os.path.join(PKG, "libfp8_b200.so")    # FP8B_LIB: A/B a differently built library
HEADER = os.path.join(ROOT, "include", "fp8_b200.h")
if os.path.join(ROOT, "oracle") not in sys.path:       # bench.py imports this module before it adds oracle/
    sys.path.insert(0, os.path.join(ROOT, "oracle"))

import fp8_oracle as o  # noqa: E402

F32, F16, BF16 = 0, 1, 2
ALGO_AUTO, ALGO_GEMV, ALGO_TCGEN05, ALGO_SIMT = 0, 1, 2, 3

_lib = None

DEV = "cuda"
GUARD_ROWS = 3
SENT = {torch.float32: 0x7FA5A5A5, torch.float16: 0x7DA5, torch.bfloat16: 0x7FA5}    # NaN payloads no kernel writes
_INT = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}
BIG_SCALE = 1024.0                                    # what sits behind per-row scales
BIG_BIAS = 30000.0                                    # what sits behind per-row biases
E4M3, E5M2 = 0, 1


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


# ------------------------------------------------------------------ structured inputs for the bit-exact matmul tests
# (test_gpu_exact.py describes the input families and why their sums are exact)

def dev_bytes(X, offset=0, guard_rows=2):
    """uint8 rows of X, then guard rows of 0x7E, starting `offset` bytes into the allocation -> (tensor, pointer)."""
    R, K = X.shape
    flat = np.full(offset + (R + guard_rows) * K + 16, 0x7E, np.uint8)
    flat[offset:offset + R * K] = X.reshape(-1)
    t = torch.from_numpy(flat).to(DEV)
    return t, t.data_ptr() + offset


def dev_bias(v, dtype, extra=8):
    """bias of `dtype` followed by large finite values -> (tensor, the fp32 values the kernel reads)."""
    t = torch.from_numpy(np.concatenate([np.asarray(v, np.float32), np.full(extra, BIG_BIAS, np.float32)])).to(DEV).to(dtype)
    return t, to_np(t[:len(v)])


def _decode(X, fmt):
    return o.decode_fmt(X, "e5m2" if fmt == E5M2 else "e4m3fn")


def oracle(A, B, sa, sb, bias, sr, odt, fmts=(E4M3, E4M3)):
    """fp8_oracle.scaled_mm (fp64 sum) restricted to the K columns where A or B has nonzeros: the other columns add
    exact zeros, and a 100000-long K then costs nothing on the host."""
    fa, fb = fmts
    K = A.shape[1]
    if K > 64:
        nz = (_decode(A, fa) != 0).any(0)
        if nz.sum() > K // 4:
            nzb = (_decode(B, fb) != 0).any(0)
            nz = nzb if nzb.sum() < nz.sum() else nz
        cols = np.flatnonzero(nz)
        A, B = A[:, cols], B[:, cols]
    return o.scaled_mm(A, B, sa, sb, bias, None if sr is None else np.array([sr], np.float32), dt_name(odt),
                       accum="f64", a_format="e5m2" if fa == E5M2 else "e4m3fn", b_format="e5m2" if fb == E5M2 else "e4m3fn")


NON_NAN = np.array([c for c in range(256) if (c & 0x7F) != 0x7F], np.uint8)
E5M2_CODES = np.array([c for c in range(256) if (c & 0x7F) < 0x60], np.uint8)       # finite, |v| < 512
SMALL_INT_CODES = o.encode(np.arange(-16, 17, dtype=np.float32))                     # exact e4m3 codes of -16..16


def codes(shape, rng, fmt=E4M3):
    return rng.choice(E5M2_CODES if fmt == E5M2 else NON_NAN, shape).astype(np.uint8)


def edges(K, bounds, rng, n_random=6):
    """k = 0, the last 16-byte vector, the 16-byte vectors on both sides of every boundary, and random positions."""
    pos = {0, 15, K - 16, K - 1}
    for b in bounds:
        pos |= {b - 16, b - 1, b, b + 15}
    pos |= set(rng.integers(0, K, n_random).tolist())
    return np.array(sorted(q for q in pos if 0 <= q < K), np.int64)


def one_hot(R, K, positions, rng, fmt=E4M3):
    """R rows, row r nonzero (a random code, the zero codes included) only at positions[r % len]; a random subset of the
    positions when there are more of them than rows."""
    X = np.zeros((R, K), np.uint8)
    n = len(positions)
    ks = positions[np.arange(R) % n] if R >= n else positions[np.sort(rng.choice(n, R, replace=False))]
    X[np.arange(R), ks] = codes(R, rng, fmt)
    return X


def few_hot(R, K, positions, rng):
    """<= 8 nonzeros per row, all at boundary positions, small integers (|v| <= 16)."""
    X = np.zeros((R, K), np.uint8)
    for r in range(R):
        ks = rng.choice(positions, min(8, len(positions)), replace=False)
        X[r, ks] = SMALL_INT_CODES[rng.integers(0, 33, len(ks))]
    return X


def small_ints(shape, rng, lo=-16, hi=16):
    return SMALL_INT_CODES[rng.integers(lo + 16, hi + 17, shape)]


def add_nan_rows(B, A, rows, rng):
    """NaN codes in a few chosen B rows: at the nonzero position of A row 0 (the product must come out as exactly 0 through
    the NaN fix-up) and at random positions (the fix-up must recompute the one real product)."""
    k0 = np.flatnonzero(A[0]) if A[0].any() else np.array([0])
    for i, n in enumerate(rows):
        B[n, rng.integers(0, B.shape[1], 3)] = 0x7F if i % 2 else 0xFF
        if i == 0:
            B[n, k0] = 0x7F
    return B


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def tc_bounds(K):
    return set(range(128, K, 128))


class Terms:
    """Random fp32 epilogue terms: per-tensor or per-row sa / sb, a bias of some dtype, scale_result."""

    def __init__(self, M, N, rng, per_row_a=False, per_row_b=False, bias_dt=None, sr=False):
        self.sa = ((rng.random(M if per_row_a else 1) + 0.5) * 0.0123).astype(np.float32)
        self.sb = ((rng.random(N if per_row_b else 1) + 0.5) * 0.0217).astype(np.float32)
        self.bias_dt = bias_dt
        self.bias_raw = (rng.standard_normal(N) * 0.7).astype(np.float32) if bias_dt is not None else None
        self.sr = float(np.float32(0.5 + rng.random())) if sr else None

    @staticmethod
    def cycle(i, M, N, rng):
        """the i-th of a fixed rotation over the term combinations."""
        return Terms(M, N, rng, per_row_a=bool(i & 1), per_row_b=bool(i & 2),
                     bias_dt=(None, torch.float32, torch.float16, torch.bfloat16)[(i >> 2) % 4], sr=bool(i % 3 == 1))

    def device(self):
        self.t_sa, self.t_sb = dev_f32(self.sa), dev_f32(self.sb)
        self.t_bias, self.bias = (None, None) if self.bias_dt is None else dev_bias(self.bias_raw, self.bias_dt)
        self.t_sr = dev_f32([self.sr]) if self.sr is not None else None
        return self
