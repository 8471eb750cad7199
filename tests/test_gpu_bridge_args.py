"""Argument preparation of the torch extension (csrc/fp8_bridge.cpp), binding by binding.

Every binding refuses what the kernels cannot take with a RuntimeError before anything is launched, and every accepted
form of a scale or a bias (host or device, float64 or int64, contiguous or not) gives the bits of the float32 device
tensor with the same values.  The multicast binding is only ever called with mc_ptr = 0: the C ABI refuses the null
destination, so no call here can store through a bogus address."""
import numpy as np
import pytest
import torch

import fp8_mps_native as nat
import fp8_mps_patch
from _util import codes

DEV = "cuda"
FP8 = torch.float8_e4m3fn


def _lib():
    return nat._get_lib()


# ------------------------------------------------------------------ CPU tensors: refused, nothing launched

def _cpu_calls():
    L = _lib()
    A, B = torch.zeros(4, 32, dtype=torch.uint8), torch.zeros(8, 32, dtype=torch.uint8)
    x, one, out = torch.zeros(4, 32), torch.ones(1), torch.zeros(4, 8)
    return {
        "fp8_scaled_mm": lambda: L.fp8_scaled_mm(A, B, one, one),
        "fp8_scaled_mm_fused": lambda: L.fp8_scaled_mm_fused(A, B, one, one, None, None, None, 0, None, 0, 0),
        "scaled_mm_patch": lambda: L.scaled_mm_patch(A, B.t(), one, one, None, None, None),
        "fp8_scaled_mm_many": lambda: L.fp8_scaled_mm_many([A[:1]], [B], [one], [one], None, None),
        "fp8_linear_dynamic": lambda: L.fp8_linear_dynamic(x, B, one, None, None, False),
        "fp8_scaled_mm_peers": lambda: L.fp8_scaled_mm_peers(A, B, one, one, None, out, torch.zeros(2, dtype=torch.int64), 0),
        "fp8_scaled_mm_push": lambda: L.fp8_scaled_mm_push(A, B, one, one, None, out, [0], 0),
        "fp8_scaled_mm_multicast": lambda: L.fp8_scaled_mm_multicast(A, B, one, one, None, torch.float32, 0, 8, 0),
        "fp8_encode": lambda: L.fp8_encode(x),
        "fp8_encode_many": lambda: L.fp8_encode_many([x]),
        "fp8_quantize": lambda: L.fp8_quantize(x),
        "fp8_quantize_rowwise": lambda: L.fp8_quantize_rowwise(x),
        "fp8_dequantize": lambda: L.fp8_dequantize(A, one),
        "fp8_dequantize_to": lambda: L.fp8_dequantize_to(A, torch.float32, 0),
        "fp8_dequantize_many": lambda: L.fp8_dequantize_many([A], torch.float32),
    }


@pytest.mark.parametrize("binding", sorted(_cpu_calls()))
def test_cpu_tensors_are_refused(binding):
    L = _lib()
    n0 = L.launch_count()
    with pytest.raises(RuntimeError):
        _cpu_calls()[binding]()
    assert L.launch_count() == n0


# ------------------------------------------------------------------ GPU: malformed arguments

M, K, N = 300, 512, 1024
FULL_N, N0 = N + 64, 32                  # exchange bindings write the column block [N0, N0 + N) of an (M, FULL_N) buffer


def _operands():
    rng = np.random.default_rng(1)
    A = torch.from_numpy(codes((M, K), rng)).to(DEV)
    B = torch.from_numpy(codes((N, K), rng)).to(DEV)
    X = torch.from_numpy(rng.standard_normal((M, K)).astype(np.float32)).to(DEV)
    sa = torch.tensor([0.013], device=DEV)
    sb = torch.from_numpy(((rng.random(N) + 0.5) * 0.02).astype(np.float32)).to(DEV)
    bias = torch.from_numpy(rng.integers(-8, 9, N).astype(np.float32)).to(DEV)
    return A, B, X, sa, sb, bias


def _out():
    return torch.zeros(M, FULL_N, device=DEV)


# binding -> (call(A, B, X, sa, sb, bias, sr) returning the (.., N) result, the faults it can be given)
_ALL = ("k", "uint8", "contiguous", "scale_a", "scale_b", "bias")


def _peers(A, B, X, sa, sb, bias, sr):
    out, peer = _out(), _out()                      # world = 2: a second local buffer stands in for the peer's
    deltas = torch.tensor([0, peer.data_ptr() - out.data_ptr()], dtype=torch.int64, device=DEV)
    _lib().fp8_scaled_mm_peers(A, B, sa, sb, bias, out, deltas, N0)
    return out[:, N0:N0 + N]


def _push(A, B, X, sa, sb, bias, sr):
    out = _out()
    _lib().fp8_scaled_mm_push(A, B, sa, sb, bias, out, [out.data_ptr()], N0)
    return out[:, N0:N0 + N]


BINDINGS = {
    "fp8_scaled_mm": (lambda A, B, X, sa, sb, bias, sr: _lib().fp8_scaled_mm(A, B, sa, sb),
                      ("k", "uint8", "contiguous", "scale_a", "scale_b")),
    "fp8_scaled_mm_fused": (lambda A, B, X, sa, sb, bias, sr:
                            _lib().fp8_scaled_mm_fused(A, B, sa, sb, bias, sr, None, 0, None, 0, 0),
                            _ALL + ("scale_result",)),
    "scaled_mm_patch": (lambda A, B, X, sa, sb, bias, sr: _lib().scaled_mm_patch(A, B.t(), sa, sb, bias, sr, None),
                        ("k", "uint8", "scale_a", "scale_b", "bias", "scale_result")),     # copies a strided operand
    "fp8_scaled_mm_many": (lambda A, B, X, sa, sb, bias, sr:
                           _lib().fp8_scaled_mm_many([A[:1]], [B], [sa], [sb], None if bias is None else [bias], None)[0],
                           _ALL),
    "fp8_linear_dynamic": (lambda A, B, X, sa, sb, bias, sr: _lib().fp8_linear_dynamic(X, B, sb, bias, None, False)[0],
                           ("k", "uint8", "contiguous", "scale_b", "bias")),
    "fp8_scaled_mm_peers": (_peers, _ALL),
    "fp8_scaled_mm_push": (_push, _ALL),
    "fp8_scaled_mm_multicast": (lambda A, B, X, sa, sb, bias, sr:
                                _lib().fp8_scaled_mm_multicast(A, B, sa, sb, bias, torch.float32, 0, FULL_N, 0),
                                _ALL),
}
_CASES = [(b, f) for b, (_, faults) in BINDINGS.items() for f in faults]


@pytest.mark.gpu
@pytest.mark.parametrize("binding,fault", _CASES, ids=[f"{b}-{f}" for b, f in _CASES])
def test_malformed_arguments_are_refused_before_any_launch(binding, fault):
    A, B, X, sa, sb, bias = _operands()
    sr = None
    match = None
    if fault == "k":
        B = B[:, :K - 16].contiguous()
    elif fault == "uint8":
        B = B.view(torch.int8)
    elif fault == "contiguous":
        B = torch.cat([B, B], dim=1)[:, :K]
    elif fault == "scale_a":
        sa, match = torch.full((3,), 0.5, device=DEV), r"scale_[ax] must have"
    elif fault == "scale_b":
        sb, match = sb[:N - 1], r"scale_[bw] must have"
    elif fault == "bias":
        bias, match = torch.zeros(N + 1, device=DEV), "bias must have"
    elif fault == "scale_result":
        sr, match = torch.ones(2, device=DEV), "scale_result must have"
    call = BINDINGS[binding][0]
    torch.cuda.synchronize()
    n0 = _lib().launch_count()
    with pytest.raises(RuntimeError, match=match):
        call(A, B, X, sa, sb, bias, sr)
    assert _lib().launch_count() == n0


@pytest.mark.gpu
def test_operands_of_the_malformed_cases_are_otherwise_accepted():
    """The base arguments of the cases above compute, so each refusal above comes from its one fault; the multicast
    binding, called with mc_ptr = 0, reaches the C ABI and comes back with its null-destination refusal."""
    A, B, X, sa, sb, bias = _operands()
    for binding, (call, _) in BINDINGS.items():
        n0 = _lib().launch_count()
        if binding == "fp8_scaled_mm_multicast":
            with pytest.raises(RuntimeError, match="invalid argument"):
                call(A, B, X, sa, sb, bias, None)
            assert _lib().launch_count() == n0
            with pytest.raises(RuntimeError, match="unsupported"):     # no float8_e4m3fn output through multicast
                _lib().fp8_scaled_mm_multicast(A, B, sa, sb, bias, FP8, 0, FULL_N, 0)
            assert _lib().launch_count() == n0
        else:
            y = call(A, B, X, sa, sb, bias, None)
            assert _lib().launch_count() > n0, binding
            assert y.shape[-1] == N and bool(torch.isfinite(y).all()), binding


# ------------------------------------------------------------------ GPU: every accepted form gives the same bits

def _bits(t):
    return t.contiguous().view(torch.int32 if t.element_size() == 4 else torch.int16)


@pytest.mark.gpu
@pytest.mark.parametrize("binding", [b for b in BINDINGS if b != "fp8_scaled_mm_multicast"])
def test_scale_and_bias_forms_give_identical_bits(binding):
    """float64 scales and an int64 bias give the bits of their float32 values; host tensors give the bits of the same
    device tensors; a strided device bias gives the bits of a contiguous one."""
    A, B, X, sa, sb, bias = _operands()
    call = BINDINGS[binding][0]
    ref = call(A, B, X, sa, sb, bias, None).clone()
    forms = {
        "host": (sa.cpu(), sb.cpu(), bias.cpu()),
        "float64 / int64 on the device": (sa.double(), sb.double(), bias.long()),
        "float64 / int64 on the host": (sa.double().cpu(), sb.double().cpu(), bias.long().cpu()),
        "strided bias": (sa, sb, torch.stack([bias, -bias], dim=1)[:, 0]),
    }
    for what, (sa2, sb2, bias2) in forms.items():
        y = call(A, B, X, sa2, sb2, bias2, None)
        assert torch.equal(_bits(y), _bits(ref)), f"{binding}: {what}"


@pytest.mark.gpu
@pytest.mark.parametrize("bias_dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_fused_patch_and_many_agree_at_m1(bias_dtype):
    """One M = 1 problem through fp8_scaled_mm_fused, the patched torch._scaled_mm and fp8_scaled_mm_many: the same
    GEMV with the same epilogue, so the same bits, whatever the bias dtype."""
    rng = np.random.default_rng(7)
    Kg, Ng = 1024, 256
    x = torch.from_numpy(codes((1, Kg), rng)).to(DEV)
    W = torch.from_numpy(codes((Ng, Kg), rng)).to(DEV)
    sa = torch.tensor([0.021], device=DEV)
    sb = torch.from_numpy(((rng.random(Ng) + 0.5) * 0.02).astype(np.float32)).to(DEV)
    bias = torch.from_numpy(rng.standard_normal(Ng).astype(np.float32)).to(DEV).to(bias_dtype)
    odt = torch.bfloat16
    y_fused = _lib().fp8_scaled_mm_fused(x, W, sa, sb, bias, None, odt, 0, None, 0, 0)
    y_many = nat.fp8_scaled_mm_many([x], [W], [sa], [sb], [bias], odt)[0]
    fp8_mps_patch.install()
    try:
        y_patch = torch._scaled_mm(x.view(FP8), W.view(FP8).t(), scale_a=sa, scale_b=sb, bias=bias, out_dtype=odt)
    finally:
        fp8_mps_patch.uninstall()
    assert y_fused.dtype == y_many.dtype == y_patch.dtype == odt
    assert torch.equal(_bits(y_patch), _bits(y_fused)), "patch vs fused"
    assert torch.equal(_bits(y_many), _bits(y_fused)), "many vs fused"
