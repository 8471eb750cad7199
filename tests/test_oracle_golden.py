"""
Pins the oracle (oracle/fp8_oracle.py and oracle/fp8_oracle.c) to the reference.

The fixtures in tests/golden/ were produced by tests/golden/make_golden.py, which imports the
reference's own pure-Python codec (test_fp8_correctness.py:22-106) and runs the reference's
host arithmetic (fp8_mps_native.py:121-122, :174-189).  Bit-exact everywhere; NaN inputs (which
the reference leaves undefined) are marked 0xFF in the fixtures and skipped.
"""
import numpy as np
import pytest

import c_oracle
import fp8_oracle as o

NAN_SENTINEL = 0xFF


def test_decode_table_matches_reference(golden):
    ref = golden["codec"]["decode_table"]
    assert np.array_equal(o.DECODE_TABLE.view(np.uint32), ref.view(np.uint32))       # incl. -0.0 at 0x80
    assert np.array_equal(c_oracle.decode_table().view(np.uint32), ref.view(np.uint32))
    assert o.DECODE_TABLE[0x7F] == 0.0 and o.DECODE_TABLE[0xFF] == 0.0               # NaN -> 0 (metal:21)
    assert o.DECODE_TABLE[0x7E] == 448.0 and o.DECODE_TABLE[0x01] == 2.0 ** -9


def test_encode_all_bf16_patterns(golden):
    ref = golden["codec"]["enc_bf16_all"]
    bits = np.arange(65536, dtype=np.uint32)
    vals = (bits << 16).view(np.float32)
    ok = ref != NAN_SENTINEL
    assert ok.sum() == 65536 - 2 * 127
    for got in (o.encode(vals), o.encode_bits(vals), c_oracle.encode(vals),
                c_oracle.encode_bf16_bits(bits.astype(np.uint16))):
        assert np.array_equal(got[ok], ref[ok])
        assert np.all(got[~ok] == 0x7F)            # build-defined NaN answer


def test_encode_all_fp16_patterns(golden):
    ref = golden["codec"]["enc_fp16_all"]
    vals = np.arange(65536, dtype=np.uint16).view(np.float16)
    ok = ref != NAN_SENTINEL
    for got in (o.encode(vals), o.encode_bits(vals), c_oracle.encode(vals)):
        assert np.array_equal(got[ok], ref[ok])


def test_encode_fp32_golden(golden):
    x = golden["codec"]["enc_f32_in"]
    ref = golden["codec"]["enc_f32_out"]
    ok = ref != NAN_SENTINEL
    assert x.size > 60000
    for got in (o.encode(x), o.encode_bits(x), c_oracle.encode(x)):
        assert np.array_equal(got[ok], ref[ok])


def test_known_answers(golden):
    kat = golden["kat"]
    for v, b in kat["encode"]:
        assert int(o.encode(np.float32(v))) == b, (v, b)
        assert int(c_oracle.encode(np.array([v], dtype=np.float32))[0]) == b
    # test_mps_vs_cpu.py:303: these five must equal torch CPU's own cast
    got = o.encode(np.array(kat["torch_cpu_equal"], dtype=np.float32)).tolist()
    assert got == kat["torch_cpu_bytes"]


def test_roundtrip_all_256(golden):
    """test_fp8_correctness.py:118-131: encode(decode(b)) == b except {0x7F,0xFF,0x80} -> 0x00."""
    b = np.arange(256, dtype=np.uint8)
    rt = o.encode(o.decode(b))
    allow = golden["kat"]["roundtrip_allow"]
    for i in range(256):
        assert rt[i] == (0 if i in allow else i)


def test_monotonic():
    """test_fp8_correctness.py:190-222: encode is monotone non-decreasing on [0, 448]."""
    x = np.linspace(0, 460, 200001, dtype=np.float32)
    e = o.encode(x).astype(np.int32)
    assert np.all(np.diff(e) >= 0)


def test_dequantize_golden(golden):
    h = golden["host"]
    u8 = np.arange(256, dtype=np.uint8)
    for i, s in enumerate(h["deq_scales"]):
        assert np.array_equal(o.fp8_dequantize(u8, s).view(np.uint16), h["deq_out"][i])
        assert np.array_equal(c_oracle.to_half(u8, s).view(np.uint16), h["deq_out"][i])
    assert np.array_equal(c_oracle.to_half(u8).view(np.uint16),
                          o.decode(u8).astype(np.float16).view(np.uint16))


def test_quantize_golden(golden):
    h = golden["host"]
    for i in range(int(h["n_quant"])):
        q, inv = o.fp8_quantize(h[f"q{i}_in"])
        assert np.array_equal(q, h[f"q{i}_bytes"])
        assert np.array_equal(inv.view(np.uint32), h[f"q{i}_inv"].view(np.uint32))


def test_quantize_rows_equals_rowwise_quantize():
    """fp8_quantize_rows == fp8_quantize row by row, special rows included; the special amax values give the
    scale and inverse scale the C ABI documents (include/fp8_b200.h)."""
    rng = np.random.default_rng(11)
    cols = 37
    X = (rng.standard_normal((40, cols)) * np.exp2(rng.integers(-20, 20, (40, 1)))).astype(np.float32)
    specials = {1: 0.0, 2: -0.0, 3: np.nan, 4: np.inf, 5: -np.inf, 6: 448.0, 7: np.finfo(np.float32).max,
                8: np.float32(2.0 ** -149), 9: np.float32(1e-37), 10: np.float32(2.0 ** -126)}
    for r, v in specials.items():
        if r in (1, 2):
            X[r] = v
        elif r in (8, 9, 10):
            X[r] = 0.0
            X[r, [0, 5, cols - 1]] = [v, -v, v]
        else:
            X[r, 3] = v
    X[11, [2, 7]] = [np.inf, np.nan]
    X[12] = -1.5
    for dt in (np.float32, np.float16):
        with np.errstate(over="ignore"):
            Xd = X.astype(dt)
        q, inv = o.fp8_quantize_rows(Xd)
        assert q.shape == X.shape and inv.shape == (X.shape[0],) and inv.dtype == np.float32
        for r in range(X.shape[0]):
            rq, rinv = o.fp8_quantize(Xd[r])
            assert np.array_equal(q[r], rq), (dt, r)
            assert inv[r].view(np.uint32) == rinv.view(np.uint32)[0], (dt, r)
    q, inv = o.fp8_quantize_rows(X)
    assert inv[1] == inv[2] == 1.0 and not q[1].any() and not q[2].any()             # amax 0: scale 1
    assert inv[3] == inv[11] == 1.0 and q[3, 3] == q[11, 7] == 0x7F and q[11, 2] == 0x7E   # NaN amax: scale 1
    for r in (4, 5):                                                                 # inf amax: scale 0, inv +inf
        assert inv[r] == np.inf
        finite = np.isfinite(X[r])
        assert (q[r][finite] == 0).all() and (q[r][~finite] == 0x7F).all()
    assert inv[12] == np.float32(1.5 / 448.0)
    for r in (8, 9):                                                                 # float32(448/amax) = inf
        assert 0.0 <= inv[r] < np.float32(2.0 ** -126)
        assert (q[r][X[r] == 0] == 0x7F).all() and q[r][0] == 0x7E and q[r][5] == 0xFE
    assert o.fp8_quantize_rows(np.zeros((3, 0), np.float32))[1].tolist() == [1.0, 1.0, 1.0]


def test_quantize_roundtrip_reference_case():
    """test_fp8_metal.py:167-188: max abs error < 50 on the reference's list (it is far smaller)."""
    x = np.array([0.0, 1.0, -1.0, 0.5, -0.5, 100.0, -100.0, 448.0], dtype=np.float32)
    q, inv = o.fp8_quantize(x)
    d = o.fp8_dequantize(q, inv).astype(np.float32)
    assert np.abs(d - x).max() < 50.0
    assert np.abs(d - x).max() <= 4.0      # 100 -> 0x6C = 96 (RNE tie, FIX_DOCUMENTATION.md:33-41)


@pytest.mark.parametrize("M,K,N", [(1, 512, 256), (1, 4096, 64), (4, 4096, 48), (64, 256, 128),
                                   (32, 64, 48), (3, 37, 5), (1, 3, 2), (16, 130, 33)])
def test_scaled_mm_numpy_vs_c(M, K, N):
    """The fp64-sum oracle and the shader-order C loops agree to fp32 summation noise;
    shapes are the reference's (test_fp8_metal.py:97-218, test_cross_validation.py:166-198)."""
    rng = np.random.default_rng(M * 1000 + K + N)
    A = rng.integers(0, 256, (M, K), dtype=np.uint8)
    B = rng.integers(0, 256, (N, K), dtype=np.uint8)
    sa = np.array([0.01], dtype=np.float32)
    sb = rng.random(N).astype(np.float32) * 0.02 + 0.001
    ref = o.scaled_mm(A, B, sa, sb)
    got = c_oracle.scaled_mm(A, B, sa, sb)
    assert o.rel_rmse(got, ref) < 2e-6
    # per-row scale_a too (reference scale_mode 1)
    if M > 1:
        sa2 = rng.random(M).astype(np.float32) + 0.5
        assert o.rel_rmse(c_oracle.scaled_mm(A, B, sa2, sb), o.scaled_mm(A, B, sa2, sb)) < 2e-6


def test_scaled_mm_quantisation_error_matches_reference_claim():
    """README.md:86 / test_fp8_metal.py:122: FP8 matmul is within 15 % rel-RMSE (about 4 %)
    of the un-quantised fp32 A@B.T."""
    rng = np.random.default_rng(7)
    M, K, N = 64, 256, 128
    A = rng.standard_normal((M, K)).astype(np.float32)
    B = rng.standard_normal((N, K)).astype(np.float32)
    qa, sa = o.fp8_quantize(A)
    qb, sb = o.fp8_quantize(B)
    r = o.scaled_mm(qa, qb, sa, sb)
    e = o.rel_rmse(r, A @ B.T)
    assert e < 0.15 and e < 0.06


def test_epilogue_order_and_out_dtypes():
    rng = np.random.default_rng(3)
    A = rng.integers(0, 127, (4, 64), dtype=np.uint8)
    B = rng.integers(0, 127, (8, 64), dtype=np.uint8)
    sa = np.array([0.5], dtype=np.float32)
    sb = np.array([0.25], dtype=np.float32)
    bias = rng.standard_normal(8).astype(np.float32)
    base = o.scaled_mm(A, B, sa, sb)
    full = o.scaled_mm(A, B, sa, sb, bias=bias, scale_result=np.array([2.0], dtype=np.float32))
    assert np.array_equal(full, (base + bias) * np.float32(2.0))         # fp8_mps_patch.py:95-100
    bf = o.scaled_mm(A, B, sa, sb, out_dtype="bf16")
    assert np.all((bf.view(np.uint32) & 0xFFFF) == 0)
    h = o.scaled_mm(A, B, sa, sb, out_dtype="f16")
    assert np.array_equal(h, base.astype(np.float16).astype(np.float32))


def test_e5m2_decode_table_matches_torch_cast():
    """float8_e5m2 has no codec in the reference (SURVEY B6); the oracle's table is pinned to PyTorch's CPU cast
    (tests/golden/e5m2_golden.npz): bit-exact for the 250 non-NaN bytes, NaN for the six NaN bytes."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "e5m2_golden.npz"))
    ref = g["decode_f32_bits"].view(np.float32)
    ours = o.decode_e5m2(np.arange(256, dtype=np.uint8))
    nan = np.isnan(ref)
    assert nan.sum() == 6 and np.array_equal(np.isnan(ours), nan)
    assert np.array_equal(ours[~nan].view(np.uint32), ref[~nan].view(np.uint32))
    assert ours[0x7C] == np.inf and ours[0xFC] == -np.inf and ours[0x7B] == 57344.0 and ours[0x01] == 2.0 ** -16
    c_tab = c_oracle.decode_table_e5m2()                     # the plain-C restatement (arithmetic, not a bit shift)
    assert np.array_equal(np.isnan(c_tab), nan) and np.array_equal(c_tab[~nan].view(np.uint32), ref[~nan].view(np.uint32))
    # every value is exactly representable in fp16 and bf16
    assert np.array_equal(g["decode_f16_bits"][~nan], (np.arange(256, dtype=np.uint16) << 8)[~nan])
    assert np.array_equal(o.f32_to_bf16_bits(ours[~nan]), g["decode_bf16_bits"][~nan])
