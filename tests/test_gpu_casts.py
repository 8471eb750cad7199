"""GPU parity: the streaming cast kernels vs the oracle / the reference-generated fixtures.
Bit-exact everywhere (integer/byte work).  Calls go through the raw C ABI (ctypes) and through
the reference-shaped Python API (fp8_mps_native)."""
import numpy as np
import pytest
import torch

import c_oracle
import fp8_oracle as o
from _util import BF16, F16, F32, capi, dt_code, make_spans, p, stream_ptr, to_np

pytestmark = pytest.mark.gpu
DEV = "cuda"
NAN_SENTINEL = 0xFF


def _encode_capi(x, prescale=None):
    out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    rc = capi().fp8b_encode(p(x), dt_code(x.dtype), p(out), x.numel(), p(prescale), stream_ptr())
    assert rc == 0, capi().fp8b_status_string(rc)
    return out


def _dequant_capi(u8, dtype, scale=None):
    out = torch.empty(u8.shape, dtype=dtype, device=u8.device)
    if scale is not None or dtype == torch.float16:
        assert dtype == torch.float16
        rc = capi().fp8b_dequant_f16(p(u8), p(out), u8.numel(), p(scale), stream_ptr())
    else:
        rc = capi().fp8b_dequant(p(u8), p(out), dt_code(dtype), u8.numel(), stream_ptr())
    assert rc == 0, capi().fp8b_status_string(rc)
    return out


# ------------------------------------------------------------------ decode

@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32])
def test_decode_all_256_patterns(golden, dtype):
    """test_fp8_metal.py:53-94 (gate 0.5 abs; README claims 0.0): here bit-exact incl. NaN->0, 0x80->-0."""
    ref = golden["codec"]["decode_table"]
    b = torch.arange(256, dtype=torch.int32).to(torch.uint8).to(DEV)
    out = _dequant_capi(b, dtype)
    got = to_np(out)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    # repeat so the vector path (not just the scalar tail) sees every pattern at every lane position
    rep = b.repeat(257)[3:]                      # misaligned start -> scalar kernel
    got2 = to_np(_dequant_capi(rep, dtype))
    assert np.array_equal(got2.view(np.uint32), np.tile(ref, 257)[3:].view(np.uint32))
    rep = b.repeat(64)                           # aligned -> vector kernel
    got3 = to_np(_dequant_capi(rep, dtype))
    assert np.array_equal(got3.view(np.uint32), np.tile(ref, 64).view(np.uint32))


def test_dequantize_scaled_golden(golden):
    """fp8_dequantize = fp16 multiply by half(scale) (fp8_mps_native.py:121-122), fixture from torch CPU."""
    import fp8_mps_native
    h = golden["host"]
    b = torch.arange(256, dtype=torch.int32).to(torch.uint8).to(DEV).repeat(16)
    for i, s in enumerate(h["deq_scales"]):
        sc = torch.tensor([float(s)], dtype=torch.float32, device=DEV)
        want = np.tile(h["deq_out"][i], 16)
        got = _dequant_capi(b, torch.float16, sc).view(torch.int16).cpu().numpy().view(np.uint16)
        assert np.array_equal(got, want), f"scale {s}"
        got2 = fp8_mps_native.fp8_dequantize(b, sc)
        assert got2.dtype == torch.float16 and got2.shape == b.shape
        assert np.array_equal(got2.view(torch.int16).cpu().numpy().view(np.uint16), want)
        got3 = fp8_mps_native.fp8_dequantize(b[5:261].cpu(), torch.tensor(float(s)))   # CPU in, odd offset
        assert got3.device.type == "cuda"
        assert np.array_equal(got3.view(torch.int16).cpu().numpy().view(np.uint16), want[5:261])


# ------------------------------------------------------------------ encode

def _check_encode(got_u8, ref_u8):
    got = got_u8.cpu().numpy().reshape(-1)
    ok = ref_u8 != NAN_SENTINEL
    bad = np.nonzero(got[ok] != ref_u8[ok])[0]
    assert bad.size == 0, f"{bad.size} mismatches, first at {bad[:5]}"
    assert np.all(got[~ok] == 0x7F)              # NaN inputs: build-defined 0x7F


def test_encode_all_bf16_patterns(golden):
    bits = torch.arange(65536, dtype=torch.int32).to(torch.int16).to(DEV)
    x = bits.view(torch.bfloat16)
    _check_encode(_encode_capi(x), golden["codec"]["enc_bf16_all"])
    _check_encode(_encode_capi(x.float()), golden["codec"]["enc_bf16_all"])          # same values via fp32 path
    _check_encode(_encode_capi(x[1:]), golden["codec"]["enc_bf16_all"][1:])          # unaligned -> scalar kernel
    one = torch.ones(1, dtype=torch.float32, device=DEV)
    _check_encode(_encode_capi(x, one), golden["codec"]["enc_bf16_all"])             # prescale path, * 1.0


def test_encode_all_fp16_patterns(golden):
    bits = torch.arange(65536, dtype=torch.int32).to(torch.int16).to(DEV)
    x = bits.view(torch.float16)
    _check_encode(_encode_capi(x), golden["codec"]["enc_fp16_all"])
    _check_encode(_encode_capi(x.float()), golden["codec"]["enc_fp16_all"])
    _check_encode(_encode_capi(x[3:]), golden["codec"]["enc_fp16_all"][3:])


def test_encode_fp32_golden(golden):
    x = torch.from_numpy(golden["codec"]["enc_f32_in"]).to(DEV)
    _check_encode(_encode_capi(x), golden["codec"]["enc_f32_out"])
    _check_encode(_encode_capi(x[1:]), golden["codec"]["enc_f32_out"][1:])


def test_known_answers_and_api(golden):
    import fp8_mps_native
    kat = golden["kat"]
    vals = torch.tensor([v for v, _ in kat["encode"]], dtype=torch.float32)
    got = fp8_mps_native.fp8_encode(vals)                       # CPU input is moved (native.py:142)
    assert got.device.type == "cuda" and got.dtype == torch.uint8
    assert got.cpu().tolist() == [b for _, b in kat["encode"]]
    t = torch.tensor(kat["torch_cpu_equal"], dtype=torch.float32, device=DEV)
    assert fp8_mps_native.fp8_encode(t).cpu().tolist() == kat["torch_cpu_bytes"]     # test_mps_vs_cpu.py:303
    assert fp8_mps_native.fp8_encode(torch.empty(0, device=DEV)).numel() == 0
    assert fp8_mps_native.fp8_encode(torch.zeros(3, 5, 7, device=DEV)).shape == (3, 5, 7)


@pytest.mark.parametrize("n", [1, 7, 8, 9, 31, 257, 4099, 1 << 20, (1 << 22) + 13])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_encode_decode_random_sizes(n, dtype):
    """Ragged sizes: vector body + scalar tail, against the C oracle."""
    g = torch.Generator().manual_seed(n)
    scale = [1.0, 0.02, 100.0][n % 3]
    x = (torch.randn(n, generator=g) * scale).to(dtype)
    xd = x.to(DEV)
    got = _encode_capi(xd).cpu().numpy()
    if dtype == torch.bfloat16:
        ref = c_oracle.encode_bf16_bits(x.view(torch.int16).numpy().view(np.uint16))
    else:
        ref = c_oracle.encode(x.numpy())
    assert np.array_equal(got, ref)
    for odt in (torch.float16, torch.bfloat16, torch.float32):
        back = to_np(_dequant_capi(torch.from_numpy(ref).to(DEV), odt))
        assert np.array_equal(back.view(np.uint32), o.decode(ref).view(np.uint32))


def test_quantize_golden_and_random(golden):
    """fp8_quantize: device-side amax -> double-precision scale -> fused multiply+encode
    must equal the reference's host arithmetic (fp8_mps_native.py:174-189) bit for bit."""
    import fp8_mps_native
    h = golden["host"]
    for i in range(int(h["n_quant"])):
        x = torch.from_numpy(h[f"q{i}_in"]).to(DEV)
        q, inv = fp8_mps_native.fp8_quantize(x)
        assert q.dtype == torch.uint8 and inv.dtype == torch.float32 and inv.shape == (1,)
        assert np.array_equal(q.cpu().numpy(), h[f"q{i}_bytes"]), i
        assert np.array_equal(inv.cpu().numpy().view(np.uint32), h[f"q{i}_inv"].view(np.uint32)), i
    g = torch.Generator().manual_seed(5)
    for n, s in [(1000003, 1.0), (4096 * 4096, 0.02), (77, 300.0)]:
        x = torch.randn(n, generator=g) * s
        q, inv = fp8_mps_native.fp8_quantize(x)
        rq, rinv = o.fp8_quantize(x.numpy())
        assert np.array_equal(q.cpu().numpy(), rq)
        assert np.array_equal(inv.cpu().numpy().view(np.uint32), rinv.view(np.uint32))
    # bf16 / fp16 inputs are widened exactly (native.py:170)
    xb = (torch.randn(50000, generator=g) * 3).to(torch.bfloat16)
    q, inv = fp8_mps_native.fp8_quantize(xb.to(DEV))
    rq, rinv = o.fp8_quantize(xb.float().numpy())
    assert np.array_equal(q.cpu().numpy(), rq) and np.array_equal(inv.cpu().numpy().view(np.uint32), rinv.view(np.uint32))
    # roundtrip gate of the reference (test_fp8_metal.py:167-188)
    x = torch.tensor([0.0, 1.0, -1.0, 0.5, -0.5, 100.0, -100.0, 448.0])
    q, sc = fp8_mps_native.fp8_quantize(x)
    d = fp8_mps_native.fp8_dequantize(q, sc)
    assert (d.cpu().float() - x).abs().max().item() < 50.0


@pytest.mark.parametrize("rows,cols,dtype", [(7, 1000, torch.float32), (64, 4096, torch.bfloat16), (3, 17, torch.float16),
                                             (12288, 3072, torch.bfloat16), (5, 8, torch.float32), (1, 1, torch.float32),
                                             # register-resident kernel, few rows: a CTA per row with 1/2/4/8 vectors per
                                             # thread; then the two-pass kernel again
                                             (19, 64, torch.bfloat16), (9, 1000, torch.float16), (33, 2048, torch.bfloat16),
                                             (21, 2048, torch.float32), (10, 8192, torch.bfloat16), (16, 14336, torch.bfloat16),
                                             (5, 8192, torch.float32), (4, 20000, torch.bfloat16), (6, 1004, torch.bfloat16),
                                             # >= 32 rows per SM (4736 on 148 SMs): 2 or 4 vectors per thread and 32 / 32 /
                                             # 64 / 128 threads per row, several rows per CTA, a partial last CTA
                                             (4801, 256, torch.float32), (4801, 500, torch.float32), (4801, 1024, torch.float32),
                                             (4801, 2048, torch.float32), (4801, 512, torch.float16), (4801, 1000, torch.float16),
                                             (4801, 2048, torch.float16), (4801, 4096, torch.float16)])
def test_quantize_rowwise(rows, cols, dtype):
    """Per-row quantise == the reference's fp8_quantize arithmetic applied row by row (oracle), bit for bit,
    and its inverse scales feed _scaled_mm as per-row scales."""
    import fp8_mps_native
    g = torch.Generator().manual_seed(rows * 31 + cols)
    x = (torch.randn(rows, cols, generator=g) * torch.rand(rows, 1, generator=g) * 10).to(dtype)
    if rows > 2:
        x[1].zero_()                                               # amax == 0 -> scale 1.0 (native.py:176)
    q, inv = fp8_mps_native.fp8_quantize_rowwise(x.to(DEV))
    assert q.shape == (rows, cols) and q.dtype == torch.uint8 and inv.shape == (rows,) and inv.dtype == torch.float32
    qn, invn = q.cpu().numpy(), inv.cpu().numpy()
    check_rows = range(rows) if rows <= 64 else range(0, rows, 97)
    for r in check_rows:
        rq, rinv = o.fp8_quantize(x[r].float().numpy())
        assert np.array_equal(qn[r], rq), r
        assert invn[r].view(np.uint32) == rinv.view(np.uint32)[0], r


def test_full_size_properties():
    """BASELINE config 5 scale (one FLUX linear, 21504x3072 = 66 M elements, and a 1 Gi-element sweep
    of raw bytes): size-independent properties instead of an element-wise CPU oracle."""
    n = 21504 * 3072
    g = torch.Generator(device=DEV).manual_seed(11)
    w = (torch.randn(n, generator=g, device=DEV) * 0.02).to(torch.bfloat16)
    q = _encode_capi(w)
    # (1) idempotence: enc(dec(enc(x))) == enc(x), except 0x80 (-0.0) -> 0x00, the reference's own
    #     round-trip allow-list (test_fp8_correctness.py:118-131)
    d = _dequant_capi(q, torch.bfloat16)
    q2 = _encode_capi(d)
    assert torch.equal(torch.where(q == 0x80, torch.zeros_like(q), q), q2)
    # (2) the encoder never emits a NaN code and never emits -0 for an input that is not negative
    assert int(((q & 0x7F) == 0x7F).sum()) == 0
    assert int(((q == 0x80) & (w >= 0)).sum()) == 0
    # (3) |dec(enc(x)) - x| <= half a grid step (relative 1/16) or the flush threshold
    err = (d.float() - w.float()).abs()
    bound = torch.maximum(w.float().abs() / 16.0, torch.full_like(err, 2.0 ** -9))
    assert bool((err <= bound).all())
    # (4) a strided 1 M sample equals the C oracle bit for bit
    idx = torch.arange(0, n, 61, device=DEV)
    sample = w[idx].cpu()
    ref = c_oracle.encode_bf16_bits(sample.view(torch.int16).numpy().view(np.uint16))
    assert np.array_equal(q[idx].cpu().numpy(), ref)
    # (5) byte histogram of the full result equals the histogram implied by the sample's law:
    #     checksum of checksums -- sum over 64 Ki-element blocks of the byte sums, GPU vs itself
    #     re-encoded from fp32 input (a different kernel instantiation must agree exactly)
    q3 = _encode_capi(w.float())
    assert torch.equal(q, q3)
    del w, d, q2, q3, err, bound
    # raw-byte sweep: dec -> enc is the identity except {0x7F,0xFF,0x80} -> 0x00
    b = torch.randint(0, 256, (1 << 30,), dtype=torch.uint8, device=DEV, generator=g)
    h = _dequant_capi(b, torch.float16)
    rb = _encode_capi(h)
    expect = torch.where(((b & 0x7F) == 0x7F) | (b == 0x80), torch.zeros_like(b), b)
    assert torch.equal(rb, expect)


# ------------------------------------------------------------------ batched casts (many tensors, one launch)

def _oracle_encode(x):
    if x.dtype == torch.bfloat16:
        return c_oracle.encode_bf16_bits(x.view(torch.int16).numpy().view(np.uint16))
    return c_oracle.encode(x.numpy())


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_batch_casts_ragged_spans(dtype):
    """fp8b_encode_batch / fp8b_dequant_batch over ragged, empty, sub-vector and MISALIGNED spans carved out of
    one arena: every span bit-exact against the C oracle, and not a byte written outside the spans."""
    sizes = [0, 1, 3, 7, 8, 9, 8191, 8192, 8193, 1024 * 8 * 3 + 5, 100003, 1 << 20, 0, 17, (1 << 21) + 11]
    gaps = [0, 16, 16, 2, 16, 6, 16, 16, 16, 16, 10, 16, 16, 16, 16]     # element gaps: some starts lose 16-B alignment
    total = sum(sizes) + sum(gaps) + 64
    g = torch.Generator().manual_seed(123)
    arena = (torch.randn(total, generator=g) * 3.0).to(dtype)
    arena[::97] = 0.0
    arena[5::1013] = -0.0
    ad = arena.to(DEV)
    out = torch.full((total,), 0xAB, dtype=torch.uint8, device=DEV)
    esz = arena.element_size()
    offs, off = [], 8
    for n, gap in zip(sizes, gaps):
        offs.append(off)
        off += n + gap
    spans = make_spans([(ad.data_ptr() + esz * o_, out.data_ptr() + o_, n) for o_, n in zip(offs, sizes)])
    rc = capi().fp8b_encode_batch(spans, len(sizes), dt_code(dtype), stream_ptr())
    assert rc == 0, capi().fp8b_status_string(rc)
    got = out.cpu().numpy()
    expect = np.full(total, 0xAB, dtype=np.uint8)
    for o_, n in zip(offs, sizes):
        expect[o_:o_ + n] = _oracle_encode(arena[o_:o_ + n])
    assert np.array_equal(got, expect)

    for odt in (torch.float16, torch.bfloat16, torch.float32):
        wide = torch.full((total,), 7.0, dtype=odt, device=DEV)
        src = torch.from_numpy(expect).to(DEV)
        spans = make_spans([(src.data_ptr() + o_, wide.data_ptr() + wide.element_size() * o_, n) for o_, n in zip(offs, sizes)])
        rc = capi().fp8b_dequant_batch(spans, len(sizes), dt_code(odt), stream_ptr())
        assert rc == 0, capi().fp8b_status_string(rc)
        w = to_np(wide)
        ref = np.full(total, 7.0, dtype=np.float32)
        for o_, n in zip(offs, sizes):
            ref[o_:o_ + n] = o.decode(expect[o_:o_ + n])
        assert np.array_equal(w.view(np.uint32), ref.view(np.uint32))


def test_batch_casts_many_tensors_python_api():
    """More tensors than one span table holds (512), mixed dtypes and shapes, through fp8_mps_native."""
    import fp8_mps_native
    g = torch.Generator().manual_seed(9)
    dts = [torch.bfloat16, torch.float16, torch.float32]
    xs = [(torch.randn(1 + (i * 37) % 300, 1 + (i * 11) % 50, generator=g) * (0.01 + i % 7)).to(dts[i % 3]) for i in range(1100)]
    xs.append(torch.empty(0, 4, dtype=torch.bfloat16))
    qs = fp8_mps_native.fp8_encode_many([x.to(DEV) for x in xs])
    assert len(qs) == len(xs)
    for x, q in zip(xs, qs):
        assert q.shape == x.shape and q.dtype == torch.uint8
        assert np.array_equal(q.cpu().numpy().reshape(-1), _oracle_encode(x.reshape(-1)))
    ws = fp8_mps_native.fp8_dequantize_many(qs, torch.bfloat16)
    for q, w in zip(qs, ws):
        assert w.shape == q.shape and w.dtype == torch.bfloat16
        assert np.array_equal(to_np(w).reshape(-1).view(np.uint32), o.decode(q.cpu().numpy().reshape(-1)).view(np.uint32))
    assert fp8_mps_native.fp8_encode_many([]) == []


def test_batch_casts_validation():
    L = capi()
    x = torch.zeros(16, dtype=torch.bfloat16, device=DEV)
    q = torch.zeros(16, dtype=torch.uint8, device=DEV)
    assert L.fp8b_encode_batch(None, 0, BF16, stream_ptr()) == 0
    assert L.fp8b_encode_batch(None, 2, BF16, stream_ptr()) == -1
    assert L.fp8b_encode_batch(make_spans([(x.data_ptr(), q.data_ptr(), 16)]), 1, 9, stream_ptr()) == -1
    assert L.fp8b_encode_batch(make_spans([(None, q.data_ptr(), 16)]), 1, BF16, stream_ptr()) == -1
    assert L.fp8b_dequant_batch(make_spans([(q.data_ptr(), None, 4)]), 1, F16, stream_ptr()) == -1
    assert L.fp8b_dequant_batch(make_spans([(None, None, 0)]), 1, F16, stream_ptr()) == 0


def test_casts_under_pdl_see_fresh_data():
    """The tile kernels are launched with programmatic dependent launch (resident before their predecessor has
    finished).  Inputs produced by the kernel just before -- a torch op, or another cast -- must still be seen:
    regenerate x on the device right before every call and chain encode -> dequant without a sync."""
    import fp8_mps_native
    g = torch.Generator(device=DEV).manual_seed(11)
    n = (1 << 22) + 24
    for it in range(25):
        x = (torch.randn(n, device=DEV, generator=g) * (0.5 + it)).to(torch.bfloat16)
        q = fp8_mps_native.fp8_encode(x)                       # predecessor: the torch cast kernel that wrote x
        h = fp8_mps_native.fp8_dequantize_to(q, torch.float16)  # predecessor: our own encode kernel
        qq, inv = fp8_mps_native.fp8_quantize(x)               # amax -> finalize -> encode(prescale) chain
        torch.cuda.synchronize()
        q_ref = fp8_mps_native.fp8_encode(x)
        torch.cuda.synchronize()
        h_ref = fp8_mps_native.fp8_dequantize_to(q_ref, torch.float16)
        torch.cuda.synchronize()
        qq_ref, inv_ref = fp8_mps_native.fp8_quantize(x)
        torch.cuda.synchronize()
        assert torch.equal(q, q_ref) and torch.equal(h, h_ref), f"iteration {it}"
        assert torch.equal(qq, qq_ref) and torch.equal(inv, inv_ref), f"iteration {it} (quantize)"
    xs = x[:70001].float().cpu()
    assert np.array_equal(q[:70001].cpu().numpy(), c_oracle.encode(xs.numpy()))


# ------------------------------------------------------------------ float8_e5m2 decode

@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_e5m2_decode_all_patterns_and_sizes(dtype):
    """e5m2 -> wide against the oracle table (pinned to torch's CPU cast): bit-exact for non-NaN, NaN stays NaN;
    vector body, ragged tail and the unaligned scalar path."""
    L = capi()
    table = o.decode_e5m2(np.arange(256, dtype=np.uint8))
    for n, off in ((256, 0), (7, 0), (4099, 0), ((1 << 20) + 5, 0), (70001, 3)):
        rng = np.random.default_rng(n)
        b = np.arange(256, dtype=np.uint8) if n == 256 else rng.integers(0, 256, n + off, dtype=np.uint8)
        src = torch.from_numpy(b).to(DEV)
        out = torch.empty(n, dtype=dtype, device=DEV)
        rc = L.fp8b_dequant_fmt(src.data_ptr() + off, 1, p(out), dt_code(dtype), n, None, stream_ptr())
        assert rc == 0, L.fp8b_status_string(rc)
        got = to_np(out)
        ref = table[b[off:off + n]]
        nan = np.isnan(ref)
        assert np.array_equal(np.isnan(got), nan)
        assert np.array_equal(got[~nan].view(np.uint32), ref[~nan].view(np.uint32))
    # same as torch's own cast on the device, and through the patched Tensor.to
    import fp8_mps_patch
    e5 = torch.arange(256, dtype=torch.int32).to(torch.uint8).to(DEV).view(torch.float8_e5m2)
    want = e5.to(dtype)
    fp8_mps_patch.install()
    try:
        got_t = e5.to(dtype)
    finally:
        fp8_mps_patch.uninstall()
    assert torch.equal(torch.nan_to_num(got_t.float(), nan=123.0), torch.nan_to_num(want.float(), nan=123.0))
    assert L.fp8b_dequant_fmt(p(src), 2, p(out), dt_code(dtype), 4, None, stream_ptr()) == -1      # unknown format


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_big_tile_paths_256bit_and_128bit(dtype):
    """Large tensors take the 64 KB-tile kernels: 256-bit loads when the tensor is 32-byte aligned, the 16-byte
    variant otherwise; both, single and batched, must give the bytes of the (oracle-checked) small-tile path."""
    L = capi()
    n = 68 * (1 << 20) + 13                                 # >= 2^26 elements -> 64 KB tiles with 256-bit loads; ragged tail
    g = torch.Generator(device=DEV).manual_seed(77)
    esz = torch.empty(0, dtype=dtype).element_size()
    arena = (torch.randn(3 * n + 64, device=DEV, generator=g) * 2.0).to(dtype)
    out = torch.zeros(3 * n + 64, dtype=torch.uint8, device=DEV)
    offs = [0, n + 16 // esz + (16 // esz) * ((n // (16 // esz)) % 2), 2 * n + 48 // esz]   # 32-B aligned, 16-B only, 16-B only
    offs[1] = ((n * esz + 31) // 32 * 32 + 16) // esz        # exactly 16 mod 32 bytes
    offs[2] = ((2 * n * esz + 64 + 31) // 32 * 32) // esz    # 32-B aligned again, but its fp8 side is offset by the same elements
    for o_ in offs:
        rc = L.fp8b_encode(arena.data_ptr() + esz * o_, dt_code(dtype), out.data_ptr() + o_, n, None, stream_ptr())
        assert rc == 0
    L.fp8b_set_option(19, 1)                                # FP8B_OPT_TUNE_CAST_SHAPE = 1: always the small 16-byte tiles
    try:
        ref = torch.zeros_like(out)
        for o_ in offs:
            assert L.fp8b_encode(arena.data_ptr() + esz * o_, dt_code(dtype), ref.data_ptr() + o_, n, None, stream_ptr()) == 0
    finally:
        L.fp8b_set_option(19, -1)
    assert torch.equal(out, ref)
    samp = slice(offs[1], offs[1] + 50001)
    x = arena[samp].cpu()
    want = _oracle_encode(x) if dtype == torch.bfloat16 else c_oracle.encode(x.numpy())
    assert np.array_equal(out[samp].cpu().numpy(), want)
    batched = torch.zeros_like(out)
    spans = make_spans([(arena.data_ptr() + esz * o_, batched.data_ptr() + o_, n) for o_ in offs])
    assert L.fp8b_encode_batch(spans, 3, dt_code(dtype), stream_ptr()) == 0
    assert torch.equal(batched, ref)
