"""GPU parity: `_scaled_mm` (GEMV, tcgen05 GEMM, SIMT GEMM) vs the fp32 dequantise-then-matmul oracle.

Tolerances (relative RMSE against oracle/fp8_oracle.scaled_mm on identical bytes, fp64-summed):
    fp32 out  <= 5e-6  for the CUDA-core kernels (exact products, fp32 accumulation; only the summation
                       order differs from the oracle)
              <= 1e-4  for the tensor-core kernel (accumulation precision of tcgen05 kind::f8f6f4 is
                       whatever the hardware does; measured and printed by test_tcgen05_accumulation_precision)
    fp16 out  <= 5e-4  (output rounding floor 2.1e-4, SURVEY 8c)
    bf16 out  <= 3e-3  (output rounding floor 1.7e-3)
plus max-abs <= 2 ulp of the output dtype at the oracle's RMS magnitude scale.
The reference's own gates are far looser: rel-RMSE < 15 % against the UN-quantised fp32 product
(test_fp8_metal.py:122,161,215) and 1e-4 abs between its two dispatchers on tiny shapes
(test_cross_validation.py:187)."""
import numpy as np
import pytest
import torch

import fp8_oracle as o
from _util import ALGO_AUTO, ALGO_GEMV, ALGO_SIMT, ALGO_TCGEN05, capi, dt_name, mm_capi, to_np

pytestmark = pytest.mark.gpu
DEV = "cuda"

TOL = {"f32": 5e-6, "f16": 5e-4, "bf16": 3e-3}
ULP = {"f32": 2.0 ** -23, "f16": 2.0 ** -10, "bf16": 2.0 ** -7}


def _rand_fp8(shape, seed, kind="bytes"):
    rng = np.random.default_rng(seed)
    if kind == "bytes":                                   # every byte value, NaN codes excluded
        b = rng.integers(0, 256, shape, dtype=np.uint8)
        b[(b & 0x7F) == 0x7F] = 0x3C
        return b
    x = rng.standard_normal(shape).astype(np.float32)     # "randn -> quantise" like the reference tests
    q, inv = o.fp8_quantize(x)
    return q, inv


def _check(got_t, ref, out_dtype, tol=None, what=""):
    name = dt_name(out_dtype)
    got = to_np(got_t)
    assert got.shape == ref.shape
    assert np.isfinite(got).all(), what
    e = o.rel_rmse(got, ref)
    rms = float(np.sqrt(np.mean(ref.astype(np.float64) ** 2)))
    mx = float(np.abs(got.astype(np.float64) - ref).max())
    tol = TOL[name] if tol is None else tol
    assert e <= tol, f"{what}: rel-RMSE {e:.3e} > {tol:.1e}"
    # max-abs: 2 ulp of the out dtype at the larger of the RMS and the element magnitude
    scale = np.maximum(np.abs(ref), rms)
    lim = 2 * ULP[name] * scale + (tol * 40) * rms
    assert (np.abs(got.astype(np.float64) - ref) <= lim).all(), f"{what}: max-abs {mx:.3e}"
    return e


def _run_case(M, K, N, out_dtype, algo, seed, per_row_a=False, per_row_b=False, bias_dtype=None,
              scale_result=False, kind="bytes", tol=None):
    A = _rand_fp8((M, K), seed, "bytes")
    B = _rand_fp8((N, K), seed + 1, "bytes")
    rng = np.random.default_rng(seed + 2)
    sa = (rng.random(M if per_row_a else 1).astype(np.float32) + 0.5) * 0.01
    sb = (rng.random(N if per_row_b else 1).astype(np.float32) + 0.5) * 0.02
    bias = rng.standard_normal(N).astype(np.float32) if bias_dtype is not None else None
    sr = np.array([0.75], dtype=np.float32) if scale_result else None
    tA, tB = torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV)
    tbias = None
    if bias is not None:
        tbias = torch.from_numpy(bias).to(DEV).to(bias_dtype)
        bias = to_np(tbias)                               # what the kernel actually sees
    tsr = torch.from_numpy(sr).to(DEV) if sr is not None else None
    rc, C = mm_capi(tA, tB, torch.from_numpy(sa), torch.from_numpy(sb), tbias, tsr, out_dtype, algo)
    assert rc == 0, capi().fp8b_status_string(rc)
    ref = o.scaled_mm(A, B, sa, sb, bias, sr, dt_name(out_dtype))
    return _check(C, ref, out_dtype, tol, f"M{M} K{K} N{N} {dt_name(out_dtype)} algo{algo}")


# ------------------------------------------------------------------ GEMV (M <= 16)

@pytest.mark.parametrize("M,K,N,odt,kw", [
    (1, 512, 256, None, {}),                                   # test_fp8_metal.py:191-218
    (1, 4096, 4096, torch.float16, {}),                        # BASELINE config 1
    (1, 14336, 4096, torch.bfloat16, {}),                      # BASELINE config 2
    (4, 4096, 4096, torch.bfloat16, {"bias_dtype": torch.bfloat16}),   # BASELINE config 3
    (1, 4096, 64, None, {}),                                   # small N -> cluster split-K
    (2, 8192, 40, None, {"per_row_b": True}),                  # split-K, ragged N
    (3, 4112, 1001, torch.float16, {"per_row_a": True, "per_row_b": True, "bias_dtype": torch.float32}),
    (5, 1024, 333, None, {"scale_result": True}),              # M > 4: two passes
    (16, 2048, 512, torch.bfloat16, {"per_row_a": True}),
    (1, 16, 8, None, {}),                                      # minimum aligned K
    (1, 100000, 24, None, {}),                                 # K panel loop (x does not fit one smem panel) + split
    (4, 65536, 16, None, {}),
    (2, 37, 5, None, {}),                                      # K % 16 != 0 -> generic kernel
    (1, 3, 2, None, {}),
    (7, 130, 33, torch.float16, {"bias_dtype": torch.float16}),
])
def test_gemv(M, K, N, odt, kw):
    _run_case(M, K, N, odt, ALGO_AUTO, seed=M * 7 + K + N, **kw)
    if odt is None:
        _run_case(M, K, N, odt, ALGO_GEMV, seed=K, kind="bytes", **kw)


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("M,K,N,odt,kw", [
    (1, 14336, 4096, torch.bfloat16, {}),
    (1, 4096, 4096, None, {}),
    (4, 4096, 4096, torch.bfloat16, {"bias_dtype": torch.bfloat16}),
    (8, 2048, 100, None, {"per_row_a": True, "per_row_b": True}),
    (9, 1040, 50, torch.float16, {"scale_result": True}),
    (16, 4096, 24, None, {"per_row_a": True}),
    (3, 80, 17, None, {}),
])
def test_gemv_both_kernels(tune, impl, M, K, N, odt, kw):
    """FP8B_GEMV_IMPL=1: CUDA-core FHFMA kernel; =2: warp-level tensor-core kernel.  Both must meet
    the same tolerance on every M in 1..16."""
    tune("GEMV_IMPL", impl)
    _run_case(M, K, N, odt, ALGO_GEMV, seed=impl + M + K + N, **kw)


@pytest.mark.parametrize("impl", [3, 4])
@pytest.mark.parametrize("M", [1, 4, 16])
def test_gemv_retired_impl_values_take_the_built_in_rule(tune, impl, M):
    """FP8B_GEMV_IMPL = 3 / 4 selected two GEMV kernels that measured slower and were removed (DESIGN.md 3.2, 3.3b).
    Such a value must still work: one launch, bit-identical to the built-in rule."""
    A = torch.from_numpy(_rand_fp8((M, 2048), 5)).to(DEV)
    B = torch.from_numpy(_rand_fp8((1000, 2048), 6)).to(DEV)
    s = torch.tensor([0.01], device=DEV)
    rc, ref = mm_capi(A, B, s, s, algo=ALGO_GEMV)
    assert rc == 0
    tune("GEMV_IMPL", impl)
    L = capi()
    n0 = L.fp8b_launch_count()
    rc, out = mm_capi(A, B, s, s, algo=ALGO_GEMV)
    assert rc == 0
    assert L.fp8b_launch_count() == n0 + 1
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


def test_gemv_mma_nan_bytes(tune):
    tune("GEMV_IMPL", 2)
    rng = np.random.default_rng(1)
    A = rng.integers(0, 256, (5, 1024), dtype=np.uint8)
    B = rng.integers(0, 256, (70, 1024), dtype=np.uint8)
    sa = np.array([0.5], np.float32)
    sb = np.array([0.25], np.float32)
    rc, C = mm_capi(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(sa), torch.from_numpy(sb))
    assert rc == 0
    _check(C, o.scaled_mm(A, B, sa, sb), None, what="mma nan bytes")


def test_gemv_matches_reference_summation_to_fp32_noise():
    """Against the plain-C restatement of the shader's own loop order (oracle/fp8_oracle.c):
    same fp32 products, different summation order only."""
    import c_oracle
    A = _rand_fp8((1, 4096), 1)
    B = _rand_fp8((512, 4096), 2)
    sa = np.array([0.01], np.float32)
    sb = np.array([0.03], np.float32)
    rc, C = mm_capi(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(sa), torch.from_numpy(sb))
    assert rc == 0
    assert o.rel_rmse(to_np(C), c_oracle.scaled_mm(A, B, sa, sb)) < 2e-6


def test_gemv_nan_bytes_decode_to_zero():
    """fp8_matmul.metal:21 -- 0x7F / 0xFF contribute 0; the fast path repairs NaN accumulators."""
    rng = np.random.default_rng(0)
    A = rng.integers(0, 256, (2, 2048), dtype=np.uint8)       # NaN codes left in
    B = rng.integers(0, 256, (96, 2048), dtype=np.uint8)
    B[5, 100] = 0x7F
    B[17, 7] = 0xFF
    A[1, 33] = 0x7F
    sa = np.array([1.0], np.float32)
    sb = np.array([1.0], np.float32)
    rc, C = mm_capi(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(sa), torch.from_numpy(sb))
    assert rc == 0
    _check(C, o.scaled_mm(A, B, sa, sb), None, what="nan bytes")


def test_gemv_rejects_large_m_when_forced():
    A = torch.zeros(17, 64, dtype=torch.uint8, device=DEV)
    B = torch.zeros(8, 64, dtype=torch.uint8, device=DEV)
    rc, _ = mm_capi(A, B, torch.ones(1), torch.ones(1), algo=ALGO_GEMV)
    assert rc == -2                                           # FP8B_ERR_UNSUPPORTED, no silent re-dispatch


# ------------------------------------------------------------------ tensor-core GEMM

def test_tcgen05_accumulation_precision():
    """Measures (and bounds) how far tcgen05 kind::f8f6f4 accumulation is from exact fp32."""
    res = {}
    for K in (128, 1024, 4096, 16384):
        res[K] = _run_case(256, K, 256, None, ALGO_TCGEN05, seed=K, tol=1e-4)
    print("tcgen05 fp32-out rel-RMSE vs exact:", {k: f"{v:.2e}" for k, v in res.items()})


@pytest.mark.parametrize("M,K,N,odt,kw", [
    (128, 128, 128, None, {}),
    (64, 256, 128, None, {}),                                 # test_fp8_metal.py:97-164 shape
    (32, 64, 48, None, {}),                                   # test_cross_validation.py:166-198 shape
    (17, 64, 40, torch.float16, {"bias_dtype": torch.float16}),
    (256, 512, 384, torch.bfloat16, {"per_row_a": True, "per_row_b": True}),
    (200, 336, 1000, torch.bfloat16, {"bias_dtype": torch.bfloat16, "scale_result": True}),   # ragged everything
    (129, 2064, 257, None, {"per_row_b": True}),
    (1000, 1024, 3000, torch.float16, {}),                    # multi-tile, both tile widths
    (2048, 3072, 4096, torch.bfloat16, {"bias_dtype": torch.float32}),   # 128x256 tiles, > 2 waves
    (4, 4096, 512, None, {}),                                 # small M forced onto tensor cores
])
def test_tcgen05_gemm(M, K, N, odt, kw):
    tol = 1e-4 if odt is None else None
    _run_case(M, K, N, odt, ALGO_TCGEN05, seed=M + K + N, tol=tol, **kw)


@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("M,K,N,odt,kw", [
    (256, 512, 384, torch.bfloat16, {"per_row_a": True, "per_row_b": True}),
    (200, 336, 1000, None, {"bias_dtype": torch.float32, "scale_result": True}),      # ragged M, N, K
    (1000, 1024, 3000, torch.float16, {"bias_dtype": torch.float16}),
    (640, 3072, 1536, torch.bfloat16, {}),                                            # an 8-way shard of the FLUX linear
    (130, 4096, 260, None, {"per_row_b": True}),
    (2304, 256, 2560, torch.bfloat16, {"per_row_b": True, "bias_dtype": torch.bfloat16}),   # 9x10 pair tiles: 74 + 16 -> last wave split in half-width tiles
    (2304, 128, 2500, None, {"per_row_a": True}),                                         # same, ragged N, fp32 out
])
def test_tcgen05_all_tile_configs(tune, cfg, M, K, N, odt, kw):
    """FP8B_GEMM_CFG: 1 = 128x256 tile, one CTA; 2 = 128x128, one CTA; 3 = 256x256, CTA pair
    (cta_group::2); 4 = 256x128, CTA pair; 5 = 256x192, CTA pair.  Every configuration must serve every shape."""
    tune("GEMM_CFG", cfg)
    tol = 1e-4 if odt is None else None
    _run_case(M, K, N, odt, ALGO_TCGEN05, seed=cfg + M + N, tol=tol, **kw)


@pytest.mark.parametrize("odt", [None, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("kind", range(8))
def test_tcgen05_every_epilogue_term_combination(tune, kind, odt):
    """The TMA-store epilogue compiles one copy of its tile loop per combination of optional terms (per-column scale_b,
    bias, scale_result): run each of the eight, for every output dtype, on a shape with a ragged column edge (the
    out-of-line edge loads), several tiles per CTA pair and a K tail."""
    tune("GEMM_SPLITK", 1)
    kw = {"per_row_b": bool(kind & 1), "scale_result": bool(kind & 4)}
    if kind & 2:
        kw["bias_dtype"] = torch.float32 if odt is None else odt
    M, K, N = 520, 400, 40 * 8 + 24 if odt is None else 1160                # N * esz % 16 == 0 -> TMA-store epilogue
    tol = 1e-4 if odt is None else None
    for cfg in (2, 4):
        tune("GEMM_CFG", cfg)
        _run_case(M, K, N, odt, ALGO_TCGEN05, seed=50 + kind, per_row_a=bool(kind & 1), tol=tol, **kw)


@pytest.mark.parametrize("split", [2, 4])
@pytest.mark.parametrize("M,K,N,odt,kw", [
    (32, 3072, 3072, torch.bfloat16, {}),                                             # 24 tiles: the shape the plan exists for
    (256, 3072, 3072, torch.bfloat16, {"bias_dtype": torch.bfloat16}),
    (100, 4096, 4096, torch.float16, {"per_row_a": True, "per_row_b": True}),
    (333, 2048, 1000, None, {"bias_dtype": torch.float32, "scale_result": True}),     # ragged M and N, fp32 out
    (17, 528, 40, None, {"per_row_b": True}),                                         # K tail block, one ragged tile
    (130, 1024, 260, torch.bfloat16, {"per_row_a": True, "bias_dtype": torch.float16}),
    (128, 512, 136, torch.float16, {}),                                               # 4 k-blocks: one per CTA when split 4 ways
    (2048, 1024, 2048, torch.bfloat16, {}),                                           # 256 tiles: more clusters than the GPU holds at once
])
def test_tcgen05_split_k(tune, split, M, K, N, odt, kw):
    """Split-K plan (cluster of 2 / 4 CTAs per 128 x 128 tile, reduce-scatter over distributed shared memory): same
    tolerances against the oracle as every other plan; bit-identical from run to run (partials are added in rank order)."""
    tune("GEMM_SPLITK", split)
    tol = 1e-4 if odt is None else None
    _run_case(M, K, N, odt, ALGO_TCGEN05, seed=split + M + N, tol=tol, **kw)


def test_tcgen05_split_k_is_deterministic_and_automatic(tune):
    import fp8_mps_native
    M, K, N = 64, 3072, 3072
    A = torch.from_numpy(_rand_fp8((M, K), 21)).to(DEV)
    B = torch.from_numpy(_rand_fp8((N, K), 22)).to(DEV)
    sa = torch.tensor([0.01], device=DEV); sb = torch.tensor([0.02], device=DEV)
    L = capi()
    n0 = L.fp8b_launch_count()
    auto = fp8_mps_native.fp8_scaled_mm_fused(A, B, sa, sb, None, None, torch.bfloat16)       # 24 tiles, 24 k-blocks -> split 4
    assert L.fp8b_launch_count() - n0 == 1
    tune("GEMM_SPLITK", 4)
    runs = [fp8_mps_native.fp8_scaled_mm_fused(A, B, sa, sb, None, None, torch.bfloat16).clone() for _ in range(5)]
    tune("GEMM_SPLITK", 1)
    plain = fp8_mps_native.fp8_scaled_mm_fused(A, B, sa, sb, None, None, torch.bfloat16)
    torch.cuda.synchronize()
    assert all(torch.equal(r, runs[0]) for r in runs)
    assert torch.equal(auto, runs[0])                          # the automatic rule picked the 4-way split for this shape
    # the one-CTA-per-tile plan rounds differently (sequential accumulation over all of K) but agrees to bf16 resolution
    err = o.rel_rmse(to_np(plain), to_np(runs[0]))
    assert err < 3e-3, err


def test_tcgen05_split_k_random_shapes(tune):
    """Stress of the cluster protocol (DSMEM bulk copies, receive barriers, short A box, ragged edges): 80 random shapes,
    both split factors, fp32 out, against the one-CTA-per-tile plan of the same kernel family -- the two differ only in
    the rounding of the partial sums (a few 1e-6 rel-RMSE at K = 6000; bound 1e-5); a lost or early-read block would be off by orders of magnitude.
    Every split result must also repeat bit for bit."""
    import fp8_mps_native
    rng = np.random.default_rng(2024)
    sa = torch.tensor([0.01], device=DEV); sb = torch.tensor([0.02], device=DEV)
    for case in range(80):
        M = int(rng.integers(17, 400)); N = int(rng.integers(8, 1500)); K = 16 * int(rng.integers(32, 400))
        split = 2 if case % 2 else 4
        A = torch.from_numpy(_rand_fp8((M, K), 1000 + case)).to(DEV)
        B = torch.from_numpy(_rand_fp8((N, K), 2000 + case)).to(DEV)
        tune("GEMM_SPLITK", 1)
        plain = fp8_mps_native.fp8_scaled_mm_fused(A, B, sa, sb, None, None, None, algo=ALGO_TCGEN05)
        tune("GEMM_SPLITK", split)
        y1 = fp8_mps_native.fp8_scaled_mm_fused(A, B, sa, sb, None, None, None, algo=ALGO_TCGEN05).clone()
        y2 = fp8_mps_native.fp8_scaled_mm_fused(A, B, sa, sb, None, None, None, algo=ALGO_TCGEN05)
        torch.cuda.synchronize()
        assert torch.equal(y1, y2), (case, M, K, N, split)
        err = o.rel_rmse(to_np(y1), to_np(plain))
        assert err <= 1e-5, (case, M, K, N, split, err)


def test_tcgen05_split_k_nan_bytes_and_strided_output(tune):
    tune("GEMM_SPLITK", 2)
    rng = np.random.default_rng(14)
    M, K, N = 96, 1024, 200
    A = rng.integers(0, 256, (M, K), dtype=np.uint8)
    B = rng.integers(0, 256, (N, K), dtype=np.uint8)          # ~0.8 % NaN codes
    sa = np.array([0.02], np.float32); sb = np.array([0.01], np.float32)
    wide = torch.full((M, 2 * N + 8), 7.0, dtype=torch.bfloat16, device=DEV)
    out = wide[:, 8:8 + N]                                    # column shard of a wider matrix (ldc > N)
    rc, C = mm_capi(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(sa),
                    torch.from_numpy(sb), out_dtype=torch.bfloat16, algo=ALGO_TCGEN05, out=out)
    assert rc == 0
    _check(out, o.scaled_mm(A, B, sa, sb, out_dtype="bf16"), torch.bfloat16, what="split-K nan+strided")
    assert bool((wide[:, :8] == 7.0).all()) and bool((wide[:, 8 + N:] == 7.0).all())   # nothing outside the shard


@pytest.mark.parametrize("M,K,N,odt,kw", [
    (33, 37, 65, None, {}),
    (64, 256, 128, torch.bfloat16, {"bias_dtype": torch.bfloat16}),
    (130, 1000, 70, torch.float16, {"per_row_a": True, "per_row_b": True, "scale_result": True}),
])
def test_simt_gemm(M, K, N, odt, kw):
    _run_case(M, K, N, odt, ALGO_SIMT, seed=M * K + N, **kw)


def test_auto_dispatch_rules():
    L = capi()
    A = torch.zeros(64, 256, dtype=torch.uint8, device=DEV)
    B = torch.zeros(128, 256, dtype=torch.uint8, device=DEV)
    sel = lambda a, b: L.fp8b_scaled_mm_select(a.data_ptr(), b.data_ptr(), None, 0, a.shape[0], b.shape[0], a.shape[1], b.shape[0])
    assert sel(A[:16], B) == ALGO_GEMV                        # M <= 16 (fp8_mps_native.py:208)
    assert sel(A, B) == ALGO_TCGEN05
    A2 = torch.zeros(64, 250, dtype=torch.uint8, device=DEV)
    B2 = torch.zeros(128, 250, dtype=torch.uint8, device=DEV)
    assert sel(A2, B2) == ALGO_SIMT                           # K % 16 != 0: TMA cannot describe it
    rc, _ = mm_capi(A2, B2, torch.ones(1), torch.ones(1), algo=ALGO_TCGEN05)
    assert rc == -2
    _run_case(40, 250, 72, None, ALGO_AUTO, seed=9)           # ... and AUTO still computes it on the GPU


def test_tcgen05_nan_bytes_and_strided_output():
    rng = np.random.default_rng(4)
    M, K, N = 160, 512, 320
    A = rng.integers(0, 256, (M, K), dtype=np.uint8)
    B = rng.integers(0, 256, (N, K), dtype=np.uint8)          # ~0.8 % NaN codes
    sa = np.array([0.02], np.float32)
    sb = np.array([0.01], np.float32)
    wide = torch.full((M, 2 * N + 8), 7.0, dtype=torch.bfloat16, device=DEV)
    out = wide[:, 8:8 + N]                                    # column shard of a wider matrix (ldc > N)
    rc, C = mm_capi(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(sa),
                    torch.from_numpy(sb), out_dtype=torch.bfloat16, algo=ALGO_TCGEN05, out=out)
    assert rc == 0
    _check(out, o.scaled_mm(A, B, sa, sb, out_dtype="bf16"), torch.bfloat16, what="nan+strided")
    assert bool((wide[:, :8] == 7.0).all()) and bool((wide[:, 8 + N:] == 7.0).all())   # nothing outside the shard


def test_flux_linear_full_size_against_oracle_and_simt():
    """BASELINE config 4 at full size: M=4096 K=3072 N=12288, per-tensor scales, bf16 out.
    Oracle: numpy fp32 BLAS dequantise-then-matmul on a 512-row slab (exact fp64 on a corner),
    plus the independent CUDA-core kernel on the whole matrix."""
    M, K, N = 4096, 3072, 12288
    g = torch.Generator().manual_seed(4)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g)
    qa, sa = o.fp8_quantize(a.numpy())
    qw, sw = o.fp8_quantize(w.numpy())
    tA, tW = torch.from_numpy(qa).to(DEV), torch.from_numpy(qw).to(DEV)
    rc, C = mm_capi(tA, tW, torch.from_numpy(sa), torch.from_numpy(sw), out_dtype=torch.bfloat16, algo=ALGO_TCGEN05)
    assert rc == 0
    rc, C32 = mm_capi(tA, tW, torch.from_numpy(sa), torch.from_numpy(sw), out_dtype=None, algo=ALGO_TCGEN05)
    assert rc == 0
    rc, S32 = mm_capi(tA, tW, torch.from_numpy(sa), torch.from_numpy(sw), out_dtype=None, algo=ALGO_SIMT)
    assert rc == 0
    e_simt = o.rel_rmse(to_np(C32), to_np(S32))
    assert e_simt < 1e-4, e_simt
    ref = o.scaled_mm(qa[:512], qw, sa, sw, out_dtype="bf16", accum="f32")
    _check(C[:512], ref, torch.bfloat16, what="flux slab")
    ref64 = o.scaled_mm(qa[-128:], qw[-256:], sa, sw)
    _check(C32[-128:, -256:], ref64, None, tol=1e-4, what="flux corner fp64")
    # the reference's own gate: within 15 % of the un-quantised product (test_fp8_metal.py:122)
    full = (a[:256] @ w.T).numpy()
    assert o.rel_rmse(to_np(C[:256]), full) < 0.15


# ------------------------------------------------------------------ through the reference-shaped API

def test_native_api_shapes_and_asserts():
    import fp8_mps_native
    M, K, N = 64, 256, 128                                    # test_fp8_metal.py:128-164
    g = torch.Generator().manual_seed(0)
    A = torch.randn(M, K, generator=g)
    B = torch.randn(N, K, generator=g)
    ref = (A @ B.T).numpy()
    qa, sa = fp8_mps_native.fp8_quantize(A)
    qb, sb = fp8_mps_native.fp8_quantize(B)
    for fn in (fp8_mps_native.fp8_scaled_mm, fp8_mps_native.fp8_scaled_mm_auto, fp8_mps_native.fp8_scaled_mm_fast):
        r = fn(qa, qb, sa, sb)
        assert r.dtype == torch.float32 and r.shape == (M, N) and r.device.type == "cuda"
        assert o.rel_rmse(to_np(r), ref) < 0.15
        assert o.rel_rmse(to_np(r), o.scaled_mm(qa.cpu().numpy(), qb.cpu().numpy(), sa.cpu().numpy(), sb.cpu().numpy())) < 1e-4
    r = fp8_mps_native.fp8_scaled_mm(qa.cpu(), qb.cpu(), sa.cpu(), sb.cpu())      # CPU inputs are moved (native.py:63-70)
    assert r.device.type == "cuda"
    with pytest.raises(AssertionError):
        fp8_mps_native.fp8_scaled_mm(qa.float(), qb, sa, sb)                     # dtype assert (native.py:55)
    with pytest.raises(AssertionError):
        fp8_mps_native.fp8_scaled_mm(qa, qb[:, :100].contiguous(), sa, sb)       # K mismatch (native.py:60)
    with pytest.raises(AssertionError):
        fp8_mps_native.fp8_scaled_mm(qa.t(), qb, sa, sb)                         # contiguity (native.py:56)
    lib = fp8_mps_native._get_lib()                                              # bridge ops (fp8_bridge.cpp:361-371)
    with pytest.raises(RuntimeError):
        lib.fp8_scaled_mm(qa, qb[:, :100].contiguous(), sa, sb)
    q2, inv2 = lib.fp8_quantize(A.to(DEV))
    assert torch.equal(q2, qa) and torch.equal(inv2, sa)
    # vecmat (test_fp8_metal.py:191-218)
    x = torch.randn(1, 512, generator=g)
    W = torch.randn(256, 512, generator=g)
    xq, xs = fp8_mps_native.fp8_quantize(x)
    Wq, Ws = fp8_mps_native.fp8_quantize(W)
    r = fp8_mps_native.fp8_scaled_mm(xq, Wq, xs, Ws)
    assert r.shape == (1, 256) and o.rel_rmse(to_np(r), (x @ W.T).numpy()) < 0.15


def test_capi_argument_validation():
    """Error convention of the C ABI (include/fp8_b200.h): negative status, nothing launched, no fallback."""
    L = capi()
    A = torch.zeros(4, 64, dtype=torch.uint8, device=DEV)
    B = torch.zeros(8, 64, dtype=torch.uint8, device=DEV)
    one = torch.ones(1)
    n0 = L.fp8b_launch_count()
    rc, _ = mm_capi(A, B, torch.ones(3), one)                     # scale_a length not in {1, M}
    assert rc == -1
    rc, _ = mm_capi(A, B, one, torch.ones(5))                     # scale_b length not in {1, N}
    assert rc == -1
    rc, _ = mm_capi(A, B, one, one, algo=9)                       # unknown algorithm
    assert rc == -1
    C = torch.empty(4, 8, device=DEV)
    rc = L.fp8b_scaled_mm(A.data_ptr(), B.data_ptr(), C.data_ptr(), 0, 4, 8, 64, 4, one.to(DEV).data_ptr(), 1,
                          one.to(DEV).data_ptr(), 1, None, 0, None, None, 0, 0, None)     # ldc < N
    assert rc == -1
    rc = L.fp8b_scaled_mm(None, B.data_ptr(), C.data_ptr(), 0, 4, 8, 64, 8, one.to(DEV).data_ptr(), 1,
                          one.to(DEV).data_ptr(), 1, None, 0, None, None, 0, 0, None)     # null A
    assert rc == -1
    assert L.fp8b_launch_count() == n0
    assert L.fp8b_status_string(-2).startswith(b"unsupported")
    rc, out = mm_capi(A[:0], B, one, one)                         # M == 0 is a valid empty problem
    assert rc == 0 and out.shape == (0, 8)


@pytest.mark.parametrize("M,K,N,xdt,odt,kw", [
    (1, 14336, 4096, torch.bfloat16, torch.bfloat16, {}),
    (1, 4096, 512, torch.float32, None, {"bias": True}),
    (4, 4096, 300, torch.float16, torch.float16, {"per_row_b": True}),
    (7, 2048, 64, torch.bfloat16, None, {}),                      # two passes of <= 4 rows, cluster split-K
    (16, 512, 40, torch.float32, torch.bfloat16, {"bias": True, "per_row_b": True}),
    (1, 100000, 24, torch.float32, None, {}),                     # K panel loop
    (2, 100000, 24, torch.float32, None, {"tol": 3e-5}),         # tensor-core accumulation over a long K
    (3, 100, 50, torch.float32, None, {"ws_only": True}),         # ragged K: only the workspace plan can serve it (ADVICE r1)
    (1, 4099, 70, torch.bfloat16, torch.float16, {"ws_only": True, "bias": True}),
])
@pytest.mark.parametrize("single", [False, True])
def test_fused_dynamic_quantize_gemv(M, K, N, xdt, odt, kw, single):
    """fp8_linear_dynamic == the reference composition fp8_quantize(x) per row -> _scaled_mm, in one launch.
    The quantised activations must be the oracle's bytes exactly, so the only difference from the oracle result
    is fp32 summation order."""
    import fp8_mps_native
    g = torch.Generator().manual_seed(M * 13 + N)
    x = (torch.randn(M, K, generator=g) * (torch.rand(M, 1, generator=g) * 5 + 0.1)).to(xdt)
    if M > 2:
        x[2].zero_()                                              # amax == 0 -> scale 1.0
    W = _rand_fp8((N, K), M + K)
    sb = (np.random.default_rng(N).random(N if kw.get("per_row_b") else 1).astype(np.float32) + 0.5) * 0.02
    bias = torch.randn(N, generator=g).to(odt or torch.float32) if kw.get("bias") else None
    if kw.get("ws_only") and single:
        with pytest.raises(RuntimeError, match="unsupported"):      # no workspace + ragged K: refused, never a fallback
            fp8_mps_native.fp8_linear_dynamic(x.to(DEV), torch.from_numpy(W).to(DEV), torch.from_numpy(sb),
                                              None if bias is None else bias.to(DEV), odt, single_kernel=True)
        return
    y, inv = fp8_mps_native.fp8_linear_dynamic(x.to(DEV), torch.from_numpy(W).to(DEV), torch.from_numpy(sb),
                                               None if bias is None else bias.to(DEV), odt, single_kernel=single)
    assert y.shape == (M, N) and y.dtype == (odt or torch.float32) and inv.shape == (M,)
    qs, invs = zip(*[o.fp8_quantize(x[m].float().numpy()) for m in range(M)])
    q = np.stack(qs)
    inv_ref = np.concatenate(invs)
    assert np.array_equal(inv.cpu().numpy().view(np.uint32), inv_ref.view(np.uint32))
    ref = o.scaled_mm(q, W, inv_ref, sb, None if bias is None else to_np(bias), None, dt_name(odt))
    _check(y, ref, odt, tol=kw.get("tol"), what=f"fused dynamic M{M} K{K} N{N}")
    # and it equals the two-step path of this library bit for bit in the quantised operands
    q2, inv2 = fp8_mps_native.fp8_quantize_rowwise(x.to(DEV))
    assert np.array_equal(q2.cpu().numpy(), q)


@pytest.mark.parametrize("M", [1, 2, 12])
def test_pdl_chain_sees_fresh_activations(M):
    """Programmatic dependent launch regression: the GEMV is resident BEFORE its predecessor has written the
    activations, so every activation load must come after griddepcontrol.wait (a non-coherent load was hoisted
    above it once and read the previous call's bytes).  x is regenerated on the device right before each call and
    the workspace address is reused, so a stale read changes the result."""
    import fp8_mps_native
    K, N = 8192, 96
    g = torch.Generator(device=DEV).manual_seed(5)
    W = torch.from_numpy(_rand_fp8((N, K), 3)).to(DEV)
    sb = torch.tensor([0.02], device=DEV)
    for it in range(40):
        x = torch.randn(M, K, device=DEV, generator=g) * (1.0 + it)        # written by the kernel just before
        y, inv = fp8_mps_native.fp8_linear_dynamic(x, W, sb, None, None)
        q, inv2 = fp8_mps_native.fp8_quantize_rowwise(x)
        torch.cuda.synchronize()
        ref = fp8_mps_native.fp8_scaled_mm_fused(q, W, inv2, sb, None, None, None)   # no PDL on this path
        torch.cuda.synchronize()
        assert torch.equal(inv, inv2)
        assert torch.equal(y, ref), f"iteration {it}: chained result differs from the unchained one"


@pytest.mark.parametrize("shape", [(256, 512, 384), (300, 1024, 1000), (64, 2048, 1024)])       # the last one: split-K plan
def test_pdl_chain_gemm_sees_fresh_operands(shape):
    """The tcgen05 GEMM is launched with programmatic dependent launch too: its prologue runs while the predecessor
    drains, and nothing global may be read before griddepcontrol.wait.  Both operands are re-quantised on the device
    (kernels that trigger their dependents early) into the SAME buffers right before every GEMM of a chain, and a GEMM
    follows a GEMM whose output buffer is reused: a stale read or an early write changes a result."""
    import fp8_mps_native
    M, K, N = shape
    g = torch.Generator(device=DEV).manual_seed(11)
    xs = [torch.randn(M, K, device=DEV, generator=g) * (1.0 + i) for i in range(12)]
    ws = [torch.randn(N, K, device=DEV, generator=g) * (0.5 + 0.1 * i) for i in range(12)]
    refs = []
    for x, w in zip(xs, ws):                                      # unchained: a synchronize after every step
        qa, ia = fp8_mps_native.fp8_quantize(x)
        qw, iw = fp8_mps_native.fp8_quantize(w)
        torch.cuda.synchronize()
        refs.append(fp8_mps_native.fp8_scaled_mm_fused(qa, qw, ia, iw, None, None, torch.bfloat16, algo=2).clone())
        torch.cuda.synchronize()
    qa_buf = torch.empty(M, K, dtype=torch.uint8, device=DEV)
    qw_buf = torch.empty(N, K, dtype=torch.uint8, device=DEV)
    out = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
    outs = []
    for x, w in zip(xs, ws):                                      # chained: no host synchronisation at all
        qa, ia = fp8_mps_native.fp8_quantize(x)
        qw, iw = fp8_mps_native.fp8_quantize(w)
        qa_buf.copy_(qa); qw_buf.copy_(qw)
        fp8_mps_native.fp8_scaled_mm_fused(qa_buf, qw_buf, ia, iw, None, None, torch.bfloat16, algo=2, out=out)
        fp8_mps_native.fp8_scaled_mm_fused(qa_buf, qw_buf, ia, iw, None, None, torch.bfloat16, algo=2, out=out)   # GEMM behind a GEMM
        outs.append(out.clone())
    torch.cuda.synchronize()
    for i, (y, ref) in enumerate(zip(outs, refs)):
        assert torch.equal(y, ref), f"step {i}: chained result differs from the unchained one"


@pytest.mark.parametrize("M", [1, 3])
def test_static_weights_option_sees_fresh_activations(M):
    """Same hazard through FP8B_OPT_STATIC_WEIGHTS: only B may be read before the wait."""
    import fp8_mps_native
    K, N = 8192, 96
    W = torch.from_numpy(_rand_fp8((N, K), 7)).to(DEV)
    base = torch.from_numpy(_rand_fp8((M, K), 8)).to(DEV)
    sa = torch.tensor([0.5], device=DEV); sb = torch.tensor([0.02], device=DEV)
    refs = []
    for it in range(24):
        x = torch.roll(base, it, dims=1).contiguous()
        refs.append(fp8_mps_native.fp8_scaled_mm_fused(x, W, sa, sb, None, None, None))
    torch.cuda.synchronize()
    fp8_mps_native.set_static_weights(True)
    try:
        buf = torch.empty_like(base)
        outs = []
        for it in range(24):
            buf.copy_(torch.roll(base, it, dims=1))                          # predecessor writes the activations
            outs.append(fp8_mps_native.fp8_scaled_mm_fused(buf, W, sa, sb, None, None, None))
        torch.cuda.synchronize()
    finally:
        fp8_mps_native.set_static_weights(False)
    for it in range(24):
        assert torch.equal(outs[it], refs[it]), f"iteration {it}"


@pytest.mark.parametrize("M,K,N,xdt,odt", [(64, 1024, 512, torch.bfloat16, torch.bfloat16),
                                           (300, 2048, 384, torch.float16, None),
                                           (17, 4096, 256, torch.float32, torch.float16)])
def test_dynamic_linear_large_m(M, K, N, xdt, odt):
    """M > 16: per-row quantise + tcgen05 GEMM with per-row scale_a, against the oracle composition."""
    import fp8_mps_native
    g = torch.Generator().manual_seed(M + N)
    x = (torch.randn(M, K, generator=g) * (torch.rand(M, 1, generator=g) * 4 + 0.05)).to(xdt)
    W = _rand_fp8((N, K), K + 1)
    sb = (np.random.default_rng(N).random(N).astype(np.float32) + 0.5) * 0.02
    bias = torch.randn(N, generator=g)
    y, inv = fp8_mps_native.fp8_linear_dynamic(x.to(DEV), torch.from_numpy(W).to(DEV), torch.from_numpy(sb), bias.to(DEV), odt)
    qs, invs = zip(*[o.fp8_quantize(x[m].float().numpy()) for m in range(M)])
    inv_ref = np.concatenate(invs)
    assert np.array_equal(inv.cpu().numpy().view(np.uint32), inv_ref.view(np.uint32))
    ref = o.scaled_mm(np.stack(qs), W, inv_ref, sb, to_np(bias), None, dt_name(odt))
    _check(y, ref, odt, what=f"dynamic linear M{M}")
    with pytest.raises(RuntimeError):
        fp8_mps_native.fp8_linear_dynamic(x.to(DEV), torch.from_numpy(W).to(DEV), torch.from_numpy(sb), None, odt, single_kernel=True)


# ------------------------------------------------------------------ float8_e5m2 operands

def _rand_e5m2(shape, seed, special=False):
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 256, shape, dtype=np.uint8)
    e = b & 0x7C
    b[e == 0x7C] = 0x3C                                   # no inf / NaN ...
    b[(b & 0x7F) >= 0x58] = 0x41                          # ... and |v| < 128 so fp32 sums of products stay finite
    if special:
        b.reshape(-1)[5] = 0x7C                           # +inf
        b.reshape(-1)[-3] = 0x7E                          # NaN
    return b


@pytest.mark.parametrize("M,K,N", [(1, 4096, 512), (4, 2048, 300), (16, 1024, 129), (3, 1000, 40),
                                   (256, 1024, 512), (130, 2048, 384), (33, 520, 70)])
@pytest.mark.parametrize("fa,fb", [("e5m2", "e4m3fn"), ("e4m3fn", "e5m2"), ("e5m2", "e5m2")])
def test_e5m2_operands(M, K, N, fa, fb):
    """`_scaled_mm` with float8_e5m2 operands decoded as e5m2 (the reference mis-decodes them as e4m3fn):
    warp-MMA GEMV for M <= 16 (generic kernel when K % 16 != 0), tcgen05 GEMM above (SIMT when not TMA-able)."""
    import fp8_mps_native
    A = _rand_e5m2((M, K), 1 + M) if fa == "e5m2" else _rand_fp8((M, K), 1 + M)
    B = _rand_e5m2((N, K), 2 + N) if fb == "e5m2" else _rand_fp8((N, K), 2 + N)
    sa = np.array([2.0 ** -6], dtype=np.float32)
    sb = (np.random.default_rng(N).random(N).astype(np.float32) + 0.5) * 2.0 ** -6
    bias = torch.randn(N, generator=torch.Generator().manual_seed(K))
    for odt in (None, torch.bfloat16):
        y = fp8_mps_native.fp8_scaled_mm_fused(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(sa),
                                               torch.from_numpy(sb), bias.to(DEV), None, odt, a_format=fa, b_format=fb)
        ref = o.scaled_mm(A, B, sa, sb, to_np(bias), None, dt_name(odt), a_format=fa, b_format=fb)
        _check(y, ref, odt, what=f"e5m2 {fa}x{fb} M{M} K{K} N{N}")


@pytest.mark.parametrize("M,K,N", [(2, 1024, 64), (128, 1024, 256)])
def test_e5m2_inf_nan_propagate_and_e4m3_nan_is_zero(M, K, N):
    """IEEE semantics for e5m2 operands (inf / NaN reach the output), reference semantics for e4m3fn ones
    (0x7F / 0xFF contribute 0) -- in the same product."""
    import fp8_mps_native
    A = _rand_fp8((M, K), 3)
    A[1, 7] = 0x7F                                       # e4m3fn NaN byte -> 0
    B = _rand_e5m2((N, K), 4)
    B[5, 9] = 0x7C                                       # +inf in weight row 5
    B[6, 3] = 0x7E                                       # NaN in weight row 6
    one = np.ones(1, dtype=np.float32)
    y = fp8_mps_native.fp8_scaled_mm_fused(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(one),
                                           torch.from_numpy(one), None, None, None, a_format="e4m3fn", b_format="e5m2")
    got = y.cpu().numpy()
    ref = o.scaled_mm(A, B, one, one, None, None, "f32", a_format="e4m3fn", b_format="e5m2")
    assert np.array_equal(np.isnan(got), np.isnan(ref)) and np.array_equal(np.isinf(got), np.isinf(ref))
    assert np.isnan(got[:, 6]).all() and not np.isfinite(got[:, 5]).any()
    fin = np.isfinite(ref)
    assert o.rel_rmse(got[fin], ref[fin]) < 5e-6


def test_e5m2_through_patched_scaled_mm():
    """torch._scaled_mm with a float8_e5m2 operand after install(): routed with the e5m2 decode."""
    import fp8_mps_patch
    M, K, N = 8, 512, 96
    A = _rand_e5m2((M, K), 9)
    W = _rand_fp8((N, K), 10)
    a = torch.from_numpy(A).to(DEV).view(torch.float8_e5m2)
    w = torch.from_numpy(W).to(DEV).view(torch.float8_e4m3fn)
    sa = torch.tensor([0.25], device=DEV); sb = torch.tensor([0.5], device=DEV)
    fp8_mps_patch.install()
    try:
        y = torch._scaled_mm(a, w.t(), sa, sb, None, None, torch.float32)
    finally:
        fp8_mps_patch.uninstall()
    ref = o.scaled_mm(A, W, np.array([0.25], np.float32), np.array([0.5], np.float32), None, None, "f32", a_format="e5m2")
    _check(y, ref, None, what="patched e5m2")


# ------------------------------------------------------------------ several GEMVs in one launch

@pytest.mark.parametrize("K,Ns,odt,shared_x", [(4096, [4096, 1024, 1024], torch.bfloat16, True),
                                               (14336, [4096, 300], None, False),
                                               (1024, [8, 1, 77, 2048] * 5, torch.float16, False),   # 20 items: two launches
                                               (16, [5], None, True)])
def test_gemv_batch_matches_single_calls_and_oracle(K, Ns, odt, shared_x):
    """fp8_scaled_mm_many == the M = 1 kernel called once per problem (same per-lane accumulation order, so
    bit-identical whenever that call does not split K) and within tolerance of the oracle, incl. a NaN weight byte,
    per-row weight scales and biases."""
    import fp8_mps_native
    g = torch.Generator().manual_seed(K + len(Ns))
    xs, Ws, sxs, sws, bs = [], [], [], [], []
    x0 = _rand_fp8((1, K), 11)
    for i, N in enumerate(Ns):
        x = x0 if shared_x else _rand_fp8((1, K), 20 + i)
        W = _rand_fp8((N, K), 40 + i)
        if i == 1:
            W[0, min(5, K - 1)] = 0x7F                        # NaN byte: contributes 0 (metal:21)
        xs.append(x); Ws.append(W)
        sxs.append(np.array([0.02 + 0.01 * i], dtype=np.float32))
        sws.append(((np.random.default_rng(i).random(N) + 0.5) * 0.01).astype(np.float32) if i % 2 else np.array([0.015], np.float32))
        bs.append(torch.randn(N, generator=g).to(odt or torch.float32) if i % 3 == 0 else None)
    to_dev = lambda a: torch.from_numpy(a).to(DEV)
    ys = fp8_mps_native.fp8_scaled_mm_many([to_dev(x) for x in xs], [to_dev(W) for W in Ws], [to_dev(s) for s in sxs],
                                           [to_dev(s) for s in sws], [None if b is None else b.to(DEV) for b in bs], odt)
    assert len(ys) == len(Ns)
    for i, N in enumerate(Ns):
        assert ys[i].shape == (1, N) and ys[i].dtype == (odt or torch.float32)
        ref = o.scaled_mm(xs[i], Ws[i], sxs[i], sws[i], None if bs[i] is None else to_np(bs[i]), None, dt_name(odt))
        _check(ys[i], ref, odt, what=f"gemv batch item {i} N{N} K{K}")
        single = fp8_mps_native.fp8_scaled_mm_fused(to_dev(xs[i]), to_dev(Ws[i]), to_dev(sxs[i]), to_dev(sws[i]),
                                                    None if bs[i] is None else bs[i].to(DEV), None, odt, algo=1)
        if N >= 2 * 148 * 8 or K < 4096:                      # the single call does not split K here: same summation order
            assert torch.equal(ys[i], single), f"item {i}"
    assert fp8_mps_native.fp8_scaled_mm_many([], [], [], []) == []


def test_gemv_batch_validation():
    from _util import GemvItem, capi, stream_ptr
    L = capi()
    x = torch.zeros(64, dtype=torch.uint8, device=DEV); W = torch.zeros(4, 64, dtype=torch.uint8, device=DEV)
    y = torch.zeros(4, device=DEV); s = torch.ones(1, device=DEV)
    def item(**kw):
        it = (GemvItem * 1)()
        d = dict(x=x.data_ptr(), W=W.data_ptr(), y=y.data_ptr(), N=4, scale_x=s.data_ptr(), scale_w=s.data_ptr(), scale_w_len=1, bias=None)
        d.update(kw)
        for k, v in d.items():
            setattr(it[0], k, v)
        return it
    assert L.fp8b_gemv_batch(item(), 1, 64, 0, 0, stream_ptr()) == 0
    assert L.fp8b_gemv_batch(None, 0, 64, 0, 0, stream_ptr()) == 0
    assert L.fp8b_gemv_batch(None, 1, 64, 0, 0, stream_ptr()) == -1
    assert L.fp8b_gemv_batch(item(scale_w_len=3), 1, 64, 0, 0, stream_ptr()) == -1
    assert L.fp8b_gemv_batch(item(W=None), 1, 64, 0, 0, stream_ptr()) == -1
    assert L.fp8b_gemv_batch(item(), 1, 64, 7, 0, stream_ptr()) == -1
    assert L.fp8b_gemv_batch(item(), 1, 24, 0, 0, stream_ptr()) == -2          # K % 16 != 0
    assert L.fp8b_gemv_batch(item(x=x.data_ptr() + 1), 1, 48, 0, 0, stream_ptr()) == -2   # unaligned x
    assert L.fp8b_gemv_batch(item(N=0), 1, 64, 0, 0, stream_ptr()) == 0
