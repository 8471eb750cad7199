"""GPU parity: the tcgen05 GEMM with the TMA-store ("push") epilogue, fp8b_scaled_mm_push.

On one GPU the 1..8 destinations are all local buffers -- the kernel neither knows nor cares whether a destination
is local HBM or a peer's symmetric buffer (tests/mgpu_sharded.py covers real peers).  Checks, through the C ABI:
bit-equality with the direct-store kernel (same accumulation, same epilogue arithmetic), parity with the oracle
at the tolerances of test_gpu_scaled_mm.py, untouched columns outside the shard block, ragged M / N edges (TMA
clipping), every out dtype, per-row scales + bias + scale_result, and every tile configuration."""
import numpy as np
import pytest
import torch

import fp8_oracle as o
from _util import ALGO_TCGEN05, capi, dt_name, mm_capi, mm_push_capi, to_np

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {"f32": 1e-4, "f16": 5e-4, "bf16": 3e-3}


def _bytes(shape, seed):
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 256, shape, dtype=np.uint8)
    b[(b & 0x7F) == 0x7F] = 0x3C
    return b


def _case(M, K, N, odt, n_dst=1, ldc=None, n0=0, per_row=False, bias_dt=None, scale_result=False, seed=0):
    A, B = _bytes((M, K), seed), _bytes((N, K), seed + 1)
    rng = np.random.default_rng(seed + 2)
    sa = (rng.random(M if per_row else 1).astype(np.float32) + 0.5) * 0.01
    sb = (rng.random(N if per_row else 1).astype(np.float32) + 0.5) * 0.02
    tA, tB = torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV)
    tsa, tsb = torch.from_numpy(sa).to(DEV), torch.from_numpy(sb).to(DEV)
    bias = tbias = None
    if bias_dt is not None:
        tbias = torch.from_numpy(rng.standard_normal(N).astype(np.float32)).to(DEV).to(bias_dt)
        bias = to_np(tbias)
    sr = np.array([0.75], np.float32) if scale_result else None
    tsr = torch.from_numpy(sr).to(DEV) if scale_result else None
    ldc = ldc or N
    dsts = [torch.full((M, ldc), -7.0, dtype=odt, device=DEV) for _ in range(n_dst)]
    rc = mm_push_capi(tA, tB, tsa, tsb, dsts, n0=n0, bias=tbias, sr=tsr)
    assert rc == 0, capi().fp8b_status_string(rc)
    rc, direct = mm_capi(tA, tB, tsa, tsb, tbias, tsr, odt, ALGO_TCGEN05)
    assert rc == 0
    torch.cuda.synchronize()
    ref = o.scaled_mm(A, B, sa, sb, bias, sr, dt_name(odt))
    for d in dsts:
        blk = d[:, n0:n0 + N]
        assert torch.equal(blk, direct), f"push != direct (M{M} K{K} N{N} {dt_name(odt)} n_dst{n_dst})"
        assert o.rel_rmse(to_np(blk), ref) <= TOL[dt_name(odt)]
        if n0 > 0:
            assert bool((d[:, :n0] == -7.0).all()), "columns left of the shard block were touched"
        if n0 + N < ldc:
            assert bool((d[:, n0 + N:] == -7.0).all()), "columns right of the shard block were touched"


@pytest.mark.parametrize("M,K,N,odt,kw", [
    (256, 512, 384, torch.bfloat16, {}),
    (4096, 3072, 1536, torch.bfloat16, dict(n_dst=8, ldc=12288, n0=3072)),      # C4's w=8 shard, eight destinations
    (1024, 1024, 2048, torch.bfloat16, dict(n_dst=2, ldc=4096, n0=2048, per_row=True, bias_dt=torch.bfloat16)),
    (300, 512, 1000, torch.bfloat16, dict(n_dst=3, ldc=2000, n0=1000, per_row=True, bias_dt=torch.float32)),   # ragged M, N
    (129, 144, 136, torch.float16, dict(n_dst=2, per_row=True, bias_dt=torch.float16, scale_result=True)),
    (512, 256, 520, torch.float32, dict(n_dst=2, ldc=1040, n0=520, bias_dt=torch.float32)),                      # fp32: 32-column boxes
    (100, 64, 72, torch.float32, dict(scale_result=True)),
    (128, 128, 8, torch.bfloat16, dict(n_dst=2, ldc=24, n0=8)),                 # one partial box
    (2048, 768, 4096 + 64, torch.bfloat16, dict(n_dst=2)),                      # last-wave split + ragged last tile
])
@pytest.mark.parametrize("store", [4, 3])
def test_push_matches_direct_and_oracle(tune, store, M, K, N, odt, kw):
    """FP8B_OPT_TUNE_GEMM_STORE = 4 / 3 once chose between two push epilogues; either value must still give the one push
    epilogue.  Either also makes the direct kernel of _case store with st.global, not with the TMA-store epilogue the
    push path uses."""
    tune("GEMM_STORE", store)
    _case(M, K, N, odt, seed=M + K + N, **kw)


@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("store", [4, 3])
def test_push_all_tile_configs(tune, cfg, store):
    """Every tile configuration (FP8B_OPT_TUNE_GEMM_CFG), with both former push-epilogue values of GEMM_STORE (see
    test_push_matches_direct_and_oracle)."""
    tune("GEMM_CFG", cfg)
    tune("GEMM_STORE", store)
    _case(640, 512, 1000, torch.bfloat16, n_dst=2, ldc=2000, n0=1000, per_row=True, bias_dt=torch.bfloat16, seed=11)
    _case(300, 256, 328, torch.float32, n_dst=1, seed=12)
    _case(1280, 384, 2560, torch.float16, n_dst=2, seed=13)


@pytest.mark.parametrize("M,K,N,odt", [(4096, 3072, 12288, torch.bfloat16), (1000, 1024, 3000, torch.float16),
                                       (200, 336, 1000, torch.float32)])
def test_plain_scaled_mm_with_tma_store_option(tune, M, K, N, odt):
    """fp8b_scaled_mm itself with FP8B_OPT_TUNE_GEMM_STORE = 2 (TMA-store epilogue) equals the st.global epilogue bit for bit."""
    A, B = _bytes((M, K), 1), _bytes((N, K), 2)
    tA, tB = torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV)
    s = torch.full((1,), 0.01, device=DEV)
    tune("GEMM_STORE", 1)
    rc, c1 = mm_capi(tA, tB, s, s, None, None, odt, ALGO_TCGEN05)
    assert rc == 0
    tune("GEMM_STORE", 2)
    rc, c2 = mm_capi(tA, tB, s, s, None, None, odt, ALGO_TCGEN05)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(c1, c2)


def test_push_nan_bytes_decode_to_zero():
    M, K, N = 256, 256, 192
    A, B = _bytes((M, K), 5), _bytes((N, K), 6)
    A[3, 7] = 0x7F; B[100, 9] = 0xFF; A[200, 0] = 0xFF
    tA, tB = torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV)
    one = torch.ones(1, device=DEV)
    dst = torch.zeros(M, N, dtype=torch.float32, device=DEV)
    assert mm_push_capi(tA, tB, one, one, [dst]) == 0
    torch.cuda.synchronize()
    ref = o.scaled_mm(A, B, np.ones(1, np.float32), np.ones(1, np.float32), None, None, "f32")
    assert np.isfinite(to_np(dst)).all()
    assert o.rel_rmse(to_np(dst), ref) <= 1e-4


def test_push_rejects_unaligned():
    L = capi()
    M, K, N = 128, 64, 36
    tA = torch.zeros(M, K, dtype=torch.uint8, device=DEV)
    tB = torch.zeros(N, K, dtype=torch.uint8, device=DEV)
    one = torch.ones(1, device=DEV)
    dst = torch.zeros(M, 37, dtype=torch.bfloat16, device=DEV)              # row pitch 74 bytes: not TMA-storable
    assert mm_push_capi(tA, tB, one, one, [dst[:, :N]]) == -2               # FP8B_ERR_UNSUPPORTED, never a fallback
    assert L.fp8b_scaled_mm_push_supported(2, M, N, K, 37, None, None, None) == 0
    assert L.fp8b_scaled_mm_push_supported(2, M, N, K, 40, None, None, None) == 0      # 36 columns = 72 bytes: not 16-byte units
    assert L.fp8b_scaled_mm_push_supported(2, M, 32, K, 40, None, None, None) == 1


@pytest.mark.parametrize("store", [4, 3])
def test_push_ragged_column_block(tune, store):
    """A column block whose rows end on a 16-byte boundary but not on a box boundary: the tensor map clips the last box,
    with both former push-epilogue values of GEMM_STORE.  A block that does not end on 16 bytes is refused (TMA stores
    move 16-byte units and would write past column N) -- and plain fp8b_scaled_mm, whose default epilogue is the TMA
    store, falls back to st.global."""
    tune("GEMM_STORE", store)
    _case(300, 256, 328, torch.bfloat16, n_dst=2, ldc=1000, n0=8, per_row=True, seed=3)
    M, K, N = 130, 64, 333
    tA = torch.from_numpy(_bytes((M, K), 1)).to(DEV)
    tB = torch.from_numpy(_bytes((N, K), 2)).to(DEV)
    one = torch.ones(1, device=DEV)
    dst = torch.full((M, 1000), -7.0, dtype=torch.bfloat16, device=DEV)
    assert mm_push_capi(tA, tB, one, one, [dst], n0=8) == -2
    assert capi().fp8b_scaled_mm_push_supported(2, M, N, K, 1000, None, None, None) == 0
    tune("GEMM_STORE", 2)
    rc, c = mm_capi(tA, tB, one, one, None, None, torch.bfloat16, ALGO_TCGEN05, out=dst[:, 8:8 + N])
    assert rc == 0
    torch.cuda.synchronize()
    assert bool((dst[:, :8] == -7.0).all()) and bool((dst[:, 8 + N:] == -7.0).all())
    ref = o.scaled_mm(_bytes((M, K), 1), _bytes((N, K), 2), np.ones(1, np.float32), np.ones(1, np.float32), None, None, "bf16")
    assert o.rel_rmse(to_np(dst[:, 8:8 + N]), ref) <= 3e-3


@pytest.mark.parametrize("M,K,N,odt", [(2304, 256, 2560, torch.bfloat16), (1000, 512, 3000, torch.float16), (300, 128, 520, torch.float32)])
def test_tile_raster_orders_agree(tune, M, K, N, odt):
    """FP8B_OPT_TUNE_GEMM_RASTER: M-fastest, N-fastest and banded (8 M-blocks per band; 2304 rows = one full band + one
    short one) tile orders, incl. the split last wave, give the same bits, with both epilogues."""
    A, B = _bytes((M, K), 21), _bytes((N, K), 22)
    tA, tB = torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV)
    s = torch.full((1,), 0.01, device=DEV)
    outs = []
    for raster in (1, 2, 3):
        for store in (1, 2):
            tune("GEMM_RASTER", raster)
            tune("GEMM_STORE", store)
            rc, c = mm_capi(tA, tB, s, s, None, None, odt, ALGO_TCGEN05)
            assert rc == 0
            outs.append(c)
    torch.cuda.synchronize()
    for c in outs[1:]:
        assert torch.equal(outs[0], c)
    ref = o.scaled_mm(A, B, np.full(1, 0.01, np.float32), np.full(1, 0.01, np.float32), None, None, dt_name(odt))
    assert o.rel_rmse(to_np(outs[0]), ref) <= TOL[dt_name(odt)]


def test_push_signal_and_peer_wait_on_one_gpu():
    """The fused closing barrier through the C ABI, both ends on one GPU: fp8b_scaled_mm_push_signal (two local
    destinations standing in for this rank and a peer) stores the epoch into the "peer's" flag word when its last box
    has landed; fp8b_peer_wait -- launched with PDL, resident while the GEMM runs -- returns only then.  (Safe on one GPU:
    the waiter depends on the GEMM, never the other way round.)  Epochs grow; the CTA counter resets itself."""
    import ctypes
    from _util import dt_code, p, stream_ptr
    L = capi()
    M, K, N = 1024, 512, 1536
    A, B = _bytes((M, K), 31), _bytes((N, K), 32)
    tA, tB = torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV)
    s = torch.full((1,), 0.01, device=DEV)
    flags = torch.zeros(16, dtype=torch.int64, device=DEV)
    counter = torch.zeros(1, dtype=torch.int32, device=DEV)
    rc, direct = mm_capi(tA, tB, s, s, None, None, torch.bfloat16, ALGO_TCGEN05)
    assert rc == 0
    for epoch in (1, 2, 3):
        d0 = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
        d1 = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
        dsts = (ctypes.c_void_p * 2)(d0.data_ptr(), d1.data_ptr())
        sig = (ctypes.c_void_p * 2)(None, flags.data_ptr() + 8 * 1)          # "peer" 1's word on "rank" 0: here, local memory
        rc = L.fp8b_scaled_mm_push_signal(p(tA), p(tB), dsts, 2, dt_code(torch.bfloat16), M, N, K, N, p(s), 1, p(s), 1, None, 0, None,
                                          sig, p(counter), epoch, stream_ptr())
        assert rc == 0, L.fp8b_status_string(rc)
        assert L.fp8b_peer_wait(p(flags), 2, 0, epoch, stream_ptr()) == 0
        after = flags.clone()                                                   # stream-ordered behind the wait kernel
        torch.cuda.synchronize()
        assert int(after[1]) == epoch and int(counter[0]) == 0
        assert torch.equal(d0, direct) and torch.equal(d1, direct)
    assert L.fp8b_peer_wait(None, 2, 0, 1, stream_ptr()) == -1
    assert L.fp8b_peer_wait(p(flags), 9, 0, 1, stream_ptr()) == -1
