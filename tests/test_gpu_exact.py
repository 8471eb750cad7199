"""Bit-exact `_scaled_mm` checks: structured inputs whose exact sum every kernel must reproduce, in guarded buffers.

The parity tests of test_gpu_scaled_mm.py use uniform random bytes and a statistical bound.  At bf16 / fp16 output that
bound is about 0.14 rms per element, several times one product term, so a dropped 16-byte K vector, a lost split-K rank,
a wrong epilogue rounding order or a neighbour's bias can pass it.  Here the inputs are built so that the exact sum of
products fits in fp32 and does not depend on summation order or accumulator width:

  1. one-hot A: each A row has one nonzero byte (any e4m3 code), so every output is one exact product;
  2. one-hot B: the mirror, which checks the A addressing (every row of every tile, CTA-pair halves, ragged M);
  3. few-hot integers: at most 8 nonzeros per A row, |a|, |b| <= 16, so every sum is an integer below 2^11;
  4. dense {-1, 0, 1}: |sum| <= K <= 4096.

The nonzeros sit where the addressing changes: k = 0 and the last 16-byte vector, split-K rank edges, shared-memory
panel edges, the 64-byte k-steps and per-warp ranges of the warp-MMA GEMV, the 128-byte k-blocks of tcgen05.  After
the sum, the epilogue is a fixed chain of separately rounded fp32 operations, (((acc * sa) * sb) + bias) * sr, and an
RNE cast, which fp8_oracle.scaled_mm(accum="f64") restates, so the result must equal the oracle bit for bit.  The
scales are random fp32 values, not powers of two, so the rounding order of the epilogue shows.  The one exception to
"bit for bit" is the sign of an exact zero sum, which depends on the summation order: +0 and -0 compare equal.

Every call writes into an interior view of a sentinel-filled buffer, with rows above and below and columns on both
sides (ldc > N); every sentinel is checked afterwards.  Operands are the leading rows of buffers whose extra rows hold
0x7E (448), and per-row scales and biases are followed by large finite values, so a read past an operand changes the
exact result.  All of it stays inside allocated memory.

Helpers here compute the kernel plans (split ranks, panels, warp ranges) from the same rules as the host code, only to
place the nonzeros; a plan that changes makes these positions less pointed, never the tests wrong."""
import ctypes

import numpy as np
import pytest
import torch

import fp8_oracle as o
from _util import (ALGO_AUTO, ALGO_GEMV, ALGO_SIMT, ALGO_TCGEN05, E4M3, E5M2, SENT, GemvItem, Out, Terms, add_nan_rows, assert_bits_equal,
                   capi, codes, dev_bytes, dev_f32, dt_code, dt_name, edges, few_hot, one_hot, oracle, p, sm_count, small_ints,
                   stream_ptr, tc_bounds, to_np)

pytestmark = pytest.mark.gpu
DEV = "cuda"
OPT_PDL, OPT_STATIC_WEIGHTS = 0, 1
ODTS = (torch.float32, torch.float16, torch.bfloat16)


# ------------------------------------------------------------------ plans (to place the nonzeros)

def fhfma_bounds(M, N, K):
    """split-K rank edges and shared-memory panel edges of the FHFMA GEMV (launch_gemv_fhfma)."""
    out = set()
    for m0 in range(0, M, 4):
        mt = min(4, M - m0)
        S, rb = 1, -(-N // 8)
        while S < 8 and rb * S < 2 * sm_count() and K // (S * 2) >= 2048:
            S *= 2
        kps = (-(-K // S) + 15) & ~15
        while S > 1 and kps * (S - 1) >= K:
            S //= 2
            kps = (-(-K // S) + 15) & ~15
        panel = min(kps, (96 * 1024 // (2 * mt)) & ~15)
        for kb in range(0, K, kps):
            out |= {kb} | set(range(kb + panel, min(K, kb + kps), panel))
    return out


def mma_bounds(K, batch=4):
    """per-warp K ranges, their first 64-byte k-steps and load groups (fp8_gemv_mma_kernel)."""
    kpw = (-(-K // 8) + 63) & ~63
    return {w * kpw + d for w in range(8) for d in (0, 64, 64 * batch)}


# ------------------------------------------------------------------ calls through the C ABI

def run_mm(A, B, odt, algo=ALGO_AUTO, terms=None, rng=None, fmts=None, a_offset=0, aligned=True, expect_rc=0, what="",
           dB=None):
    """One fp8b_scaled_mm (or _fmt when `fmts` is given) call on guarded buffers; checks the status, every sentinel and,
    when it succeeded, the exact result.  dB: B already on the device (dev_bytes(B))."""
    M, K = A.shape
    N = B.shape[0]
    t = (terms or Terms(M, N, rng or np.random.default_rng(M + N + K))).device()
    tA, pA = dev_bytes(A, offset=a_offset)
    tB, pB = dB or dev_bytes(B)
    out = Out(M, N, odt, aligned=aligned)
    L = capi()
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    args = (out.ptr, dt_code(odt), M, N, K, out.ldc, p(t.t_sa), len(t.sa), p(t.t_sb), len(t.sb), p(t.t_bias), bc, p(t.t_sr))
    if fmts is None:
        rc = L.fp8b_scaled_mm(pA, pB, *args, None, 0, algo, stream_ptr())
    else:
        rc = L.fp8b_scaled_mm_fmt(pA, fmts[0], pB, fmts[1], *args, algo, stream_ptr())
    torch.cuda.synchronize()
    what = f"{what} M{M} N{N} K{K} {dt_name(odt)} algo{algo}"
    assert rc == expect_rc, f"{what}: status {rc} ({capi().fp8b_status_string(rc).decode()}), expected {expect_rc}"
    if rc != 0:
        out.check_guard(what, interior_written=False)
        return out
    out.check_guard(what)
    assert_bits_equal(to_np(out.view), oracle(A, B, t.sa, t.sb, t.bias, t.sr, odt, fmts or (E4M3, E4M3)), what)
    return out


def run_family_rows(A_all, B, M, odt, rng, what, **kw):
    """Several calls of M rows each, so that all rows of A_all (more boundary positions than M) are covered."""
    dB = dev_bytes(B)
    for i, r0 in enumerate(range(0, A_all.shape[0], M)):
        A = A_all[r0:r0 + M]
        if A.shape[0] < M:
            A = np.concatenate([A, A_all[:M - A.shape[0]]])
        run_mm(A, B, odt, terms=Terms.cycle(i, M, B.shape[0], rng), what=f"{what} call {i}", dB=dB, **kw)


@pytest.fixture
def option():
    """option(OPT_PDL, 0): fp8b_set_option for this test, restored afterwards."""
    L = capi()
    saved = {}

    def setter(opt, value):
        saved.setdefault(opt, L.fp8b_get_option(opt))
        assert L.fp8b_set_option(opt, value) == 0

    yield setter
    for opt, value in saved.items():
        L.fp8b_set_option(opt, value)


# ------------------------------------------------------------------ GEMV, FHFMA kernel

GEMV_SHAPES = {"split": (8192, 40), "panels": (100000, 24), "wide": (4096, 1200)}     # (K, N)


@pytest.mark.parametrize("shape", sorted(GEMV_SHAPES))
@pytest.mark.parametrize("M", [1, 3, 4, 5, 16])
def test_gemv_fhfma_exact(tune, M, shape):
    """GEMV_IMPL = 1 at M in {1, 3, 4, 5, 16} (one to four passes of <= 4 rows): cluster split-K (small N, long K), panel
    loop inside the split ranks (K = 100000, 4-row passes), no split (wide N).  Families 1 and 3."""
    tune("GEMV_IMPL", 1)
    K, N = GEMV_SHAPES[shape]
    rng = np.random.default_rng(M * 1000 + K)
    pos = edges(K, fhfma_bounds(M, N, K), rng)
    A1 = one_hot(max(len(pos), M), K, pos, rng)
    B = codes((N, K), rng)
    if shape != "wide":
        B = add_nan_rows(B, A1, [1, N - 1], rng)
    odt = ODTS[M % 3]
    run_family_rows(A1, B, M, odt, rng, f"one-hot A {shape}")
    run_family_rows(few_hot(M, K, pos, rng), small_ints((N, K), rng), M, ODTS[(M + 1) % 3], rng, f"few-hot {shape}")


@pytest.mark.parametrize("unroll", [2, 4, 8])
def test_gemv_fhfma_unroll_exact(tune, unroll):
    """GEMV_UNROLL 2 / 4 / 8 (fp8_gemv_kernel<1, U>) at M = 1: split-K, and the panel loop without a split (K > 49152
    with N large enough that K is not split)."""
    tune("GEMV_IMPL", 1)
    tune("GEMV_UNROLL", unroll)
    for K, N in ((8192, 40), (50000, 2400)):
        rng = np.random.default_rng(unroll + K)
        pos = edges(K, fhfma_bounds(1, N, K), rng)
        B = codes((N, K), rng)
        run_family_rows(one_hot(len(pos), K, pos, rng), B, 1, torch.float32, rng, f"unroll {unroll} one-hot A")
        run_mm(few_hot(1, K, pos, rng), small_ints((N, K), rng), torch.bfloat16, rng=rng, what=f"unroll {unroll} few-hot")


@pytest.mark.parametrize("impl", [1, 2])
def test_gemv_dense_small_integers(tune, impl):
    """Family 4 through both GEMV kernels, M = 1 and 16, K up to 4096."""
    tune("GEMV_IMPL", impl)
    for M, K, N in ((1, 4096, 300), (16, 4096, 77), (5, 1024, 40)):
        rng = np.random.default_rng(impl * 10 + M)
        A, B = small_ints((M, K), rng, -1, 1), small_ints((N, K), rng, -1, 1)
        for i, odt in enumerate(ODTS):
            run_mm(A, B, odt, ALGO_GEMV, terms=Terms.cycle(i + M, M, N, rng), what=f"dense impl {impl}")


# ------------------------------------------------------------------ GEMV, warp-MMA kernel

@pytest.mark.parametrize("M,batch,static,pdl", [
    (1, 1, 0, 1), (1, 2, 1, 1), (1, 4, 0, 0), (4, 4, 1, 0),          # NB = 1 (M <= 8), GEMV_BATCH 1 / 2 / 4
    (8, 2, 0, 1), (8, 1, 1, 1),
    (9, 4, 1, 1), (16, 4, 0, 0), (13, 4, 1, 0),                      # NB = 2 (M = 9..16)
])
def test_gemv_mma_exact(tune, option, M, batch, static, pdl):
    """GEMV_IMPL = 2 with GEMV_BATCH, STATIC_WEIGHTS and PDL sampled: families 1, 2 and 3 on a shape with a ragged last
    16-row weight block and a K whose warp ranges do not divide evenly."""
    tune("GEMV_IMPL", 2)
    tune("GEMV_BATCH", batch)
    option(OPT_STATIC_WEIGHTS, static)
    option(OPT_PDL, pdl)
    K, N = 5008, 333
    rng = np.random.default_rng(M * 31 + batch)
    pos = edges(K, mma_bounds(K, batch), rng)
    A1 = one_hot(len(pos), K, pos, rng)
    B = add_nan_rows(codes((N, K), rng), A1, [0, N - 2], rng)
    run_family_rows(A1, B, M, ODTS[M % 3], rng, "mma one-hot A")
    run_mm(codes((M, K), rng), one_hot(N, K, pos, rng), ODTS[(M + 1) % 3], ALGO_GEMV, rng=rng, what="mma one-hot B")
    run_mm(few_hot(M, K, pos, rng), small_ints((N, K), rng), ODTS[(M + 2) % 3], ALGO_GEMV, rng=rng, what="mma few-hot")


# ------------------------------------------------------------------ generic kernel and SIMT GEMM

@pytest.mark.parametrize("algo", [ALGO_AUTO, ALGO_GEMV])
@pytest.mark.parametrize("why", ["ragged_k", "misaligned_a"])
def test_generic_kernel_exact(algo, why):
    """fp8_gemv_generic_kernel: K % 16 != 0, or A one byte off 16-byte alignment; through AUTO and forced GEMV."""
    K = 1037 if why == "ragged_k" else 1024
    off = 1 if why == "misaligned_a" else 0
    rng = np.random.default_rng(K + algo)
    pos = edges(K, range(32, K, 32), rng)
    for M in (1, 7, 16):
        A1 = one_hot(len(pos), K, pos, rng)
        B = add_nan_rows(codes((70, K), rng), A1, [3], rng)
        run_family_rows(A1, B, M, ODTS[M % 3], rng, f"generic {why} one-hot A", algo=algo, a_offset=off, aligned=False)
        run_mm(codes((M, K), rng), one_hot(70, K, pos, rng), torch.float32, algo, rng=rng, a_offset=off, what=f"generic {why} one-hot B")
        run_mm(small_ints((M, K), rng, -1, 1), small_ints((70, K), rng, -1, 1), torch.bfloat16, algo, rng=rng, a_offset=off,
               what=f"generic {why} dense")


@pytest.mark.parametrize("algo", [ALGO_SIMT, ALGO_AUTO])
def test_simt_exact(algo):
    """fp8_gemm_simt_kernel, forced and through AUTO (M > 16 with K % 16 != 0): ragged 64 x 64 tiles and 32-wide K panels."""
    M, K, N = 133, 1000 if algo == ALGO_AUTO else 1024, 197
    rng = np.random.default_rng(M + K + algo)
    pos = edges(K, range(32, K, 32), rng)
    A1 = one_hot(M, K, pos, rng)
    run_mm(A1, add_nan_rows(codes((N, K), rng), A1, [5], rng), torch.float32, algo, terms=Terms.cycle(7, M, N, rng), what="simt one-hot A")
    run_mm(codes((M, K), rng), one_hot(N, K, pos, rng), torch.bfloat16, algo, terms=Terms.cycle(3, M, N, rng), what="simt one-hot B")
    run_mm(few_hot(M, K, pos, rng), small_ints((N, K), rng), torch.float16, algo, terms=Terms.cycle(5, M, N, rng), what="simt few-hot")
    run_mm(small_ints((M, K), rng, -1, 1), small_ints((N, K), rng, -1, 1), torch.float32, algo, aligned=False,
           terms=Terms.cycle(2, M, N, rng), what="simt dense")


# ------------------------------------------------------------------ tcgen05 GEMM

def _tc_families(M, K, N, rng, what, nan=True, odts=ODTS, **kw):
    pos = edges(K, tc_bounds(K), rng)
    A1 = one_hot(M, K, pos, rng)
    B = codes((N, K), rng)
    if nan:
        B = add_nan_rows(B, A1, [2, N - 1], rng)
    run_mm(A1, B, odts[0], ALGO_TCGEN05, terms=Terms.cycle(1, M, N, rng), what=f"{what} one-hot A", **kw)
    run_mm(codes((M, K), rng), one_hot(N, K, pos, rng), odts[1 % len(odts)], ALGO_TCGEN05, terms=Terms.cycle(6, M, N, rng),
           what=f"{what} one-hot B", **kw)
    run_mm(few_hot(M, K, pos, rng), small_ints((N, K), rng), odts[2 % len(odts)], ALGO_TCGEN05, terms=Terms.cycle(11, M, N, rng),
           what=f"{what} few-hot", **kw)


@pytest.mark.parametrize("store", [1, 2])
@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
def test_tcgen05_tile_configs_exact(tune, cfg, store):
    """GEMM_CFG 1-5 x GEMM_STORE 1 (st.global) / 2 (TMA store) on ragged M, N and a K tail: every row of both CTAs of a
    pair, the last partial tile in both directions, the last partial k-block."""
    tune("GEMM_CFG", cfg)
    tune("GEMM_STORE", store)
    rng = np.random.default_rng(cfg * 10 + store)
    _tc_families(300, 400, 1000, rng, f"cfg {cfg} store {store}")
    if store == 1:                     # unaligned C: the scalar edge path of the st.global epilogue
        _tc_families(137, 144, 203, rng, f"cfg {cfg} unaligned C", aligned=False, odts=(torch.bfloat16, torch.float32))


@pytest.mark.parametrize("split", [2, 4, -1])
def test_tcgen05_split_k_exact(tune, split):
    """GEMM_SPLITK 2 / 4 and the automatic plan (-1), 32 x 3072 x 3072 (24 tiles: the shape split-K exists for) and a
    ragged one; one-hot B covers every 128-byte k-block boundary, so a lost or doubled rank shows."""
    tune("GEMM_SPLITK", split)
    rng = np.random.default_rng(split + 5)
    for M, K, N in ((32, 3072, 3072), (77, 2064, 400)):
        _tc_families(M, K, N, rng, f"split {split}", nan=(N < 1000))


@pytest.mark.parametrize("raster", [1, 2, 3])
def test_tcgen05_raster_exact(tune, raster):
    tune("GEMM_RASTER", raster)
    tune("GEMM_CFG", 4)
    _tc_families(1100, 256, 700, np.random.default_rng(raster), f"raster {raster}", nan=False)


def test_tcgen05_dense_small_integers(tune):
    """Family 4 on tcgen05 (kind::f8f6f4), one CTA and CTA-pair tiles and split-K: integer sums up to 2^12 in magnitude
    come out exact, so the accumulation holds at least this range (see test_tcgen05_accumulation_precision)."""
    rng = np.random.default_rng(44)
    for cfg, M, K, N in ((2, 200, 4096, 300), (3, 300, 4096, 520)):
        tune("GEMM_CFG", cfg)
        A, B = small_ints((M, K), rng, -1, 1), small_ints((N, K), rng, -1, 1)
        A[0], B[0] = 0x38, 0x38                                   # one output at exactly K = 4096
        run_mm(A, B, torch.float32, ALGO_TCGEN05, terms=Terms.cycle(0, M, N, rng), what=f"dense cfg {cfg}")
    tune("GEMM_CFG", -1)
    tune("GEMM_SPLITK", 4)
    A, B = small_ints((32, 4096), rng, -1, 1), small_ints((256, 4096), rng, -1, 1)
    run_mm(A, B, torch.bfloat16, ALGO_TCGEN05, terms=Terms.cycle(5, 32, 256, rng), what="dense split 4")


# ------------------------------------------------------------------ push epilogue

@pytest.mark.parametrize("n_dst,n0", [(1, 0), (2, 24), (3, 1000)])
def test_push_exact(n_dst, n0):
    """fp8b_scaled_mm_push into 1-3 local destinations, at column offset n0 of each (M, ldc) matrix: each destination
    equals the exact result, nothing outside the block changes."""
    M, K, N = 300, 400, 1000
    rng = np.random.default_rng(n_dst)
    pos = edges(K, tc_bounds(K), rng)
    L = capi()
    for fam, odt in (("one-hot A", torch.bfloat16), ("one-hot B", torch.float32), ("few-hot", torch.float16)):
        if fam == "one-hot A":
            A, B = one_hot(M, K, pos, rng), codes((N, K), rng)
        elif fam == "one-hot B":
            A, B = codes((M, K), rng), one_hot(N, K, pos, rng)
        else:
            A, B = few_hot(M, K, pos, rng), small_ints((N, K), rng)
        t = Terms.cycle(n_dst + len(fam), M, N, rng).device()
        tA, pA = dev_bytes(A)
        tB, pB = dev_bytes(B)
        outs = [Out(M, N, odt, cl=8 + n0) for _ in range(n_dst)]
        ptrs = (ctypes.c_void_p * n_dst)(*[d.ptr for d in outs])
        bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
        rc = L.fp8b_scaled_mm_push(pA, pB, ptrs, n_dst, dt_code(odt), M, N, K, outs[0].ldc, p(t.t_sa), len(t.sa), p(t.t_sb),
                                   len(t.sb), p(t.t_bias), bc, p(t.t_sr), stream_ptr())
        torch.cuda.synchronize()
        assert rc == 0, capi().fp8b_status_string(rc)
        ref = oracle(A, B, t.sa, t.sb, t.bias, t.sr, odt)
        for d, out in enumerate(outs):
            what = f"push {fam} n_dst {n_dst} n0 {n0} destination {d}"
            out.check_guard(what)
            assert_bits_equal(to_np(out.view), ref, what)


# ------------------------------------------------------------------ e5m2 operands

@pytest.mark.parametrize("fmts", [(E5M2, E4M3), (E4M3, E5M2), (E5M2, E5M2)])
@pytest.mark.parametrize("M,K,N", [(3, 2048, 100), (12, 1040, 64), (150, 512, 264), (5, 100, 33)])
def test_fmt_e5m2_exact(fmts, M, K, N):
    """fp8b_scaled_mm_fmt: warp-MMA GEMV (M <= 16), tcgen05 (M > 16), generic kernel (K % 16 != 0).  Families 1 and 2
    only: one-hot products of e5m2 and e4m3 codes are exact in fp32."""
    rng = np.random.default_rng(M + K + 7 * fmts[0] + 3 * fmts[1])
    bounds = tc_bounds(K) | mma_bounds(K) if K % 16 == 0 else set(range(32, K, 32))
    pos = edges(K, bounds, rng)
    fa, fb = fmts
    A1 = one_hot(max(M, len(pos)), K, pos, rng, fa)
    for i, r0 in enumerate(range(0, A1.shape[0], M)):
        A = A1[r0:r0 + M] if r0 + M <= A1.shape[0] else A1[-M:]
        run_mm(A, codes((N, K), rng, fb), ODTS[i % 3], terms=Terms.cycle(i, M, N, rng), fmts=fmts, what=f"fmt {fmts} one-hot A")
        if M > 16:
            break
    run_mm(codes((M, K), rng, fa), one_hot(N, K, pos, rng, fb), torch.float32, terms=Terms.cycle(3, M, N, rng), fmts=fmts,
           what=f"fmt {fmts} one-hot B")


# ------------------------------------------------------------------ batched GEMV

def test_gemv_batch_exact():
    """fp8b_gemv_batch: 22 items, 18 of them nonempty (two launches) including N = 0 items, per-row and per-tensor weight scales, biases; each
    y_i in its own guarded buffer."""
    K = 3072
    rng = np.random.default_rng(3)
    pos = edges(K, {1024, 2048}, rng)
    L = capi()
    for odt, bias_dt in ((torch.float32, torch.bfloat16), (torch.bfloat16, torch.float32), (torch.float16, torch.float16)):
        Ns = [40, 0, 1, 77, 8, 0, 300, 5, 16, 0, 9, 64, 3, 1, 200, 33, 0, 48, 2, 17, 100, 7]
        items = (GemvItem * len(Ns))()
        keep, checks = [], []
        for i, N in enumerate(Ns):
            if N == 0:
                items[i].N = 0
                continue
            if i % 3 == 0:
                x, W = codes((1, K), rng), one_hot(N, K, pos, rng)
            elif i % 3 == 1:
                x, W = one_hot(1, K, pos[i % len(pos):], rng), codes((N, K), rng)
            else:
                x, W = few_hot(1, K, pos, rng), small_ints((N, K), rng)
            t = Terms(1, N, rng, per_row_b=bool(i % 2), bias_dt=bias_dt if i % 4 else None).device()
            tx, px = dev_bytes(x)
            tW, pW = dev_bytes(W)
            y = Out(1, N, odt)
            items[i].x, items[i].W, items[i].y, items[i].N = px, pW, y.ptr, N
            items[i].scale_x, items[i].scale_w, items[i].scale_w_len = t.t_sa.data_ptr(), t.t_sb.data_ptr(), len(t.sb)
            items[i].bias = t.t_bias.data_ptr() if t.t_bias is not None else None
            keep += [tx, tW, t]
            checks.append((i, x, W, t, y))
        n0 = L.fp8b_launch_count()
        rc = L.fp8b_gemv_batch(items, len(Ns), K, dt_code(odt), dt_code(bias_dt), stream_ptr())
        torch.cuda.synchronize()
        assert rc == 0 and L.fp8b_launch_count() == n0 + 2
        for i, x, W, t, y in checks:
            what = f"gemv batch item {i} {dt_name(odt)}"
            y.check_guard(what)
            assert_bits_equal(to_np(y.view), oracle(x, W, t.sa, t.sb, t.bias, None, odt), what)


# ------------------------------------------------------------------ dynamic linear

@pytest.mark.parametrize("M,plan,ws", [(1, -1, True), (3, 1, True), (4, 2, True), (16, -1, False), (5, 1, False),
                                       (40, -1, True), (300, 2, True)])
@pytest.mark.parametrize("xdt", [torch.float32, torch.bfloat16, torch.float16])
def test_linear_dynamic_exact(tune, M, plan, ws, xdt):
    """fp8b_linear_dynamic with one-hot X rows: each row quantises to +-448 at one position, so the quantised bytes, the
    row scales (448 / amax in double) and the result are all exact.  DYNAMIC_PLAN 1 (single kernel) / 2 (quantise +
    chained GEMV) / built-in, with and without a workspace, M <= 16 and M > 16 (quantise + tcgen05 with per-row
    scale_a).  inv_scale_a_out is checked bit for bit, in a guarded buffer too."""
    tune("DYNAMIC_PLAN", plan)
    K, N = 4096, 264
    rng = np.random.default_rng(M * 3 + plan)
    pos = edges(K, fhfma_bounds(min(M, 16), N, K) | mma_bounds(K) | tc_bounds(K), rng)
    X = np.zeros((M, K), np.float32)
    X[np.arange(M), pos[np.arange(M) % len(pos)]] = (rng.standard_normal(M) * np.exp2(rng.integers(-6, 6, M))).astype(np.float32)
    Xt = torch.from_numpy(X).to(xdt)
    Xf = Xt.float().numpy()
    guard = torch.full((2, K), 1.0e4, dtype=xdt)
    tX = torch.cat([Xt, guard]).to(DEV)
    B = add_nan_rows(codes((N, K), rng), np.zeros((1, K), np.uint8), [7], rng)
    tB, pB = dev_bytes(B)
    odt = ODTS[(M + plan) % 3]
    t = Terms.cycle(M + plan, 1, N, rng).device()
    out = Out(M, N, odt)
    inv = torch.full((M + 8,), SENT[torch.float32], dtype=torch.int32, device=DEV).view(torch.float32)
    L = capi()
    need = L.fp8b_linear_dynamic_workspace_bytes(M, K)
    wsb = torch.empty(need + 16, dtype=torch.uint8, device=DEV) if ws else None
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    rc = L.fp8b_linear_dynamic(tX.data_ptr(), dt_code(xdt), pB, out.ptr, dt_code(odt), M, N, K, out.ldc, p(t.t_sb), len(t.sb),
                               p(t.t_bias), bc, p(t.t_sr), inv.data_ptr(), p(wsb), need if ws else 0, stream_ptr())
    torch.cuda.synchronize()
    what = f"linear_dynamic M{M} plan {plan} ws {ws} {dt_name(xdt)} -> {dt_name(odt)}"
    assert rc == 0, f"{what}: {capi().fp8b_status_string(rc).decode()}"
    qs, invs = zip(*[o.fp8_quantize(Xf[m]) for m in range(M)])
    q, inv_ref = np.stack(qs), np.concatenate(invs)
    assert set(np.unique(q).tolist()) <= {0x00, 0x7E, 0xFE}
    assert np.array_equal(inv[:M].cpu().numpy().view(np.uint32), inv_ref.view(np.uint32)), what
    assert (inv[M:].view(torch.int32) == SENT[torch.float32]).all(), f"{what}: written past inv_scale_a_out[M]"
    out.check_guard(what)
    assert_bits_equal(to_np(out.view), oracle(q, B, inv_ref, t.sb, t.bias, t.sr, odt), what)


# ------------------------------------------------------------------ degenerate extents

def _zero_k_expect(M, N, t, odt):
    return oracle(np.zeros((M, 0), np.uint8), np.zeros((N, 0), np.uint8), t.sa, t.sb, t.bias, t.sr, odt)


@pytest.mark.parametrize("M", [1, 16, 40])
def test_zero_k(M):
    """K = 0: the sum is 0, so C = cast(((0 * sa) * sb + bias) * sr) on every entry point that serves it (AUTO, GEMV,
    SIMT, _fmt, fp8b_linear_dynamic with a workspace); forced TCGEN05, fp8b_gemv_batch and the single-kernel dynamic
    plan refuse with FP8B_ERR_UNSUPPORTED and leave C untouched (include/fp8_b200.h)."""
    N = 50
    rng = np.random.default_rng(M)
    A, B = np.zeros((M, 0), np.uint8), np.zeros((N, 0), np.uint8)
    L = capi()
    for i, algo in enumerate((ALGO_AUTO, ALGO_GEMV, ALGO_SIMT, ALGO_TCGEN05)):
        refused = algo == ALGO_TCGEN05 or (algo == ALGO_GEMV and M > 16)
        n0 = L.fp8b_launch_count()
        run_mm(A, B, ODTS[i % 3], algo, terms=Terms.cycle(4 + i, M, N, rng), expect_rc=-2 if refused else 0, what="K = 0")
        assert (L.fp8b_launch_count() == n0) == refused
    run_mm(A, B, torch.bfloat16, terms=Terms.cycle(6, M, N, rng), fmts=(E5M2, E4M3), what="K = 0 fmt")
    # dynamic linear: the workspace plan serves K = 0 (amax 0 -> scale 1), the single-kernel plan refuses
    t = Terms.cycle(5, 1, N, rng).device()
    X = torch.zeros(M + 1, 16, dtype=torch.bfloat16, device=DEV)
    tB, pB = dev_bytes(np.zeros((N, 16), np.uint8))
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    for ws in (True, False):
        out = Out(M, N, torch.float32)
        inv = torch.full((M + 8,), SENT[torch.float32], dtype=torch.int32, device=DEV).view(torch.float32)
        wsb = torch.empty(64, dtype=torch.uint8, device=DEV)
        rc = L.fp8b_linear_dynamic(X.data_ptr(), dt_code(torch.bfloat16), pB, out.ptr, 0, M, N, 0, out.ldc, p(t.t_sb), len(t.sb),
                                   p(t.t_bias), bc, p(t.t_sr), inv.data_ptr(), p(wsb) if ws else None, 64 if ws else 0, stream_ptr())
        torch.cuda.synchronize()
        if ws:
            assert rc == 0
            out.check_guard("dynamic K = 0")
            assert (inv[:M] == 1.0).all() and (inv[M:].view(torch.int32) == SENT[torch.float32]).all()
            assert_bits_equal(to_np(out.view), _zero_k_expect(M, N, Terms_with(t, np.ones(M, np.float32)), torch.float32), "dynamic K = 0")
        else:
            assert rc == -2
            out.check_guard("dynamic K = 0 refused", interior_written=False)
    # batched GEMV: K >= 16 is required
    y = Out(1, N, torch.float32)
    s = dev_f32([1.0])
    items = (GemvItem * 1)()
    items[0].x, items[0].W, items[0].y, items[0].N = pB, pB, y.ptr, N
    items[0].scale_x, items[0].scale_w, items[0].scale_w_len = s.data_ptr(), s.data_ptr(), 1
    assert L.fp8b_gemv_batch(items, 1, 0, 0, 0, stream_ptr()) == -2
    torch.cuda.synchronize()
    y.check_guard("gemv batch K = 0", interior_written=False)


def Terms_with(t, sa):
    """the same epilogue terms with another scale_a."""
    c = Terms.__new__(Terms)
    c.__dict__.update(t.__dict__)
    c.sa = sa
    return c


def test_empty_m_or_n_launches_nothing():
    """M = 0 or N = 0: status 0, no launch, nothing written, on every entry point."""
    L = capi()
    K = 64
    one = dev_f32([1.0])
    tA, pA = dev_bytes(np.zeros((4, K), np.uint8))
    out = Out(4, 8, torch.float32)
    n0 = L.fp8b_launch_count()
    for M, N in ((0, 8), (4, 0), (0, 0)):
        for algo in (ALGO_AUTO, ALGO_GEMV, ALGO_TCGEN05, ALGO_SIMT):
            assert L.fp8b_scaled_mm(pA, pA, out.ptr, 0, M, N, K, 8, one.data_ptr(), 1, one.data_ptr(), 1, None, 0, None, None, 0,
                                    algo, stream_ptr()) == 0
        assert L.fp8b_scaled_mm_fmt(pA, E5M2, pA, E4M3, out.ptr, 0, M, N, K, 8, one.data_ptr(), 1, one.data_ptr(), 1, None, 0,
                                    None, 0, stream_ptr()) == 0
        ptrs = (ctypes.c_void_p * 1)(out.ptr)
        assert L.fp8b_scaled_mm_push(pA, pA, ptrs, 1, 0, M, N, K, 8, one.data_ptr(), 1, one.data_ptr(), 1, None, 0, None,
                                     stream_ptr()) == 0
        X = torch.zeros(4, K, device=DEV)
        assert L.fp8b_linear_dynamic(X.data_ptr(), 0, pA, out.ptr, 0, M, N, K, 8, one.data_ptr(), 1, None, 0, None, None,
                                     None, 0, stream_ptr()) == 0
    items = (GemvItem * 2)()
    for it in items:
        it.N = 0
    assert L.fp8b_gemv_batch(items, 2, K, 0, 0, stream_ptr()) == 0
    torch.cuda.synchronize()
    assert L.fp8b_launch_count() == n0
    out.check_guard("empty problems", interior_written=False)


@pytest.mark.parametrize("algo", [ALGO_AUTO, ALGO_GEMV, ALGO_TCGEN05, ALGO_SIMT])
def test_unit_sizes(tune, algo):
    """M = N = 1 at K = 16 (the smallest aligned problem) on every algorithm and both GEMV kernels, and through _fmt."""
    rng = np.random.default_rng(algo)
    for impl in ((1, 2) if algo == ALGO_GEMV else (-1,)):
        tune("GEMV_IMPL", impl)
        for k in (0, 15):
            A = one_hot(1, 16, np.array([k]), rng)
            for i, odt in enumerate(ODTS):
                run_mm(A, codes((1, 16), rng), odt, algo, terms=Terms.cycle(i + k, 1, 1, rng), what=f"unit impl {impl}")
    run_mm(one_hot(1, 16, np.array([7]), rng, E5M2), codes((1, 16), rng), torch.float32, algo if algo != ALGO_GEMV else ALGO_AUTO,
           rng=rng, fmts=(E5M2, E4M3), what="unit fmt")


@pytest.mark.parametrize("ws", [True, False])
def test_unit_sizes_dynamic_and_batch(ws):
    """M = N = 1 at K = 16 through fp8b_linear_dynamic (both plans) and fp8b_gemv_batch."""
    rng = np.random.default_rng(17)
    L = capi()
    B = codes((1, 16), rng)
    tB, pB = dev_bytes(B)
    t = Terms.cycle(6, 1, 1, rng).device()
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    X = torch.zeros(3, 16)
    X[0, 9] = -0.3
    tX = X.to(DEV)
    out = Out(1, 1, torch.float32)
    inv = torch.full((9,), SENT[torch.float32], dtype=torch.int32, device=DEV).view(torch.float32)
    wsb = torch.empty(64, dtype=torch.uint8, device=DEV) if ws else None
    rc = L.fp8b_linear_dynamic(tX.data_ptr(), 0, pB, out.ptr, 0, 1, 1, 16, out.ldc, p(t.t_sb), 1, p(t.t_bias), bc, p(t.t_sr),
                               inv.data_ptr(), p(wsb), 64 if ws else 0, stream_ptr())
    torch.cuda.synchronize()
    assert rc == 0
    q, inv_ref = o.fp8_quantize(X[0].numpy())
    assert inv[0].item() == inv_ref[0] and (inv[1:].view(torch.int32) == SENT[torch.float32]).all()
    out.check_guard("dynamic unit")
    assert_bits_equal(to_np(out.view), oracle(q[None], B, inv_ref, t.sb, t.bias, t.sr, torch.float32), "dynamic unit")
    x = one_hot(1, 16, np.array([15 if ws else 0]), rng)
    tx, px = dev_bytes(x)
    y = Out(1, 1, torch.bfloat16)
    items = (GemvItem * 1)()
    items[0].x, items[0].W, items[0].y, items[0].N = px, pB, y.ptr, 1
    items[0].scale_x, items[0].scale_w, items[0].scale_w_len = t.t_sa.data_ptr(), t.t_sb.data_ptr(), 1
    items[0].bias = p(t.t_bias)
    assert L.fp8b_gemv_batch(items, 1, 16, dt_code(torch.bfloat16), bc, stream_ptr()) == 0
    torch.cuda.synchronize()
    y.check_guard("batch unit")
    assert_bits_equal(to_np(y.view), oracle(x, B, t.sa, t.sb, t.bias, None, torch.bfloat16), "batch unit")


# ------------------------------------------------------------------ large indices

def _need_free(nbytes):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")


def _rand_dev_bytes(shape, seed):
    """uniform non-NaN e4m3 bytes generated on the device."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    t = torch.randint(0, 256, shape, dtype=torch.uint8, device=DEV, generator=g)
    t[(t & 0x7F) == 0x7F] = 0x3C
    return t


@pytest.mark.parametrize("store", [1, 2])
def test_tcgen05_output_past_2_31_elements(tune, store):
    """M * ldc > 2^31 output elements (40000 x 65536 bf16, 5.2 GB), one-hot A, both epilogues.  The reference is the same
    fp32 multiplies and an RNE cast in torch, in row chunks; it is first checked against fp8_oracle on a slice."""
    M, K, N = 40000, 128, 65536
    ldc = N + 64
    _need_free(M * ldc * 2 + 8 * 2**30)
    tune("GEMM_STORE", store)
    rng = np.random.default_rng(store)
    ks = rng.integers(0, K, M)
    ks[-8:] = [0, 15, 16, 63, 64, 112, 127, 127]
    vals = codes(M, rng)
    A = np.zeros((M, K), np.uint8)
    A[np.arange(M), ks] = vals
    tA = torch.from_numpy(A).to(DEV)
    tB = _rand_dev_bytes((N, K), 11)
    sa, sb = np.float32(0.0123 * 1.37), np.float32(0.0217 * 0.91)
    tsa, tsb = dev_f32([sa]), dev_f32([sb])
    bias = torch.from_numpy((rng.standard_normal(N) * 0.7).astype(np.float32)).to(DEV)
    C = torch.full((M + 2, ldc), SENT[torch.bfloat16], dtype=torch.int16, device=DEV).view(torch.bfloat16)
    view = C[1:M + 1, 32:32 + N]
    L = capi()
    rc = L.fp8b_scaled_mm(tA.data_ptr(), tB.data_ptr(), view.data_ptr(), dt_code(torch.bfloat16), M, N, K, ldc, tsa.data_ptr(), 1,
                          tsb.data_ptr(), 1, bias.data_ptr(), 0, None, None, 0, ALGO_TCGEN05, stream_ptr())
    assert rc == 0
    torch.cuda.synchronize()
    dec = torch.from_numpy(o.DECODE_TABLE).to(DEV)
    a_val = dec[torch.from_numpy(vals.astype(np.int64)).to(DEV)]
    k_dev = torch.from_numpy(ks).to(DEV)

    def ref_rows(r0, r1):
        bcols = dec[tB[:, k_dev[r0:r1]].long()].T                 # (rows, N): dec(B[n, k_m])
        return ((((a_val[r0:r1, None] * bcols) * sa) * sb) + bias).to(torch.bfloat16)

    # the torch reference against the oracle on a slice
    sl = slice(M - 8, M)
    ref_np = o.scaled_mm(A[sl], tB[:4096].cpu().numpy(), [sa], [sb], bias[:4096].cpu().numpy(), None, "bf16")
    assert_bits_equal(to_np(ref_rows(M - 8, M)[:, :4096]), ref_np, "torch reference vs oracle")
    raw = C.view(torch.int16)
    assert (raw[0] == SENT[torch.bfloat16]).all() and (raw[M + 1] == SENT[torch.bfloat16]).all(), "rows above / below C written"
    step = 2048
    for r0 in range(0, M, step):
        r1 = min(M, r0 + step)
        got = view[r0:r1]
        if not torch.equal(got.view(torch.int16), ref_rows(r0, r1).view(torch.int16)):
            bad = (got.view(torch.int16) != ref_rows(r0, r1).view(torch.int16)).nonzero()
            raise AssertionError(f"store {store}: {bad.shape[0]} outputs differ in rows [{r0}, {r1}), first at {(bad[0] + torch.tensor([r0, 0], device=DEV)).tolist()}")
        g = raw[1 + r0:1 + r1]
        assert (g[:, :32] == SENT[torch.bfloat16]).all() and (g[:, 32 + N:] == SENT[torch.bfloat16]).all(), \
            f"store {store}: columns beside C written in rows [{r0}, {r1})"


@pytest.mark.parametrize("impl", [1, 2])
def test_gemv_weights_past_2_31_bytes(tune, impl):
    """N * K > 2^31 weight bytes (33000 x 65536, 2.2 GB) through both GEMV kernels, M = 4, one-hot A: every output is one
    weight byte times one activation, so a 32-bit row offset shows in the rows past 32768."""
    M, K, N = 4, 65536, 33000
    _need_free(N * K + 2 * 2**30)
    tune("GEMV_IMPL", impl)
    tB = _rand_dev_bytes((N, K), 5)
    rng = np.random.default_rng(impl)
    ks = np.array([0, K - 1, 40000, 12345 + impl])
    vals = codes(M, rng)
    A = np.zeros((M, K), np.uint8)
    A[np.arange(M), ks] = vals
    tA = torch.from_numpy(A).to(DEV)
    sa = ((rng.random(M) + 0.5) * 0.01).astype(np.float32)
    sb = np.float32(0.0217)
    tsa, tsb = dev_f32(sa), dev_f32([sb])
    out = Out(M, N, torch.float32)
    L = capi()
    rc = L.fp8b_scaled_mm(tA.data_ptr(), tB.data_ptr(), out.ptr, 0, M, N, K, out.ldc, tsa.data_ptr(), M, tsb.data_ptr(), 1,
                          None, 0, None, None, 0, ALGO_GEMV, stream_ptr())
    assert rc == 0
    torch.cuda.synchronize()
    Bk = tB[:, torch.from_numpy(ks).to(DEV)].T.cpu().numpy()          # (M, N): B[n, k_m]
    ref = (((o.decode(vals)[:, None] * o.decode(Bk)) * sa[:, None]) * sb).astype(np.float32)
    out.check_guard(f"gemv impl {impl} large")
    assert_bits_equal(to_np(out.view), ref, f"gemv impl {impl} N*K > 2^31")
