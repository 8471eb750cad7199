"""Stream-order tests: every entry point replayed from CUDA graphs, on forked streams and from host threads, bit-exact
against the oracle.

The other bit-exact tests run each call eagerly, from one host thread, on torch's current stream, and synchronise after
it.  Users run the library differently: bench.py and serving loops capture their layers into CUDA graphs, fork
independent calls onto several streams, or call from several host threads.  Correctness then rests on ordering that an
eager, synchronised call never exercises:

  - every GEMV, cast and GEMM launch carries the programmatic-serialization attribute, which becomes a programmatic
    edge of the graph; kernels that start early (launch_dependents at entry) must still wait before they read what the
    node before them writes, and before they overwrite what it reads;
  - host state set up on first use (kernel attributes, device facts, the tensor-map encoder, the per-thread tensor-map
    cache, the bindings' default scale) must be right whichever stream, thread or capture makes the first call.

Inputs are the one-hot families of test_gpu_exact.py, so every output has one
exact value and a stale or reordered read shows up as a wrong bit.  A captured chain is replayed several times with new
data written into its external inputs before each replay: a node that reads before its producer has written gives the
previous replay's answer.  Every output sits in a guard-banded buffer, and the library's launch counter must not move
across replays (a graph replays the launches it captured; the host code does not run again).

The first-use checks run in fresh processes (tests/stream_order_child.py), since in this process earlier tests have
already made every first call."""
import ctypes
import os
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch

import fp8_oracle as o
from _util import (ALGO_AUTO, ALGO_GEMV, ALGO_SIMT, ALGO_TCGEN05, F32, SENT, GemvItem, Out, Terms, add_nan_rows, assert_bits_equal,
                   capi, codes, dt_code, edges, make_spans, one_hot, oracle, p, tc_bounds, to_np, u8_np)

pytestmark = pytest.mark.gpu
DEV = "cuda"
OPT_STATIC_WEIGHTS = 1
OUT_E4M3FN = 3
REPLAYS = 4
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture
def static_weights():
    """static_weights(v): FP8B_OPT_STATIC_WEIGHTS for this test, restored afterwards."""
    L = capi()
    saved = L.fp8b_get_option(OPT_STATIC_WEIGHTS)

    def setter(v):
        assert L.fp8b_set_option(OPT_STATIC_WEIGHTS, int(v)) == 0

    yield setter
    L.fp8b_set_option(OPT_STATIC_WEIGHTS, saved)


def cur_stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev_u8(X):
    return torch.from_numpy(np.ascontiguousarray(X)).to(DEV)


def dev_float(X, dtype):
    """numpy float32 -> device tensor of `dtype`, and the float32 values it holds."""
    t = torch.from_numpy(np.ascontiguousarray(X, np.float32)).to(DEV).to(dtype)
    return t, to_np(t)


def one_hot_values(R, K, positions, rng):
    """float32 rows with one nonzero each (a random normal value with a random binade) at positions[r % len]."""
    X = np.zeros((R, K), np.float32)
    n = len(positions)
    ks = positions[np.arange(R) % n] if R >= n else positions[np.sort(rng.choice(n, R, replace=False))]
    X[np.arange(R), ks] = (rng.standard_normal(R) * np.exp2(rng.integers(-6, 6, R))).astype(np.float32)
    return X


def replayed(record, feed, check, replays=REPLAYS):
    """record(stream) issues the chain and returns the status of every call.  Eager run first (data 0), then one
    capture; before replay r in 1..replays, feed(r) copies replay r's data into the external inputs (on the stream the
    graph replays on).  check(r) compares every output with the oracle for data r."""
    L = capi()
    feed(0)
    assert all(rc == 0 for rc in record(cur_stream())), "eager chain"
    torch.cuda.synchronize()
    check(0, "eager")
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rcs = record(cur_stream())
    assert all(rc == 0 for rc in rcs), f"captured chain: statuses {rcs}"
    n0 = L.fp8b_launch_count()
    for r in range(1, replays + 1):
        feed(r)
        g.replay()
        torch.cuda.synchronize()
        check(r, f"replay {r}")
    assert L.fp8b_launch_count() == n0, "replaying a graph ran the library's host code"
    del g


def check_out(out, ref, what):
    out.check_guard(what)
    assert_bits_equal(to_np(out.view), ref, what)


# ------------------------------------------------------------------ 1. chains whose producer is inside the graph

# name: (tune knobs, algo, (M, K, N))
VARIANTS = {
    "gemv_fhfma": ({"GEMV_IMPL": 1}, ALGO_GEMV, (5, 2048, 96)),
    "gemv_mma": ({"GEMV_IMPL": 2}, ALGO_GEMV, (9, 2048, 80)),
    "generic": ({}, ALGO_GEMV, (3, 1037, 70)),                                 # K % 16 != 0: fp8_gemv_generic_kernel
    "simt": ({}, ALGO_SIMT, (40, 256, 72)),
    "tc_cfg2_st1": ({"GEMM_CFG": 2, "GEMM_STORE": 1}, ALGO_TCGEN05, (200, 384, 256)),
    "tc_cfg2_st2": ({"GEMM_CFG": 2, "GEMM_STORE": 2}, ALGO_TCGEN05, (200, 384, 256)),
    "tc_cfg3_st1": ({"GEMM_CFG": 3, "GEMM_STORE": 1}, ALGO_TCGEN05, (300, 384, 512)),
    "tc_cfg3_st2": ({"GEMM_CFG": 3, "GEMM_STORE": 2}, ALGO_TCGEN05, (300, 384, 512)),
    "splitk2": ({"GEMM_SPLITK": 2}, ALGO_TCGEN05, (32, 3072, 256)),
    "splitk4": ({"GEMM_SPLITK": 4}, ALGO_TCGEN05, (32, 3072, 256)),
}
CHAIN_CASES = [(v, prod, 0) for v in sorted(VARIANTS) for prod in ("encode", "quantize_rows")] + \
              [(v, prod, 1) for v in ("gemv_fhfma", "gemv_mma", "tc_cfg2_st2") for prod in ("encode", "quantize_rows")]
X_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


@pytest.mark.parametrize("variant,producer,static", CHAIN_CASES)
def test_captured_producer_then_matmul(tune, static_weights, variant, producer, static):
    """fp8b_encode (A = the codes of X) or fp8b_quantize_rows (A = per-row quantised X, scale_a = its inverse scales)
    feeding fp8b_scaled_mm in one graph.  X changes before every replay; B changes too unless STATIC_WEIGHTS is on
    (then it is truly static).  Even replays: one-hot A rows against dense B codes with NaN rows; odd replays: dense A
    against one-hot B rows -- every output is one exact product."""
    knobs, algo, (M, K, N) = VARIANTS[variant]
    for k, v in knobs.items():
        tune(k, v)
    static_weights(static)
    vi = sorted(VARIANTS).index(variant)
    xdt = X_DTYPES[vi % 3]
    odt = (torch.float32, torch.bfloat16, torch.float16)[(vi + static) % 3]
    rng = np.random.default_rng(1000 * vi + 10 * static + (producer == "encode"))
    bounds = tc_bounds(K) if algo == ALGO_TCGEN05 else set(range(64, K, 64))
    pos = edges(K, bounds, rng)

    data = []
    B0 = add_nan_rows(codes((N, K), rng), one_hot(M, K, pos, rng), [1, N - 1], rng)
    for r in range(REPLAYS + 1):
        dense_a = r % 2 == 1 and not static
        if producer == "encode":
            A = codes((M, K), rng) if dense_a else one_hot(M, K, pos, rng)
            A[A == 0x80] = 0x00                           # -0.0 encodes to 0x00
            X = o.decode(A)
        else:
            X = (rng.standard_normal((M, K)) * 3).astype(np.float32) if dense_a else one_hot_values(M, K, pos, rng)
        B = one_hot(N, K, pos, rng) if dense_a else (B0 if static or r == 0 else
                                                     add_nan_rows(codes((N, K), rng), one_hot(M, K, pos, rng), [r, N - 2], rng))
        data.append((dev_float(X, xdt), dev_u8(B), B))

    t = Terms.cycle(vi + 2 * static, M, N, rng).device()          # (scale_a: the row scales of quantize_rows instead)
    tX = torch.empty(M, K, dtype=xdt, device=DEV)
    tB = torch.empty(N, K, dtype=torch.uint8, device=DEV)
    qA = torch.empty(M * K + 64, dtype=torch.uint8, device=DEV)
    inv = torch.empty(M + 8, dtype=torch.float32, device=DEV)
    out = Out(M, N, odt)
    L = capi()
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0

    def record(s):
        if producer == "encode":
            rc0 = L.fp8b_encode(p(tX), dt_code(xdt), p(qA), M * K, None, s)
            sa, sa_len = p(t.t_sa), len(t.sa)
        else:
            rc0 = L.fp8b_quantize_rows(p(tX), dt_code(xdt), M, K, p(qA), p(inv), s)
            sa, sa_len = p(inv), M
        rc1 = L.fp8b_scaled_mm(p(qA), p(tB), out.ptr, dt_code(odt), M, N, K, out.ldc, sa, sa_len, p(t.t_sb), len(t.sb),
                               p(t.t_bias), bc, p(t.t_sr), None, 0, algo, s)
        return rc0, rc1

    def feed(r):
        (xs, _), bs, _ = data[r]
        tX.copy_(xs)
        if r == 0 or not static:
            tB.copy_(bs)

    def check(r, what):
        (_, xv), _, B = data[r]
        what = f"{variant} {producer} static {static} {what}"
        if producer == "encode":
            A, sa = o.encode(xv), t.sa
        else:
            A, sa = o.fp8_quantize_rows(xv)
            assert_bits_equal(to_np(inv[:M]), sa, f"{what}: inverse row scales")
        assert np.array_equal(u8_np(qA[:M * K]).reshape(M, K), A), f"{what}: quantised A"
        check_out(out, oracle(A, B, sa, t.sb, t.bias, t.sr, odt), what)

    replayed(record, feed, check)


DYN_PLANS = {"chain": (4, 2048, 96, True), "single": (4, 2048, 96, False), "gemm": (40, 512, 256, True)}   # M, K, N, workspace


@pytest.mark.parametrize("static", [0, 1])
@pytest.mark.parametrize("plan", sorted(DYN_PLANS))
def test_captured_linear_dynamic(static_weights, plan, static):
    """fp8b_linear_dynamic in a graph: the quantise + chained GEMV plan (M <= 16, the GEMV starts behind the quantise
    kernel through the programmatic edge), the single-kernel plan (no workspace), and M > 16 (the quantise kernel
    writes the per-row scale_a the GEMM reads just after it).  X changes before every replay."""
    M, K, N, ws = DYN_PLANS[plan]
    static_weights(static)
    rng = np.random.default_rng(len(plan) * 7 + static)
    pos = edges(K, tc_bounds(K), rng)
    B = add_nan_rows(codes((N, K), rng), one_hot(M, K, pos, rng), [0, N - 3], rng)
    Xs = [dev_float(one_hot_values(M, K, pos, rng), torch.float32) for _ in range(REPLAYS + 1)]
    t = Terms(M, N, rng, per_row_b=True, bias_dt=torch.bfloat16, sr=bool(static)).device()
    odt = torch.bfloat16 if static else torch.float32
    tX = torch.empty(M, K, device=DEV)
    tB = dev_u8(B)
    inv = torch.empty(M + 8, device=DEV)
    L = capi()
    nws = L.fp8b_linear_dynamic_workspace_bytes(M, K) if ws else 0
    work = torch.empty(max(nws, 16), dtype=torch.uint8, device=DEV)
    out = Out(M, N, odt)

    def record(s):
        return (L.fp8b_linear_dynamic(p(tX), F32, p(tB), out.ptr, dt_code(odt), M, N, K, out.ldc, p(t.t_sb), len(t.sb), p(t.t_bias),
                                      dt_code(t.bias_dt), p(t.t_sr), p(inv), p(work) if ws else None, nws, s),)

    def feed(r):
        tX.copy_(Xs[r][0])

    def check(r, what):
        what = f"linear_dynamic {plan} static {static} {what}"
        A, sa = o.fp8_quantize_rows(Xs[r][1])
        assert_bits_equal(to_np(inv[:M]), sa, f"{what}: inverse row scales")
        check_out(out, oracle(A, B, sa, t.sb, t.bias, t.sr, odt), what)

    replayed(record, feed, check)


@pytest.mark.parametrize("M", [4, 64])
def test_captured_fp8_output_chain(M):
    """GEMM 1 writes e4m3fn bytes (FP8B_OUT_E4M3FN), GEMM 2 reads them as its A, fp8b_dequant turns them back into
    float32 -- all in one graph, A of GEMM 1 new before every replay.  M = 4: GEMVs; M = 64: tcgen05."""
    K, N1, N2 = 512, 128, 96
    rng = np.random.default_rng(M)
    pos = edges(K, tc_bounds(K), rng)
    B1 = codes((N1, K), rng)
    B2 = one_hot(N2, N1, np.arange(N1), rng)
    A1s = [one_hot(M, K, pos, rng) for _ in range(REPLAYS + 1)]
    t1 = Terms(M, N1, rng, per_row_a=True, bias_dt=torch.float32).device()
    t2 = Terms(M, N2, rng, per_row_b=True, sr=True).device()
    tA1, tB1, tB2 = torch.empty(M, K, dtype=torch.uint8, device=DEV), dev_u8(B1), dev_u8(B2)
    C1 = torch.empty(M, N1, dtype=torch.uint8, device=DEV)
    D1 = torch.empty(M * N1, dtype=torch.float32, device=DEV)
    out = Out(M, N2, torch.float32)
    L = capi()

    def record(s):
        return (L.fp8b_scaled_mm(p(tA1), p(tB1), p(C1), OUT_E4M3FN, M, N1, K, N1, p(t1.t_sa), len(t1.sa), p(t1.t_sb), len(t1.sb),
                                 p(t1.t_bias), F32, None, None, 0, ALGO_AUTO, s),
                L.fp8b_scaled_mm(p(C1), p(tB2), out.ptr, F32, M, N2, N1, out.ldc, p(t2.t_sa), len(t2.sa), p(t2.t_sb), len(t2.sb),
                                 None, 0, p(t2.t_sr), None, 0, ALGO_AUTO, s),
                L.fp8b_dequant(p(C1), p(D1), F32, M * N1, s))

    def feed(r):
        tA1.copy_(dev_u8(A1s[r]))

    def check(r, what):
        what = f"fp8 output chain M{M} {what}"
        ref1 = o.encode(oracle(A1s[r], B1, t1.sa, t1.sb, t1.bias, None, torch.float32))
        assert np.array_equal(u8_np(C1), ref1), f"{what}: e4m3fn output of GEMM 1"
        check_out(out, oracle(ref1, B2, t2.sa, t2.sb, None, t2.sr, torch.float32), f"{what}: GEMM 2")
        assert_bits_equal(to_np(D1).reshape(M, N1), o.decode(ref1), f"{what}: dequant", any_nan=True)

    replayed(record, feed, check)


def test_captured_batched_casts_and_gemv_batch():
    """fp8b_encode_batch (three float tensors -> codes) -> fp8b_gemv_batch (the codes as x of three GEMVs) and
    fp8b_dequant_batch (the codes back to float) in one graph, beside fp8b_amax_scale -> fp8b_encode on a fourth tensor:
    the amax scratch is reset by a memset node of the same graph.  The amax falls from replay to replay, so a scratch
    word left from the previous replay gives the old scale."""
    K, Ns = 1024, (40, 96, 130)
    rng = np.random.default_rng(5)
    pos = edges(K, set(range(64, K, 64)), rng)
    Ws = [codes((n, K), rng) for n in Ns]
    sws = [((rng.random(n) + 0.5) * 0.01).astype(np.float32) for n in Ns]
    biases = [(rng.standard_normal(n) * 0.5).astype(np.float32) for n in Ns]
    sx = np.float32(0.0371)
    n_big = 70001
    Xs, Bigs = [], []
    for r in range(REPLAYS + 1):
        A = one_hot(3, K, pos, rng)
        A[A == 0x80] = 0
        Xs.append([dev_float(o.decode(A[i:i + 1]), torch.float16) for i in range(3)])
        big = (rng.standard_normal(n_big) * np.exp2(rng.integers(-10, 4, n_big))).astype(np.float32)
        big[rng.integers(0, n_big)] = np.float32(3000.0 / (r + 1))            # the amax, smaller every replay
        Bigs.append(dev_float(big, torch.float32))
    tXs = [torch.empty(1, K, dtype=torch.float16, device=DEV) for _ in Ns]
    xq = [torch.empty(K, dtype=torch.uint8, device=DEV) for _ in Ns]
    back = [torch.empty(K, dtype=torch.bfloat16, device=DEV) for _ in Ns]
    ys = [Out(1, n, torch.float32) for n in Ns]
    tW = [dev_u8(w) for w in Ws]
    tsw = [torch.from_numpy(s).to(DEV) for s in sws]
    tb = [torch.from_numpy(b).to(DEV) for b in biases]
    tsx = torch.full((1,), float(sx), device=DEV)
    items = (GemvItem * 3)()
    for i in range(3):
        items[i].x, items[i].W, items[i].y, items[i].N = xq[i].data_ptr(), tW[i].data_ptr(), ys[i].ptr, Ns[i]
        items[i].scale_x, items[i].scale_w, items[i].scale_w_len, items[i].bias = tsx.data_ptr(), tsw[i].data_ptr(), Ns[i], tb[i].data_ptr()
    enc_spans = make_spans([(tXs[i].data_ptr(), xq[i].data_ptr(), K) for i in range(3)])
    dq_spans = make_spans([(xq[i].data_ptr(), back[i].data_ptr(), K) for i in range(3)])
    tBig = torch.empty(n_big, device=DEV)
    qBig = torch.empty(n_big, dtype=torch.uint8, device=DEV)
    scales = torch.empty(2, device=DEV)
    scratch = torch.empty(1, dtype=torch.int32, device=DEV)
    L = capi()

    def record(s):
        return (L.fp8b_encode_batch(enc_spans, 3, dt_code(torch.float16), s),
                L.fp8b_gemv_batch(items, 3, K, F32, F32, s),
                L.fp8b_dequant_batch(dq_spans, 3, dt_code(torch.bfloat16), s),
                L.fp8b_amax_scale(p(tBig), F32, n_big, p(scales), ctypes.c_void_p(scales.data_ptr() + 4), p(scratch), s),
                L.fp8b_encode(p(tBig), F32, p(qBig), n_big, p(scales), s))

    def feed(r):
        for i in range(3):
            tXs[i].copy_(Xs[r][i][0])
        tBig.copy_(Bigs[r][0])

    def check(r, what):
        for i in range(3):
            A = o.encode(Xs[r][i][1])
            assert np.array_equal(u8_np(xq[i]), A[0]), f"{what}: encode_batch span {i}"
            assert_bits_equal(to_np(back[i]), o.decode(A[0]), f"{what}: dequant_batch span {i}")
            check_out(ys[i], oracle(A, Ws[i], np.array([sx]), sws[i], biases[i], None, torch.float32), f"{what}: gemv_batch item {i}")
        q, inv = o.fp8_quantize(Bigs[r][1])
        assert_bits_equal(to_np(scales[1:]), inv, f"{what}: amax_scale inverse scale")
        assert np.array_equal(u8_np(qBig), q), f"{what}: prescaled encode"

    replayed(record, feed, check)


@pytest.mark.parametrize("n_dst", [1, 2, 3])
def test_captured_quantize_then_push(n_dst):
    """fp8b_quantize_rows -> fp8b_scaled_mm_push into 1-3 local destination buffers (column block [n0, n0 + N) of each),
    in one graph; X new before every replay."""
    M, K, N, full_N, n0 = 256, 384, 128, 384, 128
    rng = np.random.default_rng(40 + n_dst)
    pos = edges(K, tc_bounds(K), rng)
    B = codes((N, K), rng)
    Xs = [dev_float(one_hot_values(M, K, pos, rng), torch.float32) for _ in range(REPLAYS + 1)]
    t = Terms(M, N, rng, per_row_b=True, bias_dt=torch.float16).device()
    odt = torch.bfloat16
    tX, tB = torch.empty(M, K, device=DEV), dev_u8(B)
    q = torch.empty(M, K, dtype=torch.uint8, device=DEV)
    inv = torch.empty(M, device=DEV)
    dsts = [torch.full((M, full_N), SENT[odt], dtype=torch.int16, device=DEV).view(odt) for _ in range(n_dst)]
    arr = (ctypes.c_void_p * n_dst)(*[d.data_ptr() + n0 * 2 for d in dsts])
    L = capi()

    def record(s):
        return (L.fp8b_quantize_rows(p(tX), F32, M, K, p(q), p(inv), s),
                L.fp8b_scaled_mm_push(p(q), p(tB), arr, n_dst, dt_code(odt), M, N, K, full_N, p(inv), M, p(t.t_sb), len(t.sb),
                                      p(t.t_bias), dt_code(t.bias_dt), None, s))

    def feed(r):
        tX.copy_(Xs[r][0])

    def check(r, what):
        A, sa = o.fp8_quantize_rows(Xs[r][1])
        ref = oracle(A, B, sa, t.sb, t.bias, None, odt)
        for d, buf in enumerate(dsts):
            w = f"push {n_dst} destinations, destination {d}, {what}"
            assert_bits_equal(to_np(buf[:, n0:n0 + N]), ref, w)
            raw = buf.view(torch.int16).clone()
            raw[:, n0:n0 + N] = SENT[odt]
            assert bool((raw == SENT[odt]).all()), f"{w}: written outside its column block"

    replayed(record, feed, check)


# ------------------------------------------------------------------ 2. write-after-read inside a graph

@pytest.mark.parametrize("impl,static", [(1, 0), (1, 1), (2, 0), (2, 1)])
def test_graph_war_gemv_x(tune, static_weights, impl, static):
    """Layer 1's GEMV reads the x buffer, the next node encodes layer 2's input into that same buffer, layer 2's GEMV
    reads it: the encode must not overwrite x while layer 1 still reads it, and layer 2 must read the new x."""
    tune("GEMV_IMPL", impl)
    static_weights(static)
    M, K, N1, N2 = 4, 4096, 120, 88
    rng = np.random.default_rng(impl * 3 + static)
    pos = edges(K, set(range(64, K, 64)), rng)
    W1, W2 = codes((N1, K), rng), codes((N2, K), rng)
    feeds = []
    for r in range(REPLAYS + 1):
        pair = []
        for _ in range(2):
            A = one_hot(M, K, pos, rng)
            A[A == 0x80] = 0
            pair.append(dev_float(o.decode(A), torch.bfloat16))
        feeds.append(pair)
    t1, t2 = Terms(M, N1, rng, per_row_a=True).device(), Terms(M, N2, rng, bias_dt=torch.float32).device()
    tX1, tX2 = torch.empty(M, K, dtype=torch.bfloat16, device=DEV), torch.empty(M, K, dtype=torch.bfloat16, device=DEV)
    x = torch.empty(M, K, dtype=torch.uint8, device=DEV)
    tW1, tW2 = dev_u8(W1), dev_u8(W2)
    y1, y2 = Out(M, N1, torch.float32), Out(M, N2, torch.float16)
    L = capi()
    bf = dt_code(torch.bfloat16)

    def record(s):
        return (L.fp8b_encode(p(tX1), bf, p(x), M * K, None, s),
                L.fp8b_scaled_mm(p(x), p(tW1), y1.ptr, F32, M, N1, K, y1.ldc, p(t1.t_sa), M, p(t1.t_sb), 1, None, 0, None, None, 0,
                                 ALGO_GEMV, s),
                L.fp8b_encode(p(tX2), bf, p(x), M * K, None, s),
                L.fp8b_scaled_mm(p(x), p(tW2), y2.ptr, dt_code(torch.float16), M, N2, K, y2.ldc, p(t2.t_sa), 1, p(t2.t_sb), 1,
                                 p(t2.t_bias), F32, None, None, 0, ALGO_GEMV, s))

    def feed(r):
        tX1.copy_(feeds[r][0][0])
        tX2.copy_(feeds[r][1][0])

    def check(r, what):
        A1, A2 = o.encode(feeds[r][0][1]), o.encode(feeds[r][1][1])
        check_out(y1, oracle(A1, W1, t1.sa, t1.sb, None, None, torch.float32), f"WAR gemv layer 1 {what}")
        check_out(y2, oracle(A2, W2, t2.sa, t2.sb, t2.bias, None, torch.float16), f"WAR gemv layer 2 {what}")

    replayed(record, feed, check)


@pytest.mark.parametrize("cfg", [2, 3])
def test_graph_war_gemm_a(tune, cfg):
    """quantize_rows -> GEMM 1 -> quantize_rows of the next layer into the SAME A and scale_a buffers -> GEMM 2: the
    second quantise must not overwrite A or the row scales while GEMM 1 still reads them."""
    tune("GEMM_CFG", cfg)
    M, K, N1, N2 = 256, 512, 256, 384
    rng = np.random.default_rng(cfg)
    pos = edges(K, tc_bounds(K), rng)
    B1 = add_nan_rows(codes((N1, K), rng), one_hot(M, K, pos, rng), [4], rng)
    B2 = codes((N2, K), rng)
    Xs = [[dev_float(one_hot_values(M, K, pos, rng), torch.float32) for _ in range(2)] for _ in range(REPLAYS + 1)]
    t1 = Terms(M, N1, rng, per_row_b=True, bias_dt=torch.bfloat16).device()
    t2 = Terms(M, N2, rng, sr=True).device()
    tX1, tX2 = torch.empty(M, K, device=DEV), torch.empty(M, K, device=DEV)
    q = torch.empty(M, K, dtype=torch.uint8, device=DEV)
    inv = torch.empty(M, device=DEV)
    tB1, tB2 = dev_u8(B1), dev_u8(B2)
    c1, c2 = Out(M, N1, torch.bfloat16), Out(M, N2, torch.float32)
    L = capi()

    def record(s):
        return (L.fp8b_quantize_rows(p(tX1), F32, M, K, p(q), p(inv), s),
                L.fp8b_scaled_mm(p(q), p(tB1), c1.ptr, dt_code(torch.bfloat16), M, N1, K, c1.ldc, p(inv), M, p(t1.t_sb), N1,
                                 p(t1.t_bias), dt_code(torch.bfloat16), None, None, 0, ALGO_TCGEN05, s),
                L.fp8b_quantize_rows(p(tX2), F32, M, K, p(q), p(inv), s),
                L.fp8b_scaled_mm(p(q), p(tB2), c2.ptr, F32, M, N2, K, c2.ldc, p(inv), M, p(t2.t_sb), 1, None, 0, p(t2.t_sr), None, 0,
                                 ALGO_TCGEN05, s))

    def feed(r):
        tX1.copy_(Xs[r][0][0])
        tX2.copy_(Xs[r][1][0])

    def check(r, what):
        A1, s1 = o.fp8_quantize_rows(Xs[r][0][1])
        A2, s2 = o.fp8_quantize_rows(Xs[r][1][1])
        check_out(c1, oracle(A1, B1, s1, t1.sb, t1.bias, None, torch.bfloat16), f"WAR gemm cfg {cfg} layer 1 {what}")
        check_out(c2, oracle(A2, B2, s2, t2.sb, None, t2.sr, torch.float32), f"WAR gemm cfg {cfg} layer 2 {what}")

    replayed(record, feed, check)


# ------------------------------------------------------------------ 3. forked streams

# (M, K, N, algo, out dtype): independent problems on as many kernels
FORK_PROBLEMS = [(1, 4096, 200, ALGO_AUTO, torch.float16), (8, 2048, 96, ALGO_AUTO, torch.float32),
                 (3, 1037, 70, ALGO_GEMV, torch.bfloat16), (40, 256, 72, ALGO_SIMT, torch.float32),
                 (200, 384, 256, ALGO_AUTO, torch.bfloat16), (32, 3072, 256, ALGO_AUTO, torch.float32),
                 (600, 256, 1024, ALGO_AUTO, torch.float16), (128, 512, 384, ALGO_TCGEN05, torch.float32)]


class Problem:
    """One fp8b_scaled_mm with its own operands, terms and guarded output; A can be re-rolled."""

    def __init__(self, i, M, K, N, algo, odt, rng):
        self.M, self.K, self.N, self.algo, self.odt, self.rng = M, K, N, algo, odt, rng
        self.pos = edges(K, tc_bounds(K) | set(range(64, K, 64)), rng)
        self.B = add_nan_rows(codes((N, K), rng), one_hot(M, K, self.pos, rng), [N - 1], rng)
        self.t = Terms.cycle(i, M, N, rng).device()
        self.tA = torch.empty(M, K, dtype=torch.uint8, device=DEV)
        self.tB = dev_u8(self.B)
        self.new_a()

    def new_a(self):
        """new one-hot A rows (exact against any B)."""
        self.A = one_hot(self.M, self.K, self.pos, self.rng)

    def upload(self):
        self.tA.copy_(dev_u8(self.A))

    def call(self, out, s):
        t = self.t
        return capi().fp8b_scaled_mm(p(self.tA), p(self.tB), out.ptr, dt_code(self.odt), self.M, self.N, self.K, out.ldc, p(t.t_sa),
                                     len(t.sa), p(t.t_sb), len(t.sb), p(t.t_bias), dt_code(t.bias_dt) if t.bias_dt else 0,
                                     p(t.t_sr), None, 0, self.algo, s)

    def ref(self):
        t = self.t
        return oracle(self.A, self.B, t.sa, t.sb, t.bias, t.sr, self.odt)


def _forked(problems, outs, streams):
    """Round-robin over `streams`, each forked from and joined back into the current stream with events."""
    cur = torch.cuda.current_stream()
    for s in streams:
        s.wait_stream(cur)
    rcs = []
    for i, (pb, out) in enumerate(zip(problems, outs)):
        s = streams[i % len(streams)]
        with torch.cuda.stream(s):
            rcs.append(pb.call(out, ctypes.c_void_p(s.cuda_stream)))
    for s in streams:
        cur.wait_stream(s)
    return rcs


def test_forked_streams_eager_and_captured():
    """Eight independent matmuls (GEMVs, the generic kernel, SIMT, tcgen05 one-CTA / pair / split-K tiles) issued
    round-robin on 4 non-default streams joined by events, eagerly and inside a graph: the bits equal a one-stream
    run and the oracle.  The captured fork is replayed with new A data."""
    rng = np.random.default_rng(77)
    probs = [Problem(i, *spec, rng) for i, spec in enumerate(FORK_PROBLEMS)]
    for pb in probs:
        pb.upload()
    single = [Out(pb.M, pb.N, pb.odt) for pb in probs]
    assert all(pb.call(out, cur_stream()) == 0 for pb, out in zip(probs, single))
    torch.cuda.synchronize()
    for i, (pb, out) in enumerate(zip(probs, single)):
        check_out(out, pb.ref(), f"one stream, problem {i}")

    streams = [torch.cuda.Stream() for _ in range(4)]
    forked = [Out(pb.M, pb.N, pb.odt) for pb in probs]
    assert all(rc == 0 for rc in _forked(probs, forked, streams))
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(forked, single)):
        a.check_guard(f"eager fork, problem {i}")
        assert torch.equal(a.buf.view(torch.uint8), b.buf.view(torch.uint8)), f"eager fork, problem {i}: bits differ from one stream"

    L = capi()
    cap = [Out(pb.M, pb.N, pb.odt) for pb in probs]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rcs = _forked(probs, cap, streams)
    assert all(rc == 0 for rc in rcs), rcs
    n0 = L.fp8b_launch_count()
    for r in range(3):
        if r:
            for pb in probs:
                pb.new_a()
                pb.upload()
        g.replay()
        torch.cuda.synchronize()
        for i, (pb, out) in enumerate(zip(probs, cap)):
            check_out(out, pb.ref(), f"captured fork replay {r}, problem {i}")
        if r == 0:
            for i, (a, b) in enumerate(zip(cap, single)):
                assert torch.equal(a.buf.view(torch.uint8), b.buf.view(torch.uint8)), f"captured fork, problem {i}: bits differ"
    assert L.fp8b_launch_count() == n0


# ------------------------------------------------------------------ 4. host threads and the tensor-map cache

# per thread: (M, K, N, out dtype) problems on distinct kernels: GEMV, generic, SIMT (AUTO with K % 16 != 0), tcgen05
# one-CTA / pair / split-K, TMA-store and st.global epilogues
THREAD_PROBLEMS = [
    [(1, 4096, 300, torch.float32), (16, 1024, 64, torch.bfloat16)],
    [(200, 384, 256, torch.bfloat16), (5, 1037, 33, torch.float32)],
    [(600, 256, 1024, torch.float16), (2, 2048, 128, torch.float16)],
    [(32, 3072, 256, torch.float32), (50, 1000, 60, torch.bfloat16)],
    [(128, 512, 384, torch.bfloat16), (300, 128, 520, torch.float32)],
    [(256, 640, 200, torch.float32), (9, 4096, 80, torch.bfloat16)],
]


def test_host_threads():
    """Six host threads, each on its own stream with its own shapes (so different kernels and tensor maps are live at
    the same time), call the library through ctypes -- which releases the GIL -- from a common start.  Each runs its
    problems twice (the second round finds its maps in its cache) and every output is exact.  Every problem runs once
    on the main thread first, so a thread's first call finds its kernel attributes set and makes no runtime call that
    would bind a CUDA context before its first tensor-map encode: the library has to give the thread one."""
    rng = np.random.default_rng(123)
    work = []
    for t, specs in enumerate(THREAD_PROBLEMS):
        items = []
        for j, (M, K, N, odt) in enumerate(specs):
            pb = Problem(2 * t + j, M, K, N, ALGO_AUTO, odt, rng)
            pb.upload()
            items.append((pb, [Out(M, N, odt), Out(M, N, odt)]))
        work.append(items)
    for items in work:
        for pb, _ in items:
            assert pb.call(Out(pb.M, pb.N, pb.odt), cur_stream()) == 0
    streams = [torch.cuda.Stream() for _ in work]
    torch.cuda.synchronize()
    start = threading.Barrier(len(work))
    rcs = [[] for _ in work]
    errors = []

    def body(t):
        try:
            s = ctypes.c_void_p(streams[t].cuda_stream)
            start.wait()
            for rnd in range(2):
                for pb, outs in work[t]:
                    rc = pb.call(outs[rnd], s)
                    rcs[t].append(rc if rc == 0 else (rc, capi().fp8b_last_cuda_error()))    # the CUDA error is per thread
        except Exception as e:          # reported by the main thread
            errors.append(e)

    threads = [threading.Thread(target=body, args=(t,)) for t in range(len(work))]
    for th in threads:
        th.start()
    for th in threads:
        th.join(timeout=120)
    assert not any(th.is_alive() for th in threads), "a host thread did not finish"
    assert not errors, errors
    torch.cuda.synchronize()
    for t, items in enumerate(work):
        assert rcs[t] == [0] * (2 * len(items)), f"thread {t}: statuses (status, cuda error) {rcs[t]}"
        for j, (pb, outs) in enumerate(items):
            for rnd, out in enumerate(outs):
                check_out(out, pb.ref(), f"thread {t} problem {j} (M{pb.M} K{pb.K} N{pb.N}) round {rnd}")


def _strided_call(tA, A, tB, B, M, K, N, c_buf, c_off, ldc, rng, what):
    """One tcgen05 GEMM (A: the first M x K bytes at tA, TMA-store epilogue) into C at c_buf + c_off with row pitch ldc
    (float32); checks C and that nothing else in c_buf was written."""
    t = Terms(M, N, rng).device()
    c_buf.view(torch.int32).fill_(SENT[torch.float32])
    ptr = c_buf.data_ptr() + c_off * 4
    rc = capi().fp8b_scaled_mm(p(tA), p(tB), ctypes.c_void_p(ptr), F32, M, N, K, ldc, p(t.t_sa), 1, p(t.t_sb), 1, None, 0,
                               None, None, 0, ALGO_TCGEN05, cur_stream())
    torch.cuda.synchronize()
    assert rc == 0, what
    flat = c_buf.view(torch.int32)
    C = c_buf[c_off:c_off + M * ldc].view(M, ldc)[:, :N]
    assert_bits_equal(to_np(C), oracle(A, B, t.sa, t.sb, None, None, torch.float32), what)
    raw = flat.clone()
    raw[c_off:c_off + M * ldc].view(M, ldc)[:, :N] = SENT[torch.float32]
    assert bool((raw == SENT[torch.float32]).all()), f"{what}: written outside C"


def test_tensor_map_cache_same_base_other_geometry(tune):
    """The same base pointer with a different geometry must get its own tensor map: A with more rows, A with another
    K (row pitch), and C with another row pitch (TMA-store epilogue).  A map of the earlier geometry would read the
    wrong rows / bytes or store to the wrong rows."""
    tune("GEMM_CFG", 2)
    tune("GEMM_STORE", 2)
    rng = np.random.default_rng(9)
    abuf = torch.empty(300 * 512 + 256, dtype=torch.uint8, device=DEV)
    c_buf = torch.empty(4096 + 300 * 320, dtype=torch.float32, device=DEV)
    for (M, K, N, ldc) in [(128, 256, 128, 128), (200, 256, 128, 128), (200, 384, 128, 128), (200, 384, 128, 160),
                           (200, 384, 128, 192), (128, 256, 128, 160)]:
        pos = edges(K, tc_bounds(K), rng)
        A, B = one_hot(M, K, pos, rng), codes((N, K), rng)
        abuf[:M * K].copy_(dev_u8(A.reshape(-1)))
        _strided_call(abuf, A, dev_u8(B), B, M, K, N, c_buf, 1024, ldc, rng, f"same base: M{M} K{K} ldc{ldc}")


def test_tensor_map_cache_many_live_maps(tune):
    """More than 64 live tensor maps: 42 GEMMs with one-CTA tiles and the TMA-store epilogue (forced, so each GEMM uses
    three maps: A, B and C), whose A and B bases lie 256 bytes apart, so the 126 maps collide in the 64-slot cache.
    Two passes in the same order; every output is exact and the sentinels between the C windows stay intact.  (Every
    map here has one geometry; a cache key that ignores rows or pitch is checked by the same-base test above.)"""
    tune("GEMM_CFG", 2)
    tune("GEMM_STORE", 2)
    rng = np.random.default_rng(10)
    M, K, N, n = 128, 128, 128, 42
    gap = 64                                           # sentinel floats between consecutive C windows
    pos = edges(K, tc_bounds(K), rng)
    abig = torch.empty(n * 256 + M * K, dtype=torch.uint8, device=DEV)
    bbig = torch.empty(n * 256 + N * K, dtype=torch.uint8, device=DEV)
    cbig = torch.empty(gap + n * (M * N + gap), dtype=torch.float32, device=DEV)
    As = [one_hot(M, K, pos, rng) for _ in range(n)]
    Bs = [codes((N, K), rng) for _ in range(n)]
    t = Terms(M, N, rng).device()
    L = capi()
    for rnd in range(2):
        cbig.view(torch.int32).fill_(SENT[torch.float32])
        for i in range(n):
            abig[i * 256:i * 256 + M * K].copy_(dev_u8(As[i].reshape(-1)))
            bbig[i * 256:i * 256 + N * K].copy_(dev_u8(Bs[i].reshape(-1)))
            c0 = gap + i * (M * N + gap)
            rc = L.fp8b_scaled_mm(ctypes.c_void_p(abig.data_ptr() + i * 256), ctypes.c_void_p(bbig.data_ptr() + i * 256),
                                  ctypes.c_void_p(cbig.data_ptr() + c0 * 4), F32, M, N, K, N, p(t.t_sa), 1, p(t.t_sb), 1, None, 0,
                                  None, None, 0, ALGO_TCGEN05, cur_stream())
            assert rc == 0, f"map {i} pass {rnd}: status {rc}"
            torch.cuda.synchronize()
            got = to_np(cbig[c0:c0 + M * N]).reshape(M, N)
            assert_bits_equal(got, oracle(As[i], Bs[i], t.sa, t.sb, None, None, torch.float32), f"map {i} pass {rnd}")
        raw = cbig.view(torch.int32).clone()
        for i in range(n):
            c0 = gap + i * (M * N + gap)
            raw[c0:c0 + M * N] = SENT[torch.float32]
        assert bool((raw == SENT[torch.float32]).all()), f"pass {rnd}: a GEMM wrote outside its C window"


# ------------------------------------------------------------------ 5. fresh processes: first use inside a capture

CHILD = os.path.join(HERE, "stream_order_child.py")


@pytest.mark.parametrize("scenario", ["first_calls_captured", "default_scale_captured", "default_scale_busy_stream"])
def test_fresh_process(scenario):
    """tests/stream_order_child.py in a new process:
      first_calls_captured      the process's first call of every entry point is made inside torch.cuda.graph;
      default_scale_captured    the first default-scale `_scaled_mm` is captured, then an eager call runs before any
                                replay;
      default_scale_busy_stream the first default-scale call is made on a stream held busy by a delay kernel, and one
                                on another stream follows at once."""
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [CHILD, scenario]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout.splitlines()[-1:], f"{scenario}: exit {r.returncode}\n{r.stdout[-4000:]}"
