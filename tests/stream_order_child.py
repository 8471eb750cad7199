"""Fresh-process scenarios of test_gpu_stream_order.py (run as `python stream_order_child.py <scenario>`; not collected
by pytest).  Each scenario needs a process in which the library has made no call yet: the host state it sets up on
first use must be right when that first use is inside a graph capture or on a busy stream.  Prints "ok" last on
success; raises otherwise."""
import ctypes
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (HERE, os.path.join(ROOT, "fp8-mps-metal_b200"), os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import fp8_oracle as o  # noqa: E402
from _util import (ALGO_AUTO, ALGO_SIMT, F32, GemvItem, Out, Terms, assert_bits_equal, capi, codes, dt_code, make_spans,  # noqa: E402
                   one_hot, oracle, p, to_np, u8_np)

DEV = "cuda"


def s_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev_u8(X):
    return torch.from_numpy(np.ascontiguousarray(X)).to(DEV)


def first_calls_captured():
    """The first call of every entry point is made inside torch.cuda.graph (global capture mode); one replay must
    give the oracle's bits.  The bindings' ops follow, also first used inside a capture."""
    L = capi()
    rng = np.random.default_rng(1)
    checks = []
    calls = []

    def mm(M, K, N, odt, algo, what):
        pos = np.arange(0, K, 16)
        A, B = one_hot(M, K, pos, rng), codes((N, K), rng)
        t = Terms(M, N, rng, per_row_a=True, bias_dt=torch.float32).device()
        tA, tB, out = dev_u8(A), dev_u8(B), Out(M, N, odt)
        calls.append((what, lambda s: L.fp8b_scaled_mm(p(tA), p(tB), out.ptr, dt_code(odt), M, N, K, out.ldc, p(t.t_sa), M, p(t.t_sb), 1,
                                                        p(t.t_bias), F32, None, None, 0, algo, s), (tA, tB, t)))
        checks.append((what, lambda: (out.check_guard(what),
                                      assert_bits_equal(to_np(out.view), oracle(A, B, t.sa, t.sb, t.bias, None, odt), what))))

    mm(2, 2048, 96, torch.float32, ALGO_AUTO, "scaled_mm GEMV")
    mm(200, 384, 256, torch.bfloat16, ALGO_AUTO, "scaled_mm tcgen05")
    mm(32, 3072, 256, torch.float32, ALGO_AUTO, "scaled_mm split-K")
    mm(600, 256, 1024, torch.float16, ALGO_AUTO, "scaled_mm tcgen05 pair")
    mm(40, 256, 72, torch.float32, ALGO_SIMT, "scaled_mm SIMT")

    X = (rng.standard_normal((4, 1024)) * 3).astype(np.float32)
    tX = torch.from_numpy(X).to(DEV)
    q = torch.empty(4, 1024, dtype=torch.uint8, device=DEV)
    inv = torch.empty(4, device=DEV)
    calls.append(("quantize_rows", lambda s: L.fp8b_quantize_rows(p(tX), F32, 4, 1024, p(q), p(inv), s), ()))
    checks.append(("quantize_rows", lambda: (np.testing.assert_array_equal(u8_np(q), o.fp8_quantize_rows(X)[0]),
                                             assert_bits_equal(to_np(inv), o.fp8_quantize_rows(X)[1], "quantize_rows inv"))))
    e = torch.empty(4096, dtype=torch.uint8, device=DEV)
    calls.append(("encode", lambda s: L.fp8b_encode(p(tX), F32, p(e), 4096, None, s), ()))
    checks.append(("encode", lambda: np.testing.assert_array_equal(u8_np(e), o.encode(X.reshape(-1)))))
    d = torch.empty(4096, dtype=torch.bfloat16, device=DEV)
    calls.append(("dequant", lambda s: L.fp8b_dequant(p(e), p(d), dt_code(torch.bfloat16), 4096, s), ()))
    checks.append(("dequant", lambda: assert_bits_equal(to_np(d), o.decode(o.encode(X.reshape(-1))), "dequant")))
    h = torch.empty(4096, dtype=torch.float16, device=DEV)
    half = torch.full((1,), 0.5, device=DEV)
    calls.append(("dequant_f16", lambda s: L.fp8b_dequant_f16(p(e), p(h), 4096, p(half), s), ()))
    checks.append(("dequant_f16", lambda: np.testing.assert_array_equal(
        h.view(torch.int16).cpu().numpy(), o.fp8_dequantize(o.encode(X.reshape(-1)), 0.5).view(np.int16))))
    sc = torch.empty(2, device=DEV)
    scratch = torch.empty(1, dtype=torch.int32, device=DEV)
    qq = torch.empty(4096, dtype=torch.uint8, device=DEV)
    calls.append(("amax_scale", lambda s: L.fp8b_amax_scale(p(tX), F32, 4096, p(sc), ctypes.c_void_p(sc.data_ptr() + 4), p(scratch), s), ()))
    calls.append(("prescaled encode", lambda s: L.fp8b_encode(p(tX), F32, p(qq), 4096, p(sc), s), ()))
    checks.append(("amax_scale", lambda: (np.testing.assert_array_equal(u8_np(qq), o.fp8_quantize(X.reshape(-1))[0]),
                                          assert_bits_equal(to_np(sc[1:]), o.fp8_quantize(X.reshape(-1))[1], "amax inv"))))
    eb = [torch.empty(1024, dtype=torch.uint8, device=DEV) for _ in range(2)]
    db = [torch.empty(1024, dtype=torch.float16, device=DEV) for _ in range(2)]
    es = make_spans([(tX[i].data_ptr(), eb[i].data_ptr(), 1024) for i in range(2)])
    ds = make_spans([(eb[i].data_ptr(), db[i].data_ptr(), 1024) for i in range(2)])
    calls.append(("encode_batch", lambda s: L.fp8b_encode_batch(es, 2, F32, s), ()))
    calls.append(("dequant_batch", lambda s: L.fp8b_dequant_batch(ds, 2, dt_code(torch.float16), s), ()))
    checks.append(("batches", lambda: [(np.testing.assert_array_equal(u8_np(eb[i]), o.encode(X[i])),
                                        assert_bits_equal(to_np(db[i]), o.decode(o.encode(X[i])), "dequant_batch")) for i in range(2)]))

    K, N = 1024, 64
    W = codes((N, K), rng)
    x1 = one_hot(1, K, np.arange(0, K, 16), rng)
    tW, tx1 = dev_u8(W), dev_u8(x1)
    one = torch.ones(1, device=DEV)
    y = Out(1, N, torch.float32)
    items = (GemvItem * 1)()
    items[0].x, items[0].W, items[0].y, items[0].N = tx1.data_ptr(), tW.data_ptr(), y.ptr, N
    items[0].scale_x, items[0].scale_w, items[0].scale_w_len, items[0].bias = one.data_ptr(), one.data_ptr(), 1, None
    calls.append(("gemv_batch", lambda s: L.fp8b_gemv_batch(items, 1, K, F32, F32, s), ()))
    checks.append(("gemv_batch", lambda: assert_bits_equal(to_np(y.view), oracle(x1, W, [1.0], [1.0], None, None, torch.float32), "gemv_batch")))

    Xd = np.zeros((3, K), np.float32)
    Xd[np.arange(3), [5, 600, 1023]] = [3.5, -0.25, 100.0]
    tXd = torch.from_numpy(Xd).to(DEV)
    nws = L.fp8b_linear_dynamic_workspace_bytes(3, K)
    ws = torch.empty(nws, dtype=torch.uint8, device=DEV)
    yd, invd = Out(3, N, torch.float32), torch.empty(3, device=DEV)
    calls.append(("linear_dynamic", lambda s: L.fp8b_linear_dynamic(p(tXd), F32, p(tW), yd.ptr, F32, 3, N, K, yd.ldc, p(one), 1, None, 0,
                                                                    None, p(invd), p(ws), nws, s), ()))
    checks.append(("linear_dynamic", lambda: assert_bits_equal(
        to_np(yd.view), oracle(o.fp8_quantize_rows(Xd)[0], W, o.fp8_quantize_rows(Xd)[1], [1.0], None, None, torch.float32),
        "linear_dynamic")))

    M2, K2, N2 = 128, 256, 128
    A2, B2 = one_hot(M2, K2, np.arange(0, K2, 16), rng), codes((N2, K2), rng)
    tA2, tB2 = dev_u8(A2), dev_u8(B2)
    dst = torch.zeros(M2, 2 * N2, dtype=torch.float32, device=DEV)
    arr = (ctypes.c_void_p * 1)(dst.data_ptr() + N2 * 4)
    calls.append(("push", lambda s: L.fp8b_scaled_mm_push(p(tA2), p(tB2), arr, 1, F32, M2, N2, K2, 2 * N2, p(one), 1, p(one), 1, None, 0,
                                                          None, s), ()))
    checks.append(("push", lambda: assert_bits_equal(to_np(dst[:, N2:]), oracle(A2, B2, [1.0], [1.0], None, None, torch.float32), "push")))
    torch.cuda.synchronize()

    import fp8_mps_native
    ext = fp8_mps_native._get_lib()                     # import only; no call yet
    a8 = dev_u8(one_hot(8, 512, np.arange(0, 512, 16), rng))
    w8 = dev_u8(codes((64, 512), rng))
    sa8 = torch.full((1,), 0.25, device=DEV)

    g = torch.cuda.CUDAGraph()
    rcs = []
    with torch.cuda.graph(g):
        for what, fn, _ in calls:
            rcs.append((what, fn(s_ptr())))
        y_ext = ext.scaled_mm_patch(a8.view(torch.float8_e4m3fn), w8.view(torch.float8_e4m3fn).t(), sa8, sa8, None, None,
                                    torch.bfloat16)
        q_ext, inv_ext = ext.fp8_quantize_rowwise(tX)
    bad = [(w, rc) for w, rc in rcs if rc != 0]
    assert not bad, f"calls failed inside the capture: {bad}"
    g.replay()
    torch.cuda.synchronize()
    for what, fn in checks:
        fn()
    assert_bits_equal(to_np(y_ext), oracle(a8.cpu().numpy(), w8.cpu().numpy(), [0.25], [0.25], None, None, torch.bfloat16),
                      "scaled_mm_patch")
    np.testing.assert_array_equal(u8_np(q_ext), o.fp8_quantize_rows(X)[0])
    print(f"{len(calls) + 2} first calls captured and replayed")


def _default_scale_problem(rng):
    A, B = one_hot(4, 1024, np.arange(0, 1024, 16), rng), codes((96, 1024), rng)
    ref = oracle(A, B, [1.0], [1.0], None, None, torch.float32)
    return dev_u8(A).view(torch.float8_e4m3fn), dev_u8(B).view(torch.float8_e4m3fn).t(), ref


def default_scale_captured():
    """The first default-scale `_scaled_mm` (scale_a = scale_b = None) of the process is captured; an eager call runs
    before the graph has ever been replayed, then the graph replays."""
    import fp8_mps_native
    ext = fp8_mps_native._get_lib()
    a, b, ref = _default_scale_problem(np.random.default_rng(2))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        y_graph = ext.scaled_mm_patch(a, b)
    y_eager = ext.scaled_mm_patch(a, b)
    torch.cuda.synchronize()
    assert_bits_equal(to_np(y_eager), ref, "eager default-scale call after a captured first one")
    g.replay()
    torch.cuda.synchronize()
    assert_bits_equal(to_np(y_graph), ref, "captured default-scale call")


def default_scale_busy_stream():
    """The first default-scale call is made on stream 1 while a delay kernel keeps it busy; a call on stream 2 follows
    at once and must not read the default scale before it exists."""
    import fp8_mps_native
    ext = fp8_mps_native._get_lib()
    a, b, ref = _default_scale_problem(np.random.default_rng(3))
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(200_000_000)
        y1 = ext.scaled_mm_patch(a, b)
    with torch.cuda.stream(s2):
        y2 = ext.scaled_mm_patch(a, b)
    torch.cuda.synchronize()
    assert_bits_equal(to_np(y2), ref, "default-scale call on the second stream")
    assert_bits_equal(to_np(y1), ref, "default-scale call on the busy stream")


SCENARIOS = {f.__name__: f for f in (first_calls_captured, default_scale_captured, default_scale_busy_stream)}

if __name__ == "__main__":
    torch.cuda.set_device(0)
    SCENARIOS[sys.argv[1]]()
    print("ok")
