#!/usr/bin/env python3
"""Cost of e4m3fn matmul output (out_dtype FP8B_OUT_E4M3FN) against bf16 output and against float32 output + fp8b_encode.

  python profiles/tools/time_fp8_out.py [--iters 200] [--rounds 5]

C4 (4096 x 3072 x 12288) and a FLUX-sized M = 4096, K = 3072, N = 3072 linear, three ways each, alternated round by round:
bf16 out; fused e4m3fn out; float32 out then fp8b_encode (the unfused composition with the same bytes, asserted equal to the
fused bytes in this run).  C2 (M = 1, K = 3072, N = 12288) with bf16 and e4m3fn out, rotating through enough weight
buffers to defeat the 126 MB L2.  CUDA events over `iters` launches; prints the card and its power limit."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from _util import ALGO_AUTO, BF16, F32, capi, p, stream_ptr  # noqa: E402

OUT_E4M3FN = 3                                     # fp8b_dtype FP8B_OUT_E4M3FN (include/fp8_b200.h)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                          # the number is only reported, never needed
        pl = f"unknown ({e})"
    return f"{name}, power limit {pl}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    L = capi()
    st = stream_ptr()
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    sa = torch.full((1,), 0.0123, device=dev)
    print(card())

    def mm(A, B, C, dt, M, N, K):
        rc = L.fp8b_scaled_mm(p(A), p(B), p(C), dt, M, N, K, N, p(sa), 1, p(sb), N, None, 0, None, None, 0, ALGO_AUTO, st)
        assert rc == 0, rc

    def timed(fn, iters):
        for _ in range(3):
            fn(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1000.0 / iters        # us per launch

    for name, (M, K, N) in (("C4", (4096, 3072, 12288)), ("FLUX M=4096 3072x3072", (4096, 3072, 3072))):
        A = torch.randint(0, 0x7E, (M, K), dtype=torch.uint8, device=dev, generator=g)
        B = torch.randint(0, 0x7E, (N, K), dtype=torch.uint8, device=dev, generator=g)
        sb = (torch.rand(N, device=dev, generator=g) + 0.5) * 0.0217
        c16 = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
        c8 = torch.empty(M, N, dtype=torch.uint8, device=dev)
        c32 = torch.empty(M, N, dtype=torch.float32, device=dev)
        c8b = torch.empty(M, N, dtype=torch.uint8, device=dev)

        def two_step(_):
            mm(A, B, c32, F32, M, N, K)
            assert L.fp8b_encode(p(c32), F32, p(c8b), M * N, None, st) == 0
        ways = {"bf16 out": lambda _: mm(A, B, c16, BF16, M, N, K),
                "e4m3fn out (fused)": lambda _: mm(A, B, c8, OUT_E4M3FN, M, N, K),
                "f32 out + fp8b_encode": two_step}
        res = {k: [] for k in ways}
        for _ in range(a.rounds):
            for k, fn in ways.items():
                res[k].append(timed(fn, a.iters))
        assert torch.equal(c8, c8b), f"{name}: fused e4m3fn bytes differ from f32 + fp8b_encode"
        print(f"{name} (M={M} K={K} N={N}, per-row scale_b), us per call over {a.iters} launches x {a.rounds} alternated rounds:")
        for k, v in res.items():
            v = sorted(v)
            print(f"  {k:24s} median {v[len(v) // 2]:9.2f}  min {v[0]:9.2f}  max {v[-1]:9.2f}")
        print(f"  fused e4m3fn bytes == f32 + fp8b_encode bytes: True")
        del A, B, c16, c8, c32, c8b

    M, K, N = 1, 3072, 12288
    nbuf = 8                                          # 8 x 37.7 MB of weights > 126 MB of L2
    Ws = [torch.randint(0, 0x7E, (N, K), dtype=torch.uint8, device=dev, generator=g) for _ in range(nbuf)]
    x = torch.randint(0, 0x7E, (M, K), dtype=torch.uint8, device=dev, generator=g)
    sb = (torch.rand(N, device=dev, generator=g) + 0.5) * 0.0217
    y16 = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
    y8 = torch.empty(M, N, dtype=torch.uint8, device=dev)
    ways = {"bf16 out": lambda i: mm(x, Ws[i % nbuf], y16, BF16, M, N, K),
            "e4m3fn out (fused)": lambda i: mm(x, Ws[i % nbuf], y8, OUT_E4M3FN, M, N, K)}
    res = {k: [] for k in ways}
    for _ in range(a.rounds):
        for k, fn in ways.items():
            res[k].append(timed(fn, a.iters * 5))
    print(f"C2 (M=1 K={K} N={N}, {nbuf} rotating weight buffers), us per call:")
    for k, v in res.items():
        v = sorted(v)
        print(f"  {k:24s} median {v[len(v) // 2]:9.2f}  min {v[0]:9.2f}  max {v[-1]:9.2f}")


if __name__ == "__main__":
    main()
