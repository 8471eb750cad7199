#!/usr/bin/env python3
"""Launch one hot-path kernel a few times -- the short command ncu wraps (profiles/README.md).

    python profiles/run_kernels.py gemm|gemm_stg|gemm_push2|gemv|gemv4|gemv1k4|quant|dequant [reps]
    python profiles/run_kernels.py mm:M,K,N[:cfg] [reps]        # any fp8b_scaled_mm shape (AUTO dispatch), optional tile cfg
"""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "fp8-mps-metal_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import torch  # noqa: E402

from _util import capi, dt_code  # noqa: E402


def main():
    which = sys.argv[1]
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    L = capi()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    one = torch.full((1,), 0.01, device=dev)

    def rand_u8(*shape):
        b = torch.randint(0, 256, shape, dtype=torch.uint8, device=dev, generator=g)
        return torch.where((b & 0x7F) == 0x7F, torch.full_like(b, 0x3C), b)

    if which == "gemm_push2":              # the fused GEMM + push kernel, two destinations (both local on one GPU)
        M, K, N = 4096, 3072, 6144
        A = rand_u8(M, K)
        Bs = [rand_u8(N, K) for _ in range(4)]
        C1 = torch.empty(M, 2 * N, dtype=torch.bfloat16, device=dev)
        C2 = torch.empty(M, 2 * N, dtype=torch.bfloat16, device=dev)
        arr = (ctypes.c_void_p * 2)(C1.data_ptr(), C2.data_ptr())
        for i in range(reps):
            rc = L.fp8b_scaled_mm_push(P(A), P(Bs[i % 4]), arr, 2, dt_code(torch.bfloat16), M, N, K, 2 * N, P(one), 1, P(one), 1,
                                       None, 0, None, st)
            assert rc == 0, rc
    elif which in ("gemm", "gemm_stg", "gemv", "gemv4", "gemv1k4"):
        M, K, N, algo = {"gemm": (4096, 3072, 12288, 2), "gemm_stg": (4096, 3072, 12288, 2), "gemv": (1, 14336, 4096, 1),
                         "gemv4": (4, 4096, 4096, 1), "gemv1k4": (1, 4096, 4096, 1)}[which]
        if which == "gemm_stg":
            L.fp8b_set_option(20, 1)           # the round-1 st.global epilogue, for comparison
        A = rand_u8(M, K)
        Bs = [rand_u8(N, K) for _ in range(4)]
        C = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
        for i in range(reps):
            rc = L.fp8b_scaled_mm(P(A), P(Bs[i % 4]), P(C), dt_code(torch.bfloat16), M, N, K, N, P(one), 1, P(one), 1,
                                  None, 0, None, None, 0, algo, st)
            assert rc == 0, rc
    elif which.startswith("mm:"):
        parts = which.split(":")
        M, K, N = (int(v) for v in parts[1].split(","))
        if len(parts) > 2:
            L.fp8b_set_option(16, int(parts[2]))
        A = rand_u8(M, K)
        Bs = [rand_u8(N, K) for _ in range(4)]
        C = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
        for i in range(reps):
            rc = L.fp8b_scaled_mm(P(A), P(Bs[i % 4]), P(C), dt_code(torch.bfloat16), M, N, K, N, P(one), 1, P(one), 1,
                                  None, 0, None, None, 0, 0, st)
            assert rc == 0, rc
    elif which in ("quant", "dequant"):
        n = 21504 * 3072 * (8 if os.environ.get("FP8B_PROFILE_BIG") else 1)      # the largest FLUX tensor of C5 (198 MB of traffic)
        x = (torch.randn(n, generator=g, device=dev) * 0.02).to(torch.bfloat16)
        q = torch.empty(n, dtype=torch.uint8, device=dev)
        h = torch.empty(n, dtype=torch.float16, device=dev)
        for _ in range(reps):
            if which == "quant":
                assert L.fp8b_encode(P(x), 2, P(q), n, None, st) == 0
            else:
                assert L.fp8b_dequant_f16(P(q), P(h), n, None, st) == 0
    torch.cuda.synchronize()
    print("ok", which, reps)


if __name__ == "__main__":
    main()
