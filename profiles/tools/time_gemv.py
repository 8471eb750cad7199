#!/usr/bin/env python3
"""One GPU: the GEMV configs (C1, C2, C3, the reference's square shape) with every kernel variant
(FP8B_OPT_TUNE_GEMV_IMPL 0 = dispatch rule, 1 = FHFMA, 2 = warp-MMA), HBM-cold rotation in one
CUDA graph, default PDL; plus the static-weights option.   python profiles/tools/time_gemv.py"""
import ctypes, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "fp8-mps-metal_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import torch
from _util import capi
L = capi(); dev = torch.device("cuda", 0)
P = lambda t: ctypes.c_void_p(t.data_ptr())
g = torch.Generator(device=dev).manual_seed(0)
CFG = [("C1", 1, 4096, 4096, 1, 16_789_512, 32), ("C2", 1, 14336, 4096, 2, 58_742_784, 16), ("C3", 4, 4096, 4096, 2, 16_834_560, 32),
       ("SQ", 1, 14336, 14336, 0, 14336 * 14336 + 14336 + 4 * 14336 + 8, 4), ("M8", 8, 4096, 4096, 2, 16_777_216 + 8 * 4096 + 8 * 8192, 32),
       ("M16", 16, 4096, 4096, 2, 16_777_216 + 16 * 4096 + 16 * 8192, 32)]
for name, M, K, N, odt, nbytes, rot in CFG:
    x = torch.randint(0, 120, (M, K), dtype=torch.uint8, device=dev, generator=g)
    Ws = [torch.randint(0, 120, (N, K), dtype=torch.uint8, device=dev, generator=g) for _ in range(rot)]
    out = torch.empty(M, N, dtype=[torch.float32, torch.float16, torch.bfloat16][odt], device=dev)
    bias = torch.randn(N, device=dev).to(torch.bfloat16) if name == "C3" else None
    one = torch.full((1,), 0.01, device=dev)
    def run():
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        for W in Ws:
            rc = L.fp8b_scaled_mm(P(x), P(W), P(out), odt, M, N, K, N, P(one), 1, P(one), 1, P(bias) if bias is not None else None, 2,
                                  None, None, 0, 1, st)
            assert rc == 0, rc
    res = []
    for impl in (0, 1, 2):
        for static in (0, 1):
            L.fp8b_set_option(17, impl if impl else -1); L.fp8b_set_option(1, static)
            try:
                for _ in range(2): run()
                torch.cuda.synchronize()
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    run()
                for _ in range(3): gr.replay()
                torch.cuda.synchronize()
                best = 1e9
                for _ in range(3):
                    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(10): gr.replay()
                    e1.record(); torch.cuda.synchronize()
                    best = min(best, e0.elapsed_time(e1) * 1e3 / (10 * rot))
                res.append(f"impl{impl}{'s' if static else ' '} {best:6.2f} us {nbytes / best / 1e3:5.0f} GB/s")
            except Exception as e:
                res.append(f"impl{impl}{'s' if static else ' '} ERR {str(e)[:40]}")
    L.fp8b_set_option(17, -1); L.fp8b_set_option(1, 0)
    print(f"{name:3s} M{M} K{K} N{N}: " + " | ".join(res), flush=True)
    del Ws
    torch.cuda.empty_cache()
