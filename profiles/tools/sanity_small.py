#!/usr/bin/env python3
"""One small launch of every kernel family -- the short program compute-sanitizer wraps."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "fp8-mps-metal_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import torch
import fp8_mps_native as n
dev = "cuda"
g = torch.Generator(device=dev).manual_seed(0)
x = torch.randn(3, 1000, device=dev, generator=g)
for dt in (torch.float32, torch.float16, torch.bfloat16):
    q = n.fp8_encode(x.to(dt)); n.fp8_encode(x.to(dt).reshape(-1)[1:])
    n.fp8_dequantize_to(q, dt); n.fp8_dequantize(q.reshape(-1)[3:], torch.tensor([0.5]))
q, s = n.fp8_quantize(x); qr, sr = n.fp8_quantize_rowwise(x.to(torch.bfloat16))
def u8(*shape): return torch.randint(0, 256, shape, dtype=torch.uint8, device=dev, generator=g)
one = torch.ones(1, device=dev)
lib = n._get_lib()
for (M, K, N) in [(1, 512, 300), (1, 4096, 64), (3, 64, 40), (4, 1024, 100), (16, 256, 33), (2, 37, 5), (1, 2048, 400)]:
    for impl in ("1", "2"):
        lib.set_option(17, int(impl))            # FP8B_OPT_TUNE_GEMV_IMPL
        lib.fp8_scaled_mm_fused(u8(M, K), u8(N, K), one, one, torch.randn(N, device=dev).bfloat16(), one, torch.bfloat16, 1, None)
lib.set_option(17, -1)
for cfg in ("1", "2", "3", "4", "5"):
    lib.set_option(16, int(cfg))                 # FP8B_OPT_TUNE_GEMM_CFG
    for (M, K, N) in [(300, 336, 520), (129, 64, 257)]:
        lib.fp8_scaled_mm_fused(u8(M, K), u8(N, K), torch.rand(M, device=dev), torch.rand(N, device=dev), None, None, None, 2, None)
lib.set_option(16, -1)
lib.fp8_scaled_mm_fused(u8(2304, 128, ), u8(2500, 128), one, one, None, None, torch.bfloat16, 2, None)     # last-wave split
lib.fp8_scaled_mm_fused(u8(70, 50), u8(33, 50), one, one, None, None, None, 3, None)                      # SIMT
torch.cuda.synchronize()
print("sanity ok, launches:", lib.launch_count())
