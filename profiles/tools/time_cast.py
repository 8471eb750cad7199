#!/usr/bin/env python3
"""One GPU: fp8 -> wide dequant bandwidth of the default launch rule (FP8B_OPT_TUNE_CAST_SHAPE = -1) on FLUX-shaped
tensors, one launch per tensor, in one CUDA graph.  With the profiling library, CAST_SWEEP=11,12,... adds the fp16
launch-shape sweep (CAST_SHAPE 11..19) and checks it bit-equal to the default.
    python profiles/tools/time_cast.py"""
import ctypes, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "fp8-mps-metal_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import torch
from _util import capi
L = capi(); dev = torch.device("cuda", 0)
DOUBLE = [(9216, 3072), (3072, 3072), (12288, 3072), (3072, 12288), (18432, 3072)]
SINGLE = [(21504, 3072), (3072, 15360), (9216, 3072)]
sizes = []
for _ in range(6):
    sizes += [r * c for r, c in DOUBLE] * 2
for _ in range(12):
    sizes += [r * c for r, c in SINGLE]
total = sum(sizes)
q = torch.randint(0, 256, (total,), dtype=torch.uint8, device=dev)
offs = [0]
for s in sizes: offs.append(offs[-1] + s)
print(f"{len(sizes)} tensors, {total/1e9:.2f} G elements, {3*total/1e9:.1f} GB traffic per sweep", flush=True)
SWEEP = [int(x) for x in os.environ.get("CAST_SWEEP", "").split(",") if x]      # profiling library only: modes 11..19
for out_dt, code, esz in ((torch.float16, 1, 2), (torch.bfloat16, 2, 2), (torch.float32, 0, 4)):
    res = {}
    modes = (0,) + (tuple(SWEEP) if out_dt == torch.float16 else ())
    for mode in modes:
        h = torch.empty(total, dtype=out_dt, device=dev)
        L.fp8b_set_option(19, mode if mode else -1)
        def sweep():
            sp = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            for i, n in enumerate(sizes):
                rc = L.fp8b_dequant(ctypes.c_void_p(q.data_ptr() + offs[i]), ctypes.c_void_p(h.data_ptr() + esz * offs[i]), code, n, sp)
                assert rc == 0, rc
        sweep(); torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            sweep()
        for _ in range(2): gr.replay()
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(3):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); gr.replay(); gr.replay(); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / 2)
        res[mode] = ((1 + esz) * total / (best * 1e-3) / 1e9, h)
    L.fp8b_set_option(19, -1)
    same = all(torch.equal(res[0][1].view(torch.uint8), res[m][1].view(torch.uint8)) for m in modes[1:])
    print(f"fp8->{str(out_dt)[6:]:9s}: " + "  ".join(f"mode{m} {res[m][0]:6.0f} GB/s" for m in modes) + f"  bit-equal {same}", flush=True)
    del res
    torch.cuda.empty_cache()
# one big tensor and a small one with a ragged tail
for n in (1 << 30, 50_000_017):
    qq = q[:n]
    line = []
    ref = None
    for mode in (0,) + tuple(SWEEP):
        L.fp8b_set_option(19, mode if mode else -1)
        h = torch.empty(n, dtype=torch.float16, device=dev)
        sp = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        for _ in range(2): L.fp8b_dequant_f16(ctypes.c_void_p(qq.data_ptr()), ctypes.c_void_p(h.data_ptr()), n, None, sp)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5): L.fp8b_dequant_f16(ctypes.c_void_p(qq.data_ptr()), ctypes.c_void_p(h.data_ptr()), n, None, sp)
        e1.record(); torch.cuda.synchronize()
        if ref is None: ref = h
        line.append(f"mode{mode} {3 * n / (e0.elapsed_time(e1) / 5 * 1e-3) / 1e9:6.0f} GB/s eq {bool(torch.equal(ref.view(torch.int16), h.view(torch.int16)))}")
    L.fp8b_set_option(19, -1)
    print(f"n={n}: " + "  ".join(line), flush=True)
