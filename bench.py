#!/usr/bin/env python3
"""
bench.py -- measures the FP8 hot path on B200 and prints ONE JSON line (rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-sub] [--no-cpu] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline at every N (BASELINE.json `metric` names "_scaled_mm TFLOPS" first; configs[3], "C4", is the config that
shards): the FLUX.1-dev-shaped DiT linear  `_scaled_mm`  M=4096 K=3072 N=12288, FP8 e4m3fn operands, per-tensor
scales, bf16 out -- 309 237 645 312 flops per call (SURVEY 8d).
  * a STEP is 4 calls over a rotation of 4 distinct (A, W, C) sets (4 x 151 MB, larger than the 126 MB L2).
  * N = 1: the tcgen05 kernel through the C ABI, the step captured in a CUDA graph.
    N > 1: STRONG scaling of the same problem: W is column-sharded over the ranks (ShardedScaledMM, mode "push"):
    ONE kernel per rank computes its (M, N/w) block on the tensor cores and pushes every finished box with TMA stores
    into the row-major (M, N) result of EVERY rank over NVLink; one symmetric-memory barrier closes the call.  A call
    is complete when every rank holds the full result.  Timed like the N = 1 step, as CUDA graphs (two, replayed in
    turn: consecutive calls alternate between the two result buffers); the same calls issued one by one from Python
    are reported beside it (`sharded.plans.*.eager_us_per_call`).
  * value   = flops of all calls / time, CUDA events on the launching stream after W (>= 3) warm-up steps, barrier +
              synchronize on both sides, MAX over ranks.  Inputs resident in HBM.
  * e2e     = the same call through the public API with HOST (pinned) buffers inside the timed region:
              N = 1: fp8_mps_patch.install(); torch._scaled_mm(...) with A and W copied host->device and C copied
              device->host every step;  N > 1: ShardedScaledMM with A and this rank's W shard copied in and this
              rank's 1/N row slab of the assembled result copied out (the ranks' slabs make up exactly one C).
  * roofline = the GEMM kernel's flops / its average duration in the timed region against 2 x the measured bf16
              cuBLAS rate of MEASURED_PEAKS.json (dense-FP8 proxy); at N > 1 also the NVLink floor of the exchange.
  * sharded (N > 1): every exchange plan timed, each with `parity` = bit-equal to the un-sharded GEMM on every rank
              and <= 3e-3 rel-RMSE against the CPU oracle on a 64-row slab.
  * cpu_baseline = the oracle port of the reference's CPU path (LUT dequantise + fp32 matmul) on the host cores.
`sub` (N = 1) carries the other BASELINE configs with their own rooflines: C2 (M=1 K=14336 N=4096 GEMV, HBM-bound),
C1, C3, the reference's own square benchmark shape (M=1 K=N=14336, test_fp8_metal.py:232-236), C5 (FLUX-sized cast
sweeps) and the un-patched torch._scaled_mm (cuBLASLt FP8) time on C4 as a library yardstick.

--impl reference: the reference's CPU implementation of the same workload (oracle port, all host threads), same
`config`, same JSON shape with "impl": "reference".

--dump-outputs DIR (N = 1): after the timed steps, the results of the last step -- the C of each of the SETS calls --
are written as DIR/c4_out_set<i>.npy, float32, restricted to a fixed set of DUMP_ROWS rows (every column of those
rows; see dump_outputs).  The inputs come from fixed seeds, so two builds run with the same arguments can be
compared output for output.
"""

from __future__ import annotations

import argparse
import contextlib
import ctypes
import json
import os
import statistics
import sys
import threading
import time

sys.dont_write_bytecode = True             # the benchmark writes nothing into the tree it runs from (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "fp8-mps-metal_b200")
for _p in (PKG, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "FP8 _scaled_mm TFLOPS & M=1 GEMV/cast HBM GB/s as % roofline vs CPU ref"

C2 = dict(M=1, K=14336, N=4096)
C2_BYTES = 58_742_784                      # SURVEY 8d
C1 = dict(M=1, K=4096, N=4096)
C1_BYTES = 16_789_512
C3 = dict(M=4, K=4096, N=4096)
C3_BYTES = 16_834_560
C4 = dict(M=4096, K=3072, N=12288)
C4_FLOPS = 309_237_645_312
C4_OUT_BYTES = 100_663_296
SQ = dict(M=1, K=14336, N=14336)           # the reference's own benchmark shape (test_fp8_metal.py:232-236; README.md:80: 2.38 ms)
SQ_BYTES = 14336 * 14336 + 14336 + 2 * 14336 + 8
ROTATION = 16
PASSES = 8
SETS = 4                                   # C4 rotation: 4 x (12.6 + 37.7 + 100.7) MB > 126 MB L2
DUMP_ROWS = 128                            # --dump-outputs: 128 of 4096 rows of each C, 4 x 6.3 MB of float32
NVLINK_GBS = 770.0                         # peer-copy rate per direction per GPU quoted by B200_PROFILING.md
NVLINK_MEASURED_GBS = 690.0                # what a peer accepts on these boxes with both directions busy: copy engine 708,
                                           # st.global / cp.async.bulk from 148 SMs 687 GB/s (profiles/r2_peer_bw_w2.log)

FALLBACK_HBM_GBS = 6650.0                  # B200_PROFILING.md fallback
FALLBACK_BF16_TFLOPS = 1590.0

WORKLOAD = ("C4 _scaled_mm FLUX.1-dev DiT linear M=4096 K=3072 N=12288, FP8 e4m3fn, per-tensor scales, bf16 out "
            "(BASELINE.json configs[3]); N-sharded over the GPUs when N > 1, full row-major result on every rank")


def config_for(n_gpus):
    """The `config` object -- identical in the `ours` and `reference` arms."""
    return {"workload": WORKLOAD,
            "step": f"{SETS} _scaled_mm calls over a rotation of {SETS} distinct (A, W, C) sets",
            "l2": f"inputs larger than L2: rotation of {SETS} sets x 151 MB",
            "flops_per_call": C4_FLOPS,
            "parallelism": "single-gpu" if n_gpus == 1 else f"W column-sharded x{n_gpus}, strong scaling",
            "arith": "e4m3 operands, exact products, fp32 accumulation"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops"]),
                    bf16_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm=FALLBACK_HBM_GBS, bf16=FALLBACK_BF16_TFLOPS, bf16_sustained=1400.0, source="fallback")


def profile_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the committed ncu capture
    profiles/r2_<name>_raw.csv (else r1_), one `ncu --set full` capture of the same kernel and shape, or None."""
    import csv
    for rnd in ("r2", "r1"):
        path = os.path.join(ROOT, "profiles", f"{rnd}_{name}_raw.csv")
        if os.path.exists(path):
            break
    else:
        return None
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    found = 0
    for row in csv.reader(open(path)):
        if len(row) == 3 and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(row[1].replace(",", "")) * mult.get(row[2], 1.0)
            found += 1
    return int(tot) if found == 2 else None


# --------------------------------------------------------------------------- clocks

class ClockSampler:
    """Polls NVML for SM clock and throttle reasons while a timed region runs."""

    def __init__(self, index: int):
        self.samples = []
        self._stop = threading.Event()
        self._thread = None
        self._h = None
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                mhz = int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                self.samples.append((time.perf_counter(), mhz, r))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self._h is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1.0)

    def summary(self, t0=None, t1=None):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        sel = [s for s in self.samples if (t0 is None or s[0] >= t0) and (t1 is None or s[0] <= t1)] or self.samples
        names = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
                 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
                 0x100: "display_clock_setting"}
        bits = 0
        for s in sel:
            bits |= s[2]
        reasons = [n for b, n in names.items() if bits & b]
        return {"sm_mhz": int(statistics.median(s[1] for s in sel)), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(sel)}


# --------------------------------------------------------------------------- helpers

def _capi():
    from _util import capi
    return capi()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _mm(L, torch, A, B, C, odt_code, sa, sb, bias=None, bias_dt=0, algo=0):
    M, K = A.shape
    N = B.shape[0]
    rc = L.fp8b_scaled_mm(_ptr(A), _ptr(B), _ptr(C), odt_code, M, N, K, C.stride(0), _ptr(sa), sa.numel(),
                          _ptr(sb), sb.numel(), _ptr(bias), bias_dt, None, None, 0, algo,
                          ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    if rc != 0:
        raise RuntimeError(f"fp8b_scaled_mm failed: {L.fp8b_status_string(rc).decode()} (cuda {L.fp8b_last_cuda_error()})")


def _rand_fp8(torch, shape, gen, dev):
    """randn -> reference-codec FP8 bytes, on the device (fp8b_encode), plus amax/448 scale."""
    import fp8_mps_native
    x = torch.randn(shape, generator=gen, device=dev)
    q, inv = fp8_mps_native.fp8_quantize(x)
    return q, inv


def time_graph(torch, step_fn, steps, warmup, dist=None):
    """Capture step_fn once, replay: returns (ms_total, launches_per_step, t0, t1 wall-clock marks)."""
    L = _capi()
    step_fn()                                     # eager warm-up: lazy attribute setup happens outside capture
    torch.cuda.synchronize()
    n0 = L.fp8b_launch_count()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step_fn()
    launches = L.fp8b_launch_count() - n0
    for _ in range(max(warmup, 3)):
        g.replay()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
        torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    if dist is not None:
        dist.barrier()
    return e0.elapsed_time(e1), launches, t0, t1


def dump_outputs(torch, out_dir, outputs):
    """{name: (M, N) device tensor} -> out_dir/<name>.npy as float32 (exact for bf16), DUMP_ROWS full rows of each:
    one row from every block of M / DUMP_ROWS rows, at an offset that walks through the block, so that every
    row tile of the kernel and many row positions inside a tile are covered."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, c in outputs.items():
        block = c.shape[0] // DUMP_ROWS
        j = torch.arange(DUMP_ROWS, device=c.device)
        rows = j * block + (5 * j) % block
        np.save(os.path.join(out_dir, name + ".npy"), c[rows].float().cpu().numpy())


def max_over_ranks(torch, dist, ms):
    if dist is None:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# --------------------------------------------------------------------------- CPU baseline (oracle port)

def _use_all_host_cores():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use all the host cores it may."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        import torch
        torch.set_num_threads(n)
    except Exception:
        pass
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=n)
    except Exception:
        pass
    return n


def _cpu_c4_inputs():
    _use_all_host_cores()
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import fp8_oracle as o
    rng = np.random.default_rng(2)
    A = o.encode(rng.standard_normal((C4["M"], C4["K"])).astype(np.float32) * 50)
    W = o.encode(rng.standard_normal((C4["N"], C4["K"])).astype(np.float32) * 50)
    return A, W, np.array([0.01], np.float32), np.array([0.01], np.float32)


def _cpu_c4_candidates(A, W, sa, sb):
    """The reference's CPU path for C4 on the host cores, three statements of it, the fastest is reported:
    (a) torch CPU FP8 cast + fp32 matmul (the reference's own fallback, test_fp8_metal.py:257-271, minus the MPS hop),
    (b) numpy LUT dequantise + fp32 BLAS matmul, both full size; (c) the plain-C restatement of the shader loop
    (fp8_matmul.metal:99-147) on all cores, on a 256-row slab (it is far slower).  Returns {name: (fn, flops, what, cores)}."""
    import c_oracle
    import fp8_oracle as o
    rows = 256
    import torch
    return {"torch_cpu": (lambda: o.scaled_mm_torch_cpu(A, W, sa, sb, out_dtype="bf16"), float(C4_FLOPS),
                          "full-size C4 call (torch CPU FP8 cast of A and W + fp32 matmul + epilogue)", torch.get_num_threads()),
            "numpy_blas": (lambda: o.scaled_mm(A, W, sa, sb, out_dtype="bf16", accum="f32"), float(C4_FLOPS),
                           "full-size C4 call (LUT dequantise of A and W + sgemm + epilogue)", os.cpu_count() or 1),
            "c_threads": (lambda: c_oracle.scaled_mm(A[:rows], W, sa, sb), float(C4_FLOPS) * rows / C4["M"],
                          f"{rows}-row slab of C4 (1/{C4['M'] // rows} of the call), shader-loop port on pthreads",
                          c_oracle.num_threads())}


def cpu_c4_baseline(seconds_budget=20.0):
    A, W, sa, sb = _cpu_c4_inputs()
    res = {}
    for name, (fn, flops, what, cores) in _cpu_c4_candidates(A, W, sa, sb).items():
        t0 = time.perf_counter(); fn(); first = time.perf_counter() - t0          # warm-up (page faults, thread pool)
        best, n = first, 0
        t_start = time.perf_counter()
        while n < 3 and time.perf_counter() - t_start < seconds_budget / 2:
            t0 = time.perf_counter(); fn(); best = min(best, time.perf_counter() - t0); n += 1
        res[name] = (flops / best / 1e12, best, n, what, cores)
    pick = max(res, key=lambda k: res[k][0])
    tf, best, n, what, cores = res[pick]
    return {"value": round(tf, 4), "unit": "TFLOP/s", "cores": cores, "kind": "port",
            "sample": f"{max(n, 1)} x {what}, best; {pick}", "s_per_sample": round(best, 4),
            "alt_tflops": {k: round(v[0], 4) for k, v in res.items()}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    A, W, sa, sb = _cpu_c4_inputs()
    cands = _cpu_c4_candidates(A, W, sa, sb)
    probe = {}
    for name, (fn, flops, what, cores) in cands.items():
        fn()
        t0 = time.perf_counter(); fn(); probe[name] = flops / (time.perf_counter() - t0)
    pick = max(probe, key=probe.get)
    fn, flops, what, cores = cands[pick]
    t_call = flops / probe[pick]
    # bounded sample: one call per step; the whole run stays within a few minutes
    calls_per_step = SETS if t_call * SETS * (args.steps + max(args.warmup, 3)) < 150.0 else 1
    for _ in range(max(args.warmup, 3)):
        for _ in range(calls_per_step):
            fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for _ in range(calls_per_step):
            fn()
    dt = time.perf_counter() - t0
    value = flops * calls_per_step * args.steps / dt / 1e12
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "TFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(dt / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_for(args.gpus),
        "cpu_baseline": {"value": round(value, 4), "unit": "TFLOP/s", "cores": cores, "kind": "port",
                         "sample": f"{calls_per_step} x {what} per step; {pick}",
                         "calls_per_step": calls_per_step, "gpu_arm_calls_per_step": SETS},
        "e2e": {"value": round(value, 4), "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# --------------------------------------------------------------------------- sub-benchmarks (rank-local)

def bench_gemv_cfg(torch, L, cfg, nbytes, odt, with_bias, gen, dev, peaks, steps, warmup, rotation=ROTATION):
    from _util import dt_code
    M, K, N = cfg["M"], cfg["K"], cfg["N"]
    xs, inv_x = _rand_fp8(torch, (M, K), gen, dev)
    Ws = []
    for _ in range(rotation):
        w, inv_w = _rand_fp8(torch, (N, K), gen, dev)
        Ws.append(w)
    bias = torch.randn(N, generator=gen, device=dev).to(odt) if with_bias else None
    out = torch.empty(M, N, dtype=odt, device=dev)
    oc = dt_code(odt)

    def step():
        for w in Ws:
            _mm(L, torch, xs, w, out, oc, inv_x, inv_w, bias, dt_code(odt) if with_bias else 0)

    ms, launches, _, _ = time_graph(torch, step, steps, warmup)
    per_call_us = ms * 1e3 / (steps * rotation)
    gbs = nbytes / (per_call_us * 1e-6) / 1e9
    # L2-hot variant: one buffer only
    def step_hot():
        for _ in range(rotation):
            _mm(L, torch, xs, Ws[0], out, oc, inv_x, inv_w, bias, dt_code(odt) if with_bias else 0)
    ms_h, _, _, _ = time_graph(torch, step_hot, steps, warmup)
    hot_us = ms_h * 1e3 / (steps * rotation)
    # opt-in variant: weights declared static -> consecutive calls overlap via programmatic dependent launch
    L.fp8b_set_option(1, 1)
    try:
        ms_s, _, _, _ = time_graph(torch, step, steps, warmup)
    finally:
        L.fp8b_set_option(1, 0)
    static_us = ms_s * 1e3 / (steps * rotation)
    return {"us_per_call": round(per_call_us, 3), "value": round(gbs, 1), "unit": "GB/s",
            "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peaks["hbm"], "unit": "GB/s",
                         "frac": round(gbs / peaks["hbm"], 4), "frac_of_nominal_8000": round(gbs / 8000.0, 4),
                         "traffic": None, "peak_source": peaks["source"]},
            "l2_hot_us_per_call": round(hot_us, 3), "l2_hot_gbs": round(nbytes / (hot_us * 1e-6) / 1e9, 1),
            "static_weights_pdl": {"us_per_call": round(static_us, 3), "gbs": round(nbytes / (static_us * 1e-6) / 1e9, 1),
                                   "note": "FP8B_OPT_STATIC_WEIGHTS=1 (opt-in): B streamed before the predecessor kernel completes"},
            "rotation_buffers": rotation, "launches_per_step": launches}


def bench_gemm_c4(torch, L, gen, dev, peaks, steps, warmup, n_shard=None, algo=2, sets=4):
    from _util import dt_code
    M, K, N = C4["M"], C4["K"], C4["N"]
    Nl = n_shard or N
    bufs = []
    for _ in range(sets):                          # rotation: 4 x (12.6 + 37.7) MB of inputs > 126 MB L2
        a, inv_a = _rand_fp8(torch, (M, K), gen, dev)
        w, inv_w = _rand_fp8(torch, (Nl, K), gen, dev)
        out = torch.empty(M, Nl, dtype=torch.bfloat16, device=dev)
        bufs.append((a, inv_a, w, inv_w, out))

    def step():
        for a, inv_a, w, inv_w, out in bufs:
            _mm(L, torch, a, w, out, dt_code(torch.bfloat16), inv_a, inv_w, algo=algo)

    ms, launches, _, _ = time_graph(torch, step, steps, warmup)
    us = ms * 1e3 / (steps * sets)
    flops = 2.0 * M * K * Nl
    tf = flops / (us * 1e-6) / 1e12
    fp8_peak_meas = 2 * peaks["bf16"]
    return {"us_per_call": round(us, 2), "value": round(tf, 1), "unit": "TFLOP/s",
            "roofline": {"bound": "tensor", "achieved": round(tf, 1), "peak": round(fp8_peak_meas, 1), "unit": "TFLOP/s",
                         "frac": round(tf / fp8_peak_meas, 4), "frac_of_nominal_4500": round(tf / 4500.0, 4),
                         "traffic": None, "peak_source": peaks["source"] + " (2 x bf16 cuBLAS burst as dense-FP8 proxy)"},
            "l2": f"inputs larger than L2: rotation of {sets} (A,B,C) sets, {sets} x 151 MB", "launches_per_step": launches,
            "shape": [M, K, Nl]}, bufs[0]


FLUX_DOUBLE = [(9216, 3072), (3072, 3072), (12288, 3072), (3072, 12288), (18432, 3072)]   # x2 streams x19 blocks
FLUX_SINGLE = [(21504, 3072), (3072, 15360), (9216, 3072)]                               # x38 blocks


def flux_tensor_sizes():
    sizes = []
    for _ in range(19):
        for _ in range(2):
            sizes += [r * c for r, c in FLUX_DOUBLE]
    for _ in range(38):
        sizes += [r * c for r, c in FLUX_SINGLE]
    return sizes


def bench_casts_c5(torch, L, gen, dev, peaks, steps, warmup):
    """bf16 -> fp8 and fp8 -> fp16 over the whole FLUX-sized weight set, one launch per tensor."""
    sizes = flux_tensor_sizes()
    total = sum(sizes)
    assert total == 11_834_228_736
    src = torch.empty(total, dtype=torch.bfloat16, device=dev)
    chunk = 1 << 28
    for off in range(0, total, chunk):
        n = min(chunk, total - off)
        src[off:off + n] = (torch.randn(n, generator=gen, device=dev) * 0.02).to(torch.bfloat16)
    q = torch.empty(total, dtype=torch.uint8, device=dev)
    h = torch.empty(total, dtype=torch.float16, device=dev)
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    side = [torch.cuda.Stream(device=dev) for _ in range(4)]

    def sweep(call, n_streams):
        """One launch per tensor.  n_streams > 1: independent tensors are issued round-robin on forked
        streams (joined back before the step ends), so the drain of one launch overlaps the ramp of the next."""
        cur = torch.cuda.current_stream()
        if n_streams <= 1:
            sp = ctypes.c_void_p(cur.cuda_stream)
            for i, n in enumerate(sizes):
                call(i, n, sp)
            return
        fork = torch.cuda.Event()
        fork.record(cur)
        for s_ in side[:n_streams]:
            s_.wait_event(fork)
        for i, n in enumerate(sizes):
            call(i, n, ctypes.c_void_p(side[i % n_streams].cuda_stream))
        for s_ in side[:n_streams]:
            j = torch.cuda.Event()
            j.record(s_)
            cur.wait_event(j)

    def quant_one(i, n, sp):
        rc = L.fp8b_encode(ctypes.c_void_p(src.data_ptr() + 2 * offs[i]), 2, ctypes.c_void_p(q.data_ptr() + offs[i]), n, None, sp)
        assert rc == 0

    def dequant_one(i, n, sp):
        rc = L.fp8b_dequant_f16(ctypes.c_void_p(q.data_ptr() + offs[i]), ctypes.c_void_p(h.data_ptr() + 2 * offs[i]), n, None, sp)
        assert rc == 0

    class Span(ctypes.Structure):                      # fp8b_span, include/fp8_b200.h
        _fields_ = [("inp", ctypes.c_void_p), ("out", ctypes.c_void_p), ("n", ctypes.c_size_t)]

    q_spans = (Span * len(sizes))()
    d_spans = (Span * len(sizes))()
    for i, n in enumerate(sizes):
        q_spans[i].inp, q_spans[i].out, q_spans[i].n = src.data_ptr() + 2 * offs[i], q.data_ptr() + offs[i], n
        d_spans[i].inp, d_spans[i].out, d_spans[i].n = q.data_ptr() + offs[i], h.data_ptr() + 2 * offs[i], n
    L.fp8b_encode_batch.restype = ctypes.c_int
    L.fp8b_encode_batch.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    L.fp8b_dequant_batch.restype = ctypes.c_int
    L.fp8b_dequant_batch.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]

    def quant_batched():
        rc = L.fp8b_encode_batch(q_spans, len(sizes), 2, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0

    def dequant_batched():
        rc = L.fp8b_dequant_batch(d_spans, len(sizes), 1, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0

    out = {}
    k = max(3, min(steps, 5))
    for name, one, batched in (("quantize_bf16_to_fp8", quant_one, quant_batched),
                               ("dequant_fp8_to_fp16", dequant_one, dequant_batched)):
        res = {}
        ms_b, launches_b, _, _ = time_graph(torch, batched, k, max(warmup, 3))
        ms_b /= k
        gbs_b = 3.0 * total / (ms_b * 1e-3) / 1e9
        for ns in (1, 4):
            ms, launches, _, _ = time_graph(torch, lambda: sweep(one, ns), k, max(warmup, 3))
            ms_sweep = ms / k
            res[ns] = (ms_sweep, 3.0 * total / (ms_sweep * 1e-3) / 1e9, launches)
        ms_sweep, gbs, launches = res[1]
        out[name] = {"ms_per_sweep": round(ms_sweep, 3), "value": round(gbs, 1), "unit": "GB/s", "elements": total,
                     "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peaks["hbm"], "unit": "GB/s",
                                  "frac": round(gbs / peaks["hbm"], 4), "frac_of_nominal_8000": round(gbs / 8000.0, 4),
                                  "traffic": profile_traffic("quant" if name.startswith("quantize") else "dequant"),
                                  "traffic_note": "ncu capture of ONE launch on the largest tensor of the set (21504x3072, "
                                                  "198 180 864 algorithmic bytes); below that because part of the output "
                                                  "is still dirty in L2 when the 3-launch capture ends",
                                  "peak_source": peaks["source"]},
                     "launches_per_sweep": launches, "l2": "35.5 GB working set per sweep >> L2",
                     "four_streams": {"ms_per_sweep": round(res[4][0], 3), "value": round(res[4][1], 1), "unit": "GB/s",
                                      "frac": round(res[4][1] / peaks["hbm"], 4),
                                      "note": "same per-tensor launches issued round-robin on 4 forked streams"},
                     "batched_api": {"ms_per_sweep": round(ms_b, 3), "value": round(gbs_b, 1), "unit": "GB/s",
                                     "frac": round(gbs_b / peaks["hbm"], 4), "launches_per_sweep": launches_b,
                                     "note": "fp8b_encode_batch / fp8b_dequant_batch: all 304 tensors as one tile list, "
                                             "one persistent launch (span table in the kernel parameters)"}}
    # spot parity on the last tensor (bit-exact vs the C oracle on a strided sample)
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import numpy as np
        import c_oracle
        idx = torch.arange(0, total, 104729, device=dev)
        ref = c_oracle.encode_bf16_bits(src[idx].cpu().view(torch.int16).numpy().view(np.uint16))
        out["parity_sample_bit_exact"] = bool((q[idx].cpu().numpy() == ref).all())
    except Exception as e:  # pragma: no cover
        out["parity_sample_bit_exact"] = f"not checked: {e}"
    del src, q, h
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------- C2 GEMV block (a `sub` entry since round 2)

def bench_c2(torch, L, gen, dev, peaks, steps, warmup):
    """BASELINE configs[1]: M=1 K=14336 N=4096 bf16 out.  128 calls per step = 8 passes over 16 distinct weight
    matrices (940 MB >> L2) in one CUDA graph; plus the static-weights PDL option, four forked streams, the
    four-per-launch batched entry point, and the patched torch._scaled_mm with resident weights (host x in, y out)."""
    from _util import GemvItem, dt_code
    import fp8_mps_patch
    M, K, N = C2["M"], C2["K"], C2["N"]
    x, inv_x = _rand_fp8(torch, (M, K), gen, dev)
    Ws, inv_ws = [], []
    for _ in range(ROTATION):
        w, inv_w = _rand_fp8(torch, (N, K), gen, dev)
        Ws.append(w)
        inv_ws.append(inv_w)
    out = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
    bf16 = dt_code(torch.bfloat16)
    calls = ROTATION * PASSES

    def step():
        for _ in range(PASSES):
            for w, s in zip(Ws, inv_ws):
                _mm(L, torch, x, w, out, bf16, inv_x, s)

    def gbs(ms):
        return C2_BYTES * calls / (ms / steps * 1e-3) / 1e9

    ms, launches, _, _ = time_graph(torch, step, steps, warmup)
    L.fp8b_set_option(1, 1)
    try:
        ms_static, _, _, _ = time_graph(torch, step, steps, warmup)
    finally:
        L.fp8b_set_option(1, 0)
    side = [torch.cuda.Stream(device=dev) for _ in range(4)]
    outs4 = [torch.empty(M, N, dtype=torch.bfloat16, device=dev) for _ in range(4)]

    def step_streams():
        cur = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(cur)
        for s_ in side:
            s_.wait_event(fork)
        i = 0
        for _ in range(PASSES):
            for w, sc in zip(Ws, inv_ws):
                with torch.cuda.stream(side[i % 4]):
                    _mm(L, torch, x, w, outs4[i % 4], bf16, inv_x, sc)
                i += 1
        for s_ in side:
            j = torch.cuda.Event()
            j.record(s_)
            cur.wait_event(j)

    ms_streams, _, _, _ = time_graph(torch, step_streams, steps, warmup)
    groups = []
    for g0 in range(0, ROTATION, 4):
        arr = (GemvItem * 4)()
        for j in range(4):
            w, sc = Ws[g0 + j], inv_ws[g0 + j]
            arr[j].x, arr[j].W, arr[j].y, arr[j].N = x.data_ptr(), w.data_ptr(), outs4[j].data_ptr(), N
            arr[j].scale_x, arr[j].scale_w, arr[j].scale_w_len, arr[j].bias = inv_x.data_ptr(), sc.data_ptr(), 1, None
        groups.append(arr)

    def step_batched():
        sp = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        for _ in range(PASSES):
            for arr in groups:
                rc = L.fp8b_gemv_batch(arr, 4, K, bf16, 0, sp)
                assert rc == 0, rc

    ms_b, launches_b, _, _ = time_graph(torch, step_batched, steps, warmup)
    us = ms / steps * 1e3 / calls
    res = {"us_per_call": round(us, 3), "value": round(gbs(ms), 1), "unit": "GB/s",
           "roofline": {"bound": "hbm", "achieved": round(gbs(ms), 1), "peak": peaks["hbm"], "unit": "GB/s",
                        "frac": round(gbs(ms) / peaks["hbm"], 4), "frac_of_nominal_8000": round(gbs(ms) / 8000.0, 4),
                        "traffic": profile_traffic("gemv"), "peak_source": peaks["source"], "algorithmic_bytes": C2_BYTES},
           "step": f"{calls} GEMV calls = {PASSES} passes over {ROTATION} distinct weight matrices (940 MB), one CUDA graph",
           "launches_per_step": int(launches),
           "static_weights_pdl": {"us_per_call": round(ms_static / steps * 1e3 / calls, 3), "value": round(gbs(ms_static), 1),
                                  "note": "opt-in FP8B_OPT_STATIC_WEIGHTS=1"},
           "four_streams": {"us_per_call": round(ms_streams / steps * 1e3 / calls, 3), "value": round(gbs(ms_streams), 1),
                            "frac": round(gbs(ms_streams) / peaks["hbm"], 4),
                            "note": "the same 128 independent calls round-robin on 4 forked streams"},
           "batched_gemv": {"us_per_gemv": round(ms_b / steps * 1e3 / calls, 3), "value": round(gbs(ms_b), 1),
                            "frac": round(gbs(ms_b) / peaks["hbm"], 4), "launches_per_step": int(launches_b),
                            "note": "fp8b_gemv_batch: four independent C2 GEMVs per launch"}}
    # the deployment shape of the plug-in: weights resident, x from / y to pinned host memory, patched torch._scaled_mm
    with contextlib.redirect_stdout(sys.stderr):
        fp8_mps_patch.install()
    try:
        hx = x.cpu().pin_memory()
        hout = torch.empty(M, N, dtype=torch.bfloat16).pin_memory()
        dx = torch.empty_like(x)
        w8s = [w.view(torch.float8_e4m3fn).t() for w in Ws]

        def e2e_resident(i):
            dx.copy_(hx, non_blocking=True)
            y = torch._scaled_mm(dx.view(torch.float8_e4m3fn), w8s[i % ROTATION], inv_x, inv_ws[i % ROTATION], None, None,
                                 torch.bfloat16)
            hout.copy_(y, non_blocking=True)

        for i in range(16):
            e2e_resident(i)
        torch.cuda.synchronize()
        r0 = torch.cuda.Event(enable_timing=True)
        r1 = torch.cuda.Event(enable_timing=True)
        n_it = 256
        t_h0 = time.perf_counter()
        r0.record()
        for i in range(n_it):
            e2e_resident(i)
        r1.record()
        t_h1 = time.perf_counter()
        torch.cuda.synchronize()
        res_ms = r0.elapsed_time(r1) / n_it
        res["e2e_resident_weights"] = {
            "value": round(C2_BYTES / (res_ms * 1e-3) / 1e9, 1), "unit": "GB/s", "us_per_step": round(res_ms * 1e3, 2),
            "host_us_per_step": round((t_h1 - t_h0) / n_it * 1e6, 2),
            "frac_of_device_value": round(C2_BYTES / (res_ms * 1e-3) / 1e9 / gbs(ms), 3),
            "h2d_bytes_per_step": int(hx.numel()), "d2h_bytes_per_step": int(hout.numel() * 2),
            "note": "patched torch._scaled_mm; weights on the GPU (16-matrix rotation, HBM-cold); x copied in and y copied "
                    "out of pinned host memory every step"}
    finally:
        fp8_mps_patch.uninstall()
    return res


def bench_library_yardstick(torch, bufs, steps, warmup):
    """Un-patched torch._scaled_mm (cuBLASLt FP8) on the same C4 rotation: the library sanity bar SURVEY 2.2 allows."""
    one = torch.ones((), device=bufs[0][0].device)

    def step():
        for a, inv_a, w, inv_w, out in bufs:
            torch._scaled_mm(a.view(torch.float8_e4m3fn), w.view(torch.float8_e4m3fn).t(), inv_a.reshape(()), inv_w.reshape(()),
                             None, None, torch.bfloat16, False)
    try:
        step()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step()
        for _ in range(max(warmup, 3)):
            g.replay()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (steps * len(bufs))
        del one
        return {"us_per_call": round(us, 2), "tflops": round(C4_FLOPS / (us * 1e-6) / 1e12, 1),
                "what": "stock torch._scaled_mm (cuBLASLt FP8, fast_accum off), same rotation and CUDA graph; a yardstick, "
                        "not part of the product path"}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)[:300]}


# --------------------------------------------------------------------------- main

_JSON_OUT = None


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def pin_to_gpu_numa_node(torch, index):
    """Best effort: run this rank's host thread (and so first-touch its pinned buffers) on the CPUs NVML names as local
    to the GPU, so that N ranks' host<->device copies do not all cross one memory controller.  Inside a container the
    cpuset may not contain them; then nothing is changed and the line says so."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        ideal = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        both = ideal & allowed
        if not ideal:
            return "no affinity reported"
        if both and both != allowed:
            os.sched_setaffinity(0, both)
            return f"pinned to {len(both)} of {len(allowed)} cpus local to the GPU"
        if both == allowed:
            return f"all {len(allowed)} allowed cpus are local to the GPU"
        return "GPU-local cpus outside this process's cpuset"
    except Exception as e:
        return f"not pinned: {type(e).__name__}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-sub", action="store_true", help="headline only")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed row sample of the last timed step's results to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs is implemented for the single-GPU run of --impl ours")
    # stdout carries exactly ONE line: the JSON.  Libraries chat on fd 1 (NCCL prints its version there, the
    # patch prints like the reference), so fd 1 is pointed at stderr for the run and the line goes to the saved fd.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from _util import dt_code

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    numa = pin_to_gpu_numa_node(torch, torch.cuda.current_device())
    n_gpus = world
    steps = max(args.steps, 1)
    warmup = max(args.warmup, 3)
    peaks = load_peaks()
    fp8_peak = 2 * peaks["bf16"]
    L = _capi()                                    # fails loudly if libfp8_b200.so is missing
    import fp8_mps_native
    import fp8_mps_patch
    M, K, N = C4["M"], C4["K"], C4["N"]
    bf16 = dt_code(torch.bfloat16)

    # ---------------- data: the SAME four (A, W) sets on every rank (same seeds), randn -> reference-codec FP8 on the device
    bufs = []
    for i in range(SETS):
        g = torch.Generator(device=dev).manual_seed(100 + i)
        a, inv_a = _rand_fp8(torch, (M, K), g, dev)
        w, inv_w = _rand_fp8(torch, (N, K), g, dev)
        out = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
        bufs.append((a, inv_a, w, inv_w, out))

    def step_single():
        for a, inv_a, w, inv_w, out in bufs:
            _mm(L, torch, a, w, out, bf16, inv_a, inv_w, algo=2)

    sharded = None
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    if n_gpus == 1:
        ms, launches_per_step, t0, t1 = time_graph(torch, step_single, steps, warmup)
        if args.dump_outputs:                      # the graph's last replay wrote every `out`; nothing has run since
            dump_outputs(torch, args.dump_outputs, {f"c4_out_set{i}": b[4] for i, b in enumerate(bufs)})
        clocks = sampler.summary(t0, t1)
        kernel_us = ms / steps * 1e3 / SETS
        kernel_name = "fp8b::fp8_gemm_tcgen05_kernel<256,2,2> (CTA pairs, 256x256 tiles, TMA-store epilogue)"
    else:
        from fp8_sharded import ShardedScaledMM, shard_bounds
        lins = [ShardedScaledMM(w, inv_w, None) for (_, _, w, inv_w, _) in bufs]       # each keeps its own shard of W
        n0, n1, width = shard_bounds(N, n_gpus, rank)

        def plan_step(mode, layout="row_major"):
            def run():
                for lin, (a, inv_a, _, _, _) in zip(lins, bufs):
                    lin(a, inv_a, torch.bfloat16, layout=layout, mode=mode)
            return run

        # parity of every plan BEFORE anything is timed: bit-equal to the un-sharded GEMM on every rank, and a 64-row
        # slab of the un-sharded result against the CPU oracle
        step_single()
        torch.cuda.synchronize()
        a0, inv_a0, w0, inv_w0, full0 = bufs[0]
        oracle_err = None
        if rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import fp8_oracle as o
            ref = o.scaled_mm(a0[:64].cpu().numpy(), w0.cpu().numpy(), inv_a0.cpu().numpy(), inv_w0.cpu().numpy(), None, None,
                              "bf16", accum="f32")
            oracle_err = float(o.rel_rmse(full0[:64].float().cpu().numpy(), ref))
        GRAPH_PLANS = ("push", "peers", "multicast")
        plans = {"push_fused": ("push", "row_major"), "peer_store_fused": ("peers", "row_major"),
                 "multicast_fused": ("multicast", "row_major"), "allgather_row_major": ("allgather", "row_major"),
                 "allgather_rank_major": ("allgather", "rank_major")}
        sharded = {"world": n_gpus, "exchange_recv_bytes_per_gpu": int((n_gpus - 1) * M * (n1 - n0) * 2),
                   "oracle_slab_rel_rmse_unsharded": oracle_err, "plans": {}}
        for name, (mode, layout) in plans.items():
            entry = {}
            try:
                y = lins[0](a0, inv_a0, torch.bfloat16, layout=layout, mode=mode)
                if layout == "rank_major":
                    y = y.permute(1, 0, 2).reshape(M, -1)[:, :N]
                torch.cuda.synchronize()
                same = torch.tensor([1 if torch.equal(y, full0) else 0], device=dev)
                dist.all_reduce(same, op=dist.ReduceOp.MIN)
                entry["parity"] = bool(int(same.item()) == 1) and (oracle_err is None or oracle_err <= 3e-3)
                entry["bit_equal_to_unsharded_on_every_rank"] = bool(int(same.item()) == 1)
                fn = plan_step(mode, layout)
                for _ in range(warmup):
                    fn()
                torch.cuda.synchronize()
                dist.barrier()
                torch.cuda.synchronize()
                # the fused plans (one kernel + one barrier kernel per call) are timed like the N = 1 step: captured in
                # CUDA graphs -- TWO of them, replayed alternately, because consecutive calls of a ShardedScaledMM use
                # the two buffers of its symmetric pair in turn.  The NCCL plans allocate and call the collective from
                # the host; they stay eager (their 190-300 us per call hide the host).
                run_step, timing = fn, "eager"
                n0_l = L.fp8b_launch_count()
                graphs = []
                if mode in GRAPH_PLANS:
                    try:
                        for _ in range(2):
                            gr = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(gr):
                                fn()
                            graphs.append(gr)
                    except Exception as e:         # capture refused (the same on every rank): time the eager loop
                        entry["graph_capture_failed"] = repr(e)[:160]
                        graphs = []
                        torch.cuda.synchronize()
                if graphs:
                    launches_plan = int((L.fp8b_launch_count() - n0_l) // 2)
                    turn = [0]

                    def run_step():
                        graphs[turn[0] & 1].replay()
                        turn[0] += 1
                    timing = "cuda_graph"
                    for _ in range(max(warmup, 3)):
                        run_step()
                    torch.cuda.synchronize()
                    dist.barrier()
                    torch.cuda.synchronize()
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                n0_l = L.fp8b_launch_count()
                tw0 = time.perf_counter()
                e0.record()
                for _ in range(steps):
                    run_step()
                e1.record()
                torch.cuda.synchronize()
                tw1 = time.perf_counter()
                dist.barrier()
                t_ms = max_over_ranks(torch, dist, e0.elapsed_time(e1))
                entry["timing"] = timing
                entry["us_per_call"] = round(t_ms / steps * 1e3 / SETS, 2)
                entry["tflops_total"] = round(C4_FLOPS / (entry["us_per_call"] * 1e-6) / 1e12, 1)
                entry["launches_per_step"] = launches_plan if timing == "cuda_graph" else int((L.fp8b_launch_count() - n0_l) // steps)
                entry["_ms"], entry["_t0"], entry["_t1"] = t_ms, tw0, tw1
                if graphs:                         # the same calls issued one by one from Python, for the record
                    torch.cuda.synchronize()
                    dist.barrier()
                    torch.cuda.synchronize()
                    e0.record()
                    for _ in range(steps):
                        fn()
                    e1.record()
                    torch.cuda.synchronize()
                    dist.barrier()
                    entry["eager_us_per_call"] = round(max_over_ranks(torch, dist, e0.elapsed_time(e1)) / steps * 1e3 / SETS, 2)
            except Exception as e:                 # e.g. no NVLS multicast on this system: the plan did not run at all
                entry["unavailable"] = repr(e)[:200]
                entry["parity"] = None
            sharded["plans"][name] = entry
        # compute only (no exchange): this rank's shard through the plain kernel
        def step_local():
            for lin, (a, inv_a, _, _, _) in zip(lins, bufs):
                lin.local(a, inv_a, torch.bfloat16)
        ms_l, _, _, _ = time_graph(torch, step_local, steps, warmup, dist)
        sharded["shard_gemm_only_us"] = round(max_over_ranks(torch, dist, ms_l) / steps * 1e3 / SETS, 2)
        # the headline is the default plan of ShardedScaledMM (push); should it be unavailable on a box, the first row-major
        # plan that ran takes its place and the line says so -- a missing JSON line helps nobody
        head_name = next((k for k in ("push_fused", "multicast_fused", "peer_store_fused", "allgather_row_major")
                          if "us_per_call" in sharded["plans"][k]), None)
        if head_name is None:
            raise RuntimeError(f"no exchange plan ran: {sharded['plans']}")
        sharded["headline_plan"] = head_name
        e2e_mode = {"push_fused": "push", "multicast_fused": "multicast", "peer_store_fused": "peers",
                    "allgather_row_major": "allgather"}[head_name]
        head = sharded["plans"][head_name]
        ms, t0, t1 = head.pop("_ms"), head.pop("_t0"), head.pop("_t1")
        for e in sharded["plans"].values():
            for k in ("_ms", "_t0", "_t1"):
                e.pop(k, None)
        launches_per_step = head["launches_per_step"]
        clocks = sampler.summary(t0, t1)
        kernel_us = head["us_per_call"]
        kernel_name = ("fp8b::fp8_gemm_tcgen05_kernel<BN,2,2> (tcgen05 GEMM + TMA push to every rank), incl. the closing barrier"
                       if head_name == "push_fused" else f"exchange plan {head_name}")
        floor_link = (n_gpus - 1) / n_gpus * C4_OUT_BYTES / (NVLINK_GBS * 1e9) * 1e6
        floor_link_meas = (n_gpus - 1) / n_gpus * C4_OUT_BYTES / (NVLINK_MEASURED_GBS * 1e9) * 1e6
        floor_mma = C4_FLOPS / n_gpus / (fp8_peak * 1e12) * 1e6
        sharded["floor_us"] = {"nvlink_770GBs": round(floor_link, 1), "nvlink_measured_690GBs": round(floor_link_meas, 1),
                               "tensor_at_measured_peak": round(floor_mma, 1),
                               "bound": round(max(floor_link, floor_mma), 1),
                               "achieved_over_bound": round(max(floor_link, floor_mma) / kernel_us, 3),
                               "achieved_over_measured_link_bound": round(max(floor_link_meas, floor_mma) / kernel_us, 3),
                               "note": "a call must deliver (w-1)/w of the 100.7 MB result into every GPU; the fused kernel "
                                       "is bound by that exchange, not by the tensor pipe"}
        sharded["best_plan"] = min((k for k, v in sharded["plans"].items() if "us_per_call" in v and v.get("parity")),
                                   key=lambda k: sharded["plans"][k]["us_per_call"], default=None)
        sharded["parity"] = {k: v.get("parity") for k, v in sharded["plans"].items()}      # true / false / null = plan unavailable here

    ms = max_over_ranks(torch, dist, ms) if n_gpus == 1 else ms
    ms_per_step = ms / steps
    us_per_call = ms_per_step * 1e3 / SETS
    value = C4_FLOPS / (us_per_call * 1e-6) / 1e12             # whole job: one problem, N GPUs
    per_gpu = value / n_gpus

    # ---------------- e2e: the public call with pinned HOST buffers, copies inside the timed region
    a, inv_a, w, inv_w, _ = bufs[0]
    e2e_steps = max(min(steps, 10), 3)
    with contextlib.redirect_stdout(sys.stderr):
        fp8_mps_patch.install()
    try:
        hA = a.cpu().pin_memory()
        dA = torch.empty_like(a)
        if n_gpus == 1:
            hW = w.cpu().pin_memory()
            dW = torch.empty_like(w)
            hC = torch.empty(M, N, dtype=torch.bfloat16).pin_memory()

            def e2e_step():
                dA.copy_(hA, non_blocking=True)
                dW.copy_(hW, non_blocking=True)
                y = torch._scaled_mm(dA.view(torch.float8_e4m3fn), dW.view(torch.float8_e4m3fn).t(), inv_a, inv_w, None, None,
                                     torch.bfloat16)
                hC.copy_(y, non_blocking=True)
            h2d, d2h = hA.numel() + hW.numel(), hC.numel() * 2
            call = ("fp8_mps_patch.install(); torch._scaled_mm(A8, W8.t(), scale_a, scale_b, None, None, torch.bfloat16): A and W "
                    "copied from pinned host memory, C copied back, every call")
        else:
            lin = lins[0]
            hW = lin.weight.cpu().pin_memory()
            r0_, r1_ = rank * M // n_gpus, (rank + 1) * M // n_gpus
            hC = torch.empty(r1_ - r0_, N, dtype=torch.bfloat16).pin_memory()
            # A is the same on every rank: each rank uploads only its 1/N row slab over PCIe and the ranks all-gather the
            # slabs over NVLink (12.6 MB, NCCL) instead of every rank pulling the whole matrix through the host
            even = M % n_gpus == 0
            hA_slab = hA[r0_:r1_].contiguous().pin_memory() if even else hA

            def e2e_step():
                if even:
                    dA[r0_:r1_].copy_(hA_slab, non_blocking=True)
                    dist.all_gather_into_tensor(dA.view(-1), dA[r0_:r1_].reshape(-1))
                else:
                    dA.copy_(hA, non_blocking=True)
                lin.weight.copy_(hW, non_blocking=True)
                y = lin(dA, inv_a, torch.bfloat16, mode=e2e_mode)
                hC.copy_(y[r0_:r1_], non_blocking=True)
            h2d, d2h = hA_slab.numel() + hW.numel(), hC.numel() * 2
            call = (f"ShardedScaledMM(W8, scale_b)(A8, scale_a, torch.bfloat16, mode='{e2e_mode}'): this rank's 1/N row slab of A "
                    "(all-gathered over NVLink) and its W shard copied from pinned host memory, this rank's 1/N row slab of the "
                    "assembled (M,N) result copied back, every call")
        for _ in range(3):
            e2e_step()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()
        nl0 = L.fp8b_launch_count()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(e2e_steps * SETS):
            e2e_step()
        e1.record()
        torch.cuda.synchronize()
        e2e_launches = L.fp8b_launch_count() - nl0
        if dist is not None:
            dist.barrier()
        e2e_ms = max_over_ranks(torch, dist, e0.elapsed_time(e1)) / e2e_steps           # per step of SETS calls
        e2e = {"value": round(C4_FLOPS * SETS / (e2e_ms * 1e-3) / 1e12, 3), "unit": "TFLOP/s",
               "h2d_bytes_per_step": int(h2d * SETS), "d2h_bytes_per_step": int(d2h * SETS),
               "ms_per_step": round(e2e_ms, 4), "steps": e2e_steps, "calls_per_step": SETS, "call": call,
               "kernel_launches": int(e2e_launches), "host_numa": numa,
               "pcie_gbs_per_gpu": round((h2d + d2h) * SETS / (e2e_ms * 1e-3) / 1e9, 1)}
        if n_gpus == 1:
            w8 = w.view(torch.float8_e4m3fn).t()

            def e2e_resident():
                dA.copy_(hA, non_blocking=True)
                y = torch._scaled_mm(dA.view(torch.float8_e4m3fn), w8, inv_a, inv_w, None, None, torch.bfloat16)
                hC.copy_(y, non_blocking=True)
            for _ in range(3):
                e2e_resident()
            torch.cuda.synchronize()
            r0 = torch.cuda.Event(enable_timing=True)
            r1 = torch.cuda.Event(enable_timing=True)
            r0.record()
            for _ in range(e2e_steps * SETS):
                e2e_resident()
            r1.record()
            torch.cuda.synchronize()
            res_ms = r0.elapsed_time(r1) / (e2e_steps * SETS)
            e2e["resident_weights"] = {"value": round(C4_FLOPS / (res_ms * 1e-3) / 1e12, 3), "unit": "TFLOP/s",
                                       "ms_per_call": round(res_ms, 4), "h2d_bytes_per_call": int(hA.numel()),
                                       "d2h_bytes_per_call": int(hC.numel() * 2),
                                       "note": "the plug-in's deployment shape: FP8 weights moved to the GPU once"}
    finally:
        fp8_mps_patch.uninstall()

    line = {
        "metric": METRIC, "value": round(value, 1), "unit": "TFLOP/s", "n_gpus": n_gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_for(n_gpus),
        "roofline": {"bound": "tensor", "achieved": round(per_gpu, 1), "peak": round(fp8_peak, 1), "unit": "TFLOP/s",
                     "frac": round(per_gpu / fp8_peak, 4), "traffic": profile_traffic("gemm") if n_gpus == 1 else None,
                     "frac_of_nominal_4500": round(per_gpu / 4500.0, 4), "us_per_launch": round(kernel_us, 2),
                     "frac_of_sustained_proxy": round(per_gpu / (2 * peaks["bf16_sustained"]), 4),
                     "sustained_note": "MEASURED_PEAKS.json also has the bf16 cuBLAS rate of a seconds-long loop under the power cap; "
                                       "`frac` uses the BURST figure although the timed region is milliseconds of back-to-back GEMMs",
                     "peak_source": f"{peaks['source']}: 2 x bf16 cuBLAS burst (MEASURED_PEAKS.json) as the dense-FP8 proxy",
                     "kernel": kernel_name, "flops_per_launch": C4_FLOPS // n_gpus},
        "e2e": e2e,
        "gpu_launches": int(launches_per_step * steps),
        "clocks": clocks,
    }
    if sharded is not None:
        line["sharded"] = sharded

    # ---------------- the other BASELINE configs (single-GPU paths: casts and GEMVs are replicas-only, SURVEY 8e)
    if not args.no_sub and n_gpus == 1:
        sub = {}
        gen = torch.Generator(device=dev).manual_seed(1)
        sub["C4_library_yardstick"] = bench_library_yardstick(torch, bufs, steps, warmup)
        if "us_per_call" in sub["C4_library_yardstick"]:
            sub["C4_library_yardstick"]["ours_over_library"] = round(sub["C4_library_yardstick"]["us_per_call"] / us_per_call, 3)
        try:
            L.fp8b_set_option(20, 2)              # FP8B_OPT_TUNE_GEMM_STORE = 2: same kernel with the TMA-store epilogue
            ms_t, _, _, _ = time_graph(torch, step_single, steps, warmup)
            sub["C4_tma_store_epilogue"] = {"us_per_call": round(ms_t / steps * 1e3 / SETS, 2)}
        except Exception as e:
            sub["C4_tma_store_epilogue"] = {"error": repr(e)[:200]}
        finally:
            L.fp8b_set_option(20, -1)
        del bufs
        torch.cuda.empty_cache()
        try:
            sub["C2_gemv_M1_K14336_N4096_bf16"] = bench_c2(torch, L, gen, dev, peaks, steps, warmup)
        except Exception as e:
            sub["C2_error"] = repr(e)[:300]
        try:
            sub["C1_gemv_M1_K4096_N4096_f16"] = bench_gemv_cfg(torch, L, C1, C1_BYTES, torch.float16, False, gen, dev,
                                                               peaks, steps, warmup, rotation=32)
            sub["C3_gemv_M4_K4096_N4096_bias_bf16"] = bench_gemv_cfg(torch, L, C3, C3_BYTES, torch.bfloat16, True, gen,
                                                                     dev, peaks, steps, warmup, rotation=32)
            sub["C1_gemv_M1_K4096_N4096_f16"]["roofline"]["traffic"] = profile_traffic("gemv1k4")
            sub["C3_gemv_M4_K4096_N4096_bias_bf16"]["roofline"]["traffic"] = profile_traffic("gemv4")
            sq = bench_gemv_cfg(torch, L, SQ, SQ_BYTES, torch.float32, False, gen, dev, peaks, steps, warmup, rotation=4)
            sq["reference_published"] = "2.38 ms on Apple M4 Pro (README.md:80; test_fp8_metal.py:232-236), other hardware"
            sub["ref_bench_gemv_M1_K14336_N14336_f32"] = sq
        except Exception as e:
            sub["gemv_error"] = repr(e)[:300]
        try:
            sub["C5_casts_flux_12B"] = bench_casts_c5(torch, L, gen, dev, peaks, steps, warmup)
        except Exception as e:
            sub["cast_error"] = repr(e)[:300]
        line["sub"] = sub
    elif n_gpus > 1:
        line["sub_note"] = "C1/C2/C3/C5 are single-GPU paths (replicas only, SURVEY 8e): see the N=1 line"

    sampler.stop()
    if rank == 0 and n_gpus == 1 and not args.no_cpu:
        try:
            line["cpu_baseline"] = cpu_c4_baseline()
        except Exception as e:
            line["cpu_baseline"] = {"error": repr(e)}
    if dist is not None:
        dist.barrier()
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
