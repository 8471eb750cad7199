"""torchrun script: C4 N-sharded linear, the four exchange plans, max-over-ranks CUDA-event time.
   python -m torch.distributed.run --nnodes=1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P profiles/tools/time_sharded.py"""
import os, sys
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..")
sys.path.insert(0, os.path.join(ROOT, "fp8-mps-metal_b200"))
import torch, torch.distributed as dist

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ.get("LOCAL_RANK", rank))
torch.cuda.set_device(lr); dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
from fp8_sharded import ShardedScaledMM, shard_bounds
import fp8_mps_native as nat
M, K, N = 4096, 3072, 12288
g = torch.Generator(device=dev).manual_seed(3)
a = torch.randint(0, 120, (M, K), dtype=torch.uint8, device=dev, generator=g)
n0, n1, _ = shard_bounds(N, world, rank)
w = torch.randint(0, 120, (n1 - n0, K), dtype=torch.uint8, device=dev, generator=g)
sa = torch.tensor([0.01], device=dev); sb = torch.tensor([0.02], device=dev)
lin = ShardedScaledMM(w, sb, None, weight_is_shard=True, full_N=N)
variants = {"compute_only": lambda: lin.local(a, sa, torch.bfloat16),
            "allgather_rank_major": lambda: lin(a, sa, torch.bfloat16, layout="rank_major"),
            "multicast_fused": lambda: lin(a, sa, torch.bfloat16, mode="multicast"),
            "peer_store_fused": lambda: lin(a, sa, torch.bfloat16, mode="peers"),
            "push_fused": lambda: lin(a, sa, torch.bfloat16, mode="push")}
def push_kernel_only():
    # the fused kernel alone, without the closing symmetric-memory barrier (timing breakdown only)
    key, pair, turn = lin._symm_buffers(M, torch.bfloat16, dev)
    buf, hdl = pair[turn]
    nat._get_lib().fp8_scaled_mm_push(a, lin.weight, sa, lin.scale_b, None, buf, lin._push_order(turn, hdl), int(lin.n0))
def barrier_only():
    key, pair, turn = lin._symm_buffers(M, torch.bfloat16, dev)
    pair[turn][1].barrier(channel=0)
variants["push_kernel_only"] = push_kernel_only
variants["barrier_only"] = barrier_only
for cfg in [int(c) for c in os.environ.get("CFGS", "").split(",") if c]:
    def mk(cfg):
        def run():
            nat._get_lib().set_option(16, cfg)
            try:
                lin(a, sa, torch.bfloat16, mode="push")
            finally:
                nat._get_lib().set_option(16, -1)
        return run
    variants[f"push_cfg{cfg}"] = mk(cfg)
def mk_raster(v, kernel_only):
    def run():
        nat._get_lib().set_option(24, v)
        try:
            push_kernel_only() if kernel_only else lin(a, sa, torch.bfloat16, mode="push")
        finally:
            nat._get_lib().set_option(24, -1)
    return run
variants["push_rasterN"] = mk_raster(2, False)
variants["push_rasterN_kernel_only"] = mk_raster(2, True)
def compute_rasterN():
    nat._get_lib().set_option(24, 2)
    try:
        lin.local(a, sa, torch.bfloat16)
    finally:
        nat._get_lib().set_option(24, -1)
variants["compute_only_rasterN"] = compute_rasterN
def mk_barrier(fused):
    def run():
        keep = lin.fused_barrier
        lin.fused_barrier = fused
        try:
            lin(a, sa, torch.bfloat16, mode="push")
        finally:
            lin.fused_barrier = keep
    return run
variants["push_symm_barrier"] = mk_barrier(False)
variants["push_fused_barrier"] = mk_barrier(True)
only = os.environ.get("ONLY")
if only:
    variants = {k: v for k, v in variants.items() if k in only.split(",")}
out = {}
for name, fn in variants.items():
    try:
        for _ in range(5): fn()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20): fn()
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / 20 * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name] = round(float(t.item()), 1)
    except Exception as e:
        out[name] = repr(e)[:120]
# parity of the push plan against the all-gather of the same shards
try:
    y_push = lin(a, sa, torch.bfloat16, mode="push").clone()
    y_ag = lin(a, sa, torch.bfloat16, layout="row_major")
    torch.cuda.synchronize()
    out["push==allgather"] = bool(torch.equal(y_push, y_ag))
except Exception as e:
    out["push==allgather"] = repr(e)[:200]
if rank == 0:
    print(f"world {world}: " + "  ".join(f"{k} {v} us" for k, v in out.items()), flush=True)
dist.barrier()
dist.destroy_process_group()
