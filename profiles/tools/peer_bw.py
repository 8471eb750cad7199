"""torchrun script (>= 2 GPUs): what does a peer GPU's memory accept over NVLink?
  * copy engine: buf_peer.copy_(buf_local), 100 MB
  * SM-issued stores from the profiling library (FP8B_LIB=profiles/tools/bin/libfp8_b200_profile.so): st.global.v4,
    cp.async.bulk contiguous chunks, cp.async.bulk one row segment per copy (the GEMM tile pattern, 24 KB pitch)
  * the fused GEMM + push kernel with K = 64 (no MMA time to speak of): its exchange path alone
Every rank writes to rank+1; time = max over ranks, CUDA events.
   FP8B_LIB=... python -m torch.distributed.run --nproc-per-node 2 ... profiles/tools/peer_bw.py"""
import ctypes, os, sys
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..")
sys.path.insert(0, os.path.join(ROOT, "fp8-mps-metal_b200")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch, torch.distributed as dist
import torch.distributed._symmetric_memory as symm_mem

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ.get("LOCAL_RANK", rank))
torch.cuda.set_device(lr); dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
M, N = 4096, 12288
buf = symm_mem.empty((M, N), dtype=torch.bfloat16, device=dev)
hdl = symm_mem.rendezvous(buf, dist.group.WORLD)
peer = (rank + 1) % world
peer_ptr = int(hdl.buffer_ptrs[peer]); own_ptr = int(hdl.buffer_ptrs[rank])
peer_t = hdl.get_buffer(peer, (M, N), torch.bfloat16)
nbytes = M * N * 2
local = torch.empty(M, N, dtype=torch.bfloat16, device=dev)


def timed(fn, reps=10):
    for _ in range(3): fn()
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps * 1e3], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.barrier()
    return float(t.item())


out = []
us = timed(lambda: peer_t.copy_(local))
out.append(f"copy-engine peer copy 100 MB: {us:7.1f} us {nbytes / us / 1e3:6.0f} GB/s")
us = timed(lambda: buf.copy_(local))
out.append(f"local copy 100 MB:            {us:7.1f} us {2 * nbytes / us / 1e3:6.0f} GB/s (read+write)")

lib_path = os.environ.get("FP8B_LIB")
if lib_path:
    L = ctypes.CDLL(lib_path)
    L.fp8b_prof_fill.restype = ctypes.c_int
    L.fp8b_prof_fill.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t,
                                 ctypes.c_int, ctypes.c_void_p]
    st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for target, ptr in (("peer ", peer_ptr), ("local", own_ptr)):
        for name, mode, chunk, depth, rowb, cps in [("st.global.v4 512thr x1/SM", 0, 0, 0, 0, 1), ("st.global.v4 512thr x4/SM", 0, 0, 0, 0, 4),
                                                    ("bulk 16KB contiguous d2", 1, 16384, 2, 0, 1), ("bulk 16KB contiguous d4 x2/SM", 1, 16384, 4, 0, 2),
                                                    ("bulk 4KB contiguous d8", 1, 4096, 8, 0, 1),
                                                    ("bulk 512B row segs d16", 1, 512, 16, 512, 1), ("bulk 512B row segs d32 x4/SM", 1, 512, 32, 512, 4),
                                                    ("bulk 128B row segs d32 x4/SM", 1, 128, 32, 128, 4),
                                                    ("bulk 2KB row segs d16 x2/SM", 1, 2048, 16, 2048, 2)]:
            us = timed(lambda: L.fp8b_prof_fill(ctypes.c_void_p(ptr), nbytes, mode, chunk, depth, rowb, N * 2, cps, st()))
            out.append(f"{target} {name:32s}: {us:7.1f} us {nbytes / us / 1e3:6.0f} GB/s")

# the GEMM's exchange path alone: K = 64
import fp8_mps_native as nat
from fp8_sharded import ShardedScaledMM, shard_bounds
for K in (64, 3072):
    g = torch.Generator(device=dev).manual_seed(3)
    a = torch.randint(0, 120, (M, K), dtype=torch.uint8, device=dev, generator=g)
    n0, n1, _ = shard_bounds(N, world, rank)
    w = torch.randint(0, 120, (n1 - n0, K), dtype=torch.uint8, device=dev, generator=g)
    sa = torch.tensor([0.01], device=dev); sb = torch.tensor([0.02], device=dev)
    lin = ShardedScaledMM(w, sb, None, weight_is_shard=True, full_N=N)
    key, pair, turn = lin._symm_buffers(M, torch.bfloat16, dev)
    b2, h2 = pair[0]
    order = lin._push_order(0, h2)
    shard_bytes = M * (n1 - n0) * 2
    for name, dsts in (("local only", order[:1]), ("peer only", order[1:2]), ("local + peers", order)):
        us = timed(lambda: nat._get_lib().fp8_scaled_mm_push(a, w, sa, sb, None, b2, dsts, int(n0)))
        out.append(f"GEMM+push K={K:4d} {name:14s}: {us:7.1f} us  {shard_bytes * (len(dsts) - (1 if name != 'peer only' else 0)) / us / 1e3:6.0f} GB/s to peers")
    us = timed(lambda: lin.local(a, sa, torch.bfloat16))
    out.append(f"GEMM K={K:4d} st.global epilogue, local shard: {us:7.1f} us")
# the exchange path alone (K = 64, peer only) under the kernel's knobs: tile shape, tile order
K = 64
g = torch.Generator(device=dev).manual_seed(3)
a = torch.randint(0, 120, (M, K), dtype=torch.uint8, device=dev, generator=g)
n0, n1, _ = shard_bounds(N, world, rank)
w = torch.randint(0, 120, (n1 - n0, K), dtype=torch.uint8, device=dev, generator=g)
lin = ShardedScaledMM(w, sb, None, weight_is_shard=True, full_N=N)
key, pair, turn = lin._symm_buffers(M, torch.bfloat16, dev)
b2, h2 = pair[0]
order = lin._push_order(0, h2)
lib = nat._get_lib()
for cfg in (3, 4, 2):
    for raster in (1, 2):
        lib.set_option(16, cfg); lib.set_option(24, raster)
        try:
            us = timed(lambda: lib.fp8_scaled_mm_push(a, w, sa, sb, None, b2, order[1:2], int(n0)))
            out.append(f"K=64 peer only cfg{cfg} raster{raster}: {us:7.1f} us {M * (n1 - n0) * 2 / us / 1e3:6.0f} GB/s")
        except Exception as e:
            out.append(f"K=64 cfg{cfg} raster{raster}: {str(e)[:80]}")
lib.set_option(16, -1); lib.set_option(24, -1)
# does the destination ROW PITCH matter (NVLink / memory address interleaving)?  Same K = 64 push into wider buffers.
for pad in (0, 64, 128, 256, 320, 1024, 2048):
    wide_buf = symm_mem.empty((M, N + pad), dtype=torch.bfloat16, device=dev)
    wh = symm_mem.rendezvous(wide_buf, dist.group.WORLD)
    ptrs = [int(p_) for p_ in wh.buffer_ptrs]
    us = timed(lambda: lib.fp8_scaled_mm_push(a, w, sa, sb, None, wide_buf, [ptrs[(rank + 1) % world]], int(n0)))
    out.append(f"K=64 peer only, destination pitch {2 * (N + pad):6d} B: {us:7.1f} us {M * (n1 - n0) * 2 / us / 1e3:6.0f} GB/s")
if rank == 0:
    print(f"world {world}")
    print("\n".join(out), flush=True)
dist.barrier()
dist.destroy_process_group()
