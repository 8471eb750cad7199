"""
N-sharded FP8 linear across the GPUs of one box (one process per GPU, torch.distributed).

The reference is single-device (SURVEY 2.3): this module is the build's multi-GPU extension of its
`_scaled_mm` path for large-N DiT linears.  The weight B (N,K) is split by ROWS of B = COLUMNS of
the output: rank r owns B[n0_r:n1_r, :] (and the matching slices of a per-row scale_b and of the
bias), the activations A (M,K) are replicated, every rank runs the same tcgen05 kernel on its
shard -- no reduction is needed -- and ONE exchange step assembles the (M,N) result:

  mode="allgather"  ncclAllGather of the contiguous local (M, N/w) blocks into a rank-major
                    [w, M, N/w] buffer, exposed either as is (layout="rank_major", zero extra
                    passes) or re-laid to the row-major (M,N) tensor stock _scaled_mm returns
                    (layout="row_major", one extra device pass);
  mode="push"       fused, unicast, the default on NVLink boxes: the GEMM's epilogue warps only fill a
                    shared-memory ring and a dedicated warp pushes every finished 128 x 128-byte box with TMA
                    stores (cp.async.bulk.tensor) into this rank's result and into the same place of every
                    peer's result (symmetric memory).  Each GPU receives (w-1)/w of the output, the NVLink
                    writes overlap the next tile's MMAs, any M / N (TMA clips the edges); no NVLS needed.
  mode="peers"      the round-1 form of the same plan: the epilogue warps themselves issue st.global to
                    every peer.  Kept for comparison (CTA-pair tiles only: M > 128, N/w > 128).
  mode="multicast"  fused: the GEMM epilogue writes each output tile straight into the row-major
                    (M,N) result of EVERY rank through an NVSwitch multicast mapping
                    (multimem.st), so the exchange overlaps the math tile by tile and no gather or
                    re-layout pass exists.  Needs torch symmetric memory (CUDA, NVLS).

Every plan returns what the un-sharded kernel returns, bit for bit (no reduction crosses ranks), with one exception:
for problems with very few tiles the un-sharded call may take the library's split-K plan, which rounds differently
(fp8b_set_option(FP8B_OPT_TUNE_GEMM_SPLITK, 1) turns it off); the sharded kernels never split K.

Shards are contiguous, equal-sized (ceil(N/w) rounded up to `align` columns; the tail shard may be
short or empty) so the gather can use the fixed-size collective.
"""

from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist


def shard_bounds(N: int, world: int, rank: int, align: int = 16) -> Tuple[int, int, int]:
    """(n0, n1, width): rank's column range [n0, n1) and the common padded shard width."""
    width = -(-N // world)
    width = -(-width // align) * align
    n0 = min(N, rank * width)
    n1 = min(N, n0 + width)
    return n0, n1, width


def _refuse_fp8_out(out_dtype) -> None:
    """FP8 results are not exchanged between ranks yet: raise on every rank alike, before anything is launched or sent."""
    if out_dtype in (torch.float8_e4m3fn, torch.float8_e5m2):
        raise ValueError(f"ShardedScaledMM: out_dtype {out_dtype} is not supported (float32, float16 or bfloat16); "
                         "the single-GPU fp8_scaled_mm_fused takes out_dtype=torch.float8_e4m3fn")


def _default_mm(a, b, sa, sb, bias, out_dtype, out=None):
    import fp8_mps_native
    return fp8_mps_native.fp8_scaled_mm_fused(a, b, sa, sb, bias=bias, scale_result=None, out_dtype=out_dtype, out=out)


class ShardedScaledMM:
    """y = _scaled_mm(x, W^T) with W (N,K) row-sharded over the process group."""

    def __init__(self, weight_u8: torch.Tensor, scale_b: torch.Tensor, bias: Optional[torch.Tensor] = None,
                 group=None, mm_fn: Optional[Callable] = None, weight_is_shard: bool = False,
                 full_N: Optional[int] = None, align: int = 16):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.mm_fn = mm_fn or _default_mm
        if weight_is_shard:
            assert full_N is not None
            self.N = int(full_N)
        else:
            self.N = int(weight_u8.shape[0])
        self.align = align
        self.n0, self.n1, self.width = shard_bounds(self.N, self.world, self.rank, align)
        if weight_is_shard:
            assert weight_u8.shape[0] == self.n1 - self.n0
            self.weight = weight_u8.contiguous()
        else:
            self.weight = weight_u8[self.n0:self.n1].contiguous()
        sb = scale_b.reshape(-1)
        if sb.numel() == 1:
            self.scale_b = sb
        elif sb.numel() == self.N:
            self.scale_b = sb[self.n0:self.n1].contiguous()
        else:
            assert sb.numel() == self.n1 - self.n0, "scale_b must have 1, N or shard-width elements"
            self.scale_b = sb.contiguous()
        if bias is None:
            self.bias = None
        elif bias.numel() == self.N:
            self.bias = bias.reshape(-1)[self.n0:self.n1].contiguous()
        else:
            assert bias.numel() == self.n1 - self.n0
            self.bias = bias.reshape(-1).contiguous()
        self._symm = None
        self._sig = None
        #: push mode: fuse the closing barrier into the exchange (kernel-side signal + a PDL wait kernel) instead of a
        #: separate symmetric-memory barrier kernel after it.  Measured (profiles/r2_scaling.md): w = 2 101.1 vs 102.7 us,
        #: w = 4 144.9 vs 145.0 us, w = 8 174.8 vs 166.9 us (seven system-scope release stores from one thread, and the skew
        #: between eight ranks, cost more than the barrier kernel) -- so it is the default for two ranks only.
        self.fused_barrier = self.world <= 2

    # ------------------------------------------------------------------ local compute
    def local(self, x_u8: torch.Tensor, scale_a: torch.Tensor, out_dtype=torch.bfloat16, out=None) -> torch.Tensor:
        """This rank's (M, n1-n0) column block."""
        if self.n1 == self.n0:
            return torch.empty(x_u8.shape[0], 0, dtype=out_dtype or torch.float32, device=x_u8.device)
        return self.mm_fn(x_u8, self.weight, scale_a, self.scale_b, self.bias, out_dtype, out)

    # ------------------------------------------------------------------ NCCL all-gather path
    def __call__(self, x_u8: torch.Tensor, scale_a: torch.Tensor, out_dtype=torch.bfloat16,
                 layout: str = "row_major", mode: str = "allgather") -> torch.Tensor:
        _refuse_fp8_out(out_dtype)
        if mode == "auto":
            mode = self.best_mode(x_u8.shape[0], x_u8.shape[1], out_dtype or torch.float32, x_u8.device) \
                if layout == "row_major" else "allgather"
        if mode == "push":
            return self.forward_push(x_u8, scale_a, out_dtype)
        if mode == "multicast":
            return self.forward_multicast(x_u8, scale_a, out_dtype)
        if mode == "peers":
            return self.forward_peers(x_u8, scale_a, out_dtype)
        M = x_u8.shape[0]
        odt = out_dtype or torch.float32
        if self.world == 1:
            return self.local(x_u8, scale_a, out_dtype)
        gathered = torch.empty(self.world, M, self.width, dtype=odt, device=x_u8.device)
        mine = gathered[self.rank]                              # contiguous (M, width) block
        if self.n1 - self.n0 == self.width:
            self.local(x_u8, scale_a, out_dtype, out=mine)      # the kernel writes straight into the gather buffer
        else:                                                   # short tail shard: pad with zeros
            mine.zero_()
            if self.n1 > self.n0:
                mine[:, : self.n1 - self.n0].copy_(self.local(x_u8, scale_a, out_dtype))
        inp = mine.reshape(-1)                                  # NCCL gathers in place (input aliases its output slot)
        if dist.get_backend(self.group) != "nccl":
            inp = inp.clone()
        dist.all_gather_into_tensor(gathered.view(-1), inp, group=self.group)
        if layout == "rank_major":
            return gathered                                     # [w, M, width]; column n lives at [n // width, :, n % width]
        return gathered.permute(1, 0, 2).reshape(M, self.world * self.width)[:, : self.N].contiguous()

    # ------------------------------------------------------------------ fused multicast path
    def _symm_buffers(self, M: int, odt, device):
        import torch.distributed._symmetric_memory as symm_mem
        key = (M, odt)
        if self._symm is None or self._symm[0] != key:
            pg = self.group if self.group is not None else dist.group.WORLD
            pair = []
            for _ in range(2):                                  # double-buffered: see forward_multicast
                buf = symm_mem.empty((M, self.N), dtype=odt, device=device)
                pair.append((buf, symm_mem.rendezvous(buf, pg)))
            self._symm = (key, pair, 0)
        return self._symm

    def forward_multicast(self, x_u8: torch.Tensor, scale_a: torch.Tensor, out_dtype=torch.bfloat16) -> torch.Tensor:
        """GEMM whose epilogue stores through the NVSwitch multicast address: after the closing
        barrier every rank holds the full row-major (M,N) result.

        The result aliases one of TWO symmetric buffers used alternately, so it stays valid until the
        call after next.  That is also what makes one barrier per call enough: a rank can only pass the
        closing barrier of call i-1 after every rank has ENTERED call i-1, i.e. finished with result i-2,
        whose buffer call i is about to overwrite."""
        _refuse_fp8_out(out_dtype)
        import fp8_mps_native
        M = x_u8.shape[0]
        odt = out_dtype or torch.float32
        if self.world == 1:
            return self.local(x_u8, scale_a, out_dtype)
        if not self.fused_supported("multicast", M, x_u8.shape[1], odt, x_u8.device):
            raise RuntimeError("multicast mode needs N/world % 32 == 0 and 16-byte aligned shard columns on every rank")
        key, pair, turn = self._symm_buffers(M, odt, x_u8.device)
        buf, hdl = pair[turn]
        mc = getattr(hdl, "multicast_ptr", 0)
        if not mc:                                              # a property of the system: every rank raises alike
            raise RuntimeError("symmetric memory has no multicast mapping on this system (NVLS unavailable)")
        self._symm = (key, pair, turn ^ 1)
        if self.n1 > self.n0:
            fp8_mps_native._get_lib().fp8_scaled_mm_multicast(
                x_u8, self.weight, scale_a, self.scale_b, self.bias, odt, int(mc), int(self.N), int(self.n0))
        hdl.barrier(channel=0)                                  # every rank's tiles have landed everywhere
        return buf

    def forward_peers(self, x_u8: torch.Tensor, scale_a: torch.Tensor, out_dtype=torch.bfloat16) -> torch.Tensor:
        """Like forward_multicast, with peer stores: the GEMM epilogue writes every tile into this rank's buffer and
        into each peer's buffer (unicast over NVLink).  A rank's own shard never leaves the GPU, so the NVLink
        ingress per GPU is (w-1)/w of the output instead of all of it.  Same double-buffering and single barrier."""
        _refuse_fp8_out(out_dtype)
        import fp8_mps_native
        M = x_u8.shape[0]
        odt = out_dtype or torch.float32
        if self.world == 1:
            return self.local(x_u8, scale_a, out_dtype)
        if not self.fused_supported("peers", M, x_u8.shape[1], odt, x_u8.device):   # same verdict on every rank, before any barrier
            raise RuntimeError("peer-store mode needs M > 128 and, on every rank, N/world > 128, N/world % 32 == 0")
        key, pair, turn = self._symm_buffers(M, odt, x_u8.device)
        buf, hdl = pair[turn]
        self._symm = (key, pair, turn ^ 1)
        deltas = self._peer_deltas(turn, buf, hdl)
        if self.n1 > self.n0:
            fp8_mps_native._get_lib().fp8_scaled_mm_peers(x_u8, self.weight, scale_a, self.scale_b, self.bias, buf,
                                                          deltas, int(self.n0))
        hdl.barrier(channel=0)                                  # every rank's tiles have landed everywhere
        return buf

    def _peer_deltas(self, turn, buf, hdl):
        cache = getattr(self, "_deltas", None)
        if cache is None or cache[0] is not self._symm[1]:
            cache = (self._symm[1], {})
            self._deltas = cache
        if turn not in cache[1]:
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            assert len(ptrs) == self.world
            local = ptrs[self.rank]
            cache[1][turn] = torch.tensor([p - local for p in ptrs], dtype=torch.int64, device=buf.device)
        return cache[1][turn]

    # ------------------------------------------------------------------ which fused plans can serve a call
    def fused_supported(self, mode: str, M: int, K: int, odt, device) -> bool:
        """Whether a fused plan can serve this call ON EVERY RANK -- computed from (mode, M, K, N, world, dtype)
        only, over all ranks' shard bounds, so every rank reaches the same verdict without communicating.  (Round 1
        checked per rank inside the launch: with N = 4080, w = 2 one rank launched and waited in the barrier while
        the other raised.)"""
        if mode == "push":
            return self.push_supported(M, K, odt, device)
        if self.world <= 1 or device.type != "cuda" or not dist.is_initialized() or dist.get_backend(self.group) != "nccl":
            return False
        esz = torch.empty((), dtype=odt).element_size()
        if K < 16 or K % 16 or (self.N * esz) % 16:
            return False
        for r in range(self.world):
            n0, n1, _ = shard_bounds(self.N, self.world, r, self.align)
            nl = n1 - n0
            if nl == 0:
                continue
            if nl % 32 or (n0 * esz) % 16:                       # multimem.st / st.global.v4 have no sub-word form
                return False
            if mode == "peers" and not (M > 128 and nl > 128):   # CTA-pair tile configurations only
                return False
        return mode in ("peers", "multicast")

    def push_supported(self, M: int, K: int, odt, device) -> bool:
        """Whether mode="push" can serve this call -- evaluated from (M, K, N, world, dtype) only, so every rank
        reaches the same answer without communicating (a rank must never skip the closing barrier)."""
        if self.world <= 1 or device.type != "cuda" or not dist.is_initialized():
            return False
        if dist.get_backend(self.group) != "nccl":
            return False
        esz = torch.empty((), dtype=odt).element_size()
        if K < 16 or K % 16 or (self.N * esz) % 16:
            return False
        for r in range(self.world):                              # every rank's column block: start and length in 16-byte units
            n0, n1, _ = shard_bounds(self.N, self.world, r, self.align)
            if (n0 * esz) % 16 or ((n1 - n0) * esz) % 16:
                return False
        return True

    def forward_push(self, x_u8: torch.Tensor, scale_a: torch.Tensor, out_dtype=torch.bfloat16) -> torch.Tensor:
        """ONE kernel computes this rank's column block and pushes it, box by box, into the row-major (M,N) result
        of every rank (fp8b_scaled_mm_push: tcgen05 GEMM + TMA stores to local HBM and, over NVLink, to the peers'
        symmetric buffers).  Same double-buffering and single closing barrier as forward_multicast.

        CUDA-graph capturable once the symmetric buffers exist (call it once eagerly first); capture TWO graphs and
        replay them in turn if the double-buffering matters to the caller.  Do not let the last reference to a
        symmetric buffer die inside a capture (freeing one is not a capturable operation)."""
        _refuse_fp8_out(out_dtype)
        import fp8_mps_native
        M, K = x_u8.shape
        odt = out_dtype or torch.float32
        if self.world == 1:
            return self.local(x_u8, scale_a, out_dtype)
        if not self.push_supported(M, K, odt, x_u8.device):      # same verdict on every rank: nobody is left in a barrier
            raise RuntimeError("push mode needs NCCL ranks on CUDA, K % 16 == 0 and 16-byte aligned shard columns")
        key, pair, turn = self._symm_buffers(M, odt, x_u8.device)
        buf, hdl = pair[turn]
        self._symm = (key, pair, turn ^ 1)
        lib = fp8_mps_native._get_lib()
        if self.fused_barrier and self._all_shards_nonempty() and not torch.cuda.is_current_stream_capturing():
            # (the epoch is a host-side count baked into the launch: a captured graph would replay a stale one, so under
            # stream capture the call closes with the symmetric-memory barrier kernel below instead)
            # closing barrier fused into the exchange: the push kernel's last CTA stores this call's epoch into every
            # peer's flag word; fp8b_peer_wait (one warp, programmatic dependent launch, already resident) returns when
            # every peer's flag has arrived and this rank's own kernel has completed
            sig = self._signal_state(x_u8.device)
            sig["epoch"] += 1
            lib.fp8_scaled_mm_push(x_u8, self.weight, scale_a, self.scale_b, self.bias, buf, self._push_order(turn, hdl),
                                   int(self.n0), sig["order"], sig["counter"], sig["epoch"], sig["flags"], self.rank)
            return buf
        if self.n1 > self.n0:
            lib.fp8_scaled_mm_push(x_u8, self.weight, scale_a, self.scale_b, self.bias, buf,
                                   self._push_order(turn, hdl), int(self.n0))
        hdl.barrier(channel=0)                                  # every rank's boxes have landed everywhere
        return buf

    def _all_shards_nonempty(self) -> bool:
        return all(shard_bounds(self.N, self.world, r, self.align)[1] > shard_bounds(self.N, self.world, r, self.align)[0]
                   for r in range(self.world))

    def _signal_state(self, device):
        """Symmetric flag words for the fused barrier: flags[r] on this rank is written by rank r.  Epochs only grow."""
        if self._sig is None:
            import torch.distributed._symmetric_memory as symm_mem
            pg = self.group if self.group is not None else dist.group.WORLD
            flags = symm_mem.empty(16, dtype=torch.int64, device=device)
            flags.zero_()
            hdl = symm_mem.rendezvous(flags, pg)
            hdl.barrier(channel=0)                              # every rank's zeros are in place before anyone signals
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            order = []
            for d in range(self.world):                          # same order as _push_order: own buffer first
                r = (self.rank + d) % self.world
                order.append(0 if r == self.rank else ptrs[r] + 8 * self.rank)
            self._sig = dict(flags=flags, hdl=hdl, counter=torch.zeros(1, dtype=torch.int32, device=device), order=order, epoch=0)
        return self._sig

    def _push_order(self, turn, hdl):
        """Destination base addresses for this buffer of the pair: own buffer first, then the ring of peers starting
        at rank+1, so that at any moment the ranks write to different destinations."""
        cache = getattr(self, "_order", None)
        if cache is None or cache[0] is not self._symm[1]:
            cache = (self._symm[1], {})
            self._order = cache
        if turn not in cache[1]:
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            assert len(ptrs) == self.world
            cache[1][turn] = [ptrs[(self.rank + d) % self.world] for d in range(self.world)]
        return cache[1][turn]

    def best_mode(self, M: int = 0, K: int = 0, odt=torch.bfloat16, device=None) -> str:
        """The fused TMA-store plan whenever it applies (decided from the shape alone, identically on every rank),
        else GEMM + NCCL all-gather.  Measured on 8 x B200 (C4, bf16 out, row-major result on every rank;
        profiles/r2_scaling.md)."""
        if device is not None and self.push_supported(M, K, odt, device):
            return "push"
        return "allgather"
