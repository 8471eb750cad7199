"""Bit-exact, guarded tests of the N-sharded linear's exchange epilogues, on one GPU.

fp8b_scaled_mm_peers (the kStPeers instantiations of the tcgen05 GEMM) writes every 16-byte piece of its output once per
entry of a device table of int64 byte deltas; fp8b_scaled_mm_push writes every 128-row x 128-byte box to each pointer of
a host list.  Neither kernel can tell a peer's buffer from another local one, so every exchange can be replayed on one
GPU: all destinations of a call -- or of all W calls of an emulated exchange -- are matrices in ONE sentinel-filled
allocation.  Every delta is then small and known, a store sent to the wrong place lands on sentinels instead of faulting,
and one device-side comparison checks the whole allocation.

The inputs are the structured families of test_gpu_exact.py (one-hot A, one-hot B, few-hot small integers, NaN bytes in
B), so every destination must equal fp8_oracle.scaled_mm(accum="f64") bit for bit (+0 == -0).  The multicast epilogue is
never called here with arguments that pass validation: it needs an NVSwitch multicast mapping (tests/mgpu_sharded.py).
The completion flags of fp8b_scaled_mm_push_signal are checked on the host before any fp8b_peer_wait is enqueued, so a
signalling bug fails a test instead of leaving a wait kernel polling."""
import ctypes

import numpy as np
import pytest
import torch

from _util import (ALGO_TCGEN05, GUARD_ROWS, SENT, Terms, add_nan_rows, assert_bits_equal, capi, codes, dev_bias, dev_bytes,
                   dev_f32, dt_code, dt_name, edges, few_hot, one_hot, oracle, p, sm_count, small_ints, stream_ptr, tc_bounds,
                   to_np)
from fp8_sharded import shard_bounds

pytestmark = pytest.mark.gpu
DEV = "cuda"
OK, ERR_INVALID, ERR_UNSUPPORTED = 0, -1, -2
BN_OF_CFG = {3: 256, 4: 128, 5: 192}                  # GEMM_CFG -> tile width of the CTA-pair configurations (256 rows)
FLAG_SENT = 0x5EED                                     # flag words nobody may write


def _esz(dtype):
    return torch.empty(0, dtype=dtype).element_size()


def _int_dtype(dtype):
    return torch.int32 if _esz(dtype) == 4 else torch.int16


# ------------------------------------------------------------------ one allocation, many guarded destinations

class Arena:
    """`n` guarded (M, ldc) matrices stacked in one sentinel-filled allocation: GUARD_ROWS rows above, between and below
    them, `cl` columns left and at least 8 right of the `width` columns that may be written.  The row pitch and `cl`
    keep every row of every block on 16 bytes."""

    def __init__(self, n, M, width, dtype, cl=8):
        esz = _esz(dtype)
        self.n, self.M, self.width, self.dtype, self.cl = n, M, width, dtype, cl
        ldc = cl + width + 8
        self.ldc = ldc + (-ldc * esz) % 16 // esz
        self.raw = torch.full((GUARD_ROWS + n * (M + GUARD_ROWS), self.ldc), SENT[dtype], dtype=_int_dtype(dtype), device=DEV)
        self.buf = self.raw.view(dtype)

    def refill(self):
        self.raw.fill_(SENT[self.dtype])

    def row0(self, d):
        return GUARD_ROWS + d * (self.M + GUARD_ROWS)

    def block(self, d, c0=0, c1=None):
        """matrix d, columns [c0, c1) of its writable width."""
        r = self.row0(d)
        return self.buf[r:r + self.M, self.cl + c0:self.cl + (self.width if c1 is None else c1)]

    def ptr(self, d, c0=0):
        return self.buf.data_ptr() + (self.row0(d) * self.ldc + self.cl + c0) * _esz(self.dtype)

    def check(self, written, what):
        """nothing outside the blocks `written` = [(d, c0, c1), ...] differs from the sentinel."""
        raw = self.raw.clone()
        for d, c0, c1 in written:
            r = self.row0(d)
            raw[r:r + self.M, self.cl + c0:self.cl + c1] = SENT[self.dtype]
        bad = (raw != SENT[self.dtype]).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.shape[0]} elements written outside the destination blocks, first at " \
                                 f"allocation row {bad[0, 0].item()} col {bad[0, 1].item()} (matrices start at rows " \
                                 f"{[self.row0(d) for d in range(self.n)]}, column {self.cl})"


def assert_block(got, ref_dev, what):
    """device block == device reference bit for bit, with +0 == -0 (compared as float32 bit patterns)."""
    g = (got.float() + 0.0).view(torch.int32)
    r = (ref_dev.float() + 0.0).view(torch.int32)
    if not torch.equal(g, r):
        assert_bits_equal(to_np(got), to_np(ref_dev), what)
        raise AssertionError(what)


def ref_device(ref, odt):
    """the oracle's float32 values (already rounded to the output dtype) on the device, in the output dtype."""
    return torch.from_numpy(np.ascontiguousarray(ref, np.float32)).to(DEV).to(odt)


def launch_count():
    return capi().fp8b_launch_count()


def status(rc):
    return f"status {rc} ({capi().fp8b_status_string(rc).decode()})"


def deltas_table(arena, caller, world, trap=None):
    """device int64 table: entry r < world is the byte offset of matrix r from the caller's.  With `trap`, eight entries,
    those past `world` pointing at the trap matrix, which nothing may write: a read past the table shows as stores there."""
    base = arena.ptr(caller)
    v = [arena.ptr(r) - base for r in range(world)]
    if trap is not None:
        v += [arena.ptr(trap) - base] * (8 - world)
    t = torch.tensor(v, dtype=torch.int64, device=DEV)
    return t, t.clone()


class Operands:
    """A and B on the device (dev_bytes: followed by 0x7E rows) and the epilogue terms; remembers the operand bytes so that
    a call can be checked not to have written them."""

    def __init__(self, A, B, t):
        self.A, self.B, self.t = A, B, t.device()
        self.M, self.K = A.shape
        self.N = B.shape[0]
        self.tA, self.pA = dev_bytes(A)
        self.tB, self.pB = dev_bytes(B)
        self.a0, self.b0 = self.tA.clone(), self.tB.clone()

    def ref(self, odt):
        t = self.t
        return ref_device(oracle(self.A, self.B, t.sa, t.sb, t.bias, t.sr, odt), odt)

    def unchanged(self):
        return torch.equal(self.tA, self.a0) and torch.equal(self.tB, self.b0)

    def peers(self, odt, C_local, deltas, world, ldc, over=None):
        """fp8b_scaled_mm_peers; the dict `over` replaces any argument (M, N, K, ldc, world, sb, bias, ...)."""
        t = self.t
        a = dict(A=self.pA, B=self.pB, C=C_local, deltas=p(deltas) if isinstance(deltas, torch.Tensor) else deltas, world=world,
                 odt=dt_code(odt), M=self.M, N=self.N, K=self.K, ldc=ldc, sa=p(t.t_sa), sa_len=len(t.sa), sb=p(t.t_sb),
                 sb_len=len(t.sb), bias=p(t.t_bias), bias_dt=dt_code(t.bias_dt) if t.bias_dt is not None else 0, sr=p(t.t_sr))
        a.update(over or {})
        return capi().fp8b_scaled_mm_peers(*a.values(), stream_ptr())


def families(M, K, N, rng):
    """(name, A, B) of one-hot A with NaN bytes in B, one-hot B and few-hot small integers (test_gpu_exact.py)."""
    pos = edges(K, tc_bounds(K), rng)
    A1 = one_hot(M, K, pos, rng)
    B1 = add_nan_rows(codes((N, K), rng), A1, [2, N // 2 + 1, N - 1], rng)
    return [("one-hot A", A1, B1), ("one-hot B", codes((M, K), rng), one_hot(N, K, pos, rng)),
            ("few-hot", few_hot(M, K, pos, rng), small_ints((N, K), rng))]


def peers_case(ops, odt, world, caller, n0, what):
    """One fp8b_scaled_mm_peers call: `world` destinations and a trap matrix in one arena, C_local at column n0 > 0 of
    the caller's matrix.  Every destination block equals the oracle; the sentinels, the delta table and the operands are
    intact; one launch."""
    M, N = ops.M, ops.N
    ar = Arena(world + 1, M, n0 + N + 40, odt)
    deltas, deltas0 = deltas_table(ar, caller, world, trap=world)
    n_launch = launch_count()
    rc = ops.peers(odt, ar.ptr(caller, n0), deltas, world, ar.ldc)
    torch.cuda.synchronize()
    what = f"{what} M{M} N{N} K{ops.K} {dt_name(odt)} world {world} caller {caller} n0 {n0}"
    assert rc == OK, f"{what}: {status(rc)}"
    assert launch_count() == n_launch + 1, what
    ref = ops.ref(odt)
    for d in range(world):
        assert_block(ar.block(d, n0, n0 + N), ref, f"{what}: destination {d}")
    ar.check([(d, n0, n0 + N) for d in range(world)], what)
    assert torch.equal(deltas, deltas0), f"{what}: delta table written"
    assert ops.unchanged(), f"{what}: operands written"


# ------------------------------------------------------------------ 1. peer stores, exact

ODTS = (torch.bfloat16, torch.float32, torch.float16)
WORLD_CALLER = ((2, 0), (3, 1), (8, 5))               # caller's zero delta first, or in the middle (deltas of both signs)


@pytest.mark.parametrize("cfg", [3, 4, 5, -1])
def test_peers_exact(tune, cfg):
    """GEMM_CFG 3 / 4 / 5 and the built-in choice, ragged M (300) and N = 1056 (a multiple of 32, not of the tile width:
    the last tile's right edge takes the unstaged per-lane store), a K tail; one-hot A with NaN bytes in B, one-hot B,
    few-hot; the three output dtypes; every epilogue-term combination over the four configurations (Terms.cycle)."""
    tune("GEMM_CFG", cfg)
    M, K, N = 300, 400, 1056
    ci = (3, 4, 5, -1).index(cfg)
    rng = np.random.default_rng(100 + ci)
    for i, (fam, A, B) in enumerate(families(M, K, N, rng)):
        world, caller = WORLD_CALLER[i]
        ops = Operands(A, B, Terms.cycle(4 * ci + i, M, N, rng))
        peers_case(ops, ODTS[(i + ci) % 3], world, caller, n0=32 * (1 + i), what=f"cfg {cfg} {fam}")


def split_wave(M, N, BN):
    """(tiles, remainder, split) of the last-wave rule of launch_tcgen05_cfg (fp8_gemm_tcgen05.cu) for a CTA-pair tile
    configuration: a partial last wave of at most half the pairs runs as twice as many half-width tiles."""
    cap = sm_count() // 2
    tiles = -(-M // 256) * -(-N // BN)
    rem = tiles % cap
    return tiles, rem, BN % 64 == 0 and (BN // 4) % 8 == 0 and tiles > cap and 0 < rem and 2 * rem <= cap


@pytest.mark.parametrize("cfg", [3, 4, 5])
def test_peers_split_last_wave_exact(tune, cfg):
    """A split last wave for each pair configuration: M = 2304 (9 row blocks) and the narrowest N = nb * BN - BN / 2 (a
    half-filled last column of tiles) the host rule splits, e.g. 1632 with cfg 5 and 148 SMs: 81 tiles, remainder 7.  The
    96-wide half tiles of cfg 5 with a 16-bit output take the unstaged per-lane store."""
    tune("GEMM_CFG", cfg)
    BN = BN_OF_CFG[cfg]
    M, K = 2304, 256
    N = next(nb * BN - BN // 2 for nb in range(1, 400) if split_wave(M, nb * BN - BN // 2, BN)[2])
    tiles, rem, split = split_wave(M, N, BN)
    assert split and N % 32 == 0, (tiles, rem)
    rng = np.random.default_rng(200 + cfg)
    pos = edges(K, tc_bounds(K), rng)
    A = one_hot(M, K, pos, rng)
    B = add_nan_rows(codes((N, K), rng), A, [1, N - 2], rng)
    odt = torch.bfloat16 if cfg == 5 else (torch.float16 if cfg == 3 else torch.float32)
    peers_case(Operands(A, B, Terms.cycle(9 + cfg, M, N, rng)), odt, 2, 1, n0=64,
               what=f"cfg {cfg} split last wave ({tiles} tiles, remainder {rem})")
    if cfg == 5:
        peers_case(Operands(codes((M, K), rng), one_hot(N, K, pos, rng), Terms.cycle(3, M, N, rng)), torch.float16, 3, 2,
                   n0=32, what=f"cfg {cfg} split last wave one-hot B")


# ------------------------------------------------------------------ 2. peer stores vs. the direct kernel, random bytes

def _rand_codes(shape, seed):
    """uniform bytes over every finite e4m3 code."""
    b = np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)
    b[(b & 0x7F) == 0x7F] = 0x3C
    return b


@pytest.mark.parametrize("M,K,N,odt,world,ldc,n0", [
    (4096, 3072, 1536, torch.bfloat16, 8, 12288, 3072),         # C4's w = 8 shard
    (700, 512, 1056, torch.float32, 3, 2200, 544),
])
@pytest.mark.parametrize("cfg", [3, 4, 5])
def test_peers_match_direct_kernel(tune, cfg, M, K, N, odt, world, ldc, n0):
    """With the same pair configuration forced (which also rules out split-K) and the st.global epilogue
    (GEMM_STORE = 1), fp8b_scaled_mm_peers equals fp8b_scaled_mm(TCGEN05) bit for bit on random bytes, in every
    destination: the same accumulation and epilogue arithmetic, only the stores differ."""
    tune("GEMM_CFG", cfg)
    tune("GEMM_STORE", 1)
    rng = np.random.default_rng(cfg)
    ops = Operands(_rand_codes((M, K), M + cfg), _rand_codes((N, K), N + cfg),
                   Terms(M, N, rng, per_row_a=True, per_row_b=cfg != 4, bias_dt=torch.bfloat16 if cfg != 5 else None, sr=cfg == 5))
    t = ops.t
    direct = torch.empty(M, N, dtype=odt, device=DEV)
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    rc = capi().fp8b_scaled_mm(ops.pA, ops.pB, direct.data_ptr(), dt_code(odt), M, N, K, N, p(t.t_sa), len(t.sa), p(t.t_sb),
                               len(t.sb), p(t.t_bias), bc, p(t.t_sr), None, 0, ALGO_TCGEN05, stream_ptr())
    assert rc == OK, status(rc)
    ar = Arena(world, M, ldc - 16, odt)
    assert ar.ldc == ldc
    deltas, _ = deltas_table(ar, world // 2, world)
    rc = ops.peers(odt, ar.ptr(world // 2, n0), deltas, world, ar.ldc)
    torch.cuda.synchronize()
    assert rc == OK, status(rc)
    what = f"cfg {cfg} M{M} N{N} K{K} {dt_name(odt)}"
    for d in range(world):
        assert torch.equal(ar.block(d, n0, n0 + N).view(_int_dtype(odt)), direct.view(_int_dtype(odt))), \
            f"{what}: destination {d} != fp8b_scaled_mm"
    ar.check([(d, n0, n0 + N) for d in range(world)], what)


# ------------------------------------------------------------------ 3. deltas beyond 32 bits

def test_peers_deltas_beyond_32_bits():
    """Three destinations in one arena of 4 GiB + 7 MiB: lo at 1 MiB, mid at 3 MiB, hi at 4 GiB + 5 MiB.  Called from each
    of them, the deltas reach past 2^32 in both directions.  A delta cut to 32 bits would land 2, 4 MiB after lo or mid
    or 2, 4 MiB before hi: inside the arena, on sentinels, which are checked over the whole arena on the device."""
    M, K, N = 300, 256, 256
    odt = torch.bfloat16
    cl, ldc = 8, 272
    U = 1 << 20
    rows = M + 2 * GUARD_ROWS
    assert rows * ldc * 2 < U
    total = (1 << 32) + 7 * U
    free, _ = torch.cuda.mem_get_info()
    if free < total + (3 << 30):
        pytest.skip(f"needs {(total + (3 << 30)) / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    offs = [U, 3 * U, (1 << 32) + 5 * U]                  # byte offsets of the three matrices' first guard row
    arena = torch.full((total // 2,), SENT[odt], dtype=torch.int16, device=DEV)
    base = arena.data_ptr()

    def mat(d):
        return arena[offs[d] // 2:offs[d] // 2 + rows * ldc].view(rows, ldc)

    def c_ptr(d):
        return base + offs[d] + (GUARD_ROWS * ldc + cl) * 2

    rng = np.random.default_rng(32)
    fams = families(M, K, N, rng)
    for caller in range(3):
        fam, A, B = fams[caller]
        ops = Operands(A, B, Terms.cycle(5 + caller, M, N, rng))
        if caller:
            arena.fill_(SENT[odt])
        deltas = torch.tensor([c_ptr(d) - c_ptr(caller) for d in range(3)], dtype=torch.int64, device=DEV)
        far = [int(v) for v in deltas.cpu() if abs(int(v)) > 1 << 32]
        assert len(far) == (2 if caller == 2 else 1)
        rc = ops.peers(odt, c_ptr(caller), deltas, 3, ldc)
        torch.cuda.synchronize()
        what = f"caller {caller} ({fam}), deltas {deltas.tolist()}"
        assert rc == OK, f"{what}: {status(rc)}"
        ref = ops.ref(odt)
        for d in range(3):
            blk = mat(d)[GUARD_ROWS:GUARD_ROWS + M, cl:cl + N]
            assert_block(blk.view(odt), ref, f"{what}: destination {d}")
            blk.fill_(SENT[odt])
        step = 1 << 28
        for s in range(0, arena.numel(), step):
            n_bad = int(torch.count_nonzero(arena[s:s + step] != SENT[odt]))
            assert n_bad == 0, f"{what}: {n_bad} elements written outside the destinations in arena bytes [{2 * s}, {2 * s + 2 * step})"
    del arena
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ 4. / 5. the exchange, emulated on one GPU

class Exchange:
    """An N-sharded linear over `world` emulated ranks: rank r owns B rows / output columns shard_bounds(N, world, r,
    align), with the matching slices of a per-row scale_b and of the bias, and writes its column block into the (M, N)
    buffer of every rank -- matrix r of one arena."""

    def __init__(self, A, B, t, odt, world, align):
        self.ops = Operands(A, B, t)
        self.odt, self.world = odt, world
        self.M, self.K = A.shape
        self.N = B.shape[0]
        self.ar = Arena(world, self.M, self.N, odt)
        self.shards = []
        for r in range(world):
            n0, n1, _ = shard_bounds(self.N, world, r, align)
            tB, pB = dev_bytes(B[n0:n1])
            sb = dev_f32(t.sb if len(t.sb) == 1 else t.sb[n0:n1])
            bias = dev_bias(t.bias_raw[n0:n1], t.bias_dt)[0] if t.bias_dt is not None else None
            self.shards.append((n0, n1, tB, pB, sb, bias))

    def widths(self):
        return [n1 - n0 for n0, n1, *_ in self.shards]

    def run(self, mode, epoch=None, flags=None, counters=None):
        """the W calls of one exchange; mode "peers", "push" or "push_signal" (flags: (world, 16) int64, counters:
        (world, 4) int32, one row per rank)."""
        L, t, ar, W = capi(), self.ops.t, self.ar, self.world
        bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
        n_launch = launch_count()
        for r, (n0, n1, tB, pB, sb, bias) in enumerate(self.shards):
            common = (dt_code(self.odt), self.M, n1 - n0, self.K, ar.ldc, p(t.t_sa), len(t.sa), p(sb), 1 if len(t.sb) == 1 else n1 - n0,
                      p(bias), bc, p(t.t_sr))
            if mode == "peers":
                deltas, _ = deltas_table(ar, r, W)
                rc = L.fp8b_scaled_mm_peers(self.ops.pA, pB, ar.ptr(r, n0), p(deltas), W, *common, stream_ptr())
            else:
                order = [(r + d) % W for d in range(W)]          # own buffer first, then the ring (fp8_sharded._push_order)
                dsts = (ctypes.c_void_p * W)(*[ar.ptr(j, n0) for j in order])
                if mode == "push":
                    rc = L.fp8b_scaled_mm_push(self.ops.pA, pB, dsts, W, *common, stream_ptr())
                else:
                    sig = (ctypes.c_void_p * W)(*[None if j == r else flags[j, r:].data_ptr() for j in order])
                    rc = L.fp8b_scaled_mm_push_signal(self.ops.pA, pB, dsts, W, *common, sig, counters[r].data_ptr(), epoch,
                                                      stream_ptr())
            assert rc == OK, f"{mode} world {W} rank {r}: {status(rc)}"
        torch.cuda.synchronize()
        assert launch_count() == n_launch + W

    def check(self, ref, what):
        for d in range(self.world):
            assert_block(self.ar.block(d), ref, f"{what}: buffer of rank {d}")
        self.ar.check([(d, 0, self.N) for d in range(self.world)], what)
        assert self.ops.unchanged(), f"{what}: operands written"


EXCHANGES = {          # world, N, shard alignment, output dtype; every shard nonempty, the last one shorter
    2: (416, 32, torch.bfloat16),          # shards 224 / 192 columns (224 bf16 = 3.5 boxes of 128 bytes)
    4: (832, 32, torch.float32),           # 224 x 3 / 160
    8: (1728, 32, torch.float16),          # 224 x 7 / 160
}


@pytest.mark.parametrize("world", sorted(EXCHANGES))
def test_exchange_peers_and_push(world):
    """The whole exchange, emulated: W calls, each with its own B, scale_b and bias shard, all writing into the same W
    buffers.  Afterwards every buffer equals the oracle of the unsharded problem, first with fp8b_scaled_mm_peers (delta
    tables), then with fp8b_scaled_mm_push (destination lists) in re-filled buffers; both fill them with the same bits."""
    N, align, odt = EXCHANGES[world]
    M, K = 300, 256
    rng = np.random.default_rng(world)
    fam, A, B = families(M, K, N, rng)[sorted(EXCHANGES).index(world)]
    ex = Exchange(A, B, Terms.cycle(world + 3, M, N, rng), odt, world, align)
    w = ex.widths()
    assert min(w) > 128 and all(x % 32 == 0 for x in w) and w[-1] < w[0], w
    ref = ex.ops.ref(odt)
    ex.run("peers")
    ex.check(ref, f"peers exchange world {world} {fam}")
    peers_bits = ex.ar.raw.clone()
    ex.ar.refill()
    ex.run("push")
    ex.check(ref, f"push exchange world {world} {fam}")
    assert torch.equal(ex.ar.raw, peers_bits), f"world {world}: push and peers exchanges differ"


@pytest.mark.parametrize("world,N", [(2, 296), (4, 776), (8, 1000)])
def test_exchange_push_ragged_shards(world, N):
    """fp8b_scaled_mm_push exchanges with 16-column shard alignment: shard widths that are no multiple of a 128-byte box
    (160 / 136, 208 x 3 / 152, 128 x 7 / 104 columns), so TMA clips a partial box at every shard's right edge."""
    M, K = 333, 384
    rng = np.random.default_rng(N)
    for i, (fam, A, B) in enumerate(families(M, K, N, rng)[:2]):
        odt = (torch.bfloat16, torch.float16)[i]
        ex = Exchange(A, B, Terms.cycle(2 * world + i, M, N, rng), odt, world, 16)
        assert any((x * 2) % 128 for x in ex.widths()), ex.widths()
        ex.run("push")
        ex.check(ex.ops.ref(odt), f"push exchange world {world} N{N} {fam}")


@pytest.mark.parametrize("world", [3, 4, 5, 6, 7, 8])
def test_exchange_push_signal(world):
    """The fused closing barrier at world 3-8: rank r's fp8b_scaled_mm_push_signal stores the epoch into slot r of every
    other rank's flag array; epochs 1, 2, 3 with the buffers re-filled between them.  After the W calls the host checks
    that every peer slot holds the epoch, every own slot and the slots past W are untouched and every CTA counter is 0
    again -- only then is fp8b_peer_wait(world W, rank j) enqueued for every rank, and it must leave the flags alone."""
    M, K = 260, 256
    N = 192 * world - 64
    odt = (torch.bfloat16, torch.float16, torch.float32)[world % 3]
    rng = np.random.default_rng(50 + world)
    fam, A, B = families(M, K, N, rng)[world % 3]
    ex = Exchange(A, B, Terms.cycle(world, M, N, rng), odt, world, 16)
    assert min(ex.widths()) > 0
    ref = ex.ops.ref(odt)
    flags = torch.full((world, 16), FLAG_SENT, dtype=torch.int64, device=DEV)
    counters = torch.zeros(world, 4, dtype=torch.int32, device=DEV)
    L = capi()
    for epoch in (1, 2, 3):
        what = f"push_signal world {world} epoch {epoch} {fam}"
        if epoch > 1:
            ex.ar.refill()
        ex.run("push_signal", epoch, flags, counters)
        f = flags.cpu().numpy()
        want = np.full((world, 16), FLAG_SENT, np.int64)
        want[:, :world] = epoch
        want[np.arange(world), np.arange(world)] = FLAG_SENT
        assert np.array_equal(f, want), f"{what}: flags (row j = rank j's array)\n{f[:, :world]}"
        assert not counters.any(), f"{what}: CTA counters {counters[:, 0].tolist()} not reset"
        ex.check(ref, what)
        for j in range(world):
            assert L.fp8b_peer_wait(flags[j].data_ptr(), world, j, epoch, stream_ptr()) == OK
        torch.cuda.synchronize()
        assert np.array_equal(flags.cpu().numpy(), want), f"{what}: fp8b_peer_wait changed the flags"


# ------------------------------------------------------------------ 6. refusals

def test_peers_refusals(tune):
    """Every documented refusal of fp8b_scaled_mm_peers returns its status with no launch and nothing written:
    FP8B_ERR_UNSUPPORTED for N % 32 != 0, C / ldc / per-row scale_b / bias off the 16-byte path, M <= 128 or N <= 128
    under the built-in tile rule, GEMM_CFG 1 or 2, K % 16 != 0 and K == 0; FP8B_ERR_INVALID for a world outside 2..8 and
    a NULL delta table.  M == 0 and N == 0 return FP8B_OK without a launch."""
    M, K, N = 300, 128, 256
    rng = np.random.default_rng(6)
    ops = Operands(codes((M, K), rng), codes((N, K), rng), Terms(M, N, rng, per_row_b=True, bias_dt=torch.float16))
    odt = torch.bfloat16
    ar = Arena(3, M, N + 32, odt)
    deltas, deltas0 = deltas_table(ar, 0, 2, trap=2)
    C = ar.ptr(0, 16)
    t = ops.t
    cases = [
        ("N % 32 != 0", ERR_UNSUPPORTED, dict(N=240, sb_len=240)),
        ("C off 16 bytes", ERR_UNSUPPORTED, dict(C=C + 2)),
        ("ldc * 2 % 16 != 0", ERR_UNSUPPORTED, dict(ldc=ar.ldc - 1)),
        ("per-row scale_b off 16 bytes", ERR_UNSUPPORTED, dict(sb=t.t_sb.data_ptr() + 4)),
        ("bias off 16 bytes", ERR_UNSUPPORTED, dict(bias=t.t_bias.data_ptr() + 2)),
        ("M <= 128, built-in tiles", ERR_UNSUPPORTED, dict(M=128, sa_len=1)),
        ("N <= 128, built-in tiles", ERR_UNSUPPORTED, dict(N=128, sb_len=1)),
        ("K % 16 != 0", ERR_UNSUPPORTED, dict(K=120)),
        ("K == 0", ERR_UNSUPPORTED, dict(K=0)),
        ("world 1", ERR_INVALID, dict(world=1)),
        ("world 9", ERR_INVALID, dict(world=9)),
        ("world 0", ERR_INVALID, dict(world=0)),
        ("NULL delta table", ERR_INVALID, dict(deltas=None)),
        ("M == 0", OK, dict(M=0)),
        ("N == 0", OK, dict(N=0)),
        ("M == N == 0", OK, dict(M=0, N=0)),
    ]
    for cfg in (-1, 1, 2):
        tune("GEMM_CFG", cfg)
        for what, expect, over in (cases if cfg == -1 else [(f"GEMM_CFG {cfg}", ERR_UNSUPPORTED, {})]):
            n_launch = launch_count()
            rc = ops.peers(odt, C, deltas, 2, ar.ldc, over)
            torch.cuda.synchronize()
            assert rc == expect, f"{what}: {status(rc)}, expected {expect}"
            assert launch_count() == n_launch, f"{what}: launched"
            ar.check([], what)
    assert torch.equal(deltas, deltas0) and ops.unchanged()


@pytest.mark.parametrize("cfg", [3, 4, 5])
def test_peers_forced_pair_config_small_extents(tune, cfg):
    """A forced CTA-pair configuration serves M <= 128 and N <= 128 too (the header's M > 128, N > 128 is the built-in
    tile rule's): M = 77 (the second CTA of the pair has no rows), M = 128, N = 96, exact."""
    tune("GEMM_CFG", cfg)
    rng = np.random.default_rng(70 + cfg)
    for i, (M, N) in enumerate(((77, 256), (128, 320), (300, 96))):
        K = 144
        fam, A, B = families(M, K, N, rng)[(i + cfg) % 3]
        peers_case(Operands(A, B, Terms.cycle(i + 3 * cfg, M, N, rng)), ODTS[i], 2 + i, i, n0=16 * (i + 1),
                   what=f"forced cfg {cfg} {fam}")


# ------------------------------------------------------------------ 7. the Python binding

def test_python_binding_peers():
    """fp8_mps_native's fp8_scaled_mm_peers: a local (M, full_N) `out`, a column block at n0 > 0, an fp16 bias and a device
    delta table pointing at a second buffer; both are views of one sentinel-filled allocation.  Both buffers hold the
    oracle block, and nothing else changes."""
    import fp8_mps_native
    lib = fp8_mps_native._get_lib()
    M, K, N, full_N, n0 = 300, 256, 544, 1200, 320
    odt = torch.bfloat16
    rng = np.random.default_rng(7)
    fam, A, B = families(M, K, N, rng)[0]
    t = Terms(M, N, rng, per_row_a=True, per_row_b=True, bias_dt=torch.float16)
    bias = torch.from_numpy(t.bias_raw).to(torch.float16)
    t.bias = bias.float().numpy()
    big = torch.full((3 * GUARD_ROWS + 2 * M, full_N), SENT[odt], dtype=torch.int16, device=DEV)
    rows = (GUARD_ROWS, 2 * GUARD_ROWS + M)
    out, second = (big[r:r + M].view(odt) for r in rows)
    deltas = torch.tensor([0, second.data_ptr() - out.data_ptr()], dtype=torch.int64, device=DEV)
    lib.fp8_scaled_mm_peers(torch.from_numpy(A).to(DEV), torch.from_numpy(B).to(DEV), torch.from_numpy(t.sa).to(DEV),
                            torch.from_numpy(t.sb).to(DEV), bias.to(DEV), out, deltas, n0)
    torch.cuda.synchronize()
    ref = ref_device(oracle(A, B, t.sa, t.sb, t.bias, None, odt), odt)
    for name, buf in (("out", out), ("second buffer", second)):
        assert_block(buf[:, n0:n0 + N], ref, f"binding {fam}: {name}")
    raw = big.clone()
    for r in rows:
        raw[r:r + M, n0:n0 + N] = SENT[odt]
    assert bool((raw == SENT[odt]).all()), "binding: written outside the column block of the two buffers"
