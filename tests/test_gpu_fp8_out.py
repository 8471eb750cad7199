"""FP8 (e4m3fn) matmul output: out_dtype FP8B_OUT_E4M3FN, encoded in the fused epilogue of every kernel.

C[m,n] = enc(v) where v is the fp32 value the same call computes for float32 output and enc is the reference encoder
(fp8b_encode with no prescale).  Every output is an interior view of a buffer filled with 0xFF, the one byte the encoder
never writes, and the sentinels are checked after every call.

  1. self-consistency on random bytes: for every kernel plan, the e4m3fn bytes equal fp8b_encode of the same call's
     float32 output;
  2. the structured families of _util (one-hot, few-hot, NaN bytes in B) and e5m2 operands equal encode(oracle);
  3. every fp32 input of tests/golden/codec_golden.npz, plus NaNs, fed through the epilogue as the bias with A = 0, gives
     the golden bytes in every kernel family (saturation, flush, no-carry rounding, -0.0 and NaN inside the epilogue);
  4. the documented refusals, which return their status and launch nothing;
  5. torch._scaled_mm(..., out_dtype=torch.float8_e4m3fn) under the patch and the Python bindings."""
import ctypes

import numpy as np
import pytest
import torch

from _util import (ALGO_AUTO, ALGO_GEMV, ALGO_SIMT, ALGO_TCGEN05, BF16, E4M3, E5M2, F32, GUARD_ROWS, GemvItem, Out,
                   Terms, add_nan_rows, capi, codes, dev_bytes, dev_f32, dt_code, edges, few_hot, make_spans, one_hot,
                   oracle, p, sm_count, small_ints, stream_ptr, tc_bounds)
import fp8_oracle as o  # noqa: E402  (_util puts oracle/ on the path)

pytestmark = pytest.mark.gpu
DEV = "cuda"
FP8 = torch.float8_e4m3fn
OUT_E4M3FN = 3                                         # fp8b_dtype FP8B_OUT_E4M3FN (include/fp8_b200.h)
OK, ERR_INVALID, ERR_UNSUPPORTED = 0, -1, -2
BIAS_DTS = (torch.float32, torch.float16, torch.bfloat16)
CFG_WIDTH = {1: 256, 2: 128, 3: 256, 4: 128, 5: 192}
CFG_PAIR = {1: False, 2: False, 3: True, 4: True, 5: True}


def u8(t):
    return t.view(torch.uint8)


def code(odt):
    """fp8b_dtype of an output dtype."""
    return OUT_E4M3FN if odt == FP8 else dt_code(odt)


class Out8(Out):
    """_util.Out for e4m3fn bytes: C is an interior view of a buffer filled with 0xFF, the one byte the encoder never
    writes.  aligned=True keeps C and ldc on 16 bytes; False shifts C by one byte and makes ldc odd."""

    def __init__(self, M, N, aligned=True):
        self.dtype, self.M, self.N = torch.uint8, M, N
        self.cl = 16 if aligned else 1
        ldc = self.cl + N + 8
        self.ldc = ldc + (-ldc) % 16 if aligned else ldc | 1
        self.buf = torch.full((M + 2 * GUARD_ROWS, self.ldc), 0xFF, dtype=torch.uint8, device=DEV)
        self.view = self.buf[GUARD_ROWS:GUARD_ROWS + M, self.cl:self.cl + N]

    def check_guard(self, what, interior_written=True):
        raw = self.buf.clone()
        if interior_written:
            raw[GUARD_ROWS:GUARD_ROWS + self.M, self.cl:self.cl + self.N] = 0xFF
        bad = (raw != 0xFF).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.shape[0]} bytes written outside C, first at buffer {bad[0].tolist()}"


def out_of(M, N, odt, aligned=True):
    return Out8(M, N, aligned) if odt == FP8 else Out(M, N, odt, aligned=aligned)


def oracle8(A, B, t, fmts=(E4M3, E4M3)):
    """encode of the oracle's float32 result (fp64 sum): the bytes the reference's .to(float8_e4m3fn) gives."""
    return o.encode(oracle(A, B, t.sa, t.sb, t.bias, t.sr, torch.float32, fmts))


def launches():
    return capi().fp8b_launch_count()


def status(rc):
    return f"status {rc} ({capi().fp8b_status_string(rc).decode()})"


def terms(kind, M, N, rng, per_row_a=False):
    """kind bit 0: per-row scale_b, bit 1: a bias (dtype rotating with kind), bit 2: scale_result -- the eight
    combinations the tcgen05 epilogues specialise on."""
    return Terms(M, N, rng, per_row_a=per_row_a, per_row_b=bool(kind & 1),
                 bias_dt=BIAS_DTS[kind % 3] if kind & 2 else None, sr=bool(kind & 4)).device()


def call_mm(pA, pB, M, N, K, t, odt, out, algo=ALGO_AUTO, fmts=None):
    L = capi()
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    args = (out.ptr, code(odt), M, N, K, out.ldc, p(t.t_sa), len(t.sa), p(t.t_sb), len(t.sb), p(t.t_bias), bc, p(t.t_sr))
    if fmts is None:
        return L.fp8b_scaled_mm(pA, pB, *args, None, 0, algo, stream_ptr())
    return L.fp8b_scaled_mm_fmt(pA, fmts[0], pB, fmts[1], *args, algo, stream_ptr())


def encode_dev(x):
    """fp8b_encode (no prescale) of a float32 device tensor."""
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=torch.uint8, device=DEV)
    assert capi().fp8b_encode(p(x), F32, p(out), x.numel(), None, stream_ptr()) == OK
    return out


def assert_bytes(got, ref, what):
    """uint8 device tensor == reference bytes (numpy or device)."""
    ref = torch.as_tensor(np.ascontiguousarray(ref)).to(DEV) if isinstance(ref, np.ndarray) else ref
    ref = ref.expand_as(got)
    if not torch.equal(got, ref):
        bad = (got != ref).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{what}: {bad.shape[0]} of {got.numel()} bytes differ; first at {list(i)}: "
                             f"got 0x{int(got[i]):02X} want 0x{int(ref[i]):02X}")


def run8(A, B, t, algo=ALGO_AUTO, aligned=True, fmts=None, exact=False, what="", dAB=None):
    """One call with e4m3fn output and the same call with float32 output, both into guarded buffers: the bytes equal
    fp8b_encode of the float32 result and, with exact=True, encode(oracle f64 result)."""
    M, K = A.shape
    N = B.shape[0]
    (tA, pA), (tB, pB) = dAB or (dev_bytes(A), dev_bytes(B))
    o8, of = Out8(M, N, aligned), Out(M, N, torch.float32, aligned=aligned)
    what = f"{what} M{M} N{N} K{K} algo {algo} {'aligned' if aligned else 'shifted'}"
    rc = call_mm(pA, pB, M, N, K, t, FP8, o8, algo, fmts)
    torch.cuda.synchronize()
    assert rc == OK, f"{what}: {status(rc)}"
    o8.check_guard(what)
    rc = call_mm(pA, pB, M, N, K, t, torch.float32, of, algo, fmts)
    torch.cuda.synchronize()
    assert rc == OK, f"{what} (float32): {status(rc)}"
    assert_bytes(u8(o8.view), encode_dev(of.view), f"{what}: e4m3fn vs fp8b_encode(float32 output)")
    if exact:
        assert_bytes(u8(o8.view), oracle8(A, B, t, fmts or (E4M3, E4M3)), f"{what}: vs oracle")
    return o8


def random_case(M, K, N, seed, kinds=range(8), what="", **kw):
    """random non-NaN operand bytes, the epilogue-term combinations `kinds`, aligned and shifted outputs alternating."""
    rng = np.random.default_rng(seed)
    A, B = codes((M, K), rng), codes((N, K), rng)
    dAB = (dev_bytes(A), dev_bytes(B))
    for i, kind in enumerate(kinds):
        run8(A, B, terms(kind, M, N, rng, per_row_a=bool(i & 1)), aligned=(i % 2 == 0) if "aligned" not in kw else kw["aligned"],
             what=f"{what} kind {kind}", dAB=dAB, **{k: v for k, v in kw.items() if k != "aligned"})


# ------------------------------------------------------------------ 1. every plan, random bytes

@pytest.mark.parametrize("unroll", [2, 4, 8])
def test_gemv_fhfma(tune, unroll):
    """FHFMA GEMV (GEMV_IMPL 1): cluster split-K (N = 40, K = 8192), the panel loop (K = 100000), no split (N = 1200)."""
    tune("GEMV_IMPL", 1)
    tune("GEMV_UNROLL", unroll)
    for M, K, N in ((1, 8192, 40), (3, 100000, 24), (5, 4096, 1200), (16, 1024, 77)):
        random_case(M, K, N, unroll * 100 + M, kinds=(unroll % 8, 7 - unroll % 8), what=f"fhfma unroll {unroll}", algo=ALGO_GEMV)


@pytest.mark.parametrize("batch", [1, 2, 4])
def test_gemv_mma(tune, batch):
    """warp-MMA GEMV (GEMV_IMPL 2), GEMV_BATCH 1 / 2 / 4, one and two 8-row blocks, ragged N."""
    tune("GEMV_IMPL", 2)
    tune("GEMV_BATCH", batch)
    for M in (1, 8, 13):
        random_case(M, 5008, 333, batch * 10 + M, kinds=(M % 8, (M + 3) % 8), what=f"mma batch {batch}", algo=ALGO_GEMV)


@pytest.mark.parametrize("algo", [ALGO_SIMT, ALGO_AUTO])
def test_simt_and_generic(algo):
    """SIMT GEMM (forced, and through AUTO with K % 16 != 0) and the generic GEMV kernel (M <= 16, K % 16 != 0)."""
    random_case(133, 1000 if algo == ALGO_AUTO else 1024, 197, 7 + algo, what="simt", algo=algo)
    random_case(5, 1037, 70, 9 + algo, kinds=(3, 6), what="generic", algo=algo)


@pytest.mark.parametrize("store", [1, 2])
@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
def test_tcgen05_tile_configs(tune, cfg, store):
    """GEMM_CFG 1-5 x GEMM_STORE 1 / 2: N = 1008 (a multiple of 16, not of 32: TMA-storable, ragged last chunk),
    N = 1000 (not TMA-storable: st.global), N = 1056; M ragged; all eight term combinations; shifted outputs take the
    scalar edge path.  GEMM_CFG 5 with GEMM_STORE 2 takes the st.global epilogue (192 bytes is not a whole box)."""
    tune("GEMM_CFG", cfg)
    tune("GEMM_STORE", store)
    for j, N in enumerate((1008, 1000, 1056)):
        random_case(300, 400, N, cfg * 10 + store + j, kinds=range(j, 8, 3) if j else range(8), what=f"cfg {cfg} store {store}",
                    algo=ALGO_TCGEN05, aligned=(j != 2) or store == 2)
    random_case(137, 144, 203, cfg + store, kinds=(5,), what=f"cfg {cfg} store {store} shifted", algo=ALGO_TCGEN05, aligned=False)


def split_wave_m(cfg):
    """M such that the built-in last-wave rule of launch_tcgen05_cfg splits the last wave of 8 tile columns into
    half-width tiles: cols_per_warp 128 / 64 (one-CTA tiles), 128 / 96 / 64 (CTA pairs)."""
    rows = 256 if CFG_PAIR[cfg] else 128
    cap = sm_count() // (2 if CFG_PAIR[cfg] else 1)
    for mt in range(1, 200):
        tiles = mt * 8
        if tiles > cap and 0 < tiles % cap <= cap // 2:
            return mt * rows - 37
    raise AssertionError("no split shape")


@pytest.mark.parametrize("store", [1, 2])
@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
def test_tcgen05_split_last_wave(tune, cfg, store):
    """the split last wave: half-width tiles (96 columns for 256 x 192, 64 for 128-wide tiles) take the unstaged per-lane
    path of the st.global epilogue; the store-ring epilogue splits only where half tiles are whole 128-byte boxes."""
    tune("GEMM_CFG", cfg)
    tune("GEMM_STORE", store)
    N = 8 * CFG_WIDTH[cfg] - 16
    random_case(split_wave_m(cfg), 128, N, cfg * 7 + store, kinds=(cfg % 8, 7 - cfg % 8), what=f"split wave cfg {cfg} store {store}",
                algo=ALGO_TCGEN05, aligned=True)


@pytest.mark.parametrize("split", [2, 4, -1])
def test_tcgen05_split_k(tune, split):
    tune("GEMM_SPLITK", split)
    random_case(32, 3072, 3072, split + 40, kinds=(0, 3, 5, 6), what=f"split-K {split}", algo=ALGO_TCGEN05)
    random_case(77, 2064, 400, split + 41, kinds=(1, 2, 4, 7), what=f"split-K {split}", algo=ALGO_TCGEN05)
    random_case(77, 2064, 390, split + 42, kinds=(7,), what=f"split-K {split} ragged", algo=ALGO_TCGEN05, aligned=False)


def test_gemv_batch(tune):
    """fp8b_gemv_batch with e4m3fn output: every y_i equals fp8b_encode of the float32 batch's y_i."""
    K = 3072
    rng = np.random.default_rng(5)
    Ns = [40, 0, 1, 77, 8, 300, 5, 16, 9, 64, 3, 200, 33, 48, 2, 17, 100, 7]
    L = capi()
    tW = [torch.from_numpy(codes((N, K), rng)).to(DEV) for N in Ns]
    x = torch.from_numpy(codes((K,), rng)).to(DEV)
    sx = dev_f32([0.0123])
    sw = [dev_f32((rng.random(N if i % 2 else 1) + 0.5) * 0.02) for i, N in enumerate(Ns)]
    bias = [torch.from_numpy(rng.standard_normal(N).astype(np.float32)).to(DEV).to(torch.bfloat16) if i % 3 else None
            for i, N in enumerate(Ns)]
    res = {}
    for odt in (FP8, torch.float32):
        outs = [out_of(1, N, odt) for N in Ns]
        items = (GemvItem * len(Ns))()
        for i, N in enumerate(Ns):
            items[i].x, items[i].W, items[i].y, items[i].N = x.data_ptr(), tW[i].data_ptr(), outs[i].ptr, N
            items[i].scale_x, items[i].scale_w = sx.data_ptr(), sw[i].data_ptr()
            items[i].scale_w_len = N if i % 2 else 1
            items[i].bias = bias[i].data_ptr() if bias[i] is not None else None
        rc = L.fp8b_gemv_batch(items, len(Ns), K, code(odt), BF16, stream_ptr())
        torch.cuda.synchronize()
        assert rc == OK, status(rc)
        for i, o in enumerate(outs):
            o.check_guard(f"gemv_batch item {i}")
        res[odt] = outs
    for i in range(len(Ns)):
        assert_bytes(u8(res[FP8][i].view), encode_dev(res[torch.float32][i].view), f"gemv_batch item {i} N {Ns[i]}")


@pytest.mark.parametrize("M,plan,ws", [(1, 1, True), (3, 2, True), (4, -1, True), (16, -1, False), (5, 1, False),
                                       (40, -1, True)])
def test_linear_dynamic(tune, M, plan, ws):
    """fp8b_linear_dynamic (DYNAMIC_PLAN 1 / 2, with and without a workspace; M > 16 through the GEMM) with e4m3fn
    output equals fp8b_encode of its float32 output."""
    tune("DYNAMIC_PLAN", plan)
    K, N = 2048, 272
    rng = np.random.default_rng(M * 3 + plan)
    X = torch.from_numpy(rng.standard_normal((M, K)).astype(np.float32)).to(DEV).to(torch.bfloat16)
    B = torch.from_numpy(codes((N, K), rng)).to(DEV)
    sb = dev_f32((rng.random(N) + 0.5) * 0.02)
    bias = torch.from_numpy(rng.standard_normal(N).astype(np.float32)).to(DEV)
    sr = dev_f32([1.25])
    L = capi()
    res = {}
    for odt in (FP8, torch.float32):
        out = out_of(M, N, odt)
        wsb = L.fp8b_linear_dynamic_workspace_bytes(M, K) if ws else 0
        wst = torch.empty(max(wsb, 16), dtype=torch.uint8, device=DEV)
        rc = L.fp8b_linear_dynamic(p(X), BF16, p(B), out.ptr, code(odt), M, N, K, out.ldc, p(sb), N, p(bias), F32, p(sr),
                                   None, p(wst) if ws else None, wsb, stream_ptr())
        torch.cuda.synchronize()
        assert rc == OK, status(rc)
        out.check_guard(f"linear_dynamic M {M} plan {plan} ws {ws}")
        res[odt] = out
    assert_bytes(u8(res[FP8].view), encode_dev(res[torch.float32].view), f"linear_dynamic M {M} plan {plan} ws {ws}")


# ------------------------------------------------------------------ push and peers (one GPU, one sentinel arena)

class Arena:
    """`n` guarded (M, ldc) byte matrices in one 0xFF-filled allocation, GUARD_ROWS rows above, between and below them."""

    def __init__(self, n, M, width, cl=16):
        self.n, self.M, self.cl = n, M, cl
        self.ldc = -(-(cl + width + 16) // 16) * 16
        self.raw = torch.full((GUARD_ROWS + n * (M + GUARD_ROWS), self.ldc), 0xFF, dtype=torch.uint8, device=DEV)

    def row0(self, d):
        return GUARD_ROWS + d * (self.M + GUARD_ROWS)

    def block(self, d, c0, c1):
        r = self.row0(d)
        return self.raw[r:r + self.M, self.cl + c0:self.cl + c1]

    def ptr(self, d, c0=0):
        return self.raw.data_ptr() + self.row0(d) * self.ldc + self.cl + c0

    def check(self, written, what):
        raw = self.raw.clone()
        for d, c0, c1 in written:
            r = self.row0(d)
            raw[r:r + self.M, self.cl + c0:self.cl + c1] = 0xFF
        bad = (raw != 0xFF).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.shape[0]} bytes written outside the destination blocks, first at {bad[0].tolist()}"


def plain_ref(pA, pB, M, N, K, t):
    """the plain call's float32 output, encoded (one CTA per tile: the push / peer kernels never split K)."""
    of = Out(M, N, torch.float32)
    L = capi()
    saved = L.fp8b_get_option(25)
    L.fp8b_set_option(25, 1)
    try:
        rc = call_mm(pA, pB, M, N, K, t, torch.float32, of, ALGO_TCGEN05)
    finally:
        L.fp8b_set_option(25, saved)
    torch.cuda.synchronize()
    assert rc == OK, status(rc)
    return encode_dev(of.view)


def push_call(pA, pB, M, N, K, t, ptrs, ldc):
    bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
    arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
    return capi().fp8b_scaled_mm_push(pA, pB, arr, len(ptrs), OUT_E4M3FN, M, N, K, ldc, p(t.t_sa), len(t.sa), p(t.t_sb),
                                      len(t.sb), p(t.t_bias), bc, p(t.t_sr), stream_ptr())


@pytest.mark.parametrize("cfg", [-1, 1, 2, 3, 4])
def test_push(tune, cfg):
    """fp8b_scaled_mm_push with 1..8 destinations in one arena, each at column offset n0 (a multiple of 16); every
    destination equals the encoded plain result and nothing else is written."""
    tune("GEMM_CFG", cfg)
    rng = np.random.default_rng(60 + cfg)
    M, K, N = 300, 400, 1008
    A, B = codes((M, K), rng), codes((N, K), rng)
    (tA, pA), (tB, pB) = dev_bytes(A), dev_bytes(B)
    for n_dst in range(1, 9):
        t = terms(n_dst % 8, M, N, rng, per_row_a=bool(n_dst & 1))
        ref = plain_ref(pA, pB, M, N, K, t)
        n0 = 16 * (n_dst % 3)
        ar = Arena(n_dst, M, n0 + N)
        n_launch = launches()
        rc = push_call(pA, pB, M, N, K, t, [ar.ptr(d, n0) for d in range(n_dst)], ar.ldc)
        torch.cuda.synchronize()
        what = f"push cfg {cfg} n_dst {n_dst} n0 {n0}"
        assert rc == OK, f"{what}: {status(rc)}"
        assert launches() == n_launch + 1, what
        for d in range(n_dst):
            assert_bytes(ar.block(d, n0, n0 + N), ref, f"{what} destination {d}")
        ar.check([(d, n0, n0 + N) for d in range(n_dst)], what)


@pytest.mark.parametrize("cfg", [3, 4, 5, -1])
def test_peers(tune, cfg):
    """fp8b_scaled_mm_peers at W = 2 / 3 / 8 emulated on one GPU: every destination of one arena equals the encoded plain
    result; N = 1056 (the last tile's right edge takes the unstaged per-lane store)."""
    tune("GEMM_CFG", cfg)
    rng = np.random.default_rng(70 + cfg)
    M, K, N = 300, 400, 1056
    A, B = codes((M, K), rng), codes((N, K), rng)
    A1 = one_hot(M, K, edges(K, tc_bounds(K), rng), rng)
    B1 = add_nan_rows(codes((N, K), rng), A1, [2, N // 2 + 1, N - 1], rng)
    for i, (world, caller) in enumerate(((2, 0), (3, 1), (8, 5))):
        AA, BB = (A1, B1) if i == 1 else (A, B)
        (tA, pA), (tB, pB) = dev_bytes(AA), dev_bytes(BB)
        t = terms((3 * i + cfg) % 8, M, N, rng, per_row_a=bool(i & 1))
        ref = plain_ref(pA, pB, M, N, K, t)
        n0 = 32 * (1 + i)
        ar = Arena(world, M, n0 + N + 32)
        base = ar.ptr(caller)
        deltas = torch.tensor([ar.ptr(r) - base for r in range(world)], dtype=torch.int64, device=DEV)
        bc = dt_code(t.bias_dt) if t.bias_dt is not None else 0
        n_launch = launches()
        rc = capi().fp8b_scaled_mm_peers(pA, pB, ar.ptr(caller, n0), p(deltas), world, OUT_E4M3FN, M, N, K, ar.ldc, p(t.t_sa),
                                         len(t.sa), p(t.t_sb), len(t.sb), p(t.t_bias), bc, p(t.t_sr), stream_ptr())
        torch.cuda.synchronize()
        what = f"peers cfg {cfg} world {world} caller {caller}"
        assert rc == OK, f"{what}: {status(rc)}"
        assert launches() == n_launch + 1, what
        for d in range(world):
            assert_bytes(ar.block(d, n0, n0 + N), ref, f"{what} destination {d}")
        ar.check([(d, n0, n0 + N) for d in range(world)], what)
        if i == 1:
            assert_bytes(ar.block(0, n0, n0 + N), oracle8(AA, BB, t), f"{what}: vs oracle")


# ------------------------------------------------------------------ 2. structured inputs against the oracle

PLANS = {"fhfma": (3, ALGO_GEMV, ("GEMV_IMPL", 1)), "mma": (9, ALGO_GEMV, ("GEMV_IMPL", 2)), "simt": (133, ALGO_SIMT, None),
         "tcgen05": (300, ALGO_TCGEN05, None), "split-K": (32, ALGO_TCGEN05, ("GEMM_SPLITK", 4)),
         "cfg5": (300, ALGO_TCGEN05, ("GEMM_CFG", 5))}


@pytest.mark.parametrize("plan", sorted(PLANS))
def test_structured_families_exact(tune, plan):
    """one-hot A with NaN bytes in B, one-hot B, few-hot small integers: encode(oracle f64) exactly."""
    M, algo, knob = PLANS[plan]
    if knob:
        tune(*knob)
    K, N = 1024, 400
    rng = np.random.default_rng(len(plan) * 11 + M)
    pos = edges(K, tc_bounds(K) | set(range(64, K, 64)), rng)
    A1 = one_hot(M, K, pos, rng)
    fams = [("one-hot A", A1, add_nan_rows(codes((N, K), rng), A1, [2, N - 1], rng)),
            ("one-hot B", codes((M, K), rng), one_hot(N, K, pos, rng)),
            ("few-hot", few_hot(M, K, pos, rng), small_ints((N, K), rng))]
    for i, (fam, A, B) in enumerate(fams):
        run8(A, B, terms((3 * i + M) % 8, M, N, rng, per_row_a=bool(i & 1)), algo, aligned=(i != 2), exact=True,
             what=f"{plan} {fam}")


@pytest.mark.parametrize("fmts", [(E5M2, E4M3), (E4M3, E5M2), (E5M2, E5M2)])
@pytest.mark.parametrize("M,K,N", [(3, 2048, 100), (150, 512, 264)])
def test_e5m2_operands_exact(fmts, M, K, N):
    """fp8b_scaled_mm_fmt with e5m2 operands: one-hot rows whose nonzero is sometimes +-inf or NaN (e5m2 keeps them), so
    outputs are +-inf (-> 0x7E / 0xFE), NaN (-> 0x7F) and finite values, equal to encode(oracle)."""
    rng = np.random.default_rng(M + 3 * fmts[0] + fmts[1])
    fa, fb = fmts
    pos = edges(K, tc_bounds(K), rng)
    A = one_hot(M, K, pos, rng, fa)
    B = codes((N, K), rng, fb)
    if fa == E5M2:
        nz = A.argmax(1)
        A[np.arange(M), nz] = np.where(np.arange(M) % 3 == 0, 0x7C, np.where(np.arange(M) % 3 == 1, 0xFC, A[np.arange(M), nz]))
        A[1 % M, nz[1 % M]] = 0x7D
        B[:, nz[0]] = np.where(np.arange(N) % 7 == 0, 0, B[:, nz[0]])          # inf * 0 = NaN
    else:
        B[0, :], B[1, :] = 0x7C, 0xFE
    t = terms(5, M, N, rng)
    o8 = run8(A, B, t, fmts=fmts, exact=True, what=f"e5m2 {fmts}")
    got = set(np.unique(u8(o8.view).cpu().numpy()).tolist())
    assert ({0x7E, 0xFE, 0x7F} if fa == E5M2 else {0x7F}) <= got, f"e5m2 {fmts}: inf / NaN outputs missing"


# ------------------------------------------------------------------ 3. the encoder's edge cases inside the epilogue

EDGE_PLANS = [("fhfma", 1, ALGO_GEMV, [("GEMV_IMPL", 1)]), ("mma", 4, ALGO_GEMV, [("GEMV_IMPL", 2)]),
              ("simt", 20, ALGO_SIMT, []), ("generic", 2, ALGO_GEMV, [])] + \
             [(f"cfg{c} store{s}", 300, ALGO_TCGEN05, [("GEMM_CFG", c), ("GEMM_STORE", s), ("GEMM_SPLITK", 1)])
              for c in (1, 2, 3, 4, 5) for s in (1, 2)] + \
             [(f"split-K {s}", 100, ALGO_TCGEN05, [("GEMM_SPLITK", s)]) for s in (2, 4)]


@pytest.fixture(scope="module")
def edge_bias(golden):
    """every fp32 input of codec_golden.npz (+-inf and +-0.0 included) and NaNs of both signs and several payloads, padded
    to a multiple of 16 columns, with the expected bytes."""
    x = golden["codec"]["enc_f32_in"].astype(np.float32)
    y = golden["codec"]["enc_f32_out"].astype(np.uint8)
    nan = np.array([0x7FC00000, 0xFFC00000, 0x7F800001, 0xFF800001, 0x7FFFFFFF, 0xFFFFFFFF], np.uint32).view(np.float32)
    n_pad = (-(len(x) + len(nan))) % 16 + 16
    nans = np.resize(nan, len(nan) + n_pad)
    return np.concatenate([x, nans]), np.concatenate([y, np.full(len(nans), 0x7F, np.uint8)])


@pytest.mark.parametrize("plan", [e[0] for e in EDGE_PLANS])
def test_encoder_edges_through_epilogue(tune, edge_bias, plan):
    """A = 0, scales 1: C[m,n] = enc(0 + bias[n]) must be the golden byte of every fp32 input, in every kernel family,
    through aligned and 1-byte-shifted outputs."""
    _, M, algo, knobs = next(e for e in EDGE_PLANS if e[0] == plan)
    for k in knobs:
        tune(*k)
    bias, want = edge_bias
    N = len(bias)
    K = 1037 if plan == "generic" else 512
    A, B = np.zeros((M, K), np.uint8), np.zeros((N, K), np.uint8)
    (tA, pA), (tB, pB) = dev_bytes(A), dev_bytes(B)
    t = Terms(M, N, np.random.default_rng(2))
    t.sa, t.sb, t.bias_dt, t.bias_raw, t.sr = np.ones(1, np.float32), np.ones(1, np.float32), torch.float32, bias, None
    t.device()
    for aligned in (True, False):
        o8 = Out8(M, N, aligned)
        rc = call_mm(pA, pB, M, N, K, t, FP8, o8, algo)
        torch.cuda.synchronize()
        what = f"encoder edges {plan} {'aligned' if aligned else 'shifted'}"
        assert rc == OK, f"{what}: {status(rc)}"
        o8.check_guard(what)
        assert_bytes(u8(o8.view), torch.from_numpy(want).to(DEV).reshape(1, -1), what)


def test_encoder_edges_batch_and_dynamic(edge_bias):
    """the same bias through fp8b_gemv_batch and fp8b_linear_dynamic (X = 0: amax 0, scale 1, every q = 0)."""
    bias, want = edge_bias
    N, K = len(bias), 512
    L = capi()
    tb = torch.from_numpy(bias).to(DEV)
    W = torch.from_numpy(codes((N, K), np.random.default_rng(3))).to(DEV)
    x = torch.zeros(K, dtype=torch.uint8, device=DEV)
    one = dev_f32([1.0])
    out = Out8(1, N)
    items = (GemvItem * 1)()
    items[0].x, items[0].W, items[0].y, items[0].N = x.data_ptr(), W.data_ptr(), out.ptr, N
    items[0].scale_x, items[0].scale_w, items[0].scale_w_len, items[0].bias = one.data_ptr(), one.data_ptr(), 1, tb.data_ptr()
    assert L.fp8b_gemv_batch(items, 1, K, OUT_E4M3FN, F32, stream_ptr()) == OK
    torch.cuda.synchronize()
    out.check_guard("gemv_batch edges")
    assert_bytes(u8(out.view), torch.from_numpy(want).to(DEV).reshape(1, -1), "gemv_batch edges")
    for M in (1, 3, 40):
        X = torch.zeros(M, K, dtype=torch.float32, device=DEV)
        out = Out8(M, N)
        wsb = L.fp8b_linear_dynamic_workspace_bytes(M, K)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        rc = L.fp8b_linear_dynamic(p(X), F32, p(W), out.ptr, OUT_E4M3FN, M, N, K, out.ldc, p(one), 1, p(tb), F32, None, None,
                                   p(ws), wsb, stream_ptr())
        torch.cuda.synchronize()
        assert rc == OK, status(rc)
        out.check_guard(f"linear_dynamic edges M {M}")
        assert_bytes(u8(out.view), torch.from_numpy(want).to(DEV).reshape(1, -1), f"linear_dynamic edges M {M}")


# ------------------------------------------------------------------ 4. refusals

def test_refusals_launch_nothing(tune):
    L = capi()
    s = stream_ptr()
    buf = torch.full((4096,), 0x5A, dtype=torch.uint8, device=DEV)
    buf0 = buf.clone()
    one = dev_f32([1.0])
    scratch = torch.zeros(4, dtype=torch.int32, device=DEV)
    n0 = launches()
    src, dst = p(buf), p(buf[2048:])
    spans = make_spans([(buf.data_ptr(), buf.data_ptr() + 2048, 64)])
    checks = {
        "fp8b_dequant": L.fp8b_dequant(src, dst, OUT_E4M3FN, 64, s),
        "fp8b_dequant_fmt": L.fp8b_dequant_fmt(src, E4M3, dst, OUT_E4M3FN, 64, None, s),
        "fp8b_encode": L.fp8b_encode(src, OUT_E4M3FN, dst, 64, None, s),
        "fp8b_encode_batch": L.fp8b_encode_batch(spans, 1, OUT_E4M3FN, s),
        "fp8b_dequant_batch": L.fp8b_dequant_batch(spans, 1, OUT_E4M3FN, s),
        "fp8b_amax_scale": L.fp8b_amax_scale(src, OUT_E4M3FN, 64, p(one), None, p(scratch), s),
        "fp8b_quantize_rows": L.fp8b_quantize_rows(src, OUT_E4M3FN, 2, 32, dst, p(one), s),
    }
    for name, rc in checks.items():
        assert rc == ERR_INVALID, f"{name} with dtype 3: {status(rc)}"
    M, K, N = 256, 256, 256
    rng = np.random.default_rng(9)
    (tA, pA), (tB, pB) = dev_bytes(codes((M, K), rng)), dev_bytes(codes((N, K), rng))
    o8 = Out8(M, N)
    bias = torch.zeros(N, dtype=torch.uint8, device=DEV)
    rc = L.fp8b_scaled_mm(pA, pB, o8.ptr, OUT_E4M3FN, M, N, K, o8.ldc, p(one), 1, p(one), 1, p(bias), OUT_E4M3FN, None, None, 0,
                          ALGO_AUTO, s)
    assert rc == ERR_INVALID, f"bias_dtype 3: {status(rc)}"
    X = torch.zeros(M, K, dtype=torch.uint8, device=DEV)
    ws = torch.empty(L.fp8b_linear_dynamic_workspace_bytes(M, K), dtype=torch.uint8, device=DEV)
    rc = L.fp8b_linear_dynamic(p(X), OUT_E4M3FN, pB, o8.ptr, OUT_E4M3FN, M, N, K, o8.ldc, p(one), 1, None, F32, None, None, p(ws),
                               ws.numel(), s)
    assert rc == ERR_INVALID, f"x_dtype 3: {status(rc)}"
    items = (GemvItem * 1)()
    items[0].x, items[0].W, items[0].y, items[0].N = tA.data_ptr(), tB.data_ptr(), o8.ptr, N
    items[0].scale_x, items[0].scale_w, items[0].scale_w_len, items[0].bias = one.data_ptr(), one.data_ptr(), 1, bias.data_ptr()
    assert L.fp8b_gemv_batch(items, 1, K, OUT_E4M3FN, OUT_E4M3FN, s) == ERR_INVALID, "gemv_batch bias_dtype 3"
    rc = L.fp8b_scaled_mm_multicast(pA, pB, o8.ptr, OUT_E4M3FN, M, N, K, o8.ldc, p(one), 1, p(one), 1, None, 0, None, s)
    assert rc == ERR_UNSUPPORTED, f"multicast e4m3fn: {status(rc)}"
    # push: N % 16 != 0 and ldc % 16 != 0 are unsupported for 1-byte elements; push_supported says so
    ar = Arena(2, M, N + 32)
    t = terms(0, M, N, rng)
    rc = push_call(pA, pB, M, N - 8, K, t, [ar.ptr(0), ar.ptr(1)], ar.ldc)
    assert rc == ERR_UNSUPPORTED, f"push N % 16 != 0: {status(rc)}"
    rc = push_call(pA, pB, M, N, K, t, [ar.ptr(0)], ar.ldc - 8)
    assert rc == ERR_UNSUPPORTED, f"push ldc % 16 != 0: {status(rc)}"
    assert L.fp8b_scaled_mm_push_supported(OUT_E4M3FN, M, N - 8, K, ar.ldc, pA, pB, ar.ptr(0)) == 0
    assert L.fp8b_scaled_mm_push_supported(OUT_E4M3FN, M, N, K, ar.ldc - 8, pA, pB, ar.ptr(0)) == 0
    assert L.fp8b_scaled_mm_push_supported(OUT_E4M3FN, M, N, K, ar.ldc, pA, pB, ar.ptr(0)) == 1
    tune("GEMM_CFG", 5)
    rc = push_call(pA, pB, M, N, K, t, [ar.ptr(0), ar.ptr(1)], ar.ldc)
    assert rc == ERR_UNSUPPORTED, f"forced GEMM_CFG 5 push, e4m3fn: {status(rc)}"
    torch.cuda.synchronize()
    assert launches() == n0, "a refused call launched a kernel"
    assert torch.equal(buf, buf0), "a refused cast wrote its output"
    o8.check_guard("refusals", interior_written=False)
    ar.check([], "refused push")


def test_plan_does_not_depend_on_output_dtype():
    L = capi()
    rng = np.random.default_rng(4)
    for M, K, N in ((1, 4096, 512), (16, 1024, 77), (300, 400, 1000), (133, 1000, 197)):
        (tA, pA), (tB, pB) = dev_bytes(codes((M, K), rng)), dev_bytes(codes((N, K), rng))
        algos = {L.fp8b_scaled_mm_select(pA, pB, None, dt, M, N, K, N) for dt in (F32, BF16, OUT_E4M3FN)}
        assert len(algos) == 1, (M, K, N, algos)


# ------------------------------------------------------------------ 5. torch._scaled_mm and the bindings

@pytest.mark.parametrize("M,K,N", [(1, 4096, 512), (4, 1024, 272), (256, 512, 384), (300, 640, 1000)])
def test_scaled_mm_patch_fp8_out(M, K, N):
    """out_dtype=torch.float8_e4m3fn, keyword and positional, with bias and scale_result: a float8_e4m3fn tensor whose
    bytes equal the reference's composition _scaled_mm(..., out_dtype=float32).to(float8_e4m3fn) under the patch."""
    import fp8_mps_patch
    rng = np.random.default_rng(M + N)
    a8 = torch.from_numpy(codes((M, K), rng)).to(DEV).view(FP8)
    w8 = torch.from_numpy(codes((N, K), rng)).to(DEV).view(FP8)
    sa = torch.tensor([0.0123], device=DEV)
    sb = torch.from_numpy(((rng.random(N) + 0.5) * 0.02).astype(np.float32)).to(DEV)
    bias = torch.from_numpy(rng.standard_normal(N).astype(np.float32)).to(DEV).to(torch.bfloat16)
    sr = torch.tensor([1.5], device=DEV)
    fp8_mps_patch.install()
    try:
        y_kw = torch._scaled_mm(a8, w8.t(), scale_a=sa, scale_b=sb, bias=bias, scale_result=sr, out_dtype=FP8)
        y_pos = torch._scaled_mm(a8, w8.t(), sa, sb, bias, sr, FP8)
        ref = torch._scaled_mm(a8, w8.t(), scale_a=sa, scale_b=sb, bias=bias, scale_result=sr, out_dtype=torch.float32).to(FP8)
        y_nob = torch._scaled_mm(a8, w8.t(), scale_a=sa, scale_b=sb, out_dtype=FP8)
        ref_nob = torch._scaled_mm(a8, w8.t(), scale_a=sa, scale_b=sb).to(FP8)
        with pytest.raises(RuntimeError, match="e5m2"):
            torch._scaled_mm(a8, w8.t(), scale_a=sa, scale_b=sb, out_dtype=torch.float8_e5m2)
    finally:
        fp8_mps_patch.uninstall()
    for y in (y_kw, y_pos, y_nob):
        assert y.dtype == FP8 and tuple(y.shape) == (M, N)
    assert ref.dtype == FP8
    assert_bytes(u8(y_kw), u8(ref), "keyword")
    assert_bytes(u8(y_pos), u8(ref), "positional")
    assert_bytes(u8(y_nob), u8(ref_nob), "no bias")


def test_bindings_fp8_out(tune):
    """fp8_scaled_mm_fused (incl. out= with a wider row stride), fp8_scaled_mm_many, fp8_linear_dynamic, select_algo and
    the push / peers bindings take torch.float8_e4m3fn as the output dtype; bias dtypes stay float."""
    import fp8_mps_native as nat
    lib = nat._get_lib()
    rng = np.random.default_rng(8)
    M, K, N = 300, 512, 1024
    A = torch.from_numpy(codes((M, K), rng)).to(DEV)
    B = torch.from_numpy(codes((N, K), rng)).to(DEV)
    sa, sb = torch.tensor([0.011], device=DEV), torch.tensor([0.019], device=DEV)
    bias = torch.from_numpy(rng.standard_normal(N).astype(np.float32)).to(DEV)
    ref = encode_dev(nat.fp8_scaled_mm_fused(A, B, sa, sb, bias=bias, out_dtype=torch.float32))
    y = nat.fp8_scaled_mm_fused(A, B, sa, sb, bias=bias, out_dtype=FP8)
    assert y.dtype == FP8
    assert_bytes(u8(y), ref, "fused")
    wide = torch.full((M, N + 48), 0xFF, dtype=torch.uint8, device=DEV)
    nat.fp8_scaled_mm_fused(A, B, sa, sb, bias=bias, out_dtype=FP8, out=wide.view(FP8)[:, 16:16 + N])
    assert_bytes(wide[:, 16:16 + N], ref, "fused out=")
    assert bool((wide[:, :16] == 0xFF).all()) and bool((wide[:, 16 + N:] == 0xFF).all()), "fused out= wrote outside"
    assert lib.select_algo(A, B, FP8) == lib.select_algo(A, B, torch.float32)
    assert lib.push_supported(M, N, K, N, FP8) and not lib.push_supported(M, N - 8, K, N, FP8)
    # many
    xs = [A[:1].contiguous(), A[1:2].contiguous()]
    Ws = [B[:100].contiguous(), B[100:364].contiguous()]
    ys = nat.fp8_scaled_mm_many(xs, Ws, [sa, sa], [sb, sb], None, FP8)
    ys32 = nat.fp8_scaled_mm_many(xs, Ws, [sa, sa], [sb, sb], None, torch.float32)
    for y8, y32 in zip(ys, ys32):
        assert y8.dtype == FP8
        assert_bytes(u8(y8), encode_dev(y32), "many")
    # linear_dynamic
    X = torch.from_numpy(rng.standard_normal((5, K)).astype(np.float32)).to(DEV)
    y8, inv8 = nat.fp8_linear_dynamic(X, B, sb, bias, FP8)
    y32, inv32 = nat.fp8_linear_dynamic(X, B, sb, bias, torch.float32)
    assert y8.dtype == FP8 and torch.equal(inv8, inv32)
    assert_bytes(u8(y8), encode_dev(y32), "linear_dynamic")
    # push and peers bindings into full-width e4m3fn buffers, column block [n0, n0 + N)
    tune("GEMM_SPLITK", 1)
    n0, full = 32, N + 64
    ref = encode_dev(nat.fp8_scaled_mm_fused(A, B, sa, sb, bias=bias, out_dtype=torch.float32))
    for mode in ("push", "peers"):
        bufs = [torch.full((M, full), 0xFF, dtype=torch.uint8, device=DEV) for _ in range(2)]
        outs = [b.view(FP8) for b in bufs]
        if mode == "push":
            lib.fp8_scaled_mm_push(A, B, sa, sb, bias, outs[0], [o.data_ptr() for o in outs], n0)
        else:
            deltas = torch.tensor([0, outs[1].data_ptr() - outs[0].data_ptr()], dtype=torch.int64, device=DEV)
            lib.fp8_scaled_mm_peers(A, B, sa, sb, bias, outs[0], deltas, n0)
        torch.cuda.synchronize()
        for d, b in enumerate(bufs):
            assert_bytes(b[:, n0:n0 + N], ref, f"{mode} binding destination {d}")
            assert bool((b[:, :n0] == 0xFF).all()) and bool((b[:, n0 + N:] == 0xFF).all()), f"{mode} binding wrote outside"
