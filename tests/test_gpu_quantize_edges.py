"""Dynamic quantisation at its edges: NaN, infinities, signed zeros, the dtype maxima, subnormal amax and the amax below
which float32(448 / amax) overflows, through every amax -> scale -> encode kernel, bit for bit, in guarded buffers.

The arithmetic is the reference's fp8_quantize: amax of |x| in fp32, scale = 448 / amax in double, an fp32 multiply by
float32(scale), the encode, and inv = float32(1 / scale).  The special amax values follow from it (fp8_oracle):

  NaN amax             scale 1, inv 1; NaN elements encode to 0x7F
  inf amax             scale 0, inv +inf; finite elements -> 0x00, +-inf * 0 = NaN -> 0x7F
  amax < A* (~1.3e-36) float32(scale) = +inf, inv a subnormal or 0; zeros -> NaN -> 0x7F, nonzeros -> 0x7E / 0xFE

Each special value sits, one row or one call at a time, where the code paths change: the first element, the last
element of the vector body, the scalar tail, the last vector of the last thread of the register-resident row kernel,
and a random position.  Neighbouring rows have amax values 2^10 apart and every input is followed, inside its
allocation, by +inf, so a read past a row or past the tensor changes a scale.  Outputs are interior views of
sentinel-filled buffers, checked after every call.  The kernel variants each test must reach are computed from the
host rules and asserted from the kernel names a torch.profiler trace records."""
import re

import numpy as np
import pytest
import torch

import c_oracle
import fp8_oracle as o
from _util import F16, SENT, Out, assert_bits_equal, capi, dev_f32, dt_code, dt_name, p, stream_ptr, to_np

pytestmark = pytest.mark.gpu
DEV = "cuda"
DTYPES = (torch.float32, torch.float16, torch.bfloat16)
_ITORCH = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}
_UNP = {torch.float32: np.uint32, torch.float16: np.uint16, torch.bfloat16: np.uint16}
_SIGN = {torch.float32: 0x80000000, torch.float16: 0x8000, torch.bfloat16: 0x8000}
_INF = {torch.float32: 0x7F800000, torch.float16: 0x7C00, torch.bfloat16: 0x7F80}
_QNAN = {torch.float32: 0x7FC00000, torch.float16: 0x7E00, torch.bfloat16: 0x7FC0}
_NAN_PAYLOADS = {torch.float32: [0x7F800001, 0xFFC00001, 0x7FFFFFFF], torch.float16: [0x7C01, 0xFE00, 0x7FFF],
                 torch.bfloat16: [0x7F81, 0xFFC1, 0x7FFF]}
_MAX = {torch.float32: 0x7F7FFFFF, torch.float16: 0x7BFF, torch.bfloat16: 0x7F7F}
_MAX_SUB = {torch.float32: 0x007FFFFF, torch.float16: 0x03FF, torch.bfloat16: 0x007F}
_EPV = {torch.float32: 4, torch.float16: 8, torch.bfloat16: 8}
_PAD = 16                                                  # elements of +inf poison before and after every input
_BYTE_SENT = 0xA5


def _bits(values, dtype):
    """float values -> bit patterns of `dtype` (round to nearest)."""
    t = torch.as_tensor(np.asarray(values, np.float32)).to(dtype)
    return t.view(_ITORCH[dtype]).numpy().astype(np.int64) & (0xFFFFFFFF if dtype == torch.float32 else 0xFFFF)


def _values(bits, dtype):
    """bit patterns of `dtype` -> float32, exactly."""
    return torch.from_numpy(np.asarray(bits).astype(_UNP[dtype]).view(np.int32 if dtype == torch.float32 else np.int16)
                            ).view(dtype).float().numpy()


def a_star():
    """The smallest fp32 amax for which float32(448 / amax) is finite (bit pattern), by bisection over fp32 bit patterns
    with the oracle's arithmetic: a zero next to the amax element quantises to 0x7F exactly when the scale overflowed."""
    def overflows(b):
        return o.fp8_quantize(np.array([np.uint32(b).view(np.float32), 0.0], np.float32))[0][1] == 0x7F
    lo, hi = 1, 0x3F800000
    assert overflows(lo) and not overflows(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if overflows(mid) else (lo, mid)
    return hi


A_STAR = a_star()


def cases(dtype):
    """(name, special bit patterns, background).  The first special goes to the position under test, any others to
    random positions.  Backgrounds: normal (Gaussian, 2^10 apart from row to row), below (|x| < |special| / 2), zero,
    and the whole-row fills allzero / allnegzero / all (every element +-special)."""
    s = _SIGN[dtype]
    out = [("zero", [0], "allzero"), ("negzero", [s], "allnegzero"),
           ("nan", [_QNAN[dtype]], "normal"), ("negnan", [_QNAN[dtype] | s], "normal"),
           ("nan_payloads", _NAN_PAYLOADS[dtype], "normal"),
           ("inf", [_INF[dtype]], "normal"), ("neginf", [_INF[dtype] | s], "normal"),
           ("inf_nan", [_INF[dtype] | s, _QNAN[dtype]], "normal"),
           ("all_amax", list(_bits([3.25], dtype)), "all"), ("neg_amax", list(_bits([-1000.0], dtype)), "below"),
           ("amax448", list(_bits([448.0], dtype)), "below"), ("dtype_max", [_MAX[dtype]], "below"),
           ("min_sub", [1], "zero"), ("max_sub", [_MAX_SUB[dtype]], "zero")]
    if dtype == torch.float32:
        out += [("below_astar", [A_STAR - 1], "zero"), ("at_astar", [A_STAR], "zero")]
    elif dtype == torch.bfloat16:
        out += [("below_astar", [(A_STAR - 1) >> 16], "zero"), ("above_astar", [(A_STAR + 0xFFFF) >> 16], "zero")]
    return out


def make_row(case, pos, cols, base, dtype, rng):
    """One input row (bit patterns) for `case` with its first special value at `pos`."""
    _, sp, bg = case
    if bg == "allzero" or bg == "allnegzero":
        return np.full(cols, sp[0], np.int64)
    if bg == "all":
        return np.where(rng.random(cols) < 0.5, sp[0], sp[0] | _SIGN[dtype]).astype(np.int64)
    if bg == "normal":
        row = _bits(rng.standard_normal(cols) * base, dtype)
    elif bg == "below":
        row = _bits((rng.random(cols) - 0.5) * np.abs(_values([sp[0]], dtype)[0]), dtype)
    else:
        row = np.zeros(cols, np.int64)
    row[pos] = sp[0]
    for v in sp[1:]:
        row[rng.integers(cols)] = v
    return row


def special_rows(dtype, cols, positions, rng):
    """Every case at every position (the whole-row cases once), with plain rows between them, as bit patterns."""
    rows = []
    for case in cases(dtype):
        for i, pos in enumerate(positions):
            if case[2] in ("allzero", "allnegzero", "all") and i:
                break
            rows.append(make_row(case, pos, cols, 2.0 ** (10 * (len(rows) % 3 - 1)), dtype, rng))
    return np.stack(rows)


def poisoned(bits, dtype, offset=0):
    """bits (any shape) on the device between _PAD + offset and _PAD elements of +inf -> (buffer, pointer)."""
    flat = np.full(bits.size + 2 * _PAD + offset, _INF[dtype], np.int64)
    flat[_PAD + offset:_PAD + offset + bits.size] = bits.reshape(-1)
    npdt = np.int32 if dtype == torch.float32 else np.int16
    t = torch.from_numpy(flat.astype(_UNP[dtype]).view(npdt)).to(DEV).view(dtype)
    return t, t.data_ptr() + (_PAD + offset) * t.element_size()


class Bytes:
    """n output bytes inside a sentinel-filled buffer, starting 32 + offset bytes in."""

    def __init__(self, n, offset=0):
        self.n, self.o = n, 32 + offset
        self.buf = torch.full((n + self.o + 32,), _BYTE_SENT, dtype=torch.uint8, device=DEV)
        self.ptr = self.buf.data_ptr() + self.o

    def get(self, what):
        b = self.buf.cpu().numpy()
        assert (b[:self.o] == _BYTE_SENT).all() and (b[self.o + self.n:] == _BYTE_SENT).all(), f"{what}: wrote outside q"
        return b[self.o:self.o + self.n]


class Floats:
    """n fp32 outputs inside a sentinel-filled buffer."""

    def __init__(self, n):
        self.n = n
        self.buf = torch.full((n + 16,), SENT[torch.float32], dtype=torch.int32, device=DEV)
        self.ptr = self.buf.data_ptr() + 8 * 4

    def get(self, what):
        b = self.buf.cpu().numpy()
        assert (b[:8] == SENT[torch.float32]).all() and (b[8 + self.n:] == SENT[torch.float32]).all(), \
            f"{what}: wrote outside the scale output"
        return b[8:8 + self.n].view(np.float32)


def assert_same(got, want, what):
    if not np.array_equal(got, want):
        bad = np.flatnonzero(np.asarray(got).reshape(-1) != np.asarray(want).reshape(-1))
        raise AssertionError(f"{what}: {bad.size} of {np.size(want)} differ; first at {bad[0]}: "
                             f"got {np.asarray(got).reshape(-1)[bad[0]]!r} want {np.asarray(want).reshape(-1)[bad[0]]!r}")


def assert_f32_bits(got, want, what):
    assert_same(np.asarray(got, np.float32).view(np.uint32), np.asarray(want, np.float32).view(np.uint32), what)


def kernels(fn):
    """Run fn under torch.profiler; return the names of the CUDA kernels it launched."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


def assert_reached(names, patterns, what):
    for pat in patterns:
        assert any(re.search(pat, n) for n in names), f"{what}: no kernel matching {pat!r} ran; ran {sorted(names)}"


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------ fp8b_quantize_rows

def rows_plan(rows, cols, dtype, in_ok=True):
    """The kernel fp8b_quantize_rows picks (fp8_cast.cu): ("reg", V, TPR) or ("two_pass", vector?)."""
    epv = _EPV[dtype]
    vec_ok = in_ok and cols * (16 // epv) % 16 == 0
    nvec = cols // epv
    if vec_ok and 0 < nvec <= 2048:
        if rows * 64 < sm_count() * 2048 or nvec > 512:
            return ("reg", 1 if nvec <= 256 else 2 if nvec <= 512 else 4 if nvec <= 1024 else 8, 256)
        return ("reg",) + ((2, 32) if nvec <= 64 else (4, 32) if nvec <= 128 else (4, 64) if nvec <= 256 else (4, 128))
    return ("two_pass", vec_ok)


# (name, vectors per row or -cols, many rows, element offset of the input): one entry per kernel variant
ROW_CONFIGS = [("reg V1 TPR256", 200, False, 0), ("reg V2 TPR256", 400, False, 0), ("reg V4 TPR256", 1000, False, 0),
               ("reg V8 TPR256", 2000, False, 0), ("reg V2 TPR32", 40, True, 0), ("reg V4 TPR32", 100, True, 0),
               ("reg V4 TPR64", 200, True, 0), ("reg V4 TPR128", 400, True, 0), ("two-pass vector", 2049, False, 0),
               ("two-pass scalar, ragged cols", -1001, False, 0), ("two-pass scalar, unaligned base", 64, False, 1)]


@pytest.mark.parametrize("dtype", DTYPES, ids=dt_name)
def test_quantize_rows_edges(dtype):
    """fp8b_quantize_rows: every register-resident (V, TPR) instantiation (row counts not a multiple of the rows per
    CTA), the two-pass vector kernel and the two-pass scalar kernel, each with every special row."""
    L = capi()
    rng = np.random.default_rng(dt_code(dtype))
    epv = _EPV[dtype]
    reached = set()

    def run_all():
        for name, nv, many, off in ROW_CONFIGS:
            cols = -nv if nv < 0 else nv * epv
            plan = rows_plan(0, cols, dtype, in_ok=off == 0)
            nvec = cols // epv if plan[0] == "reg" or plan[1] else 0
            pos = {0, cols - 1, int(rng.integers(cols))}
            if nvec:
                pos.add(nvec * epv - 1)
            if plan[0] == "reg":
                V, T = rows_plan(sm_count() * 32 + 5 if many else 3, cols, dtype)[1:]
                assert (V - 1) * T < nvec, "the last of the V vectors must exist for some thread"
                pos |= {(V - 1) * T * epv, min(nvec - 1, V * T - 1) * epv + epv // 2}
            else:
                pos.add(min(cols - 1, 255 * (epv if nvec else 1) + 1))
            block = special_rows(dtype, cols, sorted(pos), rng)
            R = sm_count() * 32 + 5 if many else block.shape[0]
            bits = np.tile(block, (-(-R // block.shape[0]), 1))[:R]
            plan = rows_plan(R, cols, dtype, in_ok=off == 0)
            reached.add(plan)
            x, px = poisoned(bits, dtype, off)
            q, inv = Bytes(R * cols), Floats(R)
            rc = L.fp8b_quantize_rows(px, dt_code(dtype), R, cols, q.ptr, inv.ptr, stream_ptr())
            torch.cuda.synchronize()
            what = f"quantize_rows {name} {dt_name(dtype)} rows {R} cols {cols} plan {plan}"
            assert rc == 0, what
            rq, rinv = o.fp8_quantize_rows(_values(block, dtype))
            reps = -(-R // block.shape[0])
            assert_same(q.get(what).reshape(R, cols), np.tile(rq, (reps, 1))[:R], what + " bytes")
            assert_f32_bits(inv.get(what), np.tile(rinv, reps)[:R], what + " inv")

    names = kernels(run_all)
    regs = {pl for pl in reached if pl[0] == "reg"}
    assert {pl[1:] for pl in regs} == {(1, 256), (2, 256), (4, 256), (8, 256), (2, 32), (4, 32), (4, 64), (4, 128)}
    dcode = dt_code(dtype)
    assert_reached(names, [rf"quantize_rows_reg_kernel<{dcode}, {v}, {t}>" for _, v, t in regs] +
                   [rf"quantize_rows_kernel<{dcode}>"], f"quantize_rows {dt_name(dtype)}")


# ------------------------------------------------------------------ per tensor: fp8b_amax_scale + prescaled fp8b_encode

def _scale32(amax):
    with np.errstate(over="ignore"):
        return np.float32(448.0 / float(amax) if amax > 0 else 1.0)


def per_tensor_case(dtype, n, block_bits, case, pos, off, rng, which=("scale", "inv")):
    """One amax_scale + encode call; the input is block_bits tiled to n with the case's special value(s) at pos."""
    L = capi()
    _, sp, bg = case
    if bg in ("allzero", "allnegzero", "all"):
        block = make_row(case, 0, block_bits.size, 1.0, dtype, rng)
    elif bg in ("zero", "below"):
        block = np.zeros(block_bits.size, np.int64) if bg == "zero" else \
            _bits((rng.random(block_bits.size) - 0.5) * np.abs(_values([sp[0]], dtype)[0]), dtype)
    else:
        block = block_bits
    reps = -(-n // block.size)
    assert reps >= 2
    full = np.tile(block, reps)[:n]
    spos = {}
    if bg not in ("allzero", "allnegzero", "all"):
        spos[pos] = sp[0]
        for v in sp[1:]:
            spos[int(rng.integers(n))] = v
    for k, v in spos.items():
        full[k] = v
    x, px = poisoned(full, dtype, off)
    # the oracle on the distinct values (every block value also appears in an untouched copy of the block)
    ks = np.array(sorted(spos), np.int64)
    compact = np.concatenate([block, np.array([spos[k] for k in ks], np.int64)])
    rq, rinv = o.fp8_quantize(_values(compact, dtype))
    want_q = np.tile(rq[:block.size], reps)[:n]
    want_q[ks] = rq[block.size:]
    amax = np.max(np.abs(_values(compact, dtype)))
    out = Floats(2)
    s_ptr = out.ptr if "scale" in which else None
    i_ptr = out.ptr + 4 if "inv" in which else None
    scratch = torch.zeros(4, dtype=torch.int32, device=DEV)
    what = f"per-tensor {case[0]} {dt_name(dtype)} n {n} pos {pos} offset {off} {which}"
    assert L.fp8b_amax_scale(px, dt_code(dtype), n, s_ptr, i_ptr, scratch.data_ptr(), stream_ptr()) == 0, what
    q = None
    if s_ptr is not None:
        q = Bytes(n)
        assert L.fp8b_encode(px, dt_code(dtype), q.ptr, n, s_ptr, stream_ptr()) == 0, what
    torch.cuda.synchronize()
    got = out.get(what).copy()
    raw = out.buf.cpu().numpy()[8:10]
    if "scale" in which:
        assert_f32_bits(got[:1], [_scale32(amax)], what + " scale")
        assert_same(q.get(what), want_q, what + " bytes")
    else:
        assert raw[0] == SENT[torch.float32], what + ": scale written through a NULL pointer's slot"
    if "inv" in which:
        assert_f32_bits(got[1:], rinv, what + " inv")
    else:
        assert raw[1] == SENT[torch.float32], what
    assert scratch[0].item() == 0, what + ": amax scratch word not reset"


def _tensor_positions(n, epv, extra=()):
    nvec = n // epv
    return sorted(k for k in {0, nvec * epv - 1, n - 1, epv * 1024 + 5, *extra} if k < n)


@pytest.mark.parametrize("dtype", DTYPES, ids=dt_name)
def test_amax_scale_encode_edges(tune, dtype):
    """Per-tensor quantisation through the C ABI: amax_kernel (tail element in block 0) under the default AMAX_CAP and
    AMAX_CAP = 1 (grid-stride loop), amax_scalar_kernel with the scalar encode (input not 16-byte aligned), small and
    big 16-byte encode tiles, and for fp32 the 256-bit tiles; scale_out and inv each with the other pointer NULL."""
    rng = np.random.default_rng(40 + dt_code(dtype))
    epv = _EPV[dtype]
    sms = sm_count()
    block = _bits(rng.standard_normal(1021) * 3.0, dtype)
    all_cases = cases(dtype)
    few = [c for c in all_cases if c[0] in ("nan", "neginf", "neg_amax", "max_sub", "below_astar")]
    configs = [("small tiles", 8 * 1024 + 3, 0, None, all_cases, ()),
               ("AMAX_CAP 1", sms * 1024 * epv * 2 + 5, 0, 1, few, (sms * 1024 * epv + 1,)),
               ("unaligned", 5000, 1, None, all_cases, ()),
               ("big tiles", sms * 4096 * epv + 7, 0, None, few, ())]
    if dtype == torch.float32:
        configs.append(("256-bit tiles", (1 << 25) + 3, 0, None, few[:2], ()))

    def run_all():
        for name, n, off, cap, cs, extra in configs:
            if cap is not None:
                tune("AMAX_CAP", cap)
            for case in cs:
                for pos in _tensor_positions(n, epv, extra):
                    per_tensor_case(dtype, n, block, case, pos, off, rng)
            if cap is not None:
                tune("AMAX_CAP", -1)
        for which in (("scale",), ("inv",)):
            per_tensor_case(dtype, 4099, block, all_cases[2], 4098, 0, rng, which)

    names = kernels(run_all)
    d = dt_code(dtype)
    pats = [rf"amax_kernel<{d}>", rf"amax_scalar_kernel<{d}>", rf"wide_to_fp8_scalar_kernel<{d}, true>",
            rf"wide_to_fp8_kernel<{d}, true, 256, 4, 16>", rf"wide_to_fp8_kernel<{d}, true, 1024, 4, 16>"]
    if dtype == torch.float32:
        pats.append(rf"wide_to_fp8_kernel<{d}, true, 512, 4, 32>")
    assert_reached(names, pats, f"per-tensor {dt_name(dtype)}")


def test_amax_scale_empty_and_python_api():
    """n = 0 gives scale 1 and inv 1; fp8_mps_native.fp8_quantize gives the oracle's answer on a row with +-inf."""
    import fp8_mps_native
    L = capi()
    out = Floats(2)
    scratch = torch.zeros(1, dtype=torch.int32, device=DEV)
    assert L.fp8b_amax_scale(None, 0, 0, out.ptr, out.ptr + 4, scratch.data_ptr(), stream_ptr()) == 0
    torch.cuda.synchronize()
    assert out.get("n = 0").tolist() == [1.0, 1.0]
    x = torch.randn(1000, generator=torch.Generator().manual_seed(3))
    x[17], x[999] = float("inf"), float("-inf")
    q, inv = fp8_mps_native.fp8_quantize(x)
    rq, rinv = o.fp8_quantize(x.numpy())
    assert rinv[0] == np.inf and set(rq[[17, 999]].tolist()) == {0x7F}
    assert_same(q.cpu().numpy(), rq, "fp8_mps_native.fp8_quantize inf")
    assert_f32_bits(inv.cpu().numpy(), rinv, "fp8_mps_native.fp8_quantize inf")


# ------------------------------------------------------------------ fp8b_linear_dynamic

# (M, K, N, DYNAMIC_PLAN, workspace, kernel that computes C; at M = 40 tcgen05 takes its split-K plan)
DYN_CONFIGS = [(1, 4096, 264, 1, False, r"fp8_gemv_xq_kernel<1, "), (2, 4096, 264, 1, False, r"fp8_gemv_xq_kernel<2, "),
               (3, 4096, 264, 1, False, r"fp8_gemv_xq_kernel<3, "), (4, 4096, 264, 1, False, r"fp8_gemv_xq_kernel<4, "),
               (16, 4096, 264, 1, False, r"fp8_gemv_xq_kernel<4, "), (1, 4096, 264, 2, True, r"fp8_gemv_kernel<1, "),
               (4, 4096, 264, 2, True, r"fp8_gemv_mma_kernel"), (40, 4096, 264, -1, True, r"fp8_gemm_(tcgen05|splitk)_kernel"),
               (20, 100, 72, -1, True, r"fp8_gemm_simt_kernel")]


def _one_hot_w(N, K, positions, rng):
    """W (N, K) with one nonzero per row, at positions[n % len]: each output is one exact product."""
    codes = np.array([c for c in range(256) if (c & 0x7F) not in (0x7F, 0x00)], np.uint8)
    W = np.zeros((N, K), np.uint8)
    W[np.arange(N), np.asarray(positions)[np.arange(N) % len(positions)]] = rng.choice(codes, N)
    return W


@pytest.mark.parametrize("dtype", DTYPES, ids=dt_name)
def test_linear_dynamic_edges(tune, dtype):
    """fp8b_linear_dynamic with special X rows and one-hot W rows whose nonzeros sit on the special positions: the
    single-kernel plan at M = 1, 2, 3, 4, 16 with split-K over a 2-CTA cluster (K = 4096, N = 264), the chained plan
    (FHFMA at M = 1, warp-MMA at M = 4), and M > 16 through tcgen05 and SIMT (K = 100).  inv_scale_a_out is compared
    bit for bit; C equals the oracle, NaN where the oracle has NaN."""
    L = capi()
    rng = np.random.default_rng(70 + dt_code(dtype))
    all_cases = cases(dtype)

    def run_all():
        for M, K, N, plan, ws, _ in DYN_CONFIGS:
            tune("DYNAMIC_PLAN", plan)
            pos = sorted({0, 15, K // 2 - 1, K // 2, K - 16, K - 1, int(rng.integers(K))} if K >= 64 else {0, K - 1, 37})
            W = _one_hot_w(N, K, pos, rng)
            tW = torch.from_numpy(np.concatenate([W.reshape(-1), np.full(16 * K, 0x7E, np.uint8)])).to(DEV)
            sb = ((rng.random(N) + 0.5) * 0.0217).astype(np.float32)
            t_sb = dev_f32(sb)
            rows = [make_row(c, pp, K, 2.0 ** (10 * (i % 3 - 1)), dtype, rng)
                    for i, (c, pp) in enumerate((c, pp) for c in all_cases for pp in pos)]
            for r0 in range(0, len(rows), M):
                chunk = rows[r0:r0 + M]
                chunk += rows[:M - len(chunk)]
                bits = np.stack(chunk)
                x, px = poisoned(bits, dtype)
                out = Out(M, N, torch.float32)
                inv = Floats(M)
                need = L.fp8b_linear_dynamic_workspace_bytes(M, K)
                wsb = torch.empty(need + 16, dtype=torch.uint8, device=DEV) if ws else None
                rc = L.fp8b_linear_dynamic(px, dt_code(dtype), tW.data_ptr(), out.ptr, 0, M, N, K, out.ldc, p(t_sb), N,
                                           None, 0, None, inv.ptr, p(wsb), need if ws else 0, stream_ptr())
                torch.cuda.synchronize()
                what = f"linear_dynamic {dt_name(dtype)} M{M} K{K} N{N} plan {plan} ws {ws} rows {r0}.."
                assert rc == 0, what
                q, rinv = o.fp8_quantize_rows(_values(bits, dtype))
                assert_f32_bits(inv.get(what), rinv, what + " inv")
                out.check_guard(what)
                with np.errstate(invalid="ignore", over="ignore"):
                    ref = o.scaled_mm(q, W, rinv, sb, out_dtype="f32", accum="f64")
                assert_bits_equal(to_np(out.view), ref, what, any_nan=True)
            tune("DYNAMIC_PLAN", -1)

    names = kernels(run_all)
    assert_reached(names, [c[5] for c in DYN_CONFIGS] + [rf"quantize_rows_reg_kernel<{dt_code(dtype)}, "],
                   f"linear_dynamic {dt_name(dtype)}")


# ------------------------------------------------------------------ encode sweep and special prescales / scales

def _encode(x_ptr, dtype_code, n, prescale=None):
    q = Bytes(n)
    assert capi().fp8b_encode(x_ptr, dtype_code, q.ptr, n, prescale, stream_ptr()) == 0
    return q


def test_encode_f32_binade_sweep():
    """Every fp32 pattern with exponent field 116..136 (the binades in which the encoder's output depends on the
    fraction, and one more on each side), both signs, through the vector encode kernel; three binades through the
    scalar kernel.  Compared with the C oracle in chunks."""
    chunk = 1 << 25
    starts = [(s << 31) | (e << 23) for s in (0, 1) for e in range(116, 137, 4)]
    for s0 in starts:
        for c0 in range(s0, min(s0 + (4 << 23), (s0 & 0x80000000) | (137 << 23)), chunk):
            n = min(chunk, ((s0 & 0x80000000) | (137 << 23)) - c0)
            dev = torch.arange(c0, c0 + n, dtype=torch.int64, device=DEV).to(torch.int32)       # wraps to the bit pattern
            got = _encode(dev.data_ptr(), 0, n).get("sweep")
            want = c_oracle.encode(np.arange(c0, c0 + n, dtype=np.uint32).view(np.float32))
            assert_same(got, want, f"fp32 encode, patterns {c0:#x}..{c0 + n:#x}")
    for e in (118, 127, 135):
        c0 = e << 23
        dev = torch.arange(c0, c0 + (1 << 23) + 1, dtype=torch.int64, device=DEV).to(torch.int32)
        got = _encode(dev.data_ptr() + 4, 0, 1 << 23).get("sweep scalar")                 # 4-byte offset: scalar kernel
        want = c_oracle.encode(np.arange(c0 + 1, c0 + 1 + (1 << 23), dtype=np.uint32).view(np.float32))
        assert_same(got, want, f"fp32 scalar encode, binade {e}")


SPECIAL_PRESCALES = [0.0, -0.0, np.inf, np.nan, np.finfo(np.float32).max, np.float32(2.0 ** -140),
                     np.float32(448.0 / 3.0), np.float32(448.0 / 1e-30)]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=dt_name)
def test_encode_all_16bit_patterns_special_prescales(dtype):
    """All 65536 fp16 / bf16 patterns with the prescales 0, -0, +inf, NaN, FLT_MAX, a subnormal and two values of the
    form float32(448 / amax), through the vector and the scalar prescaled encode: enc(f32(x) * s)."""
    bits = torch.arange(65536 + 8, dtype=torch.int32).to(torch.int16).view(dtype).to(DEV)
    xf = _values(np.arange(65536 + 8) & 0xFFFF, dtype)
    for s in SPECIAL_PRESCALES:
        ts = dev_f32([s])
        with np.errstate(invalid="ignore", over="ignore"):
            want = c_oracle.encode(xf * np.float32(s))
        for off in (0, 3):
            n = 65536 + 8 - off
            got = _encode(bits.data_ptr() + 2 * off, dt_code(dtype), n, ts.data_ptr()).get("prescale")
            assert_same(got, want[off:], f"{dt_name(dtype)} encode * {s!r} offset {off}")


DEQ_SCALES = [0.0, -0.0, -1.0, 65504.0, 65520.0, 1e5, np.inf, -np.inf, np.nan, 2.0 ** -24, 2.0 ** -25, 3e-8]


@pytest.mark.parametrize("fmt", ["e4m3fn", "e5m2"])
def test_dequant_f16_special_scales(fmt):
    """fp8b_dequant_f16 / fp8b_dequant_fmt(e5m2) -> fp16 with special scales (0, -0, -1, 65504, 65520 which rounds to
    inf in fp16, 1e5, +-inf, NaN, 2^-24, 2^-25, 3e-8) through the small-tile, big-tile, tail and scalar kernels: an fp16
    multiply of the fp16 decode by half(scale), NaN-aware bit comparison."""
    L = capi()
    big = sm_count() * 4096 * 8 + 5
    codes = torch.arange(256, dtype=torch.int32).to(torch.uint8)
    sizes = [(256 * 16 + 3, 0), (big, 0), (256 * 4 + 1, 1)]
    with np.errstate(over="ignore", invalid="ignore"):
        dec = (o.decode(np.arange(256)) if fmt == "e4m3fn" else o.decode_e5m2(np.arange(256))).astype(np.float16)

    def run_all():
        for n, off in sizes:
            src = codes.repeat(-(-(n + off) // 256))[:n + off].to(DEV)
            for s in DEQ_SCALES:
                ts = dev_f32([s])
                buf = torch.full((n + 24,), SENT[torch.float16], dtype=torch.int16, device=DEV)
                pout = buf.data_ptr() + 16 + 2 * off
                if fmt == "e4m3fn":
                    rc = L.fp8b_dequant_f16(src.data_ptr() + off, pout, n, ts.data_ptr(), stream_ptr())
                else:
                    rc = L.fp8b_dequant_fmt(src.data_ptr() + off, 1, pout, F16, n, ts.data_ptr(), stream_ptr())
                assert rc == 0
                raw = buf.cpu().numpy()
                what = f"dequant {fmt} n {n} offset {off} scale {s!r}"
                assert (raw[:8 + off] == SENT[torch.float16]).all() and (raw[8 + off + n:] == SENT[torch.float16]).all(), \
                    what + ": wrote outside the output"
                with np.errstate(over="ignore", invalid="ignore"):
                    want = (np.tile(dec, -(-(n + off) // 256))[off:off + n] * np.float16(np.float32(s))).astype(np.float16)
                got = raw[8 + off:8 + off + n].view(np.float16)
                nan = np.isnan(want)
                assert_same(np.isnan(got), nan, what + " NaN positions")
                assert_same(got.view(np.uint16)[~nan], want.view(np.uint16)[~nan], what)

    names = kernels(run_all)
    f = 0 if fmt == "e4m3fn" else 1
    assert_reached(names, [rf"fp8_to_wide_kernel<{F16}, true, 256, 4, {f}>", rf"fp8_to_wide_kernel<{F16}, true, 512, 8, {f}>",
                           rf"fp8_to_wide_scalar_kernel<{F16}, true, {f}>"], f"dequant {fmt}")
