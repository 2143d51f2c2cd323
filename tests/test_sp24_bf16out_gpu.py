"""GPU tests of bf16 output with a per-row bias for the 2:4-sparse operators (libxsmm_b200_sp24_execute_bf16out /
_execute_fp8_bf16out, Sp24.linear; csrc/sp24.cu, OB = true).

The reference is the fp32-output entry on the same operator and B: its C (beta = 0) is the v = alpha acc of the contract's
step 1, and steps 2-4 are emulated on it in numpy float32 (one rounded addition each) and rounded to bf16 by torch (nearest
even).  Operands are built as in test_sp24_fp8_gpu (make24, small dyadic values), so the bf16 operator runs the same values
widened; every beta used for bit equality is a power of two or +-1, which makes fmaf(beta, C, v) one exact product and one
rounded addition."""
import numpy as np
import pytest

from test_sp24_fp8_gpu import DYADIC, FMTS, LEGAL, dec, enc, make24, operands, pad_b, widen

pytestmark = pytest.mark.gpu
KINDS = ["bf16"] + ["%s/%s" % f for f in FMTS]
NAN16 = 0x7FC1


def fmts(kind):
    return ("e4m3", "e4m3") if kind == "bf16" else tuple(kind.split("/"))


def values16(h):
    return (np.ascontiguousarray(h, np.uint16).astype(np.uint32) << 16).view(np.float32)


def bits16(x):
    """float32 -> bf16 bits, rounded to nearest even by torch"""
    import torch
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def dyadic16(shape, rng):
    return bits16(rng.choice(DYADIC, shape))


class Case:
    """one operator and one B, run through the fp32 entry and the bf16-output entry"""

    def __init__(self, xs, kind, A, B, transb):
        """A, B in the operator's encoding: uint16 bf16 bits for kind "bf16", FP8 bytes otherwise"""
        self.xs, self.kind, self.transb = xs, kind, transb
        self.a_fmt, self.b_fmt = fmts(kind)
        self.M, self.K = A.shape
        self.N = B.shape[0] if transb == "T" else B.shape[1]
        if kind == "bf16":
            self.op = xs.Sp24(A)
            self.ldb = (B.shape[1] + 7) // 8 * 8
            Bp = np.full((B.shape[0], self.ldb), NAN16, np.uint16)       # B goes through TMA: NaN in the row padding
            Bp[:, :B.shape[1]] = B
        else:
            self.op = xs.Sp24(A, fmt=self.a_fmt)
            Bp, self.ldb = pad_b(B, self.b_fmt)
        self.dB = xs.DeviceBuffer.from_numpy(Bp)
        self.kernel = "sp24_compute_kernel_bf16out" if kind == "bf16" else "sp24_compute_kernel_fp8_bf16out"

    def kw(self, alpha):
        return {} if self.kind == "bf16" else {"alpha": alpha, "b_fmt": self.b_fmt}

    def c_shape(self, transc):
        return (self.N, self.M) if transc == "T" else (self.M, self.N)

    def fp32(self, transc, alpha=1.0):
        """C of the fp32-output entry with beta = 0: the contract's v after step 1"""
        xs = self.xs
        dC = xs.DeviceBuffer(4 * self.M * self.N)
        try:
            self.op.execute(self.dB, dC, self.N, ldb=self.ldb, transb=self.transb, transc=transc, **self.kw(alpha))
            xs.synchronize()
            xs.check()
            return dC.to_numpy(np.float32, self.c_shape(transc))
        finally:
            dC.free()

    def bf16(self, transc, C0, alpha=1.0, bias=None, beta=0.0, ldc=None, c_offset=0):
        """C of the bf16-output entry: C0 (uint16, rows of ldc) uploaded at byte offset c_offset of a fresh buffer"""
        xs = self.xs
        dC = xs.DeviceBuffer(C0.nbytes + 16)
        dC.upload(np.ascontiguousarray(C0), c_offset)
        dbias = None if bias is None else xs.DeviceBuffer.from_numpy(bias)
        try:
            n0 = xs.launch_count()
            self.op.execute(self.dB, dC.ptr + c_offset, self.N, ldb=self.ldb, ldc=ldc, beta=beta, transb=self.transb, transc=transc,
                            bias=dbias, c_dtype="bf16", **self.kw(alpha))
            xs.synchronize()
            xs.check()
            assert xs.launch_count() == n0 + 1
            assert xs.last_compute_kernel() == self.kernel
            return dC.to_numpy(np.uint16, C0.shape, c_offset)
        finally:
            dC.free()
            if dbias is not None:
                dbias.free()

    def destroy(self):
        self.op.destroy()
        self.dB.free()


def encode(kind, A8, B8):
    """FP8 operands as the operator of `kind` takes them (widened to bf16 for the bf16 operator: exact)"""
    a_fmt, b_fmt = fmts(kind)
    return (widen(A8, a_fmt), widen(B8, b_fmt)) if kind == "bf16" else (A8, B8)


def make_case(xs, kind, M, N, K, transb, seed):
    a_fmt, b_fmt = fmts(kind)
    A8, B8, _ = operands(M, N, K, transb, "N", seed, a_fmt, b_fmt)
    return Case(xs, kind, *encode(kind, A8, B8), transb), A8, B8


def dense_case(xs, kind, A, B):
    """an operator and B ('N') from float32 arrays that the kind's formats hold exactly"""
    if kind == "bf16":
        Ae, Be = bits16(A), bits16(B)
        assert np.array_equal(values16(Ae), A) and np.array_equal(values16(Be), B)
    else:
        a_fmt, b_fmt = fmts(kind)
        Ae, Be = enc(A, a_fmt), enc(B, b_fmt)
        assert np.array_equal(dec(Ae, a_fmt), A) and np.array_equal(dec(Be, b_fmt), B)
    return Case(xs, kind, Ae, Be, "N")


def emulate(v, transc, bias=None, beta=0.0, C0=None):
    """steps 2-4 on the fp32 entry's C, in numpy float32; bf16 bits"""
    v = v.astype(np.float32).copy()
    with np.errstate(invalid="ignore", over="ignore"):
        if bias is not None:
            b = values16(bias)
            v = v + (b[None, :] if transc == "T" else b[:, None])
        if beta != 0.0:
            v = v + np.float32(beta) * values16(C0)
    return bits16(v)


def is_nan16(h):
    return ((h & 0x7F80) == 0x7F80) & ((h & 0x7F) != 0)


def assert_bits(got, want):
    nan = is_nan16(want)
    np.testing.assert_array_equal(is_nan16(got), nan)
    np.testing.assert_array_equal(got[~nan], want[~nan])


# ---- same accumulator: NULL bias and beta = 0 give the fp32 entry's C rounded to bf16 -----------------------------------------
def same_accumulator(xs, kind, M, N, K, transb, transc, seed=0):
    case, _, _ = make_case(xs, kind, M, N, K, transb, seed + M + N + K)
    try:
        alpha = 1.0 if kind == "bf16" else 0.5
        v = case.fp32(transc, alpha)
        C0 = np.full(case.c_shape(transc), NAN16, np.uint16)            # beta = 0: C is not read
        got = case.bf16(transc, C0, alpha)
        np.testing.assert_array_equal(got, bits16(v))
    finally:
        case.destroy()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("transb", ["N", "T"])
@pytest.mark.parametrize("transc", ["N", "T"])
def test_same_accumulator_ragged(gpu, kind, transb, transc):
    same_accumulator(gpu, kind, 300, 257, 200, transb, transc)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("M,N,K", [(2560, 2560, 384), (4096, 1024, 4096)])     # half tiles; many tiles per CTA pair
@pytest.mark.parametrize("trans", ["NN", "TT"])
def test_same_accumulator_tiles(gpu, kind, M, N, K, trans):
    same_accumulator(gpu, kind, M, N, K, trans[0], trans[1])


@pytest.mark.parametrize("kind", ["bf16", "e4m3/e5m2"])
@pytest.mark.parametrize("N", [3, 16, 130, 257])
@pytest.mark.parametrize("transc", ["N", "T"])
def test_same_accumulator_n(gpu, kind, N, transc):
    same_accumulator(gpu, kind, 300, N, 256, "N", transc)


# ---- bias, then beta, then rounding ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,alpha", [("bf16", 1.0), ("e4m3/e4m3", 1.0), ("e4m3/e4m3", 2.0 ** -6), ("e5m2/e4m3", 2.0 ** -6)])
@pytest.mark.parametrize("beta", [0.0, 1.0, 0.5, -1.0, 2.0])
@pytest.mark.parametrize("transc", ["N", "T"])
def test_bias_and_beta_order(gpu, kind, alpha, beta, transc):
    M, N, K = 520, 392, 328
    case, _, _ = make_case(gpu, kind, M, N, K, "N", 7)
    rng = np.random.default_rng(8)
    try:
        v = case.fp32(transc, alpha)
        bias = dyadic16(M, rng)
        C0 = dyadic16(case.c_shape(transc), rng)
        got = case.bf16(transc, C0, alpha, bias, beta)
        assert_bits(got, emulate(v, transc, bias, beta, C0))
        nobias = case.bf16(transc, C0, alpha, None, beta)
        assert_bits(nobias, emulate(v, transc, None, beta, C0))
    finally:
        case.destroy()


@pytest.mark.parametrize("kind", ["bf16", "e4m3/e4m3"])
def test_beta_not_dyadic_within_one_ulp(gpu, kind):
    M, N, K = 300, 264, 256
    case, _, _ = make_case(gpu, kind, M, N, K, "T", 9)
    rng = np.random.default_rng(9)
    try:
        v = case.fp32("N", 0.25)
        bias = dyadic16(M, rng)
        C0 = bits16(rng.uniform(-3, 3, (M, N)))
        got = case.bf16("N", C0, 0.25, bias, 0.3)
        vb = (v + values16(bias)[:, None]).astype(np.float64)              # exact: dyadic operands
        want64 = vb + float(np.float32(0.3)) * values16(C0).astype(np.float64)   # the exact fmaf operand sum
        assert np.all(np.abs(values16(got).astype(np.float64) - want64) <= bf16_ulp(want64))
    finally:
        case.destroy()


# ---- rounding and special values -------------------------------------------------------------------------------------------
def two_term(t, s):
    """A row m = [1, t_m, 0, ...], B column n = [1, s_n, 0, ...]^T: acc = 1 + t_m s_n"""
    M, N, K = len(t), len(s), 128
    A, B = np.zeros((M, K), np.float32), np.zeros((K, N), np.float32)
    A[:, 0], A[:, 1] = 1.0, t
    B[0, :], B[1, :] = 1.0, s
    return A, B


@pytest.mark.parametrize("kind", ["bf16", "e4m3/e4m3"])
def test_halfway_rounds_to_even(gpu, kind):
    t = np.tile(np.array([2.0 ** -8, -2.0 ** -8, 2.0 ** -7, 0.0]), 32)            # 1 + k 2^-8 with k odd is a tie
    s = np.tile(np.array([1.0, 3.0, 5.0, 7.0, 0.5, 1.5]), 11)[:64]
    case = dense_case(gpu, kind, *two_term(t, s))
    try:
        v = case.fp32("N")
        np.testing.assert_array_equal(v, (1.0 + np.outer(t, s)).astype(np.float32))
        ties = (v.view(np.uint32) & 0xFFFF) == 0x8000
        assert ties.sum() > 1000
        got = case.bf16("N", np.zeros((case.M, case.N), np.uint16))
        np.testing.assert_array_equal(got, bits16(v))
        assert np.all(got[ties] & 1 == 0)                                           # every tie went to the even neighbour
        assert list(got[0, :4]) == [0x3F80, 0x3F82, 0x3F82, 0x3F84]                 # 1 + {1, 3, 5, 7} 2^-8
    finally:
        case.destroy()


@pytest.mark.parametrize("kind", ["bf16", "e5m2/e5m2"])
def test_past_the_bf16_maximum_gives_inf(gpu, kind):
    """v = +-2^119 (alpha lifts the FP8 accumulator there) plus a bias of +-bf16 max of the same sign is finite in fp32 and a
    tie whose even neighbour is +-Inf; a bias of the other sign stays finite"""
    M, N = 128, 64
    sign = np.where(np.arange(M) % 2, 1.0, -1.0).astype(np.float32)
    big, alpha = (2.0 ** 119, 1.0) if kind == "bf16" else (2.0 ** 14, 2.0 ** 105)
    A, B = two_term(np.zeros(M), np.zeros(N))
    A[:, 0], B[0, :] = sign, big
    case = dense_case(gpu, kind, A, B)
    try:
        v = case.fp32("N", alpha)
        np.testing.assert_array_equal(v, np.outer(sign, np.full(N, 2.0 ** 119)).astype(np.float32))
        same = (np.arange(M) % 4) < 2
        bias = np.where((sign > 0) == same, 0x7F7F, 0xFF7F).astype(np.uint16)
        got = case.bf16("N", np.zeros((M, N), np.uint16), alpha, bias)
        assert_bits(got, emulate(v, "N", bias))
        assert np.all(got[same & (sign > 0)] == 0x7F80) and np.all(got[same & (sign < 0)] == 0xFF80)
        assert not np.any((got[~same] & 0x7F80) == 0x7F80)
    finally:
        case.destroy()


@pytest.mark.parametrize("kind", ["bf16", "e5m2/e5m2"])      # e5m2 encodes Inf and NaN; the bf16 operator takes them widened
@pytest.mark.parametrize("transc", ["N", "T"])
def test_non_finite_b_and_bias_reach_exactly_the_float64_outputs(gpu, kind, transc):
    """every group keeps exactly two elements, so the tensor core multiplies exactly the kept products: Inf / NaN in B reach
    the rows whose kept element meets them, a NaN or Inf bias its row, as the float64 product of the kept elements says"""
    M, N, K = 256, 272, 256
    masks = np.random.default_rng(4).choice([m for m in LEGAL if bin(m).count("1") == 2], (M, K // 4))
    A8, B8, _ = operands(M, N, K, "N", "N", 4, "e5m2", "e5m2")
    A8 = make24(M, K, 4, "e5m2", masks)
    specials = {(17, 40): 0x7C, (200, 100): 0xFC, (90, 263): 0x7E}     # +Inf, -Inf, NaN
    for (k, n), code in specials.items():
        B8[k, n] = code
    a, b = dec(A8, "e5m2"), dec(B8, "e5m2")
    want = a @ np.where(np.isfinite(b), b, 0.0)
    for (k, n) in specials:
        hit = a[:, k] != 0
        want[hit, n] = a[hit, k] * b[k, n]                                 # one non-finite product per column
    ops = (widen(A8, "e5m2"), widen(B8, "e5m2")) if kind == "bf16" else (A8, B8)
    case = Case(gpu, kind, *ops, "N")
    try:
        v = case.fp32(transc)
        vt = v.T if transc == "T" else v
        np.testing.assert_array_equal(np.isnan(vt), np.isnan(want))
        np.testing.assert_array_equal(np.isposinf(vt), np.isposinf(want))
        np.testing.assert_array_equal(np.isneginf(vt), np.isneginf(want))
        assert np.isnan(want).any() and np.isinf(want).any()
        bias = dyadic16(M, np.random.default_rng(5))
        bias[3], bias[77], bias[150] = NAN16, 0x7F80, 0xFF80
        got = case.bf16(transc, np.zeros(case.c_shape(transc), np.uint16), 1.0, bias)
        assert_bits(got, emulate(v, transc, bias))
        with np.errstate(invalid="ignore"):
            want_b = want + values16(bias).astype(np.float64)[:, None]
        gt = got.T if transc == "T" else got
        np.testing.assert_array_equal(is_nan16(gt), np.isnan(want_b))
        np.testing.assert_array_equal((gt & 0x7FFF) == 0x7F80, np.isinf(want_b))
    finally:
        case.destroy()


@pytest.mark.parametrize("kind", ["bf16", "e4m3/e4m3"])
@pytest.mark.parametrize("transc,N", [("N", 264), ("N", 130), ("T", 264)])     # TMA boxes; per-thread 'N'; per-thread 'T'
def test_nan_filled_c_is_not_read_with_beta_0(gpu, kind, transc, N):
    case, _, _ = make_case(gpu, kind, 300, N, 256, "N", 12)
    try:
        v = case.fp32(transc)
        got = case.bf16(transc, np.full(case.c_shape(transc), NAN16, np.uint16), 1.0, dyadic16(300, np.random.default_rng(1)), 0.0)
        assert not is_nan16(got).any()
    finally:
        case.destroy()


def test_negative_zero_survives_a_null_bias(gpu):
    """alpha = -1 and +1 turn a zero accumulator into -0 for one of them; a NULL bias keeps it, a bias of +0 makes it +0"""
    M, N, K = 256, 264, 256
    case, _, _ = make_case(gpu, "e4m3/e4m3", M, N, K, "N", 13)
    case.dB.upload(np.zeros((K, case.ldb), np.uint8))                  # B = +0: every accumulator is a zero
    try:
        negzero = 0
        for alpha in (-1.0, 1.0):
            v = case.fp32("N", alpha)
            assert np.all(v == 0)
            negzero += int(np.signbit(v).sum())
            got = case.bf16("N", np.full((M, N), NAN16, np.uint16), alpha)
            np.testing.assert_array_equal(got, bits16(v))
            plus = case.bf16("N", np.full((M, N), NAN16, np.uint16), alpha, np.zeros(M, np.uint16))
            assert np.all(plus == 0)
        assert negzero == M * N
    finally:
        case.destroy()


# ---- both store paths ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["bf16", "e5m2/e4m3"])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_both_store_paths_same_bits(gpu, kind, beta):
    """d_c 16-byte aligned with ldc % 8 = 0 (TMA boxes for beta = 0, 16-byte stores for beta = 1), the same C 2 bytes off
    (element stores), and a pitch of N + 4 (no 16-byte rows): identical bits"""
    M, N, K = 300, 264, 256
    case, _, _ = make_case(gpu, kind, M, N, K, "T", 14)
    rng = np.random.default_rng(14)
    try:
        bias = dyadic16(M, rng)
        C0 = dyadic16((M, N), rng)
        outs = [case.bf16("N", C0, 0.5, bias, beta, ldc=N, c_offset=0), case.bf16("N", C0, 0.5, bias, beta, ldc=N, c_offset=2)]
        Cw = np.full((M, N + 4), NAN16, np.uint16)
        Cw[:, :N] = C0
        outs.append(case.bf16("N", Cw, 0.5, bias, beta, ldc=N + 4, c_offset=0)[:, :N])
        for o in outs[1:]:
            np.testing.assert_array_equal(o, outs[0])
        assert_bits(outs[0], emulate(case.fp32("N", 0.5), "N", bias, beta, C0))
    finally:
        case.destroy()


# ---- guard bands -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["bf16", "e4m3/e4m3"])
@pytest.mark.parametrize("N", [3, 16, 130, 257])
@pytest.mark.parametrize("transc", ["N", "T"])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_guard_bands(gpu, kind, N, transc, beta):
    """NaN sentinels in C's pitch padding and in rows past C stay; with beta = 0 NaN inside C disappears"""
    M, K = 300, 256
    case, _, _ = make_case(gpu, kind, M, N, K, "N", N)
    rng = np.random.default_rng(N)
    try:
        shape = case.c_shape(transc)
        rows, ldc = (shape[0] + 5, (shape[1] + 8 + 7) // 8 * 8) if transc == "N" else (shape[0] + 5, shape[1] + 9)
        Cs = np.full((rows, ldc), NAN16, np.uint16)
        C0 = dyadic16(shape, rng)
        if beta == 0.0:
            C0[::7, ::5] = NAN16
        Cs[:shape[0], :shape[1]] = C0
        bias = dyadic16(M, rng)
        got = case.bf16(transc, Cs, 0.25, bias, beta, ldc=ldc)
        assert_bits(np.ascontiguousarray(got[:shape[0], :shape[1]]), emulate(case.fp32(transc, 0.25), transc, bias, beta, C0))
        pad = np.ones_like(got, bool)
        pad[:shape[0], :shape[1]] = False
        np.testing.assert_array_equal(got[pad], Cs[pad])
    finally:
        case.destroy()


# ---- streams and graphs ----------------------------------------------------------------------------------------------------
def test_two_handles_on_two_streams(gpu):
    xs = gpu
    cases, bufs, serial = [], [], []
    rng = np.random.default_rng(40)
    for i, (kind, M, N, K) in enumerate([("bf16", 512, 384, 256), ("e5m2/e5m2", 300, 528, 384)]):
        case, _, _ = make_case(xs, kind, M, N, K, "T", 40 + i)
        bias = dyadic16(M, rng)
        C0 = np.zeros((M, N), np.uint16)
        cases.append(case)
        serial.append(case.bf16("N", C0, 0.5, bias))
        bufs.append((xs.DeviceBuffer.from_numpy(C0), xs.DeviceBuffer.from_numpy(bias)))
    streams = [xs.Stream(), xs.Stream()]
    try:
        for rep in range(3):
            for case, (dC, dbias), st in zip(cases, bufs, streams):
                case.op.execute(case.dB, dC, case.N, ldb=case.ldb, transb="T", bias=dbias, c_dtype="bf16", stream=st, **case.kw(0.5))
            for st in streams:
                st.synchronize()
            for case, (dC, _), want in zip(cases, bufs, serial):
                np.testing.assert_array_equal(dC.to_numpy(np.uint16, (case.M, case.N)), want)
        xs.check()
    finally:
        for case in cases:
            case.destroy()
        for dC, dbias in bufs:
            dC.free(); dbias.free()
        for st in streams:
            st.destroy()


@pytest.mark.parametrize("kind", ["bf16", "e4m3/e4m3"])
def test_graph_replay_with_new_b_and_new_bias(gpu, kind):
    xs, L = gpu, gpu.load()
    M, N, K = 512, 400, 384
    case, _, _ = make_case(xs, kind, M, N, K, "N", 50)
    rng = np.random.default_rng(50)
    a_fmt, b_fmt = fmts(kind)
    Bs = [enc(rng.choice(DYADIC, (K, N)), b_fmt) for _ in range(2)]
    Bs = [widen(b, b_fmt) for b in Bs] if kind == "bf16" else Bs
    biases = [dyadic16(M, rng) for _ in range(2)]
    dC, dbias = xs.DeviceBuffer(2 * M * N), xs.DeviceBuffer.from_numpy(biases[0])
    case.dB.upload(Bs[0])
    st = xs.Stream()
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    case.op.execute(case.dB, dC, N, ldb=case.ldb, bias=dbias, c_dtype="bf16", stream=st, **case.kw(2.0))
    graph = L.libxsmm_b200_graph_end(st.ptr)
    xs.check()
    assert graph
    try:
        for B, bias in zip(Bs + Bs[:1], biases + biases[::-1][:1]):
            case.dB.upload(B)
            v = case.fp32("N", 2.0)
            dbias.upload(bias)
            n0 = xs.launch_count()
            assert 0 == L.libxsmm_b200_graph_launch(graph, st.ptr)
            st.synchronize()
            assert xs.launch_count() == n0
            assert_bits(dC.to_numpy(np.uint16, (M, N)), emulate(v, "N", bias))
    finally:
        L.libxsmm_b200_graph_destroy(graph)
        case.destroy(); dC.free(); dbias.free(); st.destroy()


# ---- rejections ------------------------------------------------------------------------------------------------------------
def test_execute_rejections_launch_nothing(gpu):
    xs = gpu
    M, N, K = 256, 64, 192
    A8, _, _ = operands(M, N, K, "N", "N", 60)
    op8, op16 = xs.Sp24(A8, fmt="e4m3"), xs.Sp24(widen(A8, "e4m3"))
    dB, dC, dbias = xs.DeviceBuffer(2 * K * max(N, K) + 64), xs.DeviceBuffer(2 * M * max(N, M) + 64), xs.DeviceBuffer(2 * M + 64)
    b, c, bs = dB.ptr, dC.ptr, dbias.ptr

    def e16(h, tb, tc, n, db, ldb, bias, dc, ldc):
        xs.sp24_execute_bf16out(h, tb, tc, n, db, ldb, bias, 0.0, dc, ldc)

    def e8(h, tb, tc, n, db, ldb, bias, dc, ldc, fmt=0):
        xs.sp24_execute_fp8_bf16out(h, tb, tc, n, db, fmt, ldb, 1.0, bias, 0.0, dc, ldc)

    h16, h8 = op16.handle, op8.handle
    cases = [
        (lambda: e16(None, "N", "N", N, b, N, bs, c, N), "NULL handle"),
        (lambda: e8(None, "N", "N", N, b, N, bs, c, N), "NULL handle"),
        (lambda: e16(h8, "N", "N", N, b, N, bs, c, N), "FP8 operator"),             # the bf16 entry refuses an FP8 handle
        (lambda: e8(h16, "N", "N", N, b, N, bs, c, N), "bf16 operator"),            # and the reverse
        (lambda: e16(h16, "X", "N", N, b, N, bs, c, N), "transb='X'"),
        (lambda: e8(h8, "N", "q", N, b, N, bs, c, N), "transc='q'"),
        (lambda: e8(h8, "N", "N", N, b, N, bs, c, N, fmt=2), "b_format=2"),
        (lambda: e16(h16, "N", "N", -1, b, N, bs, c, N), "N=-1"),
        (lambda: e16(h16, "N", "N", N, b, N - 8, bs, c, N), "ldb=56"),
        (lambda: e8(h8, "N", "T", N, b, N, bs, c, M - 1), "ldc=255"),
        (lambda: e16(h16, "N", "N", N, None, N, bs, c, N), "NULL d_b"),
        (lambda: e8(h8, "N", "N", N, b, N, bs, None, N), "NULL d_b or d_c"),
        (lambda: e16(h16, "N", "N", N, b + 2, N, bs, c, N), "16-byte aligned"),
        (lambda: e8(h8, "N", "N", N, b, N + 8, bs, c, N), "ldb=72"),
        (lambda: e16(h16, "N", "N", N, b, N, bs, c + 1, N), "2-byte aligned"),
        (lambda: e16(h16, "T", "T", N, b, K, bs + 1, c, M), "2-byte aligned"),
        (lambda: e8(h8, "N", "N", N, b, N, bs, c + 3, N), "2-byte aligned"),
        (lambda: e8(h8, "T", "N", N, b, K, bs + 1, c, N), "2-byte aligned"),
    ]
    try:
        for call, frag in cases:
            xs.clear_error()
            n0 = xs.launch_count()
            call()
            code, msg = xs.last_error()
            assert xs.launch_count() == n0, frag
            assert code == -97 and frag in msg, (frag, code, msg)
        for call in (lambda: e16(h16, "N", "N", 0, None, 0, None, None, 0), lambda: e8(h8, "N", "N", 0, None, 0, None, None, 0)):
            xs.clear_error()
            n0 = xs.launch_count()
            call()                                                                  # N = 0 does nothing
            assert xs.launch_count() == n0 and xs.last_error()[0] == 0
    finally:
        xs.clear_error()
        op8.destroy(); op16.destroy(); dB.free(); dC.free(); dbias.free()


# ---- Sp24.linear -----------------------------------------------------------------------------------------------------------
def bf16_ulp(y):
    return np.ldexp(1.0, np.frexp(np.maximum(np.abs(y), np.finfo(np.float32).tiny))[1] - 8)


@pytest.mark.parametrize("with_bias", [False, True])
def test_linear_bf16_operator(gpu, with_bias):
    import torch
    M, K = 384, 256
    rng = np.random.default_rng(70)
    masks = rng.choice(LEGAL, (M, K // 4))
    keep = ((masks[:, :, None] >> np.arange(4)) & 1).astype(bool).reshape(M, K)
    W = torch.from_numpy(bits16(np.where(keep, rng.uniform(0.25, 2.0, (M, K)) * rng.choice([-1.0, 1.0], (M, K)), 0.0)).view(np.int16)).view(torch.bfloat16).cuda()
    x = (torch.rand((3, 67, K), device="cuda") - 0.5).to(torch.bfloat16)
    bias = (torch.rand(M, device="cuda") - 0.5).to(torch.bfloat16) if with_bias else None
    op = gpu.Sp24(W)
    try:
        n0 = gpu.launch_count()
        y = op.linear(x, bias)
        torch.cuda.synchronize()
        assert gpu.launch_count() == n0 + 1 and gpu.last_compute_kernel() == "sp24_compute_kernel_bf16out"
        assert y.shape == (3, 67, M) and y.dtype == torch.bfloat16 and y.device == x.device
        y2 = torch.empty((201, M), dtype=torch.bfloat16, device="cuda")
        op.execute(x, y2, 201, ldb=K, ldc=M, transb="T", transc="T", bias=bias, stream=torch.cuda.current_stream())
        torch.cuda.synchronize()
        assert torch.equal(y.view(-1, M).view(torch.int16), y2.view(torch.int16))
        xd, wd = x.double().cpu().view(-1, K), W.double().cpu()
        want = torch.nn.functional.linear(xd, wd, None if bias is None else bias.double().cpu()).numpy()
        bound = 4e-6 * (xd.abs() @ wd.abs().t()).numpy() + (0 if bias is None else 4e-6 * np.abs(bias.double().cpu().numpy()))
        got = y.view(-1, M).double().cpu().numpy()
        assert np.all(np.abs(got - want) <= bound + 0.5 * bf16_ulp(got))
        s = torch.cuda.Stream()                                          # a non-default current stream
        with torch.cuda.stream(s):
            x_s = x * 1                                                  # produced on s: linear must be ordered after it
            y3 = op.linear(x_s, bias)
        s.synchronize()
        assert torch.equal(y3.view(torch.int16), y.view(torch.int16))
    finally:
        op.destroy()


@pytest.mark.parametrize("with_bias", [False, True])
def test_linear_fp8_operator_against_scaled_mm(gpu, with_bias):
    import torch
    M, K = 512, 512
    F8 = torch.float8_e4m3fn
    rng = np.random.default_rng(71)
    masks = rng.choice(LEGAL, (M, K // 4))
    keep = torch.from_numpy(((masks[:, :, None] >> np.arange(4)) & 1).astype(bool).reshape(M, K)).cuda()
    Wf = torch.where(keep, torch.randn((M, K), device="cuda"), torch.zeros((), device="cuda"))
    sw = float(Wf.abs().max()) / 448.0
    W8 = (Wf / sw).to(F8)
    xf = torch.randn((4, 64, K), device="cuda")
    sx = float(xf.abs().max()) / 448.0
    x8 = (xf / sx).to(F8)
    bias = (torch.rand(M, device="cuda") - 0.5).to(torch.bfloat16) if with_bias else None
    op = gpu.Sp24(W8)
    try:
        y = op.linear(x8, bias, alpha=sx * sw)
        torch.cuda.synchronize()
        assert gpu.last_compute_kernel() == "sp24_compute_kernel_fp8_bf16out"
        assert y.shape == (4, 64, M) and y.dtype == torch.bfloat16
        ref = torch._scaled_mm(x8.view(-1, K), W8.t(), scale_a=torch.tensor(sx, device="cuda"), scale_b=torch.tensor(sw, device="cuda"),
                               out_dtype=torch.bfloat16, bias=bias)
        a = x8.view(-1, K).double().cpu()
        w = W8.double().cpu()
        bound = 4e-6 * sx * sw * (a.abs() @ w.abs().t()).numpy() + (0 if bias is None else 4e-6 * np.abs(bias.double().cpu().numpy()))
        got, want = y.view(-1, M).double().cpu().numpy(), ref.double().cpu().numpy()
        assert np.all(np.abs(got - want) <= bound + bf16_ulp(np.maximum(np.abs(got), np.abs(want))))   # each rounds by half an ulp
    finally:
        op.destroy()
