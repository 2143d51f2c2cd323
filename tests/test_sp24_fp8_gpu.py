"""GPU tests of the fixed 2:4-sparse FP8 operators (libxsmm_b200_sp24_create_fp8 / _execute_fp8, csrc/sp24.cu): A in e4m3 or
e5m2 is compressed once, execute multiplies on the 8-bit structured-sparse tensor core with A, its metadata and B fetched by
TMA, and C = alpha (A . op(B)) + beta C in fp32.

Exact data: A, B and C0 hold small dyadic values ({+-0.5, +-1, +-1.5, +-2, +-3}, exact in both formats) and alpha, beta are
powers of two, so every partial sum is exact in fp32 and C must equal the float64 product bit for bit.  Random data over a
format's range is held to the bf16 operator's bound |alpha| 4e-6 (|A|.|B| + |beta| |C0|) against the float64 product of the
kept elements."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
KERNEL = "sp24_compute_kernel_fp8"
LEGAL = [m for m in range(16) if bin(m).count("1") <= 2]      # the eleven keep masks of a 2:4 group
DYADIC = np.array([0.5, -0.5, 1.0, -1.0, 1.5, -1.5, 2.0, -2.0, 3.0, -3.0])
NAN8 = {"e4m3": [0x7F, 0xFF], "e5m2": [0x7D, 0x7E, 0x7F, 0xFD, 0xFE, 0xFF]}
FMTS = [("e4m3", "e4m3"), ("e5m2", "e5m2"), ("e4m3", "e5m2"), ("e5m2", "e4m3")]


def tdtype(fmt):
    import torch
    return {"e4m3": torch.float8_e4m3fn, "e5m2": torch.float8_e5m2}[fmt]


def enc(x, fmt):
    """float values (exact in fmt, or rounded by torch) -> FP8 bytes"""
    import torch
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(tdtype(fmt)).view(torch.uint8).numpy()


def dec(u8, fmt):
    import torch
    return torch.from_numpy(np.ascontiguousarray(u8, np.uint8)).view(tdtype(fmt)).to(torch.float32).numpy().astype(np.float64)


def kept(A8, fmt):
    """float64 image of the kept elements (ordered nonzeros; +-0 and NaN dropped, Inf kept)"""
    a = dec(A8, fmt)
    return np.where(np.isnan(a), 0.0, a)


def random_range(shape, fmt, rng):
    """finite nonzero FP8 bytes spread over the whole format (both signs, every exponent)"""
    top = 0x7E if fmt == "e4m3" else 0x7B
    return (rng.integers(1, top + 1, shape) | (rng.integers(0, 2, shape) << 7)).astype(np.uint8)


def make24(M, K, seed, fmt, masks=None, exact=True):
    """random 2:4 FP8 A: every group takes one of the legal masks"""
    rng = np.random.default_rng(seed)
    G = (K + 3) // 4
    m = rng.choice(LEGAL, (M, G)) if masks is None else masks
    keep = ((m[:, :, None] >> np.arange(4)) & 1).astype(bool).reshape(M, 4 * G)[:, :K]
    v = enc(rng.choice(DYADIC, (M, K)), fmt) if exact else random_range((M, K), fmt, rng)
    return np.where(keep, v, 0).astype(np.uint8)


def pad_b(B8, fmt):
    """B goes through TMA: rows padded to 16 bytes, NaN in the padding"""
    ld = (B8.shape[1] + 15) // 16 * 16
    if ld == B8.shape[1]:
        return B8, ld
    Bp = np.full((B8.shape[0], ld), NAN8[fmt][0], np.uint8)
    Bp[:, :B8.shape[1]] = B8
    return Bp, ld


def run(xs, op, B8, b_fmt, C0, N, transb="N", transc="N", alpha=1.0, beta=0.0, ldb=None, ldc=None):
    """one execute on fresh device buffers; returns C as stored"""
    if ldb is None:
        B8, ldb = pad_b(B8, b_fmt)
    dB, dC = xs.DeviceBuffer.from_numpy(B8), xs.DeviceBuffer.from_numpy(C0)
    try:
        n0 = xs.launch_count()
        op.execute(dB, dC, N, ldb=ldb, ldc=ldc, beta=beta, transb=transb, transc=transc, alpha=alpha, b_fmt=b_fmt)
        xs.synchronize()
        assert xs.launch_count() == n0 + (1 if N > 0 else 0)
        if N > 0:
            assert xs.last_compute_kernel() == KERNEL
        return dC.to_numpy(np.float32, C0.shape)
    finally:
        dB.free(); dC.free()


def want_and_bound(A8, a_fmt, B8, b_fmt, C0, transb, transc, alpha, beta):
    a = kept(A8, a_fmt)
    b = dec(B8, b_fmt)
    if transb == "T":
        b = b.T
    c0 = C0.astype(np.float64)
    if transc == "T":
        c0 = c0.T
    want = alpha * (a @ b) + (beta * c0 if beta != 0 else 0.0)
    bound = 4e-6 * abs(alpha) * (np.abs(a) @ np.abs(b) + (abs(beta) * np.abs(c0) if beta != 0 else 0.0))
    return (want.T, bound.T) if transc == "T" else (want, bound)


def check_exact(C, *args):
    want, _ = want_and_bound(*args)
    np.testing.assert_array_equal(C.view(np.uint32), want.astype(np.float32).view(np.uint32))


def check_f64(C, *args):
    want, bound = want_and_bound(*args)
    err = np.abs(C.astype(np.float64) - want)
    assert np.all(np.isfinite(C))
    assert np.all(err <= bound), float((err - bound).max())


def operands(M, N, K, transb, transc, seed, a_fmt="e4m3", b_fmt="e4m3", exact=True):
    rng = np.random.default_rng(seed + 1)
    A8 = make24(M, K, seed, a_fmt, exact=exact)
    shape_b = (N, K) if transb == "T" else (K, N)
    B8 = enc(rng.choice(DYADIC, shape_b), b_fmt) if exact else random_range(shape_b, b_fmt, rng)
    C0 = rng.choice(DYADIC, (N, M) if transc == "T" else (M, N)).astype(np.float32)
    if not exact:
        C0 *= rng.uniform(0.5, 2.0, C0.shape).astype(np.float32)
    return A8, B8, C0


def case(xs, M, N, K, transb="N", transc="N", alpha=1.0, beta=0.0, a_fmt="e4m3", b_fmt="e4m3", seed=0, exact=True):
    A8, B8, C0 = operands(M, N, K, transb, transc, seed + M + N + K, a_fmt, b_fmt, exact)
    op = xs.Sp24(A8, fmt=a_fmt)
    try:
        C = run(xs, op, B8, b_fmt, C0, N, transb, transc, alpha, beta)
    finally:
        op.destroy()
    args = (A8, a_fmt, B8, b_fmt, C0, transb, transc, alpha, beta)
    (check_exact if exact else check_f64)(C, *args)
    xs.check()


# ---- exact parity ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [
    (300, 1, 72), (300, 3, 72), (300, 208, 72), (300, 257, 72),
    (300, 1, 200), (300, 3, 200), (300, 208, 200), (300, 257, 200),
    (300, 264, 520),              # K not a multiple of the slot's 256
    (33, 16, 256),                # one partial tile
    (4096, 2048, 256),            # 128 tiles: more than the CTA pairs
    (2560, 2560, 384),            # 100 tiles: the left-over ones are split into half tiles
    (4096, 4096, 4096),
])
def test_exact_parity(gpu, M, N, K):
    case(gpu, M, N, K, beta=0.5)


@pytest.mark.parametrize("transb", ["N", "T"])
@pytest.mark.parametrize("transc", ["N", "T"])
@pytest.mark.parametrize("beta", [0.0, 1.0, 0.5, -1.0])
@pytest.mark.parametrize("alpha", [1.0, 2.0 ** -6])
def test_trans_alpha_beta(gpu, transb, transc, beta, alpha):
    case(gpu, 520, 392, 328, transb, transc, alpha, beta, seed=7)


@pytest.mark.parametrize("a_fmt,b_fmt", FMTS)
@pytest.mark.parametrize("transb", ["N", "T"])
def test_formats_exact(gpu, a_fmt, b_fmt, transb):
    case(gpu, 300, 264, 520, transb, "N", 0.5, 1.0, a_fmt, b_fmt, seed=13)


@pytest.mark.parametrize("a_fmt,b_fmt", FMTS)
@pytest.mark.parametrize("transb,transc,beta", [("N", "N", 0.0), ("T", "T", 1.0)])
def test_float64_bound_over_the_format_range(gpu, a_fmt, b_fmt, transb, transc, beta):
    case(gpu, 520, 392, 1000, transb, transc, 2.0 ** -10, beta, a_fmt, b_fmt, seed=17, exact=False)


# ---- same product as the bf16 operator -------------------------------------------------------------------------------------
def widen(u8, fmt):
    return (dec(u8, fmt).astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)


@pytest.mark.parametrize("a_fmt,b_fmt", FMTS)
@pytest.mark.parametrize("transb,M,N,K", [("N", 512, 392, 512), ("T", 300, 257, 200), ("N", 4096, 1024, 4096)])
def test_same_bits_as_bf16(gpu, a_fmt, b_fmt, transb, M, N, K):
    A8, B8, C0 = operands(M, N, K, transb, "N", 5, a_fmt, b_fmt)
    op8, op16 = gpu.Sp24(A8, fmt=a_fmt), gpu.Sp24(widen(A8, a_fmt))
    try:
        C = run(gpu, op8, B8, b_fmt, C0, N, transb, "N", 1.0, 1.0)
        B16 = widen(B8, b_fmt)
        ld16 = (B16.shape[1] + 7) // 8 * 8
        B16p = np.zeros((B16.shape[0], ld16), np.uint16)
        B16p[:, :B16.shape[1]] = B16
        dB, dC = gpu.DeviceBuffer.from_numpy(B16p), gpu.DeviceBuffer.from_numpy(C0)
        op16.execute(dB, dC, N, ldb=ld16, beta=1.0, transb=transb)
        gpu.synchronize()
        C16 = dC.to_numpy(np.float32, C0.shape)
        dB.free(); dC.free()
        np.testing.assert_array_equal(C.view(np.uint32), C16.view(np.uint32))
    finally:
        op8.destroy(); op16.destroy()


# ---- keep rule -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["e4m3", "e5m2"])
def test_every_group_pattern_and_special_values(gpu, fmt):
    """the eleven legal masks at every group position of a 256-k slot, +-0 and every NaN encoding dropped (a group of two
    values and two NaN is legal), e5m2 +-Inf kept"""
    M, N, K = 256, 256, 512
    G = K // 4
    masks = np.array([[LEGAL[(r * 7 + g * 5 + (r >> 4)) % 11] for g in range(G)] for r in range(M)])
    A8 = make24(M, K, 3, fmt, masks)
    rng = np.random.default_rng(3)
    nans = NAN8[fmt]
    for r in range(0, M, 3):
        g = (r * 13) % G
        A8[r, 4 * g:4 * g + 4] = [0x80, nans[r % len(nans)], 0x00, nans[(r + 1) % len(nans)]]
        g2 = (g + 7) % G
        A8[r, 4 * g2:4 * g2 + 4] = enc([1.5, 0.0, -0.5, 0.0], fmt)
        A8[r, 4 * g2 + 1], A8[r, 4 * g2 + 3] = nans[-1], 0x80
    inf_rows = []
    if fmt == "e5m2":
        for r in range(1, M, 37):
            g = (r * 5 + 3) % G
            A8[r, 4 * g:4 * g + 4] = [0, 0x7C if r % 2 else 0xFC, 0, 0]
            inf_rows.append(r)
    B8 = enc(rng.choice(DYADIC, (K, N)), "e4m3")
    C0 = rng.choice(DYADIC, (M, N)).astype(np.float32)
    op = gpu.Sp24(A8, fmt=fmt)
    try:
        C = run(gpu, op, B8, "e4m3", C0, N, beta=1.0)
    finally:
        op.destroy()
    want, _ = want_and_bound(A8, fmt, B8, "e4m3", C0, "N", "N", 1.0, 1.0)
    want32 = want.astype(np.float32)
    np.testing.assert_array_equal(np.isinf(C), np.isinf(want32))
    assert np.all(np.isinf(C[inf_rows])) if inf_rows else True
    finite = np.isfinite(want32)
    np.testing.assert_array_equal(C[finite].view(np.uint32), want32[finite].view(np.uint32))


@pytest.mark.parametrize("fmt", ["e4m3", "e5m2"])
@pytest.mark.parametrize("M,K,row,group,nkept", [(256, 256, 0, 0, 3), (300, 200, 299, 49, 4), (300, 203, 137, 50, 3)])
def test_create_rejects_a_that_is_not_2_4(gpu, fmt, M, K, row, group, nkept):
    """one group keeping three or four elements -- the first, the last, or the partial tail group of a row (K % 4 = 3) --
    gives NULL with -96 naming it; the failed create gives its device memory back"""
    import torch
    A8 = make24(M, K, 9, fmt)
    A8[row, 4 * group:4 * group + nkept] = enc([1.0, -2.0, 3.0, 0.5][:nkept], fmt)
    for attempt in range(2):           # the first attempt may grow the runtime's pools; the second must leave memory as it was
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        gpu.clear_error()
        h = gpu.sp24_create_fp8(M, K, K, A8, {"e4m3": 0, "e5m2": 1}[fmt])
        code, msg = gpu.last_error()
        gpu.clear_error()
        assert not h
        assert code == -96, msg
        assert "sp24_create_fp8" in msg and "row %d, group %d" % (row, group) in msg, msg
        free1 = torch.cuda.mem_get_info()[0]
    assert free1 == free0


# ---- create paths ----------------------------------------------------------------------------------------------------------
def test_host_device_torch_and_bytes_give_identical_c(gpu):
    import torch
    M, N, K = 300, 264, 200
    lda = 224
    A8, B8, C0 = operands(M, N, K, "N", "N", 21, "e5m2", "e4m3")
    Apad = np.full((M, lda), 0x7F, np.uint8)            # NaN in A's pitch padding is never read
    Apad[:, :K] = A8
    ops = [gpu.Sp24(Apad[:, :K], fmt="e5m2")]
    assert ops[0].lda == lda
    dA = gpu.DeviceBuffer.from_numpy(A8)
    h = gpu.sp24_create_fp8(M, K, K, dA.ptr, 1)
    dA.free()                                          # read only during create
    gpu.check()
    assert h
    op_d = gpu.Sp24.__new__(gpu.Sp24)
    op_d.M, op_d.K, op_d.lda, op_d.fp8, op_d.format, op_d.handle = M, K, K, True, 1, h
    ops.append(op_d)
    ops.append(gpu.Sp24(torch.from_numpy(A8).view(torch.float8_e5m2).cuda()))
    ops.append(gpu.Sp24(torch.from_numpy(A8).view(torch.float8_e5m2)))          # a host tensor
    try:
        Cs = [run(gpu, op, B8, "e4m3", C0, N, beta=1.0) for op in ops]
        b = torch.from_numpy(pad_b(B8, "e4m3")[0]).view(torch.float8_e4m3fn).cuda()
        c = torch.from_numpy(C0).cuda()
        ops[2].execute(b, c, N, ldb=b.shape[1], beta=1.0, stream=torch.cuda.current_stream())
        torch.cuda.synchronize()
        Cs.append(c.cpu().numpy())
        for C in Cs[1:]:
            np.testing.assert_array_equal(C.view(np.uint32), Cs[0].view(np.uint32))
        check_exact(Cs[0], A8, "e5m2", B8, "e4m3", C0, "N", "N", 1.0, 1.0)
    finally:
        for op in ops:
            op.destroy()


# ---- guard bands and special values ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [3, 16, 130, 257])
@pytest.mark.parametrize("transc", ["N", "T"])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_guard_bands(gpu, N, transc, beta):
    """NaN sentinels in C's pitch padding and past M stay, NaN in B's padding columns does not leak, NaN in C0 disappears with
    beta = 0.  transc = 'N', beta = 0 with N % 4 = 0 takes the TMA-box epilogue."""
    M, K = 300, 256
    rng = np.random.default_rng(N)
    A8 = make24(M, K, N, "e4m3")
    ldb = (N + 16 + 15) // 16 * 16
    B8 = np.full((K, ldb), 0x7F, np.uint8)
    B8[:, :N] = enc(rng.choice(DYADIC, (K, N)), "e4m3")
    rows, ldc = (M + 5, (N + 7) // 4 * 4) if transc == "N" else (N + 5, M + 4)
    Cs = np.full((rows, ldc), np.nan, np.float32)
    C0 = rng.choice(DYADIC, (M, N) if transc == "N" else (N, M)).astype(np.float32)
    if beta == 0.0:
        C0[::7, ::5] = np.nan
    Cs[:C0.shape[0], :C0.shape[1]] = C0
    op = gpu.Sp24(A8, fmt="e4m3")
    try:
        C = run(gpu, op, B8, "e4m3", Cs, N, "N", transc, 0.25, beta, ldb=ldb, ldc=ldc)
    finally:
        op.destroy()
    inner = np.ascontiguousarray(C[:C0.shape[0], :C0.shape[1]])
    check_exact(inner, A8, "e4m3", np.ascontiguousarray(B8[:, :N]), "e4m3", C0, "N", transc, 0.25, beta)
    pad = np.ones_like(C, bool)
    pad[:C0.shape[0], :C0.shape[1]] = False
    np.testing.assert_array_equal(C[pad].view(np.uint32), Cs[pad].view(np.uint32))


def test_non_finite_b_taints_no_more_than_the_dense_product(gpu):
    M, N, K = 256, 272, 256
    A8, B8, C0 = operands(M, N, K, "N", "N", 8, "e4m3", "e5m2")
    B8[17, 40] = 0x7C             # +Inf
    B8[200, 100] = 0xFC           # -Inf
    B8[90, 263] = 0x7E            # NaN
    op = gpu.Sp24(A8, fmt="e4m3")
    try:
        C = run(gpu, op, B8, "e5m2", C0, N)
    finally:
        op.destroy()
    b = dec(B8, "e5m2")
    tainted = np.broadcast_to(~np.all(np.isfinite(b), axis=0), C.shape)   # the dense product multiplies every A[m, k], zeros included
    assert not np.any(~np.isfinite(C) & ~tainted)
    clean = ~tainted[0]
    want, _ = want_and_bound(A8, "e4m3", np.where(np.isfinite(b), B8, 0).astype(np.uint8), "e5m2", C0, "N", "N", 1.0, 0.0)
    np.testing.assert_array_equal(C[:, clean], want[:, clean].astype(np.float32))


# ---- launch behaviour ------------------------------------------------------------------------------------------------------
def test_two_handles_on_two_streams(gpu):
    xs = gpu
    shapes = [(512, 384, 256, "e4m3"), (300, 528, 384, "e5m2")]
    ops, bufs, serial = [], [], []
    for i, (M, N, K, fmt) in enumerate(shapes):
        A8, B8, C0 = operands(M, N, K, "T", "N", 40 + i, fmt, fmt)
        ops.append(xs.Sp24(A8, fmt=fmt))
        serial.append(run(xs, ops[-1], B8, fmt, C0, N, "T", alpha=0.5))
        bufs.append((xs.DeviceBuffer.from_numpy(B8), xs.DeviceBuffer.from_numpy(C0), N, C0.shape, fmt))
    streams = [xs.Stream(), xs.Stream()]
    try:
        for rep in range(3):
            for op, (dB, dC, N, shp, fmt), st in zip(ops, bufs, streams):
                op.execute(dB, dC, N, transb="T", alpha=0.5, b_fmt=fmt, stream=st)
            for st in streams:
                st.synchronize()
            for (dB, dC, N, shp, fmt), C in zip(bufs, serial):
                np.testing.assert_array_equal(dC.to_numpy(np.float32, shp).view(np.uint32), C.view(np.uint32))
        xs.check()
    finally:
        for op in ops:
            op.destroy()
        for dB, dC, _, _, _ in bufs:
            dB.free(); dC.free()
        for st in streams:
            st.destroy()


def test_graph_replay_with_new_b(gpu):
    xs, L = gpu, gpu.load()
    M, N, K = 512, 400, 384
    A8, _, C0 = operands(M, N, K, "N", "N", 50)
    rng = np.random.default_rng(50)
    Bs = [enc(rng.choice(DYADIC, (K, N)), "e4m3") for _ in range(2)]
    op = xs.Sp24(A8, fmt="e4m3")
    dB, dC = xs.DeviceBuffer.from_numpy(Bs[0]), xs.DeviceBuffer.from_numpy(C0)
    st = xs.Stream()
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    op.execute(dB, dC, N, alpha=2.0, b_fmt="e4m3", stream=st)
    graph = L.libxsmm_b200_graph_end(st.ptr)
    xs.check()
    assert graph
    try:
        for B8 in Bs + Bs[:1]:
            want = run(xs, op, B8, "e4m3", C0, N, alpha=2.0)
            dB.upload(B8)
            n0 = xs.launch_count()
            assert 0 == L.libxsmm_b200_graph_launch(graph, st.ptr)
            st.synchronize()
            assert xs.launch_count() == n0
            np.testing.assert_array_equal(dC.to_numpy(np.float32, C0.shape).view(np.uint32), want.view(np.uint32))
    finally:
        L.libxsmm_b200_graph_destroy(graph)
        op.destroy(); dB.free(); dC.free(); st.destroy()


def test_execute_rejections_launch_nothing(gpu):
    xs = gpu
    M, N, K = 256, 64, 192
    A8, B8, C0 = operands(M, N, K, "N", "N", 60)
    op = xs.Sp24(A8, fmt="e4m3")
    op16 = xs.Sp24(widen(A8, "e4m3"))
    dB, dC = xs.DeviceBuffer(K * max(N, K) + 64), xs.DeviceBuffer(4 * M * max(N, M) + 64)
    h = op.handle
    cases = [
        ((h, "X", "N", N, dB.ptr, 0, N, dC.ptr, N), "transb='X'"),
        ((h, "N", "q", N, dB.ptr, 0, N, dC.ptr, N), "transc='q'"),
        ((h, "N", "N", N, dB.ptr, 2, N, dC.ptr, N), "b_format=2"),
        ((h, "N", "N", -1, dB.ptr, 0, N, dC.ptr, N), "N=-1"),
        ((h, "N", "N", N, dB.ptr, 0, N - 16, dC.ptr, N), "ldb=48"),
        ((h, "T", "N", N, dB.ptr, 0, K - 16, dC.ptr, N), "ldb=176"),
        ((h, "N", "N", N, dB.ptr, 0, N, dC.ptr, N - 1), "ldc=63"),
        ((h, "N", "T", N, dB.ptr, 0, N, dC.ptr, M - 1), "ldc=255"),
        ((h, "N", "N", N, None, 0, N, dC.ptr, N), "NULL d_b"),
        ((h, "N", "N", N, dB.ptr, 0, N, None, N), "NULL d_b or d_c"),
        ((h, "N", "N", N, dB.ptr + 8, 0, N, dC.ptr, N), "16-byte aligned"),
        ((h, "N", "N", N, dB.ptr, 0, N + 8, dC.ptr, N), "ldb=72"),
        ((op16.handle, "N", "N", N, dB.ptr, 0, N, dC.ptr, N), "bf16 operator"),
    ]
    try:
        for args, frag in cases:
            xs.clear_error()
            n0 = xs.launch_count()
            xs.sp24_execute_fp8(args[0], *args[1:5], args[5], args[6], 1.0, 0.0, args[7], args[8])
            code, msg = xs.last_error()
            assert xs.launch_count() == n0, frag
            assert code == -97 and frag in msg, (frag, code, msg)
        xs.clear_error()
        n0 = xs.launch_count()
        xs.sp24_execute(h, "N", "N", N, dB.ptr, N, 0.0, dC.ptr, N)          # the bf16 entry refuses an FP8 handle
        code, msg = xs.last_error()
        assert xs.launch_count() == n0 and code == -97 and "FP8 operator" in msg, msg
        xs.clear_error()
        n0 = xs.launch_count()
        xs.sp24_execute_fp8(h, "N", "N", 0, None, 0, 0, 1.0, 0.0, None, 0)   # N = 0 does nothing
        assert xs.launch_count() == n0 and xs.last_error()[0] == 0
    finally:
        xs.clear_error()
        op.destroy(); op16.destroy(); dB.free(); dC.free()


def test_other_device_is_rejected(gpu):
    xs = gpu
    if xs.device_count() < 2:
        pytest.skip("one device")
    M, N, K = 128, 64, 128
    A8, B8, C0 = operands(M, N, K, "N", "N", 70)
    L = xs.load()
    assert 0 == L.libxsmm_b200_set_device(1)
    try:
        op = xs.Sp24(A8, fmt="e4m3")
    finally:
        L.libxsmm_b200_set_device(0)
    dB, dC = xs.DeviceBuffer.from_numpy(B8), xs.DeviceBuffer.from_numpy(C0)
    try:
        xs.clear_error()
        n0 = xs.launch_count()
        op.execute(dB, dC, N, b_fmt="e4m3")
        code, msg = xs.last_error()
        xs.clear_error()
        assert code == -97 and "created on device 1" in msg, msg
        assert xs.launch_count() == n0
    finally:
        dB.free(); dC.free()
        L.libxsmm_b200_set_device(1)
        op.destroy()
        L.libxsmm_b200_set_device(0)
