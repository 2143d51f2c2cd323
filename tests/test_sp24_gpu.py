"""GPU tests of the fixed 2:4-sparse bf16 operators (libxsmm_b200_sp24_*, csrc/sp24.cu): create compresses A once into the
structured-sparse tensor core's operand, execute multiplies with A and its metadata fetched by TMA.

Accuracy is the bf16 tensor-core contract of K4s and K4f: elementwise |C - want| <= 4e-6 (|A|.|B| + |beta| |C0|) against the
float64 product of the kept elements, on mixed-sign data.  Where K4s can run the same product (transb = 'N', K % 128 == 0,
aligned rows) the result is compared bit for bit: same instruction, same operands, same k order."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
KERNEL = "sp24_compute_kernel"
LEGAL = [m for m in range(16) if bin(m).count("1") <= 2]      # the eleven keep masks of a 2:4 group
NAN16, NZERO16 = 0x7FC1, 0x8000


def bits(x):
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) >> 16).astype(np.uint16)


def values(h):
    return (np.ascontiguousarray(h, np.uint16).astype(np.uint32) << 16).view(np.float32)


def kept(A16):
    """float64 image of the kept elements (ordered nonzeros; +-0 and NaN dropped)"""
    a = values(A16).astype(np.float64)
    return np.where(np.isnan(a), 0.0, a)


def make24(M, K, seed, masks=None):
    """random 2:4 bf16 A: every group takes one of the legal masks, mixed-sign values in [0.25, 2)"""
    rng = np.random.default_rng(seed)
    G = (K + 3) // 4
    m = rng.choice(LEGAL, (M, G)) if masks is None else masks
    keep = ((m[:, :, None] >> np.arange(4)) & 1).astype(bool).reshape(M, 4 * G)[:, :K]
    v = rng.uniform(0.25, 2.0, (M, K)) * rng.choice([-1.0, 1.0], (M, K))
    return bits(np.where(keep, v, 0.0))


def mixed(shape, rng):
    return rng.uniform(-1.0, 1.0, shape).astype(np.float32)


def run(xs, A16, B16, C0, N, transb="N", transc="N", beta=0.0, ldb=None, ldc=None, op=None):
    """one execute on fresh device buffers (an operator made from the host A unless one is given); returns C as stored"""
    own = op is None
    if own:
        op = xs.Sp24(A16)
    if ldb is None and B16.shape[1] % 8:        # B goes through TMA: rows padded to 16 bytes, NaN in the padding
        ldb = (B16.shape[1] + 7) // 8 * 8
        Bp = np.full((B16.shape[0], ldb), NAN16, np.uint16)
        Bp[:, :B16.shape[1]] = B16
        B16 = Bp
    dB, dC = xs.DeviceBuffer.from_numpy(B16), xs.DeviceBuffer.from_numpy(C0)
    try:
        n0 = xs.launch_count()
        op.execute(dB, dC, N, ldb=ldb, ldc=ldc, beta=beta, transb=transb, transc=transc)
        xs.synchronize()
        assert xs.launch_count() == n0 + (1 if N > 0 else 0)
        if N > 0:
            assert xs.last_compute_kernel() == KERNEL
        return dC.to_numpy(np.float32, C0.shape)
    finally:
        dB.free(); dC.free()
        if own:
            op.destroy()


def device_op(xs, A16):
    """an operator created from a DEVICE copy of A"""
    d = xs.DeviceBuffer.from_numpy(A16)
    try:
        M, K = A16.shape
        op = xs.Sp24.__new__(xs.Sp24)
        op.M, op.K, op.lda = M, K, K
        op.handle = xs.sp24_create_bfloat16(M, K, K, d.ptr)
        xs.check()
        assert op.handle
        return op
    finally:
        d.free()      # read only during create


def want_and_bound(A16, B16, C0, transb, transc, beta):
    a = kept(A16)
    b = values(B16).astype(np.float64)
    if transb == "T":
        b = b.T
    c0 = C0.astype(np.float64)
    if transc == "T":
        c0 = c0.T
    want = a @ b + (beta * c0 if beta != 0 else 0.0)
    bound = 4e-6 * (np.abs(a) @ np.abs(b) + (abs(beta) * np.abs(c0) if beta != 0 else 0.0))
    return (want.T, bound.T) if transc == "T" else (want, bound)


def check_f64(C, A16, B16, C0, transb="N", transc="N", beta=0.0):
    want, bound = want_and_bound(A16, B16, C0, transb, transc, beta)
    err = np.abs(C.astype(np.float64) - want)
    assert np.all(np.isfinite(C))
    assert np.all(err <= bound), float((err - bound).max())


def operands(M, N, K, transb, transc, seed):
    rng = np.random.default_rng(seed + 1)
    A16 = make24(M, K, seed)
    B = mixed((N, K) if transb == "T" else (K, N), rng)
    C0 = mixed((N, M) if transc == "T" else (M, N), rng)
    return A16, bits(B), C0


# ---- float64 parity ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [
    (4096, 4096, 4096),
    (300, 1, 72), (300, 3, 72), (300, 208, 72), (300, 257, 72),
    (300, 1, 200), (300, 3, 200), (300, 208, 200), (300, 257, 200),
    (33, 8, 128),                 # one partial tile
    (4096, 2048, 256),            # 128 tiles: more than the CTA pairs
    (2560, 2560, 384),            # 100 tiles: the left-over ones are split into half tiles
])
def test_float64_parity(gpu, M, N, K):
    A16, B16, C0 = operands(M, N, K, "N", "N", M + N + K)
    C = run(gpu, A16, B16, C0, N, beta=0.5)
    check_f64(C, A16, B16, C0, beta=0.5)
    gpu.check()


@pytest.mark.parametrize("transb", ["N", "T"])
@pytest.mark.parametrize("transc", ["N", "T"])
@pytest.mark.parametrize("beta", [0.0, 1.0, 0.5, -1.0])
def test_trans_and_beta(gpu, transb, transc, beta):
    M, N, K = 520, 392, 328
    A16, B16, C0 = operands(M, N, K, transb, transc, 7)
    C = run(gpu, A16, B16, C0, N, transb, transc, beta)
    check_f64(C, A16, B16, C0, transb, transc, beta)
    gpu.check()


def test_every_group_pattern(gpu):
    """the eleven legal masks at every group position of a 16-k span, rows of both halves of a 16-row metadata unit, plus groups
    whose only elements are -0 / NaN (dropped), or that hold them beside two kept elements"""
    M, N, K = 256, 256, 256
    G = K // 4
    masks = np.array([[LEGAL[(r * 7 + g * 5 + (r >> 4)) % 11] for g in range(G)] for r in range(M)])
    A16 = make24(M, K, 3, masks)
    rng = np.random.default_rng(3)
    for r in range(0, M, 3):
        g = (r * 13) % G
        A16[r, 4 * g:4 * g + 4] = [NZERO16, NAN16, NZERO16, NAN16 | 0x8000]
        g2 = (g + 7) % G
        A16[r, 4 * g2:4 * g2 + 4] = bits([rng.uniform(0.5, 1), 0.0, -rng.uniform(0.5, 1), 0.0])
        A16[r, 4 * g2 + 1], A16[r, 4 * g2 + 3] = NAN16, NZERO16
    B16, C0 = bits(mixed((K, N), rng)), mixed((M, N), rng)
    C = run(gpu, A16, B16, C0, N, beta=1.0)
    check_f64(C, A16, B16, C0, beta=1.0)
    C2 = k4s(gpu, A16, B16, C0, 1)
    np.testing.assert_array_equal(C.view(np.uint32), C2.view(np.uint32))


# ---- same bits as K4s ------------------------------------------------------------------------------------------------------
def k4s(xs, A16, B16, C0, beta):
    """C of the spmdm route with K4s forced"""
    import os
    saved = {k: os.environ.get(k) for k in ("LIBXSMM_B200_SPMDM_TC", "LIBXSMM_B200_TC16_SPARSE")}
    os.environ["LIBXSMM_B200_SPMDM_TC"] = "1"
    os.environ["LIBXSMM_B200_TC16_SPARSE"] = "1"
    M, K = A16.shape
    N = B16.shape[1]
    p = xs.Spmdm(M, N, K, 1)
    try:
        dA, dB, dC = (xs.DeviceBuffer.from_numpy(x) for x in (A16, B16, C0))
        p.create_slices(dA, "N", True)
        p.compute(dB, dC, "N", "N", beta, True)      # bf16 beta: the raw integer (reference quirk), 1 means beta = 1
        xs.synchronize()
        assert xs.last_compute_kernel() == "spmdm_compute_tc16s_kernel"
        C = dC.to_numpy(np.float32, C0.shape)
        for d in (dA, dB, dC):
            d.free()
        return C
    finally:
        p.destroy()
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("M,N,K", [(512, 512, 512), (300, 208, 256), (4096, 4096, 4096), (2048, 264, 384)])
@pytest.mark.parametrize("beta", [0, 1])
def test_same_bits_as_k4s(gpu, M, N, K, beta):
    A16, B16, C0 = operands(M, N, K, "N", "N", 11 + M)
    C = run(gpu, A16, B16, C0, N, beta=float(beta))
    C2 = k4s(gpu, A16, B16, C0, beta)
    np.testing.assert_array_equal(C.view(np.uint32), C2.view(np.uint32))


@pytest.mark.parametrize("M,N,K", [(512, 392, 512), (300, 257, 200), (4096, 1024, 4096)])
def test_transposed_forms_same_bits(gpu, M, N, K):
    A16, B16, C0 = operands(M, N, K, "N", "N", 5)
    op = gpu.Sp24(A16)
    try:
        C = run(gpu, A16, B16, C0, N, "N", "N", 0.0, op=op)
        Ct = run(gpu, A16, np.ascontiguousarray(B16.T), C0, N, "T", "N", 0.0, op=op)
        np.testing.assert_array_equal(C.view(np.uint32), Ct.view(np.uint32))
        C0t = np.ascontiguousarray(C0.T)
        for tb, B in (("N", B16), ("T", np.ascontiguousarray(B16.T))):
            Cc = run(gpu, A16, B, C0t, N, tb, "T", 0.0, op=op)
            np.testing.assert_array_equal(Cc.view(np.uint32), np.ascontiguousarray(C.T).view(np.uint32))
    finally:
        op.destroy()


# ---- create ------------------------------------------------------------------------------------------------------------
def test_host_and_device_a_give_identical_c(gpu):
    M, N, K = 300, 264, 200
    lda = 208
    A16, B16, C0 = operands(M, N, K, "N", "N", 21)
    Apad = np.full((M, lda), NAN16, np.uint16)            # NaN in A's pitch padding is never read
    Apad[:, :K] = A16
    op_h = gpu.Sp24(Apad[:, :K])
    assert op_h.lda == lda
    op_d = device_op(gpu, A16)
    try:
        Ch = run(gpu, A16, B16, C0, N, beta=1.0, op=op_h)
        Cd = run(gpu, A16, B16, C0, N, beta=1.0, op=op_d)
        np.testing.assert_array_equal(Ch.view(np.uint32), Cd.view(np.uint32))
        check_f64(Ch, A16, B16, C0, beta=1.0)
    finally:
        op_h.destroy(); op_d.destroy()


def test_torch_tensors(gpu):
    import torch
    M, N, K = 256, 128, 256
    A16, B16, C0 = operands(M, N, K, "N", "N", 4)
    a = torch.from_numpy(A16.view(np.int16)).view(torch.bfloat16).cuda()
    b = torch.from_numpy(B16.view(np.int16)).view(torch.bfloat16).cuda()
    c = torch.empty((M, N), dtype=torch.float32, device="cuda")
    op = gpu.Sp24(a)
    try:
        op.execute(b, c, N, stream=torch.cuda.current_stream())
        torch.cuda.synchronize()
        check_f64(c.cpu().numpy(), A16, B16, C0)
    finally:
        op.destroy()


@pytest.mark.parametrize("M,K,row,group", [(256, 256, 0, 0), (300, 200, 299, 49), (300, 203, 137, 50)])
def test_create_rejects_a_that_is_not_2_4(gpu, M, K, row, group):
    """one group keeping three elements -- the first, the last, or the partial tail group of a row (K % 4 = 3) -- gives NULL
    with -96 naming it; the failed create gives its device memory back"""
    import torch
    A16 = make24(M, K, 9)
    A16[row, 4 * group:4 * group + 3] = bits([1.0, -2.0, 3.0])
    for attempt in range(2):           # the first attempt may grow the runtime's pools; the second must leave memory as it was
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        gpu.clear_error()
        h = gpu.sp24_create_bfloat16(M, K, K, A16)
        code, msg = gpu.last_error()
        gpu.clear_error()
        assert not h
        assert code == -96, msg
        assert "row %d, group %d" % (row, group) in msg, msg
        free1 = torch.cuda.mem_get_info()[0]
    assert free1 == free0


# ---- guard bands and special values ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [3, 8, 130, 257])
@pytest.mark.parametrize("transc", ["N", "T"])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_guard_bands(gpu, N, transc, beta):
    """NaN sentinels in C's pitch padding and past M stay, NaN in B's padding columns does not leak, NaN in C0 disappears with
    beta = 0.  transc = 'N', beta = 0 with N % 4 = 0 takes the TMA-box epilogue."""
    M, K = 300, 256
    rng = np.random.default_rng(N)
    A16 = make24(M, K, N)
    ldb = ((N + 8) + 7) // 8 * 8
    B16 = np.full((K, ldb), NAN16, np.uint16)
    B16[:, :N] = bits(mixed((K, N), rng))
    rows, ldc = (M + 5, (N + 7) // 4 * 4) if transc == "N" else (N + 5, M + 4)    # 16-byte rows: N % 4 decides the epilogue
    Cs = np.full((rows, ldc), np.nan, np.float32)
    C0 = mixed((M, N) if transc == "N" else (N, M), rng)
    if beta == 0.0:
        C0[::7, ::5] = np.nan
    Cs[:C0.shape[0], :C0.shape[1]] = C0
    C = run(gpu, A16, B16, Cs, N, "N", transc, beta, ldb=ldb, ldc=ldc)
    inner = C[:C0.shape[0], :C0.shape[1]]
    check_f64(np.ascontiguousarray(inner), A16, np.ascontiguousarray(B16[:, :N]), C0, "N", transc, beta)
    pad = np.ones_like(C, bool)
    pad[:C0.shape[0], :C0.shape[1]] = False
    np.testing.assert_array_equal(C[pad].view(np.uint32), Cs[pad].view(np.uint32))


def test_non_finite_b_taints_no_more_than_the_dense_product(gpu):
    M, N, K = 256, 264, 256
    A16, B16, C0 = operands(M, N, K, "N", "N", 8)
    B16[17, 40] = 0x7F80           # +Inf
    B16[200, 100] = 0xFF80         # -Inf
    B16[90, 263] = NAN16
    C = run(gpu, A16, B16, C0, N)
    b = values(B16)
    tainted = np.broadcast_to(~np.all(np.isfinite(b), axis=0), C.shape)   # the dense product multiplies every A[m, k], zeros included
    assert not np.any(~np.isfinite(C) & ~tainted)
    clean = ~tainted[0]
    want, bound = want_and_bound(A16, np.where(np.isfinite(b), B16, 0).astype(np.uint16), C0, "N", "N", 0.0)
    assert np.all(np.abs(C[:, clean] - want[:, clean]) <= bound[:, clean])


# ---- launch behaviour ------------------------------------------------------------------------------------------------------
def test_two_handles_on_two_streams(gpu):
    xs = gpu
    shapes = [(512, 384, 256), (300, 520, 384)]
    ops, bufs, serial = [], [], []
    for i, (M, N, K) in enumerate(shapes):
        A16, B16, C0 = operands(M, N, K, "N", "N", 40 + i)
        ops.append(xs.Sp24(A16))
        serial.append(run(xs, A16, B16, C0, N, op=ops[-1]))
        bufs.append((xs.DeviceBuffer.from_numpy(B16), xs.DeviceBuffer.from_numpy(C0), N, C0.shape))
    streams = [xs.Stream(), xs.Stream()]
    try:
        for rep in range(3):
            for op, (dB, dC, N, shp), st in zip(ops, bufs, streams):
                op.execute(dB, dC, N, beta=0.0, stream=st)
            for st in streams:
                st.synchronize()
            for (dB, dC, N, shp), C in zip(bufs, serial):
                np.testing.assert_array_equal(dC.to_numpy(np.float32, shp).view(np.uint32), C.view(np.uint32))
        xs.check()
    finally:
        for op in ops:
            op.destroy()
        for dB, dC, _, _ in bufs:
            dB.free(); dC.free()
        for st in streams:
            st.destroy()


def test_graph_replay_with_new_b(gpu):
    xs, L = gpu, gpu.load()
    M, N, K = 512, 392, 384
    A16, _, C0 = operands(M, N, K, "N", "N", 50)
    rng = np.random.default_rng(50)
    Bs = [bits(mixed((K, N), rng)) for _ in range(2)]
    op = xs.Sp24(A16)
    dB, dC = xs.DeviceBuffer.from_numpy(Bs[0]), xs.DeviceBuffer.from_numpy(C0)
    st = xs.Stream()
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    op.execute(dB, dC, N, beta=0.0, stream=st)
    graph = L.libxsmm_b200_graph_end(st.ptr)
    xs.check()
    assert graph
    try:
        for B16 in Bs + Bs[:1]:
            want = run(xs, A16, B16, C0, N, op=op)
            dB.upload(B16)
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
    A16, B16, C0 = operands(M, N, K, "N", "N", 60)
    op = xs.Sp24(A16)
    dB, dC = xs.DeviceBuffer(2 * K * max(N, K) + 64), xs.DeviceBuffer(4 * M * max(N, M) + 64)
    h = op.handle
    cases = [
        (("X", "N", N, dB.ptr, N, dC.ptr, N), "transb='X'"),
        (("N", "q", N, dB.ptr, N, dC.ptr, N), "transc='q'"),
        (("N", "N", -1, dB.ptr, N, dC.ptr, N), "N=-1"),
        (("N", "N", N, dB.ptr, N - 8, dC.ptr, N), "ldb=56"),
        (("T", "N", N, dB.ptr, K - 8, dC.ptr, N), "ldb=184"),
        (("N", "N", N, dB.ptr, N, dC.ptr, N - 1), "ldc=63"),
        (("N", "T", N, dB.ptr, N, dC.ptr, M - 1), "ldc=255"),
        (("N", "N", N, None, N, dC.ptr, N), "NULL d_b"),
        (("N", "N", N, dB.ptr, N, None, N), "NULL d_b or d_c"),
        (("N", "N", N, dB.ptr + 2, N, dC.ptr, N), "16-byte aligned"),
        (("N", "N", N, dB.ptr, N + 4, dC.ptr, N), "ldb=68"),
    ]
    try:
        for (tb, tc, n, b, ldb, c, ldc), frag in cases:
            xs.clear_error()
            n0 = xs.launch_count()
            xs.sp24_execute(h, tb, tc, n, b, ldb, 0.0, c, ldc)
            code, msg = xs.last_error()
            assert xs.launch_count() == n0, frag
            assert code == -97 and frag in msg, (frag, code, msg)
        xs.clear_error()
        n0 = xs.launch_count()
        xs.sp24_execute(h, "N", "N", 0, None, 0, 0.0, None, 0)       # N = 0 does nothing
        assert xs.launch_count() == n0 and xs.last_error()[0] == 0
    finally:
        xs.clear_error()
        op.destroy(); dB.free(); dC.free()


def test_other_device_is_rejected(gpu):
    xs = gpu
    if xs.device_count() < 2:
        pytest.skip("one device")
    M, N, K = 128, 64, 128
    A16, B16, C0 = operands(M, N, K, "N", "N", 70)
    L = xs.load()
    assert 0 == L.libxsmm_b200_set_device(1)
    try:
        op = xs.Sp24(A16)
    finally:
        L.libxsmm_b200_set_device(0)
    dB, dC = xs.DeviceBuffer.from_numpy(B16), xs.DeviceBuffer.from_numpy(C0)
    try:
        xs.clear_error()
        n0 = xs.launch_count()
        op.execute(dB, dC, N)
        code, msg = xs.last_error()
        xs.clear_error()
        assert code == -97 and "created on device 1" in msg, msg
        assert xs.launch_count() == n0
    finally:
        dB.free(); dC.free()
        L.libxsmm_b200_set_device(1)
        op.destroy()
        L.libxsmm_b200_set_device(0)
