"""GPU parity of K4f, the tensor-core kernel for dense fp32 fixed operators (fsspmdm_tc_kernel, csrc/fsspmdm_tc.cu), and of
the routes around it: the unaligned-C epilogue, the generic-kernel fallback for an unaligned B, the host-pointer staging and
the dense-SMM dispatch entry.

K4f is persistent (grid = min(tiles, SMs), CTA b runs tiles b, b + grid, ...), and most of its state only turns over once a
CTA reaches its second tile: two raw B stages sharing one b_lo buffer, the double-buffered accumulator in tensor memory, the
two C staging boxes of the TMA-store epilogue, the L2 prefetch two tiles ahead.  The problems here give every CTA six or seven
tiles, so every barrier parity wraps several times.

Reference: the float64 product of the fp32 inputs.  Bound, element by element: |C - want| <= 4e-6 * (|a| @ |B| + beta |C0|)
(3xTF32: at most 24 fp32 accumulations of 8 k-steps x 3 MMAs for K <= 64, plus the dropped lo x lo term), beside the normwise
1e-5 contract.  Inputs are mixed-sign so that a wrong row or column cannot hide under max |C|.
LIBXSMM_B200_FSSPMDM_TC=1 forces the kernel wherever a test is not about the automatic choice."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K4F = "fs_tc_kernel"
GENERIC = "fs_generic_kernel"
BAKED = "fs_baked"
BN = 128                          # panel columns per tile
ELEM_BOUND = 4e-6
RTOL = 1e-5


def sm_count():
    """multiprocessors of device 0 (the grid of the persistent kernel), from the driver"""
    cu = ctypes.CDLL("libcuda.so.1")
    dev, v = ctypes.c_int(0), ctypes.c_int(0)
    assert 0 == cu.cuInit(0) and 0 == cu.cuDeviceGet(ctypes.byref(dev), 0)
    assert 0 == cu.cuDeviceGetAttribute(ctypes.byref(v), 16, dev)        # CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT
    return v.value


def persistent_n(sms):
    """N with 6 * SMs + SMs / 2 + 1 tiles, the last one ragged (48 columns): every CTA runs six or seven tiles"""
    ntiles = 6 * sms + sms // 2 + 1
    return (ntiles - 1) * BN + 48, ntiles


def inputs(M, K, ld, seed, ldc=None):
    rng = np.random.default_rng(seed)
    a = rng.uniform(-1, 1, (M, K)).astype(np.float32)
    B = rng.uniform(-1, 1, (K, ld)).astype(np.float32)
    C0 = rng.uniform(-1, 1, (M, ld if ldc is None else ldc)).astype(np.float32)
    return a, B, C0


def reference(a, B, C0, beta, N):
    """(want, mag) in float64 over the first N columns.  Products that involve a non-finite input are summed elementwise
    (IEEE: 0 * Inf = NaN), the rest goes through BLAS on the finite values."""
    with np.errstate(invalid="ignore"):
        return _reference(a, B, C0, beta, N)


def _reference(a, B, C0, beta, N):
    a64, B64 = a.astype(np.float64), B[:, :N].astype(np.float64)
    fa, fb = np.where(np.isfinite(a64), a64, 0.0), np.where(np.isfinite(B64), B64, 0.0)
    want, mag = fa @ fb, np.abs(fa) @ np.abs(fb)
    cols = np.nonzero(~np.isfinite(B64).all(axis=0))[0]
    if len(cols):
        want[:, cols] = (a64[:, :, None] * B64[None, :, cols]).sum(axis=1)
    for r in np.nonzero(~np.isfinite(a64).all(axis=1))[0]:
        want[r] = (a64[r][:, None] * B64).sum(axis=0)
    if beta:
        c = C0[:, :N].astype(np.float64)
        want += c
        mag += np.where(np.isfinite(c), np.abs(c), 0.0)
    return want, mag


def worst_ratio(C, want, mag):
    """largest |C - want| / mag over the finite reference elements; asserts the elementwise bound and the normwise contract"""
    C64 = C.astype(np.float64)
    fin = np.isfinite(want)
    err = np.where(fin, np.abs(C64 - np.where(fin, want, 0.0)), 0.0)
    assert np.isfinite(C64[fin]).all(), "non-finite output where the reference is finite"
    bad = err > ELEM_BOUND * mag
    if bad.any():
        m, n = np.argwhere(bad)[0]
        raise AssertionError("%d elements beyond the bound, first (%d, %d): got %r want %r mag %r"
                             % (bad.sum(), m, n, C64[m, n], want[m, n], mag[m, n]))
    assert err.max() <= RTOL * max(float(np.abs(want[fin]).max()), 1e-30)
    return float(np.max(np.where(mag > 0, err / np.where(mag > 0, mag, 1.0), 0.0)))


def same_bits(x, y):
    np.testing.assert_array_equal(np.ascontiguousarray(x).view(np.uint32), np.ascontiguousarray(y).view(np.uint32))


def run(xs, a, B, C0, beta, N, ldb, ldc, b_shift=0, c_shift=0):
    """one execute_stream on device copies of B (K x ldb) and C0 (M x ldc), each optionally `shift` bytes past an aligned
    base (the bytes in front of a shifted C must stay untouched); returns (C, kernel that ran)"""
    op = xs.Fsspmdm(a, N, ldb=ldb, ldc=ldc, beta=beta)
    dB, dC = xs.DeviceBuffer(B.nbytes + 16), xs.DeviceBuffer(C0.nbytes + 16)
    try:
        assert op.is_tensor_core
        lead = np.full(4, 0x7F7FFFFF, np.uint32)                            # pattern in front of a shifted C
        dB.upload(B, b_shift)
        dC.upload(lead)
        dC.upload(C0, c_shift)
        op.execute_stream(dB.ptr + b_shift, dC.ptr + c_shift)
        xs.synchronize()
        kernel = xs.last_compute_kernel()
        C = dC.to_numpy(np.float32, C0.shape, c_shift)
        if c_shift:
            assert np.array_equal(dC.to_numpy(np.uint32, (c_shift // 4,)), lead[:c_shift // 4]), "written in front of C"
        return C, kernel
    finally:
        dB.free(); dC.free(); op.destroy()
        xs.check()


@pytest.fixture
def k4f(monkeypatch):
    monkeypatch.setenv("LIBXSMM_B200_FSSPMDM_TC", "1")
    monkeypatch.delenv("LIBXSMM_B200_K4F_EPI", raising=False)
    return monkeypatch


@pytest.fixture(scope="module")
def big():
    """the persistent-loop problem: 150 x 64 operator, ldb = ldc = N + 64, references for beta 0 and 1"""
    sms = sm_count()
    N, ntiles = persistent_n(sms)
    a, B, C0 = inputs(150, 64, N + 64, seed=41)
    return dict(sms=sms, N=N, ntiles=ntiles, ld=N + 64, a=a, B=B, C0=C0, ref={b: reference(a, B, C0, b, N) for b in (0, 1)})


# ---- 1. persistent loop --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [0, 1])
def test_persistent_loop_every_element(gpu, k4f, big, beta):
    """six or seven tiles per CTA: every element within the bound, columns past N untouched, two launches the same bits"""
    xs, N, ld = gpu, big["N"], big["ld"]
    assert big["ntiles"] > 6 * big["sms"] and N % BN == 48
    outs = []
    for rep in range(2):
        C, kernel = run(xs, big["a"], big["B"], big["C0"], beta, N, ld, ld)
        assert kernel == K4F
        outs.append(C)
    worst_ratio(outs[0][:, :N], *big["ref"][beta])
    same_bits(outs[0][:, N:], big["C0"][:, N:])
    same_bits(outs[0], outs[1])


@pytest.mark.parametrize("beta", [0, 1])
def test_persistent_tiles_match_one_tile_launches(gpu, k4f, big, beta):
    """a tile's arithmetic does not depend on the CTA that ran it or on what that CTA did before: first-round tiles, tiles of
    rounds 2 to 7 and the ragged last tile are bit-identical to a launch of that tile alone (stale b_lo, accumulator or
    staging-box content would change bits)"""
    xs, sms, N, ld, ntiles = gpu, big["sms"], big["N"], big["ld"], big["ntiles"]
    a, B, C0 = big["a"], big["B"], big["C0"]
    C, kernel = run(xs, a, B, C0, beta, N, ld, ld)
    assert kernel == K4F
    tiles = sorted({r * sms + c for r in range(7) for c in (0, 37 % sms, sms // 2, sms - 1)} | {ntiles - 1})
    tiles = [t for t in tiles if t < ntiles]
    assert len(tiles) >= 24 and tiles[-1] == ntiles - 1
    dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
    try:
        for t in tiles:
            w = min(BN, N - t * BN)
            op = xs.Fsspmdm(a, w, ldb=ld, ldc=ld, beta=beta)
            op.execute_stream(dB.ptr + 4 * BN * t, dC.ptr + 4 * BN * t)
            xs.synchronize()
            assert xs.last_compute_kernel() == K4F
            op.destroy()
        one = dC.to_numpy(np.float32, C0.shape)
    finally:
        dB.free(); dC.free()
    hit = np.zeros(ld, bool)
    for t in tiles:
        hit[t * BN:min((t + 1) * BN, N)] = True
        same_bits(one[:, t * BN:(t + 1) * BN], C[:, t * BN:(t + 1) * BN])
    same_bits(one[:, ~hit], C0[:, ~hit])           # each one-tile launch wrote its own columns only
    xs.check()


@pytest.mark.parametrize("beta", [0, 1])
def test_epilogue_forms_give_identical_bits(gpu, k4f, big, beta):
    """the TMA-store epilogue (EPI = 2, default; beta = 1: TMA reduce-add), per-thread stores in 8-row chunks (EPI = 1, also
    what an unaligned C gets) and the 32-row loop (EPI = 0) store the same accumulator: identical bits"""
    xs, N, ld = gpu, big["N"], big["ld"]
    outs = {}
    for epi in ("2", "1", "0"):
        k4f.setenv("LIBXSMM_B200_K4F_EPI", epi)                      # read at create
        C, kernel = run(xs, big["a"], big["B"], big["C0"], beta, N, ld, ld)
        assert kernel == K4F
        outs[epi] = C
    worst_ratio(outs["1"][:, :N], *big["ref"][beta])
    same_bits(outs["1"], outs["2"])
    same_bits(outs["0"], outs["2"])


# ---- 2. operator geometry ------------------------------------------------------------------------------------------------
# staging boxes of 32 rows: 1 .. 6; M % 8 != 0 and M_pad (next multiple of 16) != M; K below, on and across the 8-k step
# and the 32-k chunk of the operator's layout
GEOMETRY = [(1, 1), (8, 7), (17, 9), (31, 8), (32, 33), (33, 32), (64, 31), (72, 17), (100, 63), (150, 64), (161, 64),
            (176, 40), (192, 64)]


@pytest.mark.parametrize("M,K", GEOMETRY)
@pytest.mark.parametrize("beta", [0, 1])
def test_operator_geometry(gpu, k4f, M, K, beta):
    xs = gpu
    sms = sm_count()
    N = (2 * sms + 3) * BN - 80                      # two and a bit tiles per CTA, ragged last tile
    ld = N + 32
    a, B, C0 = inputs(M, K, ld, seed=M * 100 + K)
    zero_row = M // 2 if M > 1 else None
    if zero_row is not None:
        a[zero_row] = 0                              # written as 0 (beta = 0) or as C0 (beta = 1)
    C, kernel = run(xs, a, B, C0, beta, N, ld, ld)
    assert kernel == K4F
    worst_ratio(C[:, :N], *reference(a, B, C0, beta, N))
    same_bits(C[:, N:], C0[:, N:])
    if zero_row is not None:
        if beta:
            same_bits(C[zero_row], C0[zero_row])
        else:
            assert not C[zero_row, :N].any()


# ---- 3. routes around the kernel -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("how", ["pointer", "ldc"])
@pytest.mark.parametrize("beta", [0, 1])
def test_unaligned_c_stays_on_tensor_cores(gpu, k4f, how, beta):
    """C that the store engine cannot address (base not 16-byte aligned, or a pitch of N + 1 floats): K4f with per-thread
    stores; columns outside [0, N) and the bytes in front of C untouched"""
    xs = gpu
    N = (2 * sm_count() + 1) * BN + 48
    ldb = N + 64
    ldc = N + 64 if how == "pointer" else N + 1
    a, B, C0 = inputs(150, 64, ldb, seed=51, ldc=ldc)
    C, kernel = run(xs, a, B, C0, beta, N, ldb, ldc, c_shift=4 if how == "pointer" else 0)
    assert kernel == K4F
    worst_ratio(C[:, :N], *reference(a, B, C0, beta, N))
    same_bits(C[:, N:], C0[:, N:])


@pytest.mark.parametrize("how", ["pointer", "ldb"])
@pytest.mark.parametrize("beta", [0, 1])
def test_unaligned_b_falls_back_to_generic_kernel(gpu, oracle, k4f, how, beta):
    """B the tensor map cannot describe: the operator has no baked kernel (the tensor-core one took it), so the generic
    kernel runs -- the reference's in-order fma chain, bit-exact against the oracle on the same panel"""
    xs = gpu
    N = 8192 + 48
    ldc = N + 64
    ldb = N + 64 if how == "pointer" else N + 1
    a, B, C0 = inputs(150, 64, ldb, seed=52, ldc=ldc)
    a[3] = 0
    C, kernel = run(xs, a, B, C0, beta, N, ldb, ldc, b_shift=4 if how == "pointer" else 0)
    assert kernel == GENERIC
    want = C0.copy()
    oracle.sfsspmdm_execute(a, B, want, float(beta), N=N, ldb=ldb, ldc=ldc)
    same_bits(C, want)


@pytest.mark.parametrize("beta", [0, 1])
def test_host_pointers_through_staging_chunks(gpu, k4f, beta):
    """host panels go through device staging in 65536-column chunks (here three, the last one ragged) with the chunk width
    as pitch; columns past N untouched"""
    xs = gpu
    N = 2 * 65536 + 4096 + 48
    ld = N + 64
    a, B, C0 = inputs(150, 64, ld, seed=53)
    op = xs.Fsspmdm(a, N, ldb=ld, ldc=ld, beta=beta)
    try:
        assert op.is_tensor_core
        C = C0.copy()
        op.execute(B, C)
        xs.check()
        assert xs.last_compute_kernel() == K4F
    finally:
        op.destroy()
    worst_ratio(C[:, :N], *reference(a, B, C0, beta, N))
    same_bits(C[:, N:], C0[:, N:])


def _mm_layout(m_total, layout):
    lda = ldc = max(16, (m_total + 3) // 4 * 4) + 4            # the descriptor's m (16 columns per call) <= lda, ldc
    if layout == "lda":
        lda += 1
    elif layout == "ldc":
        ldc += 1
    return lda, ldc


@pytest.mark.parametrize("m_total", [1, 5, 127, 129, "3 waves + 77"])
@pytest.mark.parametrize("layout", ["aligned", "lda", "ldc"])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_mm_dispatch_routes(gpu, oracle, monkeypatch, m_total, layout, beta):
    """libxsmm_b200_smmdispatch + execute (automatic kernel choice): a dense operator from a host pointer, then another dense
    one from a device pointer (the handle re-creates its operator), then a 20 %-dense one (baked kernel, bit-exact).  An
    unaligned panel pitch (lda) sends the dense operator to the generic kernel (bit-exact), an unaligned ldc keeps K4f.
    Any column count: columns from m_total to ldc are neither written nor read-modify-written (the store engine's boxes
    end on 16-byte boundaries, so a ragged m_total must not go through it)."""
    monkeypatch.delenv("LIBXSMM_B200_FSSPMDM_TC", raising=False)
    monkeypatch.delenv("LIBXSMM_B200_K4F_EPI", raising=False)
    xs = gpu
    if not isinstance(m_total, int):
        m_total = 3 * sm_count() * BN + 77
    M, K = 150, 64
    lda, ldc = _mm_layout(m_total, layout)
    rng = np.random.default_rng(m_total + 7 * len(layout))
    B = rng.uniform(-1, 1, (K, lda)).astype(np.float32)
    C0 = rng.uniform(-1, 1, (M, ldc)).astype(np.float32)
    C0[:, m_total:] = np.uint32(0x7FC0BEEF).view(np.float32)    # a NaN payload that any read-modify-write would lose
    sparse = rng.uniform(-1, 1, (M, K)).astype(np.float32)
    sparse[rng.random((M, K)) >= 0.2] = 0
    ops = [(rng.uniform(-1, 1, (M, K)).astype(np.float32), "host", K4F),
           (rng.uniform(-1, 1, (M, K)).astype(np.float32), "device", K4F),
           (sparse, "device", BAKED)]
    h = xs.MmDispatch(16, M, K, lda=lda, ldb=K, ldc=ldc, beta=beta, dtype=np.float32)
    dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
    try:
        for a, where, form in ops:
            dC.upload(C0)
            dA = xs.DeviceBuffer.from_numpy(a) if where == "device" else None
            h.execute(dB, dA if dA is not None else a, dC, m_total)
            xs.synchronize()
            if dA is not None:
                dA.free()
            C = dC.to_numpy(np.float32, C0.shape)
            assert h.kernel == form
            if form == K4F:
                route = GENERIC if layout == "lda" else K4F
            else:       # the baked kernel's two-column form (even pitches) takes even column counts only
                route = GENERIC if (layout == "aligned" and m_total % 2) else BAKED
            assert xs.last_compute_kernel() == route, (xs.last_compute_kernel(), route)
            if route == K4F:
                worst_ratio(C[:, :m_total], *reference(a, B, C0, beta, m_total))
            else:
                want = C0.copy()
                oracle.sfsspmdm_execute(a, B, want, beta, N=m_total, ldb=lda, ldc=ldc)
                same_bits(C, want)
            same_bits(C[:, m_total:], C0[:, m_total:])
    finally:
        dB.free(); dC.free(); h.release()
    xs.check()


# ---- 4. non-finite inputs as tracers -------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [0, 1])
def test_non_finite_inputs_stay_in_their_rows_and_columns(gpu, k4f, big, beta):
    """NaN in B in tiles of different rounds, +-Inf in other B columns and in one operator value, NaN in C0 (beta = 1): the
    set of non-finite outputs is exactly the reference's, nothing leaks into another column or into the next tile of the
    same CTA, and every other element keeps the bound.  3xTF32 cannot give Inf (Inf - trunc(Inf) is NaN, and Inf times an
    operator value that is exact in TF32 has a NaN low part), so NaN stands where the reference has +-Inf."""
    xs, sms, N, ld, ntiles = gpu, big["sms"], big["N"], big["ld"], big["ntiles"]
    a, B, C0 = big["a"].copy(), big["B"].copy(), big["C0"].copy()
    col = lambda t, c: t * BN + c                                       # noqa: E731
    for k, n in ((0, col(0, 0)), (63, col(sms + 5, 17)), (31, col(3 * sms + 7, 127)), (8, N - 1), (40, col(sms - 1, 64))):
        B[k, n] = np.nan
    B[5, col(1, 3)] = np.inf
    B[40, col(2 * sms + 1, 100)] = -np.inf
    B[17, col(5 * sms + 2, 31)] = np.inf
    a[77, 13] = -np.inf
    if beta:
        for m, n in ((0, col(4 * sms, 5)), (149, col(6 * sms + 3, 0)), (60, col(sms + 5, 18))):
            C0[m, n] = np.nan
    want, mag = reference(a, B, C0, beta, N)
    C, kernel = run(xs, a, B, C0, beta, N, ld, ld)
    assert kernel == K4F
    C = C[:, :N]
    np.testing.assert_array_equal(~np.isfinite(C), ~np.isfinite(want))
    assert np.isnan(C[np.isnan(want)]).all()
    inf = np.isinf(want)
    assert (np.isnan(C[inf]) | (C[inf] == want[inf])).all()
    assert (~np.isfinite(want)).sum() < 12 * 150 + N                     # the tracers stayed tracers
    worst_ratio(C, want, mag)


# ---- 5. subnormals -------------------------------------------------------------------------------------------------------
def tf32(x):
    """x with the 13 low mantissa bits cleared: what the tensor core reads of an fp32 operand"""
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def test_subnormal_b_columns(gpu, k4f):
    """B columns made entirely of subnormals under an O(1) operator.  Subnormal TF32 operands are not flushed: columns whose
    subnormals are exact in TF32 keep the bound.  Of any other subnormal b the low part b - trunc(b) lies below the smallest
    TF32 subnormal (2^-136), so the kernel multiplies trunc(b): those columns keep the bound against a reference built from
    trunc(b), and miss the exact one by about 1e-3 of their scale (DESIGN.md section 2)."""
    xs = gpu
    N = 4096 + 48
    a, B, C0 = inputs(150, 64, N, seed=61)
    rng = np.random.default_rng(62)
    exact, rest = [2049, N - 1], [5, 700]
    for c in exact + rest:
        B[:, c] = (rng.uniform(-1, 1, 64) * 2.0 ** -127).astype(np.float32)
    B[:, exact] = tf32(B[:, exact])
    assert (np.abs(B[:, exact + rest]) < np.finfo(np.float32).tiny).all() and (B[:, rest] != tf32(B[:, rest])).any()
    C, kernel = run(xs, a, B, C0, 0, N, N, N)
    assert kernel == K4F
    keep = np.setdiff1d(np.arange(N), rest)
    worst_ratio(C[:, keep], *(x[:, keep] for x in reference(a, B, C0, 0, N)))
    Bt = B.copy()
    Bt[:, rest] = tf32(B[:, rest])
    worst_ratio(C[:, rest], *(x[:, rest] for x in reference(a, Bt, C0, 0, N)))


@pytest.mark.parametrize("epi", ["2", "1", "0"])
def test_subnormal_c0_with_zero_b_column(gpu, k4f, epi):
    """beta = 1, B column zero, C0 subnormal in that column: the reference gives C0 exactly, and so does every epilogue form
    (the TMA reduce-add of the default one does not flush subnormals)"""
    xs = gpu
    k4f.setenv("LIBXSMM_B200_K4F_EPI", epi)
    N = 4096 + 48
    a, B, C0 = inputs(150, 64, N, seed=63)
    rng = np.random.default_rng(64)
    cols = [9, 1500, N - 2]
    for c in cols:
        B[:, c] = 0
        C0[:, c] = (rng.uniform(-1, 1, 150) * 2.0 ** -127).astype(np.float32)
    C, kernel = run(xs, a, B, C0, 1, N, N, N)
    assert kernel == K4F
    same_bits(C[:, cols], C0[:, cols])
    worst_ratio(C, *reference(a, B, C0, 1, N))
