"""Dense x SoA kernels (libxsmm_b200_[sd]rm_{ac,bc}_soa_*; the batched GPU counterparts of libxsmm_create_rm_ac_soa /
libxsmm_create_rm_bc_soa).  CPU: the oracle's restatement against a float64 product and on exact small-integer inputs, and the
argument checks of create / execute, which make no CUDA call.  GPU: the batched entry against the oracle, bit for bit (NaN
positions compared as a set: a NaN's payload is not part of the contract, the GPU and the host's fma propagate different ones).
The restatement is tests/rm_soa_oracle.c, compiled by the rm_oracle fixture."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

SENT = -7.25          # sentinel in pitch padding and element gaps of C: must survive every call


def bits(x):
    return x.view(np.uint64 if x.dtype == np.float64 else np.uint32)


def same(got, want):
    ng, nw = np.isnan(got), np.isnan(want)
    return np.array_equal(ng, nw) and np.array_equal(bits(got)[~ng], bits(want)[~nw])


def extents(form, M, N, K, lda, ldb, ldc, soa):
    """scalars of one element's first operand, second operand and C as they lie in memory"""
    ea = ((M - 1) * lda + K) * (soa if form == "ac" else 1)
    eb = ((K - 1) * ldb + N) * (soa if form == "bc" else 1)
    return ea, eb, ((M - 1) * ldc + N) * soa


def flat_case(rng, form, M, N, K, soa, dt, lda, ldb, ldc, E, sa, sb, sc, ints=False):
    """flat operand arrays for E elements at strides sa / sb / sc (0: shared); C gaps and padding hold SENT"""
    ea, eb, ec = extents(form, M, N, K, lda, ldb, ldc, soa)
    draw = (lambda n: rng.integers(-4, 5, n).astype(dt)) if ints else (lambda n: rng.uniform(-1, 1, n).astype(dt))
    a = draw(max(E - 1, 0) * sa + ea)
    b = draw(max(E - 1, 0) * sb + eb)
    c = np.full(max(E - 1, 0) * sc + ec, SENT, dt)
    for e in range(E):
        for m in range(M):
            o = e * sc + m * ldc * soa
            c[o:o + N * soa] = draw(N * soa)
    return a, b, c


def dense_views(form, M, N, K, lda, ldb, ldc, soa, a, b, c, e, sa, sb, sc):
    """element e as float64 arrays A (M x K x soa or M x K), B (K x N or K x N x soa), C (M x N x soa)"""
    from numpy.lib.stride_tricks import as_strided
    s = a.itemsize
    if form == "ac":
        A = as_strided(a[e * sa:], (M, K, soa), (lda * soa * s, soa * s, s))
        B = as_strided(b[e * sb:], (K, N), (ldb * s, s))
    else:
        A = as_strided(a[e * sa:], (M, K), (lda * s, s))
        B = as_strided(b[e * sb:], (K, N, soa), (ldb * soa * s, soa * s, s))
    C = as_strided(c[e * sc:], (M, N, soa), (ldc * soa * s, soa * s, s))
    return A.astype(np.float64), B.astype(np.float64), C.astype(np.float64)


def product64(form, A, B, C0, beta):
    """float64 product and the scale of its terms (|op1| |op2| + beta |C0|)"""
    if form == "ac":
        P, S = np.einsum("mks,kn->mns", A, B), np.einsum("mks,kn->mns", np.abs(A), np.abs(B))
    else:
        P, S = np.einsum("mk,kns->mns", A, B), np.einsum("mk,kns->mns", np.abs(A), np.abs(B))
    return P + beta * C0, S + beta * np.abs(C0)


class RmOracle:
    """ctypes front-end of tests/rm_soa_oracle.c"""

    def __init__(self, path):
        self.f = ctypes.CDLL(path).orc_rm_soa_execute
        self.f.argtypes = [ctypes.c_int] * 9 + [ctypes.c_double] + [ctypes.c_void_p] * 3 + [ctypes.c_long] * 4
        self.f.restype = None

    def rm_soa_execute(self, form, M, N, K, lda, ldb, ldc, soa, beta, a, b, c, n_elem, stride_a, stride_b, stride_c):
        """in place on the flat array c; a, b, c flat arrays of one dtype, element strides in scalars (0: shared operand)"""
        assert form in ("ac", "bc") and a.dtype == b.dtype == c.dtype and c.flags.c_contiguous
        a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
        self.f(int(c.dtype == np.float64), 0 if form == "ac" else 1, M, N, K, lda, ldb, ldc, soa, float(beta),
               a.ctypes.data, b.ctypes.data, c.ctypes.data, n_elem, stride_a, stride_b, stride_c)
        return c


@pytest.fixture(scope="module")
def rm_oracle():
    """the restatement compiled into a temporary directory (the tree may be read-only); every fma is explicit"""
    tmp = tempfile.mkdtemp(prefix="rm_soa_oracle_")
    try:
        lib = os.path.join(tmp, "librm_soa_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-shared", "-o", lib,
                               os.path.join(HERE, "rm_soa_oracle.c"), "-lm"])
        yield RmOracle(lib)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def oracle_run(rm_oracle, form, M, N, K, lda, ldb, ldc, soa, beta, a, b, c0, E, sa, sb, sc):
    want = c0.copy()
    rm_oracle.rm_soa_execute(form, M, N, K, lda, ldb, ldc, soa, beta, a, b, want, E, sa, sb, sc)
    return want


FORMS = ("ac", "bc")
DTYPES = (np.float64, np.float32)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("beta", (0.0, 1.0))
def test_oracle_against_float64_product(rm_oracle, form, dt, beta):
    rng = np.random.default_rng(40)
    for (M, N, K, soa, pad) in ((35, 9, 9, 8, 0), (35, 9, 35, 4, 2), (7, 5, 3, 3, 1), (12, 20, 64, 2, 0)):
        lda, ldb, ldc, E = K + pad, N + pad, N + pad, 3
        ea, eb, ec = extents(form, M, N, K, lda, ldb, ldc, soa)
        sa, sb, sc = ea + pad, eb + pad, ec + pad
        a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, lda, ldb, ldc, E, sa, sb, sc)
        got = oracle_run(rm_oracle, form, M, N, K, lda, ldb, ldc, soa, beta, a, b, c0, E, sa, sb, sc)
        eps = np.finfo(dt).eps
        for e in range(E):
            A, B, C0 = dense_views(form, M, N, K, lda, ldb, ldc, soa, a, b, c0, e, sa, sb, sc)
            want, scale = product64(form, A, B, C0, beta)
            C = dense_views(form, M, N, K, lda, ldb, ldc, soa, a, b, got, e, sa, sb, sc)[2]
            assert (np.abs(C - want) <= K * eps * scale).all(), (form, M, N, K, soa, e)
        untouched = np.ones(got.shape, bool)
        for e in range(E):
            for m in range(M):
                o = e * sc + m * ldc * soa
                untouched[o:o + N * soa] = False
        assert (got[untouched] == SENT).all(), "padding or element gap written"


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt", DTYPES)
def test_oracle_exact_on_small_integers(rm_oracle, form, dt):
    rng = np.random.default_rng(41)
    M, N, K, soa, E = 9, 7, 11, 4, 2
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    for beta in (0.0, 1.0):
        a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, ea, eb, ec, ints=True)
        got = oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, beta, a, b, c0, E, ea, eb, ec)
        for e in range(E):
            A, B, C0 = dense_views(form, M, N, K, K, N, N, soa, a, b, c0, e, ea, eb, ec)
            want = product64(form, A, B, C0, beta)[0]
            assert np.array_equal(dense_views(form, M, N, K, K, N, N, soa, a, b, got, e, ea, eb, ec)[2], want)


def create_raw(xs, form, dt, M, N, K, lda, ldb, ldc, soa, beta):
    return xs.rm_soa_create(form, np.dtype(dt) == np.float64, M, N, K, lda, ldb, ldc, soa, beta)


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt", DTYPES)
def test_create_rejects_invalid_arguments(xs, form, dt):
    """host only: no device needed"""
    xs.clear_error()
    h = create_raw(xs, form, dt, 35, 9, 9, 9, 9, 9, 8, 1.0)
    assert h and xs.last_error()[0] == 0
    xs.rm_soa_destroy(h)
    bad = [((0, 9, 9, 9, 9, 9, 8, 0.0), -80), ((35, 0, 9, 9, 9, 9, 8, 0.0), -80), ((35, 9, 0, 9, 9, 9, 8, 0.0), -80),
           ((35, 9, 9, 9, 9, 9, 0, 0.0), -80), ((-1, 9, 9, 9, 9, 9, 8, 0.0), -80),
           ((35, 9, 9, 8, 9, 9, 8, 0.0), -81), ((35, 9, 9, 9, 8, 9, 8, 0.0), -81), ((35, 9, 9, 9, 9, 8, 8, 0.0), -81),
           ((35, 9, 9, 9, 9, 9, 8, 0.5), -82), ((35, 9, 9, 9, 9, 9, 8, -1.0), -82), ((35, 9, 9, 9, 9, 9, 8, 2.0), -82),
           ((35, 9, 9, 9, 9, 9, 8, float("nan")), -82)]
    for args, code in bad:
        assert not create_raw(xs, form, dt, *args), args
        assert xs.last_error()[0] == code, (args, xs.last_error())
        xs.clear_error()


def test_execute_rejects_invalid_arguments_without_launching(xs):
    """checked before any CUDA call, so this runs without a device too"""
    xs.clear_error()
    h = create_raw(xs, "ac", np.float64, 35, 9, 9, 9, 9, 9, 8, 1.0)
    ec = (34 * 9 + 9) * 8
    n0 = xs.launch_count()
    for (n, sa, sb, sc) in ((2, -1, 81, ec), (2, 2520, -1, ec), (2, 2520, 81, -1), (2, 2520, 81, ec - 1), (5, 2520, 81, 0), (-1, 0, 0, ec)):
        xs.rm_soa_execute(h, 16, 16, 16, n, sa, sb, sc)
        assert xs.last_error()[0] == -83, (n, sa, sb, sc)
        xs.clear_error()
    xs.rm_soa_execute(h, 16, 16, 16, 0, 2520, 81, ec)     # no elements: nothing to do, no error
    assert xs.last_error()[0] == 0
    assert xs.launch_count() == n0
    xs.rm_soa_execute(None, 16, 16, 16, 1, 0, 0, 0)
    assert xs.last_error()[0] == -83
    xs.clear_error()
    xs.rm_soa_destroy(h)


# ---------------------------------------------------------------------------------------------------------------- GPU
def gpu_run(gpu, form, dt, M, N, K, soa, beta, lda, ldb, ldc, a, b, c0, E, sa, sb, sc, shift=(0, 0, 0), stream=None):
    """uploads, executes once and returns C; shift: scalars added to each device base pointer"""
    es = np.dtype(dt).itemsize
    bufs = []
    for arr, sh in zip((a, b, c0), shift):
        d = gpu.DeviceBuffer(arr.nbytes + sh * es + 16)
        d.upload(arr, sh * es)
        bufs.append(d)
    op = gpu.RmSoa(form, M, N, K, soa, dt, lda=lda, ldb=ldb, ldc=ldc, beta=beta)
    op.execute(bufs[0].ptr + shift[0] * es, bufs[1].ptr + shift[1] * es, bufs[2].ptr + shift[2] * es, E, sa, sb, sc, stream)
    gpu.synchronize()
    kernel = gpu.last_compute_kernel()
    C = bufs[2].to_numpy(dt, c0.shape, shift[2] * es)
    op.destroy()
    for d in bufs:
        d.free()
    return C, kernel


SHAPES = [(35, 9, 9, 0, 200), (35, 9, 35, 0, 200), (84, 9, 84, 0, 100), (1, 1, 1, 0, 3), (7, 5, 3, 2, 5), (5, 6, 200, 1, 4),
          (37, 21, 11, 3, 6)]           # W1, W2, W3 at a few hundred elements; tiny; K = 200; M and N past the register block (8)


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16), (np.float64, 1), (np.float32, 3)])
@pytest.mark.parametrize("beta", (0.0, 1.0))
@pytest.mark.parametrize("M,N,K,pad,E", SHAPES)
def test_gpu_forms_and_sizes(gpu, rm_oracle, form, dt, soa, beta, M, N, K, pad, E):
    """padded pitches and element gaps (SENT must survive), per-element operands"""
    rng = np.random.default_rng(M * 1000 + N * 10 + K)
    lda, ldb, ldc = K + pad, N + pad, N + pad
    ea, eb, ec = extents(form, M, N, K, lda, ldb, ldc, soa)
    sa, sb, sc = ea + 4 * pad, eb + 4 * pad, ec + 4 * pad
    a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, lda, ldb, ldc, E, sa, sb, sc)
    C, kernel = gpu_run(gpu, form, dt, M, N, K, soa, beta, lda, ldb, ldc, a, b, c0, E, sa, sb, sc)
    assert kernel.startswith("rm_soa_" + form), kernel
    assert same(C, oracle_run(rm_oracle, form, M, N, K, lda, ldb, ldc, soa, beta, a, b, c0, E, sa, sb, sc)), kernel
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
def test_gpu_strides(gpu, rm_oracle, form, dt, soa):
    """an input shared by all elements (stride 0) on either side, 1 and 0 elements, and 148 k + 1 elements (ragged persistent loop)"""
    rng = np.random.default_rng(7)
    M, N, K = 20, 9, 13
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    for (E, sa, sb) in ((300, 0, eb), (300, ea, 0), (300, 0, 0), (1, ea, eb), (148 * 7 + 1, ea, eb), (148 * 7 + 1, ea if form == "ac" else 0, eb if form == "bc" else 0)):
        for beta in (0.0, 1.0):
            a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, sa, sb, ec)
            C, kernel = gpu_run(gpu, form, dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, sa, sb, ec)
            assert kernel == "rm_soa_%s (staged)" % form
            assert same(C, oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, beta, a, b, c0, E, sa, sb, ec)), (E, sa, sb, beta)
    # no elements: no launch, no error
    op = gpu.RmSoa(form, M, N, K, soa, dt)
    n0 = gpu.launch_count()
    d = gpu.DeviceBuffer(64)
    op.execute(d, d, d, 0)
    gpu.synchronize()
    assert gpu.launch_count() == n0
    op.destroy(); d.free()
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
def test_gpu_64bit_offsets(gpu, rm_oracle, form):
    """two elements whose C lie more than 4 GiB apart: only the touched regions are compared"""
    rng = np.random.default_rng(8)
    dt, soa, M, N, K = np.float32, 16, 35, 9, 9
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    sc = (1 << 30) + 4096                               # scalars: element 1's C starts 4 GiB + 16 KiB in
    a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, 2, ea, eb, ec)
    want = oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, 1.0, a, b, c0, 2, ea, eb, ec)
    dA, dB = gpu.DeviceBuffer.from_numpy(a), gpu.DeviceBuffer.from_numpy(b)
    dC = gpu.DeviceBuffer((sc + ec) * 4)
    dC.upload(c0[:ec], 0); dC.upload(c0[ec:], sc * 4)
    op = gpu.RmSoa(form, M, N, K, soa, dt, beta=1.0)
    op.execute(dA, dB, dC, 2, ea, eb, sc)
    gpu.synchronize()
    assert same(dC.to_numpy(dt, (ec,), 0), want[:ec]) and same(dC.to_numpy(dt, (ec,), sc * 4), want[ec:])
    op.destroy()
    for d in (dA, dB, dC):
        d.free()
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
def test_gpu_staged_and_direct_paths(gpu, rm_oracle, form, dt, soa):
    """a base pointer or an element stride one scalar off 16 bytes, and a shape whose double buffer does not fit in shared
    memory, take the direct path; both paths give the staged path's bits"""
    rng = np.random.default_rng(9)
    M, N, K, E = 35, 9, 9, 300
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    xs_ = ea if form == "ac" else eb                      # the SoA input's element extent
    for beta in (0.0, 1.0):
        a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, ea, eb, ec)
        ref, kernel = gpu_run(gpu, form, dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, ea, eb, ec)
        assert kernel == "rm_soa_%s (staged)" % form
        assert same(ref, oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, beta, a, b, c0, E, ea, eb, ec))
        x = 0 if form == "ac" else 1
        shift = [0, 0, 0]; shift[x] = 1
        C, kernel = gpu_run(gpu, form, dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, ea, eb, ec, shift=tuple(shift))
        assert kernel == "rm_soa_%s (direct)" % form and same(C, ref)
        C, kernel = gpu_run(gpu, form, dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, ea, eb, ec, shift=(1, 1, 1))
        assert kernel == "rm_soa_%s (direct)" % form and same(C, ref)
        # element stride one scalar longer: the same data re-laid, compared element by element
        st = [ea, eb]; st[x] = xs_ + 1
        a2, b2, c2 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, st[0], st[1], ec)
        for e in range(E):
            (a2 if x == 0 else b2)[e * (xs_ + 1):e * (xs_ + 1) + xs_] = (a if x == 0 else b)[e * xs_:(e + 1) * xs_]
        (b2 if x == 0 else a2)[:] = (b if x == 0 else a)
        C, kernel = gpu_run(gpu, form, dt, M, N, K, soa, beta, K, N, N, a2, b2, c0, E, st[0], st[1], ec)
        assert kernel == "rm_soa_%s (direct)" % form and same(C, ref)
    # too large for the double buffer (2 x 1.2 MB)
    M, N, K, E = 300, 10, 64, 3
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    if form == "bc":
        M, N, K = 10, 300, 64
        ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, ea, eb, ec)
    C, kernel = gpu_run(gpu, form, dt, M, N, K, soa, 1.0, K, N, N, a, b, c0, E, ea, eb, ec)
    assert kernel == "rm_soa_%s (direct)" % form
    assert same(C, oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, 1.0, a, b, c0, E, ea, eb, ec))
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
def test_gpu_special_values(gpu, rm_oracle, form, dt, soa):
    """NaN and Inf tracers follow the chain (0 * Inf = NaN: zeros are not skipped); beta = 0 never reads C (NaN C0)"""
    rng = np.random.default_rng(10)
    M, N, K, E = 12, 9, 10, 40
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, ea, eb, ec)
    a[rng.choice(a.size, 6, replace=False)] = 0.0
    b[rng.choice(b.size, 6, replace=False)] = 0.0
    a[rng.choice(a.size, 3, replace=False)] = np.inf
    b[rng.choice(b.size, 3, replace=False)] = -np.inf
    a[rng.choice(a.size, 2, replace=False)] = np.nan
    a[:4] = 0.0; b[:4] = np.inf                                   # 0 * Inf on element 0
    b[4:8] = -0.0
    for beta in (0.0, 1.0):
        C, _ = gpu_run(gpu, form, dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, ea, eb, ec)
        want = oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, beta, a, b, c0, E, ea, eb, ec)
        assert np.isnan(want).any() and same(C, want)
    a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, ea, eb, ec)
    c0[:] = np.nan
    C, _ = gpu_run(gpu, form, dt, M, N, K, soa, 0.0, K, N, N, a, b, c0, E, ea, eb, ec)
    want = oracle_run(rm_oracle, form, M, N, K, K, N, N, soa, 0.0, a, b, c0, E, ea, eb, ec)
    assert same(C, want) and np.isnan(C).sum() == c0.size - E * M * N * soa    # only the gaps (untouched) stay NaN
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
def test_gpu_matches_sparse_entries_on_dense_operators(gpu, dt, soa):
    """ac with a shared, fully non-zero b = csc_soa built from that b; bc with a shared dense a = csr_soa with lda = 0"""
    rng = np.random.default_rng(11)
    M, N, K, E = 35, 9, 35, 150
    for beta in (0.0, 1.0):
        # ac
        ea, eb, ec = extents("ac", M, N, K, K, N, N, soa)
        a, b, c0 = flat_case(rng, "ac", M, N, K, soa, dt, K, N, N, E, ea, 0, ec)
        b[b == 0] = 0.5
        C, _ = gpu_run(gpu, "ac", dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, ea, 0, ec)
        bm = b.reshape(K, N)
        colptr = np.arange(N + 1, dtype=np.uint32) * K
        rowidx = np.tile(np.arange(K, dtype=np.uint32), N)
        op = gpu.CsrSoa(M, N, K, colptr, rowidx, np.ascontiguousarray(bm.T).ravel(), soa, beta=beta, sparse="B", fmt="csc")
        dA, dC = gpu.DeviceBuffer.from_numpy(a), gpu.DeviceBuffer.from_numpy(c0)
        op.execute(dA, dC, E, ea, ec)
        gpu.synchronize()
        S = dC.to_numpy(dt, c0.shape)
        op.destroy(); dA.free(); dC.free()
        assert np.array_equal(bits(C), bits(S)), ("ac", beta)
        # bc
        ea, eb, ec = extents("bc", M, N, K, K, N, N, soa)
        a, b, c0 = flat_case(rng, "bc", M, N, K, soa, dt, K, N, N, E, 0, eb, ec)
        a[a == 0] = 0.5
        C, _ = gpu_run(gpu, "bc", dt, M, N, K, soa, beta, K, N, N, a, b, c0, E, 0, eb, ec)
        rowptr = np.arange(M + 1, dtype=np.uint32) * K
        colidx = np.tile(np.arange(K, dtype=np.uint32), M)
        op = gpu.CsrSoa(M, N, K, rowptr, colidx, a, soa, beta=beta, sparse="A")
        dB, dC = gpu.DeviceBuffer.from_numpy(b), gpu.DeviceBuffer.from_numpy(c0)
        op.execute(dB, dC, E, eb, ec)
        gpu.synchronize()
        S = dC.to_numpy(dt, c0.shape)
        op.destroy(); dB.free(); dC.free()
        assert np.array_equal(bits(C), bits(S)), ("bc", beta)
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
def test_gpu_stream_and_graph(gpu, form):
    """on a non-default stream, and captured into a graph replayed twice: the bits of a direct call"""
    rng = np.random.default_rng(12)
    dt, soa, M, N, K, E = np.float64, 8, 35, 9, 9, 500
    ea, eb, ec = extents(form, M, N, K, K, N, N, soa)
    a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, K, N, N, E, ea, eb, ec)
    ref, _ = gpu_run(gpu, form, dt, M, N, K, soa, 0.0, K, N, N, a, b, c0, E, ea, eb, ec)
    st = gpu.Stream()
    C, _ = gpu_run(gpu, form, dt, M, N, K, soa, 0.0, K, N, N, a, b, c0, E, ea, eb, ec, stream=st)
    assert np.array_equal(bits(C), bits(ref))
    L = gpu.load()
    dA, dB, dC = (gpu.DeviceBuffer.from_numpy(x) for x in (a, b, c0))
    op = gpu.RmSoa(form, M, N, K, soa, dt, beta=0.0)
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    op.execute(dA, dB, dC, E, ea, eb, ec, st)
    g = L.libxsmm_b200_graph_end(st.ptr)
    assert g
    gpu.check()
    for _ in range(2):
        dC.upload(c0)
        assert 0 == L.libxsmm_b200_graph_launch(ctypes.c_void_p(g), st.ptr)
        st.synchronize()
        assert np.array_equal(bits(dC.to_numpy(dt, c0.shape)), bits(ref))
    L.libxsmm_b200_graph_destroy(ctypes.c_void_p(g))
    op.destroy(); st.destroy()
    for d in (dA, dB, dC):
        d.free()
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 3)])
def test_gpu_guard_bands(gpu, form, dt, soa):
    """every buffer between two 64 KiB bands of a known pattern (the pattern of test_hardening_gpu.py): bands and inputs
    bit-identical afterwards, on the staged (aligned) and the direct (one scalar off) path"""
    G = 1 << 16
    es = np.dtype(dt).itemsize

    def guarded(arr, shift=0):
        raw = np.full(2 * G + shift + arr.nbytes, 0xA5, np.uint8)
        raw[G + shift:G + shift + arr.nbytes] = arr.view(np.uint8).ravel()
        return gpu.DeviceBuffer.from_numpy(raw), raw

    def check(d, raw, nbytes, changed_ok, shift=0):
        got = d.to_numpy(np.uint8, raw.shape)
        lo, hi = G + shift, G + shift + nbytes
        assert np.array_equal(got[:lo], raw[:lo]) and np.array_equal(got[hi:], raw[hi:]), "guard band overwritten"
        if not changed_ok:
            assert np.array_equal(got, raw), "input buffer was written"
        d.free()

    rng = np.random.default_rng(13)
    for (M, N, K, pad, E) in ((35, 9, 9, 0, 7), (13, 11, 5, 3, 9)):
        for shift in (0, es):
            lda, ldb, ldc = K + pad, N + pad, N + pad
            ea, eb, ec = extents(form, M, N, K, lda, ldb, ldc, soa)
            a, b, c0 = flat_case(rng, form, M, N, K, soa, dt, lda, ldb, ldc, E, ea, eb, ec)
            (dA, rA), (dB, rB), (dC, rC) = guarded(a, shift), guarded(b, shift), guarded(c0, shift)
            op = gpu.RmSoa(form, M, N, K, soa, dt, lda=lda, ldb=ldb, ldc=ldc, beta=1.0)
            op.execute(dA.ptr + G + shift, dB.ptr + G + shift, dC.ptr + G + shift, E, ea, eb, ec)
            gpu.synchronize()
            op.destroy()
            check(dA, rA, a.nbytes, False, shift); check(dB, rB, b.nbytes, False, shift); check(dC, rC, c0.nbytes, True, shift)
    gpu.check()


@pytest.mark.gpu
def test_gpu_one_launch_per_execute(gpu):
    dt, soa, M, N, K, E = np.float32, 16, 35, 9, 35, 64
    ec = extents("bc", M, N, K, K, N, N, soa)[2]
    big = np.ones(M * K * soa, dt)                                # either operand of either form, shared by all elements
    dA, dB, dC = (gpu.DeviceBuffer.from_numpy(x) for x in (big, big, np.zeros(E * ec, dt)))
    for form in FORMS:
        op = gpu.RmSoa(form, M, N, K, soa, dt, beta=1.0)
        for i in range(3):
            n0 = gpu.launch_count()
            op.execute(dA, dB, dC, E, 0, 0, ec)
            assert gpu.launch_count() == n0 + 1
        op.destroy()
    gpu.synchronize()
    for d in (dA, dB, dC):
        d.free()
