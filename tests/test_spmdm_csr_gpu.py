"""spmdm with A given in CSR form (libxsmm_spmdm_createSparseSlice_csr_{fp32,bfloat16}_stream, kernel K1c).

The contract: for a well-formed CSR the slices -- rowidx[0..nrows], colidx / values over [0, nnz_slice) and slice_nnz -- are
bit for bit what the dense route writes for the densified A, so every multiply kernel gives the dense route's bits.  Both
routes run on the GPU here and are compared array by array, and with the oracle on the densified A."""
import numpy as np
import pytest

from test_spmdm_gpu import oracle_spmdm, valid_slices_equal

pytestmark = pytest.mark.gpu
K4 = "spmdm_compute_tc_kernel"
K4P = "spmdm_compute_tc16p_kernel"
K4S = "spmdm_compute_tc16s_kernel"


# ---- helpers ---------------------------------------------------------------------------------------------------------
def to_csr(A, keep=None):
    """CSR arrays of the entries of A where `keep` is set (default: nonzero bit pattern), ascending columns per row."""
    keep = (A.view(np.uint32 if A.dtype == np.float32 else np.uint16) != 0) if keep is None else keep
    rows, cols = np.nonzero(keep)
    row_ptr = np.zeros(A.shape[0] + 1, np.uint32)
    np.cumsum(np.bincount(rows, minlength=A.shape[0]), out=row_ptr[1:])
    return row_ptr, cols.astype(np.uint32), np.ascontiguousarray(A[rows, cols])


def densify(M, K, row_ptr, col_idx, values):
    A = np.zeros((M, K), values.dtype)
    rows = np.repeat(np.arange(M), np.diff(row_ptr.astype(np.int64)))
    A[rows, col_idx] = values
    return A


def sparse_a(M, K, density, bf16, seed, empty_rows=0.1):
    """uniform values in [0.5, 1.5) with both signs at `density`, a share of rows left empty"""
    rng = np.random.default_rng(seed)
    A = np.where(rng.random((M, K)) < density, (rng.random((M, K)) + 0.5) * rng.choice([-1.0, 1.0], (M, K)), 0.0).astype(np.float32)
    A[rng.random(M) < empty_rows] = 0
    return to_bf16(A) if bf16 else A


def to_bf16(x):
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) >> np.uint32(16)).astype(np.uint16)


def from_bf16(h):
    return (np.ascontiguousarray(h, np.uint16).astype(np.uint32) << np.uint32(16)).view(np.float32)


def dense_b_c(M, N, K, bf16, seed, transb="N", transc="N"):
    rng = np.random.default_rng(seed + 1)
    B = rng.uniform(-1, 1, (N, K) if transb == "T" else (K, N)).astype(np.float32)
    C0 = rng.uniform(-1, 1, (N, M) if transc == "T" else (M, N)).astype(np.float32)
    return (to_bf16(B) if bf16 else B), C0


def slice_nnz(xs, p):
    """the arena's true per-slice counts: they follow the values and the auxiliary words (4 bytes per entry each)"""
    h = p.handle
    ns, cap = h.mb * h.kb, h.bm * h.bk
    out = np.empty(ns, np.uint32)
    xs.load().libxsmm_b200_synchronize()
    xs.load().libxsmm_b200_memcpy_d2h(out.ctypes.data, p.slices[0].values + 2 * ns * cap * 4, out.nbytes)
    xs.check()
    return out


class Csr:
    """device copies of CSR arrays"""

    def __init__(self, xs, row_ptr, col_idx, values):
        self.nnz = len(col_idx)
        self.rp, self.ci, self.va = (xs.DeviceBuffer.from_numpy(x) for x in (row_ptr, col_idx, values))

    def upload(self, row_ptr, col_idx, values):
        assert len(col_idx) == self.nnz
        self.rp.upload(row_ptr); self.ci.upload(col_idx); self.va.upload(values)

    def free(self):
        for d in (self.rp, self.ci, self.va):
            d.free()


def run(xs, M, N, K, threads, bf16, A=None, csr=None, B=None, C0=None, transb="N", transc="N", beta=0):
    """one handle, one slicing pass (dense A or CSR arrays), optionally one multiply.  Returns (geometry, slices, slice_nnz, C,
    kernel name)."""
    import pyoracle
    p = xs.Spmdm(M, N, K, threads)
    bufs = []
    try:
        if csr is not None:
            d = Csr(xs, *csr)
            bufs += [d.rp, d.ci, d.va]
            p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16)
        else:
            dA = xs.DeviceBuffer.from_numpy(A)
            bufs.append(dA)
            p.create_slices(dA, "N", bf16)
        C, name = None, None
        if B is not None:
            dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
            bufs += [dB, dC]
            p.compute(dB, dC, transb, transc, beta, bf16)
            xs.synchronize()
            C = dC.to_numpy(np.float32, C0.shape)
            name = xs.last_compute_kernel()
        xs.synchronize()
        g = pyoracle.Geometry(p.geometry)
        g["scratch"] = 0
        return g, p.read_slices(), slice_nnz(xs, p), C, name
    finally:
        for b in bufs:
            b.free()
        p.destroy()


def assert_same_slices(oracle, g, A, got, got_nnz, dense, dense_nnz):
    """CSR route == dense route (GPU) == oracle on the densified A, array by array"""
    og, osl, _ = oracle_spmdm(oracle, g, A, np.zeros((g.k, g.n), A.dtype), np.zeros((g.m, g.n), np.float32), "N", "N", "N", 0.0)
    valid_slices_equal(og, got, dense)
    valid_slices_equal(og, got, osl)
    import pyoracle
    np.testing.assert_array_equal(got_nnz, dense_nnz)
    np.testing.assert_array_equal(got_nnz, pyoracle.slice_counts(og, osl[0]))


def both_routes_slices(gpu, oracle, M, K, A, bf16, threads, csr=None, N=16):
    csr = to_csr(A) if csr is None else csr
    g, sl, cnt, _, _ = run(gpu, M, N, K, threads, bf16, csr=csr)
    gd, sld, cntd, _, _ = run(gpu, M, N, K, threads, bf16, A=A)
    assert dict(g) == dict(gd)
    assert_same_slices(oracle, g, A, sl, cnt, sld, cntd)
    return g, cnt


# ---- 1. slices, bit for bit ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,density,dtype,bn,threads", [
    (300, 260, 0.05, "f32", 48, 1),       # partial last row block, scalar remainder (K % 128 = 4)
    (300, 260, 0.05, "bf16", 48, 1),
    (512, 384, 0.001, "f32", 96, 1),
    (512, 384, 0.50, "bf16", 96, 4),      # K % 128 == 0: the structured-sparse words too
    (1024, 256, 0.02, "bf16", 6, 1),      # simd_w 1: no vector part, NaN kept everywhere
    (700, 200, 0.20, "f32", 6, 3),
    (2048, 384, 0.01, "bf16", 48, 56),    # bm = 245
    (640, 129, 0.30, "f32", 48, 8),
])
def test_slices_match_dense_route_and_oracle(gpu, oracle, monkeypatch, M, K, density, dtype, bn, threads):
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_BN", str(bn))
    A = sparse_a(M, K, density, dtype == "bf16", seed=M + K + bn)
    g, cnt = both_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", threads)
    assert g.bn == bn
    assert cnt.sum() > 0
    gpu.check()


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_empty_matrix(gpu, oracle, dtype):
    """nnz = 0 (NULL col_idx / values allowed) gives all-empty slices"""
    M, K = 300, 260
    A = np.zeros((M, K), np.uint16 if dtype == "bf16" else np.float32)
    p = gpu.Spmdm(M, 16, K, 1)
    rp = gpu.DeviceBuffer.from_numpy(np.zeros(M + 1, np.uint32))
    try:
        p.create_slices_csr(rp, None, None, 0, dtype == "bf16")
        gpu.check()
        assert not slice_nnz(gpu, p).any()
    finally:
        rp.free()
        p.destroy()
    both_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", 1)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_full_slice_wraps_the_row_counter(gpu, oracle, dtype):
    """a fully dense 512 x 128 slice: rowidx wraps at 65536 like the reference's u16 counter, slice_nnz holds 65536"""
    M, K = 512, 128
    A = (np.random.default_rng(9).random((M, K)) + 0.5).astype(np.float32)
    A = to_bf16(A) if dtype == "bf16" else A
    g, cnt = both_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", 1, N=48)      # N = bn: the geometry keeps bm = 512
    assert g.bm == 512 and list(cnt) == [65536]


# ---- 2. special values -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_special_values(gpu, oracle, dtype):
    """explicit 0, -0, NaN (vector part and scalar remainder), +-Inf and subnormals as stored CSR entries: the kept set and the
    slices equal the dense route's"""
    M, K = 200, 260                              # last k-block: 4 columns, all in the scalar remainder
    rng = np.random.default_rng(21)
    A = np.where(rng.random((M, K)) < 0.1, rng.uniform(-1, 1, (M, K)), 0.0).astype(np.float32)
    keep = A != 0
    specials = np.array([0.0, -0.0, np.nan, np.inf, -np.inf, 1e-40, -3e-39, 1e-45], np.float32)
    if dtype == "bf16":
        specials = from_bf16(to_bf16(specials))  # bf16 bit patterns: 0x0000, 0x8000, NaN, +-Inf, subnormals
    for r in range(M):
        for c in list(rng.choice(256, 3, replace=False)) + [256 + r % 4]:
            A[r, c] = specials[(r + c) % len(specials)]
            keep[r, c] = True
    A = to_bf16(A) if dtype == "bf16" else A
    csr = to_csr(A, keep)
    assert np.array_equal(densify(M, K, *csr).view(np.uint8), A.view(np.uint8))
    both_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", 1, csr)
    gpu.check()


# ---- 3. C, bit for bit, with the same kernel ---------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tb,tc,beta", [
    ("f32", "N", "N", 0.0), ("f32", "T", "N", 1.0), ("f32", "N", "T", 0.5), ("f32", "T", "T", 1.0),
    ("bf16", "N", "N", 0), ("bf16", "T", "T", 1), ("bf16", "N", "T", 0),
])
def test_cuda_core_product_matches_oracle_and_dense_route(gpu, oracle, monkeypatch, dtype, tb, tc, beta):
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    M, N, K = 300, 203, 260
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.08, bf16, seed=4)
    B, C0 = dense_b_c(M, N, K, bf16, 4, tb, tc)
    g, sl, cnt, C, name = run(gpu, M, N, K, 1, bf16, csr=to_csr(A), B=B, C0=C0, transb=tb, transc=tc, beta=beta)
    _, sld, cntd, Cd, named = run(gpu, M, N, K, 1, bf16, A=A, B=B, C0=C0, transb=tb, transc=tc, beta=beta)
    assert name == named
    np.testing.assert_array_equal(C.view(np.uint32), Cd.view(np.uint32))
    _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", tb, tc, float(beta))
    np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
    gpu.check()


@pytest.mark.parametrize("dtype,K,sparse,kernel", [
    ("f32", 300, None, K4),       # K % 128 != 0: the dense route writes no dense image either, both take K4 on tcoff
    ("bf16", 384, "0", K4P),
    ("bf16", 384, "1", K4S),
])
def test_tensor_core_kernels_same_bits(gpu, oracle, monkeypatch, dtype, K, sparse, kernel):
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    if sparse is not None:
        monkeypatch.setenv("LIBXSMM_B200_TC16_SPARSE", sparse)
    M, N = 512, 400
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.05, bf16, seed=K)
    B, C0 = dense_b_c(M, N, K, bf16, 7)
    g, sl, _, C, name = run(gpu, M, N, K, 1, bf16, csr=to_csr(A), B=B, C0=C0, beta=1)
    _, _, _, Cd, named = run(gpu, M, N, K, 1, bf16, A=A, B=B, C0=C0, beta=1)
    assert name == named == kernel
    np.testing.assert_array_equal(C.view(np.uint32), Cd.view(np.uint32))
    _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 1.0)
    assert float(np.abs(C.astype(np.float64) - OC).max() / np.abs(OC).max()) <= 1e-5
    gpu.check()


def test_c2_default_dispatch_takes_k4s(gpu, monkeypatch):
    """bf16 4096^3 at 1 %: once the handle knows the density the CSR route runs K4s, with the dense route's bits"""
    monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    monkeypatch.delenv("LIBXSMM_B200_TC16_SPARSE", raising=False)
    M = N = K = 4096
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, 0.01, dtype="bf16", seed=2)
    out = []
    for use_csr in (True, False):
        p = gpu.Spmdm(M, N, K, 1)
        d = Csr(gpu, *to_csr(A)) if use_csr else None
        dA = None if use_csr else gpu.DeviceBuffer.from_numpy(A)
        dB, dC = gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer(C0.nbytes)
        for _ in range(3):                       # from the third pass on the density estimate is known and stable: K4s alone
            dC.upload(C0)
            if use_csr:
                p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, True)
            else:
                p.create_slices(dA, "N", True)
            p.compute(dB, dC, "N", "N", 0, True)
            gpu.synchronize()
        out.append((dC.to_numpy(np.float32, C0.shape), gpu.last_compute_kernel()))
        d.free() if use_csr else dA.free()
        dB.free(); dC.free()
        p.destroy()
    assert out[0][1] == out[1][1] == K4S
    np.testing.assert_array_equal(out[0][0].view(np.uint32), out[1][0].view(np.uint32))
    gpu.check()


# ---- 4. state between passes ---------------------------------------------------------------------------------------
def test_stale_dense_image_is_never_used(gpu, oracle, monkeypatch):
    """a dense fp32 pass of X writes the dense tile image; a CSR pass of Y follows: the multiply must be Y's product"""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    M, N, K = 512, 256, 384
    X = sparse_a(M, K, 0.2, False, seed=1, empty_rows=0)
    Y = sparse_a(M, K, 0.2, False, seed=2, empty_rows=0)
    B, C0 = dense_b_c(M, N, K, False, 3)
    p = gpu.Spmdm(M, N, K, 1)
    dX, dB, dC = gpu.DeviceBuffer.from_numpy(X), gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer.from_numpy(C0)
    d = Csr(gpu, *to_csr(Y))
    try:
        p.create_slices(dX, "N", False)
        p.compute(dB, dC, "N", "N", 0.0, False)
        gpu.synchronize()
        assert gpu.last_compute_kernel() == "spmdm_compute_tcq_kernel"      # reads the image
        dC.upload(C0)
        p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, False)
        p.compute(dB, dC, "N", "N", 0.0, False)
        gpu.synchronize()
        assert gpu.last_compute_kernel() == K4
        C = dC.to_numpy(np.float32, C0.shape)
        _, _, OC = oracle_spmdm(oracle, pyoracle_geometry(p), Y, B, C0, "N", "N", "N", 0.0)
        assert float(np.abs(C.astype(np.float64) - OC).max() / np.abs(OC).max()) <= 1e-5
    finally:
        d.free()
        for b in (dX, dB, dC):
            b.free()
        p.destroy()
    gpu.check()


def pyoracle_geometry(p):
    import pyoracle
    g = pyoracle.Geometry(p.geometry)
    g["scratch"] = 0
    return g


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_csr_then_dense_then_legacy_compute(gpu, oracle, monkeypatch, dtype):
    """a CSR pass then a dense pass on one handle, each multiplied; then a CSR pass multiplied by the legacy per-block entries"""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    M, N, K = 300, 200, 256
    bf16 = dtype == "bf16"
    X, Y = sparse_a(M, K, 0.1, bf16, seed=5), sparse_a(M, K, 0.03, bf16, seed=6)
    B, C0 = dense_b_c(M, N, K, bf16, 5)
    p = gpu.Spmdm(M, N, K, 2)
    g = pyoracle_geometry(p)
    dY, dB, dC = gpu.DeviceBuffer.from_numpy(Y), gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer.from_numpy(C0)
    d = Csr(gpu, *to_csr(X))
    try:
        for src, A in (("csr", X), ("dense", Y)):
            dC.upload(C0)
            if src == "csr":
                p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16)
            else:
                p.create_slices(dY, "N", bf16)
            p.compute(dB, dC, "N", "N", 1, bf16)
            gpu.synchronize()
            _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 1.0)
            np.testing.assert_array_equal(dC.to_numpy(np.float32, C0.shape).view(np.uint32), OC.view(np.uint32), err_msg=src)
        dC.upload(C0)
        p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16)
        gpu.synchronize()
        h = p.handle
        for blk in range(h.mb * h.nb):
            if bf16:
                gpu.libxsmm_spmdm_compute_bfloat16_thread(h, "N", "N", 0x3F80, p.slices, dB, "N", 1, dC, blk, blk % 2, 2)
            else:
                gpu.libxsmm_spmdm_compute_fp32_thread(h, "N", "N", 1.0, p.slices, dB, "N", 1.0, dC, blk, blk % 2, 2)
        gpu.synchronize()
        _, _, OC = oracle_spmdm(oracle, g, X, B, C0, "N", "N", "N", 1.0)
        np.testing.assert_array_equal(dC.to_numpy(np.float32, C0.shape).view(np.uint32), OC.view(np.uint32), err_msg="legacy")
    finally:
        d.free()
        for b in (dY, dB, dC):
            b.free()
        p.destroy()
    gpu.check()


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_two_rounds_back_to_back_on_one_stream(gpu, oracle, dtype):
    """slice + multiply of X, then of Y, enqueued on one stream with no synchronisation in between (default dispatch)"""
    M, N, K = 512, 256, 384
    bf16 = dtype == "bf16"
    X, Y = sparse_a(M, K, 0.3, bf16, seed=7), sparse_a(M, K, 0.01, bf16, seed=8)
    B, C0 = dense_b_c(M, N, K, bf16, 7)
    p = gpu.Spmdm(M, N, K, 1)
    g = pyoracle_geometry(p)
    st = gpu.Stream()
    dB = gpu.DeviceBuffer.from_numpy(B)
    dC = [gpu.DeviceBuffer.from_numpy(C0) for _ in range(2)]
    ds = [Csr(gpu, *to_csr(A)) for A in (X, Y)]
    try:
        for d, c in zip(ds, dC):
            p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16, st)
            p.compute(dB, c, "N", "N", 1, bf16, st)
        st.synchronize()
        for A, c in zip((X, Y), dC):
            _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 1.0)
            C = c.to_numpy(np.float32, C0.shape)
            assert float(np.abs(C.astype(np.float64) - OC).max() / np.abs(OC).max()) <= 1e-5
    finally:
        for d in ds:
            d.free()
        for b in [dB] + dC:
            b.free()
        st.destroy()
        p.destroy()
    gpu.check()


# ---- 5. graph --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tc_mode", [("f32", "0"), ("bf16", "0"), ("bf16", None)])
def test_graph_replay_with_new_arrays(gpu, oracle, monkeypatch, dtype, tc_mode):
    """CSR slicing + multiply captured once, replayed with new index / value contents in the same buffers (same nnz)"""
    if tc_mode is None:
        monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    else:
        monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", tc_mode)
    xs, L = gpu, gpu.load()
    M, N, K = 512, 400, 384
    bf16 = dtype == "bf16"
    nnz = M * K // 20
    rng = np.random.default_rng(30)
    mats = []
    for i in range(2):
        keep = np.zeros(M * K, bool)
        keep[rng.choice(M * K, nnz, replace=False)] = True
        A = np.where(keep.reshape(M, K), rng.uniform(0.5, 1.5, (M, K)), 0.0).astype(np.float32)
        mats.append(to_bf16(A) if bf16 else A)
    B, C0 = dense_b_c(M, N, K, bf16, 30)
    p = xs.Spmdm(M, N, K, 1)
    g = pyoracle_geometry(p)
    d = Csr(xs, *to_csr(mats[0]))
    dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
    st = xs.Stream()
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16, st)
    p.compute(dB, dC, "N", "N", 0, bf16, st)
    graph = L.libxsmm_b200_graph_end(st.ptr)
    xs.check()
    assert graph
    try:
        for A in mats + mats[:1]:
            d.upload(*to_csr(A))
            dC.upload(C0)
            assert 0 == L.libxsmm_b200_graph_launch(graph, st.ptr)
            st.synchronize()
            C = dC.to_numpy(np.float32, C0.shape)
            _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.0)
            if tc_mode == "0":
                np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
            else:
                assert float(np.abs(C.astype(np.float64) - OC).max() / np.abs(OC).max()) <= 1e-5
    finally:
        L.libxsmm_b200_graph_destroy(graph)
        d.free()
        for b in (dB, dC):
            b.free()
        st.destroy()
        p.destroy()
    gpu.check()


# ---- 6. rejections and safety ----------------------------------------------------------------------------------------
def test_host_side_rejections_launch_nothing(gpu):
    xs = gpu
    M, K = 64, 128
    p = xs.Spmdm(M, 16, K, 1)
    rp = xs.DeviceBuffer.from_numpy(np.zeros(M + 1, np.uint32))
    ci, va = xs.DeviceBuffer(64), xs.DeviceBuffer(64)
    stale = xs.libxsmm_spmdm_handle.from_buffer_copy(p.handle)     # becomes an unknown handle once p is destroyed
    other = xs.Spmdm(M, 16, K, 1)
    other.destroy()
    cases = [
        (xs.libxsmm_spmdm_handle(), rp, ci, va, 1, -10),          # never initialised
        (other.handle, rp, ci, va, 1, -10),                       # destroyed: its arena pointer is cleared
        (p.handle, None, ci, va, 1, -90),
        (p.handle, None, None, None, 0, -90),                     # row_ptr is needed even for nnz = 0
        (p.handle, rp, None, va, 1, -90),
        (p.handle, rp, ci, None, 1, -90),
        (p.handle, rp, ci, va, -1, -91),
        (p.handle, rp, ci, va, 1 << 32, -91),
    ]
    try:
        for bf16 in (False, True):
            f = xs.libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream if bf16 else xs.libxsmm_spmdm_createSparseSlice_csr_fp32_stream
            for h, r, c, v, nnz, code in cases:
                xs.clear_error()
                n0 = xs.launch_count()
                f(h, r, c, v, nnz, p.slices)
                assert xs.last_error()[0] == code, (nnz, code, xs.last_error())
                assert xs.launch_count() == n0
        p_base = p.handle.base_ptr_scratch_A
        p.destroy()
        assert p_base and stale.base_ptr_scratch_A == p_base
        xs.clear_error()
        n0 = xs.launch_count()
        xs.libxsmm_spmdm_createSparseSlice_csr_fp32_stream(stale, rp, ci, va, 1, None)
        assert xs.last_error()[0] == -11 and xs.launch_count() == n0
    finally:
        xs.clear_error()
        for b in (rp, ci, va):
            b.free()
        p.destroy()


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_malformed_arrays_stay_in_bounds(gpu, oracle, monkeypatch, dtype):
    """columns >= K, duplicated and unsorted columns, row_ptr past nnz and not monotone: the result is unspecified, but the pass
    and the multiply stay inside their arrays (a guard-banded C keeps its guards) and the next well-formed pass is exact"""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    xs = gpu
    M, N, K = 300, 200, 384
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.2, bf16, seed=12)
    row_ptr, col_idx, values = to_csr(A)
    nnz = len(col_idx)
    rng = np.random.default_rng(12)
    bad_cols = col_idx.copy()
    bad_cols[rng.choice(nnz, 200, replace=False)] = rng.integers(K, K + 70000, 200)        # columns >= K
    for r in range(0, M, 7):                                                                # unsorted / duplicated rows
        lo, hi = int(row_ptr[r]), int(row_ptr[r + 1])
        if hi - lo > 2:
            bad_cols[lo:hi] = bad_cols[lo:hi][::-1] if r % 2 else bad_cols[lo]
    bad_rp = row_ptr.copy()
    bad_rp[5] = nnz + 1000                                                                  # past nnz, then not monotone
    bad_rp[-1] = nnz + 7
    B, C0 = dense_b_c(M, N, K, bf16, 12)
    guard = 4096
    sentinel = np.float32(-12345.5)
    p = xs.Spmdm(M, N, K, 1)
    g = pyoracle_geometry(p)
    d = Csr(xs, bad_rp, bad_cols, values)
    dB = xs.DeviceBuffer.from_numpy(B)
    dCg = xs.DeviceBuffer.from_numpy(np.full(C0.size + 2 * guard, sentinel, np.float32))
    try:
        dCg.upload(C0, guard * 4)
        p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16)
        p.compute(dB, dCg.ptr + guard * 4, "N", "N", 1, bf16)
        xs.synchronize()
        out = dCg.to_numpy(np.float32, (C0.size + 2 * guard,))
        assert np.all(out[:guard] == sentinel) and np.all(out[-guard:] == sentinel)
        cnt = slice_nnz(xs, p)
        assert int(cnt.max()) <= g.bm * g.bk
        d.upload(row_ptr, col_idx, values)                          # well-formed again, same handle
        dCg.upload(C0, guard * 4)
        p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16)
        p.compute(dB, dCg.ptr + guard * 4, "N", "N", 1, bf16)
        xs.synchronize()
        out = dCg.to_numpy(np.float32, (C0.size + 2 * guard,))
        og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 1.0)
        valid_slices_equal(og, p.read_slices(), osl)
        np.testing.assert_array_equal(out[guard:-guard].reshape(C0.shape).view(np.uint32), OC.view(np.uint32))
        assert np.all(out[:guard] == sentinel) and np.all(out[-guard:] == sentinel)
    finally:
        d.free()
        for b in (dB, dCg):
            b.free()
        p.destroy()
    gpu.check()


# ---- 7. one launch per call --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_one_launch_per_csr_slicing_call(gpu, dtype):
    M, K = 1000, 640
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.05, bf16, seed=13)
    p = gpu.Spmdm(M, 64, K, 1)
    d = Csr(gpu, *to_csr(A))
    st = gpu.Stream()
    try:
        for _ in range(2):
            n0 = gpu.launch_count()
            p.create_slices_csr(d.rp, d.ci, d.va, d.nnz, bf16, st)
            assert gpu.launch_count() - n0 == 1
        st.synchronize()
    finally:
        d.free()
        st.destroy()
        p.destroy()
    gpu.check()
