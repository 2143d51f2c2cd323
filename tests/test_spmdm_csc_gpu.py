"""spmdm with A given in CSC form (libxsmm_spmdm_createSparseSlice_csc_{fp32,bfloat16}_stream, kernel K1t).

The contract: for a well-formed CSC the slices -- rowidx[0..nrows], colidx / values over [0, nnz_slice) and slice_nnz -- are
bit for bit what the dense route writes with transa = 'T' for the K x M array holding these entries, and what the CSR route
writes for A's CSR arrays.  All three routes run on the GPU here and are compared array by array, and with the oracle
(transa = 'T')."""
import numpy as np
import pytest

from test_spmdm_gpu import oracle_spmdm, valid_slices_equal
from test_spmdm_csr_gpu import Csr, dense_b_c, densify, from_bf16, pyoracle_geometry, slice_nnz, sparse_a, to_bf16, to_csr

pytestmark = pytest.mark.gpu
K4 = "spmdm_compute_tc_kernel"
K4P = "spmdm_compute_tc16p_kernel"
K4Q = "spmdm_compute_tcq_kernel"
K4S = "spmdm_compute_tc16s_kernel"


# ---- helpers ---------------------------------------------------------------------------------------------------------
def to_csc(A, keep=None):
    """CSC arrays (col_ptr[K + 1], row_idx, values) of the entries of A (M x K) where `keep` is set: the CSR arrays of A.T"""
    return to_csr(np.ascontiguousarray(A.T), None if keep is None else np.ascontiguousarray(keep.T))


def run(xs, M, N, K, threads, bf16, route, A, arrays=None, B=None, C0=None, transb="N", transc="N", beta=0):
    """one handle, one slicing pass of A (M x K) through `route`, optionally one multiply.  route: "csc" (A's CSC arrays, or
    `arrays`), "csr" (A's CSR arrays, or `arrays`), "T" (the dense K x M array A.T with transa = 'T') or "N" (A itself).
    Returns (geometry, slices, slice_nnz, C, kernel name)."""
    p = xs.Spmdm(M, N, K, threads)
    bufs = []
    try:
        if route in ("csc", "csr"):
            d = Csr(xs, *(arrays if arrays is not None else (to_csc(A) if route == "csc" else to_csr(A))))
            bufs += [d.rp, d.ci, d.va]
            (p.create_slices_csc if route == "csc" else p.create_slices_csr)(d.rp, d.ci, d.va, d.nnz, bf16)
        else:
            dA = xs.DeviceBuffer.from_numpy(np.ascontiguousarray(A.T) if route == "T" else A)
            bufs.append(dA)
            p.create_slices(dA, route, bf16)
        C, name = None, None
        if B is not None:
            dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
            bufs += [dB, dC]
            p.compute(dB, dC, transb, transc, beta, bf16)
            xs.synchronize()
            C = dC.to_numpy(np.float32, C0.shape)
            name = xs.last_compute_kernel()
        xs.synchronize()
        return pyoracle_geometry(p), p.read_slices(), slice_nnz(xs, p), C, name
    finally:
        for b in bufs:
            b.free()
        p.destroy()


def three_routes_slices(gpu, oracle, M, K, A, bf16, threads, keep=None, N=16):
    """CSC route == dense 'T' route == CSR route (GPU) == oracle with transa = 'T', array by array"""
    g, sl, cnt, _, _ = run(gpu, M, N, K, threads, bf16, "csc", A, to_csc(A, keep))
    gt, slt, cntt, _, _ = run(gpu, M, N, K, threads, bf16, "T", A)
    gr, slr, cntr, _, _ = run(gpu, M, N, K, threads, bf16, "csr", A, to_csr(A, keep))
    assert dict(g) == dict(gt) == dict(gr)
    AT = np.ascontiguousarray(A.T)
    og, osl, _ = oracle_spmdm(oracle, g, AT, np.zeros((K, N), A.dtype), np.zeros((M, N), np.float32), "T", "N", "N", 0.0)
    valid_slices_equal(og, sl, slt)
    valid_slices_equal(og, sl, slr)
    valid_slices_equal(og, sl, osl)
    import pyoracle
    np.testing.assert_array_equal(cnt, cntt)
    np.testing.assert_array_equal(cnt, cntr)
    np.testing.assert_array_equal(cnt, pyoracle.slice_counts(og, osl[0]))
    return g, cnt


def rel(C, OC):
    return float(np.abs(C.astype(np.float64) - OC).max() / np.abs(OC).max())


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
def test_slices_match_dense_t_route_csr_route_and_oracle(gpu, oracle, monkeypatch, M, K, density, dtype, bn, threads):
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_BN", str(bn))
    A = sparse_a(M, K, density, dtype == "bf16", seed=M + K + bn + 1)
    g, cnt = three_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", threads)
    assert g.bn == bn
    assert cnt.sum() > 0
    gpu.check()


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_empty_matrix(gpu, oracle, dtype):
    """nnz = 0 (NULL row_idx / values allowed) gives all-empty slices"""
    M, K = 300, 260
    A = np.zeros((M, K), np.uint16 if dtype == "bf16" else np.float32)
    p = gpu.Spmdm(M, 16, K, 1)
    cp = gpu.DeviceBuffer.from_numpy(np.zeros(K + 1, np.uint32))
    try:
        p.create_slices_csc(cp, None, None, 0, dtype == "bf16")
        gpu.check()
        assert not slice_nnz(gpu, p).any()
    finally:
        cp.free()
        p.destroy()
    three_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", 1)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_full_slice_wraps_the_row_counter(gpu, oracle, dtype):
    """a fully dense 512 x 128 slice: rowidx wraps at 65536 like the reference's u16 counter, slice_nnz holds 65536"""
    M, K = 512, 128
    A = (np.random.default_rng(10).random((M, K)) + 0.5).astype(np.float32)
    A = to_bf16(A) if dtype == "bf16" else A
    g, cnt = three_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", 1, N=48)     # N = bn: the geometry keeps bm = 512
    assert g.bm == 512 and list(cnt) == [65536]


# ---- 2. special values -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_special_values(gpu, oracle, dtype):
    """explicit 0, -0, NaN (vector part and scalar remainder), +-Inf and subnormals as stored CSC entries: the kept set and the
    slices equal the dense 'T' route's"""
    M, K = 200, 260                              # last k-block: 4 columns, all in the scalar remainder
    rng = np.random.default_rng(22)
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
    csc = to_csc(A, keep)
    assert np.array_equal(np.ascontiguousarray(densify(K, M, *csc).T).view(np.uint8), A.view(np.uint8))
    three_routes_slices(gpu, oracle, M, K, A, dtype == "bf16", 1, keep)
    gpu.check()


# ---- 3. C, bit for bit, with the same kernel ---------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tb,tc,beta", [
    ("f32", "N", "N", 0.0), ("f32", "T", "N", 1.0), ("f32", "N", "T", 0.5), ("f32", "T", "T", 1.0),
    ("bf16", "N", "N", 0), ("bf16", "T", "T", 1), ("bf16", "N", "T", 0),
])
def test_cuda_core_product_matches_oracle_and_dense_t_route(gpu, oracle, monkeypatch, dtype, tb, tc, beta):
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    M, N, K = 300, 203, 260
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.08, bf16, seed=5)
    B, C0 = dense_b_c(M, N, K, bf16, 5, tb, tc)
    g, _, _, C, name = run(gpu, M, N, K, 1, bf16, "csc", A, B=B, C0=C0, transb=tb, transc=tc, beta=beta)
    _, _, _, Ct, namet = run(gpu, M, N, K, 1, bf16, "T", A, B=B, C0=C0, transb=tb, transc=tc, beta=beta)
    assert name == namet
    np.testing.assert_array_equal(C.view(np.uint32), Ct.view(np.uint32))
    _, _, OC = oracle_spmdm(oracle, g, np.ascontiguousarray(A.T), B, C0, "T", tb, tc, float(beta))
    np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
    gpu.check()


@pytest.mark.parametrize("dtype,K,sparse,kernel", [
    ("f32", 300, None, K4),
    ("f32", 384, None, K4),       # K % 128 == 0: the sparse routes write no dense image, K4 runs on tcoff
    ("bf16", 384, "0", K4P),
    ("bf16", 384, "1", K4S),
])
def test_tensor_core_kernels_same_bits_as_csr_route(gpu, oracle, monkeypatch, dtype, K, sparse, kernel):
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    if sparse is not None:
        monkeypatch.setenv("LIBXSMM_B200_TC16_SPARSE", sparse)
    M, N = 512, 400
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.05, bf16, seed=K + 1)
    B, C0 = dense_b_c(M, N, K, bf16, 8)
    g, _, _, C, name = run(gpu, M, N, K, 1, bf16, "csc", A, B=B, C0=C0, beta=1)
    _, _, _, Cr, namer = run(gpu, M, N, K, 1, bf16, "csr", A, B=B, C0=C0, beta=1)
    assert name == namer == kernel
    np.testing.assert_array_equal(C.view(np.uint32), Cr.view(np.uint32))
    _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 1.0)
    assert rel(C, OC) <= 1e-5
    gpu.check()


def test_c2_default_dispatch_takes_k4s(gpu, monkeypatch):
    """bf16 4096^3 at 1 %: once the handle knows the density the CSC route runs K4s with the CSR route's bits; the dense 'T' route
    on the same problem writes no structured-sparse words and stays on K4p"""
    monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    monkeypatch.delenv("LIBXSMM_B200_TC16_SPARSE", raising=False)
    M = N = K = 4096
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, 0.01, dtype="bf16", seed=3)
    out = {}
    for route in ("csc", "csr", "T"):
        p = gpu.Spmdm(M, N, K, 1)
        d = Csr(gpu, *(to_csc(A) if route == "csc" else to_csr(A))) if route != "T" else None
        dA = gpu.DeviceBuffer.from_numpy(np.ascontiguousarray(A.T)) if route == "T" else None
        dB, dC = gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer(C0.nbytes)
        for _ in range(3):                       # from the third pass on the density estimate is known and stable
            dC.upload(C0)
            if route == "T":
                p.create_slices(dA, "T", True)
            else:
                (p.create_slices_csc if route == "csc" else p.create_slices_csr)(d.rp, d.ci, d.va, d.nnz, True)
            p.compute(dB, dC, "N", "N", 0, True)
            gpu.synchronize()
        out[route] = (dC.to_numpy(np.float32, C0.shape), gpu.last_compute_kernel())
        d.free() if d is not None else dA.free()
        dB.free(); dC.free()
        p.destroy()
    assert out["csc"][1] == out["csr"][1] == K4S
    assert out["T"][1] == K4P
    np.testing.assert_array_equal(out["csc"][0].view(np.uint32), out["csr"][0].view(np.uint32))
    assert rel(out["csc"][0], out["T"][0].astype(np.float64)) <= 1e-5
    gpu.check()


# ---- 4. state between passes ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("transa", ["N", "T"])
def test_stale_dense_image_is_never_used(gpu, oracle, monkeypatch, transa):
    """a dense fp32 pass of X writes the dense tile image; a CSC pass of Y follows: the multiply must be Y's product"""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    M, N, K = 512, 256, 384
    X = sparse_a(M, K, 0.2, False, seed=11, empty_rows=0)
    Y = sparse_a(M, K, 0.2, False, seed=12, empty_rows=0)
    B, C0 = dense_b_c(M, N, K, False, 13)
    p = gpu.Spmdm(M, N, K, 1)
    dX = gpu.DeviceBuffer.from_numpy(np.ascontiguousarray(X.T) if transa == "T" else X)
    dB, dC = gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer.from_numpy(C0)
    d = Csr(gpu, *to_csc(Y))
    try:
        p.create_slices(dX, transa, False)
        p.compute(dB, dC, "N", "N", 0.0, False)
        gpu.synchronize()
        assert gpu.last_compute_kernel() == K4Q      # reads the image
        dC.upload(C0)
        p.create_slices_csc(d.rp, d.ci, d.va, d.nnz, False)
        p.compute(dB, dC, "N", "N", 0.0, False)
        gpu.synchronize()
        assert gpu.last_compute_kernel() == K4
        _, _, OC = oracle_spmdm(oracle, pyoracle_geometry(p), Y, B, C0, "N", "N", "N", 0.0)
        assert rel(dC.to_numpy(np.float32, C0.shape), OC) <= 1e-5
    finally:
        d.free()
        for b in (dX, dB, dC):
            b.free()
        p.destroy()
    gpu.check()


def test_interleaved_routes_on_one_handle(gpu, oracle, monkeypatch):
    """bf16, K4s whenever the slices carry their structured-sparse words: dense 'N' (K1x writes tcsp), CSC, dense 'T' (no tcsp: the
    words the CSC pass left are stale), CSR, CSC -- each multiply is the product of the matrix just sliced"""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    monkeypatch.setenv("LIBXSMM_B200_TC16_SPARSE", "1")
    M, N, K = 512, 400, 384
    mats = [sparse_a(M, K, 0.03, True, seed=40 + i) for i in range(5)]
    B, C0 = dense_b_c(M, N, K, True, 40)
    p = gpu.Spmdm(M, N, K, 1)
    g = pyoracle_geometry(p)
    dB, dC = gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer.from_numpy(C0)
    try:
        for (route, want), A in zip((("N", K4S), ("csc", K4S), ("T", K4P), ("csr", K4S), ("csc", K4S)), mats):
            bufs = []
            if route in ("N", "T"):
                bufs.append(gpu.DeviceBuffer.from_numpy(np.ascontiguousarray(A.T) if route == "T" else A))
                p.create_slices(bufs[0], route, True)
            else:
                d = Csr(gpu, *(to_csc(A) if route == "csc" else to_csr(A)))
                bufs += [d.rp, d.ci, d.va]
                (p.create_slices_csc if route == "csc" else p.create_slices_csr)(d.rp, d.ci, d.va, d.nnz, True)
            dC.upload(C0)
            p.compute(dB, dC, "N", "N", 0, True)
            gpu.synchronize()
            assert gpu.last_compute_kernel() == want, route
            _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.0)
            assert rel(dC.to_numpy(np.float32, C0.shape), OC) <= 1e-5, route
            for b in bufs:
                b.free()
    finally:
        for b in (dB, dC):
            b.free()
        p.destroy()
    gpu.check()


# ---- 5. graph --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tc_mode", [("f32", "0"), ("bf16", "0"), ("bf16", None)])
def test_graph_replay_with_new_arrays(gpu, oracle, monkeypatch, dtype, tc_mode):
    """CSC slicing + multiply captured once, replayed with new index / value contents in the same buffers (same nnz)"""
    if tc_mode is None:
        monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    else:
        monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", tc_mode)
    xs, L = gpu, gpu.load()
    M, N, K = 512, 400, 384
    bf16 = dtype == "bf16"
    nnz = M * K // 20
    rng = np.random.default_rng(31)
    mats = []
    for i in range(2):
        keep = np.zeros(M * K, bool)
        keep[rng.choice(M * K, nnz, replace=False)] = True
        A = np.where(keep.reshape(M, K), rng.uniform(0.5, 1.5, (M, K)), 0.0).astype(np.float32)
        mats.append(to_bf16(A) if bf16 else A)
    B, C0 = dense_b_c(M, N, K, bf16, 31)
    p = xs.Spmdm(M, N, K, 1)
    g = pyoracle_geometry(p)
    d = Csr(xs, *to_csc(mats[0]))
    dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
    st = xs.Stream()
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    p.create_slices_csc(d.rp, d.ci, d.va, d.nnz, bf16, st)
    p.compute(dB, dC, "N", "N", 0, bf16, st)
    graph = L.libxsmm_b200_graph_end(st.ptr)
    xs.check()
    assert graph
    try:
        for A in mats + mats[:1]:
            d.upload(*to_csc(A))
            dC.upload(C0)
            assert 0 == L.libxsmm_b200_graph_launch(graph, st.ptr)
            st.synchronize()
            C = dC.to_numpy(np.float32, C0.shape)
            _, _, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.0)
            if tc_mode == "0":
                np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
            else:
                assert rel(C, OC) <= 1e-5
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
    cp = xs.DeviceBuffer.from_numpy(np.zeros(K + 1, np.uint32))
    ri, va = xs.DeviceBuffer(64), xs.DeviceBuffer(64)
    stale = xs.libxsmm_spmdm_handle.from_buffer_copy(p.handle)     # becomes an unknown handle once p is destroyed
    other = xs.Spmdm(M, 16, K, 1)
    other.destroy()
    cases = [
        (xs.libxsmm_spmdm_handle(), cp, ri, va, 1, -10),          # never initialised
        (other.handle, cp, ri, va, 1, -10),                       # destroyed: its arena pointer is cleared
        (p.handle, None, ri, va, 1, -90),
        (p.handle, None, None, None, 0, -90),                     # col_ptr is needed even for nnz = 0
        (p.handle, cp, None, va, 1, -90),
        (p.handle, cp, ri, None, 1, -90),
        (p.handle, cp, ri, va, -1, -91),
        (p.handle, cp, ri, va, 1 << 32, -91),
    ]
    try:
        for bf16 in (False, True):
            f = xs.libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream if bf16 else xs.libxsmm_spmdm_createSparseSlice_csc_fp32_stream
            for h, c, r, v, nnz, code in cases:
                xs.clear_error()
                n0 = xs.launch_count()
                f(h, c, r, v, nnz, p.slices)
                assert xs.last_error()[0] == code, (nnz, code, xs.last_error())
                assert xs.launch_count() == n0
        p_base = p.handle.base_ptr_scratch_A
        p.destroy()
        assert p_base and stale.base_ptr_scratch_A == p_base
        xs.clear_error()
        n0 = xs.launch_count()
        xs.libxsmm_spmdm_createSparseSlice_csc_fp32_stream(stale, cp, ri, va, 1, None)
        assert xs.last_error()[0] == -11 and xs.launch_count() == n0
    finally:
        xs.clear_error()
        for b in (cp, ri, va):
            b.free()
        p.destroy()


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_malformed_arrays_stay_in_bounds(gpu, oracle, monkeypatch, dtype):
    """rows >= M, duplicated and unsorted rows, col_ptr past nnz and not monotone: the result is unspecified, but the pass and
    the multiply stay inside their arrays (a guard-banded C keeps its guards, no slice holds more than bm x bk entries) and the
    next well-formed pass is exact"""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    xs = gpu
    M, N, K = 300, 200, 384
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.2, bf16, seed=14)
    col_ptr, row_idx, values = to_csc(A)
    nnz = len(row_idx)
    rng = np.random.default_rng(14)
    bad_rows = row_idx.copy()
    bad_rows[rng.choice(nnz, 200, replace=False)] = rng.integers(M, M + 70000, 200)          # rows >= M
    for c in range(0, K, 5):                                                                # unsorted / duplicated columns
        lo, hi = int(col_ptr[c]), int(col_ptr[c + 1])
        if hi - lo > 2:
            bad_rows[lo:hi] = bad_rows[lo:hi][::-1] if c % 2 else bad_rows[lo]
    bad_cp = col_ptr.copy()
    bad_cp[5] = nnz + 1000                                                                  # past nnz, then not monotone
    bad_cp[200] = 3
    bad_cp[-1] = nnz + 7
    B, C0 = dense_b_c(M, N, K, bf16, 14)
    guard = 4096
    sentinel = np.float32(-12345.5)
    p = xs.Spmdm(M, N, K, 1)
    g = pyoracle_geometry(p)
    d = Csr(xs, bad_cp, bad_rows, values)
    dB = xs.DeviceBuffer.from_numpy(B)
    dCg = xs.DeviceBuffer.from_numpy(np.full(C0.size + 2 * guard, sentinel, np.float32))
    try:
        dCg.upload(C0, guard * 4)
        p.create_slices_csc(d.rp, d.ci, d.va, d.nnz, bf16)
        p.compute(dB, dCg.ptr + guard * 4, "N", "N", 1, bf16)
        xs.synchronize()
        out = dCg.to_numpy(np.float32, (C0.size + 2 * guard,))
        assert np.all(out[:guard] == sentinel) and np.all(out[-guard:] == sentinel)
        cnt = slice_nnz(xs, p)
        assert int(cnt.max()) <= g.bm * g.bk
        d.upload(col_ptr, row_idx, values)                          # well-formed again, same handle
        dCg.upload(C0, guard * 4)
        p.create_slices_csc(d.rp, d.ci, d.va, d.nnz, bf16)
        p.compute(dB, dCg.ptr + guard * 4, "N", "N", 1, bf16)
        xs.synchronize()
        out = dCg.to_numpy(np.float32, (C0.size + 2 * guard,))
        og, osl, OC = oracle_spmdm(oracle, g, np.ascontiguousarray(A.T), B, C0, "T", "N", "N", 1.0)
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
def test_one_launch_per_csc_slicing_call(gpu, dtype):
    M, K = 1000, 640
    bf16 = dtype == "bf16"
    A = sparse_a(M, K, 0.05, bf16, seed=15)
    p = gpu.Spmdm(M, 64, K, 1)
    d = Csr(gpu, *to_csc(A))
    st = gpu.Stream()
    try:
        for _ in range(2):
            n0 = gpu.launch_count()
            p.create_slices_csc(d.rp, d.ci, d.va, d.nnz, bf16, st)
            assert gpu.launch_count() - n0 == 1
        st.synchronize()
    finally:
        d.free()
        st.destroy()
        p.destroy()
    gpu.check()
