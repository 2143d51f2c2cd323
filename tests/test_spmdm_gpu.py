"""GPU parity of libxsmm_spmdm (through the C ABI) against the CPU oracle.

Bars (BASELINE.json north_star):
  * slices: row pointers, column indices, values and nnz BIT-EXACT;
  * C: within 1e-5 (fp32 inputs) / 1e-2 (bf16 inputs) relative -- stated below as RTOL_*.  The kernels
    keep the reference's rounding sequence, so the tests additionally require bit equality and report
    the tolerance figure only as the contractual fallback.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def cuda_core_path(monkeypatch):
    """These tests assert BIT equality with the oracle, which holds for the CUDA-core kernels (they keep the
    reference's rounding sequence).  The tensor-core branch that takes over dense fp32 problems is covered,
    against the relative-error contract, by tests/test_spmdm_tc_gpu.py."""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")


RTOL_F32 = 1e-5
RTOL_BF16 = 1e-2


def rel_err(got, want):
    scale = max(float(np.abs(want).max()), 1e-30)
    return float(np.abs(got.astype(np.float64) - want.astype(np.float64)).max()) / scale


def valid_slices_equal(g, got, want):
    """compare rowidx[0..nrows] and colidx/values[0..nnz) of every slice."""
    import pyoracle
    ro_g, co_g, va_g = got
    ro_w, co_w, va_w = want
    cnt = pyoracle.slice_counts(g, ro_w)
    for s in range(g.nslices):
        mb = s % g.mb
        nrows = min(g.bm, g.m - mb * g.bm)
        np.testing.assert_array_equal(ro_g[s, :nrows + 1], ro_w[s, :nrows + 1], err_msg="rowidx slice %d" % s)
        n = int(min(cnt[s], g.cap))
        np.testing.assert_array_equal(co_g[s, :n], co_w[s, :n], err_msg="colidx slice %d" % s)
        np.testing.assert_array_equal(va_g[s, :n].view(np.uint32), va_w[s, :n].view(np.uint32), err_msg="values slice %d" % s)
    return int(cnt.sum())


def gpu_spmdm(xs, A, B, C0, M, N, K, transa="N", transb="N", transc="N", beta=0.0, bf16=False, max_threads=1, a_offset=0):
    """slice + compute on device buffers through the stream entries; returns (geometry, slices, C).
    a_offset: A is placed that many bytes past the start of its (256-byte aligned) device buffer."""
    import pyoracle
    p = xs.Spmdm(M, N, K, max_threads)
    try:
        A = np.ascontiguousarray(A)
        dA = xs.DeviceBuffer(max(A.nbytes + a_offset, 1))
        if A.nbytes:
            dA.upload(A, a_offset)
        dB = xs.DeviceBuffer.from_numpy(B)
        dC = xs.DeviceBuffer.from_numpy(C0)
        p.create_slices(dA.ptr + a_offset, transa, bf16)
        p.compute(dB, dC, transb, transc, beta, bf16)
        xs.synchronize()
        sl = p.read_slices()
        C = dC.to_numpy(np.float32, C0.shape)
        geo = p.geometry
        g = pyoracle.Geometry(geo)
        g["scratch"] = 0
        for d in (dA, dB, dC):
            d.free()
        return g, sl, C
    finally:
        p.destroy()


def oracle_spmdm(oracle, g, A, B, C0, transa, transb, transc, beta):
    og = oracle.geometry(g.m, g.n, g.k, 1, bn=g.bn)
    og.update(bm=g.bm, mb=g.mb)          # bm depends on max_threads; take the library's and check it separately
    sl = oracle.slices(og, A, transa)
    C = C0.copy()
    oracle.compute(og, sl, B, C, transb, transc, beta)
    return og, sl, C


CASES = [
    # M, N, K, density, dtype, ta, tb, tc, beta, max_threads
    (512, 384, 640, 0.10, "f32", "N", "N", "N", 0.0, 1),
    (512, 384, 640, 0.10, "f32", "N", "N", "N", 1.0, 1),
    (512, 384, 640, 0.10, "f32", "N", "N", "N", 0.5, 1),
    (300, 200, 260, 0.15, "f32", "N", "N", "N", 0.0, 1),      # ragged in M, N (narrow last block), K
    (300, 200, 260, 0.15, "f32", "N", "N", "N", 1.0, 4),
    (300, 203, 260, 0.15, "f32", "N", "N", "N", 0.75, 1),     # scalar tail columns as well
    (260, 200, 300, 0.50, "f32", "T", "N", "T", 0.0, 1),      # "weight update" variant of the sample
    (260, 200, 300, 0.50, "f32", "N", "T", "N", 0.0, 1),      # "backprop" variant of the sample
    (260, 203, 300, 0.50, "f32", "T", "T", "T", 1.0, 1),
    (1024, 512, 512, 0.50, "f32", "N", "N", "N", 0.0, 8),
    (2048, 256, 256, 0.10, "f32", "N", "N", "N", 0.0, 56),    # bm = 245 after the balance loop
    (64, 48, 128, 0.30, "f32", "N", "N", "N", 0.0, 1),
    (1, 16, 1, 1.00, "f32", "N", "N", "N", 0.0, 1),
    (33, 7, 129, 0.40, "f32", "N", "N", "N", 1.0, 1),
    (512, 512, 512, 0.01, "bf16", "N", "N", "N", 0, 1),
    (512, 512, 512, 0.10, "bf16", "N", "N", "N", 1, 1),       # beta bits == integer 1 -> beta 1 (quirk Q2)
    (300, 203, 256, 0.10, "bf16", "N", "N", "N", 0, 1),
    (256, 200, 384, 0.20, "bf16", "T", "N", "T", 0, 1),
    (256, 200, 384, 0.20, "bf16", "N", "T", "N", 0, 1),
    (4096, 320, 256, 0.01, "bf16", "N", "N", "N", 0, 8),
]


@pytest.mark.parametrize("M,N,K,density,dtype,ta,tb,tc,beta,threads", CASES)
def test_spmdm_matches_oracle(gpu, oracle, M, N, K, density, dtype, ta, tb, tc, beta, threads):
    w = gpu.workloads
    A, B, C0 = w.spmdm_inputs(M, N, K, density, dtype=dtype, seed=M + N + K, transa=ta, transb=tb, transc=tc)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, beta, dtype == "bf16", threads)
    # geometry is the reference's arithmetic (src/libxsmm_spmdm.c:552-608)
    og_full = oracle.geometry(M, N, K, threads, bn=g.bn)
    assert {k: g[k] for k in ("bm", "bn", "bk", "mb", "nb", "kb")} == {k: og_full[k] for k in ("bm", "bn", "bk", "mb", "nb", "kb")}
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, ta, tb, tc, float(beta))
    nnz = valid_slices_equal(og, sl, osl)
    assert nnz > 0 or density == 0
    err = rel_err(C, OC)
    assert err <= (RTOL_BF16 if dtype == "bf16" else RTOL_F32), "relative error %g" % err
    np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32), err_msg="same rounding sequence expected")
    gpu.check()


@pytest.mark.parametrize("dtype", ["bf16", "f32"])
@pytest.mark.parametrize("M,N,K,density", [(512, 768, 512, 0.02), (1024, 512, 384, 0.30), (256, 1100, 640, 0.004)])
def test_mixed_sign_denormal_overflow(gpu, oracle, dtype, M, N, K, density):
    """Inputs the uniform [0,1) workloads never produce: both signs (cancellation), denormal A and B entries, products
    that underflow, sums that overflow to +-Inf.  The order-preserving kernels (K2s uses the mixed-precision
    fma.rn.f32.bf16 for bf16 slices) must still reproduce the reference's fmaf chain bit for bit."""
    w = gpu.workloads
    rng = np.random.default_rng(M + N + K + (1 if dtype == "bf16" else 0))
    A = np.where(rng.random((M, K)) < density, rng.uniform(-1.0, 1.0, (M, K)), 0.0).astype(np.float32)
    B = rng.uniform(-1.0, 1.0, (K, N)).astype(np.float32)
    C0 = rng.uniform(-1.0, 1.0, (M, N)).astype(np.float32)
    nzr, nzc = np.nonzero(A)
    assert len(nzr) > 64
    pick = rng.permutation(len(nzr))
    for j, v in zip(pick[:16], [1e-40, -3e-39, 9.2e-41, 1e-38] * 4):          # denormal (and near-denormal) operator entries
        A[nzr[j], nzc[j]] = v
    for j in pick[16:24]:                                                     # huge entries: partial sums overflow
        A[nzr[j], nzc[j]] = 3e38
    B[rng.integers(0, K, 64), rng.integers(0, N, 64)] = np.float32(1e-39)     # denormal B entries
    B[nzc[pick[16]], :] = np.float32(2.5)                                      # 3e38 * 2.5 -> Inf in that output row
    B[rng.integers(0, K, 64), rng.integers(0, N, 64)] = np.float32(1e-30)     # tiny x tiny products underflow to denormals / 0
    if dtype == "bf16":
        A = w.to_bf16_bits(A); B = w.to_bf16_bits(B)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=1.0 if dtype == "f32" else 0, bf16=(dtype == "bf16"))
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 1.0 if dtype == "f32" else 0.0)
    valid_slices_equal(og, sl, osl)
    assert np.isinf(OC).any() and np.isfinite(OC).any()
    same = (C.view(np.uint32) == OC.view(np.uint32)) | (np.isnan(C) & np.isnan(OC))
    assert same.all(), "%d elements differ from the reference's rounding sequence" % int((~same).sum())
    gpu.check()


def test_special_values_in_a(gpu, oracle):
    """NaN / -0.0 / Inf / denormal handling of the slicing (reference quirk Q3): the vector part of the
    reference uses an ordered compare (drops NaN), the scalar remainder keeps NaN."""
    M, N, K = 40, 48, 133            # 133 = 128 + 5: second k-block is all "scalar remainder" columns
    rng = np.random.default_rng(7)
    A = np.where(rng.random((M, K)) < 0.3, rng.random((M, K)), 0).astype(np.float32)
    A[0, 0] = np.nan; A[1, 5] = -0.0; A[2, 9] = np.inf; A[3, 11] = 1e-45; A[4, 127] = -np.inf
    A[5, 130] = np.nan; A[6, 131] = -0.0; A[7, 132] = np.inf
    B = rng.random((K, N)).astype(np.float32)
    C0 = rng.random((M, N)).astype(np.float32)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.0)
    valid_slices_equal(og, sl, osl)
    # a kept NaN poisons its output row on both sides; NaN payload bits are implementation defined
    assert np.isnan(OC[5]).all() and np.isnan(C[5]).all()
    ok = ~np.isnan(OC)
    np.testing.assert_array_equal(np.isnan(C), np.isnan(OC))
    np.testing.assert_array_equal(C[ok].view(np.uint32), OC[ok].view(np.uint32))


@pytest.mark.parametrize("wide", ["2", "0"])
def test_special_values_bf16_wide_slicing(gpu, oracle, wide):
    """bf16 bit patterns through the slicing kernels for complete blocks: +-0, NaN with either sign, +-Inf, denormals,
    the largest finite value, dense and empty lanes and rows -- kept iff ordered-nonzero like the reference's vector
    loops (quirk Q3).  Slices bit for bit against the oracle.  wide = 16-byte words per lane of the kernel that slices A:
    "2" = the wide kernel (16-byte aligned rows), "0" = the generic kernel, reached with A 8 bytes past a 16-byte
    boundary (it still takes the complete-block form and 8-byte loads)."""
    M, N, K = 600, 48, 256           # two complete k-blocks, row pitch 512 B; two row blocks (512 + 88 rows)
    rng = np.random.default_rng(11)
    bits = np.where(rng.random((M, K)) < 0.05, rng.integers(1, 0x7F80, (M, K)), 0).astype(np.uint16)
    bits[rng.random((M, K)) < 0.02] |= 0x8000                      # negative values and -0.0
    special = np.array([0x0000, 0x8000, 0x7FC0, 0xFFC1, 0x7F81, 0x7F80, 0xFF80, 0x0001, 0x8001, 0x7F7F, 0xFF7F, 0x0080], np.uint16)
    idx = rng.integers(0, M * K, 4000)
    bits.reshape(-1)[idx] = special[rng.integers(0, len(special), len(idx))]
    bits[3, :] = 0x3F80              # a completely dense row
    bits[4, 16:32] = 0x4000          # one completely dense lane (two-word kernel) next to empty ones
    bits[5, :] = 0                   # an empty row
    bits[511, 120:128] = 0xC000      # last lane of the last row of the first block
    A = np.ascontiguousarray(bits)
    B = gpu.workloads.to_bf16_bits(rng.random((K, N)).astype(np.float32))
    C0 = rng.random((M, N)).astype(np.float32)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=0, bf16=True, a_offset=0 if "2" == wide else 8)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.0)
    nnz = valid_slices_equal(og, sl, osl)
    keep = ((bits & 0x7FFF) >= 1) & ((bits & 0x7FFF) <= 0x7F80)
    assert nnz == int(keep.sum())
    ok = ~np.isnan(OC)
    np.testing.assert_array_equal(np.isnan(C), np.isnan(OC))
    np.testing.assert_array_equal(C[ok].view(np.uint32), OC[ok].view(np.uint32))
    gpu.check()


def test_all_zero_and_dense_wrap(gpu, oracle):
    """empty A; and a fully dense 512 x 128 slice whose u16 counter wraps to 0 like the reference's
    (quirk Q4, template :72): row pointers are compared modulo 2^16."""
    M, N, K = 512, 96, 128            # N a multiple of bn: the balance loop keeps bm = 512
    B = np.random.default_rng(1).random((K, N)).astype(np.float32)
    C0 = np.ones((M, N), np.float32)
    A = np.zeros((M, K), np.float32)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K)
    assert not sl[0].any()
    assert not C.any()
    A = (np.random.default_rng(2).random((M, K)) + 0.5).astype(np.float32)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=1.0)
    og = oracle.geometry(M, N, K, 1, bn=g.bn)
    assert og.bm == 512
    osl = oracle.slices(og, A)
    np.testing.assert_array_equal(sl[0][0], osl[0][0])      # includes rowidx[512] == 0
    assert sl[0][0, 512] == 0


def test_legacy_block_entries_host_pointers(gpu, oracle):
    """The 8 reference entry points driven exactly like samples/spmdm/spmdm.c:88-111, HOST matrices."""
    xs = gpu
    M, N, K = 300, 203, 260
    A, B, C0 = xs.workloads.spmdm_inputs(M, N, K, 0.2, seed=11)
    h, s = xs.libxsmm_spmdm_init(M, N, K, 3)
    try:
        nthreads = 3
        for i in range(xs.libxsmm_spmdm_get_num_createSparseSlice_blocks(h)):
            xs.libxsmm_spmdm_createSparseSlice_fp32_thread(h, "N", A, s, i, i % nthreads, nthreads)
        C = C0.copy()
        for i in range(xs.libxsmm_spmdm_get_num_compute_blocks(h)):
            xs.libxsmm_spmdm_compute_fp32_thread(h, "N", "N", 1.0, s, B, "N", 0.5, C, i, i % nthreads, nthreads)
        xs.check()
        import pyoracle
        g = pyoracle.Geometry(dict(m=h.m, n=h.n, k=h.k, bm=h.bm, bn=h.bn, bk=h.bk, mb=h.mb, nb=h.nb, kb=h.kb))
        og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.5)
        np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
    finally:
        xs.libxsmm_spmdm_destroy(h)
    assert not h.base_ptr_scratch_A


def test_legacy_block_entries_bf16_transposed(gpu, oracle):
    xs = gpu
    M, N, K = 256, 200, 384
    A, B, C0 = xs.workloads.spmdm_inputs(M, N, K, 0.2, dtype="bf16", seed=12, transa="T", transc="T")
    h, s = xs.libxsmm_spmdm_init(M, N, K, 2)
    try:
        for i in range(xs.libxsmm_spmdm_get_num_createSparseSlice_blocks(h)):
            xs.libxsmm_spmdm_createSparseSlice_bfloat16_thread(h, "T", A, s, i, i % 2, 2)
        C = C0.copy()
        for i in range(xs.libxsmm_spmdm_get_num_compute_blocks(h)):
            xs.libxsmm_spmdm_compute_bfloat16_thread(h, "T", "N", 0x3F80, s, B, "T", 0, C, i, i % 2, 2)
        xs.check()
        import pyoracle
        g = pyoracle.Geometry(dict(m=h.m, n=h.n, k=h.k, bm=h.bm, bn=h.bn, bk=h.bk, mb=h.mb, nb=h.nb, kb=h.kb))
        og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "T", "N", "T", 0.0)
        np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
    finally:
        xs.libxsmm_spmdm_destroy(h)


@pytest.mark.parametrize("shape", [(384, 1000, 512), (2048, 1100, 256)])
@pytest.mark.parametrize("dtype,ta,tb,tc,beta", [("f32", "N", "N", "N", 0.0), ("f32", "T", "N", "T", 1.0),
                                                  ("f32", "N", "T", "N", 0.5), ("bf16", "N", "N", "N", 0), ("bf16", "T", "T", "T", 1)])
def test_exec_host(gpu, oracle, shape, dtype, ta, tb, tc, beta):
    """the whole-multiply host entry: uploads, slicing, compute and downloads pipelined over row blocks x column
    panels on three streams (the second shape has 8 row blocks and 5 panels, the last one ragged)."""
    xs = gpu
    M, N, K = shape
    A, B, C0 = xs.workloads.spmdm_inputs(M, N, K, 0.1, dtype=dtype, seed=5, transa=ta, transb=tb, transc=tc)
    h, s = xs.libxsmm_spmdm_init(M, N, K, 1)
    try:
        dt = xs.LIBXSMM_SPMDM_DATATYPE_BFLOAT16 if dtype == "bf16" else xs.LIBXSMM_SPMDM_DATATYPE_F32
        import pyoracle
        g = pyoracle.Geometry(dict(m=h.m, n=h.n, k=h.k, bm=h.bm, bn=h.bn, bk=h.bk, mb=h.mb, nb=h.nb, kb=h.kb))
        og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, ta, tb, tc, float(beta))
        for rep in range(2):      # second call: the density hint of the first one is in effect
            C = C0.copy()
            xs.libxsmm_spmdm_exec_host(h, s, dt, ta, tb, tc, A, B, beta, C)
            xs.check()
            np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
    finally:
        xs.libxsmm_spmdm_destroy(h)


FULL = [
    ("C1", 2048, 2048, 2048, 0.10, "f32", "N", "N", "N"),
    ("C2", 4096, 4096, 4096, 0.01, "bf16", "N", "N", "N"),
    ("C4-NNN", 2048, 2048, 2048, 0.50, "f32", "N", "N", "N"),
    ("C4-TNT", 2048, 2048, 2048, 0.50, "f32", "T", "N", "T"),
    ("C4-NTN", 2048, 2048, 2048, 0.50, "f32", "N", "T", "N"),
]


@pytest.mark.parametrize("name,M,N,K,density,dtype,ta,tb,tc", FULL)
def test_full_size_properties(gpu, oracle, name, M, N, K, density, dtype, ta, tb, tc):
    """BASELINE.json sizes: slices against the oracle (cheap), C through size-independent properties --
    (1) B = identity reproduces A exactly (one fma(a, 1, 0) per kept element; -0.0 and NaN are dropped),
    (2) the column checksum C.1 equals A.(B.1) computed in float64, (3) a random sample of rows equals
    the oracle's in-order fma chain bit for bit (full blocks only)."""
    w = gpu.workloads
    bf16 = dtype == "bf16"
    A, B, C0 = w.spmdm_inputs(M, N, K, density, dtype=dtype, seed=1, transa=ta, transb=tb, transc=tc)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, 0 if bf16 else 0.0, bf16, 1)
    og = oracle.geometry(M, N, K, 1, bn=g.bn)
    osl = oracle.slices(og, A, ta)
    nnz = valid_slices_equal(og, sl, osl)
    Af = w.from_bf16_bits(A) if bf16 else A
    Bf = w.from_bf16_bits(B) if bf16 else B
    Am = Af.T if ta == "T" else Af          # M x K
    Bm = Bf.T if tb == "T" else Bf          # K x N
    Cm = C.T if tc == "T" else C            # M x N
    assert nnz == int(np.count_nonzero(Am))
    # (2) checksum
    want = Am.astype(np.float64) @ Bm.astype(np.float64).sum(axis=1)
    got = Cm.astype(np.float64).sum(axis=1)
    assert np.abs(got - want).max() <= (RTOL_BF16 if bf16 else RTOL_F32) * np.abs(want).max()
    # (3) sampled rows, in-order fma chain (N is a multiple of bn? no: 2048 % 48 != 0 -> restrict to full blocks)
    n_full = (N // g.bn) * g.bn
    rows = np.random.default_rng(3).choice(M, 6, replace=False)
    for r in rows:
        ks = np.nonzero(Am[r])[0]
        acc = np.zeros(n_full, np.float32)
        a64 = Am[r, ks].astype(np.float64)
        for a, k in zip(a64, ks):   # fp32 fma emulated exactly: product of two fp32 is exact in fp64, one rounding of (p + acc)
            acc = (a * Bm[k, :n_full].astype(np.float64) + acc.astype(np.float64)).astype(np.float32)
        got_r = Cm[r, :n_full]
        # double rounding (fp64 then fp32) can differ from a true fma in rare ties: allow 1 ulp on < 0.1 % entries
        diff = np.abs(got_r.view(np.int32).astype(np.int64) - acc.view(np.int32).astype(np.int64))
        assert diff.max() <= 1 and (diff > 0).mean() < 1e-3, (name, r, diff.max(), (diff > 0).mean())
    # (1) identity
    eye = np.eye(K, N, dtype=np.float32)
    Bi = w.to_bf16_bits(eye) if bf16 else eye
    if tb == "T":
        Bi = np.ascontiguousarray((w.from_bf16_bits(Bi) if bf16 else Bi).T)
        Bi = w.to_bf16_bits(Bi) if bf16 else Bi
    _, _, Ci = gpu_spmdm(gpu, A, Bi, C0, M, N, K, ta, tb, tc, 0 if bf16 else 0.0, bf16, 1)
    Cim = Ci.T if tc == "T" else Ci
    np.testing.assert_array_equal(Cim[:, :min(K, N)], Am[:, :min(K, N)] + np.float32(0))
    gpu.check()


@pytest.mark.parametrize("name,M,N,K,density,dtype,ta,tb,tc", FULL[:2])
def test_full_size_vs_oracle(gpu, oracle, name, M, N, K, density, dtype, ta, tb, tc):
    """C1 and C2 at full size against the oracle, every output element."""
    w = gpu.workloads
    bf16 = dtype == "bf16"
    A, B, C0 = w.spmdm_inputs(M, N, K, density, dtype=dtype, seed=2, transa=ta, transb=tb, transc=tc)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, 0 if bf16 else 0.0, bf16, 1)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, ta, tb, tc, 0.0)
    valid_slices_equal(og, sl, osl)
    err = rel_err(C, OC)
    assert err <= (RTOL_BF16 if bf16 else RTOL_F32)
    np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))
