"""CSR "A sparse" x dense SoA kernels (SURVEY.md section 8f-1; reference libxsmm_create_xcsr_soa, caller
samples/edge/asparse_srsoa.c).  The fixture tests/golden/csr_soa.npz holds outputs of the compiled reference on real EDGE
operators (tests/golden/make_soa_golden.py).  CPU: the oracle's restatement against the fixture and against the compiled
reference where it is present.  GPU: the batched product entry against both, bit for bit.

To stay small the fixture holds every third element of each reference output (row-major) and none of the dense inputs: those
are drawn again from the generator's seeded stream (soa_inputs)."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def soa_inputs(d):
    """the dense operands of every case, drawn in the order tests/golden/make_soa_golden.py draws them from default_rng(31)"""
    rng = np.random.default_rng(31)
    rng.uniform(-1, 1, (12, 12)); rng.random((20, 28)); rng.uniform(-1, 1, (20, 28))       # its two synthetic A operators
    out = {}
    for group, first in (("names", "B"), ("bnames", "A"), ("cnames", "A")):
        if group == "cnames":
            rng.random((24, 30)); rng.uniform(-1, 1, (24, 30))                               # its synthetic CSC operator
        for key in [str(n) for n in d[group]]:
            dt = np.float64 if key.endswith("_d") else np.float32
            M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
            if key.startswith("csc_synthetic_unsorted"):                                      # the row indices it shuffled
                cp = d[key + "_colptr"]
                for n in range(N):
                    rng.shuffle(list(range(int(cp[n + 1] - cp[n]))))
            out[key + "_" + first] = rng.uniform(-1, 1, (E, K, N, soa) if first == "B" else (E, M, K, soa)).astype(dt)
            out[key + "_C0"] = rng.uniform(-1, 1, (E, M, N, soa)).astype(dt)
            probe = np.concatenate([out[key + "_" + first].ravel()[:4], out[key + "_C0"].ravel()[:4]]).astype(np.float64)
            assert np.array_equal(probe, d[key + "_probe"]), "%s: numpy's random stream differs from the one the fixture was made with" % key
    return out


@pytest.fixture(scope="module")
def cases():
    with np.load(os.path.join(ROOT, "tests", "golden", "csr_soa.npz")) as z:
        d = dict(z)
    d.update(soa_inputs(d))
    return d, [str(n) for n in d["names"]]


def bits(x):
    return x.view(np.uint64 if x.dtype == np.float64 else np.uint32)


def matches_reference(C, d, key, beta):
    return np.array_equal(bits(C).ravel()[::3], bits(d[key + "_out%d" % int(beta)]))


def test_oracle_matches_reference_outputs(oracle, cases):
    d, names = cases
    assert len(names) >= 10
    for key in names:
        M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
        for beta in (0.0, 1.0):
            C = d[key + "_C0"].copy()
            oracle.csr_soa_execute(d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"], d[key + "_B"], C, N, beta=beta)
            assert matches_reference(C, d, key, beta), "%s beta=%g" % (key, beta)


def test_oracle_matches_compiled_reference(oracle, ref):
    """ragged pitches (ldb, ldc > N), rows without nonzeros untouched"""
    rng = np.random.default_rng(3)
    for dt in (np.float64, np.float32):
        soa = ref.soa_width(dt)
        for (M, K, N, ld, dens, beta) in ((35, 35, 9, 9, 0.1, 0.0), (20, 35, 7, 11, 0.3, 1.0), (10, 10, 30, 32, 1.0, 1.0), (56, 20, 3, 5, 0.2, 1.0)):
            a = np.where(rng.random((M, K)) < dens, rng.uniform(-1, 1, (M, K)), 0).astype(dt)
            if dens < 1.0:
                a[M // 2, :] = 0
            rp, ci, va = [0], [], []
            for i in range(M):
                nz = np.nonzero(a[i])[0]
                ci += list(nz); va += list(a[i, nz]); rp.append(len(ci))
            rp, ci, va = np.array(rp, np.uint32), np.array(ci, np.uint32), np.array(va, dt)
            B = rng.uniform(-1, 1, (2, K, ld, soa)).astype(dt); C0 = rng.uniform(-1, 1, (2, M, ld, soa)).astype(dt)
            C = C0.copy(); ref.csr_soa(rp, ci, va, B, C, N, beta)
            OC = C0.copy(); oracle.csr_soa_execute(rp, ci, va, B, OC, N, beta=beta)
            assert np.array_equal(bits(C), bits(OC)), (dt.__name__, M, K, N, ld, dens, beta)
            assert np.array_equal(bits(C[:, :, N:]), bits(C0[:, :, N:]))          # columns past N untouched


def test_oracle_matches_reference_outputs_b_sparse(oracle, cases):
    d, _ = cases
    bnames = [str(n) for n in d["bnames"]]
    assert len(bnames) >= 8
    for key in bnames:
        M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
        for beta in (0.0, 1.0):
            C = d[key + "_C0"].copy()
            oracle.csr_soa_bsparse_execute(d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"], d[key + "_A"], C, N, beta=beta)
            assert matches_reference(C, d, key, beta), "%s beta=%g" % (key, beta)


def test_oracle_matches_compiled_reference_b_sparse(oracle, ref):
    """pitches lda > K, ldc > N; an all-zero column (still written: beta C or 0) and an all-zero row of B"""
    rng = np.random.default_rng(5)
    for dt in (np.float64, np.float32):
        soa = ref.soa_width(dt)
        for (M, K, N, lda, ldc, dens, beta) in ((9, 35, 35, 35, 35, 0.2, 0.0), (9, 56, 35, 60, 40, 0.1, 1.0), (4, 20, 28, 24, 28, 0.5, 0.0), (5, 10, 10, 10, 12, 1.0, 1.0)):
            b = np.where(rng.random((K, N)) < dens, rng.uniform(-1, 1, (K, N)), 0).astype(dt)
            b[:, 3] = 0; b[2, :] = 0
            rp, ci, va = [0], [], []
            for i in range(K):
                nz = np.nonzero(b[i])[0]
                ci += list(nz); va += list(b[i, nz]); rp.append(len(ci))
            rp, ci, va = np.array(rp, np.uint32), np.array(ci, np.uint32), np.array(va, dt)
            A = rng.uniform(-1, 1, (2, M, lda, soa)).astype(dt); C0 = rng.uniform(-1, 1, (2, M, ldc, soa)).astype(dt)
            C = C0.copy(); ref.csr_soa_bsparse(rp, ci, va, A, C, N, beta)
            OC = C0.copy(); oracle.csr_soa_bsparse_execute(rp, ci, va, A, OC, N, beta=beta)
            assert np.array_equal(bits(C), bits(OC)), (dt.__name__, M, K, N, dens, beta)
            if beta == 0.0:
                assert not C[:, :, 3].any()
            assert np.array_equal(bits(C[:, :, N:]), bits(C0[:, :, N:]))


def test_oracle_matches_reference_outputs_csc(oracle, cases):
    """libxsmm_create_xcsc_soa (B sparse in CSC): stored outputs of the compiled reference, incl. unsorted columns."""
    d, _ = cases
    for key in [str(n) for n in d["cnames"]]:
        M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
        for beta in (0.0, 1.0):
            C = d[key + "_C0"].copy()
            oracle.csc_soa_execute(d[key + "_colptr"], d[key + "_rowidx"], d[key + "_values"], d[key + "_A"], C, N, beta=beta)
            assert matches_reference(C, d, key, beta), "%s beta=%g" % (key, beta)


def test_oracle_matches_compiled_reference_csc(oracle, ref):
    rng = np.random.default_rng(12)
    for dt in (np.float64, np.float32):
        soa = ref.soa_width(dt)
        for K, N, dens, trail in ((20, 30, 0.2, 0), (35, 35, 0.1, 6), (10, 40, 0.5, 0)):
            b = np.where(rng.random((K, N)) < dens, rng.uniform(-1, 1, (K, N)), 0).astype(dt)
            b[:, 3] = 0
            if trail:
                b[:, N - trail:] = 0
            cp, ri, va = [0], [], []
            for n in range(N):
                ks = list(np.nonzero(b[:, n])[0]); rng.shuffle(ks)
                ri += ks; va += [b[k, n] for k in ks]; cp.append(len(ri))
            for beta in (0.0, 1.0):
                A = rng.uniform(-1, 1, (2, 9, K, soa)).astype(dt); C0 = rng.uniform(-1, 1, (2, 9, N + 2, soa)).astype(dt)
                C = C0.copy(); ref.csc_soa(cp, ri, np.array(va, dt), A, C, N, beta)
                OC = C0.copy(); oracle.csc_soa_execute(cp, ri, np.array(va, dt), A, OC, N, beta=beta)
                assert np.array_equal(bits(C), bits(OC))
                assert np.array_equal(bits(C[:, :, N:]), bits(C0[:, :, N:]))


@pytest.mark.gpu
def test_gpu_csc_matches_reference_and_oracle(gpu, oracle, cases):
    d, _ = cases
    for key in [str(n) for n in d["cnames"]]:
        M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
        for beta in (0.0, 1.0):
            op = gpu.CsrSoa(M, N, K, d[key + "_colptr"], d[key + "_rowidx"], d[key + "_values"], soa, beta=beta, sparse="B", fmt="csc")
            assert op.is_baked, key
            dA, dC = gpu.DeviceBuffer.from_numpy(d[key + "_A"]), gpu.DeviceBuffer.from_numpy(d[key + "_C0"])
            op.execute(dA, dC, E)
            gpu.synchronize()
            C = dC.to_numpy(d[key + "_C0"].dtype, d[key + "_C0"].shape)
            dA.free(); dC.free(); op.destroy()
            assert matches_reference(C, d, key, beta), "%s beta=%g" % (key, beta)
            want = d[key + "_C0"].copy()
            oracle.csc_soa_execute(d[key + "_colptr"], d[key + "_rowidx"], d[key + "_values"], d[key + "_A"], want, N, beta=beta)
            assert np.array_equal(bits(C), bits(want)), "%s beta=%g" % (key, beta)
    # duplicates inside a column (the first entry with a row index wins), rows >= K, padded pitches and strides: against the oracle
    rng = np.random.default_rng(14)
    for dt, soa in ((np.float64, 8), (np.float32, 16)):
        M, K, N, lda, ldc, E, pad = 9, 24, 18, 28, 20, 200, 8
        cp, ri, va = [0], [], []
        for n in range(N):
            ks = [int(k) for k in rng.integers(0, K + 3, size=int(rng.integers(0, 7)))]      # duplicates and k >= K on purpose
            ri += ks; va += [float(v) for v in rng.uniform(-1, 1, len(ks))]; cp.append(len(ri))
        cp, ri, va = np.array(cp, np.uint32), np.array(ri, np.uint32), np.array(va, dt)
        sa, sc = M * lda * soa + pad, M * ldc * soa + pad
        Af = rng.uniform(-1, 1, E * sa).astype(dt); Cf = rng.uniform(-1, 1, E * sc).astype(dt)
        want = Cf.copy()
        for e in range(E):
            Ae = np.ascontiguousarray(Af[e * sa:e * sa + M * lda * soa].reshape(M, lda, soa))
            Ce = np.ascontiguousarray(want[e * sc:e * sc + M * ldc * soa].reshape(M, ldc, soa))
            oracle.csc_soa_execute(cp, ri, va, Ae, Ce, N, beta=0.0, K=K)
            want[e * sc:e * sc + M * ldc * soa] = Ce.ravel()
        op = gpu.CsrSoa(M, N, K, cp, ri, va, soa, lda=lda, ldc=ldc, beta=0.0, sparse="B", fmt="csc")
        dA, dC = gpu.DeviceBuffer.from_numpy(Af), gpu.DeviceBuffer.from_numpy(Cf)
        op.execute(dA, dC, E, sa, sc)
        gpu.synchronize()
        C = dC.to_numpy(dt, Cf.shape)
        dA.free(); dC.free(); op.destroy()
        assert np.array_equal(bits(C), bits(want)), dt.__name__
    gpu.check()


@pytest.mark.gpu
def test_gpu_b_sparse_matches_reference_and_oracle(gpu, oracle, cases):
    d, _ = cases
    for key in [str(n) for n in d["bnames"]]:
        M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
        for beta in (0.0, 1.0):
            op = gpu.CsrSoa(M, N, K, d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"], soa, beta=beta, sparse="B")
            assert op.is_baked, key
            dA, dC = gpu.DeviceBuffer.from_numpy(d[key + "_A"]), gpu.DeviceBuffer.from_numpy(d[key + "_C0"])
            op.execute(dA, dC, E)
            gpu.synchronize()
            C = dC.to_numpy(d[key + "_C0"].dtype, d[key + "_C0"].shape)
            dA.free(); dC.free(); op.destroy()
            assert matches_reference(C, d, key, beta), "%s beta=%g" % (key, beta)
            want = d[key + "_C0"].copy()
            oracle.csr_soa_bsparse_execute(d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"], d[key + "_A"], want, N, beta=beta)
            assert np.array_equal(bits(C), bits(want)), "%s beta=%g" % (key, beta)
    # many elements, padded pitches and element strides, an empty column and an empty row of B, against the oracle
    rng = np.random.default_rng(10)
    for dt, soa in ((np.float64, 8), (np.float32, 16)):
        M, K, N, lda, ldc, E, pad = 9, 35, 20, 40, 24, 300, 16
        b = np.where(rng.random((K, N)) < 0.2, rng.uniform(-1, 1, (K, N)), 0).astype(dt)
        b[:, 5] = 0; b[7, :] = 0
        rp, ci, va = [0], [], []
        for i in range(K):
            nz = np.nonzero(b[i])[0]
            ci += list(nz); va += list(b[i, nz]); rp.append(len(ci))
        rp, ci, va = np.array(rp, np.uint32), np.array(ci, np.uint32), np.array(va, dt)
        sa, sc = M * lda * soa + pad, M * ldc * soa + pad
        Af = rng.uniform(-1, 1, E * sa).astype(dt); Cf = rng.uniform(-1, 1, E * sc).astype(dt)
        want = Cf.copy()
        for e in range(E):
            Ae = np.ascontiguousarray(Af[e * sa:e * sa + M * lda * soa].reshape(M, lda, soa))
            Ce = np.ascontiguousarray(want[e * sc:e * sc + M * ldc * soa].reshape(M, ldc, soa))
            oracle.csr_soa_bsparse_execute(rp, ci, va, Ae, Ce, N, beta=1.0)
            want[e * sc:e * sc + M * ldc * soa] = Ce.ravel()
        op = gpu.CsrSoa(M, N, K, rp, ci, va, soa, lda=lda, ldc=ldc, beta=1.0, sparse="B")
        dA, dC = gpu.DeviceBuffer.from_numpy(Af), gpu.DeviceBuffer.from_numpy(Cf)
        op.execute(dA, dC, E, sa, sc)
        gpu.synchronize()
        C = dC.to_numpy(dt, Cf.shape)
        dA.free(); dC.free(); op.destroy()
        assert np.array_equal(bits(C), bits(want)), dt.__name__
    gpu.check()


@pytest.mark.gpu
def test_gpu_matches_reference_outputs(gpu, oracle, cases):
    d, names = cases
    for key in names:
        M, K, N, soa, E = (int(x) for x in d[key + "_shape"])
        for beta in (0.0, 1.0):
            op = gpu.CsrSoa(M, N, K, d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"], soa, beta=beta)
            assert op.is_baked, key
            dB, dC = gpu.DeviceBuffer.from_numpy(d[key + "_B"]), gpu.DeviceBuffer.from_numpy(d[key + "_C0"])
            op.execute(dB, dC, E)
            gpu.synchronize()
            C = dC.to_numpy(d[key + "_C0"].dtype, d[key + "_C0"].shape)
            dB.free(); dC.free(); op.destroy()
            assert matches_reference(C, d, key, beta), "%s beta=%g" % (key, beta)
            want = d[key + "_C0"].copy()
            oracle.csr_soa_execute(d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"], d[key + "_B"], want, N, beta=beta)
            assert np.array_equal(bits(C), bits(want)), "%s beta=%g" % (key, beta)
    gpu.check()


@pytest.mark.gpu
def test_gpu_batched_strided_against_oracle(gpu, oracle):
    """many elements, pitches larger than N, element strides larger than one element, an operator too wide for the baked
    register kernel (falls back to the generic batched kernel), invalid arguments."""
    rng = np.random.default_rng(9)
    for dt, soa in ((np.float64, 8), (np.float32, 16)):
        for (M, K, N, ld, dens, beta, E, pad) in ((35, 35, 9, 9, 0.1, 0.0, 500, 0), (56, 56, 9, 12, 0.2, 1.0, 64, 40), (8, 260, 5, 5, 0.5, 0.0, 17, 0)):
            a = np.where(rng.random((M, K)) < dens, rng.uniform(-1, 1, (M, K)), 0).astype(dt)
            a[M // 3, :] = 0
            rp, ci, va = [0], [], []
            for i in range(M):
                nz = np.nonzero(a[i])[0]
                ci += list(nz); va += list(a[i, nz]); rp.append(len(ci))
            rp, ci, va = np.array(rp, np.uint32), np.array(ci, np.uint32), np.array(va, dt)
            sb, sc = K * ld * soa + pad, M * ld * soa + pad
            Bf = rng.uniform(-1, 1, E * sb).astype(dt); Cf = rng.uniform(-1, 1, E * sc).astype(dt)
            want = Cf.copy()
            for e in range(E):
                Be = np.ascontiguousarray(Bf[e * sb:e * sb + K * ld * soa].reshape(K, ld, soa))
                Ce = np.ascontiguousarray(want[e * sc:e * sc + M * ld * soa].reshape(M, ld, soa))
                oracle.csr_soa_execute(rp, ci, va, Be, Ce, N, beta=beta)
                want[e * sc:e * sc + M * ld * soa] = Ce.ravel()
            op = gpu.CsrSoa(M, N, K, rp, ci, va, soa, ldb=ld, ldc=ld, beta=beta)
            assert op.is_baked == (K <= 100 if dt == np.float64 else K <= 200)
            dB, dC = gpu.DeviceBuffer.from_numpy(Bf), gpu.DeviceBuffer.from_numpy(Cf)
            op.execute(dB, dC, E, sb, sc)
            gpu.synchronize()
            C = dC.to_numpy(dt, Cf.shape)
            dB.free(); dC.free(); op.destroy()
            assert np.array_equal(bits(C), bits(want)), (dt.__name__, M, K, N, ld, E)
    with pytest.raises(ValueError):
        gpu.CsrSoa(4, 9, 4, np.array([0, 1, 2, 3, 4], np.uint32), np.array([0, 1, 2, 9], np.uint32), np.ones(4), 8)     # column index out of range
    with pytest.raises(ValueError):
        gpu.CsrSoa(4, 9, 4, np.array([0, 1, 2, 3, 4], np.uint32), np.array([0, 1, 2, 3], np.uint32), np.ones(4), 8, beta=0.5)   # the reference's descriptor rejects it too
    gpu.check()
