"""GPU parity of the tensor-core branch of libxsmm_spmdm compute (tcgen05, 3xTF32, csrc/spmdm_compute_tc.cu).

The branch is selected on the device when the slices hold >= 7 % nonzeros (fp32, N/N/N, 16-byte aligned
panels); LIBXSMM_B200_SPMDM_TC=1 forces it, =0 disables it.  It does not keep the reference's rounding
sequence, so the bar is the contract of BASELINE.json: 1e-5 relative (max abs error / max |C|)."""
import numpy as np
import pytest

from test_spmdm_gpu import gpu_spmdm, oracle_spmdm, valid_slices_equal

pytestmark = pytest.mark.gpu
RTOL_F32 = 1e-5


def rel(got, want):
    return float(np.abs(got.astype(np.float64) - want.astype(np.float64)).max() / max(float(np.abs(want).max()), 1e-30))


CASES = [
    # M, N, K, density, beta, threads
    (128, 128, 128, 0.50, 0.0, 1),
    (512, 384, 640, 0.10, 0.0, 1),
    (512, 384, 640, 0.10, 1.0, 1),
    (512, 384, 640, 0.10, 0.5, 1),
    (300, 204, 260, 0.30, 0.75, 1),      # ragged M, N (204 = 4*51: narrow reference block, partial CTA columns), K tail
    (1024, 512, 512, 0.50, 0.0, 8),
    (2048, 256, 256, 0.10, 0.0, 56),     # bm = 245: row tiles 128 + 117
    (33, 8, 129, 0.40, 1.0, 1),
    (512, 128, 128, 1.00, 0.0, 1),       # completely full slice: u16 counter wraps, last row reads as empty like the reference
]


@pytest.mark.parametrize("mode", ["1", "auto"])
@pytest.mark.parametrize("M,N,K,density,beta,threads", CASES)
def test_tc_matches_oracle(gpu, oracle, monkeypatch, mode, M, N, K, density, beta, threads):
    if mode == "auto":
        monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    else:
        monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", mode)
    w = gpu.workloads
    if density >= 1.0:
        A = (np.random.default_rng(2).random((M, K)) + 0.5).astype(np.float32)
        B = np.random.default_rng(3).random((K, N)).astype(np.float32)
        C0 = np.random.default_rng(4).random((M, N)).astype(np.float32)
    else:
        A, B, C0 = w.spmdm_inputs(M, N, K, density, seed=M + N + K)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=beta, max_threads=threads)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", float(beta))
    valid_slices_equal(og, sl, osl)
    err = rel(C, OC)
    assert err <= RTOL_F32, "relative error %g" % err
    gpu.check()


@pytest.mark.parametrize("ta,tb,tc", [("T", "N", "T"), ("N", "T", "N"), ("T", "T", "T"), ("N", "N", "T"), ("T", "T", "N")])
@pytest.mark.parametrize("M,N,K,density,beta", [(260, 200, 300, 0.5, 0.0), (512, 384, 640, 0.2, 0.5), (1024, 256, 512, 0.5, 1.0)])
def test_tc_transposed_variants(gpu, oracle, monkeypatch, ta, tb, tc, M, N, K, density, beta):
    """the sample's "weight update" (T/N/T) and "backprop" (N/T/N) variants and the other flag combinations:
    B stored n x k is a K-major tensor-core operand, C stored n x m is written one full line per instruction."""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, density, seed=M + K, transa=ta, transb=tb, transc=tc)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, beta)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, ta, tb, tc, float(beta))
    valid_slices_equal(og, sl, osl)
    err = rel(C, OC)
    assert err <= RTOL_F32, "relative error %g" % err
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    _, _, C_cc = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, beta)
    if K % 4 == 0 or tb == "N":      # the panel qualified for the tensor-core kernel: different rounding sequence
        assert not np.array_equal(C.view(np.uint32), C_cc.view(np.uint32))
    gpu.check()


def test_sparse_problem_stays_bit_exact_in_auto_mode(gpu, oracle, monkeypatch):
    """below the density threshold the CUDA-core twin runs: same bits as the oracle."""
    monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    M, N, K = 512, 384, 640
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, 0.02, seed=9)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=0.5)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", 0.5)
    np.testing.assert_array_equal(C.view(np.uint32), OC.view(np.uint32))


def test_dense_problem_takes_the_tensor_core_branch(gpu, monkeypatch):
    """same inputs, TC off vs auto: results differ in the last bits (different rounding sequence), which
    shows that the dense twin actually ran; both are within the contract of each other."""
    M, N, K = 512, 512, 512
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, 0.5, seed=10)
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    _, _, C_cc = gpu_spmdm(gpu, A, B, C0, M, N, K)
    monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    _, _, C_tc = gpu_spmdm(gpu, A, B, C0, M, N, K)
    assert rel(C_tc, C_cc) <= RTOL_F32
    assert not np.array_equal(C_tc.view(np.uint32), C_cc.view(np.uint32))


@pytest.mark.parametrize("name,density", [("C1", 0.10), ("C4", 0.50)])
def test_full_size(gpu, name, density, monkeypatch):
    """BASELINE sizes (2048^3): every output element against a float64 product of the same inputs, plus
    B = identity, which must reproduce A to 3xTF32 accuracy (a_lo keeps 11 of its 13 bits: 2^-22 relative)."""
    monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    M = N = K = 2048
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, density, seed=1)
    _, _, C = gpu_spmdm(gpu, A, B, C0, M, N, K)
    want = A.astype(np.float64) @ B.astype(np.float64)
    assert np.abs(C - want).max() / np.abs(want).max() <= RTOL_F32
    _, _, Ci = gpu_spmdm(gpu, A, np.eye(K, N, dtype=np.float32), C0, M, N, K)
    assert np.abs(Ci - A).max() <= 2.0 ** -21 * np.abs(A).max()
    assert np.array_equal(Ci == 0, A == 0)      # dropped entries stay exact zeros


@pytest.mark.parametrize("mode", ["1", "auto"])
@pytest.mark.parametrize("M,N,K,density,beta,ta,tb,tc", [
    (512, 512, 512, 0.10, 0, "N", "N", "N"), (512, 512, 512, 0.10, 1, "N", "N", "N"), (300, 208, 256, 0.30, 0, "N", "N", "N"),
    (4096, 320, 256, 0.05, 0, "N", "N", "N"), (256, 200, 384, 0.20, 0, "T", "N", "T"), (256, 200, 384, 0.20, 0, "N", "T", "N"),
    (512, 256, 128, 1.00, 0, "N", "N", "N")])
def test_bf16_tensor_core_branch(gpu, oracle, monkeypatch, mode, M, N, K, density, beta, ta, tb, tc):
    """bf16 inputs on tcgen05 (kind::f16, exact products, fp32 accumulation in TMEM).  Contract 1e-2 relative;
    observed 1e-6."""
    if mode == "auto":
        monkeypatch.delenv("LIBXSMM_B200_SPMDM_TC", raising=False)
    else:
        monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", mode)
    if density >= 1.0:
        rng = np.random.default_rng(5)
        A = gpu.workloads.to_bf16_bits((rng.random((M, K)) + 0.5).astype(np.float32))
        B = gpu.workloads.to_bf16_bits(rng.random((K, N)).astype(np.float32))
        C0 = rng.random((M, N)).astype(np.float32)
    else:
        A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, density, dtype="bf16", seed=M + N, transa=ta, transb=tb, transc=tc)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, beta, True)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, ta, tb, tc, float(beta))
    valid_slices_equal(og, sl, osl)
    assert rel(C, OC) <= 1e-5
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    _, _, C_cc = gpu_spmdm(gpu, A, B, C0, M, N, K, ta, tb, tc, beta, True)
    np.testing.assert_array_equal(C_cc.view(np.uint32), OC.view(np.uint32))      # the CUDA-core path stays bit exact
    assert not np.array_equal(C.view(np.uint32), C_cc.view(np.uint32))           # ... and the tensor-core twin really ran
    gpu.check()


# pair = "1": the CTA-pair kernel (K4p), the only bf16 dense tensor-core kernel; the parameter keeps the case ids stable
@pytest.mark.parametrize("density,beta,pair", [(0.01, 0, "1"), (0.01, 1, "1"), (0.05, 0, "1"), (0.30, 0, "1")])
def test_bf16_full_size_c2(gpu, monkeypatch, density, beta, pair):
    """BASELINE C2 (bf16, 4096^3) on the tensor cores -- 256 pair tiles on 74 CTA pairs: three whole rounds and a
    last round of half tiles -- against the order-preserving CUDA-core kernels on the same device buffers
    (those are bit-exact against the oracle at the sizes the oracle can do), every output element."""
    M = N = K = 4096
    A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, density, dtype="bf16", seed=7)
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    _, _, C_tc = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=beta, bf16=True)
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "0")
    _, _, C_cc = gpu_spmdm(gpu, A, B, C0, M, N, K, beta=beta, bf16=True)
    assert rel(C_tc, C_cc) <= 1e-5
    assert not np.array_equal(C_tc.view(np.uint32), C_cc.view(np.uint32))
    rows = np.arange(0, M, 37)
    want = gpu.workloads.from_bf16_bits(A[rows]).astype(np.float64) @ gpu.workloads.from_bf16_bits(B).astype(np.float64) + beta * C0[rows]
    assert rel(C_tc[rows], want) <= 1e-5
    gpu.check()


@pytest.mark.parametrize("pair", ["1"])     # the CTA-pair kernel (K4p); the parameter keeps the case ids stable
@pytest.mark.parametrize("M,N,K,density,beta,threads", [
    (300, 204, 260, 0.30, 1, 1),        # ragged M, partial 256-column tile, K tail (260 = 2 * 128 + 4)
    (2048, 256, 200, 0.02, 0, 56),      # bm = 245 (balance loop): CTA tiles of 128 + 117 rows, pairs span row blocks
    (33, 8, 129, 0.40, 0, 1),           # one partial tile, second k-block holds a single column
    (1536, 520, 384, 0.002, 0, 1),      # nearly empty slices (most k-blocks of a tile hold no nonzero)
    (640, 256, 128, 1.00, 0, 1),        # full slices: u16 counter wraps in the first row block, dense fallback of the workers
])
def test_bf16_tensor_core_shapes(gpu, oracle, monkeypatch, pair, M, N, K, density, beta, threads):
    """geometry corners of the bf16 CTA-pair tensor-core kernel, forced on."""
    monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
    if density >= 1.0:
        rng = np.random.default_rng(5)
        A = gpu.workloads.to_bf16_bits((rng.random((M, K)) + 0.5).astype(np.float32))
        B = gpu.workloads.to_bf16_bits(rng.random((K, N)).astype(np.float32))
        C0 = rng.random((M, N)).astype(np.float32)
    else:
        A, B, C0 = gpu.workloads.spmdm_inputs(M, N, K, density, dtype="bf16", seed=M + K)
    g, sl, C = gpu_spmdm(gpu, A, B, C0, M, N, K, "N", "N", "N", beta, True, threads)
    og, osl, OC = oracle_spmdm(oracle, g, A, B, C0, "N", "N", "N", float(beta))
    valid_slices_equal(og, sl, osl)
    assert rel(C, OC) <= 1e-5
    gpu.check()
