"""The wide bf16 slicing kernel K1x (spmdm_slice_bf16x_kernel: transa 'N', complete 128-column blocks, 16-byte aligned rows)
bit for bit against two independent producers of the same slices on the same matrix:

  * the generic slicing kernel, reached by placing A 8 bytes past a 16-byte boundary: rowidx, colidx, values, the tensor-core
    word per nonzero (tcpk) and slice_nnz;
  * K1c on the CSR arrays of the same matrix: the same, and the overflow counts of the structured-sparse words (slice_ovf).
    The structured-sparse words themselves (tcsp) and the overflow lists are checked through their one reader: the
    structured-sparse multiply gives the same bits on both routes' slices.

K1x tests every lane's 16 elements for +-0 first and, when a warp's rows hold at most 32 lanes with anything else (candidates),
runs the exact keep test on the compacted candidates only; denser warps take the per-lane path.  The patterns below sit on both
sides of that bound."""
import numpy as np
import pytest

from test_spmdm_csr_gpu import to_csr

pytestmark = pytest.mark.gpu


# ---- helpers ---------------------------------------------------------------------------------------------------------
def random_bits(rng, shape, density):
    """bf16 bit patterns of both signs, magnitudes in [0.5, 2), at `density`"""
    v = ((rng.random(shape) + 0.5) * rng.choice([-1.0, 1.0], shape) * np.where(rng.random(shape) < 0.5, 1.0, 2.0)).astype(np.float32)
    bits = (v.view(np.uint32) >> np.uint32(16)).astype(np.uint16)
    return np.where(rng.random(shape) < density, bits, np.uint16(0)).astype(np.uint16)


def read_arena(xs, h, slices):
    """rowidx, colidx, values, tcpk, slice_nnz and slice_ovf of every slice of handle h (one arena: row pointers, column
    indices, values, the 32-bit auxiliary word per entry, then the per-slice counts, each count array padded to 256 bytes)"""
    ns, cap = h.mb * h.kb, h.bm * h.bk
    ro = np.empty((ns, h.bm + 1), np.uint16)
    co = np.empty((ns, cap), np.uint16)
    va = np.empty((ns, cap), np.float32)
    base = slices[0].values
    tcpk = np.empty((ns, cap), np.uint32)
    nnz = np.empty(ns, np.uint32)
    ovf = np.empty(ns, np.uint32)
    L = xs.load()
    L.libxsmm_b200_synchronize()
    L.libxsmm_b200_memcpy_d2h(ro.ctypes.data, slices[0].rowidx, ro.nbytes)
    L.libxsmm_b200_memcpy_d2h(co.ctypes.data, slices[0].colidx, co.nbytes)
    L.libxsmm_b200_memcpy_d2h(va.ctypes.data, base, va.nbytes)
    L.libxsmm_b200_memcpy_d2h(tcpk.ctypes.data, base + ns * cap * 4, tcpk.nbytes)
    L.libxsmm_b200_memcpy_d2h(nnz.ctypes.data, base + 2 * ns * cap * 4, nnz.nbytes)
    L.libxsmm_b200_memcpy_d2h(ovf.ctypes.data, base + 2 * ns * cap * 4 + ((ns * 4 + 255) & ~255), ovf.nbytes)
    xs.check()
    return dict(rowidx=ro, colidx=co, values=va.view(np.uint32), tcpk=tcpk, nnz=nnz, ovf=ovf)


def run(xs, A, N, threads, route, B=None):
    """one handle, one slicing pass of bf16 A (route: "k1x", "generic" = A 8 bytes past a 16-byte boundary, "csr"), then
    optionally one multiply on the structured-sparse path.  Returns (geometry, arena, C, kernel name)."""
    M, K = A.shape
    p = xs.Spmdm(M, N, K, threads)
    bufs = []
    try:
        if "csr" == route:
            bufs += [xs.DeviceBuffer.from_numpy(x) for x in to_csr(A)]
            p.create_slices_csr(bufs[0], bufs[1], bufs[2], int(np.count_nonzero(A)), True)
        else:
            off = 8 if "generic" == route else 0
            dA = xs.DeviceBuffer(A.nbytes + off)
            bufs.append(dA)
            dA.upload(A, off)
            p.create_slices(dA.ptr + off, "N", True)
        xs.synchronize()
        ar = read_arena(xs, p.handle, p.slices)
        C, name = None, None
        if B is not None:
            dB, dC = xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer(M * N * 4)
            bufs += [dB, dC]
            p.compute(dB, dC, "N", "N", 0, True)
            xs.synchronize()
            C = dC.to_numpy(np.float32, (M, N))
            name = xs.last_compute_kernel()
        xs.check()
        return p.geometry, ar, C, name
    finally:
        for b in bufs:
            b.free()
        p.destroy()


def assert_same(g, got, want, keys):
    for s in range(g["mb"] * g["kb"]):
        nrows = min(g["bm"], g["m"] - (s % g["mb"]) * g["bm"])
        n = int(want["nnz"][s])
        assert int(got["nnz"][s]) == n, "slice_nnz of slice %d" % s
        np.testing.assert_array_equal(got["rowidx"][s, :nrows + 1], want["rowidx"][s, :nrows + 1], err_msg="rowidx slice %d" % s)
        for k in keys:
            np.testing.assert_array_equal(got[k][s, :n], want[k][s, :n], err_msg="%s slice %d" % (k, s))


def check_k1x(xs, monkeypatch, A, N=48, threads=1, product=True):
    """K1x's slices == the generic kernel's == K1c's; the structured-sparse product on K1x's slices == on K1c's"""
    keep = ((A & 0x7FFF) >= 1) & ((A & 0x7FFF) <= 0x7F80)
    g, k1x, _, _ = run(xs, A, N, threads, "k1x")
    _, gen, _, _ = run(xs, A, N, threads, "generic")
    assert_same(g, k1x, gen, ("colidx", "values", "tcpk"))
    assert int(k1x["nnz"].sum()) == int(keep.sum())
    _, k1c, _, _ = run(xs, A, N, threads, "csr")
    assert_same(g, k1x, k1c, ("colidx", "values", "tcpk"))
    np.testing.assert_array_equal(k1x["ovf"], k1c["ovf"])
    if product:
        monkeypatch.setenv("LIBXSMM_B200_SPMDM_TC", "1")
        monkeypatch.setenv("LIBXSMM_B200_TC16_SPARSE", "1")
        B = random_bits(np.random.default_rng(A.shape[0] + A.shape[1]), (A.shape[1], N), 1.0)
        _, _, C, name = run(xs, A, N, threads, "k1x", B)
        _, _, Cc, namec = run(xs, A, N, threads, "csr", B)
        assert name == namec
        np.testing.assert_array_equal(C.view(np.uint32), Cc.view(np.uint32))
    return g, k1x


# ---- 1. random matrices across the density range -----------------------------------------------------------------------
@pytest.mark.parametrize("density", [0.0, 0.001, 0.01, 0.03, 0.06, 0.25, 1.0])
def test_density(gpu, monkeypatch, density):
    """M = 600 = 330 + 270 (bm = 330: the 16-warp form, two parts of eleven rows per warp; the last row block ragged),
    K = 384 (row pitch three times the block width)"""
    A = random_bits(np.random.default_rng(int(density * 1000) + 5), (600, 384), density)
    g, ar = check_k1x(gpu, monkeypatch, A)
    assert g["bm"] == 330 and g["mb"] == 2


# ---- 2. the candidate bound of one warp ---------------------------------------------------------------------------------
@pytest.mark.parametrize("ncand", [31, 32, 33, 64, 65, 128])
def test_candidates_per_warp(gpu, monkeypatch, ncand):
    """warp 3 of the first slice (rows 48..63, 128 lanes of 16 columns) with exactly `ncand` lanes holding something other than
    +-0 -- among them lanes with NaN only (candidates that keep nothing) and lanes with several nonzeros -- next to lanes holding
    only -0"""
    rng = np.random.default_rng(ncand)
    A = np.zeros((512, 128), np.uint16)
    A[48:64] = 0x8000                                     # -0 everywhere: no lane is a candidate by that
    lanes = rng.permutation(128)[:ncand]
    for i, l in enumerate(lanes):
        r, c0 = 48 + l // 8, (l % 8) * 16
        seg = A[r, c0:c0 + 16]
        if i % 5 == 1:
            seg[rng.integers(0, 16)] = 0x7F81 if i % 2 else 0xFFC0          # NaN only
        else:
            for e in rng.choice(16, 1 + i % 4, replace=False):
                seg[e] = 0x3F80 + rng.integers(0, 0x40)
    A[100:116, :] = random_bits(rng, (16, 128), 0.01)     # other warps: sparse, and one empty warp in between
    check_k1x(gpu, monkeypatch, A)


# ---- 3. special values -----------------------------------------------------------------------------------------------------
def test_special_lanes(gpu, monkeypatch):
    """a lane with all 16 elements kept; lanes of -0 only and of NaN only; +-Inf and denormals; more than 256 overflow groups in
    one slice (groups of four with three or four nonzeros); a completely dense row; on a 1 % background"""
    rng = np.random.default_rng(17)
    A = random_bits(rng, (1024, 256), 0.01)
    A[3, 16:32] = 0x4000                                  # one full lane
    A[5, 32:48] = 0x8000                                  # -0 only
    A[6, 48:64] = 0x7F81                                  # NaN only
    A[7, 64:80] = 0xFFC0
    A[8, 0:8] = [0x7F80, 0xFF80, 0x0001, 0x8001, 0x7F7F, 0xFF7F, 0x0080, 0x8000]
    A[9, :] = 0x3F80                                      # a dense row
    for r in range(20, 20 + 300):                         # 300 groups with three nonzeros (one overflow each) in slice 0
        c = 4 * (r % 32)
        A[r, c:c + 3] = 0x3F80
    A[700, 128:256] = 0xC000
    A[1023, 240:256] = 0x0001
    g, ar = check_k1x(gpu, monkeypatch, A)
    assert ar["ovf"][0] > 256


def test_full_slice_wraps(gpu, monkeypatch):
    """a completely full 512 x 128 slice: its u16 row pointer after the last row wraps to 0, slice_nnz holds 65536"""
    A = np.full((512, 128), 0x3F80, np.uint16)
    A[::3] = 0xBF00
    g, ar = check_k1x(gpu, monkeypatch, A, product=False)
    assert g["bm"] == 512 and int(ar["nnz"][0]) == 65536 and ar["rowidx"][0, 512] == 0


# ---- 4. geometries -------------------------------------------------------------------------------------------------------
def test_small_row_blocks(gpu, monkeypatch):
    """bm = 242 (M = 1100, N = 48): the kernel's 32-warp form with eight rows per warp"""
    A = random_bits(np.random.default_rng(23), (1100, 384), 0.01)
    A[245:250, :] = 0x3F80                                # a dense warp among sparse ones
    g, _ = check_k1x(gpu, monkeypatch, A)
    assert g["bm"] == 242


def test_exec_host_slices(gpu):
    """the host-pointer entry slices row block by row block (every k-block of one row block per launch): the same slices as the
    stream entry"""
    xs = gpu
    rng = np.random.default_rng(29)
    M, N, K = 600, 48, 384
    A = random_bits(rng, (M, K), 0.01)
    A[520:524] = 0x3F80
    B = random_bits(rng, (K, N), 1.0)
    g, want, _, _ = run(xs, A, N, 1, "k1x")
    h, s = xs.libxsmm_spmdm_init(M, N, K, 1)
    try:
        C = np.zeros((M, N), np.float32)
        xs.libxsmm_spmdm_exec_host(h, s, xs.LIBXSMM_SPMDM_DATATYPE_BFLOAT16, "N", "N", "N", A, B, 0, C)
        xs.check()
        got = read_arena(xs, h, s)
    finally:
        xs.libxsmm_spmdm_destroy(h)
    assert g["mb"] == 2
    assert_same(g, got, want, ("colidx", "values", "tcpk"))
    np.testing.assert_array_equal(got["ovf"], want["ovf"])
