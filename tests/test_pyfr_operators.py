"""All 150 operators the reference ships for its PyFR driver (samples/pyfr/mats/p1..p6/{hex,pri,quad,tet,tri}/m*-sp.mtx),
from the committed fixture tests/golden/operators_pyfr.npz (tests/golden/make_pyfr_golden.py wrote it by running the compiled
reference).  CPU part: the oracle reproduces the reference's outputs bit for bit; the product's host-side plan takes the
branch the reference took and can BAKE every one of them (registers or shared-memory strip -- none falls back to the
generic kernel).  GPU part: every operator is created, is baked, and its apply matches the reference / the oracle bit for bit."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pyfr():
    d = np.load(os.path.join(ROOT, "tests", "golden", "operators_pyfr.npz"))
    ops = []
    for i, name in enumerate(d["names"]):
        M, K = (int(x) for x in d["shapes"][i])
        lo, hi = int(d["offsets"][i]), int(d["offsets"][i + 1])
        a = np.zeros((M, K))
        a[d["rows"][lo:hi].astype(np.int64), d["cols"][lo:hi].astype(np.int64)] = d["vals"][lo:hi]
        ops.append((str(name), a))
    return d, ops


def bits(x):
    return x.view(np.uint64 if x.dtype == np.float64 else np.uint32)


def panel(a, i):
    """the seeded B / C0 panel of 16 columns the reference's stored outputs for operator i were computed from"""
    rng = np.random.default_rng(100 + i)
    return rng.uniform(-1.0, 1.0, (a.shape[1], 16)), rng.uniform(-1.0, 1.0, (a.shape[0], 16))


def matches_reference(C, d, i, beta):
    """the fixture holds every second element of the reference's output (row-major), to stay small"""
    return np.array_equal(bits(C).ravel()[::2], bits(d["out%d_%d" % (int(beta), i)]))


def test_oracle_matches_reference_outputs(oracle, pyfr):
    d, ops = pyfr
    assert len(ops) == 150 and len(d["picked"]) >= 20
    for i in d["picked"]:
        name, a = ops[int(i)]
        B, C0 = panel(a, int(i))
        for beta in (0.0, 1.0):
            C = C0.copy()
            oracle.dfsspmdm_execute(a, B, C, beta, oracle.dfsspmdm_branch(a, 16, 16, beta))
            assert matches_reference(C, d, int(i), beta), "%s beta=%g" % (name, beta)


def test_every_operator_takes_the_reference_branch_and_bakes(xs, pyfr):
    d, ops = pyfr
    forms = {}
    for i, (name, a) in enumerate(ops):
        p = xs.fsspmdm_plan(a, N=16, ldb=16, ldc=16, beta=0.0)
        assert p["sparse"] == bool(d["ref_sparse_branch"][i]), name
        assert p["nnz"] == int(d["offsets"][i + 1] - d["offsets"][i])
        for dt in (np.float64, np.float32):
            f = xs.fsspmdm_plan(a.astype(dt), N=1 << 20, beta=0.0)["form"]
            assert f != "generic", "%s (%s) would fall back to the generic kernel" % (name, dt.__name__)
            forms[f] = forms.get(f, 0) + 1
    assert forms.get("baked-strip", 0) > 20 and forms.get("baked-registers", 0) > 100, forms


@pytest.mark.gpu
def test_every_operator_on_the_gpu(gpu, oracle, pyfr):
    """fp64, beta = 0 and 1: created, baked, bit-exact -- against the oracle everywhere and, where the fixture holds them (29
    operators, 16-column panels), against the reference's stored outputs too; the others on a 64-column panel."""
    d, ops = pyfr
    picked = set(int(i) for i in d["picked"])
    rng = np.random.default_rng(77)
    for i, (name, a) in enumerate(ops):
        M, K = a.shape
        for beta in (0.0, 1.0):
            if i in picked:
                N = 16
                B, C0 = panel(a, i)
            else:
                if beta == 1.0 and i % 3:
                    continue
                N = 64
                B, C0 = rng.uniform(-1, 1, (K, N)), rng.uniform(-1, 1, (M, N))
            want = C0.copy()
            oracle.dfsspmdm_execute(a, B, want, beta, oracle.dfsspmdm_branch(a, N, N, beta))
            op = gpu.Fsspmdm(a, N, beta=beta)
            try:
                assert op.is_baked, "%s: not baked" % name
                assert op.is_sparse == bool(oracle.dfsspmdm_branch(a, N, N, beta))
                dB, dC = gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer.from_numpy(C0)
                op.execute_stream(dB, dC)
                gpu.synchronize()
                C = dC.to_numpy(np.float64, C0.shape)
                dB.free(); dC.free()
            finally:
                op.destroy()
            assert np.array_equal(bits(C), bits(want)), "%s beta=%g (%s)" % (name, beta, gpu.last_compute_kernel())
            assert i not in picked or matches_reference(C, d, i, beta), "%s beta=%g (%s)" % (name, beta, gpu.last_compute_kernel())
    gpu.check()


@pytest.mark.gpu
def test_strip_kernel_float_and_ragged_panels(gpu, oracle, pyfr):
    """the shared-memory strip form on float operators, on column counts that are not multiples of its 32-column strips, on
    panels inside wider matrices (N < ld) and with the sparse branch's untouched empty rows."""
    d, ops = pyfr
    byname = dict(ops)
    rng = np.random.default_rng(5)
    for name, dt, N, ld in (("p4/hex/m0", np.float32, 80, 80), ("p4/hex/m0", np.float64, 48, 112), ("p5/hex/m132", np.float64, 16, 16),
                            ("p5/hex/m132", np.float32, 112, 128), ("p6/pri/m132", np.float64, 96, 96)):
        a = byname[name].astype(dt).copy()
        a[3, :] = 0                                   # an empty row
        M, K = a.shape
        for beta in (0.0, 1.0):
            B = rng.uniform(-1, 1, (K, ld)).astype(dt); C0 = rng.uniform(-1, 1, (M, ld)).astype(dt)
            want = C0.copy()
            if dt == np.float64:
                oracle.dfsspmdm_execute(a, B, want, beta, oracle.dfsspmdm_branch(a, ld, ld, beta), N=N, ldb=ld, ldc=ld)
            else:
                oracle.sfsspmdm_execute(a, B, want, beta, N=N, ldb=ld, ldc=ld)
            op = gpu.Fsspmdm(a, N, ldb=ld, ldc=ld, beta=beta)
            assert gpu.fsspmdm_plan(a, N=N, ldb=ld, ldc=ld, beta=beta)["form"] == "baked-strip", name
            dB, dC = gpu.DeviceBuffer.from_numpy(B), gpu.DeviceBuffer.from_numpy(C0)
            op.execute_stream(dB, dC)
            gpu.synchronize()
            C = dC.to_numpy(dt, C0.shape)
            assert gpu.last_compute_kernel() == "fs_baked"
            dB.free(); dC.free(); op.destroy()
            assert np.array_equal(bits(C), bits(want)), "%s %s N=%d ld=%d beta=%g" % (name, dt.__name__, N, ld, beta)
    gpu.check()
