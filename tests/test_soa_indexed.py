"""Indexed execution of the batched SoA entries (libxsmm_b200_rm_soa_execute_indexed, libxsmm_b200_csr_soa_execute_indexed):
element e reads and writes its operands at slot index[e] instead of slot e.  The strided entries are pinned bit for bit against
the oracle elsewhere (test_rm_soa.py, test_csr_soa.py), so the main check here is bit for bit against the strided entry run on a
numpy-gathered compact copy, scattered back; the oracle (tests/rm_soa_oracle.c, compiled by this file's fixture) checks the
neighbour-flux pattern.  CPU: every host rejection (error -84), which makes no CUDA call."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import test_rm_soa as R

HERE = os.path.dirname(os.path.abspath(__file__))
NAN_BITS = {np.float64: np.uint64(0x7FF8DEAD0000BEEF), np.float32: np.uint32(0x7FC0BEEF)}


@pytest.fixture(scope="module")
def rm_oracle():
    tmp = tempfile.mkdtemp(prefix="rm_soa_oracle_")
    try:
        lib = os.path.join(tmp, "librm_soa_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-shared", "-o", lib,
                               os.path.join(HERE, "rm_soa_oracle.c"), "-lm"])
        yield R.RmOracle(lib)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


@pytest.fixture(scope="module")
def ops():
    with np.load(os.path.join(HERE, "golden", "csr_soa.npz")) as z:
        return dict(z)


def u32(x):
    return np.ascontiguousarray(x, np.uint32)


def slots_of(idx, E):
    return np.arange(E) if idx is None else np.asarray(idx, np.int64)


def gather(flat, stride, ext, sl):
    """compact copy of the slots sl (stride 0: the shared operand itself)"""
    if stride == 0:
        return flat.copy(), 0
    out = np.empty(max(len(sl), 1) * ext, flat.dtype)
    for e, s in enumerate(sl):
        out[e * ext:(e + 1) * ext] = flat[s * stride:s * stride + ext]
    return out, ext


def scatter(dst, stride, ext, sl, compact):
    for e, s in enumerate(sl):
        dst[s * stride:s * stride + ext] = compact[e * ext:(e + 1) * ext]


def upload(gpu, *arrays):
    return [None if x is None else gpu.DeviceBuffer.from_numpy(np.ascontiguousarray(x)) for x in arrays]


def free(*bufs):
    for d in bufs:
        if d is not None:
            d.free()


def rm_case(rng, op, dt, slots, strides):
    """flat a, b, C0 with slots[i] slots at strides[i] (0: one shared copy); C gaps hold SENT"""
    ext = op.extents
    out = []
    for i, (n, s) in enumerate(zip(slots, strides)):
        size = (n - 1) * s + ext[i] if s else ext[i]
        out.append(rng.uniform(-1, 1, size).astype(dt) if i < 2 else np.full(size, R.SENT, dt))
    c = out[2]
    for sl in range(slots[2]):
        for m in range(op.M):
            o = sl * strides[2] + m * op.ldc * op.soa
            c[o:o + op.N * op.soa] = rng.uniform(-1, 1, op.N * op.soa).astype(dt)
    return out


def rm_expected(gpu, op, a, b, c0, E, strides, idx, slots):
    """the strided entry on a numpy-gathered compact copy of the elements that run, scattered back into C0"""
    ext = op.extents
    sl = [slots_of(idx[i], E) for i in range(3)]
    run = np.ones(E, bool)
    for i in range(3):
        if idx[i] is not None:
            run &= sl[i] < slots[i]
    want = c0.copy()
    if not run.any():
        return want
    comp = [gather(x, strides[i], ext[i], sl[i][run]) for i, x in enumerate((a, b, c0))]
    d = upload(gpu, comp[0][0], comp[1][0], comp[2][0])
    op.execute(d[0], d[1], d[2], int(run.sum()), comp[0][1], comp[1][1], comp[2][1])
    gpu.synchronize()
    cc = d[2].to_numpy(c0.dtype, comp[2][0].shape)
    free(*d)
    scatter(want, strides[2], ext[2], sl[2][run], cc)
    return want


def rm_indexed(gpu, op, a, b, c0, E, strides, idx, slots, shift=(0, 0, 0)):
    """uploads (each base pointer `shift` scalars past a 16-byte boundary), runs the indexed entry once, returns C and the kernel"""
    es = a.itemsize
    bufs = []
    for x, sh in zip((a, b, c0), shift):
        dd = gpu.DeviceBuffer(x.nbytes + sh * es + 16)
        dd.upload(x, sh * es)
        bufs.append(dd)
    di = upload(gpu, *[None if i is None else u32(i) for i in idx])
    ptr = [bufs[i].ptr + shift[i] * es for i in range(3)]
    op.execute_indexed(ptr[0], ptr[1], ptr[2], E, di[0], slots[0], di[1], slots[1], di[2], slots[2], *strides)
    gpu.synchronize()
    kernel = gpu.last_compute_kernel()
    C = bufs[2].to_numpy(c0.dtype, c0.shape, shift[2] * es)
    free(*bufs, *di)
    gpu.check()
    return C, kernel


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_rm_rejects_invalid_arguments_without_launching(xs):
    """checked before any CUDA call, so this runs without a device too"""
    xs.clear_error()
    h = xs.rm_soa_create("ac", True, 35, 9, 9, 9, 9, 9, 8, 1.0)
    ea, eb, ec = 35 * 9 * 8, 81, (34 * 9 + 9) * 8
    P = 4096                                                     # a dummy device address: nothing may be launched
    n0 = xs.launch_count()
    ok = dict(n=4, sa=ea, sb=eb, sc=ec, ia=None, na=0, ib=None, nb=0, ic=None, nc=0, a=P, b=P, c=P)
    bad = [dict(n=-1), dict(sa=-1), dict(sb=-1), dict(sc=-1),
           dict(ia=P, na=0), dict(ib=P, nb=-5), dict(ic=P, nc=0), dict(ia=P, na=(1 << 32) + 1), dict(ic=P, nc=(1 << 32) + 1),
           dict(a=None), dict(b=None), dict(c=None),
           dict(sc=ec - 1), dict(sc=0),                                     # no C index, more than one element
           dict(ic=P, nc=2, sc=ec - 1), dict(ic=P, nc=1 << 20, sc=0)]       # C index, more than one slot
    for d in bad:
        k = dict(ok, **d)
        xs.rm_soa_execute_indexed(h, k["a"], k["b"], k["c"], k["n"], k["sa"], k["sb"], k["sc"], k["ia"], k["na"], k["ib"], k["nb"],
                                  k["ic"], k["nc"])
        assert xs.last_error()[0] == -84, d
        xs.clear_error()
    xs.rm_soa_execute_indexed(None, P, P, P, 1, ea, eb, ec, None, 0, None, 0, None, 0)
    assert xs.last_error()[0] == -84
    xs.clear_error()
    # no elements: nothing to do, no error -- even with NULL operands; an index's slot count is still checked
    xs.rm_soa_execute_indexed(h, None, None, None, 0, ea, eb, ec, P, 1, None, 0, P, 1 << 32)
    assert xs.last_error()[0] == 0
    xs.rm_soa_execute_indexed(h, None, None, None, 0, ea, eb, ec, P, 0, None, 0, None, 0)
    assert xs.last_error()[0] == -84
    xs.clear_error()
    assert xs.launch_count() == n0
    xs.rm_soa_destroy(h)


def test_csr_rejects_null_handle_without_launching(xs):
    xs.clear_error()
    n0 = xs.launch_count()
    xs.csr_soa_execute_indexed(None, 4096, 4096, 4, 2520, 2520, None, 0, None, 0)
    assert xs.last_error()[0] == -84
    xs.clear_error()
    assert xs.launch_count() == n0


# ---------------------------------------------------------------------------------------------------------------- GPU: rm_soa
@pytest.mark.gpu
@pytest.mark.parametrize("form", R.FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16), (np.float64, 3), (np.float32, 3)])
@pytest.mark.parametrize("beta", (0.0, 1.0))
def test_gpu_rm_random_gathers(gpu, form, dt, soa, beta):
    """random gathers of a and b (repeating), a permutation of the C slots, per-element and shared plain operands; the staged and
    (element stride one scalar longer, or a base one scalar off) the direct path"""
    rng = np.random.default_rng(100 + soa)
    M, N, K, E = 35, 9, 9 if form == "ac" else 35, 300
    op = gpu.RmSoa(form, M, N, K, soa, dt, beta=beta)
    ea, eb, ec = op.extents
    x = 0 if form == "ac" else 1
    aligned = (op.extents[x] * np.dtype(dt).itemsize) % 16 == 0
    for pad, shift in ((0, (0, 0, 0)), (1, (0, 0, 0)), (0, (1, 1, 1))):
        for shared in (False, True):
            strides = [ea + pad, eb + pad, ec + 3]
            if shared:
                strides[1 - x] = 0                                   # the plain operand shared by all elements
            slots = (400, 350, E)
            idx = [rng.integers(0, 400, E), rng.integers(0, 350, E), rng.permutation(E)]
            a, b, c0 = rm_case(rng, op, dt, slots, strides)
            want = rm_expected(gpu, op, a, b, c0, E, strides, idx, slots)
            C, kernel = rm_indexed(gpu, op, a, b, c0, E, strides, idx, slots, shift)
            assert R.same(C, want), (pad, shift, shared, kernel)
            assert kernel.startswith("rm_soa_" + form)
            if aligned:
                assert kernel.endswith("(staged)" if pad == 0 and shift == (0, 0, 0) else "(direct)"), (pad, shift, kernel)
    op.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("form", R.FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
def test_gpu_rm_identity_and_null_index(gpu, rm_oracle, form, dt, soa):
    """identity arrays, NULL indices and the strided entry give the same bits (and the oracle's), also with more elements than
    CTAs; an index on a shared operand (stride 0) still reads the shared copy"""
    rng = np.random.default_rng(7)
    M, N, K = 35, 9, 9 if form == "ac" else 35
    for E in (5, 4001):
        for beta in (0.0, 1.0):
            op = gpu.RmSoa(form, M, N, K, soa, dt, beta=beta)
            ea, eb, ec = op.extents
            strides = [ea, eb, ec]
            a, b, c0 = rm_case(rng, op, dt, (E, E, E), strides)
            ref, _ = R.gpu_run(gpu, form, dt, M, N, K, soa, beta, op.lda, op.ldb, op.ldc, a, b, c0, E, *strides)
            assert R.same(ref, R.oracle_run(rm_oracle, form, M, N, K, op.lda, op.ldb, op.ldc, soa, beta, a, b, c0, E, *strides))
            ident = np.arange(E)
            for idx in ([ident, ident, ident], [None, None, None], [ident, None, None], [None, None, ident]):
                C, _ = rm_indexed(gpu, op, a, b, c0, E, strides, idx, (E, E, E))
                assert np.array_equal(R.bits(C), R.bits(ref)), [i is None for i in idx]
            # shared plain operand with an index: every in-range slot reads the one copy
            sh = list(strides); sh[1 if form == "ac" else 0] = 0
            a2, b2, _ = rm_case(rng, op, dt, (E, E, E), sh)
            ref2, _ = R.gpu_run(gpu, form, dt, M, N, K, soa, beta, op.lda, op.ldb, op.ldc, a2, b2, c0, E, *sh)
            pidx = rng.integers(0, 7, E)
            idx = [pidx, None, None] if form == "bc" else [None, pidx, None]
            slots = (7, 0, 0) if form == "bc" else (0, 7, 0)
            C, _ = rm_indexed(gpu, op, a2, b2, c0, E, sh, idx, slots)
            assert np.array_equal(R.bits(C), R.bits(ref2))
            op.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
def test_gpu_rm_neighbour_flux(gpu, rm_oracle, dt, soa):
    """C[e] += F_f . X[neigh_f(e)] for four faces with beta = 1 (ac form: X per element, F_f shared), repeating input indices:
    the sequential oracle result on gathered inputs"""
    rng = np.random.default_rng(21)
    M, N, K, E = 35, 9, 9, 2000
    op = gpu.RmSoa("ac", M, N, K, soa, dt, beta=1.0)
    ea, eb, ec = op.extents
    X = rng.uniform(-1, 1, E * ea).astype(dt)
    F = [rng.uniform(-1, 1, eb).astype(dt) for _ in range(4)]
    c0 = rng.uniform(-1, 1, E * ec).astype(dt)
    neigh = [rng.integers(0, E, E) for _ in range(4)]
    want = c0.copy()
    for f in range(4):
        xg, _ = gather(X, ea, ea, neigh[f])
        rm_oracle.rm_soa_execute("ac", M, N, K, op.lda, op.ldb, op.ldc, soa, 1.0, xg, F[f], want, E, ea, 0, ec)
    dX, dC = upload(gpu, X, c0)
    dF = upload(gpu, *F)
    dN = upload(gpu, *[u32(n) for n in neigh])
    n0 = gpu.launch_count()
    for f in range(4):
        op.execute_indexed(dX, dF[f], dC, E, a_index=dN[f], a_slots=E, stride_b=0)
    assert gpu.launch_count() == n0 + 4
    gpu.synchronize()
    assert R.same(dC.to_numpy(dt, c0.shape), want)
    free(dX, dC, *dF, *dN)
    op.destroy()
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("form", R.FORMS)
@pytest.mark.parametrize("beta", (0.0, 1.0))
def test_gpu_rm_cluster_subset(gpu, form, beta):
    """a sorted random half of the slots as inputs and C: the other slots keep their bits exactly, and with beta = 1 only the
    indexed slots are read (the others hold NaN in every operand)"""
    rng = np.random.default_rng(22)
    dt, soa, M, N, K, S = np.float64, 8, 35, 9, 9 if form == "ac" else 35, 3000
    op = gpu.RmSoa(form, M, N, K, soa, dt, beta=beta)
    strides = list(op.extents)
    a, b, c0 = rm_case(rng, op, dt, (S, S, S), strides)
    sub = np.sort(rng.choice(S, S // 2, replace=False))
    out = np.setdiff1d(np.arange(S), sub)
    for x, st, ext in zip((a, b, c0), strides, op.extents):
        for s in out:
            x[s * st:s * st + ext].view(R.bits(x).dtype)[:] = NAN_BITS[dt]
    idx = [sub, sub, sub]
    want = rm_expected(gpu, op, a, b, c0, len(sub), strides, idx, (S, S, S))
    C, _ = rm_indexed(gpu, op, a, b, c0, len(sub), strides, idx, (S, S, S))
    assert np.array_equal(R.bits(C), R.bits(want))
    assert not np.isnan(C[[s * strides[2] for s in sub]]).any()
    op.destroy()


def guarded(gpu, arr, G=1 << 16):
    raw = np.full(2 * G + arr.nbytes, 0xA5, np.uint8)
    raw[G:G + arr.nbytes] = arr.view(np.uint8).ravel()
    return gpu.DeviceBuffer.from_numpy(raw), raw


def bands_intact(d, raw, nbytes, G=1 << 16):
    got = d.to_numpy(np.uint8, raw.shape)
    return np.array_equal(got[:G], raw[:G]) and np.array_equal(got[G + nbytes:], raw[G + nbytes:]), got[G:G + nbytes]


@pytest.mark.gpu
@pytest.mark.parametrize("form", R.FORMS)
@pytest.mark.parametrize("dt,soa", [(np.float64, 8), (np.float32, 16)])
@pytest.mark.parametrize("which", ("a", "b", "c", "all"))
def test_gpu_rm_skipped_elements(gpu, form, dt, soa, which):
    """out-of-range indices skip elements: with far more elements than CTAs every CTA's persistent loop meets skipped elements at
    its first, middle and last iterations, in both buffers, singly and in runs, and whole calls skip everything.  The other
    elements are correct, skipped C slots keep their bits, the guard bands around every buffer stay intact."""
    rng = np.random.default_rng(23)
    M, N, K = 35, 9, 9 if form == "ac" else 35
    op = gpu.RmSoa(form, M, N, K, soa, dt, beta=1.0)
    ea, eb, ec = op.extents
    for E, frac in ((6007, 0.3), (6007, 0.97), (9, 1.0), (1, 1.0)):
        S = E
        skip = rng.random(E) < frac
        skip[:3] = True; skip[-3:] = True
        skip[E // 2:E // 2 + 40] = True                       # a run: consecutive iterations of many CTAs
        if frac < 1.0:
            skip[1] = False; skip[-2] = False
        idx = [rng.integers(0, S, E), rng.integers(0, S, E), rng.permutation(E)]
        bad = rng.integers(S, S + 5, E)
        bad[::7] = 0xFFFFFFFF
        for i, w in enumerate("abc"):
            if which in (w, "all"):
                idx[i] = np.where(skip, bad, idx[i])
        strides = [ea, eb, ec]
        a, b, c0 = rm_case(rng, op, dt, (S, S, S), strides)
        want = rm_expected(gpu, op, a, b, c0, E, strides, idx, (S, S, S))
        bufs = [guarded(gpu, x) for x in (a, b, c0)]
        di = upload(gpu, *[u32(i) for i in idx])
        G = 1 << 16
        op.execute_indexed(bufs[0][0].ptr + G, bufs[1][0].ptr + G, bufs[2][0].ptr + G, E, di[0], S, di[1], S, di[2], S)
        gpu.synchronize()
        gpu.check()
        for k, (d, raw) in enumerate(bufs):
            ok, body = bands_intact(d, raw, (a, b, c0)[k].nbytes)
            assert ok, ("guard band", k, E)
            if k < 2:
                assert np.array_equal(body, raw[G:G + (a, b)[k].nbytes]), "input written"
            else:
                assert np.array_equal(body.view(R.bits(c0).dtype), R.bits(want)), (E, frac, which)
        free(*[d for d, _ in bufs], *di)
    op.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("form", R.FORMS)
def test_gpu_rm_duplicate_c_indices(gpu, form):
    """repeated C slots: unspecified values there, but the guard bands stay intact and every other slot is correct"""
    rng = np.random.default_rng(24)
    dt, soa, M, N, K, E = np.float64, 8, 35, 9, 9 if form == "ac" else 35, 3000
    op = gpu.RmSoa(form, M, N, K, soa, dt, beta=1.0)
    strides = list(op.extents)
    S = E
    ic = rng.permutation(E)
    dup = rng.choice(E, 200, replace=False)
    ic[dup] = ic[dup[0]]
    ic[rng.choice(E, 50, replace=False)] = ic[7]
    idx = [rng.integers(0, S, E), rng.integers(0, S, E), ic]
    a, b, c0 = rm_case(rng, op, dt, (S, S, S), strides)
    vals, counts = np.unique(ic, return_counts=True)
    once = np.isin(ic, vals[counts == 1])
    want = rm_expected(gpu, op, a, b, c0, int(once.sum()), strides, [idx[0][once], idx[1][once], ic[once]], (S, S, S))
    bufs = [guarded(gpu, x) for x in (a, b, c0)]
    di = upload(gpu, *[u32(i) for i in idx])
    G = 1 << 16
    op.execute_indexed(bufs[0][0].ptr + G, bufs[1][0].ptr + G, bufs[2][0].ptr + G, E, di[0], S, di[1], S, di[2], S)
    gpu.synchronize()
    ok, body = bands_intact(bufs[2][0], bufs[2][1], c0.nbytes)
    assert ok
    C = body.view(dt)
    ec = strides[2]
    untouched = np.setdiff1d(np.arange(S), ic)
    for s in np.concatenate([vals[counts == 1], untouched]):
        assert np.array_equal(R.bits(C[s * ec:(s + 1) * ec]), R.bits(want[s * ec:(s + 1) * ec])), s
    free(*[d for d, _ in bufs], *di)
    op.destroy()
    gpu.check()


@pytest.mark.gpu
def test_gpu_large_offsets(gpu, ops):
    """slot * stride past 2^32 scalars (a 16 GiB fp32 buffer) for the SoA input and for C of rm_soa, and for C of csr_soa: the
    touched region equals the strided entry's result"""
    rng = np.random.default_rng(25)
    dt = np.float32
    stride = 1 << 22
    slot = (1 << 10) + 3                                         # slot * stride = 2^32 + 3 * 2^22 scalars
    dBig = gpu.DeviceBuffer((slot + 1) * stride * 4)
    off = slot * stride * 4
    for form in R.FORMS:
        op = gpu.RmSoa(form, 35, 9, 9, 16, dt, beta=1.0)
        ea, eb, ec = op.extents
        a, b, c0 = rm_case(rng, op, dt, (1, 1, 1), (ea, eb, ec))
        want = rm_expected(gpu, op, a, b, c0, 1, (ea, eb, ec), [None, None, None], (0, 0, 0))
        x = 0 if form == "ac" else 1
        di = upload(gpu, u32([slot]))[0]
        # the SoA input far away
        dBig.upload((a, b)[x], off)
        dP, dC = upload(gpu, (b, a)[x], c0)
        if form == "ac":
            op.execute_indexed(dBig, dP, dC, 1, a_index=di, a_slots=slot + 1, stride_a=stride)
        else:
            op.execute_indexed(dP, dBig, dC, 1, b_index=di, b_slots=slot + 1, stride_b=stride)
        gpu.synchronize()
        assert np.array_equal(R.bits(dC.to_numpy(dt, c0.shape)), R.bits(want)), form
        # C far away
        dBig.upload(c0, off)
        dA, dB = upload(gpu, a, b)
        op.execute_indexed(dA, dB, dBig, 1, c_index=di, c_slots=slot + 1, stride_c=stride)
        gpu.synchronize()
        assert np.array_equal(R.bits(dBig.to_numpy(dt, c0.shape, off)), R.bits(want)), form
        free(dP, dC, dA, dB, di)
        op.destroy()
    key = "tet4_4_stiffV_0_s"
    M, K, N, soa, _ = (int(v) for v in ops[key + "_shape"])
    op = gpu.CsrSoa(M, N, K, ops[key + "_rowptr"], ops[key + "_colidx"], ops[key + "_values"], soa, beta=1.0)
    Bv = rng.uniform(-1, 1, K * N * soa).astype(dt)
    C0 = rng.uniform(-1, 1, M * N * soa).astype(dt)
    dB, dC = upload(gpu, Bv, C0)
    op.execute(dB, dC, 1)
    gpu.synchronize()
    want = dC.to_numpy(dt, C0.shape)
    dBig.upload(C0, off)
    di = upload(gpu, u32([slot]))[0]
    op.execute_indexed(dB, dBig, 1, c_index=di, c_slots=slot + 1, stride_c=stride)
    gpu.synchronize()
    assert np.array_equal(R.bits(dBig.to_numpy(dt, C0.shape, off)), R.bits(want))
    free(dB, dC, di, dBig)
    op.destroy()
    gpu.check()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("rm", "csr"))
def test_gpu_stream_graph_and_launches(gpu, ops, kind):
    """on a non-default stream after an asynchronous upload of the index (stream order); captured into a graph whose index
    arrays are rewritten on the device between replays; exactly one launch per call"""
    rng = np.random.default_rng(26)
    dt, E, S = np.float64, 500, 600
    if kind == "rm":
        op = gpu.RmSoa("ac", 35, 9, 9, 8, dt, beta=1.0)
        ex, _, ec = op.extents
    else:
        key = "tet4_4_stiffV_0_d"
        M, K, N, soa, _ = (int(v) for v in ops[key + "_shape"])
        op = gpu.CsrSoa(M, N, K, ops[key + "_rowptr"], ops[key + "_colidx"], ops[key + "_values"], soa, beta=1.0)
        ex, ec = K * N * soa, M * N * soa
    X = rng.uniform(-1, 1, S * ex).astype(dt)
    P = rng.uniform(-1, 1, 81).astype(dt)
    c0 = rng.uniform(-1, 1, S * ec).astype(dt)
    dX, dP, dC = upload(gpu, X, P, c0)
    dXi, dCi = gpu.DeviceBuffer(E * 4), gpu.DeviceBuffer(E * 4)
    st = gpu.Stream()

    def run(xi, ci, stream):
        if kind == "rm":
            op.execute_indexed(dX, dP, dC, E, a_index=xi, a_slots=S, c_index=ci, c_slots=S, stride_b=0, stream=stream)
        else:
            op.execute_indexed(dX, dC, E, x_index=xi, x_slots=S, c_index=ci, c_slots=S, stream=stream)

    def expected(xi, ci):
        cx, _ = gather(X, ex, ex, xi)
        cc, _ = gather(c0, ec, ec, ci)
        d = upload(gpu, cx, cc)
        if kind == "rm":
            op.execute(d[0], dP, d[1], E, ex, 0, ec)
        else:
            op.execute(d[0], d[1], E, ex, ec)
        gpu.synchronize()
        want = c0.copy()
        scatter(want, ec, ec, ci, d[1].to_numpy(dt, cc.shape))
        free(*d)
        return want

    L = gpu.load()
    sets = [(rng.integers(0, S, E), rng.choice(S, E, replace=False)) for _ in range(3)]
    hx = [u32(s[0]) for s in sets]; hc = [u32(s[1]) for s in sets]
    # stream order: asynchronous uploads of the index, then the call, on one stream
    assert 0 == L.libxsmm_b200_memcpy_h2d_async(ctypes.c_void_p(dXi.ptr), hx[0].ctypes.data, E * 4, st.ptr)
    assert 0 == L.libxsmm_b200_memcpy_h2d_async(ctypes.c_void_p(dCi.ptr), hc[0].ctypes.data, E * 4, st.ptr)
    n0 = gpu.launch_count()
    run(dXi, dCi, st)
    assert gpu.launch_count() == n0 + 1
    st.synchronize()
    assert np.array_equal(R.bits(dC.to_numpy(dt, c0.shape)), R.bits(expected(*sets[0])))
    # graph: the replay reads the index arrays' current contents
    assert 0 == L.libxsmm_b200_graph_begin(st.ptr)
    run(dXi, dCi, st)
    g = L.libxsmm_b200_graph_end(st.ptr)
    assert g
    gpu.check()
    for k in (1, 2):
        dXi.upload(hx[k]); dCi.upload(hc[k]); dC.upload(c0)
        assert 0 == L.libxsmm_b200_graph_launch(ctypes.c_void_p(g), st.ptr)
        st.synchronize()
        assert np.array_equal(R.bits(dC.to_numpy(dt, c0.shape)), R.bits(expected(*sets[k]))), k
    L.libxsmm_b200_graph_destroy(ctypes.c_void_p(g))
    # one launch per call, with and without indices
    for xi, ci in ((dXi, dCi), (None, None), (dXi, None)):
        n0 = gpu.launch_count()
        run(xi, ci, None)
        assert gpu.launch_count() == n0 + 1
    gpu.synchronize()
    free(dX, dP, dC, dXi, dCi)
    st.destroy(); op.destroy()
    gpu.check()


# ---------------------------------------------------------------------------------------------------------------- GPU: csr_soa
def csr_handle(gpu, ops, key, group, beta):
    M, K, N, soa, _ = (int(v) for v in ops[key + "_shape"])
    if group == "cnames":
        op = gpu.CsrSoa(M, N, K, ops[key + "_colptr"], ops[key + "_rowidx"], ops[key + "_values"], soa, beta=beta, sparse="B", fmt="csc")
    else:
        op = gpu.CsrSoa(M, N, K, ops[key + "_rowptr"], ops[key + "_colidx"], ops[key + "_values"], soa, beta=beta,
                        sparse="A" if group == "names" else "B")
    ex = K * N * soa if group == "names" else M * K * soa
    return op, ex, M * N * soa, ops[key + "_values"].dtype


@pytest.mark.gpu
@pytest.mark.parametrize("group", ("names", "bnames", "cnames"))
@pytest.mark.parametrize("jit", ("baked", "generic"))
def test_gpu_csr_indexed_matches_gathered_strided(gpu, ops, group, jit, monkeypatch):
    """every fixture operator (A sparse, B sparse, CSC), baked and generic kernel: random gathers, a C permutation, skipped
    elements (x and c), identity and NULL indices, a four-face neighbour sum with beta = 1 and a half-size subset"""
    if jit == "generic":
        monkeypatch.setenv("LIBXSMM_B200_FSSPMDM_JIT", "0")
    rng = np.random.default_rng(27)
    for key in [str(n) for n in ops[group]][:4]:
        for beta in (0.0, 1.0):
            op, ex, ec, dt = csr_handle(gpu, ops, key, group, beta)
            assert op.is_baked == (jit == "baked"), key
            E, S = 700, 800
            X = rng.uniform(-1, 1, S * ex).astype(dt)
            c0 = rng.uniform(-1, 1, S * ec).astype(dt)
            dX, dC = upload(gpu, X, c0)

            def expected(xi, ci, cbase, n):
                run = (np.asarray(xi) < S) & (np.asarray(ci) < S)
                want = cbase.copy()
                if run.any():
                    cx, _ = gather(X, ex, ex, np.asarray(xi)[run]); cc, _ = gather(cbase, ec, ec, np.asarray(ci)[run])
                    d = upload(gpu, cx, cc)
                    op.execute(d[0], d[1], int(run.sum()), ex, ec)
                    gpu.synchronize()
                    scatter(want, ec, ec, np.asarray(ci)[run], d[1].to_numpy(dt, cc.shape))
                    free(*d)
                return want

            def indexed(xi, ci, n=E):
                di = upload(gpu, None if xi is None else u32(xi), None if ci is None else u32(ci))
                n0 = gpu.launch_count()
                op.execute_indexed(dX, dC, n, x_index=di[0], x_slots=S, c_index=di[1], c_slots=S)
                assert gpu.launch_count() == n0 + 1
                gpu.synchronize()
                free(*di)
                gpu.check()
                return dC.to_numpy(dt, c0.shape)

            xi, ci = rng.integers(0, S, E), rng.choice(S, E, replace=False)
            skip = rng.random(E) < 0.2
            xi_s = np.where(skip & (rng.random(E) < 0.5), S + 3, xi)
            ci_s = np.where(skip, np.where(rng.random(E) < 0.5, 0xFFFFFFFF, S), ci)
            for (a1, a2) in ((xi, ci), (xi_s, ci_s), (np.arange(E), np.arange(E))):
                dC.upload(c0)
                assert np.array_equal(R.bits(indexed(a1, a2)), R.bits(expected(a1, a2, c0, E))), (key, beta)
            dC.upload(c0)
            assert np.array_equal(R.bits(indexed(None, None)), R.bits(expected(np.arange(E), np.arange(E), c0, E))), (key, beta)
            if beta == 1.0:
                # neighbour sum: four face calls into the same C, repeating input indices
                dC.upload(c0)
                want = c0.copy()
                for f in range(4):
                    nb = rng.integers(0, S, E)
                    got = indexed(nb, None)
                    want = expected(nb, np.arange(E), want, E)
                assert np.array_equal(R.bits(got), R.bits(want)), key
                # subset: a sorted random half; the other slots keep their bits
                dC.upload(c0)
                sub = np.sort(rng.choice(S, S // 2, replace=False))
                got = indexed(sub, sub, len(sub))
                assert np.array_equal(R.bits(got), R.bits(expected(sub, sub, c0, len(sub)))), key
            free(dX, dC)
            op.destroy()


@pytest.mark.gpu
def test_gpu_csr_rejects_invalid_arguments_without_launching(gpu, ops):
    key = "tet4_4_stiffV_0_d"
    op, ex, ec, dt = csr_handle(gpu, ops, key, "names", 1.0)
    P = 4096
    n0 = gpu.launch_count()
    for args in ((-1, ex, ec, None, 0, None, 0), (2, -1, ec, None, 0, None, 0), (2, ex, -1, None, 0, None, 0),
                 (2, ex, ec, P, 0, None, 0), (2, ex, ec, None, 0, P, (1 << 32) + 1), (2, ex, ec - 1, None, 0, None, 0),
                 (2, ex, 0, None, 0, P, 2)):
        gpu.csr_soa_execute_indexed(op.handle, P, P, *args)
        assert gpu.last_error()[0] == -84, args
        gpu.clear_error()
    for X, C in ((None, P), (P, None)):
        gpu.csr_soa_execute_indexed(op.handle, X, C, 1, ex, ec, None, 0, None, 0)
        assert gpu.last_error()[0] == -84
        gpu.clear_error()
    gpu.csr_soa_execute_indexed(op.handle, None, None, 0, ex, ec, None, 0, None, 0)
    assert gpu.last_error()[0] == 0
    assert gpu.launch_count() == n0
    op.destroy()
