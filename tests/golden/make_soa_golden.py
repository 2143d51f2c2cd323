"""Generates tests/golden/csr_soa.npz by RUNNING THE UNMODIFIED REFERENCE (oracle/_ref): libxsmm_create_xcsr_soa kernels
(src/generator_spgemm_csr_asparse_soa.c, _csr_bsparse_soa.c) and libxsmm_create_xcsc_soa kernels (_csc_bsparse_soa.c) on real EDGE operators shipped under /root/reference/samples/edge/mats
(tet4_<order>_stiffV / stiffT / fluxN, CSR files) and two synthetic ones (a dense operator, one with empty rows), for
double (SoA width 8) and float (16), beta = 0 and 1, two mesh elements each -- driven like samples/edge/asparse_srsoa.c.

    python tests/golden/make_soa_golden.py

(The largest stiffness operators, e.g. tet4_6_stiffV_2 with 1680 nonzeros and beta = 1, make the reference's generator run
past its 128 KiB code buffer -- "stack smashing detected" -- so the order-6 case here is the smaller stiffT_0.)

To keep the file below 1 MB the dense inputs are not stored -- tests/test_csr_soa.py (soa_inputs) draws them again from the
same stream, so the order of the draws below is part of the fixture; <case>_probe holds their first values to tell a changed
stream from a wrong result -- and of each output only every third element (row-major) is.
"""
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyoracle  # noqa: E402

w = importlib.import_module("libxsmm-1_b200.workloads")
MATS = "/root/reference/samples/edge/mats"


def csr_of(a):
    rp, ci, va = [0], [], []
    for i in range(a.shape[0]):
        nz = np.nonzero(a[i])[0]
        ci += list(nz); va += list(a[i, nz]); rp.append(len(ci))
    return np.array(rp, np.uint32), np.array(ci, np.uint32), np.array(va, a.dtype)


def main():
    pyoracle.build_ref("avx2")
    ref = pyoracle.Ref()
    assert ref.soa_width(np.float64) == 8, "generate on an AVX-512 host (SoA width 8 / 16)"
    rng = np.random.default_rng(31)
    ops = []
    for f in ("tet4_4_stiffV_0_csr.mtx", "tet4_5_stiffT_1_csr.mtx", "tet4_3_fluxN_5_csr.mtx", "tet4_6_stiffT_0_csr.mtx"):
        ops.append((f[:-8], w.read_mtx(os.path.join(MATS, f))))
    ops.append(("dense_12x12", rng.uniform(-1, 1, (12, 12))))
    sp = np.where(rng.random((20, 28)) < 0.15, rng.uniform(-1, 1, (20, 28)), 0.0); sp[4, :] = 0; sp[19, :] = 0
    ops.append(("synthetic_empty_rows", sp))
    out, names = {}, []
    for name, a64 in ops:
        for dt in (np.float64, np.float32):
            a = a64.astype(dt)
            rp, ci, va = csr_of(a)
            M, K = a.shape
            N, E = 9, 2
            soa = ref.soa_width(dt)
            B = rng.uniform(-1, 1, (E, K, N, soa)).astype(dt); C0 = rng.uniform(-1, 1, (E, M, N, soa)).astype(dt)
            key = "%s_%s" % (name, "d" if dt == np.float64 else "s")
            names.append(key)
            out[key + "_shape"] = np.array([M, K, N, soa, E], np.int32)
            out[key + "_rowptr"], out[key + "_colidx"], out[key + "_values"] = rp, ci, va
            out[key + "_probe"] = np.concatenate([B.ravel()[:4], C0.ravel()[:4]]).astype(np.float64)
            for beta in (0.0, 1.0):
                C = C0.copy()
                ref.csr_soa(rp, ci, va, B, C, N, beta)
                out[key + "_out%d" % int(beta)] = C.ravel()[::3].copy()
    # ---- B sparse (descriptor lda > 0, ldb = 0; samples/edge/bsparse_srsoa.c): 9 quantities x basis functions, right-multiplied
    #      by a stiffness / flux operator (K x N)
    bnames = []
    for f in ("tet4_4_stiffV_0_csr.mtx", "tet4_5_stiffT_1_csr.mtx", "tet4_4_fluxN_3_csr.mtx", "tet4_4_fluxT_2_csr.mtx"):
        b64 = w.read_mtx(os.path.join(MATS, f))
        for dt in (np.float64, np.float32):
            b = b64.astype(dt)
            rp, ci, va = csr_of(b)
            K, N = b.shape
            M, E = 9, 2
            soa = ref.soa_width(dt)
            A = rng.uniform(-1, 1, (E, M, K, soa)).astype(dt); C0 = rng.uniform(-1, 1, (E, M, N, soa)).astype(dt)
            key = "bsp_%s_%s" % (f[:-8], "d" if dt == np.float64 else "s")
            bnames.append(key)
            out[key + "_shape"] = np.array([M, K, N, soa, E], np.int32)
            out[key + "_rowptr"], out[key + "_colidx"], out[key + "_values"] = rp, ci, va
            out[key + "_probe"] = np.concatenate([A.ravel()[:4], C0.ravel()[:4]]).astype(np.float64)
            for beta in (0.0, 1.0):
                C = C0.copy()
                ref.csr_soa_bsparse(rp, ci, va, A, C, N, beta)
                out[key + "_out%d" % int(beta)] = C.ravel()[::3].copy()
    # ---- B sparse in CSC (libxsmm_create_xcsc_soa; samples/edge/bsparse_scsoa.c and its *_csc.mtx operators); one synthetic
    #      operator with UNSORTED row indices inside the columns and trailing empty columns
    cnames = []
    cops = [(f[:-8], w.read_mtx(os.path.join(MATS, f)), False) for f in ("tet4_4_stiffV_1_csc.mtx", "tet4_5_stiffT_1_csc.mtx", "tet4_4_fluxN_7_csc.mtx")]
    syn = np.where(rng.random((24, 30)) < 0.25, rng.uniform(-1, 1, (24, 30)), 0.0); syn[:, 26:] = 0; syn[:, 4] = 0
    cops.append(("synthetic_unsorted", syn, True))
    for name, b64, shuffle in cops:
        for dt in (np.float64, np.float32):
            b = b64.astype(dt)
            K, N = b.shape
            cp, ri, va = [0], [], []
            for n in range(N):
                ks = list(np.nonzero(b[:, n])[0])
                if shuffle:
                    rng.shuffle(ks)
                ri += ks; va += [b[k, n] for k in ks]; cp.append(len(ri))
            cp, ri, va = np.array(cp, np.uint32), np.array(ri, np.uint32), np.array(va, dt)
            M, E = 9, 2
            soa = ref.soa_width(dt)
            A = rng.uniform(-1, 1, (E, M, K, soa)).astype(dt); C0 = rng.uniform(-1, 1, (E, M, N, soa)).astype(dt)
            key = "csc_%s_%s" % (name, "d" if dt == np.float64 else "s")
            cnames.append(key)
            out[key + "_shape"] = np.array([M, K, N, soa, E], np.int32)
            out[key + "_colptr"], out[key + "_rowidx"], out[key + "_values"] = cp, ri, va
            out[key + "_probe"] = np.concatenate([A.ravel()[:4], C0.ravel()[:4]]).astype(np.float64)
            for beta in (0.0, 1.0):
                C = C0.copy()
                ref.csc_soa(cp, ri, va, A, C, N, beta)
                out[key + "_out%d" % int(beta)] = C.ravel()[::3].copy()
    np.savez_compressed(os.path.join(HERE, "csr_soa.npz"), names=np.array(names), bnames=np.array(bnames), cnames=np.array(cnames), **out)
    print("wrote csr_soa.npz:", len(names), "A-sparse,", len(bnames), "B-sparse CSR and", len(cnames), "B-sparse CSC cases")


if __name__ == "__main__":
    main()
