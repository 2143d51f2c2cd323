"""Generates tests/golden/operators_pyfr.npz by RUNNING THE UNMODIFIED REFERENCE (oracle/_ref) on every operator shipped under
/root/reference/samples/pyfr/mats (150 coordinate-format files, p1..p6 x hex/pri/quad/tet/tri x m0/m3/m6/m132/m460).

    python tests/golden/make_pyfr_golden.py

Stored: every operator in coordinate form (so that the tests run where /root/reference does not exist), the branch the
reference's libxsmm_dfsspmdm_create took for it (sparse_reg JIT or dense SMM; N = ld = 16), and -- for a spread of 30
operators, including the largest ones -- seeded B / C0 panels of 16 columns with the reference's outputs for beta = 0 and
beta = 1.  The remaining operators are checked against the CPU oracle, which these same outputs pin.  To keep the file below
1 MB the panels are not stored (tests/test_pyfr_operators.py draws them again from the same seeds) and of each output only
every second element (row-major) is."""
import glob
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
REF_MATS = "/root/reference/samples/pyfr/mats"


def main():
    pyoracle.build_ref("avx2")
    ref = pyoracle.Ref()
    files = sorted(glob.glob(os.path.join(REF_MATS, "p*", "*", "*-sp.mtx")))
    names, shapes, offs, rows, cols, vals, branch = [], [], [0], [], [], [], []
    ops = []
    for f in files:
        a = w.read_mtx(f)
        r, c = np.nonzero(a)
        names.append(os.path.relpath(f, REF_MATS)[:-len("-sp.mtx")])
        shapes.append(a.shape)
        rows.append(r.astype(np.uint16)); cols.append(c.astype(np.uint16)); vals.append(a[r, c])
        offs.append(offs[-1] + len(r))
        B = np.zeros((a.shape[1], 16)); C = np.zeros((a.shape[0], 16))
        sparse, _, _ = ref.fsspmdm(a, B, C, 0.0, panel=16)
        branch.append(bool(sparse))
        ops.append(a)
    # outputs: every fifth operator plus the six with the most nonzeros / widest K
    order = sorted(range(len(ops)), key=lambda i: (-ops[i].shape[1], -np.count_nonzero(ops[i])))
    picked = sorted(set(list(range(0, len(ops), 6)) + order[:5]))
    out = {}
    for i in picked:
        a = ops[i]
        rng = np.random.default_rng(100 + i)
        B = rng.uniform(-1.0, 1.0, (a.shape[1], 16)); C0 = rng.uniform(-1.0, 1.0, (a.shape[0], 16))
        for beta in (0.0, 1.0):
            C = C0.copy()
            ref.fsspmdm(a, B, C, beta, panel=16)
            out["out%d_%d" % (int(beta), i)] = C.ravel()[::2].copy()
    np.savez_compressed(os.path.join(HERE, "operators_pyfr.npz"), names=np.array(names), shapes=np.array(shapes, np.int32), offsets=np.array(offs, np.int64),
                        rows=np.concatenate(rows), cols=np.concatenate(cols), vals=np.concatenate(vals), ref_sparse_branch=np.array(branch),
                        picked=np.array(picked, np.int32), **out)
    print("wrote operators_pyfr.npz: %d operators, %d nonzeros, %d with reference outputs; sparse branch taken for %d" % (len(ops), offs[-1], len(picked), sum(branch)))


if __name__ == "__main__":
    main()
