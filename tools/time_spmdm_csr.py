"""Developer tool: times the spmdm slicing pass with A in CSR form (K1c, libxsmm_spmdm_createSparseSlice_csr_*_stream) against the
dense slicing pass of the same matrix, alone and as part of a whole slice + multiply step.  With --csc: the pass with A in CSC
form (K1t, libxsmm_spmdm_createSparseSlice_csc_*_stream) against K1c on the same A and against the dense transa = 'T' pass of the
K x M array, alone and as part of a step.

    python tools/time_spmdm_csr.py [--csc] [--reps 30] [--warmup 5] [--only C2,C1]

One JSON line per (workload, measurement).  Workloads: C2 (bf16 4096^3, 1 %) and C1 (fp32 2048^3, 10 %), default dispatch.
Each measurement enqueues `reps` back-to-back passes (or steps) on one stream after `warmup` untimed ones and records the
library's events between them; best and median are per pass.  The CSR arrays (C2: ~1 MB) and the dense A (C2: 33.6 MB) both fit
the 126 MB L2, so back-to-back passes read their input from L2 rather than HBM, as they do in a loop over one matrix; so do the
CSC arrays and the K x M array.
Algorithmic bytes of the CSR pass: read 4 (M + 1) + (4 + s) nnz (s = 2 for bf16, 4 for fp32), of the CSC pass 4 (K + 1) +
(4 + s) nnz; written by both: rowidx, colidx / values over nnz, slice_nnz and the auxiliary words the pass wrote (tcpk / tcoff,
and tcsp for bf16 with K % 128 == 0).  The card's name and power limit are read in the same run.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

# id: dtype, M = N = K, density
WORKLOADS = {"C2": ("bf16", 4096, 0.01), "C1": ("f32", 2048, 0.10)}


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:      # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def to_csr(A):
    keep = A.view(np.uint16 if A.dtype == np.uint16 else np.uint32) != 0
    rows, cols = np.nonzero(keep)
    row_ptr = np.zeros(A.shape[0] + 1, np.uint32)
    np.cumsum(np.bincount(rows, minlength=A.shape[0]), out=row_ptr[1:])
    return row_ptr, cols.astype(np.uint32), np.ascontiguousarray(A[rows, cols])


def to_csc(A):
    return to_csr(np.ascontiguousarray(A.T))          # the CSC arrays of A are the CSR arrays of A stored K x M


def timed(xs, st, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ev = [xs.Event() for _ in range(reps + 1)]
    ev[0].record(st)
    for i in range(reps):
        fn()
        ev[i + 1].record(st)
    st.synchronize()
    xs.check()
    ms = np.array([ev[i].elapsed_ms(ev[i + 1]) for i in range(reps)])
    for e in ev:
        e.destroy()
    return float(ms.min()), float(np.median(ms))


def run(xs, wid, reps, warmup, hbm_gbs, csc=False):
    dtype, n, density = WORKLOADS[wid]
    bf16 = dtype == "bf16"
    A, B, C0 = xs.workloads.spmdm_inputs(n, n, n, density, dtype=dtype, seed=1)
    row_ptr, col_idx, values = to_csr(A)
    nnz = len(col_idx)
    p = xs.Spmdm(n, n, n, 1)
    g = p.geometry
    st = xs.Stream()
    dA, dB, dC = xs.DeviceBuffer.from_numpy(A), xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer.from_numpy(C0)
    rp, ci, va = (xs.DeviceBuffer.from_numpy(x) for x in (row_ptr, col_idx, values))

    def csr_slice():
        p.create_slices_csr(rp, ci, va, nnz, bf16, st)

    def dense_slice():
        p.create_slices(dA, "N", bf16, st)

    def mult():
        p.compute(dB, dC, "N", "N", 0, bf16, st)

    if csc:
        col_ptr, row_idx, cvalues = to_csc(A)
        dAT = xs.DeviceBuffer.from_numpy(np.ascontiguousarray(A.T))
        cp, ri, cv = (xs.DeviceBuffer.from_numpy(x) for x in (col_ptr, row_idx, cvalues))
        extra_bufs = [dAT, cp, ri, cv]

        def csc_slice():
            p.create_slices_csc(cp, ri, cv, nnz, bf16, st)

        def dense_t_slice():
            p.create_slices(dAT, "T", bf16, st)

    out = []
    common = {"workload": wid, "dtype": dtype, "M": n, "N": n, "K": n, "density": density, "nnz": nnz, "launches": reps}
    s = 2 if bf16 else 4
    ns = g["mb"] * g["kb"]
    read = 4 * (n + 1) + (4 + s) * nnz                        # M = K: the same for the CSC pass
    aux = 4 if bf16 else 2                                    # tcpk / tcoff per entry
    sp = 4 if (bf16 and n % 128 == 0) else 0                  # tcsp per entry
    written = 2 * ns * (g["bm"] + 1) + (2 + 4 + aux + sp) * nnz + 4 * ns
    sparse_bytes = {"bytes_read": read, "bytes_written": written}
    if csc:
        plan = (("csc_slice", csc_slice, sparse_bytes),
                ("csr_slice", csr_slice, sparse_bytes),
                ("dense_t_slice", dense_t_slice, {"bytes_read": n * n * s}),
                ("csc_step", lambda: (csc_slice(), mult()), {}),
                ("csr_step", lambda: (csr_slice(), mult()), {}),
                ("dense_t_step", lambda: (dense_t_slice(), mult()), {}))
    else:
        plan = (("csr_slice", csr_slice, sparse_bytes),
                ("dense_slice", dense_slice, {"bytes_read": n * n * s}),
                ("csr_step", lambda: (csr_slice(), mult()), {}),
                ("dense_step", lambda: (dense_slice(), mult()), {}))
    for name, fn, extra in plan:
        best, med = timed(xs, st, fn, reps, warmup)
        r = dict(common, measurement=name, best_us=round(best * 1e3, 2), median_us=round(med * 1e3, 2))
        if name.endswith("step"):
            r["compute_kernel"] = xs.last_compute_kernel()
        r.update(extra)
        if "bytes_read" in extra:
            tot = extra["bytes_read"] + extra.get("bytes_written", 0)
            r["gbs_best"] = round(tot / best / 1e6, 1)
            r["hbm_gbs"] = hbm_gbs
        out.append(r)
    for d in [dA, dB, dC, rp, ci, va] + (extra_bufs if csc else []):
        d.free()
    st.destroy()
    p.destroy()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--only", default=None)
    ap.add_argument("--csc", action="store_true", help="time the CSC pass against the CSR and the dense transa = 'T' passes")
    args = ap.parse_args()
    assert args.reps >= 20
    xs = importlib.import_module("libxsmm-1_b200")
    xs.require_gpu()
    hbm_gbs, _ = bench.peaks()
    name, power = card()
    for wid in (args.only.split(",") if args.only else WORKLOADS):
        for r in run(xs, wid, args.reps, args.warmup, hbm_gbs, args.csc):
            r.update({"card": name, "power_limit": power})
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
