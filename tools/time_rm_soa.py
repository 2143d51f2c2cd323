"""Developer tool: times the dense SoA kernels (libxsmm_b200_[sd]rm_{ac,bc}_soa_*) on the EDGE-style workloads of DESIGN.md section 8.

    python tools/time_rm_soa.py [--reps 30] [--warmup 5] [--fma-peaks fma_peak.json] [--only W1,W2]

One JSON line per workload.  Each workload's operands and C exceed the 126 MB L2 many times over (2.4 to 4 GB), so every launch
streams from HBM.  The library's events are recorded between back-to-back launches after the warm-up; best and median are per
launch.  Floors: algorithmic bytes over the HBM figure of bench.peaks(), and flops over the FMA peak measured by tools/fma_peak.cu
(--fma-peaks: the probe's output; without it the FMA floor is not reported).  The card's name and power limit are read in the
same run.
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

# id: form, dtype, (M, N, K, soa), plain operand per element?, beta, elements
WORKLOADS = {
    "W1": ("ac", np.float64, (35, 9, 9, 8), True, 1.0, 65536),
    "W1s": ("ac", np.float32, (35, 9, 9, 16), True, 1.0, 65536),
    "W2": ("bc", np.float64, (35, 9, 35, 8), False, 1.0, 65536),
    "W2s": ("bc", np.float32, (35, 9, 35, 16), False, 1.0, 65536),
    "W3": ("bc", np.float64, (84, 9, 84, 8), False, 1.0, 16384),
    "W1-direct": ("ac", np.float64, (35, 9, 9, 8), True, 1.0, 65536),     # A's element stride one scalar past 16-byte alignment
}


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:      # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def run(xs, wid, reps, warmup, fma_peaks, hbm_gbs):
    form, dt, (M, N, K, soa), per_elem, beta, E = WORKLOADS[wid]
    es = np.dtype(dt).itemsize
    xa = M * K * soa if form == "ac" else M * K               # dense extents of one element's a, b, C
    xb = K * N if form == "ac" else K * N * soa
    xc = M * N * soa
    sa = xa if (form == "ac" or per_elem) else 0
    sb = xb if (form == "bc" or per_elem) else 0
    if wid.endswith("direct"):
        sa += 1
    rng = np.random.default_rng(1)
    bufs = []
    for n in (max(E - 1, 0) * sa + xa, max(E - 1, 0) * sb + xb, E * xc):
        d = xs.DeviceBuffer(n * es)
        chunk = 1 << 24
        for o in range(0, n, chunk):
            d.upload(rng.uniform(-1, 1, min(chunk, n - o)).astype(dt), o * es)
        bufs.append(d)
    op = xs.RmSoa(form, M, N, K, soa, dt, beta=beta)
    st = xs.Stream()
    for _ in range(warmup):
        op.execute(bufs[0], bufs[1], bufs[2], E, sa, sb, xc, st)
    kernel = xs.last_compute_kernel()
    ev = [xs.Event() for _ in range(reps + 1)]
    ev[0].record(st)
    for i in range(reps):
        op.execute(bufs[0], bufs[1], bufs[2], E, sa, sb, xc, st)
        ev[i + 1].record(st)
    st.synchronize()
    xs.check()
    ms = np.array([ev[i].elapsed_ms(ev[i + 1]) for i in range(reps)])
    nbytes = E * es * ((xa if sa else 0) + (xb if sb else 0) + xc * (2 if beta else 1)) + es * ((0 if sa else xa) + (0 if sb else xb))
    flops = 2.0 * M * N * K * soa * E
    best, med = float(ms.min()), float(np.median(ms))
    hbm_floor = nbytes / (hbm_gbs * 1e6)
    res = {"workload": wid, "form": form, "dtype": np.dtype(dt).name, "M": M, "N": N, "K": K, "soa": soa, "elements": E,
           "plain_operand": "per element" if per_elem else "shared", "beta": beta, "kernel": kernel, "launches": reps,
           "best_ms": round(best, 4), "median_ms": round(med, 4), "bytes": nbytes, "flops": flops,
           "gbs_best": round(nbytes / best / 1e6, 1), "tflops_best": round(flops / best / 1e9, 3),
           "hbm_gbs": hbm_gbs, "hbm_floor_ms": round(hbm_floor, 4), "frac_hbm_floor": round(hbm_floor / best, 3)}
    if fma_peaks:
        peak = fma_peaks["dfma" if dt == np.float64 else "ffma"]
        fma_floor = flops / (peak * 1e9)
        res.update({"fma_peak_tflops": peak, "fma_floor_ms": round(fma_floor, 4), "frac_fma_peak": round(fma_floor / best, 3),
                    "frac_floor": round(max(hbm_floor, fma_floor) / best, 3)})
    op.destroy(); st.destroy()
    for e in ev:
        e.destroy()
    for d in bufs:
        d.free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--fma-peaks", default=None, help="output of tools/fma_peak.cu (JSON lines)")
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    assert args.reps >= 20
    xs = importlib.import_module("libxsmm-1_b200")
    xs.require_gpu()
    peaks = None
    if args.fma_peaks:
        peaks = {}
        for line in open(args.fma_peaks):
            r = json.loads(line)
            if "probe" in r:
                peaks[r["probe"]] = r["tflops"]
    hbm_gbs, hbm_src = bench.peaks()
    name, power = card()
    for wid in (args.only.split(",") if args.only else WORKLOADS):
        res = run(xs, wid, args.reps, args.warmup, peaks, hbm_gbs)
        res.update({"hbm_source": hbm_src, "card": name, "power_limit": power})
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
