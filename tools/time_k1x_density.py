"""Developer tool: times the bf16 slicing pass (K1x, spmdm_slice_bf16x_kernel) of a 4096 x 4096 A at several densities with CUDA
events, back to back on one stream over a ring of five copies of A (160 MiB, more than L2), and prints one JSON line per density
with the card's name and power limit.

    python tools/time_k1x_density.py [reps] [density ...]
"""
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (q.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    densities = [float(x) for x in sys.argv[2:]] or [0.005, 0.01, 0.03, 0.10, 0.50]
    xs = importlib.import_module("libxsmm-1_b200")
    name, power = card()
    M = N = K = 4096
    st = xs.Stream()
    for d in densities:
        A, _, _ = xs.workloads.spmdm_inputs(M, 16, K, d, dtype="bf16", seed=1)
        ring = [xs.DeviceBuffer.from_numpy(A) for _ in range(5)]
        p = xs.Spmdm(M, N, K, 1)
        for i in range(5):
            p.create_slices(ring[i], "N", True, st)
        st.synchronize()
        e0, e1 = xs.Event(), xs.Event()
        e0.record(st)
        for i in range(reps):
            p.create_slices(ring[i % 5], "N", True, st)
        e1.record(st)
        st.synchronize()
        xs.check()
        us = e0.elapsed_ms(e1) / reps * 1e3
        print(json.dumps({"what": "K1x slicing pass, bf16 4096x4096, back to back", "density": d, "us": round(us, 2),
                          "GB/s": round(A.nbytes / us / 1e3, 1), "reps": reps, "gpu": name, "power_limit": power}), flush=True)
        p.destroy()
        for b in ring:
            b.free()


if __name__ == "__main__":
    main()
