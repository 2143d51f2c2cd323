"""Developer tool: times the slicing and compute kernels of one spmdm workload with CUDA events
(ring of inputs larger than L2, like bench.py) and prints one line.

    python tools/time_spmdm.py c2 [reps]
"""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "c2"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    xs = importlib.import_module("libxsmm-1_b200")
    wl = bench.WORKLOADS[name]
    gen = bench.run_spmdm_gpu(xs, wl, reps, 3, want_e2e=False)
    assert next(gen) == "ready"
    r = next(gen)
    for _ in gen:
        pass
    p = r["parts"]
    print("%s: step %.1f us  slice %.1f us (%.0f GB/s)  compute %.1f us (%.0f GB/s, %.0f GFLOP/s)" % (
        name, r["total_ms"] / reps * 1e3, p["slice_ms"] * 1e3,
        p["slice_bytes"] / p["slice_ms"] / 1e6, p["compute_ms"] * 1e3, p["compute_bytes"] / p["compute_ms"] / 1e6,
        r["flops"] / p["compute_ms"] / 1e6))


def back_to_back(name, reps):
    """compute kernel alone, `reps` launches back to back on one stream (no events in between)."""
    xs = importlib.import_module("libxsmm-1_b200")
    wl = bench.WORKLOADS[name]
    bf16 = wl["dtype"] == "bf16"
    A, B, C0 = bench.spmdm_host_inputs(xs, wl)
    p = xs.Spmdm(wl["M"], wl["N"], wl["K"], 1)
    nsets = 3
    ring = [(xs.DeviceBuffer.from_numpy(A), xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer(C0.nbytes)) for _ in range(nsets)]
    st = xs.Stream()
    ta, tb, tc = wl["trans"]
    p.create_slices(ring[0][0], ta, bf16, st)
    for i in range(3):
        p.compute(ring[i % nsets][1], ring[i % nsets][2], tb, tc, wl["beta"], bf16, st)
    st.synchronize()
    e0, e1 = xs.Event(), xs.Event()
    e0.record(st)
    for i in range(reps):
        p.compute(ring[i % nsets][1], ring[i % nsets][2], tb, tc, wl["beta"], bf16, st)
    e1.record(st)
    st.synchronize()
    t_c = e0.elapsed_ms(e1) / reps * 1e3
    e0.record(st)
    for i in range(reps):
        p.create_slices(ring[i % nsets][0], ta, bf16, st)
    e1.record(st)
    st.synchronize()
    t_s = e0.elapsed_ms(e1) / reps * 1e3
    import time
    t0 = time.perf_counter()
    for i in range(reps):
        p.compute(ring[i % nsets][1], ring[i % nsets][2], tb, tc, wl["beta"], bf16, st)
    t_host = (time.perf_counter() - t0) / reps * 1e6
    st.synchronize()
    xs.check()
    print("%s back-to-back: compute %.1f us/launch, slice %.1f us/launch, host enqueue %.1f us/launch" % (name, t_c, t_s, t_host))


if __name__ == "__main__":
    main()
    back_to_back(sys.argv[1] if len(sys.argv) > 1 else "c2", int(sys.argv[2]) if len(sys.argv) > 2 else 20)
