#!/usr/bin/env python
"""bench.py -- throughput of the sparse-A x dense-B hot path on B200 (one JSON line on stdout).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|c3|c4|c5] [--impl b200|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], "C2"): libxsmm_spmdm, bf16 inputs / fp32 accumulate,
M = K = N = 4096, A 99 % zeros, beta = 0.  One STEP = one whole multiply the way samples/spmdm/spmdm.c:88-111
performs it: all createSparseSlice blocks (dense A -> CSR slices), then all compute blocks (C = A.B).
metric = effective GFLOP/s = 2.nnz.N / t  (SURVEY.md section 8d).

  value     inputs resident in HBM, stream entries (libxsmm_spmdm_exec_stream), CUDA events on the launch
            stream, K steps back to back.  Every step uses a different copy of A/B/C out of a ring larger
            than L2, so nothing is served from cache ("inputs larger than L2").
  e2e       the same multiply through the host-pointer C-ABI call (libxsmm_spmdm_exec_host): page-locked host
            A, B in, C out, copies inside the timed region.
  roofline  the dominant kernel (spmdm compute): algorithmic bytes / its mean duration from CUDA events
            recorded around every launch inside the timed region, against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, OpenMP over block ids like the sample) on this host.

Multi-GPU (N > 1, launched by torchrun, one rank per GPU): the path shards by N-column panels with A
replicated and NO collective on the data path (SURVEY.md section 8e).  torch.distributed (NCCL) is used for
the barriers and the max-over-ranks of the device time only.
  * headline (C2): BASELINE.json names no sharding for it -- every rank multiplies its own 4096-column panel
    (replicas, WEAK scaling: global problem M = K = 4096, N = 4096.N_gpus).
  * `column_sharded` (C3: dfsspmdm N = 2^20, C5: sfsspmdm N = 2^24): the configs BASELINE.json names as column
    sharded.  ONE global problem, rank r owns columns [r.N/g, (r+1).N/g) (libxsmm-1_b200/sharding.py), STRONG
    scaling; reported device-resident and end to end at every N, so that the 1/2/4/8 curve can be read off.

--impl reference times the reference CPU implementation on the same workload (rank 0 only).

--dump-outputs DIR writes what the last timed step of the headline workload computed (C) as DIR/<name>.npy, so that two
builds can be compared output for output: the inputs are seeded, identical from run to run for the same arguments.  An output
larger than DUMP_BYTES is written as a fixed sample of its elements, see dump_outputs().  With N > 1 only rank 0 writes: its
own C for the replicated C2, its own column panel of C for the column-sharded fsspmdm workloads.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: kind, parameters (SURVEY.md section 8d)
    "c1": dict(kind="spmdm", M=2048, N=2048, K=2048, density=0.10, dtype="f32", trans="NNN", beta=0.0,
               desc="spmdm fp32 M=N=K=2048, A 90% zeros, N/N/N, beta=0"),
    "c2": dict(kind="spmdm", M=4096, N=4096, K=4096, density=0.01, dtype="bf16", trans="NNN", beta=0,
               desc="spmdm bf16-in/fp32-acc M=K=N=4096, A 99% zeros, N/N/N, beta=0"),
    "c3": dict(kind="fsspmdm", M=150, K=64, density=0.30, n_unique=8, dtype="f64", N=1 << 20, beta=0.0,
               desc="dfsspmdm fp64 150x64 30% dense (8 distinct values), N=2^20 columns, beta=0"),
    "c4": dict(kind="spmdm", M=2048, N=2048, K=2048, density=0.50, dtype="f32", trans="NNN", beta=0.0,
               desc="spmdm fp32 M=N=K=2048, A 50% zeros, N/N/N, beta=0"),
    "c4-tnt": dict(kind="spmdm", M=2048, N=2048, K=2048, density=0.50, dtype="f32", trans="TNT", beta=0.0,
                   desc="spmdm fp32 2048^3 50%, transA/transC (weight update)"),
    "c4-ntn": dict(kind="spmdm", M=2048, N=2048, K=2048, density=0.50, dtype="f32", trans="NTN", beta=0.0,
                   desc="spmdm fp32 2048^3 50%, transB (backprop)"),
    "c5": dict(kind="fsspmdm", M=150, K=64, density=0.30, n_unique=8, dtype="f32", N=1 << 24, beta=0.0,
               desc="sfsspmdm fp32 150x64 30% dense, N=2^24 columns, beta=0"),
    # dense float operator: the branch where the reference itself applies the operator through its dense SMM kernel; here the
    # tcgen05 kernel K4f (not a BASELINE.json config; reported because the north star names that branch)
    "c5-dense": dict(kind="fsspmdm", M=150, K=64, density=1.0, n_unique=None, dtype="f32", N=1 << 22, beta=0.0,
                     desc="sfsspmdm fp32 150x64 fully dense operator, N=2^22 columns, beta=0"),
    "c5-dense-b1": dict(kind="fsspmdm", M=150, K=64, density=1.0, n_unique=None, dtype="f32", N=1 << 22, beta=1.0,
                        desc="sfsspmdm fp32 150x64 fully dense operator, N=2^22 columns, beta=1"),
    "c3-b1": dict(kind="fsspmdm", M=150, K=64, density=0.30, n_unique=8, dtype="f64", N=1 << 20, beta=1.0,
                  desc="dfsspmdm fp64 150x64 30% dense (8 distinct values), N=2^20 columns, beta=1"),
    # real PyFR operators (reference samples/pyfr/mats/p4/hex/m0-sp.mtx, p4/tet/m6-sp.mtx; the matrices travel as the
    # committed fixtures tests/golden/pyfr_*.npz and are handed to the library as MatrixMarket files: create_mtx)
    "c3-hex": dict(kind="fsspmdm", fixture="pyfr_p4_hex_m0", M=150, K=125, dtype="f64", N=1 << 20, beta=0.0,
                   desc="dfsspmdm fp64 PyFR p4/hex/m0-sp (150x125, 750 nnz, 5 distinct values), N=2^20 columns, beta=0"),
    "c3-tet": dict(kind="fsspmdm", fixture="pyfr_p4_tet_m6", M=105, K=60, dtype="f64", N=1 << 20, beta=0.0,
                   desc="dfsspmdm fp64 PyFR p4/tet/m6-sp (105x60, 50% dense, 202 distinct values: reference dense branch), N=2^20 columns, beta=0"),
}
# CSR x dense SoA at EDGE sizes (SURVEY.md section 8f-1): the order-4 tetrahedral stiffness operator of the reference's EDGE proxy
# (samples/edge/mats/tet4_4_stiffV_0: 35 x 35, 108 nonzeros; fixture tests/golden/csr_soa.npz), 9 quantities x 8 fused runs per
# element ([35][9][8] doubles = 20 KB per tensor), 2^16 mesh elements per step
WORKLOADS["soa"] = dict(kind="soa", case="tet4_4_stiffV_0_d", dtype="f64", elements=1 << 16, beta=1.0,
                        desc="dcsr_soa EDGE tet4 order 4 stiffV_0 (35x35, 108 nnz) x [35][9][8] tensors, 65536 elements, beta=1")
WORKLOADS["soa-b"] = dict(kind="soa", case="bsp_tet4_4_stiffV_0_d", sparse="B", dtype="f64", elements=1 << 16, beta=1.0,
                          desc="dcsr_soa, B sparse: [9][35][8] tensors x EDGE tet4 order 4 stiffV_0 (35x35, 108 nnz), 65536 elements, beta=1")
FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 74.4: 148 SMs x 128 FMA lanes at the 1965 MHz the CUDA-core kernels run at (nominal; no measured figure in MEASURED_PEAKS.json)
L2_BYTES = 126 << 20
DUMP_BYTES = 48 << 20      # --dump-outputs writes at most this much (a dump stays below 64 MB)


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def tensor_pipe_info(res):
    """The tensor-core kernels multiply the DENSIFIED slices: their own pipe utilisation, for the reader -- the roofline
    of the line stays the algorithmic (HBM) one of the sparse product.  bf16: one kind::f16 MMA per product; fp32: three
    kind::tf32 MMAs (3xTF32) at half the bf16 rate."""
    name = res.get("kernel_name", "")
    if not name.startswith("spmdm_compute_tc") or not res.get("dense_flops"):
        return None
    tp, tsrc = tensor_peak()
    bf16 = name.startswith("spmdm_compute_tc16")
    ex = (1.0 if bf16 else 3.0) * res["dense_flops"] / (res["kernel_ms"] * 1e9)
    if name.startswith("spmdm_compute_tc16s"):
        # 2:4 structured-sparse MMAs (tcgen05.mma.sp): the tensor core skips half of every group of four k, so the dense-EQUIVALENT
        # rate is held against twice the dense bf16 peak (the instruction itself was measured at 1.94 x, tools/umma_probe/probe_sp_rate.cu)
        return {"executed_dense_equivalent_tflops": ex, "peak_tflops": 2.0 * tp, "frac": ex / (2.0 * tp), "peak_source": tsrc + " x 2 (2:4 structured-sparse instruction)",
                "note": "kind::f16 structured-sparse MMAs over the compressed A tile (two kept elements of every four k); dense-equivalent, not algorithmic, flops"}
    peak = tp if bf16 else 0.5 * tp
    return {"executed_dense_tflops": ex, "peak_tflops": peak, "frac": ex / peak, "peak_source": tsrc + ("" if bf16 else " x 0.5 (tf32)"),
            "note": ("kind::f16 MMAs" if bf16 else "3 x kind::tf32 MMAs") + " over the densified A tile; executed, not algorithmic, flops"}


def bind_to_gpu_numa_node(local_rank):
    """N > 1 ranks share one host: run this rank (and first-touch its page-locked buffers) on the CPUs NVML reports as
    local to its GPU, what `numactl` would do for a multi-GPU job.  Best effort; returns a note for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            return "rank bound to %d GPU-local CPUs" % len(use)
        return "GPU-local CPUs = allowed set (%d)" % len(allowed)
    except Exception as ex:
        return "not bound (%s)" % type(ex).__name__


def tensor_peak():
    """dense bf16 TFLOP/s (cuBLAS, burst: the kernel is timed alone) for the tensor-core kernels' own utilisation figure."""
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops)"
    except Exception:
        return 2250.0, "fallback (nominal dense bf16)"


def ncu_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full summary, or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return t.get(workload, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons of one GPU, sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], threading.Event(), None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        busy = sorted(sm)[len(sm) // 2:]          # upper half = samples taken under load
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# workload construction
# ------------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def spmdm_host_inputs(xs, wl, seed=1):
    t = wl["trans"]
    return xs.workloads.spmdm_inputs(wl["M"], wl["N"], wl["K"], wl["density"], dtype=wl["dtype"], seed=seed,
                                     transa=t[0], transb=t[1], transc=t[2])


def spmdm_bytes(wl, geo, nnz):
    sA = sB = 2 if wl["dtype"] == "bf16" else 4
    M, N, K = wl["M"], wl["N"], wl["K"]
    ptr = 2 * geo["mb"] * geo["kb"] * (geo["bm"] + 1)
    beta_nz = 1 if float(wl["beta"]) != 0.0 else 0
    compute = sB * K * N + 4 * M * N * (1 + beta_nz) + 6 * nnz + ptr
    slicing = sA * M * K + 6 * nnz + ptr
    return slicing, compute


def fs_bytes(wl, N):
    s = 8 if wl["dtype"] == "f64" else 4
    return s * N * (wl["K"] + wl["M"] * (2 if float(wl["beta"]) == 1.0 else 1))


def fs_operator(xs, wl):
    if wl.get("fixture"):
        return np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", wl["fixture"] + ".npz"))["a"],
                                    np.float64 if wl["dtype"] == "f64" else np.float32)
    return xs.workloads.fsspmdm_operator(wl["M"], wl["K"], wl["density"], wl["n_unique"],
                                         np.float64 if wl["dtype"] == "f64" else np.float32, seed=1)


def run_soa_gpu(xs, wl, steps, warmup, dump=False):
    d = np.load(os.path.join(ROOT, "tests", "golden", "csr_soa.npz"))
    key = wl["case"]
    M, K, N, soa, _ = (int(x) for x in d[key + "_shape"])
    rp, ci, va = d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"]
    E = wl["elements"]
    esz = va.dtype.itemsize
    bsp = wl.get("sparse", "A") == "B"
    bB, bC = E * (M * K if bsp else K * N) * soa * esz, E * M * N * soa * esz
    op = xs.CsrSoa(M, N, K, rp, ci, va, soa, beta=wl["beta"], sparse="B" if bsp else "A")
    nsets = max(1, int(np.ceil(2.5 * L2_BYTES / (bB + bC))))
    ring = []
    for s_ in range(nsets):
        dB, dC = xs.DeviceBuffer(bB), xs.DeviceBuffer(bC)
        fill_device_random(xs, dB, bB, va.dtype, 21 + s_)
        dC.fill(0)
        ring.append((dB, dC))
    st = xs.Stream()
    t0, t1 = xs.Event(), xs.Event()
    for i in range(warmup):
        op.execute(*ring[i % nsets], E, stream=st)
    st.synchronize(); xs.check()
    yield "ready"
    l0 = xs.launch_count()
    t0.record(st)
    for i in range(steps):
        op.execute(*ring[(warmup + i) % nsets], E, stream=st)
    t1.record(st)
    st.synchronize()
    total_ms = t0.elapsed_ms(t1)
    xs.check()
    outputs = {"C": ring[(warmup + steps - 1) % nsets][1].to_numpy(va.dtype, (E, M, N, soa))} if dump else None
    nnz = len(va)
    if bsp:      # A [M][K][soa]: the rows k with nonzeros in B are read.  beta = 0: columns 0 .. ncols-1 of C are written (ncols =
        k_used = int(np.count_nonzero(np.diff(rp)))       # 1 + the largest column index of B); beta = 1: a column without nonzeros
        ncols = int(ci.max()) + 1 if len(ci) else 0       # keeps its content, so only the columns WITH nonzeros are read and written
        c_cols = 2 * int(len(np.unique(ci[ci < N]))) if float(wl["beta"]) != 0.0 else ncols
        bytes_ = esz * E * M * soa * (k_used + c_cols)
        flops = 2.0 * nnz * M * soa * E
    else:
        rows_touched = int(np.count_nonzero(np.diff(rp)))       # rows without nonzeros are neither read nor written,
        cols_used = int(len(np.unique(ci)))                      # B rows no nonzero refers to are never read
        bytes_ = esz * E * N * soa * (cols_used + rows_touched * (2 if float(wl["beta"]) != 0.0 else 1))
        flops = 2.0 * nnz * N * soa * E
    yield dict(total_ms=total_ms, launches=xs.launch_count() - l0, nnz=nnz, flops=flops, geo=dict(baked=op.is_baked, M=M, K=K, N=N, soa=soa, elements=E, sparse_operand="B" if bsp else "A"),
               kernel_ms=total_ms / steps, kernel_bytes=bytes_, kernel_name=xs.last_compute_kernel(), parts={}, step_bytes=bytes_, ring_sets=nsets, ring_bytes=nsets * (bB + bC),
               outputs=outputs)
    for bufs in ring:
        for b in bufs:
            b.free()
    op.destroy()


def dump_outputs(directory, outputs):
    """writes each output array as <directory>/<name>.npy.  One larger than its share of DUMP_BYTES is written as the 1-D sample
    a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]: the same positions for the same shape."""
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        n = DUMP_BYTES // len(outputs) // a.itemsize
        if a.size > n:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def fill_device_random(xs, dbuf, nbytes, dtype, seed):
    """fills a device buffer with uniform [0,1) values by uploading one 64 MiB host chunk repeatedly."""
    chunk_elems = min(nbytes, 64 << 20) // np.dtype(dtype).itemsize
    host = np.random.default_rng(seed).random(chunk_elems, np.float32).astype(dtype)
    off = 0
    while off < nbytes:
        n = min(host.nbytes, nbytes - off)
        xs.load().libxsmm_b200_memcpy_h2d(dbuf.ptr + off, host.ctypes.data, n)
        off += n
    xs.check()


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def run_spmdm_gpu(xs, wl, steps, warmup, want_e2e=True, dump=False):
    bf16 = wl["dtype"] == "bf16"
    dt = xs.LIBXSMM_SPMDM_DATATYPE_BFLOAT16 if bf16 else xs.LIBXSMM_SPMDM_DATATYPE_F32
    ta, tb, tc = wl["trans"]
    M, N, K = wl["M"], wl["N"], wl["K"]
    A, B, C0 = spmdm_host_inputs(xs, wl)
    nnz = int(np.count_nonzero(A))
    p = xs.Spmdm(M, N, K, 1)
    geo = p.geometry
    b_slice, b_compute = spmdm_bytes(wl, geo, nnz)
    set_bytes = A.nbytes + B.nbytes + C0.nbytes
    nsets = max(2, int(np.ceil(2.5 * L2_BYTES / set_bytes)))       # ring > 2.5 x L2: a set is evicted before reuse
    ring = []
    for _ in range(nsets):
        ring.append((xs.DeviceBuffer.from_numpy(A), xs.DeviceBuffer.from_numpy(B), xs.DeviceBuffer(C0.nbytes)))
    st = xs.Stream()
    ev = [[xs.Event() for _ in range(3)] for _ in range(steps)]
    t_first, t_last = xs.Event(), xs.Event()

    def step(i, events=None):
        dA, dB, dC = ring[i % nsets]
        if events:
            events[0].record(st)
        p.create_slices(dA, ta, bf16, st)
        if events:
            events[1].record(st)
        p.compute(dB, dC, tb, tc, wl["beta"], bf16, st)
        if events:
            events[2].record(st)

    for i in range(warmup):
        step(i)
    st.synchronize()
    xs.check()
    yield "ready"                                  # caller barriers here
    # Timed region: the K steps exactly as a caller enqueues them, nothing between the launches.  (An event recorded
    # between the slicing kernel and the multiply serialises their programmatic dependent launch and costs ~12 us of the
    # ~95 us step; the per-kernel durations below therefore come from a SECOND pass over the same K steps with events
    # between the launches, outside the timed region.)
    l0 = xs.launch_count()
    t_first.record(st)
    for i in range(steps):
        step(warmup + i)
    t_last.record(st)
    st.synchronize()
    launches = xs.launch_count() - l0
    total_ms = t_first.elapsed_ms(t_last)
    outputs = {"C": ring[(warmup + steps - 1) % nsets][2].to_numpy(np.float32, C0.shape)} if dump else None
    for i in range(steps):
        step(warmup + steps + i, ev[i])
    st.synchronize()
    slice_ms = float(np.mean([e[0].elapsed_ms(e[1]) for e in ev]))
    comp_ms = float(np.mean([e[1].elapsed_ms(e[2]) for e in ev]))
    xs.check()
    res = dict(total_ms=total_ms, launches=launches, nnz=nnz, flops=2.0 * nnz * N, geo=geo,
               kernel_ms=comp_ms, kernel_bytes=b_compute, kernel_name=xs.last_compute_kernel(), dense_flops=2.0 * M * N * K,
               parts={"slice_ms": slice_ms, "compute_ms": comp_ms, "slice_bytes": b_slice, "compute_bytes": b_compute},
               step_bytes=b_slice + b_compute, ring_sets=nsets, ring_bytes=nsets * set_bytes, outputs=outputs)
    yield res
    # ---- e2e: host pointers through the C ABI -------------------------------------------------------
    if want_e2e:
        hA = xs.HostBuffer(A.shape, A.dtype); hA.array[...] = A
        hB = xs.HostBuffer(B.shape, B.dtype); hB.array[...] = B
        hC = xs.HostBuffer(C0.shape, np.float32); hC.array[...] = C0
        for _ in range(max(1, min(warmup, 3))):
            xs.libxsmm_spmdm_exec_host(p.handle, p.slices, dt, ta, tb, tc, hA, hB, wl["beta"], hC)
        xs.check()
        yield "ready-e2e"
        t0 = time.perf_counter()
        for _ in range(steps):
            xs.libxsmm_spmdm_exec_host(p.handle, p.slices, dt, ta, tb, tc, hA, hB, wl["beta"], hC)
        t1 = time.perf_counter()
        xs.check()
        h2d = A.nbytes + B.nbytes + (C0.nbytes if float(wl["beta"]) != 0.0 else 0)
        yield dict(e2e_ms=(t1 - t0) * 1e3, h2d=h2d, d2h=C0.nbytes, checksum=float(hC.array[::97, ::89].sum()))
        for h in (hA, hB, hC):
            h.free()
    for bufs in ring:
        for b in bufs:
            b.free()
    p.destroy()


def run_fs_gpu(xs, wl, steps, warmup, world, want_e2e=True, rank=0, dump=False):
    """C3 / C5: the N columns of ONE global problem split into contiguous panels (sharding.column_panels: multiples of 16), one
    per rank; every rank holds its own dense B / C panel (ld = panel width) and a replica of the operator."""
    dbl = wl["dtype"] == "f64"
    dtype = np.float64 if dbl else np.float32
    a = fs_operator(xs, wl)
    nnz = int(np.count_nonzero(a))
    sharding = importlib.import_module("libxsmm-1_b200.sharding")
    n0, N = sharding.column_panels(wl["N"], world, 16)[rank]      # this rank's columns [n0, n0 + N) of the global B and C

    def make_operator(ncols):
        if not wl.get("fixture"):
            return xs.Fsspmdm(a, ncols, beta=wl["beta"])
        import tempfile                          # real operator: through the library's MatrixMarket entry (create_mtx)
        with tempfile.NamedTemporaryFile("w", suffix=".mtx", delete=False) as f:
            r, c = np.nonzero(a)
            f.write("%%%%MatrixMarket matrix coordinate real general\n%d %d %d\n" % (a.shape[0], a.shape[1], len(r)))
            for i, j in zip(r, c):
                f.write("%d %d %r\n" % (i + 1, j + 1, float(a[i, j])))
        try:
            return xs.Fsspmdm.from_mtx(f.name, ncols, beta=wl["beta"], double=dbl)
        finally:
            os.unlink(f.name)

    op = make_operator(N)
    esz = 8 if dbl else 4
    bB, bC = wl["K"] * N * esz, wl["M"] * N * esz
    nsets = max(1, int(np.ceil(2.5 * L2_BYTES / (bB + bC)))) if (bB + bC) < 3 * L2_BYTES else 1
    ring = []
    for s in range(nsets):
        dB, dC = xs.DeviceBuffer(bB), xs.DeviceBuffer(bC)
        fill_device_random(xs, dB, bB, dtype, 11 + s)
        dC.fill(0)
        ring.append((dB, dC))
    st = xs.Stream()
    t_first, t_last = xs.Event(), xs.Event()
    for i in range(warmup):
        op.execute_stream(*ring[i % nsets], st)
    st.synchronize(); xs.check()
    yield "ready"
    l0 = xs.launch_count()
    t_first.record(st)
    for i in range(steps):
        op.execute_stream(*ring[(warmup + i) % nsets], st)
    t_last.record(st)
    st.synchronize()
    launches = xs.launch_count() - l0
    total_ms = t_first.elapsed_ms(t_last)
    xs.check()
    outputs = {"C": ring[(warmup + steps - 1) % nsets][1].to_numpy(dtype, (wl["M"], N))} if dump else None
    yield dict(total_ms=total_ms, launches=launches, nnz=nnz, flops=2.0 * nnz * N, geo=dict(sparse=op.is_sparse, baked=op.is_baked, first_column=n0, columns_per_rank=N),
               kernel_ms=total_ms / steps, kernel_bytes=fs_bytes(wl, N), kernel_name=xs.last_compute_kernel(),
               parts={}, step_bytes=fs_bytes(wl, N), ring_sets=nsets, ring_bytes=nsets * (bB + bC), outputs=outputs)
    if want_e2e:
        Ne = min(N, 1 << 20)                      # host panel of at most 2^20 columns per step (537 MB + 1.26 GB for fp64)
        ope = make_operator(Ne) if Ne != N else op
        hB = xs.HostBuffer((wl["K"], Ne), dtype); hB.array[...] = np.random.default_rng(5).random((wl["K"], Ne), np.float32)
        hC = xs.HostBuffer((wl["M"], Ne), dtype); hC.array[...] = 0
        ope.execute(hB, hC)
        xs.check()
        yield "ready-e2e"
        t0 = time.perf_counter()
        for _ in range(steps):
            ope.execute(hB, hC)
        t1 = time.perf_counter()
        xs.check()
        yield dict(e2e_ms=(t1 - t0) * 1e3, h2d=hB.nbytes + (hC.nbytes if float(wl["beta"]) == 1.0 else 0), d2h=hC.nbytes,
                   e2e_flops=2.0 * nnz * Ne, checksum=float(hC.array[::7, ::4099].sum()))
        hB.free(); hC.free()
        if ope is not op:
            ope.destroy()
    for bufs in ring:
        for b in bufs:
            b.free()
    op.destroy()


# ------------------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference (oracle/_ref) if present, else the oracle port
# ------------------------------------------------------------------------------------------------------
def cpu_reference(wl, budget_s, reps_min=1, reps_max=50):
    """returns dict(value GFLOP/s, ms, cores, kind, sample).  TEST INFRASTRUCTURE use of oracle/."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    w = importlib.import_module("libxsmm-1_b200.workloads")
    cores = host_cores()
    have_ref = pyoracle.Ref.available()
    if not have_ref and os.path.isdir("/root/reference/src"):
        try:
            pyoracle.build_ref("avx2")
            have_ref = pyoracle.Ref.available()
        except Exception:
            have_ref = False
    # the reference has two SIMD instantiations of spmdm (src/libxsmm_spmdm.c:557-583): AVX2 (bn = 48, what a plain GCC
    # build selects) and AVX-512 (bn = 96, `make AVX=3`).  Both are timed where the host can run them; the faster counts.
    flavors = ["avx2"]
    try:
        if pyoracle.Ref.available("avx512") and "avx512f" in open("/proc/cpuinfo").read():
            flavors.append("avx512")
    except Exception:
        pass
    if wl["kind"] == "soa":
        if not have_ref:
            raise RuntimeError("no compiled reference for the SoA kernel")
        d = np.load(os.path.join(ROOT, "tests", "golden", "csr_soa.npz"))
        key = wl["case"]
        M, K, N, soa, _ = (int(x) for x in d[key + "_shape"])
        rp, ci, va = d[key + "_rowptr"], d[key + "_colidx"], d[key + "_values"]
        ref = pyoracle.Ref()
        if ref.soa_width(va.dtype) != soa:
            raise RuntimeError("host without AVX-512: the reference's SoA width differs from the workload's")
        E = min(wl["elements"], 1 << 14)                      # bounded sample: 2^14 elements (~0.65 GB of tensors)
        rng = np.random.default_rng(3)
        bsp = wl.get("sparse", "A") == "B"
        B = rng.random((E, M, K, soa) if bsp else (E, K, N, soa)).astype(va.dtype); C = np.zeros((E, M, N, soa), va.dtype)
        timed = ref.csr_soa_bsparse_bench if bsp else ref.csr_soa_bench
        tm = timed(rp, ci, va, B, C, N, wl["beta"], threads=cores, reps=1)
        reps = int(min(reps_max, max(reps_min, budget_s / max(tm[0], 1e-4))))
        tm = timed(rp, ci, va, B, C, N, wl["beta"], threads=cores, reps=reps)
        ms = float(np.median(tm)) * 1e3
        return dict(value=2.0 * len(va) * (M if bsp else N) * soa * E / ms / 1e6, ms=ms, best_ms=float(tm.min()) * 1e3, cores=cores, kind="reference",
                    sample="2^14 of the workload's elements, %d reps, median; libxsmm_create_xcsr_soa kernel, OpenMP over elements" % reps)
    if wl["kind"] == "spmdm":
        t = wl["trans"]
        A, B, C0 = w.spmdm_inputs(wl["M"], wl["N"], wl["K"], wl["density"], dtype=wl["dtype"], seed=1, transa=t[0], transb=t[1], transc=t[2])
        nnz = int(np.count_nonzero(A))
        flops = 2.0 * nnz * wl["N"]
        if have_ref:
            best, seen = None, []
            for fl in flavors:
                ref = pyoracle.Ref(fl)
                C = C0.copy()
                _, _, tm = ref.spmdm(A, B, C, wl["M"], wl["N"], wl["K"], t[0], t[1], t[2], wl["beta"], threads=cores, reps=1, dump=False)   # warm-up
                reps = int(min(reps_max, max(reps_min, budget_s / len(flavors) / max(tm[0, 2], 1e-4))))
                _, _, tm = ref.spmdm(A, B, C, wl["M"], wl["N"], wl["K"], t[0], t[1], t[2], wl["beta"], threads=cores, reps=reps, dump=False)
                ms = float(np.median(tm[:, 2])) * 1e3
                seen.append("%s (bn=%d) %.2f ms" % (fl, 96 if fl == "avx512" else 48, ms))
                if best is None or ms < best[0]:
                    best = (ms, float(tm[:, 2].min()) * 1e3, fl, reps)
            ms, best_ms, fl, reps = best
            return dict(value=flops / ms / 1e6, ms=ms, best_ms=best_ms, cores=cores, kind="reference", flavor=fl,
                        sample="full workload (%s), %d reps after 1 warm-up, median; OpenMP over block ids; instantiations timed: %s; reported: %s" % (wl["desc"], reps, ", ".join(seen), fl))
        orc = pyoracle.Oracle()
        g = orc.geometry(wl["M"], wl["N"], wl["K"], 1, bn=48)
        t0 = time.perf_counter()
        sl = orc.slices(g, A, t[0]); C = C0.copy(); orc.compute(g, sl, B, C, t[1], t[2], float(wl["beta"]))
        ms = (time.perf_counter() - t0) * 1e3
        return dict(value=flops / ms / 1e6, ms=ms, best_ms=ms, cores=1, kind="port", sample="full workload once, scalar oracle port")
    # fsspmdm: a bounded slab of columns, ld <= 2^20 (the reference's JIT addresses with 32-bit displacements)
    a = fs_operator(importlib.import_module("libxsmm-1_b200"), wl)
    nnz = int(np.count_nonzero(a))
    Ns = 1 << 20 if wl["dtype"] == "f64" else 1 << 20
    rng = np.random.default_rng(3)
    B = rng.random((wl["K"], Ns), np.float32).astype(a.dtype); C = np.zeros((wl["M"], Ns), a.dtype)
    flops = 2.0 * nnz * Ns
    if have_ref:
        ref = pyoracle.Ref()
        _, _, tm = ref.fsspmdm(a, B, C, wl["beta"], panel=64, threads=cores, reps=1)
        reps = int(min(reps_max, max(reps_min, budget_s / max(tm[0], 1e-4))))
        sparse, chunk, tm = ref.fsspmdm(a, B, C, wl["beta"], panel=64, threads=cores, reps=reps)
        ms = float(np.median(tm)) * 1e3
        return dict(value=flops / ms / 1e6, ms=ms, best_ms=float(tm.min()) * 1e3, cores=cores, kind="reference",
                    sample="2^20-column slab of the workload (ld=2^20), %d reps, median; OpenMP over 64-column panels; branch=%s" % (reps, "sparse_reg" if sparse else "dense"))
    orc = pyoracle.Oracle()
    Ns = 1 << 14
    t0 = time.perf_counter()
    if a.dtype == np.float64:
        orc.dfsspmdm_execute(a, np.ascontiguousarray(B[:, :Ns]), np.ascontiguousarray(C[:, :Ns]), wl["beta"], 1)
    else:
        orc.sfsspmdm_execute(a, np.ascontiguousarray(B[:, :Ns]), np.ascontiguousarray(C[:, :Ns]), wl["beta"])
    ms = (time.perf_counter() - t0) * 1e3
    return dict(value=2.0 * nnz * Ns / ms / 1e6, ms=ms, best_ms=ms, cores=1, kind="port", sample="2^14-column slab, scalar oracle port")


# ------------------------------------------------------------------------------------------------------
def main():
    # exactly ONE line on stdout: libraries that write to file descriptor 1 (NCCL prints its version there) are sent to stderr
    out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--others", default="c1,c4,c4-tnt,c4-ntn,c3-b1,c3-hex,c3-tet,c5-dense,c5-dense-b1,soa,soa-b", help="extra workloads reported inside the line (N=1 only); '' = none")
    ap.add_argument("--sharded", default="c3,c5", help="column-sharded fsspmdm configs reported in `column_sharded` at every N (strong scaling); '' = none")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of reference CPU time for the headline cpu_baseline (a quarter of it per secondary workload)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the headline workload's last timed step to DIR/<name>.npy (rank 0's part when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    metric = "effective GFLOP/s (2*nnz*N)"

    if args.impl == "reference":
        if rank != 0:
            return 0
        wl = dict(wl)
        if wl["kind"] == "spmdm" and args.gpus > 1:      # the GPU arm's global problem: one 4096-column panel per GPU
            wl["N"] = wl["N"] * args.gpus
            wl["desc"] += " x %d column panels (global N = %d)" % (args.gpus, wl["N"])
        r = cpu_reference(wl, budget_s=0.0, reps_min=args.steps + args.warmup, reps_max=args.steps + args.warmup)
        line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": "GFLOP/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if wl["dtype"] in ("f32", "bf16") else "f64", "data": "synthetic",
                "config": {"workload": wl["desc"], "note": "reference CPU path on this host; one rank only"},
                "cpu_baseline": {"value": r["value"], "unit": "GFLOP/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=out, flush=True)
        return 0

    if args.gpus > 1 and world == 1:      # convenience: re-launch under torchrun like the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 500), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd, stdout=out)      # the ranks write to the real stdout, not to the redirected descriptor 1

    xs = importlib.import_module("libxsmm-1_b200")
    xs.load()
    xs.require_gpu()
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    xs.load().libxsmm_b200_set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None

    def barrier():
        if dist is not None:
            dist.barrier()
        xs.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def run(wl_, want_e2e, sample_clocks, shard=1, dump=False):
        """one workload on this rank.  shard = 1: the whole problem on every rank (replicas).  shard = world: this rank's
        N / world column panel of ONE global problem (fsspmdm; SURVEY.md section 8e)."""
        # the clock sampler (nvidia-smi every 200 ms) runs from before the warm-up until after the end-to-end
        # phase: the device-timed region alone lasts only milliseconds
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
            time.sleep(0.3)
        if wl_["kind"] == "soa":
            want_e2e = False
            gen = run_soa_gpu(xs, wl_, args.steps, args.warmup, dump)
        else:
            gen = run_spmdm_gpu(xs, wl_, args.steps, args.warmup, want_e2e, dump) if wl_["kind"] == "spmdm" else \
                run_fs_gpu(xs, wl_, args.steps, args.warmup, shard, want_e2e, rank if shard > 1 else 0, dump)
        assert next(gen) == "ready"
        barrier()
        res = next(gen)
        barrier()
        res["total_ms"] = max_over_ranks(res["total_ms"])
        res["flops_all"] = sum_over_ranks(res["flops"])
        res["launches_all"] = int(sum_over_ranks(res["launches"]))
        e2e = None
        if want_e2e:
            assert next(gen) == "ready-e2e"
            barrier()
            e = next(gen)
            barrier()
            e["e2e_ms"] = max_over_ranks(e["e2e_ms"])
            e["flops_all"] = sum_over_ranks(e.get("e2e_flops", res["flops"]))
            e2e = e
        for _ in gen:
            pass
        clocks = sampler.finish() if sampler else None
        return res, e2e, clocks

    peak, peak_src = peaks()

    def bound_of(wl_, r):
        """which roofline bounds the dominant kernel of this workload, and the fraction of it achieved: HBM for the
        sparse / streaming kernels (algorithmic bytes over the measured copy bandwidth); the tensor pipe for the tcgen05
        kernels that multiply densified tiles; the fp32 FMA pipe for the CUDA-core spmdm kernels on C1 / C4, whose
        arithmetic intensity (48-186 flop/B) is far above the FMA ridge (BASELINE.md section 3)."""
        ach = r["kernel_bytes"] / (r["kernel_ms"] * 1e6)
        out = {"kernel": r["kernel_name"], "kernel_ms": r["kernel_ms"], "hbm_achieved_gbs": ach, "hbm_frac": ach / peak}
        tp = tensor_pipe_info(r)
        if tp:
            out.update(bound="tensor", frac=tp["frac"], tensor_pipe=tp)
        elif wl_["kind"] == "spmdm" and 2.0 * r["nnz"] * wl_["N"] / r["kernel_bytes"] > 16.0:
            tf = 2.0 * r["nnz"] * wl_["N"] / (r["kernel_ms"] * 1e9)
            out.update(bound="fma", frac=tf / FP32_FMA_PEAK_TFLOPS, fma_pipe={"executed_tflops": tf, "peak_tflops": FP32_FMA_PEAK_TFLOPS, "peak_source": "nominal 148 x 128 lanes x 2 x 1.965 GHz"})
        else:
            out.update(bound="hbm", frac=ach / peak)
        return out

    def e2e_block(e, wl_):
        e_ms = e["e2e_ms"] / args.steps
        return {"value": e["flops_all"] / (e_ms * 1e6), "unit": "GFLOP/s", "ms_per_step": e_ms,
                "h2d_bytes_per_step": int(e["h2d"]), "d2h_bytes_per_step": int(e["d2h"]),
                "api": "libxsmm_spmdm_exec_host" if wl_["kind"] == "spmdm" else "libxsmm_[sd]fsspmdm_execute (host pointers)"}

    res, e2e, clocks = run(wl, not args.no_e2e, rank == 0, shard=(world if wl["kind"] == "fsspmdm" else 1), dump=bool(args.dump_outputs) and rank == 0)
    if res["outputs"] is not None:
        dump_outputs(args.dump_outputs, res.pop("outputs"))
    ms_per_step = res["total_ms"] / args.steps
    value = res["flops_all"] / (ms_per_step * 1e6)
    achieved = res["kernel_bytes"] / (res["kernel_ms"] * 1e6)
    spm = wl["kind"] == "spmdm"
    line = {
        "metric": metric, "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if spm else "strong", "vs_baseline": None,
        "dtype": "f32" if wl["dtype"] in ("f32", "bf16") else "f64", "data": "synthetic",
        "config": {"workload": wl["desc"],
                   "per_gpu": ("replicas: every rank multiplies its own 4096-column panel with its own copy of A (weak scaling; BASELINE.json names no sharding for this config); "
                               "the column-SHARDED configs (C3, C5) are in `column_sharded`" if spm else
                               "one N/%d-column panel of the global problem per rank, operator replicated, no collective on the data path (strong scaling)" % world),
                   "global_N": (wl.get("N", 0) * world if spm else wl.get("N", 0)), **({"numa": numa} if numa else {}), "inputs": "bf16" if wl["dtype"] == "bf16" else wl["dtype"],
                   "l2_policy": "inputs larger than L2: ring of %d input sets = %.0f MB, a different set every step" % (res["ring_sets"], res["ring_bytes"] / 1e6),
                   "geometry": res["geo"], "nnz": res["nnz"], "step": "createSparseSlice (all blocks) + compute (all blocks)" if spm else "execute"},
        "hbm_gbs": res["step_bytes"] * world / (ms_per_step * 1e6),
        "gpu_launches": res["launches_all"],
        "roofline": {"bound": "hbm", "kernel": res["kernel_name"], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(args.workload),
                     "traffic_note": "ncu dram bytes of one launch are BELOW the algorithmic bytes because most of C (67 MB of fp32, written once) is still dirty in the 126 MB L2 when the kernel ends; the reads (A slices, B) are counted in full",
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": res["kernel_bytes"],
                     "kernel_ms": res["kernel_ms"], "parts": res["parts"],
                     **({"parts_note": "kernel durations: CUDA events between the launches, in a second pass over the same K steps (an event between the slicing kernel and the multiply serialises their programmatic dependent launch, so the parts add up to more than ms_per_step, which is timed with nothing between the launches)"} if spm else {})},
        "clocks": clocks,
    }
    tpipe = tensor_pipe_info(res)
    if tpipe:
        line["roofline"]["tensor_pipe"] = tpipe
    if e2e is not None:
        line["e2e"] = e2e_block(e2e, wl)

    # ---- the column-sharded configs of BASELINE.json (C3: dfsspmdm N = 2^20; C5: sfsspmdm N = 2^24) at this N: STRONG scaling,
    #      rank r owns columns [r N/g, (r+1) N/g) of B and C (ld = N/g), the operator is replicated, nothing is exchanged ----
    if args.sharded and spm:
        sh = {}
        for name in [n for n in args.sharded.split(",") if n]:
            w_ = WORKLOADS[name]
            try:
                r2, e2, _ = run(w_, not args.no_e2e, False, shard=world)
                ms2 = r2["total_ms"] / args.steps
                ach2 = r2["kernel_bytes"] / (r2["kernel_ms"] * 1e6)
                sh[name] = {"workload": w_["desc"], "scaling": "strong", "n_gpus": world, "columns_per_gpu": w_["N"] // world,
                            "value": r2["flops_all"] / (ms2 * 1e6), "unit": "GFLOP/s", "ms_per_step": ms2,
                            "hbm_gbs_all_gpus": fs_bytes(w_, w_["N"]) / (ms2 * 1e6), "kernel": r2["kernel_name"],
                            "per_gpu_hbm_gbs": ach2, "per_gpu_hbm_frac": ach2 / peak, "gpu_launches": r2["launches_all"]}
                if e2 is not None:
                    sh[name]["e2e"] = e2e_block(e2, w_)
                    sh[name]["e2e"]["note"] = "host panels of min(N/g, 2^20) columns per rank and step"
            except Exception as ex:
                sh[name] = {"error": repr(ex)[:200]}
                xs.clear_error()
        line["column_sharded"] = sh

    if world == 1 and rank == 0 and args.others:
        others = {}
        names = [n for n in args.others.split(",") if n and n != args.workload]
        if spm:
            names.insert(0, args.workload + "@cuda-cores")     # same workload, LIBXSMM_B200_SPMDM_TC=0: the order-preserving (bit-exact) kernels only
        for name in names:
            try:
                forced = name.endswith("@cuda-cores")
                w_ = WORKLOADS[name.split("@")[0]]
                if forced:
                    os.environ["LIBXSMM_B200_SPMDM_TC"] = "0"
                try:
                    r2, e2, _ = run(w_, (not args.no_e2e) and not forced, False)
                finally:
                    if forced:
                        os.environ.pop("LIBXSMM_B200_SPMDM_TC", None)
                ms2 = r2["total_ms"] / args.steps
                others[name] = {"workload": w_["desc"] + (" [LIBXSMM_B200_SPMDM_TC=0]" if forced else ""), "value": r2["flops"] / (ms2 * 1e6), "unit": "GFLOP/s", "ms_per_step": ms2,
                                "hbm_gbs": r2["step_bytes"] / (ms2 * 1e6), "roofline": bound_of(w_, r2), "parts": r2["parts"], "gpu_launches": r2["launches"]}
                if e2 is not None:
                    others[name]["e2e"] = e2e_block(e2, w_)
                if not args.no_cpu and not forced:
                    c = cpu_reference(w_, budget_s=args.cpu_budget / 4.0)
                    others[name]["cpu_baseline"] = {"value": c["value"], "unit": "GFLOP/s", "cores": c["cores"], "kind": c["kind"], "sample": c["sample"], "ms_per_step": c["ms"]}
            except Exception as ex:      # a secondary workload must never take the headline down
                others[name] = {"error": repr(ex)[:200]}
                xs.clear_error()
        line["other_workloads"] = others
    if world == 1 and rank == 0 and not args.no_cpu:
        try:
            c = cpu_reference(wl, budget_s=args.cpu_budget)
            line["cpu_baseline"] = {"value": c["value"], "unit": "GFLOP/s", "cores": c["cores"], "kind": c["kind"], "sample": c["sample"], "ms_per_step": c["ms"]}
        except Exception as ex:
            line["cpu_baseline"] = {"value": None, "unit": "GFLOP/s", "cores": host_cores(), "kind": "reference", "sample": "failed: %r" % (ex,)}
    if rank == 0:
        print(json.dumps(line), file=out, flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
