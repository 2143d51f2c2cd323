"""Developer tool: times the fixed 2:4-sparse bf16 operator (libxsmm_b200_sp24_execute) against what a caller with a pruned
weight has without it.

    python tools/time_sp24.py [--reps 30] [--warmup 5] [--out profiles/sp24_time.jsonl] [--only 4096x4096x4096]

Shapes M x N x K: 4096^3, 4096 x {256, 1024, 16384} x 4096 and 14336 x 4096 x 4096; transb N and T; beta 0 and 1.  A is a
random matrix pruned to 2:4 (every group of four along k keeps two of its positions: 50 % dense, mixed signs).
Compared in the same run, on the same A, B and C:
  (a) Spmdm.compute on slices made once from A, default dispatch (K4p at this density);
  (b) the same with K4s forced (LIBXSMM_B200_SPMDM_TC=1, LIBXSMM_B200_TC16_SPARSE=1; transb N only);
  (c) torch.matmul of the dense bf16 A and B (cuBLAS, bf16 output).
Each is warmed up, then timed over --reps back-to-back calls by CUDA events around every call (best and median).  B and C
rotate over enough buffers that the working set exceeds twice the 126 MB L2, so every call reads its operands from HBM.
C of the new kernel is compared bit for bit with (b) where (b) runs, otherwise with the float64 product of 256 sampled rows
(|C - want| <= 4e-6 (|A|.|B| + |beta| |C0|)).  One JSON line per (shape, transb, beta); the card's name, power limit and
maximum SM clock are read in the same run.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SHAPES = [(4096, 4096, 4096), (4096, 256, 4096), (4096, 1024, 4096), (4096, 16384, 4096), (14336, 4096, 4096)]
L2_BYTES = 126 << 20


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True)
        return [x.strip() for x in out.splitlines()[0].split(",")]
    except Exception as e:      # noqa: BLE001
        return ["unknown (%s)" % e, "unknown", "unknown"]


def make24(M, K, g):
    """random bf16 matrix pruned to 2:4 on the GPU: each group of four keeps two of its positions"""
    legal = torch.tensor([m for m in range(16) if bin(m).count("1") == 2], device="cuda")
    masks = legal[torch.randint(0, len(legal), (M, K // 4), generator=g, device="cuda")]
    keep = ((masks[:, :, None] >> torch.arange(4, device="cuda")) & 1).bool().reshape(M, K)
    v = (torch.rand((M, K), generator=g, device="cuda") * 1.75 + 0.25) * (torch.randint(0, 2, (M, K), generator=g, device="cuda") * 2 - 1)
    return torch.where(keep, v, torch.zeros_like(v)).to(torch.bfloat16)


def timed(fn, nbuf, reps, warmup):
    for i in range(warmup):
        fn(i % nbuf)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for i in range(reps):
        fn((warmup + i) % nbuf)
        ev[i + 1].record()
    torch.cuda.synchronize()
    t = sorted(ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(reps))
    return {"best_us": round(t[0], 2), "median_us": round(t[len(t) // 2], 2)}


def spmdm_leg(xs, M, N, K, A, Bs, Cs, C0, beta, transb, force_k4s, reps, warmup):
    """Spmdm.compute on slices made once from A: timing, kernel name and C of one call from C0"""
    keys = ("LIBXSMM_B200_SPMDM_TC", "LIBXSMM_B200_TC16_SPARSE")
    saved = {k: os.environ.pop(k, None) for k in keys}
    if force_k4s:
        os.environ.update({k: "1" for k in keys})
    p = xs.Spmdm(M, N, K, 1)
    try:
        p.create_slices(A.data_ptr(), "N", True)

        def call(i, c=None):      # bf16 beta: the raw integer (reference quirk), 1 means beta = 1
            p.compute(Bs[i].data_ptr(), (Cs[i] if c is None else c).data_ptr(), transb, "N", int(beta), True)
        t = timed(call, len(Bs), reps, warmup)
        t["kernel"] = xs.last_compute_kernel()
        c = C0.clone()
        call(0, c)
        xs.synchronize()
        return t, c
    finally:
        p.destroy()
        for k in keys:
            os.environ.pop(k, None)
            if saved[k] is not None:
                os.environ[k] = saved[k]


def f64_check(A, B, C, C0, beta, transb, rows):
    a = A[rows].double().cpu().numpy()
    b = (B.t() if transb == "T" else B).double().cpu().numpy()
    want = a @ b + beta * C0[rows].double().cpu().numpy()
    bound = 4e-6 * (np.abs(a) @ np.abs(b) + abs(beta) * np.abs(C0[rows].double().cpu().numpy()))
    return bool(np.all(np.abs(C[rows].double().cpu().numpy() - want) <= bound))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    xs = importlib.import_module("libxsmm-1_b200")
    xs.require_gpu()
    name, power, clock = card()
    out = open(args.out, "a") if args.out else None
    shapes = [s for s in SHAPES if not args.only or "%dx%dx%d" % s in args.only.split(",")]
    for (M, N, K) in shapes:
        g = torch.Generator(device="cuda").manual_seed(M + N + K)
        A = make24(M, K, g)
        op = xs.Sp24(A)
        per = N * K * 2 + M * N * 4
        nbuf = max(2, -(-2 * L2_BYTES // per))
        Bn = [torch.rand((K, N), generator=g, device="cuda").sub_(0.5).to(torch.bfloat16) for _ in range(nbuf)]
        Bt = [b.t().contiguous() for b in Bn]
        C0 = torch.rand((M, N), generator=g, device="cuda").sub_(0.5)
        Cs = [C0.clone() for _ in range(nbuf)]
        rows = torch.randperm(M, generator=torch.Generator().manual_seed(M))[:256]
        for transb in ("N", "T"):
            Bs = Bn if transb == "N" else Bt
            for beta in (0.0, 1.0):
                rec = {"gpu": name, "power_limit": power, "max_sm_clock": clock, "M": M, "N": N, "K": K, "transb": transb, "beta": beta,
                       "density": round(float((A != 0).float().mean()), 4), "buffers": nbuf,
                       "working_set_mb": round(nbuf * per / 2 ** 20), "l2_note": "B and C rotate over buffers larger than twice the 126 MB L2"}
                for c in Cs:
                    c.copy_(C0)
                rec["sp24"] = timed(lambda i: op.execute(Bs[i], Cs[i], N, beta=beta, transb=transb), nbuf, args.reps, args.warmup)
                xs.check()
                c = C0.clone()                    # C of one call from C0
                op.execute(Bs[0], c, N, beta=beta, transb=transb)
                torch.cuda.synchronize()
                rec["sp24"]["kernel"] = xs.last_compute_kernel()
                rec["k4p_default"], _ = spmdm_leg(xs, M, N, K, A, Bs, Cs, C0, beta, transb, False, args.reps, args.warmup)
                if transb == "N":
                    rec["k4s_forced"], ck = spmdm_leg(xs, M, N, K, A, Bs, Cs, C0, beta, "N", True, args.reps, args.warmup)
                    rec["same_bits_as_k4s"] = bool(torch.equal(c.view(torch.int32), ck.view(torch.int32)))
                else:
                    rec["k4s_forced"] = None       # K4s has no transposed-B form
                    rec["f64_bound_256_rows"] = f64_check(A, Bs[0], c, C0, beta, transb, rows)
                if beta == 0.0:
                    if transb == "N":
                        rec["cublas_bf16_out"] = timed(lambda i: torch.matmul(A, Bs[i]), nbuf, args.reps, args.warmup)
                    else:
                        rec["cublas_bf16_out"] = timed(lambda i: torch.matmul(A, Bs[i].t()), nbuf, args.reps, args.warmup)
                line = json.dumps(rec)
                print(line, flush=True)
                if out:
                    out.write(line + "\n")
                    out.flush()
        op.destroy()
        del Bn, Bt, Cs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
