"""Developer tool: times the fixed 2:4-sparse FP8 operator (libxsmm_b200_sp24_execute_fp8) against the bf16 operator on the
same values and against the dense FP8 product a caller has without it.

    python tools/time_sp24_fp8.py [--reps 30] [--warmup 5] [--out profiles/sp24_fp8_time.jsonl] [--only 4096x4096x4096]

Shapes M x N x K: 4096^3, 4096 x {256, 1024, 16384} x 4096 and 14336 x 4096 x 4096; transb N and T; beta 0 and 1.  A is a
random matrix pruned to 2:4 (every group of four along k keeps two of its positions: 50 % dense, mixed signs) and quantised to
e4m3 with a per-tensor scale, as B is.  Compared in the same run:
  (a) the FP8 operator, alpha = scale_a * scale_b;
  (b) the bf16 operator (libxsmm_b200_sp24_execute) on the same values widened to bf16 (exact), B widened likewise;
  (c) torch._scaled_mm of the dense e4m3 A and B with fp32 output (beta = 0 only; B column-major, as it requires).
Each is warmed up, then timed over --reps back-to-back calls by CUDA events around every call (best and median).  B and C
rotate over enough buffers that the working set exceeds twice the 126 MB L2, so every call reads its operands from HBM.
C of (a) is held to |alpha| 4e-6 (|A|.|B| + |beta| |C0|) against the float64 product on 256 sampled rows, and compared with
(b).  One JSON line per (shape, transb, beta); the card's name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_sp24 import SHAPES, L2_BYTES, card, make24, timed      # noqa: E402

F8 = torch.float8_e4m3fn


def quantise(x):
    """per-tensor scale so that the largest magnitude lands on 448 (e4m3's largest finite value)"""
    scale = float(x.abs().max()) / 448.0
    return (x.float() / scale).to(F8), scale


def f64_check(A8, B8, C, C0, alpha, beta, transb, rows):
    a = A8[rows].double().cpu().numpy()
    b = (B8.t() if transb == "T" else B8).double().cpu().numpy()
    c0 = C0[rows].double().cpu().numpy()
    want = alpha * (a @ b) + beta * c0
    bound = 4e-6 * abs(alpha) * (np.abs(a) @ np.abs(b) + abs(beta) * np.abs(c0))
    err = np.abs(C[rows].double().cpu().numpy() - want)
    return bool(np.all(err <= bound)), float((err / np.maximum(bound, 1e-300)).max())


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
        A8, sa = quantise(make24(M, K, g))
        op8, op16 = xs.Sp24(A8), xs.Sp24(A8.to(torch.bfloat16))
        per = N * K * 3 + M * N * 4
        nbuf = max(2, -(-2 * L2_BYTES // per))
        Bt8, sb = quantise(torch.rand((N, K), generator=g, device="cuda").sub_(0.5))
        Bt = [Bt8] + [(torch.rand((N, K), generator=g, device="cuda").sub_(0.5) / sb).to(F8) for _ in range(nbuf - 1)]
        Bn = [b.t().contiguous() for b in Bt]
        alpha = sa * sb
        C0 = torch.rand((M, N), generator=g, device="cuda").sub_(0.5)
        Cs = [C0.clone() for _ in range(nbuf)]
        rows = torch.randperm(M, generator=torch.Generator().manual_seed(M))[:256]
        sa_t, sb_t = torch.tensor(sa, device="cuda"), torch.tensor(sb, device="cuda")
        for transb in ("N", "T"):
            Bs = Bn if transb == "N" else Bt
            Bs16 = [b.to(torch.bfloat16) for b in Bs]
            for beta in (0.0, 1.0):
                rec = {"gpu": name, "power_limit": power, "max_sm_clock": clock, "M": M, "N": N, "K": K, "transb": transb, "beta": beta,
                       "format": "e4m3 x e4m3", "density": round(float((A8.float() != 0).float().mean()), 4), "buffers": nbuf,
                       "working_set_mb": round(nbuf * per / 2 ** 20), "l2_note": "B and C rotate over buffers larger than twice the 126 MB L2"}
                for c in Cs:
                    c.copy_(C0)
                rec["sp24_fp8"] = timed(lambda i: op8.execute(Bs[i], Cs[i], N, beta=beta, transb=transb, alpha=alpha), nbuf, args.reps, args.warmup)
                xs.check()
                c8 = C0.clone()
                op8.execute(Bs[0], c8, N, beta=beta, transb=transb, alpha=alpha)
                torch.cuda.synchronize()
                rec["sp24_fp8"]["kernel"] = xs.last_compute_kernel()
                ok, worst = f64_check(A8, Bs[0], c8, C0, alpha, beta, transb, rows)
                rec["f64_bound_256_rows"], rec["f64_worst_err_over_bound"] = ok, round(worst, 4)
                for c in Cs:
                    c.copy_(C0)
                rec["sp24_bf16"] = timed(lambda i: op16.execute(Bs16[i % len(Bs16)], Cs[i], N, beta=beta, transb=transb), nbuf, args.reps, args.warmup)
                c16 = C0.clone()
                op16.execute(Bs16[0], c16, N, beta=beta, transb=transb)
                torch.cuda.synchronize()
                c16 = alpha * (c16 - beta * C0) + beta * C0
                rec["max_diff_to_bf16_over_max_c"] = float((c8 - c16).abs().max() / c16.abs().max())
                rec["speedup_over_bf16"] = round(rec["sp24_bf16"]["best_us"] / rec["sp24_fp8"]["best_us"], 3)
                if beta == 0.0:
                    try:
                        rec["scaled_mm_dense_fp8_f32_out"] = timed(
                            lambda i: torch._scaled_mm(A8, Bt[i].t(), scale_a=sa_t, scale_b=sb_t, out_dtype=torch.float32), nbuf, args.reps, args.warmup)
                        rec["speedup_over_scaled_mm"] = round(rec["scaled_mm_dense_fp8_f32_out"]["best_us"] / rec["sp24_fp8"]["best_us"], 3)
                    except RuntimeError as e:
                        rec["scaled_mm_dense_fp8_f32_out"] = "unavailable: %s" % str(e).splitlines()[0]
                line = json.dumps(rec)
                print(line, flush=True)
                if out:
                    out.write(line + "\n")
                    out.flush()
            del Bs16
        op8.destroy(); op16.destroy()
        del Bn, Bt, Cs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
