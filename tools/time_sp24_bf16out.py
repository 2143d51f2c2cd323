"""Developer tool: times the bf16-output entries of the fixed 2:4-sparse operators (libxsmm_b200_sp24_execute_bf16out /
_execute_fp8_bf16out, Sp24.linear) against the fp32-output entry and what a caller of a pruned linear layer has without them.

    python tools/time_sp24_bf16out.py [--reps 30] [--warmup 5] [--out profiles/sp24_bf16out_time.jsonl] [--only 4096x4096x4096]

Shapes M x N x K as tools/time_sp24.py; layouts transb = transc = 'T' (y = x . W^T, the linear layout: B is x, N tokens x K,
C is N x M) and 'N' / 'N', at beta = 0; beta = 1 on 4096^3 only.  Operators: bf16 (A pruned to 2:4 as time_sp24.py) and FP8
(the same A and B quantised to e4m3 with per-tensor scales, alpha = scale_a * scale_b).  Compared in the same run:
  (a) the bf16-output entry, no bias;            (b) the same with a bias;
  (c) the fp32-output entry;                     (d) (c) followed by the torch add_(bias) and .to(bfloat16) a caller needs today;
  (e) dense bf16 with bias by cuBLAS: F.linear for 'T' / 'T', addmm for 'N' / 'N' (bf16 operator, beta = 0);
  (f) torch._scaled_mm(out_dtype=bfloat16, bias=...) of the dense e4m3 operands ('T' / 'T', FP8 operator, beta = 0);
  (g) Sp24.linear(x, bias) ('T' / 'T', beta = 0): (b) with the Python-side checks and the allocation of y.
Each is warmed up, then timed over --reps back-to-back calls by CUDA events around every call (best and median).  B and C
rotate over enough buffers that the working set exceeds twice the 126 MB L2, so every call reads its operands from HBM.
C of (a) and (b) is held to the float64 product on 256 sampled rows of A (|C - want| <= |alpha| 4e-6 (|A|.|B| + |bias| +
|beta| |C0|) + half a bf16 ulp of C), and C of (a) at beta = 0 is compared bit for bit with (c) rounded to bf16.  One JSON
line per (operator, shape, layout, beta); the card's name, power limit and maximum SM clock are read in the same run.
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
from time_sp24_fp8 import F8, quantise                           # noqa: E402

BF = torch.bfloat16


def f64_check(A, B, C, C0, bias, alpha, beta, trans, rows):
    """C (M x N, or N x M for 'T' / 'T') against the float64 product on the sampled rows of A"""
    a = A[rows].double().cpu().numpy()
    b = (B.t() if trans == "T" else B).double().cpu().numpy()
    c = (C.t() if trans == "T" else C)[rows].double().cpu().numpy()
    c0 = (C0.t() if trans == "T" else C0)[rows].double().cpu().numpy()
    bv = bias[rows].double().cpu().numpy()[:, None] if bias is not None else 0.0
    want = alpha * (a @ b) + bv + beta * c0
    bound = 4e-6 * abs(alpha) * (np.abs(a) @ np.abs(b)) + 4e-6 * (np.abs(bv) + abs(beta) * np.abs(c0))
    ulp = np.ldexp(1.0, np.frexp(np.maximum(np.abs(c), 1e-30))[1] - 8)
    err = np.abs(c - want)
    return bool(np.all(err <= bound + 0.5 * ulp)), float((err / (bound + 0.5 * ulp)).max())


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
    T = lambda fn: timed(fn, nbuf, args.reps, args.warmup)      # noqa: E731
    for (M, N, K) in shapes:
        g = torch.Generator(device="cuda").manual_seed(M + N + K)
        A = make24(M, K, g)
        A8, sa = quantise(A)
        per = N * K * 2 + M * N * (4 + 2)
        nbuf = max(2, -(-2 * L2_BYTES // per))
        Bt = [torch.rand((N, K), generator=g, device="cuda").sub_(0.5).to(BF) for _ in range(nbuf)]     # x: tokens x K
        sb = float(Bt[0].float().abs().max()) / 448.0
        bias = torch.rand(M, generator=g, device="cuda").sub_(0.5).to(BF)
        rows = torch.randperm(M, generator=torch.Generator().manual_seed(M))[:256]
        for kind in ("bf16", "fp8"):
            op = xs.Sp24(A if kind == "bf16" else A8)
            alpha = 1.0 if kind == "bf16" else sa * sb
            Bt_k = Bt if kind == "bf16" else [(b.float() / sb).to(F8) for b in Bt]
            Aref = A if kind == "bf16" else A8
            kw = {} if kind == "bf16" else {"alpha": alpha}
            for trans in ("T", "N"):
                Bs = Bt_k if trans == "T" else [b.t().contiguous() for b in Bt_k]
                cshape = (N, M) if trans == "T" else (M, N)
                C16 = [torch.zeros(cshape, dtype=BF, device="cuda") for _ in range(nbuf)]
                C32 = [torch.zeros(cshape, device="cuda") for _ in range(nbuf)]
                brow = bias[None, :] if trans == "T" else bias[:, None]
                for beta in ((0.0, 1.0) if (M, N, K) == (4096, 4096, 4096) else (0.0,)):
                    rec = {"gpu": name, "power_limit": power, "max_sm_clock": clock, "operator": kind, "M": M, "N": N, "K": K,
                           "transb": trans, "transc": trans, "beta": beta, "buffers": nbuf, "working_set_mb": round(nbuf * per / 2 ** 20),
                           "l2_note": "B and C rotate over buffers larger than twice the 126 MB L2"}
                    C0 = torch.rand(cshape, generator=g, device="cuda").sub_(0.5).to(BF)
                    for c in C16:
                        c.copy_(C0)
                    ex = lambda i, c, **k: op.execute(Bs[i], c, N, beta=beta, transb=trans, transc=trans, **kw, **k)   # noqa: E731
                    rec["a_bf16out"] = T(lambda i: ex(i, C16[i]))
                    rec["a_bf16out"]["kernel"] = xs.last_compute_kernel()
                    rec["b_bf16out_bias"] = T(lambda i: ex(i, C16[i], bias=bias))
                    rec["c_fp32out"] = T(lambda i: ex(i, C32[i]))
                    rec["d_fp32out_add_cast"] = T(lambda i: (ex(i, C32[i]), C32[i].add_(brow).to(BF)))
                    xs.check()
                    ca, cb = C0.clone(), C0.clone()
                    ex(0, ca)
                    ex(0, cb, bias=bias)
                    c32 = C0.float()
                    ex(0, c32)
                    torch.cuda.synchronize()
                    if beta == 0.0:
                        rec["a_same_bits_as_c_rounded"] = bool(torch.equal(ca.view(torch.int16), c32.to(BF).view(torch.int16)))
                    for key, c, bb in (("a", ca, None), ("b", cb, bias)):
                        ok, worst = f64_check(Aref, Bs[0], c, C0, bb, alpha, beta, trans, rows)
                        rec["%s_f64_bound_256_rows" % key], rec["%s_worst_err_over_bound" % key] = ok, round(worst, 4)
                    if beta == 0.0 and kind == "bf16":
                        if trans == "T":
                            rec["e_cublas_linear_bias"] = T(lambda i: torch.nn.functional.linear(Bs[i], A, bias))
                        else:
                            rec["e_cublas_addmm_bias"] = T(lambda i: torch.addmm(bias[:, None], A, Bs[i]))
                    if beta == 0.0 and kind == "fp8" and trans == "T":
                        sa_t, sb_t = torch.tensor(sa, device="cuda"), torch.tensor(sb, device="cuda")
                        try:
                            rec["f_scaled_mm_bias"] = T(lambda i: torch._scaled_mm(Bs[i], A8.t(), scale_a=sb_t, scale_b=sa_t, out_dtype=BF, bias=bias))
                        except RuntimeError as e:
                            rec["f_scaled_mm_bias"] = "unavailable: %s" % str(e).splitlines()[0]
                    if beta == 0.0 and trans == "T":
                        rec["g_linear"] = T(lambda i: op.linear(Bs[i], bias, **kw))
                    best = lambda k: rec[k]["best_us"] if isinstance(rec.get(k), dict) else None    # noqa: E731
                    rec["a_over_c"] = round(best("a_bf16out") / best("c_fp32out"), 3)
                    rec["b_over_a"] = round(best("b_bf16out_bias") / best("a_bf16out"), 3)
                    rec["a_over_d"] = round(best("a_bf16out") / best("d_fp32out_add_cast"), 3)
                    for k in ("e_cublas_linear_bias", "f_scaled_mm_bias"):
                        if best(k) and best("g_linear"):
                            rec["g_over_" + k[0]] = round(best("g_linear") / best(k), 3)
                    line = json.dumps(rec)
                    print(line, flush=True)
                    if out:
                        out.write(line + "\n")
                        out.flush()
                del C16, C32, Bs
            op.destroy()
            del Bt_k
        del Bt
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
