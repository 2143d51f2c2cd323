"""Developer tool: times the indexed SoA entries (libxsmm_b200_rm_soa_execute_indexed, libxsmm_b200_csr_soa_execute_indexed)
against the strided ones and against today's alternative, a torch.index_select gather into a compact buffer before the strided
call (and an index_copy_ of C back for a subset).

    python tools/time_soa_indexed.py [--reps 30] [--warmup 5] [--parent-lib path/to/libxsmm_b200.so] [--only W1,soa]

Workloads: W1 (rm_ac fp64 35x9x9, soa 8, b per element) and W2 (rm_bc fp64 35x9x35, a shared) of tools/time_rm_soa.py, and
bench.py's `soa` / `soa-b` csr_soa cases; 65536 elements, beta = 1.  Every working set is over a gigabyte, well past the 126 MB
L2.  Modes: strided (with --parent-lib: the parent build's strided entry, alternated launch by launch with this build's),
identity index arrays, a random permutation of the input slots, four face calls with random neighbour maps of the SoA input, a
sorted random half of the slots for every operand; and the gather-copy alternative of the last three.  Best and median per
call (per four calls for the neighbour mode) over --reps calls after --warmup, by CUDA events.  C is checked bit for bit
between the strided and identity modes (and the parent's strided entry) at the timed sizes.  One JSON line per workload and
mode; the card's name and power limit are read in the same run.
"""
import argparse
import ctypes
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_rm_soa import card  # noqa: E402

E = 65536
VP, LL = ctypes.c_void_p, ctypes.c_longlong


class Case:
    """one workload: its operands as torch tensors [slots, extent] (a shared operand: [1, extent]), which of them are per
    element, and strided / indexed launchers for this build and (optionally) the parent build"""

    def __init__(self, xs, wid, parent):
        self.xs, self.wid = xs, wid
        dt = torch.float64
        g = torch.Generator(device="cuda").manual_seed(1)
        if wid in ("W1", "W2"):
            form = "ac" if wid == "W1" else "bc"
            M, N, K, soa = (35, 9, 9, 8) if wid == "W1" else (35, 9, 35, 8)
            self.op = xs.RmSoa(form, M, N, K, soa, np.float64, beta=1.0)
            ea, eb, ec = self.op.extents
            shared = [wid == "W2", False]                       # W2: a shared by all elements
            self.ins = [torch.rand((1 if s else E, x), generator=g, device="cuda", dtype=dt) for x, s in zip((ea, eb), shared)]
            self.soa_in = 0 if form == "ac" else 1                 # the SoA input (the one neighbour maps apply to)
            if parent:
                f = getattr(parent, "libxsmm_b200_drm_%s_soa_create" % form)
                f.restype = VP
                f.argtypes = [ctypes.c_int] * 7 + [ctypes.c_double]
                self.ph = f(M, N, K, K, N, N, soa, 1.0)
                parent.libxsmm_b200_rm_soa_execute.argtypes = [VP] * 4 + [LL] * 4 + [VP]
        else:
            d = np.load(os.path.join(ROOT, "tests", "golden", "csr_soa.npz"))
            key, bsp = ("tet4_4_stiffV_0_d", False) if wid == "soa" else ("bsp_tet4_4_stiffV_0_d", True)
            M, K, N, soa, _ = (int(v) for v in d[key + "_shape"])
            rp, ci, va = (np.ascontiguousarray(d[key + s]) for s in ("_rowptr", "_colidx", "_values"))
            self.op = xs.CsrSoa(M, N, K, rp, ci, va, soa, beta=1.0, sparse="B" if bsp else "A")
            ex, ec = (M * K if bsp else K * N) * soa, M * N * soa
            shared = [False]
            self.ins = [torch.rand((E, ex), generator=g, device="cuda", dtype=dt)]
            self.soa_in = 0
            if parent:
                f = parent.libxsmm_b200_dcsr_soa_create
                f.restype = VP
                f.argtypes = [ctypes.c_int] * 7 + [ctypes.c_double] + [VP] * 3
                self.ph = f(M, N, K, K if bsp else 0, 0 if bsp else N, N, soa, 1.0, rp.ctypes.data, ci.ctypes.data, va.ctypes.data)
                parent.libxsmm_b200_csr_soa_execute.argtypes = [VP] * 3 + [LL] * 3 + [VP]
        self.shared = shared
        self.parent = parent
        self.C0 = torch.rand((E, ec), generator=g, device="cuda", dtype=dt)
        self.C = self.C0.clone()
        self.compact = [torch.empty((E, t.shape[1]), device="cuda", dtype=dt) for t in self.ins]
        self.compact_c = torch.empty_like(self.C)
        self.st = [0 if s else t.shape[1] for t, s in zip(self.ins, shared)]

    def strided(self, ins, C, n):
        if isinstance(self.op, self.xs.RmSoa):
            self.op.execute(ins[0].data_ptr(), ins[1].data_ptr(), C.data_ptr(), n, self.st[0], self.st[1], C.shape[1])
        else:
            self.op.execute(ins[0].data_ptr(), C.data_ptr(), n, self.st[0], C.shape[1])

    def strided_parent(self):
        P = self.parent
        if isinstance(self.op, self.xs.RmSoa):
            P.libxsmm_b200_rm_soa_execute(self.ph, self.ins[0].data_ptr(), self.ins[1].data_ptr(), self.C.data_ptr(), E,
                                          self.st[0], self.st[1], self.C.shape[1], None)
        else:
            P.libxsmm_b200_csr_soa_execute(self.ph, self.ins[0].data_ptr(), self.C.data_ptr(), E, self.st[0], self.C.shape[1], None)

    def indexed(self, idx_in, idx_c, n):
        """idx_in: one int32 index tensor (or None) per input; idx_c for C"""
        p = [None if i is None else i.data_ptr() for i in idx_in]
        slots = [t.shape[0] for t in self.ins]
        pc = None if idx_c is None else idx_c.data_ptr()
        if isinstance(self.op, self.xs.RmSoa):
            self.op.execute_indexed(self.ins[0].data_ptr(), self.ins[1].data_ptr(), self.C.data_ptr(), n, p[0], slots[0], p[1], slots[1],
                                    pc, E, self.st[0], self.st[1], self.C.shape[1])
        else:
            self.op.execute_indexed(self.ins[0].data_ptr(), self.C.data_ptr(), n, p[0], slots[0], pc, E, self.st[0], self.C.shape[1])

    def gathered(self, idx_in_long, idx_c_long, n):
        """today's alternative: gather the indexed inputs (and C for a subset) into compact buffers, strided call, C back"""
        ins = []
        for t, i, buf in zip(self.ins, idx_in_long, self.compact):
            if i is None:
                ins.append(t)
            else:
                torch.index_select(t, 0, i, out=buf[:n])
                ins.append(buf)
        if idx_c_long is None:
            self.strided(ins, self.C, n)
        else:
            cc = self.compact_c[:n]
            torch.index_select(self.C, 0, idx_c_long, out=cc)
            self.strided(ins, cc, n)
            self.C.index_copy_(0, idx_c_long, cc)


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for i in range(reps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return np.array([ev[i].elapsed_time(ev[i + 1]) for i in range(reps)])


def alternated(fa, fb, reps, warmup):
    """fa and fb launch by launch in turn"""
    for _ in range(warmup):
        fa(); fb()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * reps + 1)]
    ev[0].record()
    for i in range(reps):
        fa(); ev[2 * i + 1].record()
        fb(); ev[2 * i + 2].record()
    torch.cuda.synchronize()
    t = np.array([ev[i].elapsed_time(ev[i + 1]) for i in range(2 * reps)])
    return t[0::2], t[1::2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--parent-lib", default=None, help="libxsmm_b200.so of the parent build: its strided entry is timed alternately")
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    xs = importlib.import_module("libxsmm-1_b200")
    xs.require_gpu()
    parent = ctypes.CDLL(os.path.abspath(args.parent_lib)) if args.parent_lib else None
    name, power = card()
    rng = np.random.default_rng(5)

    def i32(a):
        return torch.as_tensor(np.asarray(a, np.int32), device="cuda")

    def i64(a):
        return torch.as_tensor(np.asarray(a, np.int64), device="cuda")

    for wid in (args.only.split(",") if args.only else ("W1", "W2", "soa", "soa-b")):
        c = Case(xs, wid, parent)
        res = {}
        # C bits: strided vs identity (vs the parent's strided entry), from the same C0
        ident = np.arange(E)
        c_ident = i32(ident)
        idx_ident = [None if s else c_ident for s in c.shared]
        c.C.copy_(c.C0); c.strided(c.ins, c.C, E); torch.cuda.synchronize(); ref = c.C.clone()
        c.C.copy_(c.C0); c.indexed(idx_ident, c_ident, E); torch.cuda.synchronize()
        same_identity = bool(torch.equal(c.C.view(torch.int64), ref.view(torch.int64)))
        same_parent = None
        if parent:
            c.C.copy_(c.C0); c.strided_parent(); torch.cuda.synchronize()
            same_parent = bool(torch.equal(c.C.view(torch.int64), ref.view(torch.int64)))
        xs.check()
        c.C.copy_(c.C0)
        if parent:
            res["strided-parent"], res["strided"] = alternated(c.strided_parent, lambda: c.strided(c.ins, c.C, E), args.reps, args.warmup)
        else:
            res["strided"] = timed(lambda: c.strided(c.ins, c.C, E), args.reps, args.warmup)
        res["identity"] = timed(lambda: c.indexed(idx_ident, c_ident, E), args.reps, args.warmup)
        perm = rng.permutation(E)
        p32, p64 = i32(perm), i64(perm)
        pin32 = [None if s else p32 for s in c.shared]
        pin64 = [None if s else p64 for s in c.shared]
        res["permuted"] = timed(lambda: c.indexed(pin32, None, E), args.reps, args.warmup)
        res["permuted-gather"] = timed(lambda: c.gathered(pin64, None, E), args.reps, args.warmup)
        nb = [rng.integers(0, E, E) for _ in range(4)]
        nb32 = [[p if k == c.soa_in else None for k in range(len(c.ins))] for p in (i32(x) for x in nb)]
        nb64 = [[p if k == c.soa_in else None for k in range(len(c.ins))] for p in (i64(x) for x in nb)]

        def faces():
            for f in range(4):
                c.indexed(nb32[f], None, E)

        def faces_gather():
            for f in range(4):
                c.gathered(nb64[f], None, E)
        res["neighbour4"] = timed(faces, args.reps, args.warmup)
        res["neighbour4-gather"] = timed(faces_gather, args.reps, args.warmup)
        sub = np.sort(rng.choice(E, E // 2, replace=False))
        s32, s64 = i32(sub), i64(sub)
        res["subset"] = timed(lambda: c.indexed([None if s else s32 for s in c.shared], s32, E // 2), args.reps, args.warmup)
        res["subset-gather"] = timed(lambda: c.gathered([None if s else s64 for s in c.shared], s64, E // 2), args.reps, args.warmup)
        torch.cuda.synchronize()
        xs.check()
        for mode, t in res.items():
            line = {"workload": wid, "mode": mode, "elements": E // 2 if mode.startswith("subset") else E,
                    "calls_per_sample": 4 if mode.startswith("neighbour") else 1, "samples": len(t),
                    "best_ms": round(float(t.min()), 4), "median_ms": round(float(np.median(t)), 4),
                    "c_bits_identity_equal_strided": same_identity, "card": name, "power_limit": power}
            if same_parent is not None:
                line["c_bits_parent_equal_strided"] = same_parent
            print(json.dumps(line), flush=True)
        c.op.destroy()


if __name__ == "__main__":
    main()
