"""The batch calls on host arrays against their variants on caller-owned device buffers (blu_batch_*_dev), at 4,096 bases
of configs[1]'s shape (gen.batch(4096, 2000, 700, 5.0, ...)).

Two batches with identical history, one driven through the host calls (numpy arrays), one through the _dev calls
(torch tensors on the GPU), in the same process; every measured call runs on both, alternating, and every output of the
device variant (statuses, nzlhs, the ilhs order, values) is compared with the host variant's.  Rows:
- one basis change ('N' with the solution, 'T', update) on the whole batch (d_run = NULL against the whole-batch calls)
  and on 64 bases (a device mask against the *_subset calls);
- solve_sparse with R = 16 right-hand sides of ~4 entries per basis;
- solve_dense_multi with R = 8;
- factorize_subset of 64 and of 4,096 bases.
Wall time is the host clock around one C call, which ends in a stream synchronise; min of 3 after a warm-up.  Kernel
time (the sum of the kernels' durations) and the H2D / D2H bytes per call come from a torch.profiler run of its own, one
call of each kind.  The card's name and power limit are read with nvidia-smi in the same run.  Prints one JSON object
and writes it to --out."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from blu_b200 import BLUBatch, gen  # noqa: E402
from blu_b200.blu import i32p  # noqa: E402

M, NSLACK = 2000, 700
CUDA = torch.device("cuda", 0)


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    return [s.strip() for s in out.split(",")]


def p64(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def pf(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def vp(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def T(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a)).to(CUDA).to(dtype)


class Step:
    """the inputs and outputs of one basis change of a selection (None: every basis) on both twins"""

    def __init__(self, nmat, sel, pool, it):
        self.nmat, self.sel = nmat, sel
        ks = list(range(nmat)) if sel is None else list(sel)
        pi, px, pb = pool
        cols = [(pi[pb[k * 8 + it % 8]:pb[k * 8 + it % 8 + 1]], px[pb[k * 8 + it % 8]:pb[k * 8 + it % 8 + 1]]) for k in ks]
        # host layout: compacted by selection; device layout: per basis, empty ranges for the others
        self.h_rb = np.concatenate([[0], np.cumsum([len(c[0]) for c in cols])]).astype(np.int64)
        self.h_ir = np.concatenate([c[0] for c in cols]).astype(np.int64)
        self.h_xr = np.concatenate([c[1] for c in cols])
        lens = np.zeros(nmat, np.int64)
        lens[ks] = [len(c[0]) for c in cols]
        order = np.argsort(ks)
        self.d_rb = T(np.concatenate([[0], np.cumsum(lens)]), torch.int64)
        self.d_ir = T(np.concatenate([cols[r][0] for r in order]), torch.int64)
        self.d_xr = T(np.concatenate([cols[r][1] for r in order]), torch.float64)
        self.ks = ks
        n = len(ks)
        self.h_out = (np.zeros(n, np.int64), np.zeros(n * M, np.int64), np.zeros(n * M), np.zeros(n, np.int32))
        self.d_out = (torch.zeros(nmat, dtype=torch.int64, device=CUDA), torch.zeros(nmat * M, dtype=torch.int64, device=CUDA),
                      torch.zeros(nmat * M, dtype=torch.float64, device=CUDA), torch.zeros(nmat, dtype=torch.int32, device=CUDA))
        run = np.zeros(nmat, np.int32); run[ks] = 1
        self.run = None if sel is None else T(run, torch.int32)
        self.sel64 = None if sel is None else np.ascontiguousarray(sel, np.int64)


def call_N(b, s, dev):
    L = b._L
    if dev:
        nz, il, xl, st = s.d_out
        return L.blu_batch_solve_for_update_dev(b._h, vp(s.run), vp(s.d_rb), vp(s.d_ir), vp(s.d_xr), 1, vp(nz), vp(il), vp(xl), vp(st), b"N")
    nz, il, xl, st = s.h_out
    if s.sel is None:
        return L.blu_batch_solve_for_update(b._h, p64(s.h_rb), p64(s.h_ir), pf(s.h_xr), 1, p64(nz), p64(il), pf(xl), st.ctypes.data_as(i32p), b"N")
    return L.blu_batch_solve_for_update_subset(b._h, len(s.sel64), p64(s.sel64), p64(s.h_rb), p64(s.h_ir), pf(s.h_xr), 1, p64(nz), p64(il),
                                               pf(xl), st.ctypes.data_as(i32p), b"N")


def leaving(s):
    """argmax |x| of each selected basis' 'N' solution (host twin's), in selection order; checks the device twin's"""
    nz, il, xl, st = s.h_out
    dnz, dil, dxl, dst = (t.cpu().numpy() for t in s.d_out)
    lv, xt = [], []
    for r, k in enumerate(s.ks):
        n = int(nz[r])
        assert st[r] == dst[k] == 0 and dnz[k] == n
        assert np.array_equal(il[r * M:r * M + n], dil[k * M:k * M + n]) and np.array_equal(xl[r * M:r * M + n], dxl[k * M:k * M + n])
        j = int(np.argmax(np.abs(xl[r * M:r * M + n])))
        lv.append(il[r * M + j]); xt.append(xl[r * M + j])
    return np.array(lv, np.int64), np.array(xt)


class StepT:
    def __init__(self, s, lv, xt):
        self.s = s
        self.h_rb = np.arange(len(lv) + 1, dtype=np.int64)
        self.h_ir, self.h_xt = lv, xt
        dl = np.zeros(s.nmat, np.int64); dl[s.ks] = lv
        dx = np.zeros(s.nmat); dx[s.ks] = xt
        self.d_rb = T(np.arange(s.nmat + 1), torch.int64)
        self.d_ir, self.d_xt = T(dl, torch.int64), T(dx, torch.float64)
        self.h_st = np.zeros(len(lv), np.int32)
        self.d_st = torch.zeros(s.nmat, dtype=torch.int32, device=CUDA)


def call_T(b, t, dev):
    L, s = b._L, t.s
    if dev:
        return L.blu_batch_solve_for_update_dev(b._h, vp(s.run), vp(t.d_rb), vp(t.d_ir), None, 0, None, None, None, vp(t.d_st), b"T")
    if s.sel is None:
        return L.blu_batch_solve_for_update(b._h, p64(t.h_rb), p64(t.h_ir), None, 0, None, None, None, t.h_st.ctypes.data_as(i32p), b"T")
    return L.blu_batch_solve_for_update_subset(b._h, len(s.sel64), p64(s.sel64), p64(t.h_rb), p64(t.h_ir), None, 0, None, None, None,
                                               t.h_st.ctypes.data_as(i32p), b"T")


def call_U(b, t, dev):
    L, s = b._L, t.s
    if dev:
        return L.blu_batch_update_dev(b._h, vp(s.run), vp(t.d_xt), vp(t.d_st))
    if s.sel is None:
        return L.blu_batch_update(b._h, pf(t.h_xt), t.h_st.ctypes.data_as(i32p))
    return L.blu_batch_update_subset(b._h, len(s.sel64), p64(s.sel64), pf(t.h_xt), t.h_st.ctypes.data_as(i32p))


def check_status(t):
    d = t.d_st.cpu().numpy()
    assert (t.h_st == 0).all() and all(d[k] == 0 for k in t.s.ks)


def timed(fn):
    t0 = time.perf_counter()
    st = fn()
    dt = time.perf_counter() - t0
    assert st == 0, st
    return dt * 1e3


def profile(fns):
    """kernel milliseconds and H2D / D2H bytes of each fn, from one torch.profiler run"""
    out = []
    for fn in fns:
        path = os.path.join(tempfile.mkdtemp(), "t.json")
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
            assert fn() == 0
            torch.cuda.synchronize()
        prof.export_chrome_trace(path)
        ev = json.load(open(path))["traceEvents"]
        kms = sum(e.get("dur", 0) for e in ev if e.get("cat") == "kernel") / 1e3
        h2d = sum(int(e["args"].get("bytes", 0)) for e in ev if e.get("cat") == "gpu_memcpy" and "HtoD" in e.get("name", ""))
        d2h = sum(int(e["args"].get("bytes", 0)) for e in ev if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", ""))
        out.append(dict(kernel_ms=round(kms, 3), h2d_bytes=h2d, d2h_bytes=d2h))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmat", type=int, default=4096)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "batch_dev_b200.json"))
    a = ap.parse_args()
    nmat = a.nmat
    name, power = gpu_card()
    bb, be, bi, bx, _ = gen.batch(nmat, M, NSLACK, 5.0, 50000, 60000)
    cap = int((be - bb).reshape(nmat, M).sum(1).max()) + 4 * M
    h, d = BLUBatch(nmat, M, cap, device=0), BLUBatch(nmat, M, cap, device=0)
    assert h.factorize(bb, be, bi, bx)[0] == 0 and d.factorize(bb, be, bi, bx)[0] == 0
    # 8 entering columns per basis
    idx, val, begin = [], [], [0]
    for k in range(nmat):
        cp, ri, v = gen.basis(70000 + k, M, 0, 3.0)
        for c in range(8):
            idx.append(ri[cp[c]:cp[c + 1]]); val.append(v[cp[c]:cp[c + 1]]); begin.append(begin[-1] + cp[c + 1] - cp[c])
    pool = (np.concatenate(idx).astype(np.int64), np.concatenate(val), np.array(begin, np.int64))
    rows = []
    it = [0]

    def step_rows(label, sel):
        res = {"N": [], "T": [], "update": []}
        for rep in range(4):
            s = Step(nmat, sel, pool, it[0]); it[0] += 1
            wN = [timed(lambda: call_N(h, s, False)), timed(lambda: call_N(d, s, True))]
            lv, xt = leaving(s)
            t = StepT(s, lv, xt)
            wT = [timed(lambda: call_T(h, t, False)), timed(lambda: call_T(d, t, True))]
            check_status(t)
            wU = [timed(lambda: call_U(h, t, False)), timed(lambda: call_U(d, t, True))]
            check_status(t)
            if rep:
                res["N"].append(wN); res["T"].append(wT); res["update"].append(wU)
        # one more step for the profile
        s = Step(nmat, sel, pool, it[0]); it[0] += 1
        pN = profile([lambda: call_N(h, s, False), lambda: call_N(d, s, True)])
        lv, xt = leaving(s)
        t = StepT(s, lv, xt)
        pT = profile([lambda: call_T(h, t, False), lambda: call_T(d, t, True)])
        pU = profile([lambda: call_U(h, t, False), lambda: call_U(d, t, True)])
        for call, w, p in (("N", res["N"], pN), ("T", res["T"], pT), ("update", res["update"], pU)):
            rows.append(dict(row=f"{label} {call}", host_wall_ms=round(min(x[0] for x in w), 3), dev_wall_ms=round(min(x[1] for x in w), 3),
                             host=p[0], dev=p[1]))

    step_rows("basis change, all 4,096", None)
    step_rows("basis change, 64 in the mask", np.unique(np.linspace(0, nmat - 1, 64).round().astype(np.int64)))

    # solve_sparse, R = 16 right-hand sides of 4 entries per basis
    R = 16
    nunits = R * nmat
    rng = np.random.default_rng(3)
    ir = np.concatenate([np.sort(rng.choice(M, 4, replace=False)) for _ in range(nunits)]).astype(np.int64)
    xr = rng.uniform(-1, 1, len(ir))
    ub = np.arange(0, nunits + 1, R, dtype=np.int64)
    rb = np.arange(0, 4 * nunits + 1, 4, dtype=np.int64)
    hN = (np.zeros(nunits, np.int64), np.zeros(nunits * M, np.int64), np.zeros(nunits * M), np.zeros(nunits, np.int32))
    dN = (torch.zeros(nunits, dtype=torch.int64, device=CUDA), torch.zeros(nunits * M, dtype=torch.int64, device=CUDA),
          torch.zeros(nunits * M, dtype=torch.float64, device=CUDA), torch.zeros(nunits, dtype=torch.int32, device=CUDA))
    dub, drb, dir_, dxr = T(ub, torch.int64), T(rb, torch.int64), T(ir, torch.int64), T(xr, torch.float64)
    hs = lambda: h._L.blu_batch_solve_sparse(h._h, p64(ub), p64(rb), p64(ir), pf(xr), p64(hN[0]), p64(hN[1]), pf(hN[2]), hN[3].ctypes.data_as(i32p), b"N")
    ds = lambda: d._L.blu_batch_solve_sparse_dev(d._h, nunits, vp(dub), vp(drb), vp(dir_), vp(dxr), vp(dN[0]), vp(dN[1]), vp(dN[2]), vp(dN[3]), b"N")
    w = [[timed(hs), timed(ds)] for _ in range(4)][1:]
    nz, il, xl, st = (t.cpu().numpy() for t in dN)
    assert np.array_equal(nz, hN[0]) and np.array_equal(st, hN[3])
    for u in range(nunits):
        n = int(nz[u])
        assert np.array_equal(il[u * M:u * M + n], hN[1][u * M:u * M + n]) and np.array_equal(xl[u * M:u * M + n], hN[2][u * M:u * M + n])
    p = profile([hs, ds])
    rows.append(dict(row="solve_sparse R = 16", host_wall_ms=round(min(x[0] for x in w), 3), dev_wall_ms=round(min(x[1] for x in w), 3),
                     host=p[0], dev=p[1]))
    del dN, hN

    # solve_dense_multi, R = 8
    R = 8
    rhs = np.random.default_rng(4).uniform(-1, 1, nmat * R * M)
    hx, hst = np.zeros(nmat * R * M), np.zeros(nmat * R, np.int32)
    drhs, dx, dst = T(rhs, torch.float64), torch.zeros(nmat * R * M, dtype=torch.float64, device=CUDA), torch.zeros(nmat * R, dtype=torch.int32, device=CUDA)
    hd = lambda: h._L.blu_batch_solve_dense_multi(h._h, R, pf(rhs), pf(hx), b"N", hst.ctypes.data_as(i32p))
    dd = lambda: d._L.blu_batch_solve_dense_multi_dev(d._h, R, vp(drhs), vp(dx), b"N", vp(dst))
    w = [[timed(hd), timed(dd)] for _ in range(4)][1:]
    assert np.array_equal(dx.cpu().numpy(), hx) and np.array_equal(dst.cpu().numpy(), hst)
    p = profile([hd, dd])
    rows.append(dict(row="solve_dense_multi R = 8", host_wall_ms=round(min(x[0] for x in w), 3), dev_wall_ms=round(min(x[1] for x in w), 3),
                     host=p[0], dev=p[1]))
    del drhs, dx

    # factorize_subset of 64 and of all bases, each from its original B
    dB = [T(x, dt) for x, dt in ((bb, torch.int64), (be, torch.int64), (bi, torch.int64), (bx, torch.float64))]
    for nsel in (64, nmat):
        sel = np.unique(np.linspace(0, nmat - 1, nsel).round().astype(np.int64))
        cb = np.concatenate([bb[k * M:(k + 1) * M] for k in sel]); ce = np.concatenate([be[k * M:(k + 1) * M] for k in sel])
        run = np.zeros(nmat, np.int32); run[sel] = 1
        drun = T(run, torch.int32)
        hst, dst = np.zeros(nsel, np.int32), torch.zeros(nmat, dtype=torch.int32, device=CUDA)
        hf = lambda: h._L.blu_batch_factorize_subset(h._h, nsel, p64(sel), p64(cb), p64(ce), p64(bi), pf(bx), len(bi), hst.ctypes.data_as(i32p))
        df = lambda: d._L.blu_batch_factorize_subset_dev(d._h, vp(drun), vp(dB[0]), vp(dB[1]), vp(dB[2]), vp(dB[3]), len(bi), vp(dst))
        w, kms = [], []
        for _ in range(4):
            w.append([timed(hf), timed(df)])
            kms.append([h.last_kernel_ms(0), d.last_kernel_ms(0)])
        w, kms = w[1:], kms[1:]
        assert (hst == 0).all() and (dst.cpu().numpy()[sel] == 0).all()
        for k in sel[::max(1, nsel // 16)]:
            fh, fd = h.get_factors(int(k))[1], d.get_factors(int(k))[1]
            assert all(np.array_equal(fh[q], fd[q]) for q in fh), k
        p = profile([hf, df])
        rows.append(dict(row=f"factorize_subset {nsel}", host_wall_ms=round(min(x[0] for x in w), 3), dev_wall_ms=round(min(x[1] for x in w), 3),
                         host=dict(p[0], last_kernel_ms=round(min(x[0] for x in kms), 3)),
                         dev=dict(p[1], last_kernel_ms=round(min(x[1] for x in kms), 3))))
    res = dict(gpu=name, power_limit=power, nmat=nmat, m=M, workload="gen.batch(4096, 2000, 700, 5.0, 50000, 60000)",
               timing="wall: host clock around one C call ending in a stream synchronise, min of 3 after a warm-up; kernel_ms and "
                      "bytes: one call in a torch.profiler run of its own (sum of kernel durations, memcpy bytes by direction)",
               rows=rows)
    print(json.dumps(res))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
