"""Batch solves with many right-hand sides per basis at scale: 1,024 bases of configs[1]'s shape (2,000 x 2,000,
gen.basis(seed, 2000, 700, 5.0)), factorized once and advanced by a few batch basis changes (untimed), so that the
solves run through row etas too.

GPU arm, each timed call after a warm-up call of the same shape:
  blu_batch_solve_sparse, 'N' and 'T', R in {1, 4, 16} right-hand sides per basis of 20 entries (gen.sparse_rhs);
  blu_batch_solve_dense_multi, R = 8.
For each: the host wall time around the C call (it ends in a stream synchronise), the kernel time from CUDA events
(blu_batch_last_kernel_ms(1): the compaction launch and every chunk), and microseconds per solve.  --sweep runs the
R = 16 sparse calls once per BLU_B200_SOLVE_UNITS value (read at batch creation) on a fresh batch.

CPU arm: the oracle on every host core, one instance per worker thread; each worker factorizes its basis and applies
the same basis changes untimed, then times only that basis' solves (a loop of ctypes calls, which release the GIL;
the comparison runs the solves again, untimed).  The
figure reported is the per-basis solve times summed and divided by the thread count.  Every solve of every basis is
compared with the GPU's: status, nzlhs, the order of ilhs and the values (np.array_equal).  The card's name and power
limit are read with nvidia-smi in the same run.  Prints one JSON object and writes it to --out."""
import argparse
import concurrent.futures
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from blu_b200 import BLUBatch, gen, load_library  # noqa: E402
from blu_b200.blu import f64p, i32p, i64p  # noqa: E402
from oracle_lib import Oracle  # noqa: E402

NNZ_RHS = 20


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return name, power


def bases(a):
    return [gen.basis(a.seed + k, a.m, a.nslack, 5.0) for k in range(a.nmat)]


def entering(a, k, it):
    cp, ri, v = gen.basis(a.seed + 500000 + k, a.m, 0, 3.0)
    return ri[cp[it]:cp[it + 1]], v[cp[it]:cp[it + 1]]


def leaving(il, xl):
    """the first (lowest) index of the largest |x|: what np.argmax over the scattered vector picks"""
    mx = np.abs(xl).max()
    return int(il[np.abs(xl) == mx].min()), float(xl[np.abs(xl) == mx][np.argmin(il[np.abs(xl) == mx])])


def gpu_batch(a, B, lib):
    b = BLUBatch(a.nmat, a.m, max(len(ri) for _, ri, _ in B), device=0 if lib is None else -1, lib=lib)
    off = np.cumsum([0] + [len(ri) for _, ri, _ in B])
    st, status = b.factorize(np.concatenate([cp[:-1] + off[k] for k, (cp, _, _) in enumerate(B)]),
                             np.concatenate([cp[1:] + off[k] for k, (cp, _, _) in enumerate(B)]),
                             np.concatenate([ri for _, ri, _ in B]), np.concatenate([v for _, _, v in B]))
    assert st == 0 and (status == 0).all(), status
    for it in range(a.updates):
        st, stat, out = b.solve_for_update([entering(a, k, it) for k in range(a.nmat)], "N", want_solution=1)
        assert st == 0
        lv = [leaving(*out[k]) for k in range(a.nmat)]
        st, _, _ = b.solve_for_update([(np.array([j]), None) for j, _ in lv], "T")
        assert st == 0
        st, _ = b.update(np.array([x for _, x in lv]))
        assert st == 0
    return b


class SparseCall:
    """the arguments of one blu_batch_solve_sparse call, built once, so that the timed window holds the C call only"""

    def __init__(self, a, R, seed):
        self.R = R
        self.rhs = [[gen.sparse_rhs(seed + k * R + r, a.m, NNZ_RHS) for r in range(R)] for k in range(a.nmat)]
        n = a.nmat * R
        self.unit_begin = np.arange(a.nmat + 1, dtype=np.int64) * R
        self.rhs_begin = np.arange(n + 1, dtype=np.int64) * NNZ_RHS
        self.irhs = np.concatenate([i for lst in self.rhs for i, _ in lst]).astype(np.int64)
        self.xrhs = np.concatenate([x for lst in self.rhs for _, x in lst])
        self.nz = np.zeros(n, np.int64); self.il = np.zeros(n * a.m, np.int64); self.xl = np.zeros(n * a.m)
        self.st = np.zeros(n, np.int32)

    def run(self, b, trans):
        L = b._L
        t0 = time.perf_counter()
        st = L.blu_batch_solve_sparse(b._h, self.unit_begin.ctypes.data_as(i64p), self.rhs_begin.ctypes.data_as(i64p),
                                      self.irhs.ctypes.data_as(i64p), self.xrhs.ctypes.data_as(f64p),
                                      self.nz.ctypes.data_as(i64p), self.il.ctypes.data_as(i64p),
                                      self.xl.ctypes.data_as(f64p), self.st.ctypes.data_as(i32p), trans.encode())
        return st, time.perf_counter() - t0, b.last_kernel_ms(1)

    def results(self, m):
        """per unit: (status, ilhs, values)"""
        return [(int(self.st[u]), self.il[u * m:u * m + max(int(self.nz[u]), 0)].copy(),
                 self.xl[u * m:u * m + max(int(self.nz[u]), 0)].copy()) for u in range(len(self.nz))]


def timed(fn, reps):
    fn()                        # warm-up call of the same shape
    runs = [fn() for _ in range(reps)]
    assert all(r[0] == 0 for r in runs), [r[0] for r in runs]
    return dict(wall_s=[r[1] for r in runs], kernel_ms=[r[2] for r in runs], wall_s_min=min(r[1] for r in runs),
                kernel_ms_min=min(r[2] for r in runs))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmat", type=int, default=1024)
    ap.add_argument("--m", type=int, default=2000)
    ap.add_argument("--nslack", type=int, default=700)
    ap.add_argument("--seed", type=int, default=60000)
    ap.add_argument("--updates", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rs", default="1,4,16")
    ap.add_argument("--dense-r", type=int, default=8)
    ap.add_argument("--sweep", default="", help="comma-separated BLU_B200_SOLVE_UNITS values for the R=16 sparse calls")
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--lib", default=None, help="another build of the library (a rehearsal under the emulator)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lib = load_library(a.lib) if a.lib else None
    name, power = gpu_card() if lib is None else ("not measured (emulator)", "n/a")
    B = bases(a)
    Rs = [int(r) for r in a.rs.split(",")]
    calls = {R: SparseCall(a, R, a.seed + 100000 * (i + 1)) for i, R in enumerate(Rs)}
    dense_rhs = np.random.default_rng(a.seed).uniform(-1.0, 1.0, (a.nmat, a.dense_r, a.m))

    b = gpu_batch(a, B, lib)
    gpu, got = {}, {}
    for R in Rs:
        for tr in "NT":
            l0 = b.launch_count()
            gpu[f"sparse_{tr}_R{R}"] = r = timed(lambda: calls[R].run(b, tr), a.reps)
            r["launches_per_call"] = int(b.launch_count() - l0) // (a.reps + 1)
            r["us_per_solve"] = 1e6 * r["wall_s_min"] / (a.nmat * R)
            r["kernel_us_per_solve"] = 1e3 * r["kernel_ms_min"] / (a.nmat * R)
            got[(R, tr)] = calls[R].results(a.m)
    dense_x = np.zeros_like(dense_rhs)
    dstat = np.zeros((a.nmat, a.dense_r), np.int32)

    def dense_call():
        t0 = time.perf_counter()
        st = b._L.blu_batch_solve_dense_multi(b._h, a.dense_r, dense_rhs.ctypes.data_as(f64p), dense_x.ctypes.data_as(f64p),
                                              b"N", dstat.ctypes.data_as(i32p))
        return st, time.perf_counter() - t0, b.last_kernel_ms(1)
    gpu[f"dense_multi_N_R{a.dense_r}"] = r = timed(dense_call, a.reps)
    r["us_per_solve"] = 1e6 * r["wall_s_min"] / (a.nmat * a.dense_r)
    r["kernel_us_per_solve"] = 1e3 * r["kernel_ms_min"] / (a.nmat * a.dense_r)
    del b

    sweep = {}
    for units in [int(u) for u in a.sweep.split(",") if u]:
        os.environ["BLU_B200_SOLVE_UNITS"] = str(units)
        bs = gpu_batch(a, B, lib)
        R = max(Rs)
        sweep[str(units)] = {tr: timed(lambda: calls[R].run(bs, tr), a.reps) for tr in "NT"}
        del bs
    os.environ.pop("BLU_B200_SOLVE_UNITS", None)

    def cpu_basis(k):
        cp, ri, v = B[k]
        o = Oracle(a.m, 60 * len(ri) + 100)
        assert o.factorize(cp[:-1], cp[1:], ri, v) == 0
        for it in range(a.updates):
            ii, xx = entering(a, k, it)
            assert o.solve_for_update(len(ii), ii, xx, "N", 1) == 0
            lhs = o.lhs
            j = int(np.argmax(np.abs(lhs)))
            assert o.solve_for_update(1, np.array([j]), None, "T", 0) == 0
            assert o.update(lhs[j]) == 0
        times, bad = {}, []
        for R in Rs:
            for tr in "NT":
                # timed: the ctypes calls alone; compared: the same solves again, untimed
                t0 = time.perf_counter()
                for ii, xx in calls[R].rhs[k]:
                    o.solve_sparse(len(ii), ii, xx, tr)
                times[(R, tr)] = time.perf_counter() - t0
                for r, (ii, xx) in enumerate(calls[R].rhs[k]):
                    st = o.solve_sparse(len(ii), ii, xx, tr)
                    gst, gil, gxl = got[(R, tr)][k * R + r]
                    n = o.nzlhs
                    ilo = o.ilhs[:n]
                    if not (st == gst == 0 and len(gil) == n and np.array_equal(gil, ilo) and np.array_equal(gxl, o.lhs[ilo])):
                        bad.append((R, tr, r))
        t0 = time.perf_counter()
        for r in range(a.dense_r):
            o.solve_dense(dense_rhs[k, r], "N")
        times[("dense", "N")] = time.perf_counter() - t0
        for r in range(a.dense_r):
            st, xo = o.solve_dense(dense_rhs[k, r], "N")
            if not (st == dstat[k, r] == 0 and np.array_equal(xo, dense_x[k, r])):
                bad.append((a.dense_r, "dense", r))
        return times, bad

    with concurrent.futures.ThreadPoolExecutor(max_workers=a.threads) as ex:
        cres = list(ex.map(cpu_basis, range(a.nmat)))
    cpu = {}
    for R in Rs:
        for tr in "NT":
            s = sum(t[(R, tr)] for t, _ in cres) / a.threads
            cpu[f"sparse_{tr}_R{R}"] = dict(seconds_sum_over_threads=s, us_per_solve=1e6 * s / (a.nmat * R))
    s = sum(t[("dense", "N")] for t, _ in cres) / a.threads
    cpu[f"dense_multi_N_R{a.dense_r}"] = dict(seconds_sum_over_threads=s, us_per_solve=1e6 * s / (a.nmat * a.dense_r))
    for key in gpu:
        gpu[key]["gpu_wall_over_cpu_speedup"] = cpu[key]["seconds_sum_over_threads"] / gpu[key]["wall_s_min"]
    mism = [(k, x) for k, (_, bad) in enumerate(cres) for x in bad]
    res = dict(
        workload=f"{a.nmat} bases of configs[1]'s shape (m={a.m}, gen.basis(seed, {a.m}, {a.nslack}, 5.0)), "
                 f"{a.updates} batch basis changes before the solves; sparse right-hand sides of {NNZ_RHS} entries "
                 f"(gen.sparse_rhs), dense ones uniform in [-1, 1]",
        card=name, power_limit=power, solve_units_default=8192,
        gpu=gpu, solve_units_sweep_R16=sweep,
        cpu_oracle=cpu, cpu_threads=a.threads,
        cpu_note="per-basis solve times (each a ctypes call of the oracle) summed over the bases, divided by the thread count",
        parity_every_solve_of_every_basis=len(mism) == 0, parity_mismatches=[list(map(str, x)) for x in mism[:10]],
    )
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")
    return 0 if not mism else 1


if __name__ == "__main__":
    sys.exit(main())
