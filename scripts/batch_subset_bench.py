"""The batch calls on a subset of the bases at scale: 4,096 bases of configs[1]'s shape (gen.batch(4096, 2000, 700,
5.0, ...)), factorized once, untimed.

(a) blu_batch_factorize_subset for nsel in {1, 16, 128, 512, 1,024, 4,096} bases spread over the batch, each
refactorizing from its own B (handed over compacted, as a caller holding only those bases would).  Wall time is the
host clock around the C call (it ends in a stream synchronise); kernel time is blu_batch_last_kernel_ms(0), every
kernel of the call, with the head / tail / build launches (3, 4, 5) and the condest kernel (2) also reported, so that
the rebuild of the resident B is kernel - head - tail - build - condest.  Min of 3 after a warm-up call.  Against
blu_batch_factorize of the whole batch in the same run, and the CPU oracle refactorizing the same nsel bases on every
host core (one oracle per worker thread).
(b) One basis change -- solve_for_update_subset 'N' (with the solution) and 'T', update_subset -- for nsel in
{64, 1,024, 4,096}, against the whole-batch calls: a warm-up step, then min of 3 steps per call.
Every factorization of a sample of the selected bases (16 spread over them) is compared with the oracle's
(get_factors); in (b) those bases' oracles follow every call they are selected in and their solutions, statuses and
getters are compared.  The card's name and power limit are read with nvidia-smi in the same run.  Prints one JSON
object and writes it to --out."""
import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from blu_b200 import BLUBatch, gen, load_library  # noqa: E402
from oracle_lib import Oracle  # noqa: E402


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return name, power


def spread(nmat, nsel):
    return np.unique(np.linspace(0, nmat - 1, nsel).round().astype(np.int64))


def compact(B, sel):
    """b_begin, b_end, b_i, b_x of the bases sel only"""
    off = np.cumsum([0] + [len(B[k][1]) for k in sel])
    return (np.concatenate([B[k][0][:-1] + off[r] for r, k in enumerate(sel)]),
            np.concatenate([B[k][0][1:] + off[r] for r, k in enumerate(sel)]),
            np.concatenate([B[k][1] for k in sel]), np.concatenate([B[k][2] for k in sel]))


def oracle(a, nnz):
    return Oracle(a.m, 20 * nnz + 100)


def check_factors(b, B, a, ks):
    for k in ks:
        cp, ri, v = B[k]
        o = oracle(a, len(v))
        assert o.factorize(cp[:-1], cp[1:], ri, v) == b.info(int(k), "status")
        sto, fo = o.get_factors()
        stg, fg = b.get_factors(int(k))
        assert sto == stg
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (k, key)


def cpu_refactor(a, B, sel):
    """the oracle refactorizing the bases sel on a.threads host threads (ctypes releases the GIL); wall seconds"""
    local = threading.local()
    maxnz = max(len(B[k][2]) for k in sel)

    def one(k):
        if not hasattr(local, "o"):
            local.o = oracle(a, maxnz)
        cp, ri, v = B[k]
        return local.o.factorize(cp[:-1], cp[1:], ri, v)

    with concurrent.futures.ThreadPoolExecutor(max_workers=a.threads) as ex:
        list(ex.map(one, sel[:a.threads]))                   # warm-up: every worker has its oracle
        t0 = time.perf_counter()
        st = list(ex.map(one, sel))
        t = time.perf_counter() - t0
    assert all(s == 0 for s in st)
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmat", type=int, default=4096)
    ap.add_argument("--m", type=int, default=2000)
    ap.add_argument("--nslack", type=int, default=700)
    ap.add_argument("--seed", type=int, default=70000)
    ap.add_argument("--nsel", default="1,16,128,512,1024,4096")
    ap.add_argument("--nsel-step", default="64,1024,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--lib", default=None, help="another build of the library (a rehearsal under the emulator)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lib = load_library(a.lib) if a.lib else None
    name, power = gpu_card() if lib is None else ("not measured (emulator)", "n/a")
    B = [gen.basis(a.seed + k, a.m, a.nslack, 5.0) for k in range(a.nmat)]
    allb = compact(B, range(a.nmat))
    b = BLUBatch(a.nmat, a.m, max(len(v) for _, _, v in B), device=0 if lib is None else -1, lib=lib)
    st, status = b.factorize(*allb)
    assert st == 0 and (status == 0).all()

    def timed(fn):
        fn()
        best = None
        for _ in range(a.reps):
            t0 = time.perf_counter()
            r = fn()
            t = time.perf_counter() - t0
            ks = {q: b.last_kernel_ms(q) for q in range(6)}
            if best is None or t < best[0]:
                best = (t, ks, r)
        return best

    t, ks, _ = timed(lambda: b.factorize(*allb))
    whole = dict(wall_ms=1e3 * t, kernel_ms=ks[0])
    fact = []
    for nsel in [int(x) for x in a.nsel.split(",")]:
        sel = spread(a.nmat, nsel)
        args = compact(B, sel)
        t, ks, r = timed(lambda: b.factorize_subset(sel, *args))
        assert r[0] == 0 and (r[1] == 0).all(), r
        check_factors(b, B, a, sel[::max(1, len(sel) // 16)])
        parts = ks[3] + ks[4] + ks[5]
        row = dict(nsel=int(len(sel)), wall_ms=1e3 * t, kernel_ms=ks[0], head_tail_build_ms=[ks[3], ks[4], ks[5]], condest_ms=ks[2],
                   rebuild_ms=ks[0] - parts - ks[2], cpu_oracle_ms=1e3 * cpu_refactor(a, B, list(sel)) if lib is None else None,
                   whole_batch_wall_ms=whole["wall_ms"])
        print(json.dumps(row), flush=True)
        fact.append(row)

    # (b) basis changes: the batch afresh, a sample of bases followed by oracles
    st, status = b.factorize(*allb)
    assert st == 0
    oracles, npool = {}, {}

    def follow(k):
        if k not in oracles:
            cp, ri, v = B[k]
            oracles[k] = oracle(a, len(v) + 8 * a.m)
            assert oracles[k].factorize(cp[:-1], cp[1:], ri, v) == 0
        return oracles[k]

    def entering(k):
        cp, ri, v = gen.basis(a.seed + 500000 + k, a.m, 0, 3.0)
        j = npool.get(k, 0)
        npool[k] = j + 1
        return ri[cp[j]:cp[j + 1]], v[cp[j]:cp[j + 1]]

    def step(sel, whole_batch, sample):
        cols = [entering(int(k)) for k in sel]
        t = []
        t0 = time.perf_counter()
        if whole_batch:
            st, stat, out = b.solve_for_update(cols, "N", want_solution=1)
        else:
            st, stat, out = b.solve_for_update_subset(sel, cols, "N", want_solution=1)
        t.append(time.perf_counter() - t0)
        assert st == 0, (st, stat)
        lv = []
        for r, k in enumerate(sel):
            il, xl = out[r]
            mx = np.abs(xl).max()
            j = int(il[np.abs(xl) == mx].min())
            lv.append((j, float(xl[il == j][0])))
        rhs_t = [(np.array([j]), None) for j, _ in lv]
        t0 = time.perf_counter()
        st, stat, _ = b.solve_for_update(rhs_t, "T") if whole_batch else b.solve_for_update_subset(sel, rhs_t, "T")
        t.append(time.perf_counter() - t0)
        assert st == 0
        xt = np.array([x for _, x in lv])
        t0 = time.perf_counter()
        st, stat = b.update(xt) if whole_batch else b.update_subset(sel, xt)
        t.append(time.perf_counter() - t0)
        assert st == 0 and (stat == 0).all()
        pos = {int(k): r for r, k in enumerate(sel)}
        for k in sample:
            o, r = follow(int(k)), pos[int(k)]
            assert o.solve_for_update(len(cols[r][0]), cols[r][0], cols[r][1], "N", 1) == 0
            n = o.nzlhs
            assert np.array_equal(out[r][0], o.ilhs[:n]) and np.array_equal(out[r][1], o.lhs[o.ilhs[:n]]), k
            assert o.solve_for_update(1, np.array([lv[r][0]]), None, "T", 0) == 0
            assert o.update(lv[r][1]) == 0
            for nm in ("nupdate", "nforrest", "u_nz", "r_nz", "pivot_error", "l_flops", "u_flops", "r_flops", "update_cost"):
                assert b.info(int(k), nm) == o.info(nm), (k, nm)
        return t

    changes = []
    for nsel in [int(x) for x in a.nsel_step.split(",")] + [0]:
        whole_batch = nsel == 0
        sel = np.arange(a.nmat) if whole_batch else spread(a.nmat, nsel)
        sample = [int(k) for k in sel[::max(1, len(sel) // 16)]]
        for k in sample:
            follow(k)
        step(sel, whole_batch, sample)
        ts = np.array([step(sel, whole_batch, sample) for _ in range(a.reps)])
        row = dict(nsel=int(len(sel)), call="whole batch" if whole_batch else "subset",
                   solve_n_ms=1e3 * ts[:, 0].min(), solve_t_ms=1e3 * ts[:, 1].min(), update_ms=1e3 * ts[:, 2].min())
        print(json.dumps(row), flush=True)
        changes.append(row)
    res = dict(card=name, power_limit=power, nmat=a.nmat, m=a.m, nslack=a.nslack, threads=a.threads,
               whole_batch_factorize=whole, factorize_subset=fact, basis_change=changes,
               checked="every factorization of 16 selected bases per nsel against the oracle's get_factors; in the "
                       "basis changes 16 selected bases per nsel followed by their oracles (solutions, statuses, getters)")
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
