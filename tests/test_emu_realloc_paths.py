"""The could-not-grow path of every call that grows the stores on Reallocate, under the SIMT emulator.

Two objects with the same history, the control with realloc_factor 1 and the probe, are driven in lockstep through
seeded basis changes on stores far too small.  At the first call of each kind during which the control grows a store,
the probe makes the same call with realloc_factor 1e12: every growth then fails its size guard and reports
BLU_ERROR_OUT_OF_MEMORY before it allocates anything.  The call's return value, its per-basis statuses and nzlhs and
its launch count are checked; then the probe, with the factor restored, repeats the call for the bases that could not
grow and must end exactly where the control is."""
import os
import subprocess

import numpy as np
import pytest
import torch

from blu_b200 import BLU, BLUBatch, load_library
from blu_b200.blu import i32p
from dev_cases import TWIN_GETTERS
from mv_cases import make_pool, run_batch
from subset_cases import Lane, _pf, _pi, csc, layout

HERE = os.path.dirname(os.path.abspath(__file__))
OOM = -102
HUGE = 1e12


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


def tight(obj):
    """stores of one entry without padding, grown by no more than asked: the spikes and etas outgrow them again and
    again"""
    if isinstance(obj, BLUBatch):
        obj.threads_per_basis = 64
    obj.realloc_factor = 1.0
    obj.l_mem = 1; obj.u_mem = 1; obj.w_mem = 1; obj.pad = 0; obj.stretch = 0.0
    return obj


def T(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype)


def solve(b, variant, sel, rhs, trans, want):
    """solve_for_update on the bases sel (every basis for the whole-batch call) -> (return value, status, nzlhs, [(ilhs,
    values)]) per selected basis; nzlhs and the solutions are None without want"""
    n, m, ns = b.nmat, b.m, len(sel)
    if variant == "dev":
        full = {k: rhs[r] for r, k in enumerate(sel)}
        ii = [np.asarray(full[k][0], np.int64) if k in full else np.zeros(0, np.int64) for k in range(n)]
        xx = None if rhs[0][1] is None else np.concatenate([full[k][1] if k in full else np.zeros(0) for k in range(n)])
        run = np.zeros(n, np.int32); run[sel] = 1
        st, s, nz, il, xl = b.solve_for_update_dev(T(np.cumsum([0] + [len(i) for i in ii]), torch.int64), T(np.concatenate(ii), torch.int64),
                                                   None if xx is None else T(xx, torch.float64), trans, want, run=T(run, torch.int32))
        s = s.numpy()[sel]
        if not want:
            return st, s, None, None
        nz, il, xl = nz.numpy()[sel], il.numpy()[sel], xl.numpy()[sel]
        return st, s, nz, [(il[r, :max(z, 0)], xl[r, :max(z, 0)]) for r, z in enumerate(nz)]
    begin = np.cumsum([0] + [len(ii) for ii, _ in rhs]).astype(np.int64)
    irhs = np.concatenate([np.asarray(ii, np.int64) for ii, _ in rhs])
    xrhs = None if rhs[0][1] is None else np.concatenate([x for _, x in rhs])
    nz, il, xl, stat = np.full(ns, 77, np.int64), np.zeros(ns * m, np.int64), np.zeros(ns * m), np.zeros(ns, np.int32)
    outs = (_pi(nz), _pi(il), _pf(xl)) if want else (None, None, None)
    if variant == "host":
        assert sel == list(range(n))
        st = b._L.blu_batch_solve_for_update(b._h, _pi(begin), _pi(irhs), _pf(xrhs), int(want), *outs, stat.ctypes.data_as(i32p),
                                             trans.encode())
    else:
        st = b._L.blu_batch_solve_for_update_subset(b._h, ns, _pi(np.asarray(sel, np.int64)), _pi(begin), _pi(irhs), _pf(xrhs),
                                                    int(want), *outs, stat.ctypes.data_as(i32p), trans.encode())
    if not want:
        return st, stat, None, None
    return st, stat, nz, [(il[r * m:r * m + max(z, 0)], xl[r * m:r * m + max(z, 0)]) for r, z in enumerate(nz)]


def update(b, variant, sel, xt):
    """update on the bases sel with xt[r] -> (return value, status per selected basis)"""
    if variant == "subset":
        return b.update_subset(sel, xt)
    x = np.full(b.nmat, np.nan)
    x[sel] = xt
    if variant == "host":
        assert sel == list(range(b.nmat))
        return b.update(x)
    run = np.zeros(b.nmat, np.int32); run[sel] = 1
    st, s = b.update_dev(T(x, torch.float64), run=T(run, torch.int32))
    return st, s.numpy()[sel]


def same(r, c):
    """two results of solve / update are equal"""
    assert r[0] == c[0] and np.array_equal(r[1], c[1])
    for q in (2, 3):
        if len(r) > q and r[q] is not None:
            x, y = r[q], c[q]
            assert (np.array_equal(x, y) if q == 2 else
                    all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(x, y)))


def launches(obj):
    return obj._L.blu_batch_launch_count(obj._h)


def assert_alike(ctl, prb, batch, skip):
    for k in range(ctl.nmat) if batch else [None]:
        for name in TWIN_GETTERS:
            if name in skip:
                continue
            a, b = (ctl.info(k, name), prb.info(k, name)) if batch else (ctl.info(name), prb.info(name))
            assert a == b or (a != a and b != b), (k, name, a, b)


class Lockstep:
    """control and probe through the same calls; probe(kind, call, redo) does a call on both and, the first time one of
    that kind grows a store of the control, makes the probe's copy fail to grow instead (see the module docstring).
    call(obj) -> result tuple (return value, statuses, ...); redo(probe, its result, the control's) checks the failed call
    and repeats it for the bases that could not grow.  self.hit records the launch count and the result of each probed
    call."""

    def __init__(self, ctl, prb, batch=True):
        self.ctl, self.prb, self.batch = ctl, prb, batch
        self.hit = {}

    def nrealloc(self, obj):
        return obj.info(0, "nrealloc") if self.batch else obj.info("nrealloc")

    def probe(self, kind, call, redo):
        nr = self.nrealloc(self.ctl)
        rc = call(self.ctl)
        if kind in self.hit or self.nrealloc(self.ctl) == nr:
            same(call(self.prb), rc)
            return rc
        self.prb.realloc_factor = HUGE
        l0 = launches(self.prb)
        rp = call(self.prb)
        self.hit[kind] = (launches(self.prb) - l0, rp)
        self.prb.realloc_factor = 1.0
        assert self.nrealloc(self.prb) == nr
        redo(self.prb, rp, rc)
        assert self.nrealloc(self.prb) == self.nrealloc(self.ctl)
        # an update that ran out of room had compressed its row file already, and the repeat compresses it again
        assert_alike(self.ctl, self.prb, self.batch, ("ngarbage",) if kind == "update" else ())
        return rc


def batch_drive(emu, variant, seed):
    """basis changes on four bases of m = 40 until an 'N' solve, a 'T' solve and an update have each been probed"""
    m, n = 40, 4
    lanes = [Lane(seed + k, m, nslack=10) for k in range(n)]
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m
    ls = Lockstep(*[tight(BLUBatch(n, m, cap, lib=emu)) for _ in range(2)])
    rng = np.random.default_rng(seed)

    def factorize(sel):
        for b in (ls.ctl, ls.prb):
            st, stat = b.factorize_subset(sel, *layout([lanes[k].cols for k in sel]))
            assert st == 0 and (stat == 0).all()

    def redo_solve(sel, rhs, trans, want):
        def redo(b, rp, rc):
            st, stat = rp[0], rp[1]
            oom = [r for r in range(len(sel)) if stat[r] != 0]
            assert oom and st == OOM and all(stat[r] == OOM for r in oom), (st, stat)
            ok = [r for r in range(len(sel)) if stat[r] == 0]
            assert np.array_equal(rc[1][ok], stat[ok])
            if want:
                assert all(rp[2][r] == -1 and len(rp[3][r][0]) == 0 for r in oom)
                assert all(rp[2][r] == rc[2][r] and np.array_equal(rp[3][r][1], rc[3][r][1]) for r in ok)
            again = solve(b, "subset", [sel[r] for r in oom], [rhs[r] for r in oom], trans, want)
            same(again, (0, rc[1][oom]) + ((rc[2][oom], [rc[3][r] for r in oom]) if want else (None, None)))
        return redo

    def redo_update(sel, xt):
        def redo(b, rp, rc):
            st, stat = rp
            oom = [r for r in range(len(sel)) if stat[r] != 0]
            assert oom and st == OOM and all(stat[r] == OOM for r in oom), (st, stat)
            assert all(stat[r] == rc[1][r] for r in range(len(sel)) if r not in oom)
            same(update(b, "subset", [sel[r] for r in oom], [xt[r] for r in oom]), (0, rc[1][oom]))
        return redo

    factorize(list(range(n)))
    for rd in range(40):
        sel = list(range(n)) if variant == "host" else sorted(set(rng.choice(n, int(rng.integers(1, n + 1)), replace=False).tolist()))
        cols = [lanes[k].next_column() for k in sel]
        want = rd % 2
        st, stat, nz, out = ls.probe("solve_n", lambda b: solve(b, variant, sel, cols, "N", 1), redo_solve(sel, cols, "N", 1))
        assert st == 0
        leave = [int(np.argmax(np.abs(x))) for _, x in out]
        rhs_t = [(np.array([out[r][0][leave[r]]]), None) for r in range(len(sel))]
        assert ls.probe("solve_t", lambda b: solve(b, variant, sel, rhs_t, "T", want), redo_solve(sel, rhs_t, "T", want))[0] == 0
        xt = [out[r][1][leave[r]] for r in range(len(sel))]
        st, stat = ls.probe("update", lambda b: update(b, variant, sel, xt), redo_update(sel, xt))
        refactor = []
        for r, k in enumerate(sel):
            if stat[r] == 0:
                lanes[k].cols[int(rhs_t[r][0][0])] = cols[r]
            if stat[r] != 0 or ls.ctl.info(k, "nforrest") >= 20:
                refactor.append(k)
        if refactor:
            factorize(refactor)
        if len(ls.hit) == 3:
            break
    return ls.hit


@pytest.mark.parametrize("variant", ["host", "subset", "dev"])
def test_emu_batch_could_not_grow(emu, variant):
    """blu_batch_solve_for_update / _update, their _subset and their _dev variants: the bases whose store could not
    grow report BLU_ERROR_OUT_OF_MEMORY (nzlhs -1), the others keep their results; the call returns the first of them;
    one launch of the kernel and nothing after it but what the call does anyway (the _dev calls: the argument check
    and k_dev_finish; the subset solve: the packing of the solutions that are there)."""
    hit = batch_drive(emu, variant, {"host": 41000, "subset": 41100, "dev": 41200}[variant])
    assert sorted(hit) == ["solve_n", "solve_t", "update"], sorted(hit)
    for kind, (launches, rp) in hit.items():
        if kind == "update":
            assert launches == {"host": 1, "subset": 1, "dev": 2}[variant], (kind, launches)
            continue
        want = rp[2] is not None
        packed = want and any(z > 0 for z in rp[2])
        assert launches == {"host": 1, "subset": 1 + packed, "dev": 3}[variant], (kind, launches)


def test_emu_object_could_not_grow(emu):
    """BLU.solve_for_update ('N' and 'T') and BLU.update return the failed growth's BLU_ERROR_OUT_OF_MEMORY after one
    launch; repeated with the factor restored, each call lands where the control is."""
    m = 40
    L = Lane(42000, m, nslack=10)
    cp, ri, v = csc(L.cols)
    ls = Lockstep(*[tight(BLU(m, len(v), lib=emu)) for _ in range(2)], batch=False)
    for obj in (ls.ctl, ls.prb):
        assert obj.factorize(cp[:-1], cp[1:], ri, v) == 0

    def solve(obj, ii, xx, trans, want):
        st = obj.solve_for_update(len(ii), ii, xx, trans, want_solution=want)
        nz = obj.nzlhs if want else 0
        return st, np.array([st]), np.array([nz]), [(obj.ilhs[:nz].copy(), obj.lhs[obj.ilhs[:nz]].copy())]

    def redo(call):
        def again(obj, rp, rc):
            assert rp[0] == OOM, rp[0]
            same(call(obj), rc)
        return again

    for rd in range(60):
        col = L.next_column()
        call_n = lambda obj: solve(obj, col[0], col[1], "N", 1)
        st, _, _, ((il, xl),) = ls.probe("solve_n", call_n, redo(call_n))
        assert st == 0
        q = int(np.argmax(np.abs(xl)))
        call_t = lambda obj: solve(obj, np.array([il[q]]), None, "T", rd % 2)
        assert ls.probe("solve_t", call_t, redo(call_t))[0] == 0
        call_u = lambda obj: (obj.update(xl[q]), np.zeros(1))
        if ls.probe("update", call_u, redo(call_u))[0] == 0:
            L.cols[int(il[q])] = col
        if ls.ctl.info("nforrest") >= 20 or ls.ctl.info("nupdate") < 0:
            cp, ri, v = csc(L.cols)
            for obj in (ls.ctl, ls.prb):
                assert obj.factorize(cp[:-1], cp[1:], ri, v) == 0
        if len(ls.hit) == 3:
            break
    assert sorted(ls.hit) == ["solve_n", "solve_t", "update"], sorted(ls.hit)
    assert all(l == 1 for l, _ in ls.hit.values()), ls.hit


@pytest.mark.parametrize("mem,nup,nlaunch", [
    ((5000, 600, 5000), [19, 20, 21], 180),       # U runs out first: in the 'N' solve
    ((400, 5000, 5000), [11, 11, 11], 95),        # L: in the 'T' solve and k_mv_absorb
    ((5000, 5000, 600), [17, 17, 18], 154),       # W: in the update and the refactorization decision
])
def test_emu_maxvolume_could_not_grow(emu, mem, nup, nlaunch):
    """blu_batch_maxvolume on three bases of m = 50: the first store that cannot grow stops the pass with
    BLU_ERROR_OUT_OF_MEMORY, every basis still running reports it with the updates it made; a second call with the
    factor restored gives what a batch that could grow all along gives."""
    m = 50
    pools = [make_pool(4600 + k, m, 70, scale=3.0) for k in range(3)]

    def batch():
        b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), lib=emu)
        b.threads_per_basis = 64
        b.l_mem, b.u_mem, b.w_mem = mem
        return b
    ctl, prb = batch(), batch()
    want = run_batch(ctl, pools, 1.2)
    assert want[0] == 0 and ctl.info(0, "nrealloc") > 0
    prb.realloc_factor = HUGE
    l0 = launches(prb)
    st, status, got_nup, _, _ = run_batch(prb, pools, 1.2)
    assert launches(prb) - l0 == nlaunch
    assert st == OOM and (status == OOM).all() and list(got_nup) == nup, (st, status, got_nup)
    assert prb.info(0, "nrealloc") == 0
    prb.realloc_factor = 1.0
    again = run_batch(prb, pools, 1.2)
    assert all(np.array_equal(x, y) for x, y in zip(again, want))
