"""blu_solve_dense_multi / blu_solve_sparse_multi of a BLU object under the SIMT emulator: many right-hand sides against
the object's one factorization equal one-by-one oracle solves, in chunks of BLU_B200_SOLVE_UNITS units, around a pending
basis change, and after batch calls made on the object; a malformed rhs_begin is refused before anything runs."""
import os
import subprocess

import numpy as np
import pytest

from blu_b200 import BLU, gen, load_library
from blu_b200.blu import i32p
from parity import oracle_for
from subset_cases import _pf, _pi

HERE = os.path.dirname(os.path.abspath(__file__))
INVALID_CALL, INVALID_ARGUMENT = -2, -4
COUNTERS = ("l_flops", "u_flops", "r_flops", "update_cost", "nupdate", "nforrest", "u_nz", "r_nz", "pivot_error", "max_eta")


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


def pair(emu, m, seed):
    cp, ri, v = gen.basis(seed, m, 30, 4.0)
    o = oracle_for(m, len(v))
    g = BLU(m, len(v), lib=emu)
    assert o.factorize(cp[:-1], cp[1:], ri, v) == g.factorize(cp[:-1], cp[1:], ri, v) == 0
    return g, o


def launches(g):
    return g._L.blu_batch_launch_count(g._h)


def sparse_multi(g, rhs, trans, begin=None, fill=0.0):
    """the raw call on output arrays prefilled with fill -> (status, nzlhs, ilhs[nrhs, m], xlhs[nrhs, m], status[])"""
    n, m = len(rhs), g.m
    if begin is None:
        begin = np.cumsum([0] + [len(i) for i, _ in rhs]).astype(np.int64)
    irhs = np.concatenate([np.asarray(i, np.int64) for i, _ in rhs])
    xrhs = np.concatenate([np.asarray(x, np.float64) for _, x in rhs])
    nz, stat = np.full(n, 77, np.int64), np.full(n, 77, np.int32)
    il, xl = np.full(n * m, int(fill), np.int64), np.full(n * m, fill)
    st = g._L.blu_solve_sparse_multi(g._h, n, _pi(begin), _pi(irhs), _pf(xrhs), _pi(nz), _pi(il), _pf(xl),
                                     stat.ctypes.data_as(i32p), trans.encode())
    return st, nz, il.reshape(n, m), xl.reshape(n, m), stat


def sparse_rhs(m, seed, n):
    """n right-hand sides of 1 .. m/2 entries; the first one has half of m, so that row 0 is in most solutions"""
    sizes = [m // 2] + [1 + (7 * k) % (m // 2) for k in range(1, n)]
    return [gen.sparse_rhs(seed + k, m, nz) for k, nz in enumerate(sizes)]


def assert_sparse(g, o, rhs, trans):
    st, nz, il, xl, stat = sparse_multi(g, rhs, trans)
    assert st == 0 and (stat == 0).all()
    for r, (idx, val) in enumerate(rhs):
        assert o.solve_sparse(len(idx), idx, val, trans) == 0
        n = o.nzlhs
        assert nz[r] == n and np.array_equal(il[r, :n], o.ilhs[:n]), (trans, r)
        assert np.array_equal(xl[r, :n], o.lhs[o.ilhs[:n]]), (trans, r)
    return nz, il, xl


def assert_dense(g, o, R, trans):
    st, X = g.solve_dense_multi(R, trans)
    assert st == 0
    for r in range(len(R)):
        assert np.array_equal(X[r], o.solve_dense(R[r], trans)[1]), (trans, r)


def assert_counters(g, o):
    for name in COUNTERS:
        assert g.info(name) == o.info(name), name


def test_emu_object_multi_after_batch_update(emu):
    """A batch basis-change call on the object that it refuses leaves the object's multi solves as they were."""
    m = 120
    g, o = pair(emu, m, 3100)
    rhs = sparse_rhs(m, 3200, 6)
    first = [sparse_multi(g, rhs, tr) for tr in "NT"]
    stat = np.full(1, 77, np.int32)
    assert g._L.blu_batch_update(g._h, _pf(np.array([2.5])), stat.ctypes.data_as(i32p)) == INVALID_CALL
    assert stat[0] == INVALID_CALL
    for tr, a in zip("NT", first):
        b = sparse_multi(g, rhs, tr)
        assert b[0] == a[0] == 0 and np.array_equal(a[1], b[1]) and np.array_equal(a[4], b[4])
        for r, n in enumerate(a[1]):      # entries past nzlhs[r] are unspecified
            assert np.array_equal(a[2][r, :n], b[2][r, :n]) and np.array_equal(a[3][r, :n], b[3][r, :n]), (tr, r)
    for tr in "NT":
        assert_sparse(g, o, rhs, tr)      # and still the oracle's


def test_emu_object_multi_chunks(emu, monkeypatch):
    """With BLU_B200_SOLVE_UNITS=3, 8 right-hand sides run as 3 + 3 + 2 units: the results are those of one-by-one
    solves, and each call is one compaction launch and one launch per chunk."""
    monkeypatch.setenv("BLU_B200_SOLVE_UNITS", "3")
    m = 110
    g, o = pair(emu, m, 3300)
    R = np.stack([gen.rhs(3400 + k, m) for k in range(8)])
    rhs = sparse_rhs(m, 3500, 8)
    for tr in "NT":
        l0 = launches(g)
        assert_dense(g, o, R, tr)
        assert launches(g) - l0 == 1 + 3
        l0 = launches(g)
        assert_sparse(g, o, rhs, tr)
        assert launches(g) - l0 == 1 + 3
        assert_counters(g, o)


def test_emu_object_multi_pending_update(emu):
    """Both multi solves between solve_for_update ('N' and 'T') and update do not disturb the pending basis change."""
    m = 100
    g, o = pair(emu, m, 3600)
    R = np.stack([gen.rhs(3700 + k, m) for k in range(4)])
    rhs = sparse_rhs(m, 3800, 5)
    pcp, pri, pv = gen.basis(3900, m, 0, 3.0)
    for it in range(3):
        ci, cx = pri[pcp[it]:pcp[it + 1]], pv[pcp[it]:pcp[it + 1]]
        assert g.solve_for_update(len(ci), ci, cx, "N", 1) == o.solve_for_update(len(ci), ci, cx, "N", 1) == 0
        assert np.array_equal(g.lhs, o.lhs)
        j = int(np.argmax(np.abs(o.lhs)))
        xtbl = o.lhs[j]
        assert g.solve_for_update(1, np.array([j]), None, "T", 0) == o.solve_for_update(1, np.array([j]), None, "T", 0) == 0
        for tr in "NT":
            assert_dense(g, o, R, tr)
            assert_sparse(g, o, rhs, tr)
        assert g.update(xtbl) == o.update(xtbl) == 0
        assert_counters(g, o)
        for tr in "NT":
            assert np.array_equal(g.solve_dense(R[0], tr)[1], o.solve_dense(R[0], tr)[1])


def test_emu_object_multi_bad_unit_and_bad_begin(emu):
    """A rejected right-hand side is reported for itself only; an rhs_begin offset outside [0, tot] is refused with
    nothing launched and nothing written."""
    m = 90
    g, o = pair(emu, m, 4000)
    rhs = sparse_rhs(m, 4100, 4)
    rhs[2] = (np.array([3, m, 5]), np.array([1.0, 2.0, 3.0]))      # index m: rejected
    st, nz, il, xl, stat = sparse_multi(g, rhs, "N")
    assert st == INVALID_ARGUMENT and list(stat) == [0, 0, INVALID_ARGUMENT, 0] and nz[2] == -1
    for r in (0, 1, 3):
        idx, val = rhs[r]
        assert o.solve_sparse(len(idx), idx, val, "N") == 0
        n = o.nzlhs
        assert nz[r] == n and np.array_equal(il[r, :n], o.ilhs[:n]) and np.array_equal(xl[r, :n], o.lhs[o.ilhs[:n]]), r
    for bad in ([0, 3, 999, 12, 16], [0, -1, 4, 12, 16]):
        rhs = [gen.sparse_rhs(4200 + k, m, 4) for k in range(4)]
        l0 = launches(g)
        st, nz, il, xl, stat = sparse_multi(g, rhs, "N", begin=np.array(bad, np.int64), fill=-7.0)
        assert st == INVALID_ARGUMENT and launches(g) == l0
        assert (nz == 77).all() and (stat == 77).all() and (il == -7).all() and (xl == -7.0).all()
