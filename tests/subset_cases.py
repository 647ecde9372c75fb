"""Shared pieces of the tests of the batch calls on a subset of the bases (blu_batch_factorize_subset,
blu_batch_solve_for_update_subset, blu_batch_update_subset): one oracle object per basis, each basis on its own
schedule, and the comparison of every basis with its oracle after every call."""
import ctypes

import numpy as np

from blu_b200 import gen
from blu_b200.blu import I as INFO, i32p
from bs_cases import COUNTERS
from parity import SPARSE_STATS, STATS, oracle_for

# the per-basis getters compared with the oracle after every call
GETTERS = sorted(set(STATS + SPARSE_STATS + COUNTERS + ["nfactorize"]))
# every per-basis selector of a batch (not the object-level time_* and nrealloc)
PER_BASIS = [n for n in INFO if not n.startswith("time_") and n != "nrealloc"]


class Lane:
    """One basis: its current B (a list of m columns), the oracle that runs exactly the calls the basis is selected
    in, and a pool of entering columns."""

    def __init__(self, seed, m, nslack=None, pmean=4.0, policy=0):
        cp, ri, v = gen.basis(seed, m, m // 3 if nslack is None else nslack, pmean)
        self.m = m
        self.cols = [(ri[cp[j]:cp[j + 1]].copy(), v[cp[j]:cp[j + 1]].copy()) for j in range(m)]
        self.pool = gen.basis(seed + 50000, m, 0, 3.0)
        self.npool = 0
        self.oracle = oracle_for(m, len(v) + 8 * m, 400 if m <= 200 else 20)
        self.factored = None         # the B the basis was last factorized from
        self.rejected = False        # B was rejected (InvalidArgument): matrix_nz and the like are not compared
        self.pending = None          # (leaving position, xtbl, entering column) between 'N' + 'T' and the update
        self.refactor = False        # the basis must refactorize before its next basis change
        # when the basis refactorizes: 0 after update_cost > 1 or nforrest == m, 1 after nforrest == m, 2 and 3 only
        # after MaximumUpdates / SingularUpdate; 3 sometimes leaves a position where x is zero (SingularUpdate)
        self.policy = policy

    def next_column(self):
        cp, ri, v = self.pool
        j = self.npool % self.m
        self.npool += 1
        return ri[cp[j]:cp[j + 1]].copy(), v[cp[j]:cp[j + 1]].copy()


def layout(bases):
    """blu_batch_factorize_subset's b_begin, b_end, b_i, b_x for a list of column lists.  The bases are stored in
    reverse order with a gap in front of each, so that B is read through its pointers and not by position."""
    m = len(bases[0])
    bb = np.zeros(len(bases) * m, np.int64)
    be = np.zeros(len(bases) * m, np.int64)
    bi, bx, off = [], [], 0
    for r in reversed(range(len(bases))):
        bi.append(np.full(3, -7, np.int64)); bx.append(np.full(3, np.nan)); off += 3
        for j, (ri, v) in enumerate(bases[r]):
            bb[r * m + j] = off; be[r * m + j] = off + len(ri)
            bi.append(np.asarray(ri, np.int64)); bx.append(np.asarray(v, np.float64)); off += len(ri)
    return bb, be, np.concatenate(bi), np.concatenate(bx)


def csc(cols):
    cp = np.concatenate([[0], np.cumsum([len(r) for r, _ in cols])]).astype(np.int64)
    return cp, np.concatenate([r for r, _ in cols]).astype(np.int64), np.concatenate([x for _, x in cols])


def assert_getters(b, lanes, ks=None):
    for k in (range(len(lanes)) if ks is None else ks):
        if lanes[k].rejected:
            continue
        o = lanes[k].oracle
        for name in GETTERS:
            assert b.info(k, name) == o.info(name), (k, name, b.info(k, name), o.info(name))
        assert b.info(k, "internal_error") == 0, k


def factorize(b, lanes, sel):
    """factorize_subset of the bases sel from their current B, the oracles alongside"""
    st, stat = b.factorize_subset(sel, *layout([lanes[k].cols for k in sel]))
    for r, k in enumerate(sel):
        cp, ri, v = csc(lanes[k].cols)
        ost = lanes[k].oracle.factorize(cp[:-1], cp[1:], ri, v)
        assert stat[r] == ost, (k, stat[r], ost)
        lanes[k].factored = list(lanes[k].cols)
        lanes[k].refactor = False
        lanes[k].pending = None
    assert st == next((int(s) for s in stat if s != 0), 0), (st, stat)
    assert_getters(b, lanes)
    return st, stat


def solve_n(b, lanes, sel, stats=None, rng=None):
    """solve_for_update 'N' with the next pool column on the bases sel; returns {k: (leaving position, xtbl, column)}
    for those whose solve succeeded.  The leaving position is argmax |x|; with rng, a basis of policy 3 leaves a
    position where x is zero one time in four."""
    cols = {k: lanes[k].next_column() for k in sel}
    st, stat, out = b.solve_for_update_subset(sel, [cols[k] for k in sel], "N", want_solution=1)
    res = {}
    for r, k in enumerate(sel):
        o = lanes[k].oracle
        ost = o.solve_for_update(len(cols[k][0]), cols[k][0], cols[k][1], "N", want_solution=1)
        assert stat[r] == ost, (k, stat[r], ost)
        if ost != 0:
            assert len(out[r][0]) == 0
            lanes[k].refactor = True
            if stats is not None:
                stats[str(ost)] = stats.get(str(ost), 0) + 1
            continue
        n = o.nzlhs
        assert np.array_equal(out[r][0], o.ilhs[:n]), (k, "ilhs order")
        assert np.array_equal(out[r][1], o.lhs[o.ilhs[:n]]), (k, "values")
        lhs = o.lhs
        j = int(np.argmax(np.abs(lhs)))
        if rng is not None and lanes[k].policy == 3 and rng.uniform() < 0.25 and (lhs == 0).any():
            j = int(np.flatnonzero(lhs == 0)[0])
        res[k] = (j, lhs[j], cols[k])
    assert st == next((int(s) for s in stat if s != 0), 0)
    assert_getters(b, lanes)
    return res


def solve_t(b, lanes, pend, want):
    """solve_for_update 'T' on the bases of pend ({k: (j, xtbl, column)}); the ones that succeed become pending"""
    sel = sorted(pend)
    st, stat, out = b.solve_for_update_subset(sel, [(np.array([pend[k][0]]), None) for k in sel], "T", want_solution=want)
    for r, k in enumerate(sel):
        o = lanes[k].oracle
        ost = o.solve_for_update(1, np.array([pend[k][0]]), None, "T", want_solution=want)
        assert stat[r] == ost, (k, stat[r], ost)
        if ost != 0:
            lanes[k].refactor = True
            continue
        if want:
            n = o.nzlhs
            assert np.array_equal(out[r][0], o.ilhs[:n]) and np.array_equal(out[r][1], o.lhs[o.ilhs[:n]]), k
        lanes[k].pending = pend[k]
    assert_getters(b, lanes)
    return st


def update(b, lanes, sel, stats=None):
    """update on the pending bases sel; B takes the entering column where the update succeeds.  stats counts what
    makes a basis refactorize."""
    st, stat = b.update_subset(sel, [lanes[k].pending[1] for k in sel])
    for r, k in enumerate(sel):
        L = lanes[k]
        o = L.oracle
        j, xtbl, col = L.pending
        ost = o.update(xtbl)
        assert stat[r] == ost, (k, stat[r], ost)
        L.pending = None
        if ost == 0:
            L.cols[j] = col
        why = str(ost) if ost != 0 else "nforrest" if L.policy < 2 and o.info("nforrest") == L.m else \
            "update_cost" if L.policy == 0 and o.info("update_cost") > 1.0 else None
        if why:
            L.refactor = True
            if stats is not None:
                stats[why] = stats.get(why, 0) + 1
    assert st == next((int(s) for s in stat if s != 0), 0)
    assert_getters(b, lanes)
    return stat


def assert_dense(b, lanes, seed):
    """solve_dense 'N' / 'T' on the whole batch against every oracle"""
    m = lanes[0].m
    rhs = np.random.default_rng(seed).uniform(-1.0, 1.0, len(lanes) * m)
    for tr in "NT":
        _, x, stat = b.solve_dense(rhs, tr)
        for k, L in enumerate(lanes):
            ost, xo = L.oracle.solve_dense(rhs[k * m:(k + 1) * m], tr)
            assert stat[k] == ost, (k, tr, stat[k], ost)
            if ost == 0 and not L.refactor:
                assert np.array_equal(x[k], xo), (k, tr)


def replay(b, lanes, rounds, seed, dense_every=4, stats=None):
    """Every basis on its own schedule.  Each round each basis draws: stay idle, a full basis change ('N' with the
    solution, 'T', update), 'N' + 'T' now with the update in a later round, or a refactorization from its current B
    -- forced by the basis' policy (Lane.policy) after MaximumUpdates / SingularUpdate, update_cost > 1 or
    nforrest == m.  The calls of a round go out as one subset call each; every basis is compared with its oracle
    after every call.  stats (a dict) counts the refactorization triggers and the calls inside which a store grew."""
    rng = np.random.default_rng(seed)
    stats = {} if stats is None else stats
    for k in ("realloc_factorize", "realloc_solve", "realloc_update"):
        stats.setdefault(k, 0)
    for it in range(rounds):
        fact, full, half, upd = [], [], [], []
        for k, L in enumerate(lanes):
            a = rng.integers(0, 32)
            if L.refactor or a == 0:
                fact.append(k)
            elif L.pending is not None:
                if a < 16:
                    upd.append(k)
            elif 4 <= a < 24:
                full.append(k)
            elif a >= 24:
                half.append(k)
        rng.shuffle(fact)
        nr = b.info(0, "nrealloc")
        if fact:
            factorize(b, lanes, [int(k) for k in fact])
        stats["realloc_factorize"] += b.info(0, "nrealloc") > nr
        nr = b.info(0, "nrealloc")
        pend = solve_n(b, lanes, full + half, stats, rng) if full + half else {}
        if pend:
            solve_t(b, lanes, pend, want=it % 2)
        stats["realloc_solve"] += b.info(0, "nrealloc") > nr
        upd += [k for k in full if lanes[k].pending is not None]
        if upd:
            nr = b.info(0, "nrealloc")
            update(b, lanes, upd, stats)
            stats["realloc_update"] += b.info(0, "nrealloc") > nr
        if dense_every and it % dense_every == dense_every - 1:
            assert_dense(b, lanes, seed + it)
    return stats


def snapshot(b, ks, seed=1, lanes=None):
    """everything observable of the bases ks: every per-basis getter, get_factors where nupdate == 0, solve_dense.
    The dense solves run on every basis first (they compact the pivot sequence, as the reference's do, so that a
    second snapshot sees the same pivotlen): lanes, when given, have their oracles run them too."""
    m = b.m
    rhs = np.random.default_rng(seed).uniform(-1.0, 1.0, (b.nmat, 1, m))
    xs = {}
    for tr in "NT":
        _, x, stat = b.solve_dense_multi(rhs, tr)
        xs[tr] = (None, x[:, 0], stat[:, 0])
    for k, L in enumerate(lanes or []):
        for tr in "NT":
            L.oracle.solve_dense(rhs[k, 0], tr)
    snap = {}
    for k in ks:
        s = {n: b.info(k, n) for n in PER_BASIS}
        if s["nupdate"] == 0:
            st, f = b.get_factors(k)
            s["factors"] = (st, f)
        for tr in "NT":
            s["dense" + tr] = (xs[tr][2][k], xs[tr][1][k].copy())
        snap[k] = s
    return snap


def assert_same_snapshot(a, c):
    assert a.keys() == c.keys()
    for k in a:
        for n in a[k]:
            x, y = a[k][n], c[k][n]
            if n == "factors":
                assert x[0] == y[0] and all(np.array_equal(x[1][q], y[1][q]) for q in x[1]), (k, n)
            elif n.startswith("dense"):
                assert x[0] == y[0] and np.array_equal(x[1], y[1], equal_nan=True), (k, n)
            else:
                assert np.array_equal(x, y, equal_nan=True), (k, n, x, y)


def _pi(a):
    return None if a is None else np.ascontiguousarray(a, np.int64).ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def _pf(a):
    return None if a is None else np.ascontiguousarray(a, np.float64).ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def raw_factorize_subset(b, nsel, sel, bb, be, bi, bx, bnz_total):
    """blu_batch_factorize_subset with the arguments exactly as given (None = NULL)"""
    arrs = [None if a is None else np.ascontiguousarray(a, t) for a, t in
            ((sel, np.int64), (bb, np.int64), (be, np.int64), (bi, np.int64), (bx, np.float64))]
    stat = np.zeros(max(nsel, 1), np.int32)
    return b._L.blu_batch_factorize_subset(b._h, nsel, _pi(arrs[0]), _pi(arrs[1]), _pi(arrs[2]), _pi(arrs[3]), _pf(arrs[4]),
                                           bnz_total, stat.ctypes.data_as(i32p))


def raw_solve_subset(b, nsel, sel, rhs_begin, irhs, xrhs, want=1, trans="N"):
    """blu_batch_solve_for_update_subset with the arguments exactly as given (None = NULL)"""
    arrs = [None if a is None else np.ascontiguousarray(a, t) for a, t in
            ((sel, np.int64), (rhs_begin, np.int64), (irhs, np.int64), (xrhs, np.float64))]
    n = max(nsel, 1)
    nz, il, xl, stat = np.zeros(n, np.int64), np.zeros(n * b.m, np.int64), np.zeros(n * b.m), np.zeros(n, np.int32)
    return b._L.blu_batch_solve_for_update_subset(b._h, nsel, _pi(arrs[0]), _pi(arrs[1]), _pi(arrs[2]), _pf(arrs[3]), want,
                                                  _pi(nz) if want else None, _pi(il) if want else None, _pf(xl) if want else None,
                                                  stat.ctypes.data_as(i32p), trans.encode())


def raw_update_subset(b, nsel, sel, xtbl):
    """blu_batch_update_subset with the arguments exactly as given (None = NULL)"""
    s = None if sel is None else np.ascontiguousarray(sel, np.int64)
    x = None if xtbl is None else np.ascontiguousarray(xtbl, np.float64)
    stat = np.zeros(max(nsel, 1), np.int32)
    return b._L.blu_batch_update_subset(b._h, nsel, _pi(s), _pf(x), stat.ctypes.data_as(i32p))
