"""Shared pieces of the batch multi-RHS solve tests: a factorized batch with one oracle per basis, and the
comparison of blu_batch_solve_sparse / blu_batch_solve_dense_multi with the oracle running the same solves on
that basis, in order."""
import ctypes

import numpy as np

from blu_b200 import BLUBatch, gen
from blu_b200.blu import i32p
from parity import oracle_for

# per-basis getters the solves move; update_cost = update_cost_numer / update_cost_denom
COUNTERS = ["l_flops", "u_flops", "r_flops", "update_cost"]


def dup_first_column(cp, ri, v):
    """the basis with column 1 replaced by a copy of column 0: WarningSingularMatrix"""
    cols = [(ri[cp[j]:cp[j + 1]], v[cp[j]:cp[j + 1]]) for j in range(len(cp) - 1)]
    cols[1] = cols[0]
    cp2 = np.concatenate([[0], np.cumsum([len(r) for r, _ in cols])]).astype(np.int64)
    return cp2, np.concatenate([r for r, _ in cols]).astype(np.int64), np.concatenate([x for _, x in cols])


def make_batch(lib, nmat, m, seed0, nslack=None, mem=None, singular=(), factorize=True, pmean=4.0, sample=None):
    """nmat synthetic bases (gen.basis(seed0 + k, ...)) factorized on the batch and on one oracle each (sample:
    only on those bases, the other entries of the oracle list are None)"""
    nslack = m // 3 if nslack is None else nslack
    bases = [gen.basis(seed0 + k, m, nslack, pmean) for k in range(nmat)]
    bases = [dup_first_column(*bs) if k in singular else bs for k, bs in enumerate(bases)]
    b = BLUBatch(nmat, m, max(len(bs[1]) for bs in bases), lib=lib)
    if mem:
        b.l_mem = mem; b.u_mem = mem; b.w_mem = mem
    oracles = [oracle_for(m, len(bs[1]), 400) if sample is None or k in sample else None for k, bs in enumerate(bases)]
    if factorize:
        off = np.cumsum([0] + [len(bs[1]) for bs in bases])
        bb = np.concatenate([bs[0][:-1] + off[k] for k, bs in enumerate(bases)])
        be = np.concatenate([bs[0][1:] + off[k] for k, bs in enumerate(bases)])
        st, status = b.factorize(bb, be, np.concatenate([bs[1] for bs in bases]), np.concatenate([bs[2] for bs in bases]))
        for k, (o, (cp, ri, v)) in enumerate(zip(oracles, bases)):
            if o is not None:
                assert o.factorize(cp[:-1], cp[1:], ri, v) == status[k], k
    return b, oracles


def rhs_lists(m, seed, counts, sizes=(0, 1, 2, 5, 17, 40)):
    """counts[k] right-hand sides for basis k, their entry counts cycling through sizes"""
    out, n = [], 0
    for c in counts:
        lst = []
        for _ in range(c):
            nz = min(sizes[n % len(sizes)], m)
            lst.append(gen.sparse_rhs(seed + n, m, nz) if nz else (np.zeros(0, np.int64), np.zeros(0)))
            n += 1
        out.append(lst)
    return out


def assert_sparse_parity(b, oracles, lists, trans, sample=None, result=None):
    """blu_batch_solve_sparse against the oracles: status, nzlhs, the order of ilhs, values with np.array_equal and
    the counters afterwards.  sample: only these bases are compared (their oracles run every solve).  Returns the
    batch's result."""
    m = b.m
    st, out, ustat = result if result is not None else b.solve_sparse(lists, trans)
    first = next((int(s) for us in ustat for s in us if s != 0), 0)
    assert st == first, (st, first)
    for k in (range(len(oracles)) if sample is None else sample):
        o = oracles[k]
        assert len(out[k]) == len(lists[k]) == len(ustat[k])
        for u, (idx, val) in enumerate(lists[k]):
            ost = o.solve_sparse(len(idx), idx, val, trans)
            assert ustat[k][u] == ost, (k, u, ustat[k][u], ost)
            il, xl = out[k][u]
            if ost == 0:
                n = o.nzlhs
                ilo = o.ilhs[:n]
                assert len(il) == n and np.array_equal(il, ilo), (k, u, "pattern order")
                assert np.array_equal(xl, o.lhs[ilo]), (k, u, "values")
            else:
                assert len(il) == 0
        for name in COUNTERS:
            assert b.info(k, name) == o.info(name), (k, name, b.info(k, name), o.info(name))
        assert b.info(k, "internal_error") == 0
    return st, out, ustat


def assert_dense_parity(b, oracles, nrhs, seed, trans):
    m, nmat = b.m, b.nmat
    R = np.random.default_rng(seed).uniform(-1.0, 1.0, (nmat, nrhs, m))
    st, X, S = b.solve_dense_multi(R, trans)
    assert X.shape == (nmat, nrhs, m) and S.shape == (nmat, nrhs)
    first = 0
    for k, o in enumerate(oracles):
        for r in range(nrhs):
            ost, xo = o.solve_dense(R[k, r], trans)
            assert S[k, r] == ost, (k, r)
            first = first or ost
            if ost == 0:
                assert np.array_equal(X[k, r], xo), (k, r, trans)
    assert st == first
    return st, X, S


def update_round(b, oracles, seed, it):
    """one basis change on every basis (batch solve_for_update 'N' + 'T' and update) in lockstep with the
    oracles; the entering column of basis k is column `it` of gen.basis(seed + k, m, 0, 3.0)"""
    m = b.m
    cols = []
    for k in range(len(oracles)):
        cp, ri, v = gen.basis(seed + k, m, 0, 3.0)
        cols.append((ri[cp[it]:cp[it + 1]], v[cp[it]:cp[it + 1]]))
    st, stat, out = b.solve_for_update(cols, "N", want_solution=1)
    assert st == 0, (st, stat)
    leave, xt = [], []
    for k, o in enumerate(oracles):
        assert o.solve_for_update(len(cols[k][0]), cols[k][0], cols[k][1], "N", want_solution=1) == 0
        j = int(np.argmax(np.abs(o.lhs)))
        leave.append((np.array([j]), None)); xt.append(o.lhs[j])
    st, stat, _ = b.solve_for_update(leave, "T", want_solution=0)
    assert st == 0
    for k, o in enumerate(oracles):
        assert o.solve_for_update(1, leave[k][0], None, "T", want_solution=0) == 0
    return xt


def finish_update(b, oracles, xt):
    st, stat = b.update(np.array(xt))
    for k, o in enumerate(oracles):
        assert o.update(xt[k]) == stat[k], k
        for name in ("nupdate", "nforrest", "u_nz", "r_nz", "pivot_error", "max_eta") + tuple(COUNTERS):
            assert b.info(k, name) == o.info(name), (k, name)


def raw_solve_sparse(b, unit_begin, rhs_begin, irhs, xrhs, trans="N"):
    """blu_batch_solve_sparse with the arrays exactly as given (for malformed input)"""
    ub, rb = np.ascontiguousarray(unit_begin, np.int64), np.ascontiguousarray(rhs_begin, np.int64)
    ir, xr = np.ascontiguousarray(irhs, np.int64), np.ascontiguousarray(xrhs, np.float64)
    n = max(int(ub[-1]), 1)
    nz = np.zeros(n, np.int64); il = np.zeros(n * b.m, np.int64); xl = np.zeros(n * b.m); stat = np.zeros(n, np.int32)
    p = lambda a, t: a.ctypes.data_as(ctypes.POINTER(t))
    return b._L.blu_batch_solve_sparse(b._h, p(ub, ctypes.c_int64), p(rb, ctypes.c_int64), p(ir, ctypes.c_int64),
                                       p(xr, ctypes.c_double), p(nz, ctypes.c_int64), p(il, ctypes.c_int64),
                                       p(xl, ctypes.c_double), stat.ctypes.data_as(i32p), trans.encode())
