"""Shared pieces of the batch maxvolume tests: a pool of columns per basis, the batch layout of
blu_batch_maxvolume, and the comparison of every basis with its own oracle running maxvolume alone."""
import numpy as np

from blu_b200 import gen
from oracle_lib import Oracle

# the getters of the LU state maxvolume leaves behind, compared with ==
GETTERS = ["nupdate", "nforrest", "nfactorize", "nupdate_total", "nforrest_total", "nsymperm_total", "pivot_error"]


class Pool:
    """One basis' pool in CSC: its m starting columns first (basis = 0..m-1, all basic), then ncand candidates."""

    def __init__(self, a_p, a_i, a_x, m):
        self.a_p, self.a_i, self.a_x = np.asarray(a_p, np.int64), np.asarray(a_i, np.int64), np.asarray(a_x, np.float64)
        self.m = m
        self.ncol = len(self.a_p) - 1
        self.basis = np.arange(m, dtype=np.int64)
        self.isbasic = np.zeros(self.ncol, dtype=np.int64)
        self.isbasic[:m] = 1


def make_pool(seed, m, ncand, nslack=None, pmean=4.0, scale=1.0, nnz_col=6, identity=False):
    if identity:
        cp, ri, v = np.arange(m + 1, dtype=np.int64), np.arange(m, dtype=np.int64), np.ones(m)
    else:
        cp, ri, v = gen.basis(seed, m, m // 3 if nslack is None else nslack, pmean)
    qp, qi, qx = gen.column_pool(seed + 7919, m, ncand, nnz_col)
    return Pool(np.concatenate([cp, cp[-1] + qp[1:]]), np.concatenate([ri, qi]), np.concatenate([v, scale * qx]), m)


def config1_pools(nmat, ncand, seed0, scale=3.0):
    """configs[1]'s bases (gen.batch(nmat, 2000, 700, 5.0, seed0, ...): basis k is gen.basis(seed0 + k, ...)), each
    followed by ncand fresh candidate columns of 8 entries scaled by `scale`, so that columns do enter"""
    m = 2000
    pools = []
    for k in range(nmat):
        cp, ri, v = gen.basis(seed0 + k, m, 700, 5.0)
        qp, qi, qx = gen.column_pool(seed0 + 50000 + k, m, ncand, 8)
        pools.append(Pool(np.concatenate([cp, cp[-1] + qp[1:]]), np.concatenate([ri, qi]), np.concatenate([v, scale * qx]), m))
    return pools


def replace_column(p, j, rows, vals):
    """a copy of pool p whose column j holds (rows, vals)"""
    cols = [(p.a_i[p.a_p[c]:p.a_p[c + 1]], p.a_x[p.a_p[c]:p.a_p[c + 1]]) for c in range(p.ncol)]
    cols[j] = (np.asarray(rows, np.int64), np.asarray(vals, np.float64))
    a_p = np.concatenate([[0], np.cumsum([len(r) for r, _ in cols])])
    q = Pool(a_p, np.concatenate([r for r, _ in cols]), np.concatenate([x for _, x in cols]), p.m)
    q.basis, q.isbasic = p.basis.copy(), p.isbasic.copy()
    return q


def layout(pools):
    """blu_batch_maxvolume's arguments for a list of pools of one ncol: a_begin, a_end, a_i, a_x, basis, isbasic"""
    ncol = pools[0].ncol
    assert all(p.ncol == ncol for p in pools)
    ab, ae, off = [], [], 0
    for p in pools:
        ab.append(p.a_p[:-1] + off); ae.append(p.a_p[1:] + off)
        off += len(p.a_i)
    return (np.concatenate(ab), np.concatenate(ae), np.concatenate([p.a_i for p in pools]),
            np.concatenate([p.a_x for p in pools]), np.concatenate([p.basis for p in pools]),
            np.concatenate([p.isbasic for p in pools]))


def oracle_maxvolume(p, volumetol):
    """maxvolume of one basis alone on the CPU oracle (stores large enough never to reallocate, so that
    factor_flops and with it update_cost count every pivot step once)."""
    o = Oracle(p.m, 60 * len(p.a_i) + 100 * p.m)
    basis, isbasic = p.basis.copy(), p.isbasic.copy()
    st, nup = o.maxvolume(p.ncol, p.a_p, p.a_i, p.a_x, basis, isbasic, volumetol)
    return o, st, nup, basis, isbasic


def run_batch(b, pools, volumetol):
    ab, ae, ai, ax, basis, isbasic = layout(pools)
    st, status, nup = b.maxvolume(pools[0].ncol, ab, ae, ai, ax, basis, isbasic, volumetol)
    m, ncol = pools[0].m, pools[0].ncol
    return st, status, nup, basis.reshape(len(pools), m), isbasic.reshape(len(pools), ncol)


def assert_parity(b, pools, volumetol, result, rhs_seed=0, oracles=None):
    """Every basis against its own oracle: status, nupdate, basis, isbasic, the getters, and solve_dense
    'N' / 'T' on the bases that ended OK.  Returns the oracle results."""
    st, status, nup, basis, isbasic = result
    ores = oracles or [oracle_maxvolume(p, volumetol) for p in pools]
    first = next((int(s) for s in status if s != 0), 0)
    assert st == first, (st, status)
    m = pools[0].m
    rhs = np.concatenate([gen.rhs(rhs_seed + k, m) for k in range(len(pools))])
    xs = {tr: b.solve_dense(rhs, tr) for tr in "NT"}
    for k, (o, ost, onup, obasis, oisbasic) in enumerate(ores):
        assert status[k] == ost, (k, status[k], ost)
        assert nup[k] == onup, (k, nup[k], onup)
        assert np.array_equal(basis[k], obasis), k
        assert np.array_equal(isbasic[k], oisbasic), k
        for name in GETTERS:
            assert b.info(k, name) == o.info(name), (k, name, b.info(k, name), o.info(name))
        assert b.info(k, "internal_error") == 0, k
        if ost == 0:
            for tr in "NT":
                _, xo = o.solve_dense(rhs[k * m:(k + 1) * m], tr)
                assert np.array_equal(xs[tr][1][k], xo), (k, tr)
    return ores


def refactor_triggers(p, volumetol):
    """maxvolume's loop restated on the oracle's calls (as blu_b200/maxvolume.py does it), recording which of the
    conditions of maxvolume.rs:161-170 held at each refactorization.  Returns (status, nupdate, basis, isbasic,
    triggers): triggers lists one set per refactorization out of {"nforrest", "pivot_error", "update_cost"}."""
    o = Oracle(p.m, 60 * len(p.a_i) + 100 * p.m)
    basis, isbasic = p.basis.copy(), p.isbasic.copy()
    a_p, a_i, a_x, m = p.a_p, p.a_i, p.a_x, p.m
    triggers, nupdate = [], 0

    def factorize():
        return o.factorize(a_p[basis], a_p[basis + 1], a_i, a_x)

    st = factorize()
    for j in range(p.ncol):
        if st != 0:
            break
        if isbasic[j]:
            continue
        b, e = a_p[j], a_p[j + 1]
        st = o.solve_for_update(e - b, a_i[b:e], a_x[b:e], "N", 1)
        if st != 0:
            break
        lhs = o.lhs
        xmax, xtbl, imax = 0.0, 0.0, 0
        for i in o.ilhs[:o.nzlhs]:
            if abs(lhs[i]) > xmax:
                xtbl, xmax, imax = lhs[i], abs(lhs[i]), int(i)
        if xmax <= volumetol:
            continue
        isbasic[basis[imax]] = 0
        isbasic[j] = 1
        basis[imax] = j
        nupdate += 1
        st = o.solve_for_update(0, np.array([imax], np.int64), None, "T", 0)
        if st == 0:
            st = o.update(xtbl)
        if st != 0:
            break
        why = {n for n, hit in (("nforrest", o.info("nforrest") == m), ("pivot_error", o.info("pivot_error") > 1e-8),
                                ("update_cost", o.info("update_cost") > 1.0)) if hit}
        if why:
            triggers.append(why)
            st = factorize()
    return st, nupdate, basis, isbasic, triggers
