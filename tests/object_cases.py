"""Shared pieces of the tests of blu_clone / blu_save / blu_restore: BLU objects seen as the slots of a batch, so that
the lane machinery of subset_cases and copy_cases (one logged oracle per basis, replay, snapshot) drives objects, and
everything observable of one object (getters, parameters, its image) in one comparable record."""
import numpy as np

from blu_b200.blu import I as INFO, P as PARAMS

# every getter of an object but the accumulated wall-clock times, which two objects running the same calls do not share
LOCKSTEP = [n for n in INFO if not n.startswith("time_")]


def first_error(stat):
    return next((int(s) for s in stat if s != 0), 0)


class Objects:
    """slot k of this "batch" is the list of objects slots[k]: every call runs on each of them, their results must be
    bit-identical (statuses, nzlhs, ilhs order, values, dense solutions, get_factors) and so must every getter but the
    times after each call; the first object's results are returned, as the batch calls return them"""

    def __init__(self, slots):
        self.slots = [list(s) for s in slots]
        self.m = self.slots[0][0].m

    @property
    def nmat(self):
        return len(self.slots)

    def _each(self, k, fn):
        res = [fn(o) for o in self.slots[k]]
        for r in res[1:]:
            assert_same_result(res[0], r)
        for o in self.slots[k][1:]:
            for n in LOCKSTEP:
                x, y = self.slots[k][0].info(n), o.info(n)
                assert x == y or (x != x and y != y), (k, n, x, y)
        return res[0]

    def info(self, k, name):
        return self.slots[k][0].info(name)

    def factorize_subset(self, sel, bb, be, bi, bx):
        m = self.m
        stat = np.array([self._each(k, lambda o: o.factorize(bb[r * m:(r + 1) * m], be[r * m:(r + 1) * m], bi, bx))
                         for r, k in enumerate(sel)], np.int32)
        return first_error(stat), stat

    def solve_for_update_subset(self, sel, rhs_list, trans="N", want_solution=0):
        def one(o, ir, xr):
            st = o.solve_for_update(len(ir), ir, xr, trans, want_solution)
            n = o.nzlhs if want_solution and st == 0 else 0
            return st, (o.ilhs[:n].copy(), o.lhs[o.ilhs[:n]].copy())
        res = [self._each(k, lambda o: one(o, ir, xr)) for k, (ir, xr) in zip(sel, rhs_list)]
        stat = np.array([r[0] for r in res], np.int32)
        return first_error(stat), stat, [r[1] for r in res]

    def update_subset(self, sel, xtbl):
        stat = np.array([self._each(k, lambda o: o.update(x)) for k, x in zip(sel, xtbl)], np.int32)
        return first_error(stat), stat

    def solve_dense(self, rhs, trans="N"):
        m, r = self.m, np.asarray(rhs, np.float64).reshape(self.nmat, self.m)
        res = [self._each(k, lambda o: o.solve_dense(r[k], trans)) for k in range(self.nmat)]
        stat = np.array([s for s, _ in res], np.int32)
        return first_error(stat), np.stack([x for _, x in res]).reshape(self.nmat, m), stat

    def solve_dense_multi(self, rhs, trans="N"):
        r = np.asarray(rhs, np.float64).reshape(self.nmat, -1, self.m)
        res = [self._each(k, lambda o: o.solve_dense_multi(r[k], trans)) for k in range(self.nmat)]
        stat = np.array([[s] * r.shape[1] for s, _ in res], np.int32)
        return first_error(stat.reshape(-1)), np.stack([x for _, x in res]), stat

    def solve_sparse(self, rhs_lists, trans="N"):
        out, ustat = [], []
        for k, lst in enumerate(rhs_lists):
            res = []
            for ir, xr in lst:
                def one(o):
                    st = o.solve_sparse(len(ir), ir, xr, trans)
                    n = o.nzlhs if st == 0 else 0
                    return st, (o.ilhs[:n].copy(), o.lhs[o.ilhs[:n]].copy())
                res.append(self._each(k, one))
            out.append([r[1] for r in res])
            ustat.append(np.array([r[0] for r in res], np.int32))
        return first_error(np.concatenate(ustat) if ustat else []), out, ustat

    def get_factors(self, k):
        return self._each(k, lambda o: o.get_factors())


def assert_same_result(a, b):
    """two results of the same call: tuples, arrays and dicts of arrays compared bit for bit"""
    if isinstance(a, tuple):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert_same_result(x, y)
    elif isinstance(a, dict):
        assert a.keys() == b.keys()
        for q in a:
            assert_same_result(a[q], b[q])
    elif isinstance(a, np.ndarray):
        assert a.shape == b.shape and np.array_equal(a, b, equal_nan=True)
    else:
        assert a == b or (a != a and b != b), (a, b)


def record(o):
    """everything an object shows without changing: every getter (times and nrealloc included), every parameter, and
    its image"""
    return dict(info={n: o.info(n) for n in INFO}, params={n: o.get_param(n) for n in PARAMS}, image=o.save())


def assert_same_record(a, b, times=True):
    for n in a["info"]:
        if times or not n.startswith("time_"):
            x, y = a["info"][n], b["info"][n]
            assert x == y or (x != x and y != y), (n, x, y)
    assert a["params"] == b["params"]
    assert np.array_equal(a["image"], b["image"])
