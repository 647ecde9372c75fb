"""Shared pieces of the tests of the batch calls on device buffers (blu_batch_*_dev): twin batches with identical
history, one driven through the host calls and one through the _dev calls with torch tensors, compared bit for bit
after every call.  Twin has the interface the helpers of subset_cases and bs_cases drive, so the same schedules also
compare every basis with its oracle."""
import numpy as np
import torch

from blu_b200 import BLUBatch
from blu_b200.blu import I as INFO

# out-tensor fill for the entries of bases and units that do not run: they must come back as they went in
SENT_I, SENT_X = -77, 7.25
# every per-basis getter but the wall-clock times and the cycle counters (diagnostics that differ run to run on a GPU;
# n_kind7 counts the cycles of the dense tail's pivot search)
TWIN_GETTERS = [n for n in INFO if not n.startswith(("time_", "t_phase", "norms_cyc")) and n != "n_kind7"]


def first_bad(stats):
    return next((int(s) for s in stats if s != 0), 0)


class Twin:
    """Two batches made alike by make(); every call runs on both: `h` through the host calls, `d` through the _dev
    calls with tensors on `dev`.  Outputs, statuses, return values and every getter are asserted equal after each
    call; the host variant's results are returned."""

    def __init__(self, make, dev):
        self.h, self.d = make(), make()
        self.dev = dev
        self.nmat, self.m = self.h.nmat, self.h.m

    def T(self, a, dtype):
        return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(self.dev)

    def mask(self, sel):
        run = np.zeros(self.nmat, np.int32)
        run[list(sel)] = 1
        return self.T(run, torch.int32)

    def sentinels(self, n, wide):
        s = torch.full((n,), SENT_I, dtype=torch.int32, device=self.dev)
        if not wide:
            return s
        return (s, torch.full((n,), SENT_I, dtype=torch.int64, device=self.dev),
                torch.full((n * self.m,), SENT_I, dtype=torch.int64, device=self.dev),
                torch.full((n * self.m,), SENT_X, dtype=torch.float64, device=self.dev))

    def assert_state(self):
        for k in range(self.nmat):
            for name in TWIN_GETTERS:
                a, b = self.h.info(k, name), self.d.info(k, name)
                assert a == b or (a != a and b != b), (k, name, a, b)
        assert self.h.info(0, "nrealloc") == self.d.info(0, "nrealloc")

    def assert_untouched(self, outs, run):
        """entries of the masked-out bases of the out tensors still hold the sentinels"""
        off = np.flatnonzero(np.asarray(run) == 0)
        for t in outs:
            if t is None:
                continue
            a = t.cpu().numpy().reshape(self.nmat, -1)[off]
            assert (a == (SENT_X if t.dtype == torch.float64 else SENT_I)).all()

    # ---- the subset interface (subset_cases) ----
    def factorize_subset(self, sel, bb, be, bi, bx):
        st, stat = self.h.factorize_subset(sel, bb, be, bi, bx)
        m = self.m
        pb, pe = np.zeros(self.nmat * m, np.int64), np.zeros(self.nmat * m, np.int64)
        for r, k in enumerate(sel):
            pb[k * m:(k + 1) * m] = bb[r * m:(r + 1) * m]
            pe[k * m:(k + 1) * m] = be[r * m:(r + 1) * m]
        run = np.zeros(self.nmat, np.int32); run[list(sel)] = 1
        sd = self.sentinels(self.nmat, False)
        std, sd = self.d.factorize_subset_dev(self.T(pb, torch.int64), self.T(pe, torch.int64), self.T(bi, torch.int64),
                                              self.T(bx, torch.float64), run=self.mask(sel), status=sd)
        sd = sd.cpu().numpy()
        assert [sd[k] for k in sel] == list(stat)
        assert std == first_bad(sd[k] for k in sorted(sel))
        self.assert_untouched([torch.as_tensor(sd)], run)
        self.assert_state()
        return st, stat

    def solve_for_update_subset(self, sel, rhs_list, trans="N", want_solution=0):
        st, stat, out = self.h.solve_for_update_subset(sel, rhs_list, trans, want_solution)
        n, m = self.nmat, self.m
        cols = {k: rhs_list[r] for r, k in enumerate(sel)}
        begin, irhs, xrhs = np.zeros(n + 1, np.int64), [], []
        for k in range(n):
            ii = np.asarray(cols[k][0], np.int64).reshape(-1) if k in cols else np.zeros(0, np.int64)
            begin[k + 1] = begin[k] + len(ii)
            irhs.append(ii)
            if k in cols and cols[k][1] is not None:
                xrhs.append(np.asarray(cols[k][1], np.float64))
            elif k not in cols:
                xrhs.append(np.zeros(0))
        have_x = len(sel) > 0 and rhs_list[0][1] is not None
        s, nz, il, xl = self.sentinels(n, True)
        r = self.solve_dev(begin, np.concatenate(irhs), np.concatenate(xrhs) if have_x else None, trans, want_solution,
                           self.mask(sel), s, nz, il, xl)
        self.check_solve(st, stat, out, sel, r, want_solution)
        run = np.zeros(n, np.int32); run[list(sel)] = 1
        self.assert_untouched([r[1]] + ([r[2], r[3], r[4]] if want_solution else []), run)
        self.assert_state()
        return st, stat, out

    def solve_dev(self, begin, irhs, xrhs, trans, want, run, s, nz, il, xl):
        return self.d.solve_for_update_dev(self.T(begin, torch.int64), self.T(irhs, torch.int64),
                                           None if xrhs is None else self.T(xrhs, torch.float64), trans, want, run=run,
                                           status=s, nzlhs=nz if want else None, ilhs=il if want else None,
                                           xlhs=xl if want else None)

    def check_solve(self, st, stat, out, sel, r, want):
        std, sd, nzd, ild, xld = r
        sd = sd.cpu().numpy()
        assert [int(sd[k]) for k in sel] == [int(x) for x in stat], (list(stat), sd)
        assert std == first_bad(sd[k] for k in sorted(sel))
        if want:
            nzd, ild, xld = nzd.cpu().numpy(), ild.cpu().numpy().reshape(self.nmat, -1), xld.cpu().numpy().reshape(self.nmat, -1)
            for q, k in enumerate(sel):
                n = int(nzd[k])
                assert n == (len(out[q][0]) if stat[q] == 0 else -1), (k, n)
                assert np.array_equal(ild[k, :max(n, 0)], out[q][0]) and np.array_equal(xld[k, :max(n, 0)], out[q][1]), k

    def update_subset(self, sel, xtbl):
        st, stat = self.h.update_subset(sel, xtbl)
        x = np.full(self.nmat, np.nan)
        for r, k in enumerate(sel):
            x[k] = xtbl[r]
        s = self.sentinels(self.nmat, False)
        std, sd = self.d.update_dev(self.T(x, torch.float64), run=self.mask(sel), status=s)
        sd = sd.cpu().numpy()
        assert [int(sd[k]) for k in sel] == [int(v) for v in stat]
        assert std == first_bad(sd[k] for k in sorted(sel))
        run = np.zeros(self.nmat, np.int32); run[list(sel)] = 1
        self.assert_untouched([torch.as_tensor(sd)], run)
        self.assert_state()
        return st, stat

    # ---- the whole-batch interface (bs_cases) ----
    def solve_for_update(self, rhs_list, trans="N", want_solution=0):
        st, stat, out = self.h.solve_for_update(rhs_list, trans, want_solution)
        begin = np.concatenate([[0], np.cumsum([len(np.asarray(ii).reshape(-1)) for ii, _ in rhs_list])]).astype(np.int64)
        irhs = np.concatenate([np.asarray(ii, np.int64).reshape(-1) for ii, _ in rhs_list])
        xrhs = np.concatenate([np.asarray(x, np.float64) for _, x in rhs_list]) if rhs_list[0][1] is not None else None
        r = self.solve_dev(begin, irhs, xrhs, trans, want_solution, None, None, None, None, None)
        assert st == r[0]
        self.check_solve(st, stat, out if want_solution else None, list(range(self.nmat)), r, want_solution)
        self.assert_state()
        return st, stat, out

    def update(self, xtbl):
        st, stat = self.h.update(xtbl)
        std, sd = self.d.update_dev(self.T(xtbl, torch.float64))
        assert std == st and np.array_equal(sd.cpu().numpy(), stat)
        self.assert_state()
        return st, stat

    def solve_sparse(self, lists, trans="N"):
        res = self.h.solve_sparse(lists, trans)
        st, out, ustat = res
        counts = [len(r) for r in lists]
        ub = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        units = [p for r in lists for p in r]
        rb = np.concatenate([[0], np.cumsum([len(ii) for ii, _ in units])]).astype(np.int64)
        ir = np.concatenate([np.asarray(ii, np.int64).reshape(-1) for ii, _ in units]) if units else np.zeros(0, np.int64)
        xr = np.concatenate([np.asarray(x, np.float64).reshape(-1) for _, x in units]) if units else np.zeros(0)
        std, sd, nzd, ild, xld = self.d.solve_sparse_dev(self.T(ub, torch.int64), self.T(rb, torch.int64), self.T(ir, torch.int64),
                                                         self.T(xr, torch.float64), trans)
        assert std == st
        sd, nzd = sd.cpu().numpy(), nzd.cpu().numpy()
        ild, xld = ild.cpu().numpy(), xld.cpu().numpy()
        for k in range(self.nmat):
            for q, u in enumerate(range(ub[k], ub[k + 1])):
                assert sd[u] == ustat[k][q]
                n = int(nzd[u])
                assert n == (len(out[k][q][0]) if sd[u] == 0 else -1)
                assert np.array_equal(ild[u, :max(n, 0)], out[k][q][0]) and np.array_equal(xld[u, :max(n, 0)], out[k][q][1])
        self.assert_state()
        return res

    def solve_dense_multi(self, rhs, trans="N"):
        st, x, stat = self.h.solve_dense_multi(rhs, trans)
        std, xd, sd = self.d.solve_dense_multi_dev(self.T(rhs, torch.float64), trans)
        assert std == st and np.array_equal(sd.cpu().numpy(), stat)
        assert np.array_equal(xd.cpu().numpy(), x, equal_nan=True)
        self.assert_state()
        return st, x, stat

    # ---- calls both batches make through the same (host) path ----
    def solve_dense(self, rhs, trans="N"):
        a, b = self.h.solve_dense(rhs, trans), self.d.solve_dense(rhs, trans)
        assert a[0] == b[0] and np.array_equal(a[1], b[1], equal_nan=True) and np.array_equal(a[2], b[2])
        return a

    def get_factors(self, k):
        a, b = self.h.get_factors(k), self.d.get_factors(k)
        assert a[0] == b[0] and all(np.array_equal(a[1][q], b[1][q]) for q in a[1])
        return a

    def info(self, k, name):
        return self.h.info(k, name)

    def launch_count(self):
        return self.h.launch_count()


def make_twin(lib, dev, nmat, m, bnz_cap, mem=None, threads=None, realloc_factor=None):
    def make():
        b = BLUBatch(nmat, m, bnz_cap, lib=lib)
        if threads:
            b.threads_per_basis = threads
        if mem:
            b.l_mem = mem; b.u_mem = mem; b.w_mem = mem
        if realloc_factor is not None:
            b.realloc_factor = realloc_factor
        return b
    return Twin(make, dev)
