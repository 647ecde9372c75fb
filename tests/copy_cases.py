"""Shared pieces of the tests of blu_batch_copy / blu_batch_copy_dev: lanes (subset_cases.Lane) whose oracle logs every
call, so that forking lane s into lane d gives d a fresh oracle that went through s's history -- the object a copy of
basis s must behave as -- while d keeps its own pool of entering columns and so its own future."""
import numpy as np
import torch

from dev_cases import Twin
from parity import oracle_for
from subset_cases import PER_BASIS, Lane, assert_same_snapshot


class LoggedOracle:
    """an oracle object that records every call that changes its state, so that the history can be replayed"""

    def __init__(self, m, nnz, factor):
        self.args = (m, nnz, factor)
        self.o = oracle_for(m, nnz, factor)
        self.log = []

    def _call(self, name, *args, **kw):
        self.log.append((name, [a.copy() if isinstance(a, np.ndarray) else a for a in args], dict(kw)))
        return getattr(self.o, name)(*args, **kw)

    def factorize(self, *a, **kw):
        return self._call("factorize", *a, **kw)

    def solve_dense(self, *a, **kw):      # compacts the pivot sequence (pivotlen)
        return self._call("solve_dense", *a, **kw)

    def solve_sparse(self, *a, **kw):
        return self._call("solve_sparse", *a, **kw)

    def solve_for_update(self, *a, **kw):
        return self._call("solve_for_update", *a, **kw)

    def update(self, *a, **kw):
        return self._call("update", *a, **kw)

    def set_param(self, *a, **kw):
        return self._call("set_param", *a, **kw)

    def __getattr__(self, name):
        return getattr(self.o, name)

    def replica(self):
        """a fresh oracle that ran this one's history"""
        r = LoggedOracle(*self.args)
        for name, args, kw in self.log:
            r._call(name, *args, **kw)
        return r


class CLane(Lane):
    """a Lane whose oracle logs its calls"""

    def __init__(self, seed, m, nslack=None, pmean=4.0, policy=0):
        super().__init__(seed, m, nslack=nslack, pmean=pmean, policy=policy)
        nnz = sum(len(r) for r, _ in self.cols)
        self.oracle = LoggedOracle(m, nnz + 8 * m, 400 if m <= 200 else 20)

    def adopt(self, src):
        """this lane becomes what basis src's copy is: its oracle, B, factored B and pending pair; the pool and the
        policy stay this lane's own"""
        self.oracle = src.oracle.replica()
        self.cols = list(src.cols)
        self.factored = None if src.factored is None else list(src.factored)
        self.rejected = src.rejected
        self.pending = src.pending
        self.refactor = src.refactor


def fork(b, lanes, dst, src):
    """copy on the batch (b may be a dev_cases.Twin) and on the lanes; bases past the last lane have no oracle"""
    st = b.copy(dst, src)
    assert st == 0, st
    for d, s in zip(dst, src):
        if d < len(lanes):
            lanes[d].adopt(lanes[s])


def snapshot(b, ks, seed=1, lanes=None):
    """subset_cases.snapshot with one right-hand side for every basis, so that a copy and its source can be compared:
    every per-basis getter, get_factors where nupdate == 0, solve_dense 'N' and 'T' (which compact the pivot sequence;
    lanes, when given, have their oracles run them too)"""
    m = b.m
    rhs = np.tile(np.random.default_rng(seed).uniform(-1.0, 1.0, m), (b.nmat, 1, 1))
    xs = {tr: b.solve_dense_multi(rhs, tr) for tr in "NT"}
    for L in lanes or []:
        for tr in "NT":
            L.oracle.solve_dense(rhs[0, 0], tr)
    snap = {}
    for k in ks:
        s = {n: b.info(k, n) for n in PER_BASIS}
        if s["nupdate"] == 0:
            s["factors"] = b.get_factors(k)
        for tr in "NT":
            s["dense" + tr] = (xs[tr][2][k, 0], xs[tr][1][k, 0].copy())
        snap[k] = s
    return snap


def assert_copies(snap, dst, src):
    """every observable of basis d equals that of its source s (one snapshot of both)"""
    for d, s in zip(dst, src):
        assert_same_snapshot({0: snap[d]}, {0: snap[s]})


def fork_and_check(b, lanes, dst, src, seed):
    """fork, then check that each destination shows exactly what its source shows"""
    fork(b, lanes, dst, src)
    ks = sorted(set(dst) | set(src))
    assert_copies(snapshot(b, ks, seed=seed, lanes=lanes), dst, src)


class CopyTwin(Twin):
    """twin batches: `h` copies through blu_batch_copy, `d` through blu_batch_copy_dev with the map as a tensor"""

    def copy(self, dst, src):
        st = self.h.copy(dst, src)
        f = np.full(self.nmat, -1, np.int32)
        f[list(dst)] = src
        assert self.d.copy_dev(self.T(f, torch.int32)) == st
        self.assert_state()
        return st


def make_copy_twin(lib, dev, nmat, m, bnz_cap):
    from blu_b200 import BLUBatch
    return CopyTwin(lambda: BLUBatch(nmat, m, bnz_cap, device=0 if lib is None else -1, lib=lib), dev)
