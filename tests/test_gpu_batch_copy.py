"""blu_batch_copy on the B200 at configs[1]'s shape (gen.basis(seed, 2000, 700, 5.0)): 4,096 bases with update history,
64 parents each copied to 63 children; a sample of 256 parent and child lanes then goes on against its oracles, every
basis that was not a destination keeps its dense solves bit for bit, and the children refactorize from their parents'
resident B."""
import numpy as np
import pytest
import torch

from blu_b200 import BLUBatch, gen
from copy_cases import CLane, assert_copies, fork, make_copy_twin, snapshot
from subset_cases import assert_getters, csc, factorize, replay, solve_n, solve_t, update

pytestmark = pytest.mark.gpu

M, NSLACK, NMAT, NPAR, TRACK = 2000, 700, 4096, 64, 256


def assert_dense_tracked(b, lanes, seed):
    """solve_dense 'N' / 'T' on the whole batch (a right-hand side for every one of its bases) against the oracles of
    the tracked lanes, which hold bases 0 .. len(lanes)-1"""
    rhs = np.random.default_rng(seed).uniform(-1.0, 1.0, b.nmat * M)
    for tr in "NT":
        _, x, stat = b.solve_dense(rhs, tr)
        for k, L in enumerate(lanes):
            ost, xo = L.oracle.solve_dense(rhs[k * M:(k + 1) * M], tr)
            assert stat[k] == ost, (k, tr, stat[k], ost)
            if ost == 0 and not L.refactor:
                assert np.array_equal(x[k], xo), (k, tr)


def history(b, lanes, ks, rounds):
    for _ in range(rounds):
        pend = solve_n(b, lanes, ks)
        solve_t(b, lanes, pend, want=1)
        ok = [k for k in ks if lanes[k].pending is not None]
        if ok:
            update(b, lanes, ok)
        redo = [k for k in ks if lanes[k].refactor]
        if redo:
            factorize(b, lanes, redo)


def test_gpu_copy_4096_fanout():
    bb, be, bi, bx, _ = gen.batch(NMAT, M, NSLACK, 5.0, 61000, 62000)
    lanes = [CLane(63000 + k, M, nslack=NSLACK, pmean=5.0, policy=k % 2) for k in range(TRACK)]
    # the tracked bases 0..255 are factorized from their lanes' B (appended to the batch's b_i / b_x), the others from gen.batch
    bb, be, ext_i, ext_x, off = bb.copy(), be.copy(), [bi], [bx], len(bi)
    for k, L in enumerate(lanes):
        cp, ri, v = csc(L.cols)
        bb[k * M:(k + 1) * M] = cp[:-1] + off
        be[k * M:(k + 1) * M] = cp[1:] + off
        ext_i.append(ri); ext_x.append(v); off += len(ri)
    bi, bx = np.concatenate(ext_i), np.concatenate(ext_x)
    b = BLUBatch(NMAT, M, int((be - bb).reshape(NMAT, M).sum(1).max()) + 4 * M, device=0)
    st, status = b.factorize(bb, be, bi, bx)
    assert st == 0 and (status == 0).all()
    for L in lanes:
        cp, ri, v = csc(L.cols)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.factored = list(L.cols)
    assert_getters(b, lanes)
    # one basis change on every untracked basis; the tracked ones go through theirs against the oracles
    rest = list(range(TRACK, NMAT))
    cols = []
    for k in rest:
        cp, ri, v = gen.basis(64000 + k, M, 0, 3.0)
        cols.append((ri[cp[0]:cp[1]], v[cp[0]:cp[1]]))
    st, stat, out = b.solve_for_update_subset(rest, cols, "N", want_solution=1)
    assert st == 0
    leave = [(np.array([int(o[0][np.argmax(np.abs(o[1]))])]), None) for o in out]
    xt = np.array([o[1][np.argmax(np.abs(o[1]))] for o in out])
    assert b.solve_for_update_subset(rest, leave, "T")[0] == 0 and b.update_subset(rest, xt)[0] == 0
    history(b, lanes, list(range(TRACK)), 3)
    # pattern (a): parent p < 64 to 3 tracked children in [64, 256) and 60 untracked ones in [256, 4096)
    dst, src = [], []
    for p in range(NPAR):
        kids = [NPAR + 3 * p + q for q in range(3)] + [TRACK + 60 * p + q for q in range(60)]
        dst += kids
        src += [p] * len(kids)
    parents = list(range(NPAR))
    x = np.tile(np.random.default_rng(5).uniform(-1, 1, M), NMAT)
    before = {tr: b.solve_dense(x, tr) for tr in "NT"}
    for L in lanes:      # (the dense solves run on every basis and compact its pivot sequence)
        for tr in "NT":
            L.oracle.solve_dense(x[:M], tr)
    assert b.graph_capture("N") == 0
    launches = b.launch_count()
    fork(b, lanes, dst, src)
    assert b.launch_count() == launches + 1
    assert b.graph_launch() == -2
    after = {tr: b.solve_dense(x, tr) for tr in "NT"}
    for tr in "NT":
        assert np.array_equal(before[tr][1][parents], after[tr][1][parents]), tr
        for d, s in zip(dst, src):
            assert np.array_equal(after[tr][1][d], before[tr][1][s]), (tr, d, s)
    for L in lanes:
        for tr in "NT":
            L.oracle.solve_dense(x[:M], tr)
    sample = list(range(0, TRACK, 5))
    snap = snapshot(b, sample + [src[dst.index(k)] for k in sample if k in dst], seed=9, lanes=lanes)
    assert_copies(snap, [k for k in sample if k in dst], [src[dst.index(k)] for k in sample if k in dst])
    # divergent futures of parents and children, every tracked basis against its oracle after every call
    for r in range(2):      # (replay's own dense checks size the right-hand sides to the lanes, not the batch)
        replay(b, lanes, 5, 65000 + r, dense_every=0)
        assert_dense_tracked(b, lanes, 65050 + r)
    # the children refactorize from their parents' resident B
    assert b.factorize_resident() == 0
    for L in lanes:
        cp, ri, v = csc(L.factored)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.cols = list(L.factored); L.pending = None; L.refactor = False
    assert_getters(b, lanes)
    assert b.graph_capture("N") == 0 and b.graph_launch() == 0
    for L in lanes:
        cp, ri, v = csc(L.factored)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
    assert_getters(b, lanes)
    assert_dense_tracked(b, lanes, 65100)
    b.close()


def test_gpu_copy_dev_twins():
    """one copy_dev pass on twin batches of 64 configs[1]-shaped bases: bit-identical to copy, then on against the oracles"""
    nmat = 64
    lanes = [CLane(66000 + k, M, nslack=NSLACK, pmean=5.0, policy=k % 2) for k in range(nmat)]
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * M
    tw = make_copy_twin(None, torch.device("cuda", 0), nmat, M, cap)
    factorize(tw, lanes, list(range(nmat)))
    history(tw, lanes, list(range(nmat)), 2)
    dst = list(range(16, nmat))
    src = [k % 16 for k in dst]
    fork(tw, lanes, dst, src)
    assert_copies(snapshot(tw, range(nmat), seed=3, lanes=lanes), dst, src)
    replay(tw, lanes, 4, 66100, dense_every=2)
