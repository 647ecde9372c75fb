"""blu_batch_save / blu_batch_restore on the B200 at configs[1]'s shape (gen.basis(seed, 2000, 700, 5.0)): 4,096 bases
with update history, 64 parents saved and each restored into 63 slots; a sample of 256 lanes then goes on against its
oracles, and every basis that was not a destination keeps its dense solves bit for bit.  Restore equals copy on twin
batches; cross-batch on one device and (with two GPUs) across devices; the wrong-m rejection."""
import numpy as np
import pytest
import torch

from blu_b200 import BLUBatch, gen
from copy_cases import CLane, assert_copies, snapshot
from save_cases import SaveTwin, fork, restore_fork
from subset_cases import assert_getters, csc, factorize, replay, solve_n, solve_t, update

pytestmark = pytest.mark.gpu

M, NSLACK, NMAT, NPAR, TRACK = 2000, 700, 4096, 64, 256


def assert_dense_tracked(b, lanes, seed):
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


def test_gpu_restore_4096_fanout():
    bb, be, bi, bx, _ = gen.batch(NMAT, M, NSLACK, 5.0, 81000, 82000)
    lanes = [CLane(83000 + k, M, nslack=NSLACK, pmean=5.0, policy=k % 2) for k in range(TRACK)]
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
    rest = list(range(TRACK, NMAT))
    cols = []
    for k in rest:
        cp, ri, v = gen.basis(84000 + k, M, 0, 3.0)
        cols.append((ri[cp[0]:cp[1]], v[cp[0]:cp[1]]))
    st, stat, out = b.solve_for_update_subset(rest, cols, "N", want_solution=1)
    assert st == 0
    leave = [(np.array([int(o[0][np.argmax(np.abs(o[1]))])]), None) for o in out]
    xt = np.array([o[1][np.argmax(np.abs(o[1]))] for o in out])
    assert b.solve_for_update_subset(rest, leave, "T")[0] == 0 and b.update_subset(rest, xt)[0] == 0
    history(b, lanes, list(range(TRACK)), 3)
    # parent p < 64 to 3 tracked children in [64, 256) and 60 untracked ones in [256, 4096)
    dst, src = [], []
    for p in range(NPAR):
        kids = [NPAR + 3 * p + q for q in range(3)] + [TRACK + 60 * p + q for q in range(60)]
        dst += kids
        src += [p] * len(kids)
    x = np.tile(np.random.default_rng(5).uniform(-1, 1, M), NMAT)
    before = {tr: b.solve_dense(x, tr) for tr in "NT"}
    for L in lanes:
        for tr in "NT":
            L.oracle.solve_dense(x[:M], tr)
    imgs = b.save_dev(list(range(NPAR)))
    assert all(t.data_ptr() % 256 == 0 for t in imgs)
    assert b.restore_dev(dst, [imgs[s] for s in src]) == 0
    for d, s in zip(dst, src):
        if d < len(lanes):
            lanes[d].adopt(lanes[s])
    after = {tr: b.solve_dense(x, tr) for tr in "NT"}
    keep = sorted(set(range(NMAT)) - set(dst))
    for tr in "NT":
        assert np.array_equal(before[tr][1][keep], after[tr][1][keep]), tr
        for d, s in zip(dst, src):
            assert np.array_equal(after[tr][1][d], before[tr][1][s]), (tr, d, s)
    for L in lanes:
        for tr in "NT":
            L.oracle.solve_dense(x[:M], tr)
    sample = list(range(0, TRACK, 5))
    pairs = [(k, src[dst.index(k)]) for k in sample if k in dst]
    snap = snapshot(b, sample + [s for _, s in pairs], seed=9, lanes=lanes)
    assert_copies(snap, [d for d, _ in pairs], [s for _, s in pairs])
    for r in range(2):
        replay(b, lanes, 5, 85000 + r, dense_every=0)
        assert_dense_tracked(b, lanes, 85050 + r)
    # the destinations refactorize from their parents' B, which the images carried
    assert b.factorize_resident() == 0
    for L in lanes:
        cp, ri, v = csc(L.factored)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.cols = list(L.factored); L.pending = None; L.refactor = False
    assert_getters(b, lanes)
    assert_dense_tracked(b, lanes, 85100)
    b.close()


def twin_lanes(nmat, seed):
    return [CLane(seed + k, M, nslack=NSLACK, pmean=5.0, policy=k % 2) for k in range(nmat)]


def test_gpu_restore_equals_copy():
    """256-basis twin batches, one forking with copy and one with save_dev + restore_dev: bit-identical after every call"""
    nmat = 256
    lanes = twin_lanes(nmat, 86000)
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * M
    tw = SaveTwin(lambda: BLUBatch(nmat, M, cap, device=0), torch.device("cuda", 0), "dev")
    factorize(tw, lanes, list(range(nmat)))
    history(tw, lanes, list(range(nmat)), 2)
    pend = solve_n(tw, lanes, list(range(16)))
    solve_t(tw, lanes, pend, want=0)
    dst = list(range(16, nmat))
    src = [k % 16 for k in dst]
    fork(tw, lanes, dst, src)
    pairs = [(d, s) for d, s in zip(dst, src) if d % 7 == 0]
    snap = snapshot(tw, sorted({k for p in pairs for k in p}), seed=3, lanes=lanes)
    assert_copies(snap, [d for d, _ in pairs], [s for _, s in pairs])
    assert update(tw, lanes, [k for k in range(nmat) if lanes[k].pending is not None])[0] == 0
    replay(tw, lanes, 3, 86100, dense_every=3)


def cross(device_b):
    """64 bases saved from a batch on cuda:0 and restored into a batch on device_b with other capacities"""
    nmat = 64
    lanes = twin_lanes(nmat, 87000)
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * M
    a = BLUBatch(nmat, M, cap, device=0)
    factorize(a, lanes, list(range(nmat)))
    history(a, lanes, list(range(nmat)), 2)
    pend = solve_n(a, lanes, list(range(0, nmat, 2)))
    solve_t(a, lanes, pend, want=1)
    other = twin_lanes(48, 87500)
    with torch.cuda.device(device_b):
        b = BLUBatch(48, M, 16, device=device_b)
        b.l_mem = 6 * cap; b.u_mem = 6 * cap; b.w_mem = 20 * cap
    factorize(b, other, list(range(48)))
    imgs = a.save_dev(list(range(nmat)))
    dev_b = torch.device("cuda", device_b)
    moved = [t.to(dev_b) for t in imgs]
    dst = list(range(0, 48, 3))
    src = list(range(0, 2 * len(dst), 2))
    with torch.cuda.device(device_b):
        assert b.restore_dev(dst, [moved[s] for s in src]) == 0
    for d, s in zip(dst, src):
        other[d].adopt(lanes[s])
    sa = snapshot(a, src, seed=4, lanes=lanes)
    sb = snapshot(b, dst, seed=4, lanes=other)
    from subset_cases import assert_same_snapshot
    for d, s in zip(dst, src):
        assert_same_snapshot({0: sa[s]}, {0: sb[d]})
    assert update(b, other, [d for d in dst if other[d].pending is not None])[0] == 0
    replay(b, other, 4, 87100, dense_every=2)


def test_gpu_restore_cross_batch():
    cross(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_gpu_restore_cross_device():
    cross(1)


def test_gpu_restore_rejects_wrong_m():
    """an image of another dimension is refused from its header, before any launch"""
    a, b = BLUBatch(2, 50, 400, device=0), BLUBatch(2, 60, 400, device=0)
    cp, ri, v = gen.basis(88000, 50, 10, 4.0)
    bb = np.concatenate([cp[:-1], cp[:-1]]); be = np.concatenate([cp[1:], cp[1:]])
    assert a.factorize(bb, be, ri, v)[0] == 0
    img = a.save_dev([0])
    n = b.launch_count()
    assert b.restore_dev([1], img) == -4 and b.launch_count() == n + 1      # (the header gather)
    assert restore_fork(a, [1], [0], "dev") == 0
