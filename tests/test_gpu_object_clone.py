"""blu_clone and object images on the B200: an m = 1,000 object and a configs[2]-shaped object (gen.config3, m =
100,000) cloned after basis changes, the clone's solves and getters equal to the source's bit for bit; and a root object
of configs[1]'s shape restored into 64 slots of a 256-basis batch whose bases then run divergent _dev rounds against
their oracles."""
import numpy as np
import pytest
import torch

from blu_b200 import BLU, gen
from copy_cases import CLane
from dev_cases import make_twin
from object_cases import Objects, assert_same_record, record
from subset_cases import factorize, replay, solve_n, solve_t, update

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def test_gpu_clone_m1000():
    """m = 1,000: after 12 rounds of basis changes and with a pending 'N' + 'T' pair, the clone's record equals the
    source's, which is unchanged; then source and clone run in lockstep and a second clone on its own schedule, all
    against their oracles"""
    m = 1000
    lanes = [CLane(66000, m, nslack=300, pmean=5.0), CLane(66100, m, nslack=300, pmean=5.0, policy=1)]
    src = BLU(m, sum(len(r) for r, _ in lanes[0].cols) + 4 * m, device=0)
    one = Objects([[src]])
    factorize(one, lanes[:1], [0])
    replay(one, lanes[:1], 12, 66200, dense_every=4)
    if lanes[0].refactor:
        factorize(one, lanes[:1], [0])
    pend = solve_n(one, lanes[:1], [0])
    solve_t(one, lanes[:1], pend, want=1)
    before = record(src)
    c, d = src.clone(), src.clone()
    assert_same_record(before, record(src))
    assert_same_record(before, record(c))
    assert_same_record(before, record(d))
    lanes[1].adopt(lanes[0])
    pair = Objects([[src, c], [d]])
    if lanes[0].pending is not None:
        update(pair, lanes, [0, 1])
    replay(pair, lanes, 10, 66300, dense_every=3)


def test_gpu_clone_config3():
    """configs[2]'s shape (100,000 rows, a 2,000-wide bump) after 40 column replacements and a pending 'N' solve: the
    clone's record (getters, parameters, image) equals the source's; both then take 10 more replacements in lockstep
    with bit-identical solutions, and their dense and sparse solves agree bit for bit"""
    m, bump = 100000, 2000
    cp, ri, v = gen.config3(m, bump, seed=7001)
    pcp, pri, pv = gen.column_pool(7002, m, 60)
    dense = bump * bump
    src = BLU(m, len(v), device=0)
    src.threads_per_basis = 1024
    src.l_mem = int(2.2 * (dense // 2 + 10 * m)) + 40 * m
    src.u_mem = int(1.2 * (dense // 2 + 10 * m)) + 40 * m
    src.w_mem = int(3.0 * dense + 40 * m)
    assert src.factorize(cp[:-1], cp[1:], ri, v) == 0
    objs = [src]

    def change(it):
        idx, val = pri[pcp[it]:pcp[it + 1]], pv[pcp[it]:pcp[it + 1]]
        out = []
        for o in objs:
            assert o.solve_for_update(len(idx), idx, val, "N", 1) == 0
            out.append((o.nzlhs, o.ilhs[:o.nzlhs].copy(), o.lhs.copy()))
        for x in out[1:]:
            assert x[0] == out[0][0] and np.array_equal(x[1], out[0][1]) and np.array_equal(x[2], out[0][2])
        j = int(np.argmax(np.abs(out[0][2])))
        for o in objs:
            assert o.solve_for_update(1, np.array([j]), None, "T", 0) == 0
            assert o.update(out[0][2][j]) == 0

    for it in range(40):
        change(it)
    idx, val = pri[pcp[40]:pcp[41]], pv[pcp[40]:pcp[41]]
    assert src.solve_for_update(len(idx), idx, val, "N", 0) == 0
    before = record(src)
    c = src.clone()
    assert_same_record(before, record(src))
    assert_same_record(before, record(c))
    objs.append(c)
    for it in range(41, 51):
        change(it)
    for n in ("nupdate", "nforrest", "u_nz", "r_nz", "pivot_error", "max_eta", "nrealloc"):
        assert src.info(n) == c.info(n), n
    b = gen.rhs(7003, m)
    for tr in "NT":
        s0, x0 = src.solve_dense(b, tr)
        s1, x1 = c.solve_dense(b, tr)
        assert s0 == s1 == 0 and np.array_equal(x0, x1), tr
        sidx, sval = gen.sparse_rhs_np(7004, m, 100)
        assert src.solve_sparse(100, sidx, sval, tr) == c.solve_sparse(100, sidx, sval, tr) == 0
        assert src.nzlhs == c.nzlhs and np.array_equal(src.ilhs[:src.nzlhs], c.ilhs[:c.nzlhs]) and np.array_equal(src.lhs, c.lhs)


def test_gpu_root_object_into_batch_slots():
    """A root object of configs[1]'s shape (m = 2,000), after basis changes, restored from one device image into 64 of
    the 256 slots of a batch (host and _dev twins); every basis then runs its own schedule through the _dev calls
    against its oracle"""
    m, nmat = 2000, 256
    root = CLane(67000, m, nslack=700, pmean=5.0)
    g = BLU(m, sum(len(r) for r, _ in root.cols) + 4 * m, device=0)
    one = Objects([[g]])
    factorize(one, [root], [0])
    replay(one, [root], 6, 67100, dense_every=0)
    if root.pending is not None or root.refactor:
        factorize(one, [root], [0])
    lanes = [CLane(67200 + k, m, nslack=700, pmean=5.0, policy=k % 2) for k in range(nmat)]
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m
    tw = make_twin(None, DEV, nmat, m, cap)
    factorize(tw, lanes, list(range(nmat)))
    img = g.save_dev()
    assert img.device == DEV and img.data_ptr() % 256 == 0
    dst = list(range(0, nmat, 4))
    assert tw.d.restore_dev(dst, [img] * len(dst)) == 0
    assert tw.h.restore(dst, [img.cpu().numpy()] * len(dst)) == 0
    tw.assert_state()
    for k in dst:
        lanes[k].adopt(root)
    rhs = np.random.default_rng(3).uniform(-1.0, 1.0, m)
    st, x = g.solve_dense(rhs, "N")
    _, xb, stat = tw.solve_dense(np.tile(rhs, nmat), "N")
    root.oracle.solve_dense(rhs, "N")
    for k, L in enumerate(lanes):
        L.oracle.solve_dense(rhs, "N")
    for k in dst:
        assert stat[k] == st and np.array_equal(xb[k], x), k
    replay(tw, lanes, 6, 67300, dense_every=3)
