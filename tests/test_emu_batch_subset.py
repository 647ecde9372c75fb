"""The batch calls on a subset of the bases under the SIMT emulator: each basis ends exactly as its own oracle object
after the calls it was selected in, and the bases that were not selected do not move."""
import os
import subprocess

import numpy as np
import pytest

from blu_b200 import BLU, BLUBatch, load_library
from mv_cases import layout as mv_layout, make_pool
from subset_cases import (Lane, _pf, _pi, assert_dense, assert_getters, assert_same_snapshot, csc, factorize, layout,
                          raw_factorize_subset, raw_solve_subset, raw_update_subset, replay, snapshot, solve_n, solve_t,
                          update)

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


def new_batch(emu, lanes, mem=None):
    m = lanes[0].m
    b = BLUBatch(len(lanes), m, max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m, lib=emu)
    b.threads_per_basis = 64
    if mem:
        b.l_mem = mem; b.u_mem = mem; b.w_mem = mem
    return b


def start(emu, nmat, m, seed0, mem=None, nslack=None):
    lanes = [Lane(seed0 + k, m, nslack=nslack, policy=k % 4) for k in range(nmat)]
    b = new_batch(emu, lanes, mem)
    factorize(b, lanes, list(range(nmat)))
    return b, lanes


def test_emu_subset_schedule_replay(emu):
    """8 bases at m = 40 and 6 at m = 80 over 30 rounds, then 8 at m = 16 over 90 rounds (nforrest == m needs m
    updates), each basis on its own schedule: every refactorization trigger fires on some basis, and every basis
    matches its oracle after every call."""
    stats = {}
    for nmat, m, nslack, rounds, seed in ((8, 40, 20, 30, 11000), (6, 80, 40, 30, 11100), (8, 16, 10, 90, 11200)):
        b, lanes = start(emu, nmat, m, seed, nslack=nslack)
        replay(b, lanes, rounds, seed + 50, stats=stats)
        assert_dense(b, lanes, seed + 99)
    assert all(stats.get(k, 0) > 0 for k in ("update_cost", "nforrest", "-5", "-6")), str(stats)


def test_emu_subset_untouched(emu):
    """The bases not selected keep every per-basis getter, their factors and their dense solves bit for bit across
    the three subset calls on other bases -- also while one of them has a pending solve_for_update pair."""
    m = 50
    b, lanes = start(emu, 6, m, 12000)
    pend = solve_n(b, lanes, [0, 1, 2, 3])
    solve_t(b, lanes, pend, want=1)
    update(b, lanes, [0, 1])                          # bases 0, 1 updated; 2, 3 pending; 4, 5 fresh
    for sel, call in (([4, 0], "factorize"), ([5, 1], "solve"), ([1], "update")):
        other = [k for k in range(6) if k not in sel]
        before = snapshot(b, other, seed=len(sel), lanes=lanes)
        if call == "factorize":
            factorize(b, lanes, sel)
        elif call == "solve":
            solve_t(b, lanes, solve_n(b, lanes, sel), want=0)
        else:
            update(b, lanes, sel)
        assert_same_snapshot(before, snapshot(b, other, seed=len(sel), lanes=lanes))
    update(b, lanes, [2, 3])
    assert_dense(b, lanes, 12050)


def test_emu_subset_pending_pair_survives(emu):
    """Basis A does 'N' + 'T', the others refactorize, then update_subset([A]) matches the oracle."""
    m = 60
    b, lanes = start(emu, 5, m, 12100)
    solve_t(b, lanes, solve_n(b, lanes, [2]), want=1)
    factorize(b, lanes, [4, 0, 1, 3])
    assert update(b, lanes, [2])[0] == 0
    assert b.info(2, "nupdate") == 1 and all(b.info(k, "nupdate") == 0 for k in (0, 1, 3, 4))
    assert_dense(b, lanes, 12150)


def test_emu_subset_malformed(emu):
    """Every call-level reject: BLU_ERROR_INVALID_ARGUMENT, no launch, no state change.  nsel == 0 launches nothing."""
    m = 40
    b, lanes = start(emu, 4, m, 12200)
    solve_t(b, lanes, solve_n(b, lanes, [1]), want=0)     # a pending pair on basis 1
    bb, be, bi, bx = layout([lanes[0].cols, lanes[2].cols])
    nz = len(bi)
    before = snapshot(b, range(4), lanes=lanes)
    launches = b.launch_count()
    F = lambda *a: raw_factorize_subset(b, *a)
    assert F(-1, [0], bb, be, bi, bx, nz) == -4
    assert F(5, [0, 1, 2, 3, 0], np.tile(bb, 3)[:5 * m], np.tile(be, 3)[:5 * m], bi, bx, nz) == -4      # nsel > nmat
    assert F(2, [0, 4], bb, be, bi, bx, nz) == -4                                        # index outside [0, nmat)
    assert F(2, [-1, 2], bb, be, bi, bx, nz) == -4
    assert F(2, [2, 2], bb, be, bi, bx, nz) == -4                                        # duplicate
    assert F(2, None, bb, be, bi, bx, nz) == -4                                          # missing arrays
    assert F(2, [0, 2], None, be, bi, bx, nz) == -4
    assert F(2, [0, 2], bb, None, bi, bx, nz) == -4
    assert F(2, [0, 2], bb, be, None, bx, nz) == -4
    assert F(2, [0, 2], bb, be, bi, None, nz) == -4
    assert F(2, [0, 2], bb, be, bi, bx, -1) == -4
    bad = be.copy(); bad[7] = nz + 1
    assert F(2, [0, 2], bb, bad, bi, bx, nz) == -4                                       # b_end beyond bnz_total
    bad = bb.copy(); bad[3] = -1
    assert F(2, [0, 2], bad, be, bi, bx, nz) == -4                                       # negative b_begin
    S = lambda *a, **k: raw_solve_subset(b, *a, **k)
    ir, xr = np.array([1, 2, 3]), np.ones(3)
    assert S(-1, [0], [0, 3], ir, xr) == -4
    assert S(5, [0, 1, 2, 3, 0], [0, 1, 1, 1, 2, 3], ir, xr) == -4
    assert S(1, [4], [0, 3], ir, xr) == -4
    assert S(2, [3, 3], [0, 1, 3], ir, xr) == -4
    assert S(1, None, [0, 3], ir, xr) == -4
    assert S(1, [0], None, ir, xr) == -4
    assert S(1, [0], [0, 3], None, xr) == -4
    p = lambda a: _pi(np.array(a))
    assert emu.blu_batch_solve_for_update_subset(b._h, 1, p([0]), p([0, 3]), p(ir), _pf(xr), 1, None, None, None, None, b"N") == -4
    assert raw_solve_subset(b, 2, [0, 2], [0, 4, 3], ir, xr) == -4                          # offset beyond rhs_begin[nsel]
    assert raw_solve_subset(b, 2, [0, 2], [-1, 1, 3], ir, xr) == -4                         # negative offset
    assert raw_solve_subset(b, 2, [0, 2], [0, 1, -1], ir, xr) == -4                         # negative total
    U = lambda *a: raw_update_subset(b, *a)
    assert U(-1, [1], [1.0]) == -4
    assert U(5, [0, 1, 2, 3, 0], np.ones(5)) == -4
    assert U(1, [4], [1.0]) == -4
    assert U(2, [1, 1], [1.0, 1.0]) == -4
    assert U(1, None, [1.0]) == -4
    assert U(1, [1], None) == -4
    assert F(0, None, None, None, None, None, 0) == 0 and S(0, None, None, None, None) == 0 and U(0, None, None) == 0
    assert b.launch_count() == launches
    assert_same_snapshot(before, snapshot(b, range(4), lanes=lanes))
    # a single object from blu_create
    g = BLU(m, 400, lib=emu)
    assert emu.blu_batch_factorize_subset(g._h, 0, None, None, None, None, None, 0, None) == -4
    assert emu.blu_batch_update_subset(g._h, 0, None, None, None) == -4
    assert emu.blu_batch_solve_for_update_subset(g._h, 0, None, None, None, None, 0, None, None, None, None, b"N") == -4
    update(b, lanes, [1])          # the pending pair is still intact


def test_emu_subset_per_basis_errors(emu):
    """One selected basis has a row index >= m, one a column with b_end < b_begin, one a duplicate row; the fourth
    factorizes.  An update of a basis never factorized (or without both solves) answers InvalidCall for it alone."""
    m = 45
    lanes = [Lane(12300 + k, m) for k in range(6)]
    b = new_batch(emu, lanes)
    bad_row = list(lanes[0].cols); bad_row[5] = (np.array([1, m]), np.array([1.0, 2.0]))
    dup_row = list(lanes[2].cols); dup_row[7] = (np.array([3, 3]), np.array([1.0, 2.0]))
    lanes[0].cols, lanes[2].cols = bad_row, dup_row
    bb, be, bi, bx = layout([lanes[k].cols for k in (0, 1, 2, 3)])
    be[m + 9] = bb[m + 9] - 1                                   # basis 1, column 9: b_end < b_begin
    st, stat = b.factorize_subset([0, 1, 2, 3], bb, be, bi, bx)
    exp = []
    for r, k in enumerate((0, 1, 2, 3)):
        cp, ri, v = csc(lanes[k].cols)
        e = cp[1:].copy()
        if k == 1:
            e[9] = cp[9] - 1
        exp.append(lanes[k].oracle.factorize(cp[:-1], e, ri, v))
    assert list(stat) == exp and exp[0] == -4 and exp[1] == -4 and exp[2] < 0 and exp[3] == 0, (stat, exp)
    assert st == -4
    for k in (0, 1, 2):
        lanes[k].rejected = True
    assert_getters(b, lanes, [3])
    pend = solve_n(b, lanes, [3])
    solve_t(b, lanes, pend, want=0)
    # basis 4 was never factorized, basis 3 has both solves
    st, stat = b.update_subset([4, 3], [1.0, lanes[3].pending[1]])
    assert lanes[4].oracle.update(1.0) == stat[0] == -2
    assert lanes[3].oracle.update(lanes[3].pending[1]) == stat[1] == 0
    assert st == -2
    lanes[3].pending = None
    assert_getters(b, lanes, [3])
    # basis 3 again: an update without the solves
    st, stat = b.update_subset([3], [1.0])
    assert stat[0] == lanes[3].oracle.update(1.0) == -2


def test_emu_subset_tight_stores(emu):
    """Stores far too small, grown by no more than asked (realloc_factor 1): Reallocate happens inside
    factorize_subset and solve_for_update_subset over and over, and nothing changes in the results."""
    m = 60
    lanes = [Lane(12400 + k, m, nslack=10) for k in range(5)]
    b = new_batch(emu, lanes, mem=90)
    b.realloc_factor = 1.0
    nr = b.info(0, "nrealloc")
    factorize(b, lanes, [3, 1, 0, 4, 2])
    assert b.info(0, "nrealloc") > nr
    stats = replay(b, lanes, 30, 12450)
    assert stats["realloc_factorize"] > 0 and stats["realloc_solve"] > 0, stats
    assert_dense(b, lanes, 12490)


@pytest.mark.parametrize("kd,tail", [(64, 128)])
def test_emu_subset_split_factorization(emu, kd, tail):
    """The subset factorization through the head / tail / build launches (split_min = 0, dense_k), the way
    test_emu_split_batch runs the whole batch."""
    m = 170
    lanes = [Lane(12500 + k, m, nslack=30, pmean=5.0) for k in range(4)]
    b = new_batch(emu, lanes)
    b.dense_k = kd; b.split_min = 0; b.tail_threads = tail
    l0 = b.launch_count()
    factorize(b, lanes, [2, 0])
    assert b.launch_count() - l0 == 2 + 4          # rebuild of the resident B, then head, tail, build, condest
    assert all(b.info(k, "n_kind5") > 0 for k in (0, 2)) and all(b.info(k, "nfactorize") == 0 for k in (1, 3))
    factorize(b, lanes, [1, 3])
    replay(b, lanes, 4, 12550, dense_every=2)


@pytest.mark.parametrize("seed", [1, 2])
def test_emu_subset_random_lane_order(emu, seed, monkeypatch):
    monkeypatch.setenv("EMU_SEED", str(seed))
    b, lanes = start(emu, 5, 50, 12600 + 10 * seed)
    replay(b, lanes, 8, 12650 + seed, dense_every=4)


def assert_resident(b, lanes, run=None):
    """factorize_resident (or a graph replay) refactorizes every basis from the B it was last factorized from"""
    assert (run or b.factorize_resident)() == 0
    for k, L in enumerate(lanes):
        L.cols = list(L.factored)
        cp, ri, v = csc(L.cols)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == b.info(k, "status"), k
        L.pending = None; L.refactor = False
        sto, fo = L.oracle.get_factors()
        stg, fg = b.get_factors(k)
        assert sto == stg
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (k, key)
    assert_getters(b, lanes)


def test_emu_subset_resident_b_and_graph(emu):
    """After subset refactorizations the resident B of every basis is the B it was last factorized from, also after
    a maxvolume call; a graph captured before a subset factorization is refused afterwards until recaptured."""
    m = 40
    b, lanes = start(emu, 5, m, 12700)
    replay(b, lanes, 6, 12750, dense_every=0)
    factorize(b, lanes, [3])
    assert b.upload(rhs=np.ones(5 * m)) == 0
    assert b.graph_capture("N") == 0
    factorize(b, lanes, [0, 4])
    assert b.graph_launch() == -2
    assert_resident(b, lanes)
    assert b.graph_capture("N") == 0
    assert_resident(b, lanes, run=b.graph_launch)
    # after maxvolume (every basis' oracle runs maxvolume from where it is): B of every basis is its final columns
    # of the pool
    pools = [make_pool(12800 + k, m, 30, scale=3.0) for k in range(5)]
    ab, ae, ai, ax, basis, isbasic = mv_layout(pools)
    st, stat, nup = b.maxvolume(pools[0].ncol, ab, ae, ai, ax, basis, isbasic, 1.2)
    assert st == 0 and (nup > 0).all()
    basis = basis.reshape(5, m)
    for k, (L, p) in enumerate(zip(lanes, pools)):
        ob, oi = p.basis.copy(), p.isbasic.copy()
        assert L.oracle.maxvolume(p.ncol, p.a_p, p.a_i, p.a_x, ob, oi, 1.2) == (stat[k], nup[k])
        assert np.array_equal(ob, basis[k])
        L.cols = [(p.a_i[p.a_p[c]:p.a_p[c + 1]].copy(), p.a_x[p.a_p[c]:p.a_p[c + 1]].copy()) for c in basis[k]]
        L.factored = list(L.cols)
    assert_getters(b, lanes)
    factorize(b, lanes, [1, 2])
    assert_resident(b, lanes)
