"""blu_batch_copy / blu_batch_copy_dev under the SIMT emulator: a destination shows exactly what its source shows right
after the copy, then goes on as an oracle object that went through the source's history -- on its own schedule, with
its own entering columns -- while sources and every other basis do not move."""
import os
import subprocess

import numpy as np
import pytest
import torch

from blu_b200 import BLUBatch, load_library
from copy_cases import CLane, CopyTwin, assert_copies, fork, fork_and_check, snapshot
from subset_cases import assert_dense, assert_getters, assert_same_snapshot, csc, factorize, replay, solve_n, solve_t, update

HERE = os.path.dirname(os.path.abspath(__file__))
CPU = torch.device("cpu")


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


def lanes_for(nmat, m, seed0):
    """alternately sparse (many slack columns) and dense bases, so that with small stores only some grow private ones"""
    return [CLane(seed0 + k, m, nslack=m - 4 if k % 2 else 0, pmean=3.0 if k % 2 else 6.0, policy=k % 2) for k in range(nmat)]


def refactorize_resident(b, lanes, call=True):
    """blu_batch_factorize_resident (call=False: a graph launch that did it): every basis from the B it was last
    factorized from, the oracles alongside"""
    if call:
        assert b.factorize_resident() == 0
    for L in lanes:
        cp, ri, v = csc(L.factored)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.cols = list(L.factored)
        L.pending, L.refactor = None, False
    assert_getters(b, lanes)


def dirty(b, lanes, ks, rounds):
    """full basis changes on the bases ks only, so that they carry a longer history (more etas, more updates)"""
    for _ in range(rounds):
        pend = solve_n(b, lanes, ks)
        solve_t(b, lanes, pend, want=1)
        ok = [k for k in ks if lanes[k].pending is not None]
        if ok:
            update(b, lanes, ok)
        redo = [k for k in ks if lanes[k].refactor]
        if redo:
            factorize(b, lanes, redo)


@pytest.mark.parametrize("point,small", [("factorized", True), ("updated", True), ("pending_n", True), ("pending_nt", True),
                                         ("never_factorized", True), ("pending_nt", False)],
                         ids=["factorized", "updated", "pending_n", "pending_nt", "never_factorized", "pending_nt-uniform"])
def test_emu_copy_overwrites_dirty_slots(emu, point, small):
    """Destinations first carry a different and longer history than their sources, with private stores forced by
    small l_mem / u_mem / w_mem (small) or in the uniform stores; the copy at each fork point makes them show exactly
    their sources' state, and every lane then matches its oracle through 12 rounds of its own schedule."""
    nmat, m = 8, 16
    lanes = lanes_for(nmat, m, 31000)
    b = new_batch(emu, lanes, mem=3 * m if small else None)
    src, dst = [0, 1, 2], [5, 6, 4]
    if point == "never_factorized":
        factorize(b, lanes, [k for k in range(nmat) if k not in src])
    else:
        factorize(b, lanes, list(range(nmat)))
    assert (b.info(0, "nrealloc") > 0) == small
    dirty(b, lanes, dst, 6)
    if point == "updated":
        dirty(b, lanes, src, 2)
    elif point in ("pending_n", "pending_nt"):
        pend = solve_n(b, lanes, src)
        if point == "pending_nt":
            solve_t(b, lanes, pend, want=0)
    fork_and_check(b, lanes, dst, src, seed=7)
    if point == "never_factorized":
        for d in dst:
            assert b.info(d, "nupdate") == -1      # None
        factorize(b, lanes, src + dst)
    if point == "pending_nt":
        ks = src + dst
        assert update(b, lanes, ks)[0] == 0
    replay(b, lanes, 12, 31100)
    assert_dense(b, lanes, 31200)


def test_emu_copy_pending_n_then_t(emu):
    """A copy taken between 'N' and 'T' finishes the pair on its own: 'T' and update on source and copy match the
    oracles."""
    nmat, m = 6, 20
    lanes = lanes_for(nmat, m, 32000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, [3, 4], 3)
    cols = {0: lanes[0].next_column()}
    st, stat, out = b.solve_for_update_subset([0], [cols[0]], "N", want_solution=1)
    o = lanes[0].oracle
    assert o.solve_for_update(len(cols[0][0]), cols[0][0], cols[0][1], "N", want_solution=1) == stat[0] == 0
    j = int(np.argmax(np.abs(o.lhs)))
    pend = (j, o.lhs[j], cols[0])
    fork_and_check(b, lanes, [3, 4], [0, 0], seed=3)
    solve_t(b, lanes, {k: pend for k in (0, 3, 4)}, want=1)
    assert update(b, lanes, [0, 3, 4])[0] == 0
    replay(b, lanes, 8, 32100)


def test_emu_copy_capacities_both_ways(emu):
    """private to uniform, uniform to private, private to a private store of another size, and a fan-out of one
    source to every other basis; every lane then goes on against its oracle."""
    nmat, m = 8, 16
    lanes = lanes_for(nmat, m, 33000)
    b = new_batch(emu, lanes, mem=3 * m)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, list(range(nmat)), 3)
    # dense (even) bases grew private stores, sparse (odd) ones may not have: copy across both kinds
    fork_and_check(b, lanes, [1, 2], [0, 3], seed=11)
    replay(b, lanes, 6, 33100)
    fork_and_check(b, lanes, [4, 6], [2, 0], seed=12)
    replay(b, lanes, 6, 33200)
    fork_and_check(b, lanes, [k for k in range(nmat) if k != 5], [5] * (nmat - 1), seed=13)
    replay(b, lanes, 10, 33300)
    assert_dense(b, lanes, 33400)


def test_emu_copy_untouched(emu):
    """Sources and the bases not named as destinations keep their snapshot bit for bit, one of them with a pending
    solve_for_update pair."""
    nmat, m = 7, 24
    lanes = lanes_for(nmat, m, 34000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, [0, 1, 2], 2)
    solve_t(b, lanes, solve_n(b, lanes, [6]), want=1)          # basis 6: pending pair
    keep = [0, 1, 3, 6]
    before = snapshot(b, keep, seed=5, lanes=lanes)
    fork(b, lanes, [2, 4, 5], [0, 1, 0])
    assert_same_snapshot(before, snapshot(b, keep, seed=5, lanes=lanes))
    assert update(b, lanes, [6])[0] == 0
    replay(b, lanes, 6, 34100)


def test_emu_copy_resident_b(emu):
    """After a copy, factorize_resident refactorizes the destination from its source's B, also when B was caller-owned
    (factorize_dev); a later factorize_subset of other bases keeps that B; a graph captured before is refused."""
    nmat, m = 6, 20
    lanes = lanes_for(nmat, m, 35000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, list(range(nmat)), 2)
    assert b.graph_capture("N") == 0
    fork(b, lanes, [3, 4], [0, 1])
    assert b.graph_launch() == -2
    refactorize_resident(b, lanes)
    dirty(b, lanes, [0, 1, 2], 2)
    fork(b, lanes, [5], [2])
    factorize(b, lanes, [0, 1])                     # other bases: the resident B keeps basis 5's
    refactorize_resident(b, lanes)
    assert b.graph_capture("N") == 0 and b.graph_launch() == 0
    refactorize_resident(b, lanes, call=False)
    # caller-owned B
    bb = np.zeros(nmat * m, np.int64); be = np.zeros(nmat * m, np.int64); bi, bx, off = [], [], 0
    for k, L in enumerate(lanes):
        for j, (ri, v) in enumerate(L.cols):
            bb[k * m + j] = off; be[k * m + j] = off + len(ri); bi.append(np.asarray(ri, np.int64)); bx.append(np.asarray(v)); off += len(ri)
    bi, bx = np.concatenate(bi), np.concatenate(bx)
    assert b.factorize_dev(bb.ctypes.data, be.ctypes.data, bi.ctypes.data, bx.ctypes.data, len(bi)) == 0
    for L in lanes:
        cp, ri, v = csc(L.cols)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.factored = list(L.cols); L.pending = None; L.refactor = False
    assert_getters(b, lanes)
    dirty(b, lanes, [2], 2)
    bb0, be0 = bb.copy(), be.copy()
    fork(b, lanes, [0, 1], [2, 2])
    fork(b, lanes, [5], [4])                        # a second copy on the moved column pointers
    assert np.array_equal(bb, bb0) and np.array_equal(be, be0)      # the caller's B is read, never written
    refactorize_resident(b, lanes)
    assert_dense(b, lanes, 35100)


def test_emu_copy_resident_b_after_maxvolume(emu):
    """After maxvolume the resident B of every basis is its final basis; a copy takes the source's, and
    factorize_resident refactorizes each destination from its source's final columns, as the oracle does."""
    from mv_cases import make_pool, run_batch
    from oracle_lib import Oracle
    m = 40
    pools = [make_pool(36500 + k, m, 60, scale=3.0) for k in range(4)]
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), lib=emu)
    b.threads_per_basis = 64
    res = run_batch(b, pools, 1.2)
    assert res[0] == 0 and (res[2] > 0).all()
    dst, src = [2, 3], [0, 0]
    assert b.copy(dst, src) == 0
    assert b.factorize_resident() == 0
    owner = {0: 0, 1: 1, 2: 0, 3: 0}
    for k in range(len(pools)):
        p, bas = pools[owner[k]], res[3][owner[k]]
        o = Oracle(m, 60 * len(p.a_i))
        assert o.factorize(p.a_p[bas], p.a_p[bas + 1], p.a_i, p.a_x) == 0
        sto, fo = o.get_factors()
        stg, fg = b.get_factors(k)
        assert sto == stg == 0
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (k, key)


def test_emu_copy_argument_errors(emu):
    """Each rejected case returns BLU_ERROR_INVALID_ARGUMENT and changes nothing; ncopy == 0 returns BLU_OK."""
    nmat, m = 5, 16
    lanes = lanes_for(nmat, m, 36000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, [0, 1], 2)
    before = snapshot(b, range(nmat), seed=2, lanes=lanes)
    L, h = b._L, b._h
    from subset_cases import _pi
    cases = [([1], [5]), ([-1], [0]), ([2], [-3]), ([2, 2], [0, 1]), ([3], [3]), ([2, 3], [0, 2]), ([0, 1], [2, 0])]
    for dst, src in cases:
        assert b.copy(dst, src) == -4, (dst, src)
    d, s = np.array([1, 2], np.int64), np.array([0, 0], np.int64)
    assert L.blu_batch_copy(h, -1, _pi(d), _pi(s)) == -4
    assert L.blu_batch_copy(h, nmat + 1, _pi(np.arange(nmat + 1)), _pi(np.zeros(nmat + 1, np.int64))) == -4
    assert L.blu_batch_copy(h, 2, None, _pi(s)) == -4 and L.blu_batch_copy(h, 2, _pi(d), None) == -4
    assert L.blu_batch_copy(h, 0, None, None) == 0 and b.copy([], []) == 0
    assert_same_snapshot(before, snapshot(b, range(nmat), seed=2, lanes=lanes))
    from blu_b200 import BLU
    g = BLU(m, 64, lib=emu)
    assert L.blu_batch_copy(g._h, 1, _pi(np.array([0])), _pi(np.array([0]))) == -4
    g.close()


def test_emu_copy_dev_twins(emu):
    """copy_dev leaves its batch bit-identical to copy's; an invalid map (out of range, self, chain, another negative
    value) returns BLU_ERROR_INVALID_ARGUMENT and changes nothing."""
    nmat, m = 6, 20
    lanes = lanes_for(nmat, m, 37000)

    def make():
        return new_batch(emu, lanes)
    tw = CopyTwin(make, CPU)
    factorize(tw, lanes, list(range(nmat)))
    dirty(tw, lanes, [0, 1, 4], 2)
    before = snapshot(tw, range(nmat), seed=4, lanes=lanes)
    for bad in ([-1, -1, 6, -1, -1, -1], [-1, 1, -1, -1, -1, -1], [-1, 0, 1, -1, -1, -1], [-1, -1, -2, -1, -1, -1]):
        assert tw.d.copy_dev(torch.as_tensor(np.array(bad, np.int32))) == -4
    assert tw.d.copy_dev(torch.full((nmat,), -1, dtype=torch.int32)) == 0
    assert_same_snapshot(before, snapshot(tw, range(nmat), seed=4, lanes=lanes))
    fork(tw, lanes, [2, 3, 5], [0, 0, 4])
    assert_copies(snapshot(tw, range(nmat), seed=6, lanes=lanes), [2, 3, 5], [0, 0, 4])
    replay(tw, lanes, 8, 37100)


@pytest.mark.parametrize("env,case", [("EMU_SEED=1", "test_emu_copy_overwrites_dirty_slots[pending_nt]"),
                                      ("EMU_STRICT=1", "test_emu_copy_overwrites_dirty_slots[pending_nt-uniform]")])
def test_emu_copy_env(env, case):
    """the dirty-slot case at the 'N' + 'T' fork point under a shuffled lane order, and under the strict barrier check.
    The strict run keeps the uniform stores: with stores forced small, the factorization kernel's Reallocate path
    (k_factorize, phase_setup_bump), which this change does not touch, trips the strict check on its own."""
    k, v = env.split("=")
    r = subprocess.run([os.sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider",
                        os.path.abspath(__file__) + "::" + case],
                       env=dict(os.environ, **{k: v}), cwd=HERE, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
