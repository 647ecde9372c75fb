"""blu_batch_solve_sparse / blu_batch_solve_dense_multi under the SIMT emulator: every basis' results equal the
oracle running the same solves on that basis in order (nzlhs, the order of ilhs, values, unit statuses, and the
counters l_flops / u_flops / r_flops / update_cost afterwards)."""
import os
import subprocess

import numpy as np
import pytest

from blu_b200 import load_library
from bs_cases import (COUNTERS, assert_dense_parity, assert_sparse_parity, finish_update, make_batch, raw_solve_sparse,
                      rhs_lists, update_round)

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


@pytest.mark.parametrize("trans", ["N", "T"])
def test_emu_batch_solve_sparse_ragged(emu, trans):
    """Ragged unit counts (bases with none), empty right-hand sides, and right-hand sides from 1 to 60 entries at
    m = 120, so that both the depth-first and the sequential second triangle run (sparse_thres * m = 6)."""
    m = 120
    b, oracles = make_batch(emu, 5, m, 7100)
    lists = rhs_lists(m, 7200, [3, 0, 7, 1, 0], sizes=(1, 0, 2, 60, 5, 30, 1))
    assert_sparse_parity(b, oracles, lists, trans)
    # and again on the same objects: the pool's scratch is reused, marks and vectors start clean
    assert_sparse_parity(b, oracles, rhs_lists(m, 7300, [2, 4, 0, 3, 1]), trans)


def test_emu_batch_solve_sparse_thresholds(emu):
    """sparse_thres at both ends: every second triangle sequential (0.0), every one depth-first (1.0)"""
    m = 90
    for thres in (0.0, 1.0):
        b, oracles = make_batch(emu, 3, m, 7400)
        b.sparse_thres = thres
        for o in oracles:
            o.set_param("sparse_thres", thres)
        for tr in "NT":
            assert_sparse_parity(b, oracles, rhs_lists(m, 7500, [4, 2, 3]), tr)


def test_emu_batch_solve_sparse_singular_and_bad_unit(emu):
    """A singular basis (WarningSingularMatrix: its solves are still valid); one unit with an index >= m and one
    with more than m entries report ErrorInvalidArgument while the other units of their basis succeed."""
    m = 60
    b, oracles = make_batch(emu, 3, m, 7600, singular=(1,))
    assert oracles[1].info("rank") < m
    lists = rhs_lists(m, 7700, [3, 3, 3])
    lists[2][1] = (np.array([4, m, 7]), np.array([1.0, 2.0, 3.0]))
    lists[0][2] = (np.arange(m + 1) % m, np.ones(m + 1))
    for tr in "NT":
        st, out, ustat = assert_sparse_parity(b, oracles, lists, tr)
        assert st == -4 and list(ustat[2]) == [0, -4, 0] and list(ustat[0]) == [0, 0, -4]
        assert all(s == 0 for s in ustat[1])


def test_emu_batch_solve_never_factorized(emu):
    m = 40
    b, oracles = make_batch(emu, 3, m, 7800, factorize=False)
    lists = rhs_lists(m, 7900, [2, 1, 2])
    st, out, ustat = assert_sparse_parity(b, oracles, lists, "N")
    assert st == -2 and all((us == -2).all() for us in ustat)
    st, X, S = assert_dense_parity(b, oracles, 2, 7950, "N")
    assert st == -2 and (S == -2).all()


def test_emu_batch_solve_malformed(emu):
    """Malformed unit_begin / rhs_begin: ErrorInvalidArgument before anything runs, no getter moves"""
    m = 40
    b, oracles = make_batch(emu, 3, m, 8000)
    update_round(b, oracles, 8050, 0)      # a pending basis change: spike and row eta in place
    names = COUNTERS + ["pivotlen", "nupdate", "nforrest"]
    before = [[b.info(k, n) for n in names] for k in range(3)]
    launches = b.launch_count()
    ir, xr = np.array([1, 2, 3, 4]), np.ones(4)
    assert raw_solve_sparse(b, [1, 1, 2, 3], [0, 1, 2, 4], ir, xr) == -4         # unit_begin[0] != 0
    assert raw_solve_sparse(b, [0, 2, 1, 3], [0, 1, 2, 4], ir, xr) == -4         # decreasing
    assert raw_solve_sparse(b, [0, 1, 2, 3], [0, 5, 2, 4], ir, xr) == -4         # offset beyond rhs_begin[nunits]
    assert raw_solve_sparse(b, [0, 1, 2, 3], [-1, 1, 2, 4], ir, xr) == -4        # negative offset
    assert raw_solve_sparse(b, [0, 1, 2, 3], [0, 1, 2, -1], ir, xr) == -4        # negative total
    assert b._L.blu_batch_solve_dense_multi(b._h, -1, None, None, b"N", None) == -4
    assert b.launch_count() == launches
    assert [[b.info(k, n) for n in names] for k in range(3)] == before


@pytest.mark.parametrize("mem", [None, 450])
def test_emu_batch_solve_after_updates(emu, mem):
    """After several batch basis changes (row etas, permuted pivots, nforrest > 0); mem=450: tight stores, so
    that the bases run from private stores after the factorization and from grown ones later."""
    m = 90
    b, oracles = make_batch(emu, 3, m, 8100, mem=mem)
    if mem:
        assert b.info(0, "nrealloc") >= 1
        assert_sparse_parity(b, oracles, rhs_lists(m, 8150, [2, 3, 1]), "N")     # straight from the private stores
    for it in range(6):
        finish_update(b, oracles, update_round(b, oracles, 8200, it))
    assert all(b.info(k, "nforrest") > 0 for k in range(3))
    for tr in "NT":
        assert_sparse_parity(b, oracles, rhs_lists(m, 8300, [3, 2, 4], sizes=(1, 4, 30, 0, 2)), tr)
        assert_dense_parity(b, oracles, 3, 8350, tr)


def test_emu_batch_solve_between_solve_for_update_and_update(emu):
    """The solves leave the spike, the row eta and the pending flags alone: the update after them still matches"""
    m = 80
    b, oracles = make_batch(emu, 3, m, 8400)
    for it in range(3):
        xt = update_round(b, oracles, 8450, it)
        for tr in "NT":
            assert_sparse_parity(b, oracles, rhs_lists(m, 8500 + 10 * it, [2, 1, 3]), tr)
        assert_dense_parity(b, oracles, 2, 8550 + it, "T")
        finish_update(b, oracles, xt)
    assert_sparse_parity(b, oracles, rhs_lists(m, 8600, [2, 2, 2]), "N")


def test_emu_batch_solve_chunks(emu, monkeypatch):
    """BLU_B200_SOLVE_UNITS = 7: the units go through the pool in chunks of 7, a basis' units straddle chunks,
    the results are those of an unchunked run; one compaction launch plus one launch per chunk."""
    m = 70
    lists = rhs_lists(m, 8700, [5, 9, 0, 6])
    b1, o1 = make_batch(emu, 4, m, 8650)
    for it in range(2):
        finish_update(b1, o1, update_round(b1, o1, 8680, it))
    res1 = {tr: b1.solve_sparse(lists, tr) for tr in "NT"}
    monkeypatch.setenv("BLU_B200_SOLVE_UNITS", "7")
    b7, o7 = make_batch(emu, 4, m, 8650)
    for it in range(2):
        finish_update(b7, o7, update_round(b7, o7, 8680, it))
    for tr in "NT":
        l0 = b7.launch_count()
        res7 = assert_sparse_parity(b7, o7, lists, tr)
        assert b7.launch_count() - l0 == 1 + 3          # 20 units
        assert res7[0] == res1[tr][0]
        for k in range(4):
            assert np.array_equal(res7[2][k], res1[tr][2][k])
            for (a, x), (c, y) in zip(res7[1][k], res1[tr][1][k]):
                assert np.array_equal(a, c) and np.array_equal(x, y)
        l0 = b7.launch_count()
        assert_dense_parity(b7, o7, 4, 8750, tr)         # 16 units
        assert b7.launch_count() - l0 == 1 + 3
    for k in range(4):                                   # both sides have run the 'N' and the 'T' solves
        for name in COUNTERS:
            assert b7.info(k, name) == b1.info(k, name)


@pytest.mark.parametrize("seed", [1, 2])
def test_emu_batch_solve_random_lane_order(emu, seed, monkeypatch):
    monkeypatch.setenv("EMU_SEED", str(seed))
    m = 75
    b, oracles = make_batch(emu, 3, m, 8800 + seed)
    finish_update(b, oracles, update_round(b, oracles, 8850, 0))
    for tr in "NT":
        assert_sparse_parity(b, oracles, rhs_lists(m, 8900 + seed, [3, 1, 4]), tr)
        assert_dense_parity(b, oracles, 2, 8950 + seed, tr)


@pytest.mark.parametrize("trans", ["N", "T"])
def test_emu_batch_solve_dense_multi(emu, trans):
    m = 80
    b, oracles = make_batch(emu, 4, m, 9000, singular=(2,))
    assert_dense_parity(b, oracles, 3, 9050, trans)
    b, oracles = make_batch(emu, 3, m, 9060)
    for it in range(4):
        finish_update(b, oracles, update_round(b, oracles, 9100, it))
    assert_dense_parity(b, oracles, 3, 9150, trans)
    st, X, S = b.solve_dense_multi(np.zeros((3, 0, m)), trans)
    assert st == 0 and X.shape == (3, 0, m)
