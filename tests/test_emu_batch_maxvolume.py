"""blu_batch_maxvolume under the SIMT emulator: every basis of the batch ends exactly as the oracle's maxvolume
leaves it when run alone on the same pool (maxvolume.rs:64-224)."""
import os
import subprocess

import numpy as np
import pytest

from blu_b200 import BLUBatch, load_library
from mv_cases import layout, make_pool, replace_column, run_batch, assert_parity, oracle_maxvolume, refactor_triggers

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


def new_batch(emu, pools, tight=False):
    m = pools[0].m
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), lib=emu)
    b.threads_per_basis = 64
    if tight:
        nnz = max(len(p.a_i) for p in pools) // 4
        b.l_mem = nnz; b.u_mem = nnz; b.w_mem = nnz
    return b


def mixed_pools(m, seed0):
    """one basis singular from the start, one whose candidate column 12 has a row index >= m, ordinary ones"""
    pools = [make_pool(seed0 + k, m, 60, scale=3.0) for k in range(5)]
    p = pools[0]
    p.basis[1] = p.basis[0]                      # the same column twice: WarningSingularMatrix, nupdate 0
    p.isbasic[1] = 0
    q = pools[1]
    pools[1] = replace_column(q, m + 12, [2, m, 5], [3.0, 1.0, -2.0])
    return pools


def test_emu_maxvolume_mixed_outcomes(emu):
    m = 60
    pools = mixed_pools(m, 4100)
    b = new_batch(emu, pools)
    res = run_batch(b, pools, 1.5)
    ores = assert_parity(b, pools, 1.5, res, rhs_seed=4200)
    status, nup = res[1], res[2]
    assert status[0] == 2 and nup[0] == 0
    assert status[1] == -4 and 0 < nup[1]
    assert all(s == 0 for s in status[2:]) and all(n > 0 for n in nup[2:])
    assert ores[1][1] == -4


@pytest.mark.parametrize("seed", [1, 2])
def test_emu_maxvolume_random_lane_order(emu, seed, monkeypatch):
    monkeypatch.setenv("EMU_SEED", str(seed))
    pools = mixed_pools(44, 4300 + 10 * seed)
    b = new_batch(emu, pools)
    assert_parity(b, pools, 1.5, run_batch(b, pools, 1.5), rhs_seed=4400)


def test_emu_maxvolume_refactorizes(emu):
    """Small m and many entering columns: nforrest == m and update_cost > 1 both trigger refactorizations
    inside the pass, not on every basis alike."""
    m = 40
    pools = [make_pool(seed, m, 120, scale=3.0) for seed in (101, 102, 103, 104)]
    b = new_batch(emu, pools)
    assert_parity(b, pools, 1.0, run_batch(b, pools, 1.0), rhs_seed=4500)
    nf = [b.info(k, "nfactorize") for k in range(len(pools))]
    assert len(set(nf)) > 1 and max(nf) >= 3, nf


def test_emu_maxvolume_refactor_triggers(emu):
    """Both conditions of maxvolume.rs:161-170 that the pass can meet start refactorizations here: update_cost > 1
    first, nforrest == m later (the restatement of the loop on the oracle says which held)."""
    m = 30
    pools = [make_pool(seed, m, 150, nslack=25, scale=5.0) for seed in (101, 102, 103)]
    seen = set()
    for p in pools:
        for why in refactor_triggers(p, 1.0)[4]:
            seen |= why
    assert {"nforrest", "update_cost"} <= seen, seen
    b = new_batch(emu, pools)
    assert_parity(b, pools, 1.0, run_batch(b, pools, 1.0), rhs_seed=4550)
    assert all(b.info(k, "nfactorize") >= 3 for k in range(len(pools)))


def test_emu_maxvolume_all_bases_stop(emu):
    """Every basis stops: the call still ends, at the first factorization or partway through the pass."""
    m = 40
    pools = [make_pool(5600 + k, m, 30, scale=3.0) for k in range(2)]
    for p in pools:
        p.basis[1] = p.basis[0]; p.isbasic[1] = 0
    b = new_batch(emu, pools)
    res = run_batch(b, pools, 1.5)
    assert_parity(b, pools, 1.5, res, rhs_seed=5650)
    assert (res[1] == 2).all() and (res[2] == 0).all()
    pools = [replace_column(make_pool(5700 + k, m, 30, scale=3.0), m + 5 + 7 * k, [1, m + k], [2.0, 1.0]) for k in range(2)]
    b = new_batch(emu, pools)
    res = run_batch(b, pools, 1.5)
    assert_parity(b, pools, 1.5, res, rhs_seed=5750)
    assert (res[1] == -4).all()


def test_emu_maxvolume_resident_b(emu):
    """Afterwards the resident B of every basis is its final basis: refactorizing it gives the factors the
    oracle gets from those columns."""
    m = 40
    pools = [make_pool(5800 + k, m, 60, scale=3.0) for k in range(3)]
    b = new_batch(emu, pools)
    res = run_batch(b, pools, 1.2)
    assert res[0] == 0 and (res[2] > 0).all()
    assert b.factorize_resident() == 0
    from oracle_lib import Oracle
    for k, p in enumerate(pools):
        o = Oracle(m, 60 * len(p.a_i))
        bas = res[3][k]
        assert o.factorize(p.a_p[bas], p.a_p[bas + 1], p.a_i, p.a_x) == 0
        sto, fo = o.get_factors()
        stg, fg = b.get_factors(k)
        assert sto == stg == 0
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (k, key)


def test_emu_maxvolume_tight_stores(emu):
    """Stores far below what the pass needs: the sparse calls and the refactorizations reallocate, the
    results do not change."""
    m = 50
    pools = [make_pool(4600 + k, m, 70, scale=3.0) for k in range(3)]
    b = new_batch(emu, pools, tight=True)
    nr0 = b.info(0, "nrealloc")
    assert_parity(b, pools, 1.2, run_batch(b, pools, 1.2), rhs_seed=4700)
    assert b.info(0, "nrealloc") > nr0


def test_emu_maxvolume_ties(emu):
    """Identity basis, a candidate with equal magnitudes of both signs: the first entry in ilhs order leaves."""
    m = 40
    pools = []
    for k in range(3):
        p = make_pool(4800 + k, m, 10, identity=True, scale=0.1)
        rows = [3 + k, 17, 9, 30 - k]
        pools.append(replace_column(p, m + 2, rows, [-2.5, 2.5, 2.5, -2.5]))
    b = new_batch(emu, pools)
    res = run_batch(b, pools, 1.0)
    assert_parity(b, pools, 1.0, res, rhs_seed=4900)
    assert all(n >= 1 for n in res[2])
    assert all((res[3][k] == m + 2).sum() == 1 for k in range(3))


def test_emu_maxvolume_edges(emu):
    m = 45
    # ncol == m: nothing to examine, only the first factorization
    pools = [make_pool(5000 + k, m, 0) for k in range(3)]
    b = new_batch(emu, pools)
    res = run_batch(b, pools, 1.5)
    assert_parity(b, pools, 1.5, res, rhs_seed=5100)
    assert res[0] == 0 and (res[2] == 0).all()
    # empty pool columns among the candidates
    pools = [make_pool(5200 + k, m, 20, scale=3.0) for k in range(3)]
    pools = [replace_column(replace_column(p, m + 1, [], []), m + 7, [], []) for p in pools]
    b = new_batch(emu, pools)
    assert_parity(b, pools, 1.5, run_batch(b, pools, 1.5), rhs_seed=5300)
    # volumetol < 1: ErrorInvalidArgument for the call, nothing runs
    b = new_batch(emu, pools)
    st, status, nup, basis, isbasic = run_batch(b, pools, 0.5)
    assert st == -4 and (status == -4).all() and (nup == 0).all()
    assert all(b.info(k, "nfactorize") == 0 for k in range(3))
    assert all(oracle_maxvolume(p, 0.5)[1] == -4 for p in pools)
    assert np.array_equal(basis[0], pools[0].basis)


def test_emu_maxvolume_malformed(emu):
    m = 40
    pools = [make_pool(5400 + k, m, 10) for k in range(3)]
    b = new_batch(emu, pools)
    ab, ae, ai, ax, basis, isbasic = layout(pools)
    ncol = pools[0].ncol
    bad = basis.copy(); bad[5] = ncol
    assert b.maxvolume(ncol, ab, ae, ai, ax, bad, isbasic.copy(), 1.5)[0] == -4
    bad = ae.copy(); bad[3] = len(ai) + 1
    assert b.maxvolume(ncol, ab, bad, ai, ax, basis.copy(), isbasic.copy(), 1.5)[0] == -4
    assert all(b.info(k, "nfactorize") == 0 for k in range(3))


def test_emu_maxvolume_launch_count(emu):
    """The launches grow with the number of columns, not with the number of bases."""
    m = 40
    p = make_pool(5500, m, 50, scale=3.0)
    deltas = []
    for nmat in (3, 8):
        pools = [p] * nmat
        b = new_batch(emu, pools)
        l0 = b.launch_count()
        res = run_batch(b, pools, 1.2)
        assert res[0] == 0
        nfact = int(b.info(0, "nfactorize"))
        deltas.append(b.launch_count() - l0)
    assert deltas[0] == deltas[1], deltas
    assert deltas[0] <= 8 * p.ncol + 8 * nfact, (deltas, nfact)
