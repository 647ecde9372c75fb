"""blu_batch_maxvolume on the GPU: every basis ends exactly as the oracle's maxvolume leaves it when run alone on
the same pool (maxvolume.rs:64-224)."""
import numpy as np
import pytest

from blu_b200 import BLUBatch
from mv_cases import GETTERS, config1_pools, make_pool, replace_column, run_batch, assert_parity, oracle_maxvolume, refactor_triggers

pytestmark = pytest.mark.gpu


def new_batch(pools, tight=False):
    m = pools[0].m
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), device=0)
    if tight:
        nnz = max(len(p.a_i) for p in pools) // 4
        b.l_mem = nnz; b.u_mem = nnz; b.w_mem = nnz
    return b


def test_gpu_maxvolume_mixed_outcomes():
    m, nmat = 300, 64
    pools = [make_pool(6000 + k, m, 150, scale=3.0) for k in range(nmat)]
    p = pools[0]
    p.basis[1] = p.basis[0]; p.isbasic[1] = 0                        # singular from the start
    pools[1] = replace_column(pools[1], m + 40, [7, m + 3, 11], [2.0, 1.0, -3.0])   # row index >= m
    b = new_batch(pools)
    res = run_batch(b, pools, 1.5)
    assert_parity(b, pools, 1.5, res, rhs_seed=6100)
    status, nup = res[1], res[2]
    assert status[0] == 2 and nup[0] == 0
    assert status[1] == -4 and nup[1] > 0
    assert (status[2:] == 0).all() and (nup[2:] > 0).all()


def test_gpu_maxvolume_refactorizes():
    m, nmat = 300, 64
    pools = [make_pool(6200 + k, m, 400, scale=3.0) for k in range(nmat)]
    b = new_batch(pools)
    assert_parity(b, pools, 1.0, run_batch(b, pools, 1.0), rhs_seed=6300)
    nf = [b.info(k, "nfactorize") for k in range(nmat)]
    assert max(nf) >= 2, nf


def test_gpu_maxvolume_tight_stores():
    m, nmat = 300, 64
    pools = [make_pool(6400 + k, m, 150, scale=3.0) for k in range(nmat)]
    b = new_batch(pools, tight=True)
    nr0 = b.info(0, "nrealloc")
    assert_parity(b, pools, 1.2, run_batch(b, pools, 1.2), rhs_seed=6500)
    assert b.info(0, "nrealloc") > nr0


def test_gpu_maxvolume_config1_batch():
    nmat = 256
    pools = config1_pools(nmat, 500, 9000)
    b = new_batch(pools)
    st, status, nup, basis, isbasic = run_batch(b, pools, 2.0)
    assert st == 0 and (status == 0).all() and (nup > 0).all(), (st, status, nup)
    sample = np.random.default_rng(7).choice(nmat, 16, replace=False)
    for k in sample:
        o, ost, onup, obasis, oisbasic = oracle_maxvolume(pools[k], 2.0)
        assert ost == 0 and nup[k] == onup, (k, nup[k], onup)
        assert np.array_equal(basis[k], obasis) and np.array_equal(isbasic[k], oisbasic), k
        for name in GETTERS:
            assert b.info(k, name) == o.info(name), (k, name)


def test_gpu_maxvolume_ties_and_edges():
    m, nmat = 300, 64
    # identity bases, a candidate with equal magnitudes of both signs: the first entry in ilhs order leaves
    pools = [replace_column(make_pool(6600 + k, m, 10, identity=True, scale=0.1), m + 2, [3 + k, 170, 90, 290 - k],
                            [-2.5, 2.5, 2.5, -2.5]) for k in range(nmat)]
    b = new_batch(pools)
    res = run_batch(b, pools, 1.0)
    assert_parity(b, pools, 1.0, res, rhs_seed=6700)
    assert all((res[3][k] == m + 2).sum() == 1 for k in range(nmat))
    # ncol == m
    pools = [make_pool(6800 + k, m, 0) for k in range(nmat)]
    b = new_batch(pools)
    res = run_batch(b, pools, 1.5)
    assert_parity(b, pools, 1.5, res, rhs_seed=6900)
    assert res[0] == 0 and (res[2] == 0).all()
    # empty candidate columns
    pools = [replace_column(replace_column(make_pool(7000 + k, m, 40, scale=3.0), m + 1, [], []), m + 9, [], [])
             for k in range(nmat)]
    b = new_batch(pools)
    assert_parity(b, pools, 1.5, run_batch(b, pools, 1.5), rhs_seed=7100)
    # volumetol < 1: nothing runs
    b = new_batch(pools)
    st, status, nup, _, _ = run_batch(b, pools, 0.5)
    assert st == -4 and (status == -4).all() and (nup == 0).all()
    assert all(b.info(k, "nfactorize") == 0 for k in range(nmat))


def test_gpu_maxvolume_all_bases_stop_and_triggers():
    # every basis singular from the start: the call ends
    m, nmat = 300, 64
    pools = [make_pool(7200 + k, m, 20, scale=3.0) for k in range(nmat)]
    for p in pools:
        p.basis[1] = p.basis[0]; p.isbasic[1] = 0
    b = new_batch(pools)
    res = run_batch(b, pools, 1.5)
    assert_parity(b, pools, 1.5, res, rhs_seed=7300)
    assert (res[1] == 2).all()
    # both refactorization conditions the pass meets (update_cost > 1, then nforrest == m)
    m = 30
    pools = [make_pool(7400 + k, m, 150, nslack=25, scale=5.0) for k in range(nmat)]
    seen = set()
    for p in pools[:4]:
        for why in refactor_triggers(p, 1.0)[4]:
            seen |= why
    assert {"nforrest", "update_cost"} <= seen, seen
    b = new_batch(pools)
    assert_parity(b, pools, 1.0, run_batch(b, pools, 1.0), rhs_seed=7500)
