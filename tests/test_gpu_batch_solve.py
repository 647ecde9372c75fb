"""blu_batch_solve_sparse / blu_batch_solve_dense_multi on the GPU: bit-identical to the oracle running the same
solves on each basis in order, at configs[1]'s size."""
import numpy as np
import pytest

from bs_cases import (COUNTERS, assert_dense_parity, assert_sparse_parity, finish_update, make_batch, rhs_lists,
                      update_round)

pytestmark = pytest.mark.gpu

M = 2000


def config1_batch(nmat, seed0, sample=None):
    """configs[1]-shaped bases: 2,000 rows, 35 % slack, 1 + Poisson(5) entries per column"""
    return make_batch(None, nmat, M, seed0, nslack=700, pmean=5.0, sample=sample)


def test_gpu_batch_solve_256x16():
    """256 bases with 16 right-hand sides each, 'N' and 'T', before and after batch basis changes; then the
    existing batch calls on the same object still agree with the oracle."""
    b, oracles = config1_batch(256, 30000)
    sizes = (20, 1, 3, 60, 20, 0, 200, 20)
    for tr in "NT":
        assert_sparse_parity(b, oracles, rhs_lists(M, 31000, [16] * 256, sizes=sizes), tr)
    assert_dense_parity(b, oracles, 4, 31500, "N")
    for it in range(3):
        finish_update(b, oracles, update_round(b, oracles, 32000, it))
    xt = update_round(b, oracles, 32000, 3)
    for tr in "NT":      # between solve_for_update and update
        assert_sparse_parity(b, oracles, rhs_lists(M, 33000, [16] * 256, sizes=sizes), tr)
        assert_dense_parity(b, oracles, 2, 33500, tr)
    finish_update(b, oracles, xt)
    rhs = np.random.default_rng(34000).uniform(-1.0, 1.0, (256, M))
    for tr in "NT":
        st, x, status = b.solve_dense(rhs, tr)
        assert st == 0 and (status == 0).all()
        for k, o in enumerate(oracles):
            assert np.array_equal(x[k], o.solve_dense(rhs[k], tr)[1]), (k, tr)


def test_gpu_batch_solve_4096_sample():
    sample = list(range(0, 4096, 257)) + [4095]
    b, oracles = config1_batch(4096, 40000, sample=sample)
    counts = [(k * 7) % 5 for k in range(4096)]
    lists = rhs_lists(M, 41000, counts, sizes=(20, 5, 40, 1))
    for tr in "NT":
        assert_sparse_parity(b, oracles, lists, tr, sample=sample)
    R = np.random.default_rng(42000).uniform(-1.0, 1.0, (4096, 2, M))
    st, X, S = b.solve_dense_multi(R, "T")
    assert st == 0 and (S == 0).all()
    for k in sample:
        for r in range(2):
            assert np.array_equal(X[k, r], oracles[k].solve_dense(R[k, r], "T")[1]), (k, r)


def test_gpu_batch_solve_chunks(monkeypatch):
    """BLU_B200_SOLVE_UNITS = 1000: 4,096 units in five chunks; identical to one chunk, one compaction launch
    plus one launch per chunk"""
    lists = rhs_lists(M, 51000, [16] * 256, sizes=(20, 2, 60))
    b1, o1 = config1_batch(256, 50000, sample=[])
    res = {tr: b1.solve_sparse(lists, tr) for tr in "NT"}
    R = np.random.default_rng(52000).uniform(-1.0, 1.0, (256, 16, M))
    X1 = b1.solve_dense_multi(R, "N")
    monkeypatch.setenv("BLU_B200_SOLVE_UNITS", "1000")
    b, oracles = config1_batch(256, 50000, sample=[0, 77, 255])
    for tr in "NT":
        l0 = b.launch_count()
        r = assert_sparse_parity(b, oracles, lists, tr, sample=[0, 77, 255])
        assert b.launch_count() - l0 == 1 + 5
        assert r[0] == res[tr][0]
        for k in range(256):
            assert np.array_equal(r[2][k], res[tr][2][k])
            for (a, x), (c, y) in zip(r[1][k], res[tr][1][k]):
                assert np.array_equal(a, c) and np.array_equal(x, y), (k, tr)
    for k in range(256):
        for name in COUNTERS:
            assert b.info(k, name) == b1.info(k, name), (k, name)
    l0 = b.launch_count()
    X = b.solve_dense_multi(R, "N")
    assert b.launch_count() - l0 == 1 + 5
    assert X[0] == X1[0] and np.array_equal(X[1], X1[1]) and np.array_equal(X[2], X1[2])
