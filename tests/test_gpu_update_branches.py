"""The explicit-basis checks of tests/update_cases.py on the B200: single bases up to m = 2,000 bit-identical to the oracle
with their own solves checked against the explicit B', and 256 configs[1]-shaped bases (gen.basis(seed, 2000, 700,
5.0)) through masked update_dev rounds, every basis checked against its explicit B' after every round."""
import time

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from blu_b200 import BLU, BLUBatch, gen
from oracle_lib import Oracle
from subset_cases import layout
from mv_cases import config1_pools, run_batch
from update_cases import Cols, Stats, batch_rounds, check_maxvolume, single_case

pytestmark = pytest.mark.gpu


def gpu_objs(m, nnz, t):
    o = Oracle(m, (400 if m <= 200 else 40) * nnz + 2000)
    g = BLU(m, nnz, device=0)
    for k, x in t.items():
        o.set_param(k, x)
        setattr(g, k, x)
    return [o, g]


def test_gpu_blu_update_branches():
    """Twelve small structured cases (20 steps each) and two gen.basis cases at m = 1,000 and 2,000 (10 steps each)."""
    t0 = time.time()
    stats = Stats()
    for seed in range(12):
        single_case(seed, gpu_objs, nsteps=20, stats=stats)
    for seed, m in ((7001, 1000), (7002, 2000)):
        cp, ri, v = gen.basis(seed, m, 700 * m // 2000, 5.0)
        B = sp.csc_matrix((v, ri, cp), shape=(m, m)).toarray()
        single_case(seed, gpu_objs, nsteps=10, stats=stats, case=(m, 6, B, {}, np.random.default_rng(seed)))
    print(stats, f"{time.time() - t0:.1f} s")
    for b in ("ft", "sym", "unsym", "refused"):
        assert stats.count[b] > 0, str(stats)


def test_gpu_batch_update_dev_every_basis():
    """256 configs[1]-shaped bases, 10 rounds of update_dev with a run mask: every basis against its oracle and its
    explicit basis (B'x accumulated in long double on the host) after every round."""
    t0 = time.time()
    n, m = 256, 2000
    bases = [Cols(*gen.basis(40000 + k, m, 700, 5.0)) for k in range(n)]
    nnz = max(len(c.csc()[1]) for c in bases)
    b = BLUBatch(n, m, nnz + 8 * m, device=0)
    oracles = [Oracle(m, 20 * nnz + 8 * m) for _ in range(n)]
    st, stat = b.factorize_subset(list(range(n)), *layout([c.cols for c in bases]))
    assert st == 0 and (stat == 0).all()
    for o, c in zip(oracles, bases):
        cp, ri, v = c.csc()
        assert o.factorize(cp[:-1], cp[1:], ri, v) == 0
    dev = torch.device("cuda", 0)
    stats = batch_rounds(b, oracles, bases, {}, 10, 40000, update_dev=lambda a, dt: torch.as_tensor(a, dtype=dt).to(dev),
                         dev_only=True, construct_rate=0.5)
    print(stats, f"{time.time() - t0:.1f} s")
    for k in ("ft", "sym", "unsym", "refused"):
        assert stats.count[k] > 0, str(stats)
    b.close()


def test_gpu_maxvolume_against_explicit_basis():
    """Batch maxvolume on 64 configs[1]-shaped bases with 200 candidates each: B rebuilt from the returned basis of every
    basis, the later dense and sparse solves checked against it."""
    t0 = time.time()
    pools = config1_pools(64, 200, 9100)
    m = pools[0].m
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), device=0)
    st, status, nup, basis, _ = run_batch(b, pools, 1.0)
    assert st == 0 and (nup > 0).all(), (status, nup)
    stats = Stats()
    assert check_maxvolume(b, pools, status, basis, {}, np.random.default_rng(9), stats) == len(pools)
    print(stats, f"{time.time() - t0:.1f} s")
    assert stats.steps == len(pools), str(stats)
    b.close()
