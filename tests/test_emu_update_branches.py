"""The explicit-basis checks of tests/update_cases.py on the device library under the SIMT emulator: a BLU bit-identical to
the oracle after every call with its own solves checked against the explicit B', and a BLUBatch of mixed structures
stepped through update_subset and update_dev with run masks, where every basis is checked against its explicit B'
after every round, with a row file so small that the update's Reallocate fires inside both calls; and the bases batch
maxvolume returns, rebuilt from its `basis` and checked the same way."""
import os
import subprocess

import numpy as np
import pytest
import torch

from blu_b200 import BLU, BLUBatch, load_library
from mv_cases import make_pool, run_batch
from oracle_lib import Oracle
from subset_cases import layout
from update_cases import Cols, Stats, batch_rounds, check_maxvolume, csc_of, draw_case, fresh_oracle, single_case

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


def test_emu_blu_update_branches(emu):
    """BLU against the oracle and the explicit basis on 16 seeded cases (m = 8..40, every structure, default and drawn
    tunables): every branch occurs."""
    def objs(m, nnz, t):
        o = Oracle(m, 400 * nnz + 2000)
        g = BLU(m, nnz, lib=emu)
        for k, x in t.items():
            o.set_param(k, x)
            setattr(g, k, x)
        return [o, g]
    stats = Stats()
    for seed in range(16):
        single_case(seed, objs, nsteps=16, stats=stats, mmin=8, mmax=40)
    print(stats)
    for b in ("ft", "sym", "unsym", "refused"):
        assert stats.count[b] > 0, str(stats)


# a row file of one entry without padding, grown by no more than asked: the updates' spikes outgrow it again and again,
# so that Reallocate fires inside update_subset and update_dev themselves
TIGHT = dict(pad=0, stretch=0.0)


def mixed_batch(lib, seed0, n, m):
    """n bases of dimension m of every structure (draw_case's kinds but 4), each nonsingular, one oracle each, under the
    TIGHT tunables and w_mem = 1"""
    bases, seed = [], seed0
    while len(bases) < n:
        _, kind, B, _, _ = draw_case(seed, m, m)
        seed += 1
        if kind == 4 or fresh_oracle(B, {})[0] != 0:    # kind 4's growth makes the bound vacuous; covered on one basis
            continue
        bases.append(Cols(*csc_of(B)))
    nnz = max(len(c.csc()[1]) for c in bases)
    b = BLUBatch(n, m, nnz + 8 * m, lib=lib)
    b.threads_per_basis = 64
    b.realloc_factor = 1.0
    b.w_mem = 1
    oracles = [Oracle(m, 400 * nnz + 2000) for _ in range(n)]
    for k, x in TIGHT.items():
        setattr(b, k, x)
        for o in oracles:
            o.set_param(k, x)
    st, stat = b.factorize_subset(list(range(n)), *layout([c.cols for c in bases]))
    assert st == 0 and (stat == 0).all(), stat
    for o, c in zip(oracles, bases):
        cp, ri, v = c.csc()
        assert o.factorize(cp[:-1], cp[1:], ri, v) == 0
    return b, oracles, bases


def test_emu_batch_update_branches(emu):
    """Six bases through 16 rounds of masked update_subset / update_dev: every basis against its oracle and its explicit
    basis after every round; all four outcomes occur, and Reallocate fires inside update_subset and inside update_dev
    (nrealloc grows during the update call itself)."""
    stats = Stats()
    for seed0, m in ((31000, 30), (31100, 24)):
        b, oracles, bases = mixed_batch(emu, seed0, 6, m)
        batch_rounds(b, oracles, bases, TIGHT, 16, seed0, update_dev=lambda a, dt: torch.as_tensor(a, dtype=dt),
                     stats=stats, zero_rate=0.08)
    print(stats)
    for k in ("ft", "sym", "unsym", "refused", "realloc_subset", "realloc_dev"):
        assert stats.count[k] > 0, str(stats)


def test_emu_maxvolume_against_explicit_basis(emu):
    """Batch maxvolume on four bases: B rebuilt from the returned basis, the later dense and sparse solves of every
    basis checked against it."""
    m = 40
    pools = [make_pool(seed, m, 120, scale=3.0) for seed in (101, 102, 103, 104)]
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), lib=emu)
    b.threads_per_basis = 64
    st, status, nup, basis, _ = run_batch(b, pools, 1.0)
    assert st == 0 and (nup > 0).all(), (status, nup)
    stats = Stats()
    assert check_maxvolume(b, pools, status, basis, {}, np.random.default_rng(5), stats) == len(pools)
    print(stats)
    assert stats.steps == len(pools), str(stats)
