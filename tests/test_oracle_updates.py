"""Every branch of the oracle's update (Forrest-Tomlin, symmetric permutation, unsymmetric permutation through the BFS
path, SingularUpdate) checked against an explicitly kept basis: the solves after each update must be as accurate as a
fresh factorization of the same B' allows, up to the growth the update admits (tests/update_cases.py has the bound and
the measurements behind it).  The device is bit-identical to the oracle, so these checks also pin what the device's
update computes."""
import numpy as np

from oracle_lib import Oracle
from update_cases import Stats, draw_case, single_case

NCASE = 300
# measured on seeds 0..299: ft 6426, sym 1593, unsym 505, refused 291; a generator change that loses half of a
# branch's cases fails here instead of silently testing less
MIN_COUNT = dict(ft=3000, sym=800, unsym=250, refused=140)


def oracles(m, nnz, t):
    o = Oracle(m, 400 * nnz + 2000)
    for k, x in t.items():
        o.set_param(k, x)
    return [o]


def test_oracle_update_branches_against_explicit_basis():
    """300 seeded cases, m = 8..120, structured_matrix kinds 0..5 and gen.basis, default and drawn tunables; every
    accepted update is checked against the explicit B' and each branch occurs at least MIN_COUNT times."""
    stats = Stats()
    for seed in range(NCASE):
        single_case(seed, oracles, stats=stats)
    print(stats)
    for b, n in MIN_COUNT.items():
        assert stats.count[b] >= n, str(stats)
    assert stats.count["realloc"] == 0


def test_oracle_updates_with_compression():
    """Tunables under which the update compresses its files, compress_thres 0.05 with small stretch and pad, and the
    opposite, wide padding that never compresses.  Same checks as above.  Counted once with counters at the two call
    sites in blo_k_update: in the 30 slim cases compress_packed (U) runs 177 times and blo_file_compress (the row file)
    137 times over 732 updates; in the 30 wide cases neither runs."""
    stats = Stats()
    for seed in range(5000, 5060):
        case = draw_case(seed)
        t = case[3]
        if seed % 2:
            t.update(compress_thres=0.05, stretch=0.1, pad=1)
        else:
            t.update(compress_thres=1.0, stretch=1.0, pad=8)
        single_case(seed, oracles, stats=stats, case=case)
    print(stats)
    for b in ("ft", "sym", "unsym", "refused"):
        assert stats.count[b] > 0, str(stats)


def test_constructed_column_takes_the_unsymmetric_branch():
    """Named case: right after a factorization the constructed entering column (spike = one off-diagonal entry) sends
    the update through the BFS / unsymmetric permutation, and the result solves like the explicit B'."""
    stats = Stats()
    for seed in (6, 13, 20):
        single_case(seed, oracles, nsteps=12, construct_rate=1.0, zero_rate=0.0, stats=stats)
    assert stats.count["unsym"] >= 3, str(stats)
    np.testing.assert_array_less(stats.worst_eta["unsym"], 1e-12)
