"""The batch calls on device buffers under the SIMT emulator ("device" memory is host memory there, so the _dev calls take
CPU tensors): twin batches, one driven through the host calls and one through the _dev calls, stay equal bit for bit,
every basis matches its oracle, bases that do not run do not move, malformed input is rejected on the device, and the
solve and update calls move a fixed number of bytes between host and device whatever the size of the batch."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from blu_b200 import gen, load_library
from bs_cases import (assert_dense_parity, assert_sparse_parity, dup_first_column, finish_update, make_batch, rhs_lists,
                      update_round)
from dev_cases import SENT_I, SENT_X, make_twin
from subset_cases import (Lane, assert_dense, assert_same_snapshot, csc, factorize, layout, replay, snapshot, solve_n,
                          solve_t, update)

HERE = os.path.dirname(os.path.abspath(__file__))
CPU = torch.device("cpu")


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


@pytest.fixture(scope="module")
def emu_traffic(emu):
    """the emulation build with every host<->device copy of the library counted (tests/emu_traffic)"""
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "emu_traffic")])
    return load_library(os.path.join(HERE, "emu_traffic", "libblu_emu_traffic.so"))


def copied(emu):
    c = (ctypes.c_ulonglong * 5)()
    emu.cuda_emu_memcpy_bytes(c)
    return c[1], c[2]          # host to device, device to host


def start(emu, nmat, m, seed0, mem=None, nslack=None, realloc_factor=None):
    lanes = [Lane(seed0 + k, m, nslack=nslack, policy=k % 4) for k in range(nmat)]
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m
    t = make_twin(emu, CPU, nmat, m, cap, mem=mem, threads=64, realloc_factor=realloc_factor)
    factorize(t, lanes, list(range(nmat)))
    return t, lanes


def test_emu_dev_schedule_replay(emu):
    """Each basis on its own schedule through the masked _dev calls, its twin through the subset calls: equal after
    every call, and equal to the oracles; MaximumUpdates, SingularUpdate, update_cost > 1 and nforrest == m all make
    bases refactorize through factorize_subset_dev."""
    stats = {}
    for nmat, m, nslack, rounds, seed in ((8, 40, 20, 30, 21000), (8, 16, 10, 90, 21200)):
        t, lanes = start(emu, nmat, m, seed, nslack=nslack)
        replay(t, lanes, rounds, seed + 50, stats=stats)
        assert_dense(t, lanes, seed + 99)
    assert all(stats.get(k, 0) > 0 for k in ("update_cost", "nforrest", "-5", "-6")), str(stats)


def test_emu_dev_whole_batch(emu):
    """d_run == NULL: factorize_subset_dev, solve_for_update_dev, update_dev, solve_sparse_dev and solve_dense_multi_dev
    against the whole-batch host calls and the oracles, with singular bases and ragged unit counts."""
    nmat, m = 5, 40
    _, oracles = make_batch(emu, nmat, m, 22000, singular=(3,), factorize=False)
    bases = [gen.basis(22000 + k, m, m // 3, 4.0) for k in range(nmat)]
    bases = [dup_first_column(*bs) if k == 3 else bs for k, bs in enumerate(bases)]
    t = make_twin(emu, CPU, nmat, m, max(len(bs[1]) for bs in bases))
    off = np.cumsum([0] + [len(bs[1]) for bs in bases])
    bb = np.concatenate([bs[0][:-1] + off[k] for k, bs in enumerate(bases)])
    be = np.concatenate([bs[0][1:] + off[k] for k, bs in enumerate(bases)])
    bi, bx = np.concatenate([bs[1] for bs in bases]), np.concatenate([bs[2] for bs in bases])
    st, stat = t.h.factorize(bb, be, bi, bx)
    std, sd = t.d.factorize_subset_dev(t.T(bb, torch.int64), t.T(be, torch.int64), t.T(bi, torch.int64), t.T(bx, torch.float64))
    assert np.array_equal(sd.numpy(), stat) and stat[3] == 2 and std == 2
    for k, (o, (cp, ri, v)) in enumerate(zip(oracles, bases)):
        assert o.factorize(cp[:-1], cp[1:], ri, v) == stat[k]
    t.assert_state()
    for tr in "NT":
        assert_sparse_parity(t, oracles, rhs_lists(m, 22100, [3, 0, 1, 4, 2]), tr)
        assert_dense_parity(t, oracles, 3, 22200, tr)
    for it in range(3):
        finish_update(t, oracles, update_round(t, oracles, 22300, it))
        assert_sparse_parity(t, oracles, rhs_lists(m, 22400 + it, [1, 2, 0, 0, 3]), "N")


def test_emu_dev_untouched(emu):
    """Bases that do not run keep every getter, their factors, dense solves and a pending pair; their entries of the out
    tensors keep what they held (Twin checks them after every call)."""
    m = 50
    t, lanes = start(emu, 6, m, 23000)
    pend = solve_n(t, lanes, [0, 1, 2, 3])
    solve_t(t, lanes, pend, want=1)
    update(t, lanes, [0, 1])                          # bases 0, 1 updated; 2, 3 pending; 4, 5 fresh
    for sel, call in (([4, 0], "factorize"), ([5, 1], "solve"), ([1], "update"), ([], "solve"), ([], "update")):
        other = [k for k in range(6) if k not in sel]
        before = snapshot(t, other, seed=len(sel), lanes=lanes)
        if call == "factorize":
            factorize(t, lanes, sel)
        elif call == "solve":
            solve_t(t, lanes, solve_n(t, lanes, sel), want=0)
        else:
            update(t, lanes, sel)
        assert_same_snapshot(before, snapshot(t, other, seed=len(sel), lanes=lanes))
    update(t, lanes, [2, 3])


def test_emu_dev_rejects(emu):
    """Every device-validated reject: BLU_ERROR_INVALID_ARGUMENT, no launch but the check, no state change, out tensors
    untouched; a missing pointer is rejected on the host without a launch."""
    m, n = 30, 4
    t, lanes = start(emu, n, m, 24000)
    solve_t(t, lanes, solve_n(t, lanes, [1]), want=0)       # a pending pair on basis 1
    b = t.d
    T = t.T
    before = snapshot(t, range(n), lanes=lanes)
    bb, be, bi, bx = layout([L.cols for L in lanes])       # (per-basis layout: basis k's columns at k * m)
    I64, F64, I32 = torch.int64, torch.float64, torch.int32
    run = T([1, 0, 1, 1], I32)
    outs = t.sentinels(n, True)
    ub = T([0, 1, 1, 2, 3], I64)

    def same_outs():
        assert (outs[0] == SENT_I).all() and (outs[1] == SENT_I).all() and (outs[2] == SENT_I).all() and (outs[3] == SENT_X).all()

    def check(call, launches=1):
        l0 = b.launch_count()
        assert call() == -4
        assert b.launch_count() - l0 == launches
        same_outs()

    F = lambda bb_, be_, nz, r=run: b._L.blu_batch_factorize_subset_dev(b._h, b._ptr(r), b._ptr(bb_), b._ptr(be_), b._ptr(T(bi, I64)),
                                                                          b._ptr(T(bx, F64)), nz, b._ptr(outs[0]))
    nz = len(bi)
    bad = be.copy(); bad[2 * m + 7] = nz + 1
    check(lambda: F(T(bb, I64), T(bad, I64), nz))                          # b_end of a running basis beyond bnz_total
    bad = bb.copy(); bad[3 * m] = -1
    check(lambda: F(T(bad, I64), T(be, I64), nz))                          # negative b_begin
    check(lambda: F(T(bb, I64), T(be, I64), -1), 0)                        # negative bnz_total (host)
    check(lambda: F(None, T(be, I64), nz), 0)                              # missing array (host)
    ok = bb.copy(); ok[1 * m + 3] = -5                                      # basis 1 does not run: its B is not read
    l0 = b.launch_count()
    assert F(T(ok, I64), T(be, I64), nz, T([0, 0, 0, 0], I32)) == 0 and b.launch_count() == l0      # all-zero mask
    S = lambda rb, ir=T([1, 2, 3], I64), want=1, r=run: b._L.blu_batch_solve_for_update_dev(
        b._h, b._ptr(r), b._ptr(rb), b._ptr(ir), b._ptr(T(np.ones(3), F64)), want, b._ptr(outs[1]), b._ptr(outs[2]), b._ptr(outs[3]),
        b._ptr(outs[0]), b"N")
    check(lambda: S(T([0, 1, 1, 4, 3], I64)))                              # offset of a running basis beyond rhs_begin[nmat]
    check(lambda: S(T([-1, 1, 1, 2, 3], I64)))                             # negative offset of a running basis
    check(lambda: S(T([0, 1, 1, 2, -1], I64)))                             # negative total
    check(lambda: S(T([0, 1, 1, 2, 3], I64), ir=None))                     # entries without irhs
    check(lambda: S(None), 0)
    check(lambda: b._L.blu_batch_solve_for_update_dev(b._h, None, b._ptr(T([0, 1, 1, 2, 3], I64)), None, None, 1, None, None, None, None, b"N"), 0)
    U = lambda nu, ub_, rb, ir, xr: b._L.blu_batch_solve_sparse_dev(b._h, nu, b._ptr(ub_), b._ptr(rb), b._ptr(ir), b._ptr(xr),
                                                                    b._ptr(outs[1]), b._ptr(outs[2]), b._ptr(outs[3]), b._ptr(outs[0]), b"N")
    ir3, xr3, rb3 = T([1, 2, 3], I64), T(np.ones(3), F64), T([0, 1, 2, 3], I64)
    check(lambda: U(3, T([1, 1, 1, 2, 3], I64), rb3, ir3, xr3))            # unit_begin[0] != 0
    check(lambda: U(3, T([0, 2, 1, 2, 3], I64), rb3, ir3, xr3))            # decreasing
    check(lambda: U(2, ub, rb3[:3], ir3, xr3))                             # unit_begin[nmat] != nunits
    check(lambda: U(3, ub, T([0, 4, 2, 3], I64), ir3, xr3))                # unit offset beyond rhs_begin[nunits]
    check(lambda: U(3, ub, T([0, 1, -2, 3], I64), ir3, xr3))               # negative unit offset
    check(lambda: U(3, ub, T([0, 1, 2, -3], I64), ir3, xr3))               # negative total
    check(lambda: U(3, ub, rb3, ir3, None))                                # entries without xrhs
    check(lambda: U(-1, ub, rb3, ir3, xr3), 0)
    check(lambda: U(3, None, rb3, ir3, xr3), 0)
    check(lambda: b._L.blu_batch_solve_dense_multi_dev(b._h, -1, b._ptr(T(np.ones(n * m), F64)), b._ptr(outs[3]), b"N", b._ptr(outs[0])), 0)
    check(lambda: b._L.blu_batch_update_dev(b._h, b._ptr(run), None, b._ptr(outs[0])), 0)
    assert_same_snapshot(before, snapshot(t, range(n), lanes=lanes))
    # the Python layer: wrong dtype, device, length, contiguity
    with pytest.raises(TypeError):
        b.update_dev(T(np.ones(n), torch.float32))
    with pytest.raises(ValueError):
        b.update_dev(T(np.ones(n + 1), F64))
    with pytest.raises(ValueError):
        b.update_dev(T(np.ones(2 * n), F64)[::2])
    with pytest.raises(ValueError):
        b.update_dev(T(np.ones(n), F64), run=T(np.ones(n + 1), I32))
    if torch.cuda.is_available():
        with pytest.raises(ValueError):
            b.update_dev(T(np.ones(n), F64).cuda())
    # the pending pair of basis 1 is intact on both twins
    update(t, lanes, [1])


def test_emu_dev_per_basis_errors(emu):
    """A row index >= m in one running basis' B, an update of a basis never factorized: the basis' status word, the
    others carry on; the return value is the first non-OK status in index order."""
    m = 35
    lanes = [Lane(25000 + k, m) for k in range(4)]
    t = make_twin(emu, CPU, 4, m, max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m, threads=64)
    bad_row = list(lanes[2].cols); bad_row[5] = (np.array([1, m]), np.array([1.0, 2.0]))
    lanes[2].cols = bad_row
    sel = [3, 2, 0]
    st, stat = t.factorize_subset(sel, *layout([lanes[k].cols for k in sel]))
    exp = []
    for k in sel:
        cp, ri, v = csc(lanes[k].cols)
        exp.append(lanes[k].oracle.factorize(cp[:-1], cp[1:], ri, v))
    assert list(stat) == exp == [0, -4, 0] and st == -4
    st, stat = t.update_subset([1, 3], [1.0, 1.0])
    assert list(stat) == [-2, -2]


def test_emu_dev_tight_stores(emu):
    """Stores far too small, grown by no more than asked: Reallocate fires inside factorize_subset_dev,
    solve_for_update_dev and update_dev (a row file of one entry without padding, so that the update outgrows it), and
    the twins and the oracles still agree."""
    stats = {}
    m = 60
    lanes = [Lane(26000 + k, m, nslack=10, policy=k % 4) for k in range(5)]
    t = make_twin(emu, CPU, 5, m, max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m, mem=90, threads=64, realloc_factor=1.0)
    nr = t.info(0, "nrealloc")
    factorize(t, lanes, [3, 1, 0, 4, 2])
    assert t.info(0, "nrealloc") > nr
    replay(t, lanes, 30, 26050, stats=stats)
    assert_dense(t, lanes, 26090)
    m = 40
    lanes = [Lane(31040 + k, m, nslack=10, policy=k % 4) for k in range(4)]
    t = make_twin(emu, CPU, 4, m, max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m, threads=64, realloc_factor=1.0)
    for x in (t.h, t.d):
        x.w_mem = 1; x.pad = 0; x.stretch = 0.0
    factorize(t, lanes, list(range(4)))
    replay(t, lanes, 12, 31050, dense_every=4, stats=stats)
    assert stats["realloc_solve"] > 0 and stats["realloc_update"] > 0, stats      # (the first factorization grew the stores)


def test_emu_dev_host_traffic(emu_traffic):
    """solve_for_update_dev, update_dev, solve_sparse_dev and solve_dense_multi_dev copy the same bytes between host and
    device at nmat = 4 and at nmat = 32 with more units: the summary reads and nothing else.  (The host variants, for
    comparison, copy bytes that grow with the batch.)"""
    emu = emu_traffic
    per, host = {}, {}
    for nmat in (4, 32):
        m = 24
        b, oracles = make_batch(emu, nmat, m, 27000)
        rec = []

        def measure(fn):
            emu.cuda_emu_memcpy_reset()
            r = fn()
            rec.append(copied(emu))
            return r
        cols = []
        for k in range(nmat):
            cp, ri, v = gen.basis(27100 + k, m, 0, 3.0)
            cols.append((ri[cp[0]:cp[1]], v[cp[0]:cp[1]]))
        rb = np.concatenate([[0], np.cumsum([len(c[0]) for c in cols])]).astype(np.int64)
        T = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt)
        st, stat, nz, il, xl = measure(lambda: b.solve_for_update_dev(T(rb, torch.int64), T(np.concatenate([c[0] for c in cols]), torch.int64),
                                                                       T(np.concatenate([c[1] for c in cols]), torch.float64), "N", 1))
        assert st == 0
        xl = xl.numpy(); il = il.numpy(); nz = nz.numpy()
        lv = np.array([int(il[k, np.argmax(np.abs(xl[k, :nz[k]]))]) for k in range(nmat)])
        xt = np.array([xl[k, :nz[k]][np.argmax(np.abs(xl[k, :nz[k]]))] for k in range(nmat)])
        st, *_ = measure(lambda: b.solve_for_update_dev(T(np.arange(nmat + 1), torch.int64), T(lv, torch.int64), None, "T", 0))
        assert st == 0
        st, _ = measure(lambda: b.update_dev(T(xt, torch.float64)))
        assert st == 0
        lists = rhs_lists(m, 27200, [nmat // 4 + (k % 3) for k in range(nmat)])
        units = [p for r in lists for p in r]
        ub = np.concatenate([[0], np.cumsum([len(r) for r in lists])]).astype(np.int64)
        urb = np.concatenate([[0], np.cumsum([len(ii) for ii, _ in units])]).astype(np.int64)
        st, *_ = measure(lambda: b.solve_sparse_dev(T(ub, torch.int64), T(urb, torch.int64), T(np.concatenate([ii for ii, _ in units]), torch.int64),
                                                    T(np.concatenate([x for _, x in units]), torch.float64), nunits=len(units)))
        assert st == 0
        st, *_ = measure(lambda: b.solve_dense_multi_dev(T(np.ones(nmat * 3 * m), torch.float64)))
        assert st == 0
        per[nmat] = rec
        emu.cuda_emu_memcpy_reset()
        assert b.solve_dense_multi(np.ones(nmat * 3 * m))[0] == 0
        host[nmat] = copied(emu)
    assert per[4] == per[32], per
    assert host[32][0] == 8 * host[4][0] > 0 and host[32][1] == 8 * host[4][1] > 0, host      # the counters see the copies
    assert all(h2d == 0 and d2h <= 128 for h2d, d2h in per[4]), per[4]


def test_emu_dev_resident_b_and_graph(emu):
    """After factorize_subset_dev the resident B is the one factorize_subset leaves (factorize_resident reproduces the
    factors on both twins, and the oracles' factors); a graph captured before is refused until recaptured."""
    m = 40
    t, lanes = start(emu, 5, m, 28000)
    replay(t, lanes, 5, 28050, dense_every=0)
    for x in (t.h, t.d):
        assert x.upload(rhs=np.ones(5 * m)) == 0 and x.graph_capture("N") == 0
    factorize(t, lanes, [0, 4])
    for x in (t.h, t.d):
        assert x.graph_launch() == -2
    assert t.h.factorize_resident() == 0 and t.d.factorize_resident() == 0
    for k, L in enumerate(lanes):
        L.cols = list(L.factored)
        cp, ri, v = csc(L.cols)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == t.info(k, "status")
        L.pending = None; L.refactor = False
        sto, fo = L.oracle.get_factors()
        _, fg = t.get_factors(k)
        assert all(np.array_equal(fo[q], fg[q]) for q in fo), k
    t.assert_state()
    for x in (t.h, t.d):
        assert x.graph_capture("N") == 0 and x.graph_launch() == 0
    t.assert_state()


@pytest.mark.parametrize("seed", [3])
def test_emu_dev_random_lane_order(emu, seed, monkeypatch):
    monkeypatch.setenv("EMU_SEED", str(seed))
    t, lanes = start(emu, 5, 40, 29000 + 10 * seed)
    replay(t, lanes, 6, 29050 + seed, dense_every=3)
