"""The batch calls on a subset of the bases on the B200, at configs[1]'s shape (gen.basis(seed, 2000, 700, 5.0)):
each selected basis matches its own oracle object, the others do not move."""
import numpy as np
import pytest

from blu_b200 import BLUBatch, gen
from parity import oracle_for
from subset_cases import Lane, factorize, layout, replay

pytestmark = pytest.mark.gpu

M, NSLACK = 2000, 700


def test_gpu_subset_schedule_replay():
    """256 bases over 15 rounds, each on its own schedule, every basis compared with its oracle after every call"""
    lanes = [Lane(13000 + k, M, nslack=NSLACK, pmean=5.0, policy=k % 4) for k in range(256)]
    b = BLUBatch(256, M, max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * M, device=0)
    factorize(b, lanes, list(range(256)))
    replay(b, lanes, 15, 13500, dense_every=5)
    assert sum(b.info(k, "nupdate_total") for k in range(256)) > 0


def test_gpu_subset_4096_bases():
    """4,096 bases with update history; 64 of them spread over the batch refactorize from a new B.  A sample of them
    matches the oracle, and every other basis' dense solves are unchanged bit for bit."""
    nmat = 4096
    bb, be, bi, bx, rhs = gen.batch(nmat, M, NSLACK, 5.0, 14000, 24000)
    b = BLUBatch(nmat, M, int((be - bb).reshape(nmat, M).sum(1).max()) + 4 * M, device=0)
    st, status = b.factorize(bb, be, bi, bx)
    assert st == 0 and (status == 0).all()
    cols = []
    for k in range(nmat):
        cp, ri, v = gen.basis(34000 + k, M, 0, 3.0)
        cols.append((ri[cp[0]:cp[1]], v[cp[0]:cp[1]]))
    st, stat, out = b.solve_for_update(cols, "N", want_solution=1)
    assert st == 0
    leave = [(np.array([int(out[k][0][np.argmax(np.abs(out[k][1]))])]), None) for k in range(nmat)]
    xt = np.array([out[k][1][np.argmax(np.abs(out[k][1]))] for k in range(nmat)])
    assert b.solve_for_update(leave, "T")[0] == 0 and b.update(xt)[0] == 0
    before = {tr: b.solve_dense(rhs, tr) for tr in "NT"}
    sel = [int(k) for k in np.linspace(5, nmat - 3, 64).astype(int)]
    newB = [gen.basis(44000 + r, M, NSLACK, 5.0) for r in range(64)]
    st, stat = b.factorize_subset(sel, *layout([[(ri[cp[j]:cp[j + 1]], v[cp[j]:cp[j + 1]]) for j in range(M)] for cp, ri, v in newB]))
    assert st == 0 and (stat == 0).all()
    after = {tr: b.solve_dense(rhs, tr) for tr in "NT"}
    other = np.setdiff1d(np.arange(nmat), sel)
    for tr in "NT":
        assert np.array_equal(before[tr][1][other], after[tr][1][other]), tr
        assert (after[tr][2] == 0).all()
    assert all(b.info(int(k), "nupdate") == 1 for k in other[::97])
    for r in range(0, 64, 9):
        cp, ri, v = newB[r]
        o = oracle_for(M, len(v), 20)
        assert o.factorize(cp[:-1], cp[1:], ri, v) == 0
        sto, fo = o.get_factors()
        stg, fg = b.get_factors(sel[r])
        assert sto == stg == 0
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (r, key)
        for tr in "NT":
            _, xo = o.solve_dense(rhs[sel[r] * M:(sel[r] + 1) * M], tr)
            assert np.array_equal(after[tr][1][sel[r]], xo), (r, tr)


def oracle_check(b, Bs, rhs):
    x = b.download()[1] if rhs is not None else None
    for k, (cp, ri, v) in enumerate(Bs):
        o = oracle_for(M, len(v), 20)
        assert o.factorize(cp[:-1], cp[1:], ri, v) == b.info(k, "status") == 0
        sto, fo = o.get_factors()
        stg, fg = b.get_factors(k)
        assert sto == stg == 0
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (k, key)
        if rhs is not None:
            _, xo = o.solve_dense(rhs[k * M:(k + 1) * M], "N")
            assert np.array_equal(x[k], xo), k


def test_gpu_subset_caller_owned_b():
    """B in caller-owned device memory (factorize_dev), then factorize_subset: the resident B becomes library-owned,
    the caller's buffers can be overwritten, and factorize_resident refactorizes every basis from its last B."""
    import torch
    nmat = 16
    bb, be, bi, bx, _ = gen.batch(nmat, M, NSLACK, 5.0, 15000, 25000)
    Bs = [gen.basis(15000 + k, M, NSLACK, 5.0) for k in range(nmat)]
    b = BLUBatch(nmat, M, max(len(v) for _, _, v in Bs) + 4 * M, device=0)
    t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (bb, be, bi, bx)]
    torch.cuda.synchronize()
    assert b.factorize_dev(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), len(bi)) == 0
    b.synchronize()
    sel = [3, 9, 14]
    for r, k in enumerate(sel):
        Bs[k] = gen.basis(35000 + r, M, NSLACK, 5.0)
    st, stat = b.factorize_subset(sel, *layout([[(ri[cp[j]:cp[j + 1]], v[cp[j]:cp[j + 1]]) for j in range(M)]
                                                for cp, ri, v in (Bs[k] for k in sel)]))
    assert st == 0 and (stat == 0).all()
    for x in t:
        x.zero_()
    torch.cuda.synchronize()
    assert b.factorize_resident() == 0
    oracle_check(b, Bs, None)


def test_gpu_subset_graph_recapture():
    """A graph captured before factorize_subset is refused afterwards; recaptured, its replay refactorizes every
    basis from its last B and solves with it, as the oracles do."""
    nmat = 16
    bb, be, bi, bx, rhs = gen.batch(nmat, M, NSLACK, 5.0, 16000, 26000)
    Bs = [gen.basis(16000 + k, M, NSLACK, 5.0) for k in range(nmat)]
    b = BLUBatch(nmat, M, max(len(v) for _, _, v in Bs) + 4 * M, device=0)
    assert b.factorize(bb, be, bi, bx)[0] == 0
    assert b.upload(rhs=rhs) == 0
    assert b.graph_capture("N") == 0 and b.graph_launch() == 0
    sel = [0, 7]
    for r, k in enumerate(sel):
        Bs[k] = gen.basis(36000 + r, M, NSLACK, 5.0)
    st, stat = b.factorize_subset(sel, *layout([[(ri[cp[j]:cp[j + 1]], v[cp[j]:cp[j + 1]]) for j in range(M)]
                                                for cp, ri, v in (Bs[k] for k in sel)]))
    assert st == 0
    assert b.graph_launch() == -2
    assert b.graph_capture("N") == 0 and b.graph_launch() == 0
    oracle_check(b, Bs, rhs)
