"""The batch calls on device buffers on the B200, at configs[1]'s shape (gen.basis(seed, 2000, 700, 5.0)): a loop driven
entirely on the device against a twin batch driven through the host calls, stream ordering with a producer on a side
stream, and the host traffic of a steady step at 4,096 bases."""
import json
import os
import tempfile

import numpy as np
import pytest
import torch

from blu_b200 import BLUBatch, gen
from dev_cases import TWIN_GETTERS
from parity import oracle_for

pytestmark = pytest.mark.gpu

M, NSLACK, NPOOL = 2000, 700, 16
CUDA = torch.device("cuda", 0)


def setup(nmat, seed):
    bb, be, bi, bx, rhs = gen.batch(nmat, M, NSLACK, 5.0, seed, seed + 10000)
    cap = int((be - bb).reshape(nmat, M).sum(1).max()) + 4 * M
    return (bb, be, bi, bx), cap


def pool(nmat, seed):
    """NPOOL entering columns per basis: column c of basis k is pi/px[pb[k*NPOOL+c] : pb[k*NPOOL+c+1]]"""
    idx, val, begin = [], [], [0]
    for k in range(nmat):
        cp, ri, v = gen.basis(seed + k, M, 0, 3.0)
        for c in range(NPOOL):
            idx.append(ri[cp[c]:cp[c + 1]]); val.append(v[cp[c]:cp[c + 1]]); begin.append(begin[-1] + cp[c + 1] - cp[c])
    return np.concatenate(idx).astype(np.int64), np.concatenate(val), np.array(begin, np.int64)


def gather_columns(pi, px, pb, col, mask):
    """rhs_begin per basis, irhs, xrhs: basis k's pool column col[k] where mask is set, an empty range elsewhere"""
    lens = torch.where(mask, pb[col + 1] - pb[col], torch.zeros_like(col))
    rb = torch.cat([torch.zeros(1, dtype=torch.int64, device=CUDA), torch.cumsum(lens, 0)])
    pos = torch.arange(int(rb[-1]), device=CUDA) - torch.repeat_interleave(rb[:-1], lens)
    g = torch.repeat_interleave(pb[col], lens) + pos
    return rb, pi[g], px[g]


def compacted(bb, be, sel):
    return (np.concatenate([bb[k * M:(k + 1) * M] for k in sel]), np.concatenate([be[k * M:(k + 1) * M] for k in sel]))


@pytest.fixture(autouse=True)
def release_memory():
    """a 4,096-basis batch takes a good part of the card: free each test's batches and torch's cache before the next"""
    yield
    import gc
    gc.collect()
    torch.cuda.empty_cache()


def assert_twins(h, d, ks):
    for k in ks:
        for name in TWIN_GETTERS:
            a, b = h.info(int(k), name), d.info(int(k), name)
            assert a == b or (a != a and b != b), (k, name, a, b)


def test_gpu_dev_driven_loop():
    """1,024 bases over 16 rounds.  The bases that refactorize (6 updates of their own since the last time, staggered,
    or a failed step), the ones that pivot (3 in 4 of the others), the entering columns and the leaving rows (argmax |x|
    on the device) are chosen in torch and fed to the _dev calls; the twin follows the same choices through the subset
    calls.  Statuses, solutions and every getter are equal bit for bit after every round, and three bases follow their
    oracles through every call."""
    nmat = 1024
    (bb, be, bi, bx), cap = setup(nmat, 17000)
    h, d = BLUBatch(nmat, M, cap, device=0), BLUBatch(nmat, M, cap, device=0)
    Bd = [torch.from_numpy(np.ascontiguousarray(a)).to(CUDA) for a in (bb, be, bi, bx)]
    st, stat = h.factorize(bb, be, bi, bx)
    std, sd = d.factorize_subset_dev(*Bd)
    assert st == std == 0 and np.array_equal(sd.cpu().numpy(), stat)
    pin, pxn, pbn = pool(nmat, 37000)
    pi, px, pb = (torch.from_numpy(a).to(CUDA) for a in (pin, pxn, pbn))
    ar = torch.arange(nmat, device=CUDA)
    nup = (ar % 6).to(torch.int64)                     # staggered refactorization schedules
    need = torch.zeros(nmat, dtype=torch.bool, device=CUDA)
    rng = torch.Generator(device=CUDA).manual_seed(5)
    sample = [3, 511, 1000]
    oracles = {}
    for k in sample:
        cp, ri, v = gen.basis(17000 + k, M, NSLACK, 5.0)
        oracles[k] = oracle_for(M, len(v), 20)
        assert oracles[k].factorize(cp[:-1], cp[1:], ri, v) == 0
    counts = dict(refactor=0, pivots=0)
    for it in range(16):
        refac = need | (nup >= 6)
        if refac.any():
            sel = torch.nonzero(refac).flatten().cpu().numpy().tolist()
            st, stat = h.factorize_subset(sel, *compacted(bb, be, sel), bi, bx)
            std, sd = d.factorize_subset_dev(*Bd, run=refac.to(torch.int32))
            sd = sd.cpu().numpy()
            assert st == std == 0 and [sd[k] for k in sel] == list(stat)
            for k in set(sel) & set(sample):
                cp, ri, v = gen.basis(17000 + k, M, NSLACK, 5.0)
                assert oracles[k].factorize(cp[:-1], cp[1:], ri, v) == 0
            nup = torch.where(refac, torch.zeros_like(nup), nup)
            need = torch.zeros_like(need)
            counts["refactor"] += len(sel)
        pivot = (~refac) & (torch.rand(nmat, device=CUDA, generator=rng) < 0.75)
        col = ar * NPOOL + it % NPOOL
        rb, irhs, xrhs = gather_columns(pi, px, pb, col, pivot)
        std, sN, nz, il, xl = d.solve_for_update_dev(rb, irhs, xrhs, "N", 1, run=pivot.to(torch.int32))
        sel = torch.nonzero(pivot).flatten().cpu().numpy().tolist()
        rbn, irn, xrn = rb.cpu().numpy(), irhs.cpu().numpy(), xrhs.cpu().numpy()
        st, stat, out = h.solve_for_update_subset(sel, [(irn[rbn[k]:rbn[k + 1]], xrn[rbn[k]:rbn[k + 1]]) for k in sel], "N", 1)
        sNn, nzn, iln, xln = sN.cpu().numpy(), nz.cpu().numpy(), il.cpu().numpy(), xl.cpu().numpy()
        assert st == std and [sNn[k] for k in sel] == list(stat)
        for r, k in enumerate(sel):
            n = int(nzn[k])
            assert n == (len(out[r][0]) if stat[r] == 0 else -1)
            assert np.array_equal(iln[k, :max(n, 0)], out[r][0]) and np.array_equal(xln[k, :max(n, 0)], out[r][1]), k
            if k in oracles:
                o = oracles[k]
                assert o.solve_for_update(rbn[k + 1] - rbn[k], irn[rbn[k]:rbn[k + 1]], xrn[rbn[k]:rbn[k + 1]], "N", 1) == stat[r]
                if stat[r] == 0:
                    assert np.array_equal(out[r][0], o.ilhs[:o.nzlhs]) and np.array_equal(out[r][1], o.lhs[o.ilhs[:o.nzlhs]])
        # the leaving row on the device: the first largest |x| among the basis' solution entries
        ok = pivot & (sN == 0) & (nz > 0)
        valid = torch.arange(M, device=CUDA)[None, :] < nz[:, None]
        j = torch.where(valid, xl.abs(), torch.full_like(xl, -1.0)).argmax(1)
        leave, xt = il[ar, j], xl[ar, j]
        std, sT, _, _, _ = d.solve_for_update_dev(torch.arange(nmat + 1, device=CUDA), leave, None, "T", 0, run=ok.to(torch.int32))
        sel = torch.nonzero(ok).flatten().cpu().numpy().tolist()
        lv, xtn = leave.cpu().numpy(), xt.cpu().numpy()
        st, stat, _ = h.solve_for_update_subset(sel, [(np.array([lv[k]]), None) for k in sel], "T", 0)
        sTn = sT.cpu().numpy()
        assert st == std and [sTn[k] for k in sel] == list(stat)
        for r, k in enumerate(sel):
            if k in oracles:
                assert oracles[k].solve_for_update(1, np.array([lv[k]]), None, "T", 0) == stat[r]
        ok2 = ok & (sT == 0)
        std, sU = d.update_dev(xt, run=ok2.to(torch.int32))
        sel = torch.nonzero(ok2).flatten().cpu().numpy().tolist()
        st, stat = h.update_subset(sel, [xtn[k] for k in sel])
        sUn = sU.cpu().numpy()
        assert st == std and [sUn[k] for k in sel] == list(stat)
        for r, k in enumerate(sel):
            if k in oracles:
                assert oracles[k].update(xtn[k]) == stat[r]
        done = ok2 & (sU == 0)
        nup = nup + done.to(torch.int64)
        need = need | (pivot & ~done)
        counts["pivots"] += len(sel)
        assert_twins(h, d, range(0, nmat, 7) if it % 4 else range(nmat))
    assert_twins(h, d, range(nmat))
    for k, o in oracles.items():
        for name in ("nupdate", "nforrest", "u_nz", "r_nz", "l_flops", "u_flops", "r_flops", "update_cost", "pivot_error"):
            assert d.info(k, name) == o.info(name), (k, name)
    assert counts["refactor"] > nmat and counts["pivots"] > 8 * nmat, counts


def test_gpu_dev_side_stream_producer():
    """The inputs come from torch kernels on a side stream that starts with a long sleep; the calls are made with that
    stream current, so the library must wait for it.  The results equal those of the same inputs made ready first."""
    nmat = 64
    (bb, be, bi, bx), cap = setup(nmat, 18000)
    a, b = BLUBatch(nmat, M, cap, device=0), BLUBatch(nmat, M, cap, device=0)
    assert a.factorize(bb, be, bi, bx)[0] == 0 and b.factorize(bb, be, bi, bx)[0] == 0
    pin, pxn, pbn = pool(nmat, 38000)
    pi, px, pb = (torch.from_numpy(x).to(CUDA) for x in (pin, pxn, pbn))
    col = torch.arange(nmat, device=CUDA) * NPOOL
    every = torch.ones(nmat, dtype=torch.bool, device=CUDA)
    rb, irhs, xrhs = gather_columns(pi, px, pb, col, every)
    torch.cuda.synchronize()
    ref = a.solve_for_update_dev(rb, irhs, xrhs, "N", 1)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                 # ~0.1 s of spinning before the producer writes
        x2 = xrhs * 2.0 - xrhs                         # the same values, written by a kernel queued after the sleep
        r2 = b.solve_for_update_dev(rb, irhs, x2, "N", 1)
    assert r2[0] == ref[0] == 0
    for p, q in zip(ref[1:], r2[1:]):
        assert torch.equal(p, q)
    dense = torch.rand(nmat * 3 * M, dtype=torch.float64, device=CUDA)
    ref = a.solve_dense_multi_dev(dense)
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        d2 = dense + 0.0
        r2 = b.solve_dense_multi_dev(d2)
    assert torch.equal(ref[1], r2[1]) and torch.equal(ref[2], r2[2])


def test_gpu_dev_steady_step_traffic():
    """4,096 bases: 'N' with the solution, 'T', update and solve_sparse (R = 4) through the _dev calls.  The torch.profiler
    trace of the step lists no copy larger than the summary (5 words); the results match a twin through the host calls."""
    nmat = 4096
    (bb, be, bi, bx), cap = setup(nmat, 19000)
    h, d = BLUBatch(nmat, M, cap, device=0), BLUBatch(nmat, M, cap, device=0)
    assert h.factorize(bb, be, bi, bx)[0] == 0 and d.factorize(bb, be, bi, bx)[0] == 0
    pin, pxn, pbn = pool(nmat, 39000)
    pi, px, pb = (torch.from_numpy(x).to(CUDA) for x in (pin, pxn, pbn))
    ar = torch.arange(nmat, device=CUDA)
    every = torch.ones(nmat, dtype=torch.bool, device=CUDA)
    rb, irhs, xrhs = gather_columns(pi, px, pb, ar * NPOOL, every)
    # solve_sparse units: 4 per basis, pool columns 1..4 as right-hand sides
    R = 4
    ucol = (ar[:, None] * NPOOL + torch.arange(1, R + 1, device=CUDA)[None, :]).reshape(-1)
    ulen = pb[ucol + 1] - pb[ucol]
    urb = torch.cat([torch.zeros(1, dtype=torch.int64, device=CUDA), torch.cumsum(ulen, 0)])
    ug = torch.repeat_interleave(pb[ucol], ulen) + torch.arange(int(urb[-1]), device=CUDA) - torch.repeat_interleave(urb[:-1], ulen)
    uir, uxr = pi[ug], px[ug]
    ub = torch.arange(0, R * nmat + 1, R, device=CUDA, dtype=torch.int64)
    nunits = R * nmat
    outs = dict(nN=torch.zeros(nmat, dtype=torch.int64, device=CUDA), iN=torch.zeros(nmat * M, dtype=torch.int64, device=CUDA),
                xN=torch.zeros(nmat * M, dtype=torch.float64, device=CUDA), sN=torch.zeros(nmat, dtype=torch.int32, device=CUDA),
                sT=torch.zeros(nmat, dtype=torch.int32, device=CUDA), sU=torch.zeros(nmat, dtype=torch.int32, device=CUDA),
                nS=torch.zeros(nunits, dtype=torch.int64, device=CUDA), iS=torch.zeros(nunits * M, dtype=torch.int64, device=CUDA),
                xS=torch.zeros(nunits * M, dtype=torch.float64, device=CUDA), sS=torch.zeros(nunits, dtype=torch.int32, device=CUDA))
    leave = torch.zeros(nmat, dtype=torch.int64, device=CUDA)
    tb = torch.arange(nmat + 1, device=CUDA)
    xt = torch.zeros(nmat, dtype=torch.float64, device=CUDA)
    # host twin: the same step through the host calls (their inputs fetched before the trace)
    rbn, irn, xrn = rb.cpu().numpy(), irhs.cpu().numpy(), xrhs.cpu().numpy()
    stH, statH, outH = h.solve_for_update([(irn[rbn[k]:rbn[k + 1]], xrn[rbn[k]:rbn[k + 1]]) for k in range(nmat)], "N", 1)
    lvH = np.array([int(o[0][np.argmax(np.abs(o[1]))]) for o in outH])
    xtH = np.array([o[1][np.argmax(np.abs(o[1]))] for o in outH])
    leave.copy_(torch.from_numpy(lvH)); xt.copy_(torch.from_numpy(xtH))
    torch.cuda.synchronize()
    trace = os.path.join(tempfile.mkdtemp(), "step.json")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
        rN = d.solve_for_update_dev(rb, irhs, xrhs, "N", 1, status=outs["sN"], nzlhs=outs["nN"], ilhs=outs["iN"], xlhs=outs["xN"])
        rT = d.solve_for_update_dev(tb, leave, None, "T", 0, status=outs["sT"])
        rU = d.update_dev(xt, status=outs["sU"])
        rS = d.solve_sparse_dev(ub, urb, uir, uxr, "N", nunits=nunits, status=outs["sS"], nzlhs=outs["nS"], ilhs=outs["iS"], xlhs=outs["xS"])
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace)
    ev = json.load(open(trace))["traceEvents"]
    copies = [e for e in ev if e.get("cat") == "gpu_memcpy"]
    sizes = [int(e.get("args", {}).get("bytes", 0)) for e in copies]
    assert copies and max(sizes) <= 40, sorted(sizes)[-5:]
    assert rN[0] == rT[0] == rU[0] == rS[0] == 0
    # the twin
    assert h.solve_for_update([(np.array([lvH[k]]), None) for k in range(nmat)], "T", 0)[0] == 0
    assert h.update(xtH)[0] == 0
    lists = []
    uin, uxn, urn = uir.cpu().numpy(), uxr.cpu().numpy(), urb.cpu().numpy()
    for k in range(nmat):
        lists.append([(uin[urn[u]:urn[u + 1]], uxn[urn[u]:urn[u + 1]]) for u in range(k * R, (k + 1) * R)])
    stS, outS, ustS = h.solve_sparse(lists, "N")
    nN, iN, xN = outs["nN"].cpu().numpy(), outs["iN"].cpu().numpy().reshape(nmat, M), outs["xN"].cpu().numpy().reshape(nmat, M)
    nS, iS, xS = outs["nS"].cpu().numpy(), outs["iS"].cpu().numpy().reshape(nunits, M), outs["xS"].cpu().numpy().reshape(nunits, M)
    for k in range(nmat):
        assert nN[k] == len(outH[k][0]) and np.array_equal(iN[k, :nN[k]], outH[k][0]) and np.array_equal(xN[k, :nN[k]], outH[k][1])
        for q in range(R):
            u = k * R + q
            assert nS[u] == len(outS[k][q][0]) and np.array_equal(iS[u, :nS[u]], outS[k][q][0]) and np.array_equal(xS[u, :nS[u]], outS[k][q][1])
    assert (outs["sU"] == 0).all() and (outs["sS"] == 0).all()
    assert_twins(h, d, range(0, nmat, 13))
