"""blu_batch_save / blu_batch_restore and their _dev variants under the SIMT emulator: a restored basis shows exactly
what its source shows and then goes on as an oracle object that went through the source's history; a restore within a
batch leaves it as blu_batch_copy does, bit for bit; a restore into another batch (other capacities, a smaller bnz_cap,
through a file) behaves as the saved basis; save changes nothing; every malformed call or image is rejected and
changes nothing; the _dev variants read back only sizes, headers and a verdict."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from blu_b200 import BLU, BLUBatch, load_library
from copy_cases import CLane, assert_copies, snapshot
from save_cases import (SaveTwin, checksum, field, fork, fork_and_check, header_bytes, reseal, restore_fork, sections,
                        set_field)
from subset_cases import (_pi, assert_dense, assert_getters, assert_same_snapshot, csc, factorize, layout, replay, solve_n,
                          solve_t, update)

HERE = os.path.dirname(os.path.abspath(__file__))
CPU = torch.device("cpu")


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


@pytest.fixture(scope="module")
def emu_traffic(emu):
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "emu_traffic")])
    return load_library(os.path.join(HERE, "emu_traffic", "libblu_emu_traffic.so"))


def new_batch(emu, lanes, mem=None, nmat=None, bnz_cap=None):
    m = lanes[0].m
    cap = max(sum(len(r) for r, _ in L.cols) for L in lanes) + 4 * m if bnz_cap is None else bnz_cap
    b = BLUBatch(nmat or len(lanes), m, cap, lib=emu)
    b.threads_per_basis = 64
    if mem:
        b.l_mem = mem; b.u_mem = mem; b.w_mem = mem
    return b


def lanes_for(nmat, m, seed0):
    """alternately sparse (many slack columns) and dense bases, so that with small stores only some grow private ones"""
    return [CLane(seed0 + k, m, nslack=m - 4 if k % 2 else 0, pmean=3.0 if k % 2 else 6.0, policy=k % 2) for k in range(nmat)]


def dirty(b, lanes, ks, rounds):
    """full basis changes on the bases ks only, so that they carry a longer history"""
    for _ in range(rounds):
        pend = solve_n(b, lanes, ks)
        solve_t(b, lanes, pend, want=1)
        ok = [k for k in ks if lanes[k].pending is not None]
        if ok:
            update(b, lanes, ok)
        redo = [k for k in ks if lanes[k].refactor]
        if redo:
            factorize(b, lanes, redo)


def refactorize_resident(b, lanes):
    """blu_batch_factorize_resident: every basis from the B it was last factorized from, the oracles alongside"""
    assert b.factorize_resident() == 0
    for k, L in enumerate(lanes):
        cp, ri, v = csc(L.factored)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == b.info(k, "status")
        L.cols = list(L.factored)
        L.pending, L.refactor = None, False
    assert_getters(b, lanes)


@pytest.mark.parametrize("point,small,mode", [("factorized", True, "dev"), ("updated", True, "host"), ("pending_n", True, "dev"),
                                              ("pending_nt", True, "cross"), ("never_factorized", True, "dev"),
                                              ("pending_nt", False, "dev"), ("updated", False, "host")],
                         ids=["factorized", "updated", "pending_n", "pending_nt", "never_factorized", "pending_nt-uniform",
                              "updated-uniform"])
def test_emu_restore_overwrites_dirty_slots(emu, point, small, mode):
    """Destinations first carry a different and longer history than their sources, with private stores forced by small
    stores or in the uniform ones; restoring the sources' images at each fork point makes them show exactly their
    sources' state, and every lane then matches its oracle through 12 rounds of its own schedule."""
    nmat, m = 8, 16
    lanes = lanes_for(nmat, m, 41000)
    b = new_batch(emu, lanes, mem=3 * m if small else None)
    src, dst = [0, 1, 2], [5, 6, 4]
    if point == "never_factorized":
        factorize(b, lanes, [k for k in range(nmat) if k not in src])
    else:
        factorize(b, lanes, list(range(nmat)))
    assert (b.info(0, "nrealloc") > 0) == small
    dirty(b, lanes, dst, 6)
    if point == "updated":
        dirty(b, lanes, src, 2)
    elif point in ("pending_n", "pending_nt"):
        pend = solve_n(b, lanes, src)
        if point == "pending_nt":
            solve_t(b, lanes, pend, want=0)
    fork_and_check(b, lanes, dst, src, seed=7, mode=mode)
    if point == "never_factorized":
        for d in dst:
            assert b.info(d, "nupdate") == -1
        factorize(b, lanes, src + dst)
    if point == "pending_nt":
        assert update(b, lanes, src + dst)[0] == 0
    replay(b, lanes, 12, 41100)
    assert_dense(b, lanes, 41200)


@pytest.mark.parametrize("mode", ["dev", "host", "cross"])
def test_emu_restore_equals_copy(emu, mode):
    """Twin batches, one forking with copy and one through images: bit-identical after every call, at several fork
    points (with a pending pair, with private and uniform stores, a fan-out), and every lane against its oracle."""
    nmat, m = 8, 16
    lanes = lanes_for(nmat, m, 42000)
    tw = SaveTwin(lambda: new_batch(emu, lanes, mem=3 * m), CPU, mode)
    factorize(tw, lanes, list(range(nmat)))
    dirty(tw, lanes, [0, 1, 4], 2)
    fork(tw, lanes, [2, 3, 5], [0, 0, 4])
    assert_copies(snapshot(tw, range(nmat), seed=6, lanes=lanes), [2, 3, 5], [0, 0, 4])
    replay(tw, lanes, 5, 42100, dense_every=2)
    pend = solve_n(tw, lanes, [1, 6])
    solve_t(tw, lanes, pend, want=1)
    fork(tw, lanes, [0, 7], [1, 6])
    replay(tw, lanes, 5, 42200, dense_every=2)
    fork(tw, lanes, [k for k in range(nmat) if k != 3], [3] * (nmat - 1))
    replay(tw, lanes, 4, 42300, dense_every=2)


def test_emu_restore_cross_batch(emu, tmp_path):
    """Images of a batch with small forced stores go into a second batch with other uniform capacities and a bnz_cap
    smaller than their row-wise B: private stores of the images' sizes and a grown row-wise B; the restored lanes match
    their oracles.  Then the same through a file read back into a batch made afterwards."""
    nmat, m = 6, 16
    lanes = lanes_for(nmat, m, 43000)
    a = new_batch(emu, lanes, mem=3 * m)
    factorize(a, lanes, list(range(nmat)))
    dirty(a, lanes, list(range(nmat)), 3)
    pend = solve_n(a, lanes, [2])
    solve_t(a, lanes, pend, want=0)      # basis 2: a pending pair travels with it
    imgs = a.save(range(nmat))
    assert all(field(im, "bt_n") > 4 for im in imgs)
    other = [CLane(43500 + k, m, nslack=m - 2, pmean=2.0) for k in range(5)]
    b = new_batch(emu, other, bnz_cap=4)
    factorize(b, other, list(range(5)))
    dirty(b, other, list(range(5)), 2)
    # the dense bases 0, 2, 4 need more row-wise B room than b's bnz_cap, which their own factorization never needed
    assert max(field(imgs[k], "bt_n") for k in (0, 2, 4)) > max(sum(len(r) for r, _ in L.cols) for L in other)
    dst, src = [3, 0, 4], [0, 2, 4]
    assert b.restore(dst, [imgs[s] for s in src]) == 0
    for d, s in zip(dst, src):
        other[d].adopt(lanes[s])
    before = snapshot(a, src, seed=8, lanes=lanes)
    after = snapshot(b, dst, seed=8, lanes=other)
    for d, s in zip(dst, src):
        assert_same_snapshot({0: before[s]}, {0: after[d]})
    assert update(b, other, [0])[0] == 0
    replay(b, other, 10, 43100)
    assert_dense(b, other, 43200)
    # through a file, into a batch created afterwards
    path = tmp_path / "basis.img"
    a.save([5])[0].tofile(path)
    c = new_batch(emu, lanes, nmat=3)
    back = np.fromfile(path, np.uint8)
    assert c.restore([1], [back]) == 0
    three = [CLane(43800 + k, m) for k in range(3)]
    three[1].adopt(lanes[5])
    factorize(c, three, [0, 2])
    replay(c, three, 8, 43300)


def test_emu_restore_resident_b(emu):
    """After a restore, factorize_resident refactorizes the destination from the saved basis' B: a library-owned B, a
    caller-owned B from factorize_dev (whose arrays stay unchanged), a basis whose last factorization answered
    InvalidArgument, and (test_emu_restore_resident_b_after_maxvolume) the B left by maxvolume."""
    nmat, m = 6, 20
    lanes = lanes_for(nmat, m, 44000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, list(range(nmat)), 2)
    fork(b, lanes, [3, 4], [0, 1], mode="host")
    refactorize_resident(b, lanes)
    # caller-owned B
    bb = np.zeros(nmat * m, np.int64); be = np.zeros(nmat * m, np.int64); bi, bx, off = [], [], 0
    for k, L in enumerate(lanes):
        for j, (ri, v) in enumerate(L.cols):
            bb[k * m + j] = off; be[k * m + j] = off + len(ri); bi.append(np.asarray(ri, np.int64)); bx.append(np.asarray(v)); off += len(ri)
    bi, bx = np.concatenate(bi), np.concatenate(bx)
    arrays = [a.copy() for a in (bb, be, bi, bx)]
    assert b.factorize_dev(bb.ctypes.data, be.ctypes.data, bi.ctypes.data, bx.ctypes.data, len(bi)) == 0
    for L in lanes:
        cp, ri, v = csc(L.cols)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.factored = list(L.cols); L.pending = None; L.refactor = False
    assert_getters(b, lanes)
    dirty(b, lanes, [2], 2)
    fork(b, lanes, [0, 1], [2, 2], mode="dev")
    fork(b, lanes, [5], [4], mode="dev")
    assert all(np.array_equal(x, y) for x, y in zip((bb, be, bi, bx), arrays))      # the caller's B is read, never written
    refactorize_resident(b, lanes)
    # a basis whose last factorization answered InvalidArgument (a column with b_end < b_begin): its negative length
    # travels with the image, and the destination answers InvalidArgument again
    bad_b, bad_e, bad_i, bad_x = layout([lanes[1].cols])
    bad_e[9] = bad_b[9] - 1
    st, stat = b.factorize_subset([1], bad_b, bad_e, bad_i, bad_x)
    assert stat[0] == -4
    assert restore_fork(b, [3], [1], "dev") == 0
    assert b.factorize_resident() == 0
    assert b.info(3, "status") == b.info(1, "status") == -4
    for k in (0, 2, 4, 5):
        assert b.info(k, "status") == 0


def test_emu_restore_resident_b_after_maxvolume(emu):
    """After maxvolume the resident B of every basis is its final basis; a restore takes the saved basis' columns, and
    factorize_resident refactorizes each destination from them, as the oracle does."""
    from mv_cases import make_pool, run_batch
    from oracle_lib import Oracle
    m = 40
    pools = [make_pool(44500 + k, m, 60, scale=3.0) for k in range(4)]
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), lib=emu)
    b.threads_per_basis = 64
    res = run_batch(b, pools, 1.2)
    assert res[0] == 0 and (res[2] > 0).all()
    assert restore_fork(b, [2, 3], [0, 0], "host") == 0
    assert b.factorize_resident() == 0
    owner = {0: 0, 1: 1, 2: 0, 3: 0}
    for k in range(len(pools)):
        p, bas = pools[owner[k]], res[3][owner[k]]
        o = Oracle(m, 60 * len(p.a_i))
        assert o.factorize(p.a_p[bas], p.a_p[bas + 1], p.a_i, p.a_x) == 0
        sto, fo = o.get_factors()
        stg, fg = b.get_factors(k)
        assert sto == stg == 0
        for key in fo:
            assert np.array_equal(fo[key], fg[key]), (k, key)


def test_emu_save_changes_nothing_fanout_and_graph(emu):
    """Save (host and _dev) leaves every basis as it was and a captured graph launchable; images are deterministic; a
    fan-out restore of one image into every other slot works; a restore drops the graph."""
    nmat, m = 6, 20
    lanes = lanes_for(nmat, m, 45000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, [0, 1, 2], 2)
    pend = solve_n(b, lanes, [4])
    solve_t(b, lanes, pend, want=1)                      # basis 4: a pending pair
    assert b.graph_capture("N") == 0
    before = snapshot(b, range(nmat), seed=5, lanes=lanes)
    one = b.save(range(nmat))
    dev = b.save_dev([4, 4, 0])
    assert np.array_equal(dev[0].numpy(), one[4]) and np.array_equal(dev[1].numpy(), one[4]) and np.array_equal(dev[2].numpy(), one[0])
    assert all(np.array_equal(x, y) for x, y in zip(one, b.save(range(nmat))))
    assert all(field(im, "checksum") == checksum(im) for im in one)
    assert_same_snapshot(before, snapshot(b, range(nmat), seed=5, lanes=lanes))
    assert b.graph_launch() == 0                         # (the graph refactorizes every basis from its resident B)
    refactorize_resident_after_graph(b, lanes)
    pend = solve_n(b, lanes, [2])
    solve_t(b, lanes, pend, want=0)
    img = b.save_dev([2])[0]
    dst = [k for k in range(nmat) if k != 2]
    assert b.restore_dev(dst, [img] * len(dst)) == 0
    for d in dst:
        lanes[d].adopt(lanes[2])
    assert_copies(snapshot(b, range(nmat), seed=9, lanes=lanes), dst, [2] * len(dst))
    assert b.graph_launch() == -2
    assert update(b, lanes, list(range(nmat)))[0] == 0
    replay(b, lanes, 8, 45100)


def refactorize_resident_after_graph(b, lanes):
    for L in lanes:
        cp, ri, v = csc(L.factored)
        assert L.oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
        L.cols = list(L.factored)
        L.pending, L.refactor = None, False
    assert_getters(b, lanes)


def raw_save(b, fn, n, idx, bufs, cap, nbytes):
    ptrs = None if bufs is None else (ctypes.c_void_p * max(len(bufs), 1))(*bufs)
    return getattr(b._L, fn)(b._h, n, _pi(idx), ptrs, _pi(cap), _pi(nbytes))


def raw_restore(b, fn, n, dst, bufs, cap):
    ptrs = None if bufs is None else (ctypes.c_void_p * max(len(bufs), 1))(*bufs)
    return getattr(b._L, fn)(b._h, n, _pi(dst), ptrs, _pi(cap))


def test_emu_save_restore_rejections(emu):
    """Every rejected call returns BLU_ERROR_INVALID_ARGUMENT, launches nothing past the check that decides, and changes nothing: bad
    header fields (each resealed with a valid checksum so that the header check alone decides), a length over the
    capacity, an extent over its capacity, a flipped byte in each section, unaligned buffers, bad n, bad or repeated
    destinations, missing arrays, a blu_create object.  Size queries, a too small capacity on save, n == 0."""
    nmat, m = 5, 16
    lanes = lanes_for(nmat, m, 46000)
    b = new_batch(emu, lanes)
    factorize(b, lanes, list(range(nmat)))
    dirty(b, lanes, [0, 1], 2)
    pend = solve_n(b, lanes, [0])
    solve_t(b, lanes, pend, want=1)
    img = b.save([0])[0]
    secs = sections(img)
    assert [s[0] for s in secs[:3]] == ["header", "l_idx", "l_val"] and secs[0][2] == header_bytes(img)
    before = snapshot(b, range(nmat), seed=2, lanes=lanes)
    launches = b.launch_count()
    # save: size query, too small a capacity, n == 0, argument errors
    nb = np.zeros(2, np.int64)
    assert raw_save(b, "blu_batch_save", 2, [0, 0], None, None, nb) == 0 and nb[0] == nb[1] == len(img)
    assert b.launch_count() == launches + 1                      # k_save_extents
    buf = np.zeros(len(img) + 32, np.uint8)
    k = (-buf.ctypes.data) % 16
    nb[:] = 0
    assert raw_save(b, "blu_batch_save", 1, [0], [buf.ctypes.data + k], [len(img) - 16], nb) == -4 and nb[0] == len(img)
    assert not buf.any()                                          # no image written
    assert raw_save(b, "blu_batch_save", 1, [0], [buf.ctypes.data + k + 4], [len(img)], nb) == -4      # unaligned
    for fn in ("blu_batch_save", "blu_batch_save_dev"):
        assert raw_save(b, fn, 0, None, None, None, None) == 0
        assert raw_save(b, fn, -1, [0], None, None, nb) == -4
        assert raw_save(b, fn, 1, [nmat], None, None, nb) == -4 and raw_save(b, fn, 1, [-1], None, None, nb) == -4
        assert raw_save(b, fn, 1, None, None, None, nb) == -4 and raw_save(b, fn, 1, [0], None, None, None) == -4
        assert raw_save(b, fn, 1, [0], [buf.ctypes.data + k], None, nb) == -4                           # no cap
    launches = b.launch_count()
    # restore: argument errors (nothing launched)
    p = img.ctypes.data
    for fn in ("blu_batch_restore", "blu_batch_restore_dev"):
        assert raw_restore(b, fn, 0, None, None, None) == 0
        assert raw_restore(b, fn, -1, [1], [p], [len(img)]) == -4
        assert raw_restore(b, fn, nmat + 1, list(range(nmat)) + [0], [p] * (nmat + 1), [len(img)] * (nmat + 1)) == -4
        assert raw_restore(b, fn, 1, [nmat], [p], [len(img)]) == -4 and raw_restore(b, fn, 1, [-1], [p], [len(img)]) == -4
        assert raw_restore(b, fn, 2, [1, 1], [p, p], [len(img)] * 2) == -4
        assert raw_restore(b, fn, 1, None, [p], [len(img)]) == -4 and raw_restore(b, fn, 1, [1], None, [len(img)]) == -4
        assert raw_restore(b, fn, 1, [1], [p], None) == -4 and raw_restore(b, fn, 1, [1], [0], [len(img)]) == -4
        mis = np.zeros(len(img) + 32, np.uint8)
        q = (-mis.ctypes.data) % 16 + 8
        mis[q:q + len(img)] = img
        assert raw_restore(b, fn, 1, [1], [mis.ctypes.data + q], [len(img)]) == -4                         # not 16-byte aligned
        assert raw_restore(b, fn, 1, [1], [p], [len(img) - 16]) == -4                                      # length > cap
    assert b.launch_count() == launches + 1      # (restore_dev gathers the header of the length > cap case on the device)
    # headers: each field wrong, resealed
    def bad(name, value):
        x = img.copy()
        set_field(x, name, value)
        return reseal(x)
    heads = [bad("magic", 0x1234), bad("version", 2), bad("m", m + 1), bad("info_bytes", int(field(img, "info_bytes")) + 8),
             bad("length", int(field(img, "length")) + 16), bad("l_n", int(field(img, "l_mem")) + 1),
             bad("u_n", int(field(img, "u_mem")) + 1), bad("w_n", int(field(img, "w_mem")) + 1), bad("bt_n", -1),
             bad("l_mem", int(field(img, "l_n")) - 1)]
    for x in heads:
        assert b.restore([1], [x]) == -4
        assert b.restore_dev([1], [torch.as_tensor(x)]) == -4
    # another batch's dimension
    o = new_batch(emu, lanes_for(2, m + 4, 46100))
    factorize(o, lanes_for(2, m + 4, 46100), [0, 1])
    assert b.restore([1], o.save([0])) == -4
    # one flipped byte in each section: the checksum
    launches = b.launch_count()
    for name, off, n in secs:
        if n == 0:
            continue
        x = img.copy()
        at = off + n // 2 if name != "header" else HDR_FLIP
        x[at] ^= 0x10
        assert b.restore_dev([1], [torch.as_tensor(x)]) == -4, name
    assert b.launch_count() == launches + 3 * sum(1 for s in secs if s[2])      # headers, checksum, verdict
    x = img.copy(); x[len(img) - 1] ^= 1                                         # the last padding byte
    assert b.restore([1], [x]) == -4
    assert_same_snapshot(before, snapshot(b, range(nmat), seed=2, lanes=lanes))
    # and the image itself restores: launches of a restore
    launches = b.launch_count()
    assert b.restore_dev([1], [torch.as_tensor(b.save([0])[0])]) == 0
    launches += 4      # (the save: the size query, then extents, images and checksums)
    assert b.launch_count() == launches + 8      # headers, checksum, verdict, B staging, rebuild_b (3), restore
    lanes[1].adopt(lanes[0])
    assert update(b, lanes, [0, 1])[0] == 0
    g = BLU(m, 64, lib=emu)
    assert emu.blu_batch_save(g._h, 0, None, None, None, None) == -4
    assert emu.blu_batch_restore(g._h, 0, None, None, None) == -4
    assert emu.blu_batch_save_dev(g._h, 0, None, None, None, None) == -4
    assert emu.blu_batch_restore_dev(g._h, 0, None, None, None) == -4
    g.close()


HDR_FLIP = 112 + 4 * 7      # a byte inside the header's BluInfo (pivotlen): only the checksum catches it


def test_emu_save_restore_host_traffic(emu_traffic):
    """save_dev copies the n image sizes to the host and nothing else; restore_dev the n headers and two fixed-size
    summaries (the checksum verdict, the new resident B's size): the same at two dimensions, batch sizes and image
    sizes."""
    emu = emu_traffic
    per = {}
    for nmat, m, n in ((4, 16, 2), (7, 40, 5)):
        lanes = lanes_for(nmat, m, 47000 + m)
        b = new_batch(emu, lanes)
        factorize(b, lanes, list(range(nmat)))
        dirty(b, lanes, list(range(nmat)), 2)
        emu.cuda_emu_memcpy_reset()
        imgs = b.save_dev(list(range(n)))
        c = (ctypes.c_ulonglong * 5)()
        emu.cuda_emu_memcpy_bytes(c)
        assert c[2] == 2 * 8 * n, c[2]                  # (save_dev's size query, then the save: n sizes each)
        emu.cuda_emu_memcpy_reset()
        assert b.restore_dev(list(range(nmat - n, nmat)), imgs) == 0
        emu.cuda_emu_memcpy_bytes(c)
        per[m] = c[2] - n * header_bytes(imgs[0].numpy())
    assert per[16] == per[40] <= 128, per


@pytest.mark.parametrize("env,case", [("EMU_SEED=1", "test_emu_restore_overwrites_dirty_slots[pending_nt]"),
                                      ("EMU_STRICT=1", "test_emu_restore_overwrites_dirty_slots[pending_nt-uniform]")])
def test_emu_save_env(env, case):
    """the dirty-slot case at the 'N' + 'T' fork point under a shuffled lane order, and under the strict barrier check
    (uniform stores: with stores forced small the factorization's Reallocate path trips the strict check on its own)"""
    k, v = env.split("=")
    r = subprocess.run([os.sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider",
                        os.path.abspath(__file__) + "::" + case],
                       env=dict(os.environ, **{k: v}), cwd=HERE, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
