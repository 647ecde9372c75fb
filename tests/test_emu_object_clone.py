"""blu_clone, blu_save / blu_restore and their _dev variants under the SIMT emulator, against the CPU oracle: a clone
taken at every fork point shows exactly what its source shows, then follows the same schedule bit for bit or its own
against an oracle that replays the source's history; the source does not change; parameters and capacities are copied
and Reallocate fires on the same call; images move a basis between objects and batch slots both ways; a restore into
an object with other capacities rebuilds what a factorization leaves; every rejection changes nothing."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from blu_b200 import BLU, BLUBatch, load_library
from copy_cases import CLane, snapshot
from object_cases import Objects, assert_same_record, record
from save_cases import INFO_AT, field, header_bytes, reseal, sections, set_field
from subset_cases import assert_getters, assert_same_snapshot, csc, factorize, replay, solve_n, solve_t, update

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HAVE_UR = INFO_AT + 4 * 15          # BluInfo.have_ur in an image's header (blu_types.h)

POINTS = ["never_factorized", "factorized", "singular", "updated", "pending_n", "pending_nt", "c0ntinue"]


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "emu")])
    return load_library(os.path.join(HERE, "emu", "libblu_emu.so"))


@pytest.fixture(scope="module")
def emu_traffic(emu):
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "emu_traffic")])
    return load_library(os.path.join(HERE, "emu_traffic", "libblu_emu_traffic.so"))


def new_object(emu, lane, b_nz=None):
    o = BLU(lane.m, sum(len(r) for r, _ in lane.cols) + 4 * lane.m if b_nz is None else b_nz, lib=emu)
    o.threads_per_basis = 64
    return o


def launches(o):
    return o._L.blu_batch_launch_count(o._h)


def reach(b, lanes, point):
    """the object of slot 0 (lanes[0]) goes to the fork point; returns the pending 'N' solve, if any"""
    L, o = lanes[0], b.slots[0][0]
    if point == "never_factorized":
        return {}
    if point == "singular":
        L.cols[3] = L.cols[2]
    if point == "c0ntinue":
        o.l_mem = o.u_mem = o.w_mem = 8
        cp, ri, v = csc(L.cols)
        assert o.factorize_c0ntinue(cp[:-1], cp[1:], ri, v, False) == 1
        assert o.info("addmem_l") + o.info("addmem_u") + o.info("addmem_w") > 0
        return {}
    st, _ = factorize(b, lanes[:1], [0])
    assert st == (2 if point == "singular" else 0)
    if point == "updated":
        for _ in range(3):
            pend = solve_n(b, lanes[:1], [0])
            solve_t(b, lanes[:1], pend, want=1)
            if L.pending is not None:
                update(b, lanes[:1], [0])
        assert o.info("nupdate") > 0
    pend = {}
    if point in ("pending_n", "pending_nt"):
        pend = solve_n(b, lanes[:1], [0])
        assert pend
        if point == "pending_nt":
            solve_t(b, lanes[:1], pend, want=0)
    return pend


def finish(b, lanes, point, pend, restored=()):
    """every slot of b, a copy of the fork point, takes the step that point leaves open.  Slots in restored came from
    an image: their pending c0ntinue was dropped, so they refactorize instead."""
    ks = list(range(b.nmat))
    if point == "never_factorized":
        factorize(b, lanes, ks)
    elif point == "c0ntinue":
        for k in ks:
            L = lanes[k]
            cp, ri, v = csc(L.cols)
            for o in b.slots[k]:
                if k in restored:
                    assert o.factorize_c0ntinue(cp[:-1], cp[1:], ri, v, True) == -2      # InvalidCall
                    continue
                st = 1
                for _ in range(20):      # the caller's side of lu_realloc_obj, until the factorization completes
                    o.l_mem = o.get_param("l_mem") + o.info("addmem_l") + 16
                    o.u_mem = o.get_param("u_mem") + o.info("addmem_u") + 16
                    o.w_mem = o.get_param("w_mem") + o.info("addmem_w") + 16
                    st = o.factorize_c0ntinue(cp[:-1], cp[1:], ri, v, True)
                    if st != 1:
                        break
                assert st == 0
        done = [k for k in ks if k not in restored]
        for k in done:
            cp, ri, v = csc(lanes[k].cols)
            assert lanes[k].oracle.factorize(cp[:-1], cp[1:], ri, v) == 0
            lanes[k].factored = list(lanes[k].cols)
        if len(done) < len(ks):
            factorize(b, lanes, [k for k in ks if k in restored])
        assert_getters(b, lanes)
    elif point == "pending_n":
        solve_t(b, lanes, {k: pend[0] for k in ks}, want=1)
        update(b, lanes, [k for k in ks if lanes[k].pending is not None])
    elif point == "pending_nt":
        assert update(b, lanes, ks)[0] == 0


@pytest.mark.parametrize("point", POINTS)
def test_emu_clone_fork_points(emu, point):
    """Clone at each fork point: the source's record (every getter with the times and nrealloc, every parameter, its
    image) is unchanged and the clone's equals it.  Then the source and one clone follow the same schedule in lockstep
    (bit-identical statuses, nzlhs, ilhs order, values, getters, get_factors and dense solves after every call, both
    against the oracle), while a second clone follows its own schedule against an oracle that replays the source's
    history."""
    m = 16
    lanes = [CLane(60000, m), CLane(60100, m, nslack=2, pmean=5.0, policy=1)]
    src = new_object(emu, lanes[0])
    pend = reach(Objects([[src]]), lanes, point)
    before = record(src)
    assert_same_record(before, record(src))                 # save changes nothing
    c = src.clone()
    d = src.clone()
    assert_same_record(before, record(src))                 # neither does a clone
    assert_same_record(before, record(c))
    assert_same_record(before, record(d))
    if point == "never_factorized":
        assert c.info("nupdate") == -1
    lanes[1].adopt(lanes[0])
    pair = Objects([[src, c], [d]])
    finish(pair, lanes, point, pend)
    replay(pair, lanes, 10, 60200 + POINTS.index(point), dense_every=3)
    snapshot(pair, [0, 1], seed=4, lanes=lanes)


def test_emu_clone_parameters_and_memory(emu):
    """Non-default parameters and capacities are copied exactly.  With small stores, source and clone run a long
    schedule in lockstep: every Reallocate (factorization, solve_for_update, update) fires on the same call in both,
    with the same nrealloc, and both match the oracle."""
    m = 20
    lanes = [CLane(61000, m, nslack=2, pmean=6.0)]
    src = new_object(emu, lanes[0])
    numeric = dict(droptol=1e-18, abstol=1e-13, reltol=0.2, pad=2, stretch=0.5, compress_thres=0.4, sparse_thres=0.1)
    for n, v in numeric.items():
        src.set_param(n, v)
        lanes[0].oracle.set_param(n, v)
    src.realloc_factor = 1.2
    src.tail_threads = 256
    src.split_min = 3
    src.tree_min = 64
    src.dense_k = 0
    src.l_mem, src.u_mem, src.w_mem = 3 * m, 3 * m + 1, 3 * m + 2
    factorize(Objects([[src]]), lanes, [0])
    assert src.info("nrealloc") > 0
    c = src.clone()
    assert_same_record(record(src), record(c))
    for n in list(numeric) + ["realloc_factor", "tail_threads", "split_min", "tree_min", "dense_k", "threads_per_basis"]:
        assert c.get_param(n) == src.get_param(n), n
    for n in ("l_mem", "u_mem", "w_mem"):
        assert c.get_param(n) == src.get_param(n), n
    nr = src.info("nrealloc")
    stats = replay(Objects([[src, c]]), lanes, 16, 61100, dense_every=4)
    assert src.info("nrealloc") == c.info("nrealloc") > nr
    assert stats["realloc_solve"] + stats["realloc_update"] > 0, stats
    for n in ("l_mem", "u_mem", "w_mem"):
        assert c.get_param(n) == src.get_param(n), n


def assert_same_solves(sides, seed):
    """sides = [(container, basis, lanes)]: every basis shows what the first shows -- every per-basis getter,
    get_factors, dense and sparse solves 'N' and 'T', bit for bit (the lanes' oracles run the same solves)"""
    snaps = [snapshot(c, [k], seed=seed, lanes=la)[k] for c, k, la in sides]
    for s in snaps[1:]:
        assert_same_snapshot({0: snaps[0]}, {0: s})
    rng = np.random.default_rng(seed)
    m = sides[0][0].m
    for tr in "NT":
        ir = np.sort(rng.choice(m, 3, replace=False)).astype(np.int64)
        xr = rng.uniform(-1.0, 1.0, 3)
        res = [c.solve_sparse([[(ir, xr)] if q == k else [] for q in range(c.nmat)], tr) for c, k, _ in sides]
        for (c, k, la), r in zip(sides, res):
            st0, out0 = res[0][2][sides[0][1]], res[0][1][sides[0][1]]
            assert np.array_equal(r[2][k], st0), tr
            assert all(np.array_equal(x, y) for x, y in zip(r[1][k][0], out0[0])), tr
            la[k].oracle.solve_sparse(3, ir, xr, tr)


@pytest.mark.parametrize("point", POINTS)
def test_emu_object_batch_interchange(emu, point):
    """At each fork point: object -> image -> batch slot, batch slot -> image -> another object (other capacities,
    a smaller b_nz), and object -> image -> object.  The batch slot and the objects show exactly what the source shows,
    with dense and sparse solves equal bit for bit; the object -> object round trip gives a byte-identical image; every
    one then continues against its oracle."""
    m = 16
    lanes = [CLane(62000, m), CLane(62100, m), CLane(62200, m)]
    src = new_object(emu, lanes[0])
    pend = reach(Objects([[src]]), lanes, point)
    img = src.save()
    blanes = [CLane(62300 + k, m) for k in range(3)]
    bt = BLUBatch(3, m, 4 * m + max(sum(len(r) for r, _ in L.cols) for L in blanes), lib=emu)
    bt.threads_per_basis = 64
    factorize(bt, blanes, [0, 1, 2])
    assert bt.restore([1], [img]) == 0
    blanes[1].adopt(lanes[0])
    back = bt.save([1])[0]
    o2 = new_object(emu, lanes[0], b_nz=4)
    assert o2.get_param("u_mem") != field(back, "u_mem")
    assert o2.restore(back) == 0
    for n in ("l_mem", "u_mem", "w_mem"):
        assert o2.get_param(n) == field(back, n), n
    lanes[1].adopt(lanes[0])
    o3 = new_object(emu, lanes[2])
    assert o3.restore(img) == 0
    assert np.array_equal(o3.save(), img)
    lanes[2].adopt(lanes[0])
    objs = Objects([[src], [o2], [o3]])
    assert_same_solves([(objs, 0, lanes), (bt, 1, blanes), (objs, 1, lanes), (objs, 2, lanes)], 5)
    restored = (1, 2)
    finish(objs, lanes, point, pend, restored=restored)
    if point in ("never_factorized", "c0ntinue"):      # (a batch slot has no c0ntinue: it refactorizes)
        factorize(bt, blanes, [1])
    elif point == "pending_n":
        solve_t(bt, blanes, {1: pend[0]}, want=1)
        update(bt, blanes, [k for k in (1,) if blanes[k].pending is not None])
    elif point == "pending_nt":
        assert update(bt, blanes, [1])[0] == 0
    replay(objs, lanes, 8, 62400 + POINTS.index(point), dense_every=4)
    replay(bt, blanes, 8, 62500 + POINTS.index(point), dense_every=4)


def test_emu_object_restore_rebuilds_row_wise_u(emu):
    """A restore into an object rebuilds the sorted row-wise U exactly when the basis is fresh (nupdate 0, status OK or
    WarningSingularMatrix): a batch image (where it is never built) restored into an object and saved again says
    have_ur = 1 then, 0 otherwise, and the rest of the image is unchanged."""
    m = 16
    cases = []
    for point in POINTS:
        lanes = [CLane(63000, m)]
        bt = BLUBatch(1, m, 8 * m, lib=emu)
        bt.threads_per_basis = 64
        L = lanes[0]
        if point == "singular":
            L.cols[3] = L.cols[2]
        if point != "never_factorized":
            factorize(bt, lanes, [0])
        if point == "updated":
            pend = solve_n(bt, lanes, [0])
            solve_t(bt, lanes, pend, want=0)
            update(bt, lanes, [0])
        if point in ("pending_n", "pending_nt"):
            pend = solve_n(bt, lanes, [0])
            if point == "pending_nt":
                solve_t(bt, lanes, pend, want=0)
        if point == "c0ntinue":      # (a batch has no c0ntinue: a basis that answered InvalidArgument instead)
            continue
        img = bt.save([0])[0]
        assert img[HAVE_UR:HAVE_UR + 4].view(np.int32)[0] == 0
        o = new_object(emu, L)
        assert o.restore(img) == 0
        out = o.save()
        fresh = point in ("factorized", "singular", "pending_n", "pending_nt")
        assert out[HAVE_UR:HAVE_UR + 4].view(np.int32)[0] == int(fresh), point
        x = img.copy()
        x[HAVE_UR:HAVE_UR + 4] = out[HAVE_UR:HAVE_UR + 4]
        assert np.array_equal(reseal(x), out), point
        cases.append(point)
    assert len(cases) == 6


def raw(o, fn, *args):
    return getattr(o._L, fn)(o._h, *args)


def test_emu_object_rejections(emu):
    """Every rejected call returns BLU_ERROR_INVALID_ARGUMENT, launches nothing past the check that decides, and changes
    nothing (the object's record: getters, parameters, image): NULL arguments, a batch passed to the object calls (and
    an object to the batch calls), unaligned buffers, a too small capacity, a capacity below the header, a length over
    the capacity, each header field wrong (resealed), another m, a flipped byte in each section."""
    m = 16
    lanes = [CLane(64000, m)]
    o = new_object(emu, lanes[0])
    factorize(Objects([[o]]), lanes, [0])
    pend = solve_n(Objects([[o]]), lanes, [0])
    solve_t(Objects([[o]]), lanes, pend, want=1)
    img = o.save()
    secs = sections(img)
    before = record(o)
    n0 = launches(o)
    nrej = 0
    bt = BLUBatch(2, m, 8 * m, lib=emu)
    nb = ctypes.c_int64(0)
    ref = ctypes.byref(nb)
    buf = np.zeros(len(img) + 48, np.uint8)
    al = buf.ctypes.data + (-buf.ctypes.data) % 16
    # clone
    h = ctypes.c_void_p()
    for args in ((None, o._h), (ctypes.byref(h), None), (ctypes.byref(h), bt._h)):
        assert emu.blu_clone(*args) == -4
        nrej += 1
    assert not h.value
    # save and save_dev
    for fn in ("blu_save", "blu_save_dev"):
        assert raw(o, fn, None, 0, None) == -4
        assert emu.__getattr__(fn)(None, None, 0, ref) == -4
        assert emu.__getattr__(fn)(bt._h, None, 0, ref) == -4
        assert raw(o, fn, ctypes.c_void_p(al + 4), len(img), ref) == -4          # unaligned
        nrej += 4
    assert launches(o) == n0
    assert raw(o, "blu_save", None, 0, ref) == 0 and nb.value == len(img)       # size query: k_save_extents
    assert raw(o, "blu_save", ctypes.c_void_p(al), len(img) - 16, ref) == -4 and nb.value == len(img)
    assert not buf.any()
    nrej += 1
    assert launches(o) == n0 + 2
    # restore and restore_dev: arguments
    p = ctypes.c_void_p(img.ctypes.data)
    mis = np.zeros(len(img) + 32, np.uint8)
    q = (-mis.ctypes.data) % 16 + 8
    mis[q:q + len(img)] = img
    for fn in ("blu_restore", "blu_restore_dev"):
        assert emu.__getattr__(fn)(None, p, len(img)) == -4
        assert emu.__getattr__(fn)(bt._h, p, len(img)) == -4
        assert raw(o, fn, None, len(img)) == -4
        assert raw(o, fn, ctypes.c_void_p(mis.ctypes.data + q), len(img)) == -4
        assert raw(o, fn, p, 16) == -4                                           # below the header
        nrej += 5
    assert launches(o) == n0 + 2
    assert raw(o, "blu_restore", p, len(img) - 16) == -4                          # length > cap: on the host
    assert launches(o) == n0 + 2
    assert raw(o, "blu_restore_dev", p, len(img) - 16) == -4                      # (the header gathered on the device)
    assert launches(o) == n0 + 3
    nrej += 2

    def bad(name, value):
        x = img.copy()
        set_field(x, name, value)
        return reseal(x)
    heads = [bad("magic", 0x1234), bad("version", 2), bad("m", m + 1), bad("info_bytes", int(field(img, "info_bytes")) + 8),
             bad("length", int(field(img, "length")) + 16), bad("l_n", int(field(img, "l_mem")) + 1),
             bad("u_n", int(field(img, "u_mem")) + 1), bad("w_n", int(field(img, "w_mem")) + 1), bad("bt_n", -1),
             bad("l_mem", int(field(img, "l_n")) - 1)]
    for x in heads:
        assert o.restore(x) == -4
        assert o.restore_dev(torch.as_tensor(x)) == -4
        nrej += 2
    assert launches(o) == n0 + 3 + len(heads)
    other = CLane(64100, m + 4)
    g = new_object(emu, other)
    factorize(Objects([[g]]), [other], [0])
    assert o.restore(g.save()) == -4                                              # another m
    nrej += 1
    n1 = launches(o)
    for name, off, n in secs:
        if n == 0:
            continue
        x = img.copy()
        x[off + n // 2 if name != "header" else INFO_AT + 4 * 7] ^= 0x10
        assert o.restore_dev(torch.as_tensor(x)) == -4, name
        assert o.restore(x) == -4, name
        nrej += 2
    nsec = sum(1 for s in secs if s[2])
    assert launches(o) == n1 + 2 * 3 * nsec                                       # headers, checksum, verdict
    x = img.copy(); x[len(img) - 1] ^= 1                                          # the last padding byte
    assert o.restore(x) == -4
    nrej += 1
    assert_same_record(before, record(o))
    # the batch calls keep refusing objects
    assert emu.blu_batch_save(o._h, 0, None, None, None, None) == -4
    assert emu.blu_batch_restore(o._h, 0, None, None, None) == -4
    assert emu.blu_batch_copy(o._h, 0, None, None) == -4
    # and the image restores: launches of a restore into an object (the batch's eight and k_build_ur)
    n2 = launches(o)
    assert o.restore_dev(torch.as_tensor(img)) == 0
    assert launches(o) == n2 + 9
    assert_same_record(before, record(o))
    print(f"rejections checked: {nrej}")
    assert nrej >= 60


def test_emu_object_host_traffic(emu_traffic):
    """save_dev copies the image size to the host and nothing else; restore_dev the header and two fixed-size
    summaries: the same at two dimensions, and what the batch calls copy for one basis"""
    emu = emu_traffic
    per = {}
    c = (ctypes.c_ulonglong * 5)()
    for m in (16, 40):
        lanes = [CLane(65000 + m, m)]
        o = new_object(emu, lanes[0])
        factorize(Objects([[o]]), lanes, [0])
        emu.cuda_emu_memcpy_reset()
        img = o.save_dev()
        emu.cuda_emu_memcpy_bytes(c)
        assert c[2] == 2 * 8, c[2]                   # (the size query, then the save)
        emu.cuda_emu_memcpy_reset()
        assert o.restore_dev(img) == 0
        emu.cuda_emu_memcpy_bytes(c)
        per[m] = c[2] - header_bytes(img.numpy())
        bt = BLUBatch(2, m, 8 * m, lib=emu)
        emu.cuda_emu_memcpy_reset()
        assert bt.restore_dev([1], [img]) == 0
        emu.cuda_emu_memcpy_bytes(c)
        assert c[2] - header_bytes(img.numpy()) == per[m]
    assert per[16] == per[40] <= 128, per


def test_emu_clone_c_program(emu, tmp_path):
    """tests/abi/clone_check.c, plain C99 against include/blu_b200.h: clones the 10 x 10 example, moves it through an
    image, and gets the same solution bit for bit from all three objects"""
    exe = str(tmp_path / "clone_check")
    lib = os.path.join(HERE, "emu")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(HERE, "abi", "clone_check.c"), "-L", lib, "-lblu_emu", "-Wl,-rpath," + lib, "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "solve alike" in out.stdout


@pytest.mark.parametrize("env,case", [("EMU_SEED=1", "test_emu_clone_fork_points[pending_nt]"),
                                      ("EMU_STRICT=1", "test_emu_object_batch_interchange[updated]")])
def test_emu_clone_env(env, case):
    """a clone at the 'N' + 'T' fork point under a shuffled lane order, and the interchange after updates under the
    strict barrier check"""
    k, v = env.split("=")
    r = subprocess.run([os.sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider",
                        os.path.abspath(__file__) + "::" + case],
                       env=dict(os.environ, **{k: v}), cwd=HERE, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
