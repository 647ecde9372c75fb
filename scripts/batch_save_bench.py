"""blu_batch_save / blu_batch_restore at scale: 4,096 bases of configs[1]'s shape (gen.batch(4096, 2000, 700, 5.0)), each
factorized and given three basis changes (the setup of batch_copy_bench.py).  Timed, with CUDA events on the batch
stream, best and median of --reps after a warm-up:
  - save_dev of all 4,096 bases and of 64 (the parents 0, 64, 128, ...), into preallocated device buffers;
  - restore_dev of the 64 parents' images into the 4,032 other slots (each image to the 63 slots after its parent), and
    of all 4,096 images into their own slots;
  - copy of the same 4,032 pairs;
  - factorize_subset_dev of the same destinations from their sources' B, already in device memory (no upload timed);
  - the host save and restore of 256 bases (pageable numpy buffers).
Bytes: image bytes read plus written, over the call's time (save reads the basis' live state and writes its image;
restore reads the image twice -- checksum and copy -- and writes the state; counted here once each way, so a lower
bound).  After the fan-out restore every restored basis' dense solves ('N' and 'T') are checked equal to its source's.
The card's name and power limit are read with nvidia-smi in the same run.  Prints one JSON line (and writes --out)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from blu_b200 import BLUBatch, gen  # noqa: E402


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmat", type=int, default=4096)
    ap.add_argument("--m", type=int, default=2000)
    ap.add_argument("--nslack", type=int, default=700)
    ap.add_argument("--rounds", type=int, default=3, help="basis changes every basis gets first")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host", type=int, default=256, help="bases of the host save / restore")
    ap.add_argument("--seed", type=int, default=71000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ctypes
    import torch
    name, power = gpu_card()
    n, m = a.nmat, a.m
    dev = torch.device("cuda", 0)
    bb, be, bi, bx, _ = gen.batch(n, m, a.nslack, 5.0, a.seed, a.seed + 10000)
    b = BLUBatch(n, m, int((be - bb).reshape(n, m).sum(1).max()) + 4 * m, device=0)
    st, status = b.factorize(bb, be, bi, bx)
    assert st == 0 and (status == 0).all()
    for r in range(a.rounds):
        cols = []
        for k in range(n):
            cp, ri, v = gen.basis(a.seed + 20000 + r * n + k, m, 0, 3.0)
            cols.append((ri[cp[0]:cp[1]], v[cp[0]:cp[1]]))
        st, stat, out = b.solve_for_update(cols, "N", want_solution=1)
        leave = [(np.array([int(out[k][0][np.argmax(np.abs(out[k][1]))]) if len(out[k][0]) else 0]), None) for k in range(n)]
        xt = np.array([out[k][1][np.argmax(np.abs(out[k][1]))] if len(out[k][1]) else 1.0 for k in range(n)])
        b.solve_for_update(leave, "T")
        b.update(xt)
    stream = torch.cuda.ExternalStream(b._L.blu_batch_stream(b._h), device=dev)

    def timed(fn):
        fn()
        ms = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            r = fn()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
            assert (r if isinstance(r, int) else r[0]) == 0, r
        return dict(best_ms=min(ms), median_ms=float(np.median(ms)))

    L = b._L
    everyone = list(range(n))
    _, size = b._save(L.blu_batch_save_dev, everyone, None)
    size = [int(s) for s in size]
    stride = [(s + 255) & ~255 for s in size]
    block = torch.empty(sum(stride) + 256, dtype=torch.uint8, device=dev)
    at, imgs = (-block.data_ptr()) % 256, []
    for s, z in zip(size, stride):
        imgs.append(block[at:at + s])
        at += z
    res = dict(card=name, power_limit=power, nmat=n, m=m, nslack=a.nslack, rounds=a.rounds, reps=a.reps,
               image_bytes=dict(mean=float(np.mean(size)), max=int(max(size)), min=int(min(size))))

    def save_dev(idx):
        return b._save(L.blu_batch_save_dev, idx, [(imgs[k].data_ptr(), imgs[k].numel()) for k in idx])

    npar = 64
    kids = n // npar - 1
    parents = [p * (kids + 1) for p in range(npar)]
    dst = [p * (kids + 1) + 1 + q for p in range(npar) for q in range(kids)]
    src = [p * (kids + 1) for p in range(npar) for _ in range(kids)]
    tot_all, tot_par = sum(size), sum(size[p] for p in parents)
    res["save_dev_all"] = t = timed(lambda: save_dev(everyone))
    t["bytes"] = 2 * tot_all; t["gb_per_s"] = 2 * tot_all / (t["best_ms"] * 1e-3) / 1e9
    res["save_dev_64"] = t = timed(lambda: save_dev(parents))
    t["bytes"] = 2 * tot_par; t["gb_per_s"] = 2 * tot_par / (t["best_ms"] * 1e-3) / 1e9
    print(json.dumps({k: res[k] for k in ("image_bytes", "save_dev_all", "save_dev_64")}), flush=True)
    assert save_dev(everyone)[0] == 0
    I64P = ctypes.POINTER(ctypes.c_int64)

    def restore_call(dd, ts):
        """blu_batch_restore_dev with its arrays made once, outside the timed window"""
        d = np.array(dd, np.int64)
        ptrs = (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
        cap = np.array([t.numel() for t in ts], np.int64)
        return lambda: L.blu_batch_restore_dev(b._h, len(d), d.ctypes.data_as(I64P), ptrs, cap.ctypes.data_as(I64P))
    par_imgs = [imgs[s] for s in src]
    x = np.tile(np.random.default_rng(5).uniform(-1, 1, m), n)
    before = {tr: b.solve_dense(x, tr)[1] for tr in "NT"}
    res["restore_dev_64_to_4032"] = t = timed(restore_call(dst, par_imgs))
    fan = sum(size[s] for s in src)
    t["bytes"] = 2 * fan; t["gb_per_s"] = 2 * fan / (t["best_ms"] * 1e-3) / 1e9
    after = {tr: b.solve_dense(x, tr)[1] for tr in "NT"}
    ok = all(np.array_equal(after[tr][d], before[tr][s]) for tr in "NT" for d, s in zip(dst, src)) and \
        all(np.array_equal(after[tr][p], before[tr][p]) for tr in "NT" for p in parents)
    res["dense_solves_equal_sources"] = bool(ok)
    res["copy_64_to_4032"] = timed(lambda: b.copy(dst, src))
    res["restore_dev_all"] = t = timed(restore_call(everyone, imgs))
    t["bytes"] = 2 * tot_all; t["gb_per_s"] = 2 * tot_all / (t["best_ms"] * 1e-3) / 1e9
    print(json.dumps({k: res[k] for k in ("restore_dev_64_to_4032", "dense_solves_equal_sources", "copy_64_to_4032", "restore_dev_all")}), flush=True)
    # factorize_subset_dev of the same destinations, each from its source's B (the batch's B is gen.batch's, restores
    # and copies keep every basis' B its source's)
    tbi, tbx = torch.as_tensor(bi).to(dev), torch.as_tensor(bx).to(dev)
    for key, (dd, ss) in {"64_to_4032": (dst, src), "all": (everyone, everyone)}.items():
        pb, pe = bb.copy(), be.copy()
        run = np.zeros(n, np.int32)
        for d, s in zip(dd, ss):
            pb[d * m:(d + 1) * m] = bb[s * m:(s + 1) * m]
            pe[d * m:(d + 1) * m] = be[s * m:(s + 1) * m]
            run[d] = 1
        tb, te, tr = torch.as_tensor(pb).to(dev), torch.as_tensor(pe).to(dev), torch.as_tensor(run).to(dev)
        torch.cuda.synchronize(dev)
        res["factorize_subset_dev_" + key] = f = timed(lambda: b.factorize_subset_dev(tb, te, tbi, tbx, run=tr))
        r = res["restore_dev_" + ("64_to_4032" if key == "64_to_4032" else "all")]
        r["factorize_subset_dev_over_restore"] = f["best_ms"] / r["best_ms"]
        print(json.dumps({"factorize_subset_dev_" + key: f}), flush=True)
    # the host variants, 256 bases
    hidx = list(range(a.host))
    himg = [b._aligned_host(size[k]) for k in hidx]
    hbufs = [(h.ctypes.data, h.size) for h in himg]
    res["save_host_%d" % a.host] = t = timed(lambda: b._save(L.blu_batch_save, hidx, hbufs))
    hb = sum(size[k] for k in hidx)
    t["bytes"] = hb; t["gb_per_s"] = hb / (t["best_ms"] * 1e-3) / 1e9
    ptrs = (ctypes.c_void_p * len(hidx))(*[h.ctypes.data for h in himg])
    cap = np.array([h.size for h in himg], np.int64)
    hd = np.array(hidx, np.int64)
    res["restore_host_%d" % a.host] = t = timed(lambda: L.blu_batch_restore(b._h, len(hd), hd.ctypes.data_as(I64P), ptrs, cap.ctypes.data_as(I64P)))
    t["bytes"] = hb; t["gb_per_s"] = hb / (t["best_ms"] * 1e-3) / 1e9
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
