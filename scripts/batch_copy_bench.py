"""blu_batch_copy at scale: 4,096 bases of configs[1]'s shape (gen.batch(4096, 2000, 700, 5.0)), factorized and given a
few basis changes each, then copied in two patterns:
  (a) 64 parents, each to 63 children (the parents are bases 0, 64, 128, ...; a parent's children follow it);
  (b) bases 0..2047 to 2048..4095.
Beside each, factorize_subset_dev of the same destinations from their parents' B, already in device memory (so no
upload is timed) -- what a driver does without the copy, and which does not even carry the update history.

Times are CUDA events on the batch stream around the call (warm-up first, best and median of --reps), with the card's
name and power limit read with nvidia-smi in the same run.

Bytes: per destination, the live state the copy reads and writes, computed from the source's getters with the extents
rule of blu_copy.cuh.  Entries are 4-byte index + 8-byte value = 12 bytes:
  L = 2 * (l_nz + m) + r_nz entries   (column-wise and row-wise L with their unit diagonals, and the row etas)
  U = u_nz + m entries                (columns of U; replaced columns left behind by updates are not counted)
  W = u_nz + m entries                (the row file of U in the live half; the gaps between its lines are not counted)
  Bt = matrix_nz entries              (the row-wise copy of B)
plus the O(m) arrays (state_words(m) * 4 bytes), BluInfo and two resident B rows (16 * m bytes).  Each byte is read once
and written once, so the traffic is twice that; it is a lower bound on what the kernel moves.  Prints one JSON line."""
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


def state_words(m):
    """4-byte words of the O(m) arrays k_copy_slots copies (blu_copy.cuh) and of BluInfo (about 200 words)"""
    ints = (m + 1) + 4 * m + 6 * m + 8 * (m + 1) + 4 * m + 2 * (2 * m + 2) + 3 * m + (2 * m + 2) + 2 * m + (4 * m + 4)
    return ints + 2 * (2 * m) + 2 * (2 * m) + 2 * m + 200


def live_bytes(b, k, m):
    g = {n: b.info(k, n) for n in ("l_nz", "u_nz", "r_nz", "matrix_nz")}
    entries = 2 * (g["l_nz"] + m) + g["r_nz"] + 2 * (g["u_nz"] + m) + g["matrix_nz"]
    return 12 * entries + 4 * state_words(m) + 16 * m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmat", type=int, default=4096)
    ap.add_argument("--m", type=int, default=2000)
    ap.add_argument("--nslack", type=int, default=700)
    ap.add_argument("--rounds", type=int, default=3, help="basis changes every basis gets before the copies")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=71000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    name, power = gpu_card()
    n, m = a.nmat, a.m
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
    nup = [b.info(k, "nupdate") for k in range(0, n, 97)]
    stream = torch.cuda.ExternalStream(b._L.blu_batch_stream(b._h), device=torch.device("cuda", 0))

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

    per = 2 if n >= 2 else 1
    npar = min(64, n // 2)
    kids = n // npar - 1
    pat = {
        "a_64x63": ([p * (kids + 1) + 1 + q for p in range(npar) for q in range(kids)], [p * (kids + 1) for p in range(npar) for _ in range(kids)]),
        "b_half": (list(range(n // per, n)), list(range(n // per))),
    }
    res = dict(card=name, power_limit=power, nmat=n, m=m, nslack=a.nslack, rounds=a.rounds, reps=a.reps, sample_nupdate=nup)
    dev = torch.device("cuda", 0)
    tbi, tbx = torch.as_tensor(bi).to(dev), torch.as_tensor(bx).to(dev)
    for key, (dst, src) in pat.items():
        byt = sum(live_bytes(b, s, m) for s in src)
        t = timed(lambda: b.copy(dst, src))
        # the B each source was last factorized from (the batch was factorized from gen.batch), in the per-basis layout
        # of factorize_subset_dev: destination d reads its source's columns
        pb, pe = bb.copy(), be.copy()
        run = np.zeros(n, np.int32)
        for d, s in zip(dst, src):
            pb[d * m:(d + 1) * m] = bb[s * m:(s + 1) * m]
            pe[d * m:(d + 1) * m] = be[s * m:(s + 1) * m]
            run[d] = 1
        tb, te, tr = torch.as_tensor(pb).to(dev), torch.as_tensor(pe).to(dev), torch.as_tensor(run).to(dev)
        torch.cuda.synchronize(dev)
        f = timed(lambda: b.factorize_subset_dev(tb, te, tbi, tbx, run=tr))
        res[key] = dict(ncopy=len(dst), copy=t, bytes_state=int(byt), bytes_moved=int(2 * byt),
                        copy_gb_per_s=2 * byt / (t["best_ms"] * 1e-3) / 1e9, factorize_subset_dev=f,
                        factorize_over_copy=f["best_ms"] / t["best_ms"])
        print(json.dumps({key: res[key]}), flush=True)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
