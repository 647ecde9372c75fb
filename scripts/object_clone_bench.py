"""blu_clone and object images at configs[2]'s shape (gen.config3: 100,000 rows, a 4,000-wide bump that fills to full
density; the stores of scripts/configs_bench.py), after 0 and after --updates column replacements (solve_for_update
'N' + 'T', update, entering columns from gen.column_pool).  Timed with a host clock around each call, which returns
only after its work on the device is done, best and median of --reps after a warm-up:
  - clone: blu_clone (the clone is destroyed between repetitions, outside the timed window);
  - save_dev: blu_save_dev into a preallocated device buffer;
  - restore_dev: blu_restore_dev of that image into a second object of the same capacities;
  - factorize: blu_factorize of the same B from host arrays, which is what a clone or a restore replaces.
Bytes: the image bytes.  Clone writes the image and reads it back (and copies the sorted row-wise U beside it when the
basis is fresh); save_dev writes it once; restore_dev reads it twice (checksum, restore).  After each clone, the clone's
dense solve ('N') is checked equal to the source's, bit for bit.  The card's name and power limit are read with
nvidia-smi in the same run.  Prints one JSON line (and writes --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from blu_b200 import BLU, gen  # noqa: E402


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return name, power


def timed(fn, reps, sync):
    fn()      # warm-up
    ts = []
    for _ in range(reps):
        sync()
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t0)
    return {"best_ms": 1e3 * min(ts), "median_ms": 1e3 * float(np.median(ts))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=100000)
    ap.add_argument("--bump", type=int, default=4000)
    ap.add_argument("--updates", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    name, power = gpu_card()
    m, bump = a.m, a.bump
    cp, ri, v = gen.config3(m, bump)
    pcp, pri, pv = gen.column_pool(4101, m, a.updates)
    dense = bump * bump
    mem = (int(2.2 * (dense // 2 + 10 * m)) + 40 * m, int(1.2 * (dense // 2 + 10 * m)) + 40 * m, int(3.0 * dense + 40 * m))

    def make():
        g = BLU(m, len(v), device=0)
        g.threads_per_basis = 1024
        g.l_mem, g.u_mem, g.w_mem = mem
        return g

    sync = torch.cuda.synchronize
    g, other = make(), make()
    b = gen.rhs(4002, m)
    rec = {"what": "blu_clone / blu_save_dev / blu_restore_dev of one object at configs[2]'s shape, against blu_factorize",
           "gpu": name, "power_limit": power, "m": m, "bump": bump, "reps": a.reps, "timing": "host clock around each call, best / median",
           "points": []}
    assert g.factorize(cp[:-1], cp[1:], ri, v) == 0
    fact = timed(lambda: g.factorize(cp[:-1], cp[1:], ri, v), a.reps, sync)
    launches = g._L.blu_batch_launch_count
    for nupd in (0, a.updates):
        if nupd:
            for it in range(nupd):
                idx, val = pri[pcp[it]:pcp[it + 1]], pv[pcp[it]:pcp[it + 1]]
                assert g.solve_for_update(len(idx), idx, val, "N", 1) == 0
                j = int(np.argmax(np.abs(g.lhs)))
                xt = g.lhs[j]
                assert g.solve_for_update(1, np.array([j]), None, "T", 0) == 0
                assert g.update(xt) == 0
        _, x0 = g.solve_dense(b, "N")
        clones = []

        def clone():
            clones.append(g.clone())
        n0 = launches(g._h)
        t_clone = timed(clone, a.reps, sync)
        src_launches = (launches(g._h) - n0) // (a.reps + 1)
        clone_launches = launches(clones[0]._h)
        same = all(np.array_equal(c.solve_dense(b, "N")[1], x0) for c in clones)
        for c in clones:
            c.close()
        img = g.save_dev()
        t_save = timed(lambda: g.save_dev(), a.reps, sync)
        t_restore = timed(lambda: other.restore_dev(img), a.reps, sync)
        assert other.restore_dev(img) == 0
        same = same and np.array_equal(other.solve_dense(b, "N")[1], x0)
        nbytes = int(img.numel())
        pt = {"nupdate": int(g.info("nupdate")), "image_bytes": nbytes,
              "clone": dict(t_clone, launches_on_source=int(src_launches), launches_on_clone=int(clone_launches),
                            image_bytes_moved=2 * nbytes),
              "save_dev": dict(t_save, gb_per_s=nbytes / (1e-3 * t_save["best_ms"]) / 1e9),
              "restore_dev": dict(t_restore, gb_per_s=2 * nbytes / (1e-3 * t_restore["best_ms"]) / 1e9),
              "factorize": fact if nupd == 0 else None,
              "clone_over_factorize": t_clone["best_ms"] / fact["best_ms"],
              "dense_solves_bit_identical": bool(same)}
        rec["points"].append(pt)
        del img
    rec["factorize"] = fact
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
