"""blu_batch_maxvolume at scale: 1,024 bases of configs[1]'s shape (2,000 x 2,000, gen.batch(nmat, 2000, 700, 5.0,
...)), each with 500 fresh candidate columns, one maxvolume pass on every basis (maxvolume.rs:64-224).

GPU arm: the wall time of one blu_batch_maxvolume call (a host clock around the call, which ends in a stream
synchronise), after a warm-up call on a small batch.  CPU arm: the oracle's blo_maxvolume on the same pools, one
basis per task on a thread pool over every core (ctypes releases the GIL).  Every basis' status, nupdate, basis and
isbasic are compared between the two, and the LU getters for a sample of bases.  The card's name and power limit are
read with nvidia-smi in the same run.  Prints one JSON object and writes it to --out."""
import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from blu_b200 import BLUBatch  # noqa: E402
from mv_cases import GETTERS, config1_pools, layout, oracle_maxvolume  # noqa: E402


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return name, power


def gpu_pass(pools, volumetol):
    m = pools[0].m
    b = BLUBatch(len(pools), m, max(int(np.diff(p.a_p[:m + 1]).sum()) for p in pools), device=0)
    ab, ae, ai, ax, basis, isbasic = layout(pools)
    l0 = b.launch_count()
    t0 = time.perf_counter()
    st, status, nup = b.maxvolume(pools[0].ncol, ab, ae, ai, ax, basis, isbasic, volumetol)
    dt = time.perf_counter() - t0
    return b, dict(seconds=dt, st=int(st), status=status, nupdate=nup, launches=int(b.launch_count() - l0),
                   basis=basis.reshape(len(pools), m), isbasic=isbasic.reshape(len(pools), -1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmat", type=int, default=1024)
    ap.add_argument("--ncand", type=int, default=500)
    ap.add_argument("--volumetol", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sample", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = gpu_card()
    pools = config1_pools(a.nmat, a.ncand, 9000)
    m = pools[0].m

    gpu_pass(config1_pools(8, 50, 100), a.volumetol)      # warm-up: module load, first launches
    runs = []
    for _ in range(a.reps):
        b, r = gpu_pass(pools, a.volumetol)
        runs.append(r)
    gsec = [r["seconds"] for r in runs]
    r = runs[-1]
    nfact = np.array([b.info(k, "nfactorize") for k in range(a.nmat)])

    def oracle(p):
        # the oracle object is dropped here: 1,024 of them at once would not fit in host memory
        o, ost, onup, obasis, oisbasic = oracle_maxvolume(p, a.volumetol)
        return {g: o.info(g) for g in GETTERS}, ost, onup, obasis, oisbasic

    workers = os.cpu_count() or 1
    t0 = time.perf_counter()
    with concurrent.futures.ThreadPoolExecutor(max_workers=workers) as ex:
        ores = list(ex.map(oracle, pools))
    csec = time.perf_counter() - t0

    mism = [k for k, (o, ost, onup, obasis, oisbasic) in enumerate(ores)
            if not (r["status"][k] == ost and r["nupdate"][k] == onup and np.array_equal(r["basis"][k], obasis)
                    and np.array_equal(r["isbasic"][k], oisbasic))]
    sample = np.random.default_rng(11).choice(a.nmat, min(a.sample, a.nmat), replace=False)
    getter_mism = [int(k) for k in sample if any(b.info(int(k), g) != ores[k][0][g] for g in GETTERS)]
    examined = a.nmat * a.ncand     # the candidates are never basic when the pass reaches them
    res = dict(
        workload=f"{a.nmat} bases of configs[1]'s shape (m={m}, gen.basis(seed, 2000, 700, 5.0)), {a.ncand} fresh "
                 f"candidate columns each (8 entries, values x3), volumetol {a.volumetol}",
        card=name, power_limit=power,
        gpu_call_seconds=gsec, gpu_call_seconds_min=min(gsec),
        gpu_us_per_examined_column_per_basis=1e6 * min(gsec) / examined,
        gpu_launches_per_call=r["launches"],
        cpu_oracle_seconds=csec, cpu_threads=workers,
        cpu_us_per_examined_column_per_basis=1e6 * csec / examined,
        gpu_over_cpu_speedup=csec / min(gsec),
        status_ok=int((r["status"] == 0).sum()), updates_total=int(r["nupdate"].sum()),
        updates_min_per_basis=int(r["nupdate"].min()),
        refactorizations_in_pass=int((nfact - 1).clip(0).sum()),
        parity_all_bases_status_nupdate_basis_isbasic=len(mism) == 0, parity_mismatches=mism[:10],
        parity_getters_sampled_bases=[int(k) for k in sample], parity_getters_ok=len(getter_mism) == 0,
    )
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")
    return 0 if not mism and not getter_mism else 1


if __name__ == "__main__":
    sys.exit(main())
