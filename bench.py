#!/usr/bin/env python
"""bench.py -- headline benchmark of the BLU hot path on B200 (BASELINE.json `metric`).

Workload (BASELINE.json configs[1]): a batch of 4,096 independent 2,000 x 2,000 simplex-style
bases (35 % slack columns, structural columns 1+Poisson(5) entries, synthetic, seeded), each
basis = factorize + solve_dense('N').  A *step* is one pass over the whole batch.  The bases
shard across GPUs by index with no data-path collective (SURVEY.md 8e, blu_b200/shard.py): under
torchrun the ONE 4,096-basis batch of BASELINE.json is split into contiguous ranges of 4096/N bases
per rank ("strong" scaling, the default; --scaling weak gives every rank its own 4,096) and `value` is
all ranks' bases divided by the max-over-ranks device time.

    python bench.py [--gpus N] [--steps K] [--warmup W]         # the CUDA path (libblu_b200.so)
    python bench.py --impl reference ...                         # the CPU restatement of rwl/blu
    python bench.py ... --dump-outputs DIR                       # also write the last timed step's outputs (dump_outputs)

The reference is a Rust crate and this image has no Rust toolchain, so `--impl reference` and the
`cpu_baseline` leg time oracle/ (the C restatement, kind "port"), one instance per host core.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "factorize+solve matrices/sec (batched)"
UNIT = "matrices/s"
M, NSLACK, PMEAN = 2000, 700, 5.0
DUMP_BYTES = 48 * 10**6      # --dump-outputs: solutions beyond this are sampled, so that a dump stays under 64 MB
DUMP_INFO = ["rank", "l_nz", "u_nz", "min_pivot", "max_pivot", "condest_l", "condest_u", "onenorm", "infnorm", "residual_test"]


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy bandwidth, burst)"
        except Exception:
            pass
    return 6500.0, "fallback of /opt/skills/guides/B200_PROFILING.md (no MEASURED_PEAKS.json)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def algorithmic_bytes(b, nmat, m):
    """SURVEY.md 8(d): bytes(factorize) = singletons + setup_bump + elimination + build_factors, from
    the device's own counters (the same ones the oracle keeps); 12 B per stored nonzero, 4 B per
    pattern index or pointer, 8 B per vector element.  Returns (whole factorization, the part done by the
    head launch of a split factorization = singletons + setup_bump + its share of the elimination,
    solve_dense)."""
    tot_f = tot_h = tot_s = 0.0
    for k in range(nmat):
        nnz = b.info(k, "matrix_nz"); lnz = b.info(k, "l_nz"); unz = b.info(k, "u_nz")
        bump_nz = b.info(k, "bump_nz"); bump = b.info(k, "bump_size")
        sing = 36.0 * nnz + 12.0 * max(nnz - bump_nz, 0.0) + 16.0 * m   # nnzL0+nnzU0 <= nnz - bump_nz
        setup = 12.0 * bump_nz + 16.0 * bump_nz + 16.0 * bump
        build = 48.0 * (lnz + unz) + 40.0 * m
        tot_f += sing + setup + b.info(k, "elim_bytes") + build
        tot_h += sing + setup + b.info(k, "elim_bytes_head")
        tot_s += 12.0 * (lnz + unz) + 24.0 * m + 12.0 * m
    return tot_f, tot_h, tot_s


def kernel_source_hash():
    """Identifies the kernel sources a profile was taken with (profiles/traffic.json is only quoted when
    it matches the sources being benchmarked)."""
    import glob
    import hashlib
    h = hashlib.sha1()
    for f in sorted(glob.glob(os.path.join(ROOT, "blu_b200", "csrc", "*.cu*")) + glob.glob(os.path.join(ROOT, "blu_b200", "csrc", "*.h"))):
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def dump_outputs(out_dir, x, status, info=None):
    """What the last timed step returned, as float64 .npy files, so that two builds can be compared output for output
    on the same seeded inputs.  x.npy holds the solutions [bases, m] of every basis, or of a fixed seeded sample of
    them when all of them would exceed DUMP_BYTES; bases.npy gives their indices in the batch.  status.npy and
    factor_info.npy (the per-basis getters DUMP_INFO, one column each) cover every basis."""
    n, m = x.shape
    keep = max(1, DUMP_BYTES // (8 * m))
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    out = {"x": x[idx], "bases": idx, "status": status}
    if info is not None:
        out["factor_info"] = info
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def run_reference(args, rank, world):
    if rank != 0:
        return
    import oracle_lib
    from blu_b200 import gen
    cores = host_cores()
    nsample = int(min(args.nmat, max(cores * args.ref_per_core, 8)))
    bb, be, bi, bx, rhs = gen.batch(nsample, M, NSLACK, PMEAN, 2000, 3000)
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        nt, x, st = oracle_lib.batch_factorize_solve(nsample, M, bb, be, bi, bx, rhs, nthreads=cores, check_file_diff=1)
        dt = time.perf_counter() - t0
        assert (st == 0).all()
        if it >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x, st)
    T = sum(times)
    value = nsample * len(times) / T
    sample = f"{nsample} of the {args.nmat} bases per step (seeds 2000..), factorize+solve_dense each, {nt} threads, file_diff asserts on (setup_bump.rs:228-251)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * T / len(times), "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]: 4096 x (2000x2000 simplex-style basis, ~6 nnz/col) factorize+solve_dense",
                       "m": M, "bases": args.nmat, "reference_arm": "CPU only: rwl/blu restated in C (oracle/), no Rust toolchain in the image; "
                       "one instance per host core of this box whatever --gpus says (rank 0 alone runs it)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nt, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nmat", type=int, default=4096, help="bases of the batch (strong scaling: in all; weak: per GPU)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--dense-k", type=int, default=-1, help="dense-tail order (library default if < 0)")
    ap.add_argument("--dense-k-big", type=int, default=-1, help="order of the HBM/L2 stage in front of the shared-memory dense tail (library default if < 0, 0 = none)")
    ap.add_argument("--threads-per-basis", type=int, default=0)
    ap.add_argument("--ref-per-core", type=int, default=16, help="bases per host core in one reference step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    # stdout carries exactly ONE line, the JSON record: everything else that libraries print there
    # (NCCL prints its version banner on stdout) is sent to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from blu_b200 import BLUBatch, gen
    from blu_b200.shard import gather_rows, shard_range

    if args.scaling == "strong":
        lo, hi = shard_range(args.nmat, rank, world)      # rank's contiguous range of the ONE batch
        total = args.nmat
    else:
        lo, hi = rank * args.nmat, (rank + 1) * args.nmat
        total = args.nmat * world
    nmat = hi - lo
    t0 = time.time()
    bb, be, bi, bx, rhs = gen.batch(nmat, M, NSLACK, PMEAN, 2000 + lo, 3000 + lo)
    t_gen = time.time() - t0
    cap = int((be - bb).reshape(nmat, M).sum(1).max())

    # pinned host staging for the end-to-end leg
    def pin(a):
        t = torch.from_numpy(a).pin_memory()
        return t, t.numpy()
    keep = [pin(a) for a in (bb, be, bi, bx, rhs)]
    pbb, pbe, pbi, pbx, prhs = [k[1] for k in keep]
    lhs_t = torch.empty(nmat * M, dtype=torch.float64).pin_memory()

    # default store sizes (BLU::new-style, blu_host.cu create_common): a basis that needs more gets private
    # stores and re-runs alone (blu.rs:95-118), during the warm-up steps
    b = BLUBatch(nmat, M, cap, device=local)
    if args.threads_per_basis:
        b.threads_per_basis = args.threads_per_basis
    if args.dense_k >= 0:
        b.dense_k = args.dense_k
    if args.dense_k_big >= 0:
        b.dense_k_big = args.dense_k_big
    stream = torch.cuda.Stream()
    b.set_stream(stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def resident_step():
        st = b.factorize_resident()
        assert st == 0, st
        st = b.solve_dense_resident("N")
        assert st == 0, st

    # ---------------- device-resident throughput (`value`) ----------------
    assert b.upload(pbb, pbe, pbi, pbx, prhs) == 0
    for _ in range(args.warmup):
        resident_step()
    nrealloc = int(b.info(0, "nrealloc"))      # bases that outgrew the default stores got private ones in the first pass
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = b.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fact_ms, head_ms, tail_ms, build_ms, norms_ms = [], [], [], [], []
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            resident_step()
            fact_ms.append(b.last_kernel_ms(0) - b.last_kernel_ms(2))   # the k_factorize launches (2 = the condest/residual kernel)
            head_ms.append(b.last_kernel_ms(3)); tail_ms.append(b.last_kernel_ms(4)); build_ms.append(b.last_kernel_ms(5))
            norms_ms.append(b.last_kernel_ms(2))
        e1.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = b.launch_count() - l0
    ms = e0.elapsed_time(e1)
    _, x, status = b.download()
    nbad = int((status != 0).sum())
    assert nbad == 0, f"{nbad} bases did not solve"
    nrealloc_after = int(b.info(0, "nrealloc"))
    if args.dump_outputs:
        info = np.array([[b.info(k, n) for n in DUMP_INFO] for k in range(nmat)])
        x_all, status_all, info_all = (gather_rows(a, total) for a in (x, status, info))
        if rank == 0:
            dump_outputs(args.dump_outputs, x_all, status_all, info_all)

    # ---------------- end to end through the C ABI with host buffers ----------------
    import ctypes
    from blu_b200.blu import _pi, _pf, i32p
    stat = np.zeros(nmat, dtype=np.int32)
    lhs_np = lhs_t.numpy()

    def e2e_step():
        st = b._L.blu_batch_factorize(b._h, _pi(pbb), _pi(pbe), _pi(pbi), _pf(pbx), len(pbi), stat.ctypes.data_as(i32p))
        assert st == 0, st
        st = b._L.blu_batch_solve_dense(b._h, _pf(prhs), _pf(lhs_np), b"N", stat.ctypes.data_as(i32p))
        assert st == 0, st

    e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        f0.record(stream)
        for _ in range(args.steps):
            e2e_step()
        f1.record(stream)
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    h2d = int(pbb.nbytes + pbe.nbytes + pbi.nbytes + pbx.nbytes + prhs.nbytes)
    d2h = int(lhs_np.nbytes + stat.nbytes + nmat * 8 * 40)

    # max over ranks
    if world > 1:
        t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])

    if rank == 0:
        value = total * args.steps / (ms * 1e-3)
        e2e_value = total * args.steps / (ms_e2e * 1e-3)
        bytes_f, bytes_h, bytes_s = algorithmic_bytes(b, nmat, M)
        peak, peak_src = peaks()
        split = float(np.mean(tail_ms)) > 0.0
        # the dominant kernel: the longer of the two big launches of the split factorization -- HEAD (singletons, bump
        # set-up and the sparse part of the elimination) or TAIL (the dense tail: first stage in HBM/L2, second in
        # shared memory, and the last sparse pivots); not split: the one k_factorize launch with everything in it
        hm, tm = float(np.mean(head_ms)), float(np.mean(tail_ms))
        build_b = bytes_f - sum(b.info(k, "elim_bytes") for k in range(nmat)) - (bytes_h - sum(b.info(k, "elim_bytes_head") for k in range(nmat)))
        bytes_t = bytes_f - bytes_h - build_b          # the tail's share of the elimination (device counter elim_bytes)
        kinds = {"head": ("mode HEAD (singletons + setup_bump + sparse elimination)", hm, bytes_h),
                 "tail": ("mode TAIL (dense tail: HBM/L2 stage, then shared memory)", tm, bytes_t)}
        dom = "head" if hm >= tm else "tail"
        dom_ms = kinds[dom][1] if split else float(np.mean(fact_ms))
        dom_bytes = kinds[dom][2] if split else bytes_f
        other = "tail" if dom == "head" else "head"
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
        nt_dom = int(b.get_param("threads_per_basis")) if (dom == "head" or not split) else int(b.get_param("tail_threads"))
        roofline = {"bound": "hbm", "kernel": "k_factorize<%d> %s" % (nt_dom, kinds[dom][0] if split else "(whole factorization)"),
                    "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": dom_bytes, "avg_launch_ms": dom_ms,
                    "whole_factorization": {"algorithmic_bytes": bytes_f, "ms": float(np.mean(fact_ms)),
                                            "achieved_GBps": bytes_f / (float(np.mean(fact_ms)) * 1e-3) / 1e9,
                                            "frac": bytes_f / (float(np.mean(fact_ms)) * 1e-3) / 1e9 / peak},
                    "other_kernels_ms_per_step": {"k_factorize %s" % kinds[other][0]: kinds[other][1],
                                                  "k_factorize mode BUILD (build_factors)": float(np.mean(build_ms)),
                                                  "k_factor_norms (condest x2 + residual_test, factorize.rs:121-147)": float(np.mean(norms_ms)),
                                                  "k_solve_dense": float(b.last_kernel_ms(1))},
                    "other_kernels_algorithmic_bytes": {"k_factorize %s" % kinds[other][0]: kinds[other][2], "k_factorize mode BUILD": build_b}}
        roofline["dominant"] = dom
        tf = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tf):
            try:
                t = json.load(open(tf))
                # dram__bytes_read.sum + dram__bytes_write.sum of one steady-state launch of that kernel (ncu --set
                # full), per basis, scaled to this launch's batch -- quoted only if taken with these very sources
                if t.get("kernel_source_hash") == kernel_source_hash() and t.get("dominant", "head") == (dom if split else "whole"):
                    roofline["traffic"] = t["dram_bytes_per_basis"] * nmat
                    roofline["traffic_source"] = t["source"]
                else:
                    roofline["traffic_source"] = "none: profiles/traffic.json was captured with other kernel sources or for another kernel (%s %s, now %s %s)" % (t.get("kernel_source_hash"), t.get("dominant", "head"), kernel_source_hash(), dom)
            except Exception:
                pass
        cpu = None
        if not args.no_cpu_baseline and world == 1:      # reported at N=1 only (rank 0)
            import oracle_lib
            cores = host_cores()
            ns = int(min(nmat, max(cores * args.ref_per_core, 8)))
            t0 = time.perf_counter()
            nt, xo, so = oracle_lib.batch_factorize_solve(ns, M, bb[:ns * M], be[:ns * M], bi, bx, rhs[:ns * M], nthreads=cores, check_file_diff=1)
            dt = time.perf_counter() - t0
            err = float(np.abs(x[:ns] - xo).max() / np.abs(xo).max())
            t0 = time.perf_counter()
            oracle_lib.batch_factorize_solve(ns, M, bb[:ns * M], be[:ns * M], bi, bx, rhs[:ns * M], nthreads=cores, check_file_diff=0)
            dt_nofd = time.perf_counter() - t0
            cpu = {"value": ns / dt, "unit": UNIT, "cores": nt, "kind": "port",
                   "value_without_file_diff_asserts": ns / dt_nofd,   # D11: the reference keeps these O(sum rownz*colnz) asserts in release builds; without them the CPU is faster
                   "sample": f"first {ns} bases of rank 0's batch, factorize+solve_dense each, one oracle instance per core ({nt} threads), file_diff asserts on",
                   "max_rel_diff_gpu_vs_cpu_solution": err}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "configs[1]: 4096 x (2000x2000 simplex-style basis, ~6 nnz/col) factorize+solve_dense",
                           "m": M, "bases": total, "bases_per_gpu": nmat, "nnz_per_basis": float(len(bi)) / nmat,
                           "sharding": f"bases by index (shard_range), {world} rank(s), no collective",
                           "dense_k": int(b.get_param("dense_k")), "dense_k_big": int(b.get_param("dense_k_big")), "tail_threads": int(b.get_param("tail_threads")),
                           "store_entries_per_basis": {"l_mem": int(b.get_param("l_mem")), "u_mem": int(b.get_param("u_mem")), "w_mem": int(b.get_param("w_mem"))},
                           "l2": "inputs exceed L2: %.0f MB of B + rhs are re-read every step (L2 126 MB)" % ((pbi.nbytes + pbx.nbytes + pbb.nbytes + pbe.nbytes + prhs.nbytes) / 1e6),
                           "threads_per_basis": int(b.get_param("threads_per_basis")), "reallocations_in_warmup": nrealloc, "reallocations_in_timed_steps": nrealloc_after - nrealloc,
                           "gen_seconds": t_gen},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps, "api": "blu_batch_factorize + blu_batch_solve_dense (host pointers, pinned)"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline}
        if cpu:
            line["cpu_baseline"] = cpu
        emit(line)
    b.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
