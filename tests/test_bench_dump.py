"""bench.py --dump-outputs: what the timed path returned in its last step, as float64 .npy files, equal to the oracle
on the bench's seeded inputs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from blu_b200 import gen
from oracle_lib import Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out, *args):
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--nmat", "6",
                    "--dump-outputs", str(out), *args], check=True, capture_output=True, timeout=900)
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float64 for a in d.values())
    return d


def check_with_oracle(d):
    """The dumped solutions are those of bench.py's bases (gen.config2_matrix k), bit for bit."""
    assert d["x"].shape == (6, bench.M) and list(d["bases"]) == list(range(6))
    assert (d["status"] == 0).all()
    for row, k in enumerate(d["bases"].astype(int)):
        (cp, ri, v), rhs = gen.config2_matrix(k, bench.M)
        o = Oracle(bench.M, 60 * len(v))
        assert o.factorize(cp[:-1], cp[1:], ri, v) == 0
        _, xo = o.solve_dense(rhs, "N")
        assert np.array_equal(d["x"][row], xo), k
        if "factor_info" in d:
            assert list(d["factor_info"][row]) == [o.info(n) for n in bench.DUMP_INFO], k
    return d


def test_dump_outputs_sample(tmp_path, monkeypatch):
    """Solutions beyond DUMP_BYTES are cut to a fixed seeded sample of bases, listed in bases.npy."""
    n, m = 50, 8
    monkeypatch.setattr(bench, "DUMP_BYTES", 10 * 8 * m)
    x = np.random.default_rng(3).random((n, m))
    status = np.zeros(n, np.int32)
    for out in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(out), x, status, np.ones((n, 2)))
    a, b = ({f[:-4]: np.load(out / f) for f in os.listdir(out)} for out in (tmp_path / "a", tmp_path / "b"))
    assert sorted(a) == ["bases", "factor_info", "status", "x"]
    idx = a["bases"].astype(int)
    assert len(idx) == 10 and (np.diff(idx) > 0).all()
    assert np.array_equal(a["x"], x[idx]) and a["status"].shape == (n,) and a["factor_info"].shape == (n, 2)
    assert all(np.array_equal(a[k], b[k]) for k in a)


def test_dump_outputs_reference(tmp_path):
    check_with_oracle(run_bench(tmp_path, "--impl", "reference", "--ref-per-core", "1"))


@pytest.mark.gpu
def test_dump_outputs_cuda(tmp_path):
    d = check_with_oracle(run_bench(tmp_path, "--no-cpu-baseline"))
    assert d["factor_info"].shape == (6, len(bench.DUMP_INFO))
