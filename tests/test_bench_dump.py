"""bench.py --dump-outputs: the kNN lists of the last timed step as float64 .npy files, at most 64 MB in
all, the same rows on every run -- so that the outputs of two builds can be compared file for file."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(d):
    return {name: np.load(os.path.join(d, f"knn_{name}.npy")) for name in ("rows", "idx", "w")}


def test_dump_writes_every_row_of_small_tables_and_a_fixed_sample_of_large_ones(tmp_path):
    import bench
    for n, k in ((1000, 16), (300_000, 16), (20_000, 1000)):
        idx = torch.arange(n * k, dtype=torch.int64).reshape(n, k)
        w = idx % 257
        a, b = tmp_path / f"a{n}", tmp_path / f"b{n}"
        bench.dump_knn(str(a), idx, w)
        bench.dump_knn(str(b), idx, w)
        got = _read(a)
        assert sum(os.path.getsize(a / f) for f in os.listdir(a)) <= 64 << 20
        assert all(v.dtype == np.float64 for v in got.values())
        rows = got["rows"].astype(np.int64)
        if n * k * 16 <= bench.DUMP_BYTES:
            np.testing.assert_array_equal(rows, np.arange(n))
        else:
            assert len(rows) == bench.DUMP_BYTES // (16 * k) and np.all(np.diff(rows) > 0) and rows[-1] < n
        np.testing.assert_array_equal(got["idx"], idx.numpy()[rows])
        np.testing.assert_array_equal(got["w"], w.numpy()[rows])
        again = _read(b)
        assert all(np.array_equal(got[key], again[key]) for key in got)


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_build(tmp_path):
    """A short bench run on the symmetric path (bootstrap + symmetric sweep per step): the JSON line
    reports the requested steps, the timed window held exactly that many builds, and the dumped lists
    equal the oracle's on sampled rows."""
    from oracle import prograph_oracle as O
    import bench
    n, L, k, steps = 70_000, 64, 16, 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--length", str(L), "--k", str(k),
                          "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-eps",
                          "--no-queries", "--dump-outputs", str(tmp_path)],
                         cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["parity"]["ok"]
    assert line["roofline"]["bootstrap"] is not None          # two sweeps per timed step, `steps` steps
    got = _read(tmp_path)
    np.testing.assert_array_equal(got["rows"], np.arange(n))
    X = bench.make_tokens(n, L, "uniform")
    sample = np.random.default_rng(5).choice(n, size=24, replace=False)
    ri, rw = O.knn_from_distances(O.hamming(X, X[sample]), k)
    np.testing.assert_array_equal(got["idx"][sample], ri)
    np.testing.assert_array_equal(got["w"][sample], rw)
