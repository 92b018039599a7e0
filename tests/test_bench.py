"""bench.py's command line and --dump-outputs: the arguments it refuses (CPU), the files it writes (CPU), and on a B200
that they hold exactly what the timed steps computed (config 1 against the oracle's committed result)."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, "bench.py", *args], capture_output=True, text=True, cwd=ROOT, timeout=600)


@pytest.mark.parametrize("args", [["--steps", "0"], ["--warmup", "-1"], ["--gpus", "2", "--dump-outputs", "x"],
                                  ["--impl", "reference", "--dump-outputs", "x"]])
def test_bad_arguments_are_refused(args):
    r = run_bench(*args)
    assert r.returncode == 2 and "error:" in r.stderr, r.stderr


def test_dump_outputs_files(tmp_path):
    merges = np.arange(100, dtype=np.uint32).reshape(-1, 2)
    short = np.arange(1000, dtype=np.uint32)
    bench.dump_outputs(str(tmp_path / "short"), merges, short)
    assert sorted(os.listdir(tmp_path / "short")) == ["ids.npy", "merges.npy"]
    m = np.load(tmp_path / "short" / "merges.npy")
    ids = np.load(tmp_path / "short" / "ids.npy")
    assert m.dtype == ids.dtype == np.float64 and np.array_equal(m, merges) and np.array_equal(ids, short)

    long = np.random.default_rng(1).integers(0, 50256, 3 * bench.DUMP_IDS, dtype=np.uint32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), None, long)
    assert sorted(os.listdir(tmp_path / "a")) == ["ids.npy", "ids_index.npy"]
    idx = np.load(tmp_path / "a" / "ids_index.npy")
    ids = np.load(tmp_path / "a" / "ids.npy")
    assert idx.size == ids.size == bench.DUMP_IDS and np.all(np.diff(idx) > 0)
    assert np.array_equal(ids, long[idx.astype(np.int64)])
    for f in ("ids.npy", "ids_index.npy"):   # fixed positions: the same stream gives the same files
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
    # the largest merge list of the workloads (c5: 50,000) and a sampled stream stay below 64 MB
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) + 50000 * 2 * 8
    assert total < 64 << 20


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_result(tmp_path):
    """Config 1 (random_text.txt to exhaustion) with two timed steps: the dumped merge list and ids are the oracle's."""
    out = tmp_path / "out"
    r = run_bench("--workload", "c1", "--steps", "2", "--warmup", "1", "--quick", "--no-cpu-baseline", "--dump-outputs", str(out))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2 and line["checks"]["equals_oracle_digest"]
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "c1_exhaustion.json")))
    want = np.load(os.path.join(ROOT, "tests", "golden", "full", "c1_exhaustion_merges.npz"))["merges"]
    assert sorted(os.listdir(out)) == ["ids.npy", "merges.npy"]
    assert np.array_equal(np.load(out / "merges.npy"), want)
    ids = np.load(out / "ids.npy").astype("<u4")
    assert ids.size == g["n_ids"] and hashlib.sha256(ids.tobytes()).hexdigest() == g["ids_sha256"]
