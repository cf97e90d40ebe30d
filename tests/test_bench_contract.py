"""bench.py contract on CPU: the reference arm (oracle C/OpenMP port on host cores) prints ONE JSON line with the keys the
driver reads; the B200 arm refuses to run without a GPU instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          cwd=ROOT, env=dict(os.environ, **(env or {})), timeout=600)


def test_reference_arm_json_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample-rows", "20000"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "kmeans_fit_samples_per_sec" and j["unit"] == "samples/s"
    assert j["higher_is_better"] is True and j["steps"] == 1 and j["value"] > 0
    assert j["cpu_baseline"]["kind"] in ("port", "reference") and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert j["e2e"]["value"] == j["value"]


def test_reference_arm_nonzero_ranks_do_no_work():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="checks the no-GPU failure mode")
def test_b200_arm_fails_loudly_without_gpu():
    r = _run(["--steps", "1", "--warmup", "1", "--no-e2e", "--no-cpu-baseline"])
    assert r.returncode != 0
    assert "{\"metric\"" not in r.stdout


def test_reference_arm_dumps_the_timed_result(tmp_path):
    """--dump-outputs DIR: the centres and inertia of the timed loop, i.e. --steps Lloyd iterations from the first k rows
    of the seeded sample, as the fp64 oracle computes them."""
    import numpy as np

    import bench
    from oracle import kmeans_oracle as ko

    rows, d, k = 20000, 128, 64
    X = bench.cpu_sample(rows, d, k)
    for steps in (2, 1):
        out = tmp_path / str(steps)
        r = _run(["--impl", "reference", "--steps", str(steps), "--warmup", "1", "--cpu-sample-rows", str(rows),
                  "--dump-outputs", str(out)])
        assert r.returncode == 0, r.stderr[-2000:]
        C, inertia = np.load(out / "cluster_centers.npy"), np.load(out / "inertia.npy")
        assert C.dtype == np.float32 and C.shape == (k, d) and inertia.dtype == np.float64
        ref = ko.lloyd([X], X[:k].copy(), steps, -1.0)
        assert ko.max_center_rel_err(C, ref["centers"]) <= 1e-6
        assert abs(float(inertia) - ref["inertia"]) <= 1e-9 * ref["inertia"]


@pytest.mark.gpu
def test_b200_arm_dumps_the_timed_result(tmp_path):
    """The same for the sm_100a arm: the dumped centres are, bit for bit, what the library's Lloyd loop returns after
    --steps iterations on the benchmark's seeded device blobs, and two runs with the same arguments agree."""
    import numpy as np
    import torch

    import bench
    from spark_rapids_ml_b200 import _native

    n, d, k = 50_000, 128, 64
    args = ["--config", "small", "--n-per-gpu", str(n), "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--no-cfg3",
            "--long-steps", "0"]
    got = {}
    for tag, steps in (("a", 3), ("b", 3), ("c", 1)):
        r = _run(args + ["--steps", str(steps), "--dump-outputs", str(tmp_path / tag)])
        assert r.returncode == 0, r.stderr[-2000:]
        got[tag] = np.load(tmp_path / tag / "cluster_centers.npy")
        assert got[tag].dtype == np.float32 and got[tag].shape == (k, d)
        assert np.load(tmp_path / tag / "shift.npy").dtype == np.float64
    np.testing.assert_array_equal(got["a"], got["b"])
    X, _ = bench.make_blobs_device(torch, torch.device("cuda", 0), n, d, k, 0)
    with _native.Context(0) as ctx:
        for tag, steps in (("a", 3), ("c", 1)):
            C = X[:k].clone()
            assert ctx.kmeans_lloyd(X, C, steps, -1.0)[0] == steps
            np.testing.assert_array_equal(got[tag], C.cpu().numpy())
