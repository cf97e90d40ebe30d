"""Regenerates/validates tests/golden/*.

kmeans_known_answers.json is TRANSCRIBED (not computed) from the reference's own tests — the
reference's arithmetic (cuML) cannot run in this container (SURVEY.md 8c).  Running this script
(a) re-checks that the transcribed literals still appear in the reference test sources when
/root/reference is present, and (b) writes lloyd_golden_*.npz: seeded inputs + fp64-oracle
outputs that the GPU parity tests replay on the box (where /root/reference and sklearn's
cross-check are not needed).  The oracle outputs stored here are cross-checked against
scikit-learn's Lloyd in tests/test_oracle.py, which is what pins them.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import kmeans_oracle as ko  # noqa: E402


def check_transcription() -> None:
    ref = "/root/reference/python/tests/test_kmeans.py"
    if not os.path.exists(ref):
        print("reference not present; transcription check skipped")
        return
    src = open(ref).read()
    for lit in ["[[1.0, 1.0], [1.0, 2.0], [3.0, 2.0], [4.0, 3.0]]", "[1.0, 1.5]", "[3.5, 2.5]",
                "[[0.5, 0.5], [8.5, 8.5]]", "Vectors.dense([9.0, 8.0])"]:
        assert lit in src, lit
    print("transcription literals found in", ref)


def write_lloyd_golden() -> None:
    cases = [
        # name, n, d, k, generator, max_iter, tol
        ("blobs_small", 4096, 16, 8, "blobs", 30, 1e-4),
        ("blobs_d128_k64", 1536, 128, 64, "blobs", 12, 1e-4),   # X barely compresses: 1536 rows keep the file < 1 MB
        ("uniform_d32_k8", 6000, 32, 8, "uniform", 8, 0.0),
        ("ragged_d20_k5", 1000, 20, 5, "blobs", 20, 1e-4),
    ]
    for name, n, d, k, gen, max_iter, tol in cases:
        if gen == "blobs":
            X, _ = ko.make_blobs(n, d, k, seed=1234)
        else:
            X = ko.make_uniform(n, d, seed=1234)
        C0 = X[:k].copy()  # deterministic "array" init: first k rows (SURVEY.md 8d)
        out = ko.lloyd([X], C0, max_iter, tol)
        np.savez_compressed(
            os.path.join(HERE, f"lloyd_golden_{name}.npz"),
            X=X, C0=C0, centers=out["centers"], labels=out["labels"][0],
            n_iter=np.int32(out["n_iter"]), inertia=np.float64(out["inertia"]),
            max_iter=np.int32(max_iter), tol=np.float64(tol),
        )
        print(name, "n_iter", out["n_iter"], "inertia", out["inertia"])


if __name__ == "__main__":
    json.load(open(os.path.join(HERE, "kmeans_known_answers.json")))
    check_transcription()
    write_lloyd_golden()
