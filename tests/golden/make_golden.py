"""Generates the golden fixtures in this directory.

    python tests/golden/make_golden.py

The reference (mrocklin/dask-ml) cannot be imported in the build image (dask is absent), so the vectors
are produced by the oracle restatement (oracle/kmeans_oracle.py), whose per-chunk arithmetic is the
reference's own dependency (scikit-learn pairwise_distances_argmin_min) plus the restated scatter-add,
and whose results are asserted equal to scikit-learn's Lloyd in tests/test_oracle.py exactly as the
reference's tests do.  scikit-learn / numpy versions are recorded in MANIFEST.json.  The input rows are not
stored: a fixture keeps the parameters of ``tests/_util.blobs`` and the SHA-256 of the rows it was computed from
(``tests/_util.load_golden`` regenerates and checks them).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import kmeans_oracle as ok  # noqa: E402
from _util import blobs, x_digest  # noqa: E402

CASES = {
    # name: (n, d, k, k_true, dtype, chunks, max_iter, tol, seed)
    "lloyd_f32_64x256": (6000, 64, 256, 80, "float32", 2500, 6, 1e-4, 11),
    "lloyd_f64_16x8": (4000, 16, 8, 8, "float64", 1000, 50, 1e-4, 12),
    "lloyd_f32_41x100": (5000, 41, 100, 30, "float32", 5000, 6, 1e-4, 13),
}


def main():
    import sklearn
    manifest = {"numpy": np.__version__, "sklearn": sklearn.__version__, "cases": {}}
    for name, (n, d, k, kt, dt, chunks, max_iter, tol, seed) in CASES.items():
        X = blobs(n, d, kt, seed, dt)
        init = X[:k].copy()
        lab, inertia, C, n_iter = ok.kmeans_single_lloyd(ok.to_blocks(X, chunks), k, init=init, max_iter=max_iter,
                                                        tol=tol)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), blobs=np.array([n, d, kt, seed]), dtype=dt,
                            X_sha256=x_digest(X), init=init, k=k, chunks=chunks,
                            max_iter=max_iter, tol=tol, labels=np.concatenate(lab), centers=C,
                            inertia=inertia, n_iter=n_iter)
        manifest["cases"][name] = {"n": n, "d": d, "k": k, "dtype": dt, "n_iter": int(n_iter),
                                   "inertia": float(inertia)}
    with open(os.path.join(HERE, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1)


if __name__ == "__main__":
    main()
