"""Helpers shared by the parity tests."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def blobs(n, d, k_true, seed, dtype):
    """Isotropic blobs drawn from numpy's legacy ``RandomState``, whose streams numpy keeps fixed across releases:
    the Lloyd fixtures in tests/golden/ store these parameters instead of the rows."""
    rng = np.random.RandomState(seed)
    cent = rng.uniform(-10, 10, size=(k_true, d))
    return (cent[rng.randint(0, k_true, size=n)] + rng.standard_normal((n, d))).astype(dtype)


def x_digest(X):
    return hashlib.sha256(np.ascontiguousarray(X).tobytes()).hexdigest()


def load_golden(name):
    """A Lloyd fixture of tests/golden/ as a dict, with its input rows ``X`` regenerated from the stored
    ``blobs`` parameters and checked against the SHA-256 of the rows the fixture was computed from."""
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    n, d, k_true, seed = (int(v) for v in g["blobs"])
    X = blobs(n, d, k_true, seed, str(g["dtype"]))
    assert x_digest(X) == str(g["X_sha256"]), "%s: regenerated input rows differ from the fixture's" % name
    g["X"] = X
    return g


def d2_f64(X, C):
    X = np.asarray(X, dtype=np.float64)
    C = np.asarray(C, dtype=np.float64)
    return ((X[:, None, :] - C[None, :, :]) ** 2).sum(-1) if X.shape[0] * C.shape[0] * X.shape[1] < 5e7 else \
        np.maximum((X * X).sum(1)[:, None] - 2 * X @ C.T + (C * C).sum(1)[None, :], 0)


def assert_labels_match(got, want, X, C, rtol=1e-9, max_frac=1e-3):
    """Labels must be identical except on float64 near-ties: rows where the two chosen centres are
    equidistant to `rtol` relative to (||x||^2+||c||^2).  This is the documented tie-breaking."""
    got = np.asarray(got).astype(np.int64)
    want = np.asarray(want).astype(np.int64)
    assert got.shape == want.shape
    bad = np.nonzero(got != want)[0]
    if len(bad) == 0:
        return 0
    Xb = np.asarray(X, dtype=np.float64)[bad]
    C = np.asarray(C, dtype=np.float64)
    dg = ((Xb - C[got[bad]]) ** 2).sum(1)
    dw = ((Xb - C[want[bad]]) ** 2).sum(1)
    scale = (Xb ** 2).sum(1) + (C ** 2).sum(1).max()
    rel = np.abs(dg - dw) / scale
    assert rel.max() <= rtol, "label mismatch that is not a float64 near-tie: rel margin %g at row %d" % (
        rel.max(), bad[rel.argmax()])
    assert len(bad) <= max(1, max_frac * len(got)), "%d near-tie mismatches of %d rows" % (len(bad), len(got))
    return len(bad)
