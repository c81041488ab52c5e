"""The CPU oracle pinned against the reference's own test expectations (which are run-time comparisons
with scikit-learn — the reference holds no golden vectors, SURVEY.md §8c) and against the committed
fixtures in tests/golden/.  Runs without a GPU."""
import json
import os

import numpy as np
import pytest
import sklearn.datasets
import sklearn.metrics
from sklearn.cluster import KMeans as SKKMeans, kmeans_plusplus
from sklearn.utils.extmath import row_norms

from _util import load_golden

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _easy(oracle):
    centers = np.array([[-7, -7], [0, 0], [7, 7]])
    Xs, ys = oracle.make_blobs(cluster_std=0.1, centers=centers, chunks=50, random_state=0)
    return Xs, ys


def test_fit_given_init_equals_sklearn(oracle):
    """reference tests/test_kmeans.py:87-98: identical init => sklearn's Lloyd result."""
    X, _ = sklearn.datasets.make_blobs(n_samples=1000, n_features=4, random_state=1)
    init, _ = kmeans_plusplus(X, 3, random_state=np.random.RandomState(0))
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(oracle.to_blocks(X, 500), 3, init=init)
    sk = SKKMeans(3, init=init, random_state=0, n_init=1).fit(X)
    np.testing.assert_allclose(inertia, sk.inertia_, rtol=1e-12)
    np.testing.assert_array_equal(np.concatenate(lab), sk.labels_)
    # the number SURVEY.md §7 records for this restatement
    np.testing.assert_allclose(inertia, 3966.9294065453428, rtol=1e-13)


def test_argmin_min_exact_vs_sklearn_per_block(oracle):
    """reference tests/metrics/test_metrics.py:23-43: EXACT equality with sklearn, block-wise."""
    X, _ = sklearn.datasets.make_classification(n_samples=1000, n_features=4, random_state=1)
    centers = X[::100]
    a_, b_ = sklearn.metrics.pairwise_distances_argmin_min(X, centers)
    a, b = oracle.pairwise_distances_argmin_min(oracle.to_blocks(X, 500), centers)
    np.testing.assert_array_equal(np.concatenate(a), a_)
    np.testing.assert_allclose(np.concatenate(b), b_, rtol=0, atol=1e-12)


def test_plain_c_estep_agrees_with_sklearn(oracle):
    """oracle_c.c is an independent restatement of the float64 formula + first-index tie rule."""
    rng = np.random.RandomState(0)
    for dt in (np.float32, np.float64):
        X = rng.standard_normal((2000, 13)).astype(dt)
        C = X[:37].copy()
        C[5] = C[2]                      # duplicate centre: the lower index must win
        la, ma = oracle.argmin_min_c(X, C)
        lb, mb = sklearn.metrics.pairwise_distances_argmin_min(X, C, metric_kwargs={"squared": True})
        np.testing.assert_array_equal(la, lb)
        np.testing.assert_allclose(ma, mb, rtol=0, atol=1e-5 if dt == np.float32 else 1e-11)
        assert not (la == 5).any()


def test_centers_dense_c_vs_numpy(oracle):
    rng = np.random.RandomState(1)
    X = rng.standard_normal((5000, 7)).astype(np.float32)
    lab = rng.randint(0, 11, size=5000).astype(np.int32)
    got = oracle.centers_dense(X, lab, 11)
    want = np.zeros((11, 7))
    np.add.at(want, lab, X.astype(np.float64))
    np.testing.assert_allclose(got, want, rtol=1e-12)
    assert got.dtype == np.float64          # k_means.py:576


def test_row_norms(oracle):
    """reference tests/test_kmeans.py:27-30."""
    X, _ = sklearn.datasets.make_classification(n_samples=1000, n_features=4, random_state=1)
    from dask_ml_b200.utils import row_norms as rn
    from dask_ml_b200 import ChunkedArray
    got = rn(ChunkedArray.from_array(X, 500), squared=True).compute()
    np.testing.assert_allclose(got, row_norms(X, squared=True))


def test_basic_easy_blobs_vs_sklearn(oracle):
    """reference tests/test_kmeans.py:55-85 with the default k-means|| init."""
    Xs, _ = _easy(oracle)
    X = np.concatenate(Xs)
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(Xs, 3, random_state=0)
    b = SKKMeans(n_clusters=3, random_state=0, n_init=10).fit(X)
    a_order = np.argsort(C, 0)[:, 0]
    b_order = np.argsort(b.cluster_centers_, 0)[:, 0]
    np.testing.assert_allclose(C[a_order], b.cluster_centers_[b_order], rtol=1e-3)
    # inertia_ follows the reference's Q4 rule (sum of d, not d^2, unless shift <= 1e-7); compare d^2
    d2 = ((X[:, None, :] - C[None]) ** 2).sum(-1).min(1).sum()
    assert abs(d2 - b.inertia_) < 0.01


def test_quirks_q1_q3_q4(oracle):
    """Q1 empty cluster -> origin; Q3 old centres on convergence; Q4 inertia branch."""
    rng = np.random.RandomState(0)
    X = rng.standard_normal((500, 3)) + 5.0
    init = np.vstack([X[:2], [[100.0, 100.0, 100.0]]])
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd([X], 3, init=init, max_iter=1, tol=0.0)
    assert (C[2] == 0).all()                                   # Q1
    Xs, _ = _easy(oracle)
    init = np.array([[-7.0, -7.0], [0.0, 0.0], [7.0, 7.0]])
    tr = []
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(Xs, 3, init=init, tol=1e-4, trace=tr)
    Xn = np.concatenate(Xs)
    assert n_iter == len(tr)
    d = np.sqrt(((Xn[:, None, :] - C[None]) ** 2).sum(-1)).min(1)
    if tr[-1]["shift"] > 1e-7:
        np.testing.assert_allclose(inertia, d.sum(), rtol=1e-9)          # Q4: plain distances
    else:
        np.testing.assert_allclose(inertia, (d ** 2).sum(), rtol=1e-9)   # Q4: squared distances


def test_k_init_errors(oracle):
    """reference tests/test_kmeans.py:131-147."""
    Xs, _ = _easy(oracle)
    X = np.concatenate(Xs)
    with pytest.raises(ValueError):
        oracle.k_init(Xs, 3, X[:2])
    with pytest.raises(ValueError):
        oracle.k_init(Xs, 2, X[:2, :-1])
    with pytest.raises(ValueError):
        oracle.k_init(Xs, 2, "invalid")
    with pytest.raises(TypeError):
        oracle.k_init(Xs, 2, 2)


def test_make_blobs_contract(oracle):
    """datasets.py:178-189: block i is sklearn.make_blobs(random_state=i) around the prototype centres."""
    Xs, ys = oracle.make_blobs(n_samples=300, n_features=3, centers=4, chunks=100, random_state=7)
    Xs2, _ = oracle.make_blobs(n_samples=300, n_features=3, centers=4, chunks=100, random_state=7)
    assert len(Xs) == 3 and all(x.shape == (100, 3) for x in Xs)
    for a, b in zip(Xs, Xs2):
        np.testing.assert_array_equal(a, b)
    assert Xs[0].dtype == np.float64 and ys[0].dtype.kind == "i"


def test_philox_known_answers(oracle):
    """Philox4x32-10 known-answer vectors (Random123 kat_vectors): counter/key all zero and all ones."""
    # first output word for ctr = 0, key = 0 is 0x6627e8d5 ; for ctr = key = 0xffffffff.. is 0x408f276d
    u0 = oracle.philox_uniform(0, np.array([0], dtype=np.uint64))[0]
    assert int(round(u0 * 2 ** 32)) == 0x6627E8D5


@pytest.mark.parametrize("name", ["lloyd_f32_64x256", "lloyd_f64_16x8", "lloyd_f32_41x100"])
def test_golden_fixtures(oracle, name):
    """Committed golden vectors (tests/golden/make_golden.py): the oracle must reproduce them bit for bit
    on labels and to 1e-12 on centres/inertia (guards the oracle against dependency drift)."""
    g = load_golden(name)
    blocks = oracle.to_blocks(g["X"], int(g["chunks"]))
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(blocks, int(g["k"]), init=g["init"],
                                                        max_iter=int(g["max_iter"]), tol=float(g["tol"]))
    assert n_iter == int(g["n_iter"])
    np.testing.assert_array_equal(np.concatenate(lab), g["labels"])
    np.testing.assert_allclose(C, g["centers"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(inertia, float(g["inertia"]), rtol=1e-12)


REF_CASES = ["ref_lloyd_f32_64x256", "ref_lloyd_f64_16x8", "ref_lloyd_f32_41x100", "ref_lloyd_f32_13x20_conv"]


@pytest.mark.parametrize("name", REF_CASES)
def test_oracle_reproduces_the_reference_itself(oracle, name):
    """Fixtures written by tests/golden/ref_shim.py, i.e. by the UNMODIFIED reference source files
    (dask_ml/cluster/k_means.py, metrics/pairwise.py, utils.py) executed over an eager stand-in for dask:
    KMeans(init=ndarray).fit -> labels_, cluster_centers_, inertia_, n_iter_.  The oracle must agree bit for bit
    on labels / n_iter and to float64 round-off on centres and inertia (both inertia branches of Q4 occur)."""
    g = load_golden(name)
    blocks = oracle.to_blocks(g["X"], int(g["chunks"]))
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(blocks, int(g["k"]), init=g["init"],
                                                        max_iter=int(g["max_iter"]), tol=float(g["tol"]))
    assert n_iter == int(g["n_iter"])
    np.testing.assert_array_equal(np.concatenate(lab), g["labels"])
    assert np.concatenate(lab).dtype == g["labels"].dtype == np.int32
    np.testing.assert_allclose(C, g["centers"], rtol=1e-13, atol=0)
    assert C.dtype == g["centers"].dtype
    np.testing.assert_allclose(inertia, float(g["inertia"]), rtol=1e-13)
    tr = np.concatenate(oracle.euclidean_distances(blocks, g["centers"]))[:256]
    np.testing.assert_allclose(tr, g["transform"], rtol=1e-12, atol=1e-12)


def test_oracle_pairwise_ops_vs_reference(oracle):
    """dask_ml.metrics.pairwise_distances_argmin_min / pairwise_distances run by the reference code itself."""
    g = np.load(os.path.join(GOLD, "ref_pairwise_ops.npz"))
    blocks = oracle.to_blocks(g["X"], 500)
    a, b = oracle.pairwise_distances_argmin_min(blocks, g["centers"])
    np.testing.assert_array_equal(np.concatenate(a), g["argmin"])
    np.testing.assert_allclose(np.concatenate(b), g["mins"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(np.concatenate(oracle.pairwise_distances(blocks, g["centers"])), g["dists"], atol=1e-12)
