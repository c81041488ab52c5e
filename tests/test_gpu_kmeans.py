"""GPU end-to-end tests of the estimator against the CPU oracle and scikit-learn, modelled on the
reference's tests/test_kmeans.py (run with -m gpu)."""
import numpy as np
import pytest
import sklearn.datasets
from sklearn.cluster import KMeans as SKKMeans, kmeans_plusplus

from _util import assert_labels_match, load_golden

pytestmark = pytest.mark.gpu


def _easy_blobs(oracle):
    centers = np.array([[-7, -7], [0, 0], [7, 7]])
    Xs, ys = oracle.make_blobs(cluster_std=0.1, centers=centers, chunks=50, random_state=0)
    return Xs, ys


def replace(a, old, new):
    arr = np.empty(a.max() + 1, dtype=new.dtype)
    arr[old] = new
    return arr[a]


def test_fit_given_init_matches_oracle_and_sklearn(oracle):
    """tests/test_kmeans.py:87-98 — identical init => identical result."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    X_, _ = sklearn.datasets.make_blobs(n_samples=1000, n_features=4, random_state=1)
    init, _ = kmeans_plusplus(X_, 3, random_state=np.random.RandomState(0))
    X = ChunkedArray.from_array(X_, chunks=500)
    dkkm = KMeans(3, init=init, random_state=0).fit(X)
    skkm = SKKMeans(3, init=init, random_state=0, n_init=1).fit(X_)
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(oracle.to_blocks(X_, 500), 3, init=init)
    np.testing.assert_allclose(dkkm.inertia_, skkm.inertia_)
    np.testing.assert_allclose(dkkm.inertia_, inertia, rtol=1e-12)
    assert dkkm.n_iter_ == n_iter
    np.testing.assert_array_equal(dkkm.labels_.compute(), np.concatenate(lab))
    np.testing.assert_allclose(dkkm.cluster_centers_, C, rtol=1e-12)


def test_basic_vs_sklearn(oracle):
    """tests/test_kmeans.py:55-85 (default init='k-means||')."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    Xs, _ = _easy_blobs(oracle)
    X = ChunkedArray(Xs)
    Xn = np.concatenate(Xs)
    a = KMeans(n_clusters=3, random_state=0).fit(X)
    b = SKKMeans(n_clusters=3, random_state=0, n_init=10).fit(Xn)
    assert abs(a.inertia_ - b.inertia_) < 0.01
    a_order = np.argsort(a.cluster_centers_, 0)[:, 0]
    b_order = np.argsort(b.cluster_centers_, 0)[:, 0]
    a_centers = a.cluster_centers_[a_order]
    b_centers = b.cluster_centers_[b_order]
    np.testing.assert_allclose(a_centers, b_centers, rtol=1e-3)
    b_labels = replace(b.labels_, [0, 1, 2], a_order[b_order]).astype(b.labels_.dtype)
    np.testing.assert_array_equal(a.labels_.compute(), b_labels)
    assert a.n_iter_
    b.cluster_centers_ = b_centers
    a.cluster_centers_ = a_centers
    np.testing.assert_allclose(a.transform(X).compute(), b.transform(Xn), rtol=1e-3)
    np.testing.assert_array_equal(a.predict(X).compute(), b.predict(Xn))


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("n,d,k,chunks", [(20000, 64, 256, 7000), (30000, 41, 100, 30000), (50000, 13, 20, 12500)])
def test_lloyd_parity_fixed_init(oracle, dtype, n, d, k, chunks):
    """North-star parity: identical inputs + identical init centroids -> labels equal (modulo float64
    near-ties), inertia within 1e-4 relative (here far tighter), same n_iter, same centres."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    rng = np.random.RandomState(42)
    cent = rng.uniform(-10, 10, size=(max(2, k // 3), d))
    X = (cent[rng.randint(0, len(cent), size=n)] + rng.standard_normal((n, d))).astype(dtype)
    init = X[:k].copy()
    km = KMeans(k, init=init, max_iter=8, tol=1e-4).fit(ChunkedArray.from_array(X, chunks))
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(oracle.to_blocks(X, chunks), k, init=init, max_iter=8,
                                                        tol=1e-4)
    assert km.n_iter_ == n_iter
    np.testing.assert_allclose(km.cluster_centers_, C, rtol=1e-4, atol=1e-5)
    assert_labels_match(km.labels_.compute(), np.concatenate(lab), X, C, rtol=1e-6)
    assert abs(km.inertia_ - inertia) <= 1e-6 * inertia
    assert km.cluster_centers_.dtype == X.dtype
    assert km.labels_.dtype == np.int32
    assert isinstance(km.inertia_, np.float64)


def test_converged_branch_and_old_centres(oracle):
    """Q3/Q4: on convergence the OLD centres are returned and, when shift <= 1e-7, inertia is the sum
    of SQUARED distances of the last E-step; otherwise the sum of plain distances after a re-label."""
    from dask_ml_b200.cluster import KMeans

    Xs, _ = _easy_blobs(oracle)
    X = np.concatenate(Xs)
    init = np.array([[-7.0, -7.0], [0.0, 0.0], [7.0, 7.0]])
    for tol, max_iter in ((1e-4, 300), (0.5, 300), (0.0, 3)):
        km = KMeans(3, init=init, tol=tol, max_iter=max_iter).fit(X)
        lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(oracle.to_blocks(X, 50), 3, init=init, tol=tol,
                                                            max_iter=max_iter)
        assert km.n_iter_ == n_iter
        np.testing.assert_allclose(km.inertia_, inertia, rtol=1e-9)
        np.testing.assert_allclose(km.cluster_centers_, C, rtol=1e-12, atol=1e-14)


def test_empty_cluster_goes_to_origin(oracle):
    """Q1: a centre that attracts no rows becomes the zero vector (no relocation)."""
    from dask_ml_b200.cluster import KMeans

    rng = np.random.RandomState(0)
    X = rng.standard_normal((500, 3)) + 5.0
    init = np.vstack([X[:2], [[100.0, 100.0, 100.0]]])
    km = KMeans(3, init=init, max_iter=1, tol=0.0).fit(X)
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd([X], 3, init=init, max_iter=1, tol=0.0)
    np.testing.assert_allclose(km.cluster_centers_, C, rtol=1e-12, atol=1e-14)
    assert (km.cluster_centers_[2] == 0).all()
    np.testing.assert_allclose(km.inertia_, inertia, rtol=1e-9)


def test_kmeanspp_and_random_init(oracle):
    """tests/test_kmeans.py:100-117."""
    from dask_ml_b200.cluster import KMeans

    Xs, _ = _easy_blobs(oracle)
    X = np.concatenate(Xs)
    a = KMeans(3, init="k-means++", random_state=np.random.RandomState(0)).fit(X)
    b = SKKMeans(3, init="k-means++", random_state=np.random.RandomState(0), n_init=1).fit(X)
    assert abs(a.inertia_ - b.inertia_) < 1e-4 or abs(np.sqrt(a.inertia_) - np.sqrt(b.inertia_)) < 1.0
    assert a.init == "k-means++"
    KMeans(3, init="k-means++").fit(X)
    KMeans(3, init="random", random_state=0).fit(X)


def test_too_small_and_inputs():
    """tests/test_kmeans.py:39-42,149-160: default k=8 on 20 rows; ndarray / chunked / DataFrame / tensor."""
    import pandas as pd
    import torch

    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    rng = np.random.RandomState(0)
    KMeans().fit(ChunkedArray.from_array(rng.uniform(size=(20, 2)), 10))
    for X in (rng.uniform(size=(100, 4)),
              ChunkedArray.from_array(rng.uniform(size=(100, 4)), (10, 4)),
              pd.DataFrame(rng.uniform(size=(100, 4))),
              torch.rand(100, 4, device="cuda"),
              rng.randint(0, 50, size=(100, 4)).astype(np.int32),
              rng.randint(0, 50, size=(100, 4)).astype(np.int64)):
        km = KMeans(n_clusters=3).fit(X)
        t = km.transform(X)
        assert t.shape == (100, 3)


def test_fit_raises():
    """tests/test_kmeans.py:45-51 and NaN/inf handling (k_means.py:179-185)."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    km = KMeans()
    with pytest.raises(ValueError):
        km.fit(np.array([]).reshape(0, 1))
    with pytest.raises(ValueError):
        km.fit(np.array([]).reshape(1, 0))
    X = np.random.RandomState(0).uniform(size=(100, 3))
    X[7, 1] = np.nan
    with pytest.raises(ValueError):
        km.fit(ChunkedArray.from_array(X, 25))
    X[7, 1] = np.inf
    with pytest.raises(ValueError):
        km.fit(ChunkedArray.from_array(X.astype(np.float32), 25))


def test_dtypes():
    """tests/test_kmeans.py:168-182."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    X = np.random.RandomState(0).uniform(size=(100, 2))
    X2 = X.astype("f4")
    for xx, yy in [(X, X), (X2, X2), (X, X2), (X2, X)]:
        a = KMeans().fit(ChunkedArray.from_array(xx, 50))
        b = SKKMeans(n_init=1).fit(xx)
        assert a.cluster_centers_.dtype == b.cluster_centers_.dtype
        assert a.inertia_.dtype == np.float64
        assert a.labels_.dtype == b.labels_.dtype
        assert a.transform(xx).dtype == b.transform(xx).dtype
        assert a.transform(yy).dtype == b.transform(yy).dtype


def test_kmeans_parallel_init_quality(oracle):
    """k-means|| (init_scalable): with enough rounds the candidate set covers every blob, so the fit
    reaches the same inertia as scikit-learn's (smoke-level pin, see SURVEY §8c)."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    rng = np.random.RandomState(1)
    cent = rng.uniform(-20, 20, size=(5, 8))
    X = (cent[rng.randint(0, 5, size=20000)] + 0.2 * rng.standard_normal((20000, 8))).astype(np.float32)
    a = KMeans(5, random_state=0, oversampling_factor=10).fit(ChunkedArray.from_array(X, 6000))
    b = SKKMeans(5, random_state=0, n_init=10).fit(X)
    # inertia_ follows the reference's Q4 rule; compare through predict on the fitted centres
    d = ((X[:, None, :].astype(np.float64) - a.cluster_centers_[None].astype(np.float64)) ** 2).sum(-1).min(1).sum()
    assert d <= 1.05 * b.inertia_


def test_check_estimator():
    """reference tests/test_kmeans.py:21-24 — scikit-learn API conformance."""
    import warnings

    from sklearn.utils.estimator_checks import check_estimator

    from dask_ml_b200.cluster import KMeans

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = check_estimator(KMeans(), on_fail=None)
    bad = [(r["check_name"], str(r["exception"])[:200]) for r in res if r["status"] == "failed"]
    assert not bad, bad


REF_CASES = ["ref_lloyd_f32_64x256", "ref_lloyd_f64_16x8", "ref_lloyd_f32_41x100", "ref_lloyd_f32_13x20_conv"]


@pytest.mark.parametrize("name", REF_CASES)
def test_engine_matches_fixtures_written_by_the_reference(name):
    """The CUDA engine against outputs of the UNMODIFIED reference code (tests/golden/ref_shim.py): same
    n_iter, labels (modulo float64 near-ties), centres, inertia (both Q4 branches), predict and transform."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    g = load_golden(name)
    X = ChunkedArray.from_array(g["X"], int(g["chunks"]))
    km = KMeans(int(g["k"]), init=g["init"], max_iter=int(g["max_iter"]), tol=float(g["tol"])).fit(X)
    assert km.n_iter_ == int(g["n_iter"])
    np.testing.assert_allclose(km.cluster_centers_, g["centers"], rtol=2e-5, atol=2e-5)
    assert km.cluster_centers_.dtype == g["centers"].dtype
    assert_labels_match(km.labels_.compute(), g["labels"], g["X"], g["centers"], rtol=1e-6)
    np.testing.assert_allclose(km.inertia_, float(g["inertia"]), rtol=1e-6)
    km.cluster_centers_ = g["centers"]
    assert_labels_match(km.predict(X).compute(), g["predict"], g["X"], g["centers"], rtol=1e-6)
    tr = km.transform(X).compute()[:256]
    scale = np.sqrt((g["X"][:256].astype(np.float64) ** 2).sum(1)[:, None] + (g["centers"].astype(np.float64) ** 2).sum(1)[None])
    assert np.max(np.abs(tr - g["transform"]) / scale) < (2e-3 if g["X"].dtype == np.float32 else 1e-9)


def test_make_blobs_device_generator_and_c1_through_the_package(oracle):
    """BASELINE config C1 through the package: datasets.make_blobs (100k x 16 float64, 8 blocks, k = 8) -> KMeans.fit,
    against the oracle on the same blocks; plus the device generator's per-block seeding contract."""
    import torch
    from dask_ml_b200.cluster import KMeans
    from dask_ml_b200.datasets import make_blobs

    X, y = make_blobs(n_samples=100_000, n_features=16, centers=8, random_state=0, chunks=12_500)
    init = X.blocks[0][:8].copy()
    km = KMeans(8, init=init, max_iter=20).fit(X)
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd([np.asarray(b) for b in X.blocks], 8, init=init, max_iter=20)
    assert km.n_iter_ == n_iter
    assert int((km.labels_.compute() != np.concatenate(lab)).sum()) == 0
    assert abs(km.inertia_ - inertia) <= 1e-9 * inertia
    # device generator: blocks live on the GPU, block i depends on (centres, i) only
    Xd, yd = make_blobs(n_samples=40_000, n_features=16, centers=8, random_state=0, chunks=10_000, device="cuda")
    Xe, ye = make_blobs(n_samples=25_000, n_features=16, centers=8, random_state=0, chunks=10_000, device="cuda")
    assert Xd.blocks[0].is_cuda and Xd.dtype == np.float64 and yd.dtype == np.int64
    assert torch.equal(Xd.blocks[1], Xe.blocks[1]) and torch.equal(yd.blocks[1], ye.blocks[1])
    assert not torch.equal(Xd.blocks[0], Xd.blocks[1])
    Xh, yh = Xd.compute(), yd.compute()
    Xp, yp = make_blobs(n_samples=10_000, n_features=16, centers=8, random_state=0, chunks=10_000)    # same prototype
    for c in range(8):
        assert abs((yh == c).mean() - 0.125) < 0.01
        np.testing.assert_allclose(Xh[yh == c].mean(0), Xp.compute()[yp.compute() == c].mean(0), atol=0.1)
        assert abs(Xh[yh == c].std(0).mean() - 1.0) < 0.02
    X32, _ = make_blobs(n_samples=1000, n_features=5, centers=3, random_state=1, chunks=500, device="cuda", dtype="float32")
    assert X32.dtype == np.float32
    KMeans(3, init="k-means||", random_state=0).fit(X32)


def test_kmeans_parallel_candidates_match_oracle_with_the_same_philox_stream(oracle):
    """k-means|| steps 1-6 on the GPU against the oracle's restatement of k_means.py:396-435 driven by the SAME
    Philox draws (the reference's own dask draws cannot be reproduced: sampling parity is pinned to this stream):
    identical candidate sets, hence identical cost phi after every round."""
    import torch
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import k_means as km

    rng = np.random.RandomState(4)
    cent = rng.uniform(-15, 15, size=(12, 10))
    X = (cent[rng.randint(0, 12, size=60_000)] + rng.standard_normal((60_000, 10))).astype(np.float32)
    ell = 12
    Xd = km._to_device_data(ChunkedArray.from_array(X, 17_000))
    rs = np.random.RandomState(11)
    got = km._scalable_candidates(Xd, rs, None, ell)
    # the oracle's loop with the engine's per-round seeds
    rs2 = np.random.RandomState(11)
    blocks = oracle.to_blocks(X, 17_000)
    c_idx = {0}
    cost = oracle.evaluate_cost(blocks, oracle._rows(blocks, [0]))
    n_iter = int(np.round(np.log(cost)))
    for _ in range(n_iter):
        seed = int(rs2.randint(0, 2 ** 31 - 1)) | (int(rs2.randint(0, 2 ** 31 - 1)) << 32)
        draw = lambda off, n, seed=seed: oracle.philox_uniform(seed, np.arange(n, dtype=np.uint64) + np.uint64(off))
        c_idx |= set(oracle.sample_points(blocks, oracle._rows(blocks, sorted(c_idx)), ell, draw))
    want = sorted(c_idx)
    # float32 distances vs the oracle's float64: a draw within rounding of its threshold may flip
    assert len(set(got) ^ set(want)) <= max(2, len(want) // 100), (len(got), len(want))
    phi_got = km.evaluate_cost(Xd, Xd.global_rows(got))
    phi_want = oracle.evaluate_cost(blocks, oracle._rows(blocks, want))
    assert abs(phi_got - phi_want) <= 0.02 * phi_want


def test_gpu_candidate_reduce_unweighted_and_weighted():
    """Steps 7-8 on the GPU: the reduced init must be about as good as scikit-learn's KMeans on the same candidates
    (what the reference runs, k_means.py:457-463), and the weighted variant at least as good in cost over X."""
    from sklearn.cluster import KMeans as SK
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import k_means as km

    rng = np.random.RandomState(9)
    cent = rng.uniform(-20, 20, size=(15, 6))
    X = (cent[rng.randint(0, 15, size=40_000)] + 0.5 * rng.standard_normal((40_000, 6))).astype(np.float32)
    Xd = km._to_device_data(ChunkedArray.from_array(X, 10_000))
    cand_idx = km._scalable_candidates(Xd, np.random.RandomState(0), None, 30)
    cand = Xd.global_rows(cand_idx)
    assert len(cand) > 15
    a = km._reduce_candidates(cand, 15, 123, Xd.backend)
    b = SK(15, random_state=0, n_init=10).fit(cand).cluster_centers_
    ca, cb = km.evaluate_cost(Xd, a), km.evaluate_cost(Xd, b)
    assert ca <= 1.25 * cb, (ca, cb)
    c_unw = km.k_init(Xd, 15, "k-means||", random_state=2, oversampling_factor=30)
    c_w = km.k_init(Xd, 15, "k-means||", random_state=2, oversampling_factor=30, weighted=True)
    assert c_unw.shape == c_w.shape == (15, 6)
    assert km.evaluate_cost(Xd, c_w) <= 1.5 * km.evaluate_cost(Xd, c_unw)


def test_host_resident_streaming_on_the_gpu(oracle):
    """Out-of-core ingestion: X stays in (pinned) host memory and is streamed through two device buffers on every sweep;
    same labels / centres as the resident fit and as the oracle."""
    import torch
    from dask_ml_b200.cluster import KMeans
    from dask_ml_b200.engine import host_resident

    rng = np.random.RandomState(8)
    cent = rng.uniform(-10, 10, size=(30, 41))
    X = (cent[rng.randint(0, 30, size=50_000)] + rng.standard_normal((50_000, 41))).astype(np.float32)
    init = X[:100].copy()
    a = KMeans(100, init=init, max_iter=6, tol=0.0).fit(X)
    Xh = host_resident(X, block_rows=12_000)
    assert not isinstance(Xh.chunks, list) and len(Xh.chunks) == 5
    b = KMeans(100, init=init, max_iter=6, tol=0.0).fit(Xh)
    assert a.n_iter_ == b.n_iter_ == 6
    assert int((a.labels_.compute() != b.labels_.compute()).sum()) == 0
    np.testing.assert_allclose(a.cluster_centers_, b.cluster_centers_, rtol=1e-6, atol=1e-6)
    assert abs(a.inertia_ - b.inertia_) <= 1e-9 * a.inertia_
    assert int((b.predict(Xh).compute() != a.predict(X).compute()).sum()) == 0
    tr = b.transform(Xh).compute()
    np.testing.assert_allclose(tr, a.transform(X).compute(), rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_fit_predict_transform_wide_rows(oracle, dtype):
    """784 features (the MNIST shape the reference's users cluster): fit / predict / transform against the oracle."""
    from dask_ml_b200 import ChunkedArray
    from dask_ml_b200.cluster import KMeans

    rng = np.random.RandomState(5)
    n, d, k = 3000, 784, 10
    cent = rng.uniform(0, 1, size=(k, d))
    X = (cent[rng.randint(0, k, size=n)] + 0.1 * rng.standard_normal((n, d))).astype(dtype)
    init = X[:k].copy()
    km = KMeans(k, init=init, max_iter=5, tol=0.0).fit(ChunkedArray.from_array(X, 1100))
    lab, inertia, C, n_iter = oracle.kmeans_single_lloyd(oracle.to_blocks(X, 1100), k, init=init, max_iter=5, tol=0.0)
    assert km.n_iter_ == n_iter
    assert int((km.labels_.compute() != np.concatenate(lab)).sum()) == 0
    assert abs(km.inertia_ - inertia) / inertia < 1e-5
    np.testing.assert_allclose(km.cluster_centers_, C, rtol=1e-4, atol=1e-5)
    assert int((km.predict(X).compute() != np.concatenate(lab)).sum()) == 0
    T = km.transform(X[:500]).compute()
    want = np.sqrt(((X[:500, None, :].astype(np.float64) - km.cluster_centers_[None].astype(np.float64)) ** 2).sum(-1))
    np.testing.assert_allclose(T, want, rtol=2e-4, atol=1e-4)
