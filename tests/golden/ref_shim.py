"""TEST INFRASTRUCTURE — run the UNMODIFIED reference source files without dask.

    python tests/golden/ref_shim.py          # regenerates tests/golden/ref_*.npz  (needs /root/reference)

The reference (mrocklin/dask-ml @ 0310a90) cannot be imported in this image: dask / distributed / toolz are
absent and the 2018 code targets Python <= 3.9 / scikit-learn 0.19.  Its KMeans path, however, only uses a
small slice of dask: row-chunked arrays that are mapped block-wise and reduced on the client.  This module
installs an EAGER stand-in for exactly that slice (``dask``, ``dask.array``, ``dask.dataframe``) into
``sys.modules``, stubs the two removed scikit-learn names the reference imports, and then loads the reference's
own files from ``/root/reference`` with importlib — ``dask_ml/utils.py``, ``dask_ml/metrics/pairwise.py``,
``dask_ml/cluster/k_means.py`` — byte for byte, nothing copied into this repository.  The per-chunk arithmetic
therefore runs through the reference's own code: its graph construction (``pairwise_distances_argmin_min``,
``da.atop(_centers_dense, ...)``, the sequential ``sum`` of block partials, ``da.bincount``), its numba kernel
``_centers_dense`` and its Lloyd control flow.

The outputs are written as golden fixtures (inputs + reference outputs) that tests/test_oracle.py replays
against the oracle and tests/test_gpu_kmeans.py against the CUDA engine, without the reference checkout.  The
Lloyd fixtures store the parameters of ``tests/_util.blobs`` and the SHA-256 of the input rows instead of the
rows themselves (``tests/_util.load_golden`` regenerates and checks them).
"""
import collections
import collections.abc
import importlib.util
import os
import sys
import types

import numpy as np

REF = os.environ.get("BKM_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from _util import blobs, x_digest  # noqa: E402


# --------------------------------------------------------------------------------------------------
# eager stand-in for the slice of dask.array the KMeans path touches
# --------------------------------------------------------------------------------------------------
class Array(object):
    """Row-chunked array evaluated eagerly: a list of numpy blocks (chunks on axis 0 only)."""

    def __init__(self, blocks):
        self.blocks = [np.asarray(b) for b in blocks]

    # metadata -----------------------------------------------------------------
    @property
    def ndim(self):
        return self.blocks[0].ndim

    @property
    def dtype(self):
        return self.blocks[0].dtype

    @property
    def shape(self):
        n = sum(b.shape[0] for b in self.blocks) if self.ndim else ()
        return (n,) + tuple(self.blocks[0].shape[1:]) if self.ndim else ()

    @property
    def chunks(self):
        if self.ndim == 0:
            return ()
        return (tuple(b.shape[0] for b in self.blocks),) + tuple((s,) for s in self.blocks[0].shape[1:])

    @property
    def numblocks(self):
        return tuple(len(c) for c in self.chunks)

    @property
    def nbytes(self):
        return sum(b.nbytes for b in self.blocks)

    def __len__(self):
        return self.shape[0]

    # evaluation ----------------------------------------------------------------
    def compute(self):
        if self.ndim == 0:
            return self.blocks[0][()]
        return self.blocks[0] if len(self.blocks) == 1 else np.concatenate(self.blocks, axis=0)

    def __array__(self, dtype=None, copy=None):
        a = self.compute()
        return a.astype(dtype) if dtype is not None else a

    def _like(self, full):
        """Re-chunk a full result like self (same row split) when the leading dim matches."""
        full = np.asarray(full)
        if full.ndim and self.ndim and full.shape[0] == self.shape[0]:
            out, s = [], 0
            for b in self.blocks:
                out.append(full[s:s + b.shape[0]])
                s += b.shape[0]
            return Array(out)
        return Array([full])

    # block-wise ops -------------------------------------------------------------
    def map_blocks(self, func, *args, **kwargs):
        for k in ("dtype", "chunks", "drop_axis", "new_axis"):
            kwargs.pop(k, None)
        return Array([func(b, *args, **kwargs) for b in self.blocks])

    def to_delayed(self):
        arr = np.empty(len(self.blocks), dtype=object)
        for i, b in enumerate(self.blocks):
            arr[i] = b
        return arr

    def astype(self, dt):
        return Array([b.astype(dt) for b in self.blocks])

    def rechunk(self, *a, **k):
        return self

    def persist(self):
        return self

    # reductions / elementwise ------------------------------------------------------
    def sum(self, axis=None):
        return Array([np.asarray(self.compute().sum(axis=axis))])

    def min(self, axis=None):
        return self._like(self.compute().min(axis=axis))

    def any(self):
        return Array([np.asarray(self.compute().any())])

    def _bin(self, other, op):
        o = other.compute() if isinstance(other, Array) else other
        return self._like(op(self.compute(), o))

    def __add__(self, o): return self._bin(o, np.add)
    def __radd__(self, o): return self._bin(o, lambda a, b: b + a)
    def __sub__(self, o): return self._bin(o, np.subtract)
    def __mul__(self, o): return self._bin(o, np.multiply)
    def __rmul__(self, o): return self._bin(o, lambda a, b: b * a)
    def __truediv__(self, o): return self._bin(o, np.true_divide)
    def __pow__(self, o): return self._bin(o, np.power)
    def __gt__(self, o): return self._bin(o, np.greater)
    def __lt__(self, o): return self._bin(o, np.less)

    @property
    def T(self):
        return Array([self.compute().T])

    def __getitem__(self, key):
        return self._like(self.compute()[key])


def _compute(*args, **kwargs):
    def ev(x):
        if isinstance(x, Array):
            return x.compute()
        if isinstance(x, (tuple, list)):
            return type(x)(ev(v) for v in x)
        return x
    return tuple(ev(a) for a in args)


def _delayed(func=None, pure=None, nout=None, **kw):
    """dask.delayed evaluated immediately (the value IS the 'delayed' object)."""
    def wrap(*args, **kwargs):
        return func(*[a.compute() if isinstance(a, Array) else a for a in args], **kwargs)
    return wrap


def _from_array(x, chunks=None):
    x = np.asarray(x)
    rows = chunks[0] if isinstance(chunks, (tuple, list)) else chunks
    if isinstance(rows, (tuple, list)):
        out, s = [], 0
        for m in rows:
            out.append(x[s:s + m]); s += m
        return Array(out)
    rows = max(1, int(rows))
    return Array([x[i:i + rows] for i in range(0, len(x), rows)] or [x])


def _from_delayed(value, shape=None, dtype=None):
    return Array([np.asarray(value)])


def _concatenate(arrs, axis=0):
    blocks = []
    for a in arrs:
        blocks.extend(a.blocks if isinstance(a, Array) else [np.asarray(a)])
    return Array(blocks)


def _atop(func, out_ind, *args, **kwargs):
    """da.atop / blockwise for the single pattern the reference uses (k_means.py:531-544): every array
    argument is chunked identically along 'i'; literal arguments carry index None."""
    adjust = kwargs.pop("adjust_chunks", None)
    kwargs.pop("dtype", None)
    pairs = list(zip(args[0::2], args[1::2]))
    nblk = max(len(a.blocks) for a, ind in pairs if isinstance(a, Array))
    outs = []
    for b in range(nblk):
        call = [a.blocks[b] if isinstance(a, Array) else a for a, ind in pairs]
        outs.append(func(*call, **kwargs))
    return Array(outs)


def _bincount(x, minlength=0):
    return Array([np.bincount(x.compute(), minlength=minlength)])


def _elementwise(fn):
    def f(x, *a):
        a = [v.compute() if isinstance(v, Array) else v for v in a]
        return x._like(fn(x.compute(), *a)) if isinstance(x, Array) else fn(x, *a)
    return f


class _RandomState(object):
    """Stands in for dask.array.random.RandomState: numpy draws (the reference's per-chunk seeding scheme lives
    in dask itself and is not reproducible here — k-means|| sampling parity stays unpinned, see DESIGN.md)."""

    def __init__(self, seed=None):
        self._rs = np.random.RandomState(seed)

    def uniform(self, low=0.0, high=1.0, size=None, chunks=None):
        n = size if isinstance(size, int) else size[0]
        full = self._rs.uniform(low, high, size=n)
        if chunks is not None and isinstance(chunks, tuple) and isinstance(chunks[0], tuple):
            out, s = [], 0
            for m in chunks[0]:
                out.append(full[s:s + m]); s += m
            return Array(out)
        return Array([full])

    def randint(self, low, high=None, size=None, chunks=None, **kw):
        return Array([np.asarray(self._rs.randint(low, high, size=size, dtype=np.int64))])

    def choice(self, a, size=None, replace=True, chunks=None):
        return Array([self._rs.choice(a, size=size, replace=replace)])


def install():
    """Put the stand-in modules into sys.modules and return the loaded reference modules."""
    if not hasattr(collections, "Sequence"):
        collections.Sequence = collections.abc.Sequence          # dask_ml/utils.py:5 (Python < 3.10 name)

    dask = types.ModuleType("dask")
    dask.__version__ = "0.18.0"
    dask.compute = _compute
    dask.delayed = _delayed
    da = types.ModuleType("dask.array")
    da.Array = Array
    da.from_array = _from_array
    da.from_delayed = _from_delayed
    da.concatenate = _concatenate
    da.vstack = lambda arrs: _concatenate(arrs)
    da.hstack = lambda arrs: _concatenate(arrs)
    da.atop = _atop
    da.blockwise = _atop
    da.bincount = _bincount
    da.compute = _compute
    da.maximum = _elementwise(np.maximum)
    da.sqrt = _elementwise(np.sqrt)
    da.isnull = _elementwise(lambda x: np.isnan(x))
    da.isinf = _elementwise(np.isinf)
    da.dot = lambda a, b: a._like(np.dot(a.compute(), b.compute() if isinstance(b, Array) else b))
    da.where = lambda c: tuple(Array([v]) for v in np.where(c.compute()))
    dar = types.ModuleType("dask.array.random")
    dar.RandomState = _RandomState
    dar.doc_wraps = lambda f: (lambda g: g)
    da.random = dar
    dau = types.ModuleType("dask.array.utils")
    dau.assert_eq = lambda a, b, **k: np.testing.assert_allclose(np.asarray(a), np.asarray(b), **k)
    da.utils = dau
    dac = types.ModuleType("dask.array.core")
    da.core = dac
    dd = types.ModuleType("dask.dataframe")

    class _DF(object):
        pass
    dd.DataFrame = _DF
    dd.Series = _DF
    ddu = types.ModuleType("dask.dataframe.utils")
    ddu.assert_eq = lambda *a, **k: None
    dd.utils = ddu
    dask.array = da
    dask.dataframe = dd
    for name, mod in (("dask", dask), ("dask.array", da), ("dask.array.random", dar), ("dask.array.utils", dau),
                      ("dask.array.core", dac), ("dask.dataframe", dd), ("dask.dataframe.utils", ddu)):
        sys.modules[name] = mod

    # scikit-learn names removed since the reference was written (k_means.py:12, test_kmeans.py:15)
    import sklearn.cluster
    from sklearn.cluster import KMeans as _KM, kmeans_plusplus
    from sklearn.utils.extmath import row_norms
    km_ = types.ModuleType("sklearn.cluster.k_means_")

    def _k_init(X, n_clusters, x_squared_norms=None, random_state=None, **kw):
        centers, _ = kmeans_plusplus(np.asarray(X), n_clusters, random_state=random_state)
        return centers
    km_._k_init = _k_init
    km_.KMeans = lambda n_clusters, random_state=None: _KM(n_clusters, random_state=random_state, n_init=10)
    km_.row_norms = row_norms
    sys.modules["sklearn.cluster.k_means_"] = km_
    sklearn.cluster.k_means_ = km_

    # package skeleton + the reference's own files
    def pkg(name, path):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m
        return m

    def load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    root = os.path.join(REF, "dask_ml")
    pkg("dask_ml", root)
    load("dask_ml._compat", os.path.join(root, "_compat.py"))
    utils = load("dask_ml.utils", os.path.join(root, "utils.py"))
    mpk = pkg("dask_ml.metrics", os.path.join(root, "metrics"))
    pw = load("dask_ml.metrics.pairwise", os.path.join(root, "metrics", "pairwise.py"))
    for n in ("pairwise_distances", "pairwise_distances_argmin_min", "euclidean_distances"):
        setattr(mpk, n, getattr(pw, n))
    pkg("dask_ml.cluster", os.path.join(root, "cluster"))
    km = load("dask_ml.cluster.k_means", os.path.join(root, "cluster", "k_means.py"))
    return types.SimpleNamespace(da=da, utils=utils, pairwise=pw, k_means=km)


# --------------------------------------------------------------------------------------------------
# fixture generation
# --------------------------------------------------------------------------------------------------
CASES = {
    # name: (n, d, k, k_true, dtype, chunks, max_iter, tol, seed)
    "ref_lloyd_f32_64x256": (6000, 64, 256, 80, "float32", 2500, 6, 1e-4, 21),
    "ref_lloyd_f64_16x8": (4000, 16, 8, 8, "float64", 1000, 100, 1e-4, 22),
    "ref_lloyd_f32_41x100": (5000, 41, 100, 30, "float32", 2000, 6, 1e-4, 23),
    "ref_lloyd_f32_13x20_conv": (8000, 13, 20, 20, "float32", 3000, 300, 1e-9, 24),
}


def main():
    ref = install()
    da, KM = ref.da, ref.k_means.KMeans
    manifest = {}
    for name, (n, d, k, kt, dt, chunks, max_iter, tol, seed) in CASES.items():
        X = blobs(n, d, kt, seed, dt)
        init = X[:k].copy()
        Xd = da.from_array(X, chunks=(chunks, d))
        est = KM(n_clusters=k, init=init, max_iter=max_iter, tol=tol).fit(Xd)          # the reference's own fit
        labels = np.asarray(est.labels_.compute())
        pred = np.asarray(est.predict(Xd).compute())
        trans = np.asarray(est.transform(Xd).compute())
        np.savez_compressed(os.path.join(HERE, name + ".npz"), blobs=np.array([n, d, kt, seed]), dtype=dt,
                            X_sha256=x_digest(X), init=init, k=k, chunks=chunks, max_iter=max_iter,
                            tol=tol, labels=labels, centers=est.cluster_centers_, inertia=np.float64(est.inertia_),
                            n_iter=est.n_iter_, predict=pred, transform=trans[:256])
        manifest[name] = dict(n=n, d=d, k=k, dtype=dt, n_iter=int(est.n_iter_), inertia=float(est.inertia_))
        print(name, manifest[name])
    # per-chunk operator pins (reference tests/metrics/test_metrics.py:16-43)
    Xc = blobs(1000, 4, 5, 31, "float64")
    centers = Xc[::100]
    a, b = ref.pairwise.pairwise_distances_argmin_min(da.from_array(Xc, chunks=(500, 4)), centers)
    pd_ = ref.pairwise.pairwise_distances(da.from_array(Xc, chunks=(500, 4)), centers)
    np.savez_compressed(os.path.join(HERE, "ref_pairwise_ops.npz"), X=Xc, centers=centers, argmin=a.compute(),
                        mins=b.compute(), dists=pd_.compute())
    import json
    with open(os.path.join(HERE, "REF_MANIFEST.json"), "w") as f:
        json.dump({"reference": "mrocklin/dask-ml @ 0310a90 run through tests/golden/ref_shim.py", "cases": manifest},
                  f, indent=1)


if __name__ == "__main__":
    main()
