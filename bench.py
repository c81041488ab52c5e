#!/usr/bin/env python
"""bench.py — Lloyd-iteration samples/sec of the B200 KMeans engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1], "C2"): synthetic blobs 10M x 64 float32, k = 256, one chunk per GPU,
fixed init = first k rows.  A *step* is one full Lloyd iteration as ``KMeans.fit`` runs it
(``dask_ml_b200.cluster.k_means.lloyd_loop`` -> ``LloydState.run``): fused E+M kernel over the resident chunk -> (N>1:
one all-reduce of [k*d sums | k counts | inertia]) -> ``bkm_finalize_step`` (centre update + shift + the stop test of
dask_ml/cluster/k_means.py:552-559 ON THE DEVICE + the next iteration's centre pack); the host reads the loop state
once per batch of 8 iterations.  With N>1 every rank holds its own 10M-row chunk (weak scaling).
Rank 0 prints ONE JSON line.

Numbers reported:
  value         whole-job samples/s with X resident in HBM (CUDA events around the K iterations, max over ranks)
  e2e           same metric through ``lloyd_iteration_host`` with X in pinned HOST memory: every step copies X
                host->device (double-buffered row blocks) and reads the new centres back
  roofline      the fused chunk kernel against the tensor (dense 16-bit) and HBM roofs, algorithmic work 2*d*k flops and
                d*4+4 bytes per sample (SURVEY.md §8d)
  parity_check  labels of the LAST timed iteration on a >= 1M-row slice against the float64 arg-min evaluated on the
                device (mismatches must be float64 near-ties; worst relative margin reported) + deferred-row fraction
  configs       the other BASELINE shapes as sub-records, same loop, same parity check: C3 (4.9M x 41, k=100; with N>1
                the SAME 4.9M rows are split across ranks = strong scaling), C4 (15M x 13, k=20 per GPU = the 8-GPU
                shard of 120M x 13; weak), C5 (125M x 128 bf16 rows per GPU in 8 resident chunks, k=1024; `--configs C5s` = an 8M-row slice)
  allreduce_us  N>1: latency of the per-iteration collective on the [k*d+k+1] float64 buffer, CUDA events
  cpu_baseline  the dask-ml path restated without dask (oracle/: scikit-learn float64 E-step + the reference's numba
                scatter-add, thread pool over row blocks) on a bounded row sample of C2
``--impl reference`` times that CPU path alone on the FULL 10M-row C2 chunk and prints the same line shape.
``--dump-outputs DIR`` writes what the last timed headline step computed (rank 0): ``centers.npy`` (k, d) float64,
``labels.npy`` float32 (every row up to DUMP_LABEL_ROWS, else a fixed seeded sample of that many rows, in row order)
and ``shift.npy`` (1,) float64.  The inputs depend only on the arguments, so two builds can be compared file by file,
with a tolerance: the float64 re-check adds its deferred rows to the sums with atomics, so repeated runs differ in the
last bits, and over many steps such a difference can flip a near-tied label and move the centres further (NVIDIA B200,
1000 W limit, 20 steps: centres within 1e-7 in two of three repeats, within 3e-3 in the third).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# the CPU baseline runs one BLAS thread per row-block task (set before numpy/scipy load their BLAS)
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
os.environ.setdefault("OMP_NUM_THREADS", "1")
os.environ.setdefault("MKL_NUM_THREADS", "1")

import numpy as np  # noqa: E402

METRIC = "kmeans_lloyd_iter_samples_per_sec"

# name -> rows (per GPU for weak configs, total for the strong one), features, clusters, input dtype, scaling
CONFIGS = {
    "C2": dict(n=10_000_000, d=64, k=256, dtype="f32", scaling="weak", gen="blobs", seed=0,
               what="synthetic blobs 10M x 64 float32, k=256 (BASELINE configs[1])"),
    "C3": dict(n=4_898_431, d=41, k=100, dtype="f32", scaling="strong", gen="kdd", seed=1,
               what="KDD-Cup-99-shaped 4,898,431 x 41 float32, k=100 (benchmarks/k_means_kdd.py shape); N>1 splits the SAME rows"),
    "C4": dict(n=15_000_000, d=13, k=20, dtype="f32", scaling="weak", gen="airline", seed=2,
               what="airline-shaped 15M x 13 float32 per GPU, k=20 (the 8-GPU shard of 120M x 13, benchmarks/kmeans_airline.py shape)"),
    "C5": dict(n=125_000_000, chunks=8, d=128, k=1024, dtype="bf16", scaling="weak", gen="blobs", seed=3,
               what="C5: 125M x 128 bf16 rows per GPU (1B rows on 8 GPUs) in 8 resident chunks of 15.6M rows, k=1024 (BASELINE configs[4])"),
    "C5s": dict(n=8_000_000, d=128, k=1024, dtype="bf16", scaling="weak", gen="blobs", seed=3,
                what="slice of C5: 8M x 128 bf16 per GPU, k=1024 (C5 is 125M rows per GPU; samples/s is linear in n)"),
}
N_ROWS, N_FEAT, N_CLUST = CONFIGS["C2"]["n"], CONFIGS["C2"]["d"], CONFIGS["C2"]["k"]
# --dump-outputs: at most 12M labels as float32 (48 MB), so that one dump stays under 64 MB
DUMP_LABEL_ROWS = 12_000_000


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            m = json.load(f)
        src = "measured"
    else:
        m = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
        src = "fallback"
    return m, src


# ------------------------------------------------------------------------------------------ synthetic inputs
def synth_blobs_device(n, d, k_true, seed, device, dtype):
    """k_true isotropic blobs, centres ~U(-10,10)^d, sigma=1, generated on the device in row blocks."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    cent = (torch.rand((k_true, d), generator=g, device=device, dtype=torch.float32) * 20.0 - 10.0)
    X = torch.empty((n, d), device=device, dtype=dtype)
    blk = 1 << 20
    for s in range(0, n, blk):
        m = min(blk, n - s)
        idx = torch.randint(0, k_true, (m,), generator=g, device=device)
        X[s:s + m] = (cent[idx] + torch.randn((m, d), generator=g, device=device, dtype=torch.float32)).to(dtype)
    return X


def synth_config_device(name, n, seed, device):
    """SURVEY.md §8(d) generators.  C3: 38 blob columns + 3 low-cardinality integer-coded columns (values 0..69) like the
    coded categoricals of the KDD table; C4: 20 true centres, heterogeneous column scales 1 ... 1e3."""
    import torch

    cfg = CONFIGS[name]
    d, k = cfg["d"], cfg["k"]
    tdt = torch.bfloat16 if cfg["dtype"] == "bf16" else torch.float32
    if cfg["gen"] == "blobs":
        return synth_blobs_device(n, d, k, 1000 * cfg["seed"] + seed, device, tdt)
    g = torch.Generator(device=device)
    g.manual_seed(1000 * cfg["seed"] + seed)
    X = torch.empty((n, d), device=device, dtype=torch.float32)
    blk = 1 << 20
    if cfg["gen"] == "kdd":
        cent = torch.rand((k, 38), generator=g, device=device) * 20.0 - 10.0
        codes = torch.randint(0, 70, (k, 3), generator=g, device=device).float()
        for s in range(0, n, blk):
            m = min(blk, n - s)
            idx = torch.randint(0, k, (m,), generator=g, device=device)
            X[s:s + m, :38] = cent[idx] + torch.randn((m, 38), generator=g, device=device)
            # the coded columns follow the row's cluster 90 % of the time, else a random code
            rnd = torch.randint(0, 70, (m, 3), generator=g, device=device).float()
            keep = torch.rand((m, 3), generator=g, device=device) < 0.9
            X[s:s + m, 38:] = torch.where(keep, codes[idx], rnd)
    else:   # airline
        scales = torch.logspace(0, 3, d, device=device)
        cent = (torch.rand((k, d), generator=g, device=device) * 20.0 - 10.0) * scales
        for s in range(0, n, blk):
            m = min(blk, n - s)
            idx = torch.randint(0, k, (m,), generator=g, device=device)
            X[s:s + m] = cent[idx] + torch.randn((m, d), generator=g, device=device) * scales
    return X


def synth_blobs_host(n, d, k_true, seed):
    rng = np.random.default_rng(seed)
    cent = rng.uniform(-10, 10, size=(k_true, d)).astype(np.float32)
    X = np.empty((n, d), dtype=np.float32)
    blk = 1 << 20
    for s in range(0, n, blk):
        m = min(blk, n - s)
        idx = rng.integers(0, k_true, size=m)
        X[s:s + m] = cent[idx] + rng.standard_normal((m, d), dtype=np.float32)
    return X


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                pynvml.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            while not self._stop_evt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.02)
        except Exception as e:  # pragma: no cover
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------
# CPU baseline (oracle) — the only place bench.py touches oracle/
# ------------------------------------------------------------------------------------------
def _cpu_versions():
    import sklearn
    import scipy

    v = {"sklearn": sklearn.__version__, "numpy": np.__version__, "scipy": scipy.__version__}
    try:
        import numba

        v["numba"] = numba.__version__
    except Exception:
        v["numba"] = None
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    v["cpu"] = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    return v


def cpu_lloyd_baseline(sample_rows, iters, warm):
    """The dask-ml Lloyd iteration restated without dask (oracle/kmeans_oracle.py: scikit-learn float64 E-step per row
    block + the reference's numba ``_centers_dense``, k_means.py:572-582), row blocks = worker threads = host threads."""
    from oracle import kmeans_oracle as ok
    import subprocess

    if not os.path.exists(os.path.join(ROOT, "oracle", "liboracle_c.so")):
        subprocess.call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    # every host thread; OpenBLAS in this image is built for at most 128 threads
    cores = min(os.cpu_count() or 1, 128)
    try:
        cores = min(cores, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    X = synth_blobs_host(sample_rows, N_FEAT, N_CLUST, 0)
    init = X[:N_CLUST].copy()
    blocks = ok.to_blocks(X, max(1, -(-sample_rows // cores)))
    pool = ok.make_pool(cores)
    mstep, mname = ok.centers_dense, "C scatter-add"
    try:
        ok.centers_dense_numba(X[:1000], np.zeros(1000, dtype=np.int32), N_CLUST)      # JIT warm-up
        mstep, mname = ok.centers_dense_numba, "numba _centers_dense"
    except Exception:
        pass
    centers = init
    times = []
    for i in range(warm + iters):
        t0 = time.perf_counter()
        _, _, centers = ok.lloyd_iteration(blocks, centers, N_CLUST, pool, mstep=mstep)
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
    pool.shutdown()
    t = float(np.median(times))
    return {"value": sample_rows / t, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": "%d of %d rows of C2, %d Lloyd iterations (median), %d row blocks on %d threads, "
                      "scikit-learn float64 E-step + %s" % (sample_rows, N_ROWS, iters, len(blocks), cores, mname),
            "ms_per_iter": t * 1e3, "host_threads": os.cpu_count(), "versions": _cpu_versions()}


def c2_config(n):
    return {"workload": "C2: synthetic blobs %d x %d float32 per GPU, k=%d, one chunk per GPU, fixed init (first k rows)"
                        % (n, N_FEAT, N_CLUST),
            "n_samples_per_gpu": n, "n_features": N_FEAT, "n_clusters": N_CLUST}


def run_reference(args, rank, world):
    if rank != 0:
        return
    n = args.rows
    steps = max(1, args.steps)
    res = cpu_lloyd_baseline(n, steps, max(1, min(args.warmup, 2)))
    line = {
        "metric": METRIC, "value": res["value"], "unit": "samples/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_iter"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
        "config": c2_config(n),
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "host_threads", "versions")},
        "e2e": {"value": res["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# device-side helpers
# ------------------------------------------------------------------------------------------
def parity_check(X, labels, C_used, be, k, rows=1 << 20):
    """Labels of the timed kernel on a slice of rows against the float64 arg-min evaluated on the device.
    A mismatch is acceptable only where float64 itself is (nearly) tied: relative margin <= 1e-9."""
    import torch

    n = int(X.shape[0])
    rows = min(rows, n)
    # slice from the middle of the chunk (tile tails and CTA boundaries included)
    s0 = max(0, (n - rows) // 2) // 32 * 32
    C64 = C_used.double()
    cn = (C64 * C64).sum(1)
    mism = 0
    worst = 0.0
    for s in range(s0, s0 + rows, 1 << 17):
        e = min(s + (1 << 17), s0 + rows)
        xb = X[s:e].double()
        d2 = (xb * xb).sum(1, keepdim=True) + cn[None, :] - 2.0 * xb @ C64.T
        want = d2.argmin(1)
        got = labels[s:e].long()
        bad = got != want
        nb = int(bad.sum())
        if nb:
            mism += nb
            scale = (xb * xb).sum(1)[bad] + cn.max()
            dg = d2[bad].gather(1, got[bad][:, None])[:, 0]
            dw = d2[bad].gather(1, want[bad][:, None])[:, 0]
            worst = max(worst, float(((dg - dw).abs() / scale).max()))
    d = int(X.shape[1])
    fam = int(be.kernel_family(d, k, X.dtype)) if hasattr(be, "kernel_family") else None
    deferred = None
    if fam in (1, 3):
        dr = be.deferred_rows(n, d, k, X.dtype)
        deferred = None if dr is None else dr / float(n)
    return {"rows": int(rows), "mismatches": int(mism), "worst_margin": worst,
            "ok": bool(worst <= 1e-9), "deferred_frac": deferred}


def time_lloyd(st, steps, warmup, barrier, world, dev):
    """W untimed + K timed iterations of ``lloyd_loop`` (tol = 0: every iteration runs); returns (ms per step, mean ms
    of the fused chunk kernel(s) inside a step, kernel launches of this library inside the timed region), max over ranks."""
    import torch
    import torch.distributed as dist
    from dask_ml_b200.cluster.k_means import lloyd_loop

    lloyd_loop(st, warmup, 0.0)
    barrier()
    kev = []

    def hook():
        pair = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        kev.append(pair)
        return pair

    st.kernel_event_hook = hook
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = st.be.launch_count()
    ev0.record()
    _, last, _ = lloyd_loop(st, steps, 0.0)
    ev1.record()
    barrier()
    launches = st.be.launch_count() - l0
    st.kernel_event_hook = None
    if last + 1 != steps:
        raise RuntimeError("the timed loop ran %d of %d iterations" % (last + 1, steps))
    ms_total = ev0.elapsed_time(ev1)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    t = torch.tensor([ms_total, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0]) / steps, float(t[1]), int(launches)


def dump_outputs(out_dir, st):
    """Write what the last step of the timed loop computed (see the module docstring); returns the written shapes."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    labels = st.labels[0]
    n = int(labels.shape[0])
    if n > DUMP_LABEL_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LABEL_ROWS, replace=False))
        labels = labels[torch.from_numpy(rows).to(labels.device)]
    out = {"centers": st.C.cpu().numpy().astype(np.float64),
           "labels": labels.cpu().numpy().astype(np.float32),
           "shift": st.shift.cpu().numpy().astype(np.float64).reshape(1)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "label_rows": "%d of %d" % (out["labels"].shape[0], n),
            "files": {name + ".npy": list(a.shape) for name, a in out.items()}}


def _static_traffic(name):
    """DRAM bytes per launch of the config's dominant kernel from the committed ncu --set full capture
    (profiles/ncu_traffic.json; not measured in this run), or None."""
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(tp) as f:
            return json.load(f).get("configs", {}).get(name, {}).get("dram_bytes_per_launch")
    except (OSError, ValueError):
        return None


def run_config(name, args, be, comm, dev, rank, world, barrier, peaks):
    """One BASELINE shape as a sub-record: same loop, same parity check, HBM roofline."""
    import torch
    from dask_ml_b200.cluster.k_means import LloydState
    from dask_ml_b200.engine import DeviceData

    cfg = CONFIGS[name]
    d, k = cfg["d"], cfg["k"]
    Xs = None
    if cfg["scaling"] == "strong":
        n_total = cfg["n"]
        per = -(-n_total // world)
        lo, hi = rank * per, min(n_total, (rank + 1) * per)
        # every rank generates the same stream and keeps its slice: the N-GPU job clusters the SAME rows
        Xfull = synth_config_device(name, n_total, 0, dev)
        X = Xfull[lo:hi].clone()
        del Xfull
        torch.cuda.empty_cache()
    else:
        n_total = cfg["n"] * world
        nch = int(cfg.get("chunks", 1))
        if nch > 1:
            # several resident chunks per GPU (each its own allocation), generated with their own seeds
            per = -(-cfg["n"] // nch)
            Xs = [synth_config_device(name, min(per, cfg["n"] - c * per), rank * nch + c, dev) for c in range(nch)]
        else:
            X = synth_config_device(name, cfg["n"], rank, dev)
    if Xs is None:
        if d % 4 and be.kernel_family(d, k, X.dtype) == 1:
            X = be.to_device(X, X.dtype)          # the tensor path wants a 16-byte row pitch (padded view)
        Xs = [X]
    X = Xs[0]
    n_local = int(sum(int(x.shape[0]) for x in Xs))
    data = DeviceData(Xs, be, comm)
    init = data.global_rows(list(range(k))).astype(np.float64)
    st = LloydState(data, init)
    steps = max(5, args.steps)
    ms, kern_ms, _ = time_lloyd(st, steps, args.warmup, barrier, world, dev)
    C_used = st.C_new.clone()                 # after accept(): the centres the last E-step ran against
    par = parity_check(X, st.labels[0], C_used, be, k)
    esz = 2 if cfg["dtype"] == "bf16" else 4
    bytes_alg = (d * esz + 4) * n_local
    gbs = bytes_alg / (kern_ms * 1e-3) / 1e9
    flops = 2.0 * d * k * n_local
    tf = flops / (kern_ms * 1e-3) / 1e12
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    t_hbm = bytes_alg / (float(peaks["hbm_gbs"]) * 1e9)
    t_tc = flops / (peak_tf * 1e12)
    bound = "hbm" if t_hbm >= t_tc else "tensor"
    rec = {
        "workload": cfg["what"], "scaling": cfg["scaling"], "n_total": int(n_total), "rows_per_gpu": n_local,
        "chunks_per_gpu": len(Xs),
        "n_features": d, "n_clusters": k, "dtype": cfg["dtype"], "row_pitch_elems": int(X.stride(0)),
        "steps": steps, "ms_per_step": ms, "value": n_total / (ms * 1e-3), "unit": "samples/s",
        "kernel_family": int(be.kernel_family(d, k, X.dtype)), "kernel_ms": kern_ms,
        "roofline": {"bound": bound,
                     "achieved": gbs if bound == "hbm" else tf, "peak": float(peaks["hbm_gbs"]) if bound == "hbm" else peak_tf,
                     "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
                     "frac": (gbs / float(peaks["hbm_gbs"])) if bound == "hbm" else tf / peak_tf,
                     "hbm_gbs": gbs, "tflops": tf,
                     "traffic": _static_traffic(name),
                     "algorithmic": {"bytes_per_sample": d * esz + 4, "flops_per_sample": 2 * d * k}},
        "parity_check": par, "final_shift": float(st.shift.item()),
    }
    del st, data, X, Xs
    torch.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=N_ROWS, help="rows per GPU of the headline workload (default: C2)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3/C4/C5 sub-records")
    ap.add_argument("--configs", default="C3,C4,C5", help="comma-separated sub-records to run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the centres, labels and shift of the last timed headline step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (the hot path is sm_100a CUDA; there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from dask_ml_b200.cluster.k_means import LloydState, lloyd_iteration_host
    from dask_ml_b200.engine import Comm, CudaBackend, DeviceData

    be = CudaBackend(dev)
    comm = Comm()
    peaks, peak_src = _peaks()
    n = args.rows
    X = synth_blobs_device(n, N_FEAT, N_CLUST, 1000 + rank, dev, torch.float32)
    data = DeviceData([X], be, comm)
    init = X[:N_CLUST].cpu().numpy().astype(np.float64)
    if world > 1:
        init = comm.bcast_obj(init)
    st = LloydState(data, init)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- headline: W + K Lloyd iterations exactly as fit runs them (device-resident X, 2.56 GB per GPU >> L2) ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_per_step, kern_ms, launches = time_lloyd(st, args.steps, args.warmup, barrier, world, dev)
    clocks = sampler.stop()
    value = n * world / (ms_per_step * 1e-3)
    shift = float(st.shift.item())
    dumped = dump_outputs(args.dump_outputs, st) if args.dump_outputs and rank == 0 else None
    C_used = st.C_new.clone()
    par = parity_check(X, st.labels[0], C_used, be, N_CLUST)

    # ---- latency of the per-iteration collective (N > 1) ----
    allreduce_us = None
    if world > 1:
        buf = torch.zeros_like(st.red)
        for _ in range(5):
            comm.allreduce_sum_(buf)
        barrier()
        a0 = torch.cuda.Event(enable_timing=True)
        a1 = torch.cuda.Event(enable_timing=True)
        reps = 50
        a0.record()
        for _ in range(reps):
            comm.allreduce_sum_(buf)
        a1.record()
        barrier()
        ta = torch.tensor([a0.elapsed_time(a1) / reps * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(ta, op=dist.ReduceOp.MAX)
        allreduce_us = {"value": float(ta[0]), "payload_bytes": int(buf.numel() * 8),
                        "how": "mean of %d back-to-back all-reduces of the step's [k*d+k+1] float64 buffer, CUDA events, max over ranks" % reps,
                        "bus_gbs": float(buf.numel() * 8 * 2 * (world - 1) / world / (float(ta[0]) * 1e-6) / 1e9)}

    # ---- e2e: host-resident X, H2D inside the timed region, through the public host-buffer call ----
    e2e = None
    if not args.no_e2e:
        e_rows = n
        Xh = torch.empty((e_rows, N_FEAT), dtype=torch.float32, pin_memory=True)
        blk = 1 << 20
        for s in range(0, e_rows, blk):
            Xh[s:s + blk].copy_(X[s:s + blk])
        torch.cuda.synchronize()
        centers = init.copy()
        e_steps = max(2, min(args.steps, 4))
        lloyd_iteration_host(Xh, centers, backend=be, comm=comm)      # warm-up (allocations, pinned pages)
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(e_steps):
            centers, inertia_h, shift_h = lloyd_iteration_host(Xh, centers, backend=be, comm=comm)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ems = max(e0.elapsed_time(e1), wall * 1e3) / e_steps
        te = torch.tensor([ems], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        ems = float(te[0])
        e2e = {"value": e_rows * world / (ems * 1e-3), "unit": "samples/s",
               "h2d_bytes_per_step": int(e_rows * N_FEAT * 4 + N_CLUST * N_FEAT * 8),
               "d2h_bytes_per_step": int(N_CLUST * N_FEAT * 8 + 16), "ms_per_step": ems, "steps": e_steps,
               "api": "dask_ml_b200.cluster.k_means.lloyd_iteration_host (pinned host X, double-buffered H2D)"}
        del Xh
    fam_c2 = int(be.kernel_family(N_FEAT, N_CLUST, torch.float32))
    # ---- KMeans.transform on C2: (n, k) float32 distances = 10.24 GB of output per pass: the HBM WRITE roof binds ----
    xform = None
    try:
        tn = min(n, 4_000_000)                      # 4M x 256 float32 = 4.1 GB output block (linear in n)
        out = torch.empty((tn, N_CLUST), dtype=torch.float32, device=dev)
        pack = be.pack_centers(C_used, torch.float32)
        for _ in range(2):
            be.transform_chunk(X[:tn], pack, N_CLUST, out)
        barrier()
        x0 = torch.cuda.Event(enable_timing=True)
        x1 = torch.cuda.Event(enable_timing=True)
        x0.record()
        reps = 5
        for _ in range(reps):
            be.transform_chunk(X[:tn], pack, N_CLUST, out)
        x1.record()
        barrier()
        xms = x0.elapsed_time(x1) / reps
        xb = tn * (N_CLUST * 4 + N_FEAT * 4)
        ref = torch.sqrt(torch.clamp(((X[:4096].double()[:, None, :] - C_used[None, :, :]) ** 2).sum(-1), min=0.0))
        xerr = float(((out[:4096].double() - ref).abs() / (1.0 + ref)).max())
        xform = {"what": "KMeans.transform / euclidean_distances: (n, k) float32 block, %d x %d -> %d" % (tn, N_FEAT, N_CLUST),
                 "ms": xms, "rows": tn, "samples_per_s": tn / (xms * 1e-3),
                 "roofline": {"bound": "hbm", "achieved": xb / (xms * 1e-3) / 1e9, "peak": float(peaks["hbm_gbs"]),
                              "unit": "GB/s", "frac": xb / (xms * 1e-3) / 1e9 / float(peaks["hbm_gbs"]),
                              "algorithmic": {"bytes_per_sample": N_CLUST * 4 + N_FEAT * 4}},
                 "max_rel_err_vs_float64": xerr}
        del out
    except Exception as e:
        xform = {"error": "%s: %s" % (type(e).__name__, e)}
    del st, data, X
    torch.cuda.empty_cache()

    # ---- the other BASELINE shapes ----
    configs = {}
    if not args.no_configs:
        for name in [c for c in args.configs.split(",") if c]:
            if name not in CONFIGS or name == "C2":
                continue
            if CONFIGS[name]["dtype"] == "bf16" and not getattr(be, "supports_bf16", False):
                configs[name] = {"workload": CONFIGS[name]["what"], "unavailable": "bf16 input is not supported by this build"}
                continue
            try:
                configs[name] = run_config(name, args, be, comm, dev, rank, world, barrier, peaks)
            except Exception as e:  # a sub-record must never take the headline down
                configs[name] = {"workload": CONFIGS[name]["what"], "error": "%s: %s" % (type(e).__name__, e)}
                torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    flops = 2.0 * N_FEAT * N_CLUST * n
    bytes_alg = (N_FEAT * 4 + 4) * n
    ach_tf = flops / (kern_ms * 1e-3) / 1e12
    ach_gbs = bytes_alg / (kern_ms * 1e-3) / 1e9
    # The product runs on the kind::f16 tensor pipe (split-fp16, 3 products + the ||c||^2 step = 3.25x the
    # algorithmic flops), so the roof is the measured dense 16-bit peak: the sustained figure, because the
    # kernel is timed inside a long step.
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    peak_note = "%s dense bf16/fp16 tensor peak, sustained (MEASURED_PEAKS.json)" % peak_src
    issued_ratio = 3.25
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    roofline = {
        "bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
        "traffic": traffic, "traffic_source": "static: ncu --set full capture committed under profiles/ (not measured in this run)",
        "peak_source": peak_note, "kernel_ms": kern_ms,
        "kernel": "tc_chunk_kernel<true,false> (tcgen05 split-fp16 fused E+M) + tc_recheck + reduce_partials",
        "limiter": "three 128-column TMEM accumulator buffers x (epilogue ~3.0-3.6k cycles at ~6.8 B/clk of TMEM reads per warp "
                   "+ MMA refill ~1.0-1.5k) per 2-unit tile; tensor pipe 43 %, issue slots 71 % (DESIGN.md (d), profiles/r02_ncu_tc_chunk_C2.md)",
        "issued": {"tflops": ach_tf * issued_ratio, "frac": ach_tf * issued_ratio / peak_tf,
                   "note": "tensor-pipe work actually issued: 3 fp16 products + ||c||^2 step per algorithmic product"},
        "hbm": {"achieved": ach_gbs, "peak": float(peaks["hbm_gbs"]), "unit": "GB/s",
                "frac": ach_gbs / float(peaks["hbm_gbs"]), "peak_source": peak_src},
        "algorithmic": {"flops_per_sample": 2 * N_FEAT * N_CLUST, "bytes_per_sample": N_FEAT * 4 + 4,
                        "samples_per_launch": n},
    }
    cpu = None
    if not args.no_cpu:
        cpu = cpu_lloyd_baseline(1_000_000, 3, 1)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "host_threads", "versions")}
    cfg = c2_config(n)
    line = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "detail": {"arithmetic": "split-fp16 (hi,lo) x3 product on tcgen05 kind::f16, fp32 accumulate, float64 re-check of near-ties + float64 centre update",
                   "l2": "inputs (%.2f GB per GPU) are larger than L2 (126 MB); no explicit flush" % (n * N_FEAT * 4 / 1e9),
                   "step": "lloyd_loop() as KMeans.fit runs it: fused E+M kernel + reduce + re-check (+ all-reduce) + finalize_step (centre update, shift, device-side stop test, next pack); one host read of the loop state per 8 iterations",
                   "kernel_family": fam_c2, "final_shift": shift},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "parity_check": par,
        "allreduce_us": allreduce_us, "transform": xform, "configs": configs, "cpu_baseline": cpu,
    }
    if dumped:
        line["dump_outputs"] = dumped
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
