"""Metric measurement: the 1M x 100 headline mixture of bench.py (knn=5, decay=40, thresh=1e-4) built as a kNN graph
under euclidean, sqeuclidean, cosine and correlation, the four metrics alternating round by round after one warm-up
round, then a 50k x 50 exact correlation graph.  One JSON line per (metric, round) and one summary line per metric
(median device seconds over the rounds) go to stdout and to --out, with the card's name, power limit and maximum SM
clock read in the same call.

Device time is CUDA events around the graph constructor, which builds K and P in HBM: the window covers the upload
of the host rows, the search, the refine, the radius pass, the symmetrisation and the normalisation, and no copy of
the results to the host."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import graphtools_b200 as gt  # noqa: E402
from graphtools_b200 import pipeline, synth  # noqa: E402

METRICS = ("euclidean", "sqeuclidean", "cosine", "correlation")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def timed_build(X, **kw):
    """(device seconds, graph): CUDA events around the build of K and P on the device."""
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        G = gt.Graph(X, verbose=0, **kw)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3, G


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--d", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--exact-n", type=int, default=50_000)
    ap.add_argument("--exact-d", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03b_metrics_1gpu.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_metrics.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    gpu = gpu_info()
    rows = []

    def emit(rec):
        rec["gpu"] = gpu
        print(json.dumps(rec), flush=True)
        rows.append(rec)

    X, _ = synth.gaussian_mixture(a.n, a.d, n_clusters=50, intrinsic_dim=10, seed=3)
    params = dict(knn=5, decay=40, thresh=1e-4)
    times = {m: [] for m in METRICS}
    for r in range(a.rounds + 1):                       # round 0 is the warm-up of every shape
        for m in METRICS:
            dt, G = timed_build(X, distance=m, **params)
            st = pipeline.stats()
            nnz = int(G._dev_kernel.nnz) if isinstance(G._dev_kernel, pipeline.DeviceCSR) else None
            del G
            if r == 0:
                continue
            times[m].append(dt)
            emit(dict(what="knn", metric=m, n=a.n, d=a.d, round=r, device_s=dt, impl=st.get("impl"),
                      radius_rows=st.get("radius_rows"), euclidean_fallback_rows=st.get("euclidean_fallback_rows"),
                      nnz_K=nnz, **params))
    base = statistics.median(times["euclidean"])
    for m in METRICS:
        med = statistics.median(times[m])
        emit(dict(what="knn_summary", metric=m, n=a.n, d=a.d, rounds=a.rounds, median_device_s=med,
                  min_device_s=min(times[m]), max_device_s=max(times[m]), vs_euclidean=med / base,
                  points_per_s=a.n / med))

    Xe, _ = synth.gaussian_mixture(a.exact_n, a.exact_d, n_clusters=20, intrinsic_dim=10, seed=5)
    te = []
    for r in range(a.rounds + 1):
        dt, G = timed_build(Xe, graphtype="exact", distance="correlation", **params)
        del G
        torch.cuda.empty_cache()
        if r:
            te.append(dt)
            emit(dict(what="exact", metric="correlation", n=a.exact_n, d=a.exact_d, round=r, device_s=dt, **params))
    emit(dict(what="exact_summary", metric="correlation", n=a.exact_n, d=a.exact_d, rounds=a.rounds,
              median_device_s=statistics.median(te), min_device_s=min(te), max_device_s=max(te)))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in rows:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
