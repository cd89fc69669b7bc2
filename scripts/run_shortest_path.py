"""K10 measurement: G.shortest_path() end to end on the device against scipy's Dijkstra on the host, one JSON line
per graph (the C1 digits graph, then kNN graphs of N x 100 Gaussian-mixture data).

scipy is timed on the same -log(K) lengths with method="D".  Where running all N sources would take too long, it is
timed on the first --scipy-sources sources and extrapolated linearly in the number of sources (each source is an
independent Dijkstra over the same graph); such rows carry "scipy_fit": "linear_in_sources".

The traversal kernel is timed with CUDA events in a separate run of the same call.  Its byte model is
sum over sources of the edges in the source's component x 12 B (int32 index + float64 length) + 8 N^2 (the distance
block written); achieved bytes / s over the 7.7 TB/s HBM3e figure of the B200 data sheet is its share of peak."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import sparse  # noqa: E402
from scipy.sparse.csgraph import shortest_path as scipy_shortest_path  # noqa: E402

import graphtools_b200 as gt  # noqa: E402
from graphtools_b200 import _engine as E, paths, synth  # noqa: E402

HBM_PEAK = 7.7e12


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def scipy_seconds(G, n_src):
    L = sparse.csr_matrix(G.K, copy=True)
    L.data = -1 * np.log(L.data)
    n = L.shape[0]
    t = time.perf_counter()
    scipy_shortest_path(L, method="D", indices=np.arange(min(n_src, n)))
    dt = time.perf_counter() - t
    return dt if n_src >= n else dt * n / n_src


def device_seconds(G, reps):
    best = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        D = G.shortest_path()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
        del D
    return best


def traversal_ms(G):
    E.timing, E.timing_only = {}, None
    try:
        G.shortest_path()
        return {k: round(ms, 3) for k, (_, ms) in E.timings_ms().items()}
    finally:
        E.timing = None


def row(name, G, args):
    dev_s = device_seconds(G, args.reps)
    st = paths.stats()
    ms = traversal_ms(G)
    n = st["n"]
    full = n <= args.scipy_full_max
    sp_s = scipy_seconds(G, n if full else args.scipy_sources)
    trav_bytes = 12 * st["source_edges"] + 8 * n * n
    t_ms = ms.get("gtb_sp_traverse", float("nan"))
    return dict(graph=name, n=n, nnz=st["nnz"], components=st["components"], batches=st["batches"],
                device_s=round(dev_s, 4), scipy_s=round(sp_s, 3),
                scipy_fit=None if full else "linear_in_sources",
                scipy_sources=n if full else args.scipy_sources, speedup=round(sp_s / dev_s, 1),
                kernel_ms=ms, traversal_model_bytes=trav_bytes,
                traversal_bytes_per_s=trav_bytes / (t_ms * 1e-3),
                traversal_share_of_hbm_peak=round(trav_bytes / (t_ms * 1e-3) / HBM_PEAK, 4), gpu=gpu_info())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="10000,20000,50000")
    ap.add_argument("--dim", type=int, default=100)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--scipy-full-max", type=int, default=10000)
    ap.add_argument("--scipy-sources", type=int, default=1000)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    E.require_cuda()
    rows = []
    from sklearn.datasets import load_digits
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        graphs = [("C1_digits_knn5_decay40", lambda: gt.Graph(load_digits().data.astype(np.float32), knn=5, decay=40,
                                                              verbose=0))]
        for n in [int(s) for s in args.sizes.split(",") if s]:
            graphs.append(("knn5_decay40_%dx%d" % (n, args.dim),
                           lambda n=n: gt.Graph(synth.gaussian_mixture(n, args.dim, n_clusters=10, intrinsic_dim=10,
                                                                       seed=5)[0], knn=5, decay=40, verbose=0)))
        for name, make in graphs:
            G = make()
            G.shortest_path()                      # warm-up of every kernel and allocation of this shape
            try:
                r = row(name, G, args)
            except MemoryError as e:
                r = dict(graph=name, error=str(e))
            print(json.dumps(r), flush=True)
            rows.append(r)
            del G
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
