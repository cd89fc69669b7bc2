"""Diffusion-map measurement: G.diffusion_map(10) end to end on the device against scipy's eigsh on the host, one
JSON line per graph (kNN graphs, knn=5 decay=40, of the bench's Gaussian mixture: N x 100, intrinsic dimension 10,
seed 3).

Each size runs twice: with the bench's 50 clusters, which lie far apart, so the graph has one component per cluster
and the eigenvalue 1 as many times (more than the solver's block width: the top 11 eigenvalues are all 1); and with
one cluster, a connected graph whose wanted eigenvalues sit just below 1 -- the case a Krylov-type method finds
hard.  Every row records the number of connected components.

* end to end: host clock around diffusion_map(10) (11 eigenpairs, tol 1e-8) and a device synchronise, best of --reps
  after one warm-up call with the same random_state;
* the solver's counters: block width, outer iterations, filter steps;
* the filter-step kernel gtb_spmm_cheb alone, at the solver's block width, on the graph's own diff_aff values: CUDA
  events around --launches launches rotating three [N, b] buffers as the recurrence does.  Its byte model is
  nnz (12 + 8b) + 8 N (3b + 1) (CSR, row gathers, the own rows of Y and Z, the write, indptr); bytes / s over the
  7.7 TB/s HBM3e figure of the B200 data sheet is its share of peak.  The row records whether that working set
  fits the 126 MB L2;
* scipy.sparse.linalg.eigsh(G.diff_aff, k=11, which="LA", tol=1e-8) in a child process with a time cap
  (--eigsh-cap seconds); a run that does not finish in time is recorded as such.  Its eigenvalues are compared with
  the device's.  (With 50 components the eigenvalue 1 has multiplicity 50; single-vector Lanczos may then return
  fewer copies of it than there are.)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import sparse  # noqa: E402
from scipy.sparse.csgraph import connected_components  # noqa: E402

import graphtools_b200 as gt  # noqa: E402
from graphtools_b200 import _engine as E, eigen, spectral, synth  # noqa: E402
from run_shortest_path import HBM_PEAK, gpu_info  # noqa: E402

L2_BYTES = 126e6
EIGSH = """
import sys, time, numpy as np
from scipy import sparse
from scipy.sparse.linalg import eigsh
A = sparse.load_npz(sys.argv[1])
t = time.perf_counter()
w = eigsh(A, k=11, which="LA", tol=1e-8)[0]
print(time.perf_counter() - t, *np.sort(w)[::-1])
"""


def end_to_end(G, reps):
    best = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        G.diffusion_map(10, random_state=0)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    return best


def kernel_row(G, b, launches):
    K = G._dev_kernel
    vals = spectral.diff_aff_values(K, G._dev_degree)
    n, nnz = K.shape[0], K.nnz
    gen = torch.Generator(device="cuda").manual_seed(0)
    bufs = [torch.randn((n, b), dtype=torch.float64, device="cuda", generator=gen) for _ in range(3)]
    coef = eigen.cheb_coefficients(0.99, launches)

    def run():
        cur, prev, out = bufs
        for alpha, beta, gamma in coef:
            E.call("gtb_spmm_cheb", K.indptr, K.indices, vals, n, cur, b, b, alpha, beta, gamma, prev, b, out, b)
            prev, cur, out = cur, out, prev
    run()                                                          # warm-up
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    run()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / launches
    model = nnz * (12 + 8 * b) + 8 * n * (3 * b + 1)
    working_set = nnz * 12 + 8 * (n + 1) + 3 * 8 * n * b
    return dict(cheb_block=b, cheb_launches=launches, cheb_kernel_ms=round(ms, 4), cheb_model_bytes=model,
                cheb_bytes_per_s=model / (ms * 1e-3), cheb_share_of_hbm_peak=round(model / (ms * 1e-3) / HBM_PEAK, 4),
                cheb_working_set_bytes=working_set, cheb_fits_l2=working_set < L2_BYTES)


def eigsh_row(G, w_dev, cap):
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "diff_aff.npz")
        sparse.save_npz(path, sparse.csr_matrix(G.diff_aff), compressed=False)
        try:
            out = subprocess.run([sys.executable, "-c", EIGSH, path], capture_output=True, text=True, timeout=cap)
        except subprocess.TimeoutExpired:
            return dict(eigsh_s=None, eigsh_finished=False, eigsh_cap_s=cap)
    if out.returncode != 0:
        return dict(eigsh_s=None, eigsh_finished=False, eigsh_error=out.stderr.strip().splitlines()[-1:])
    vals = [float(v) for v in out.stdout.split()]
    w = np.array(vals[1:])
    return dict(eigsh_s=round(vals[0], 2), eigsh_finished=True, eigsh_cap_s=cap, eigsh_w=w.tolist(),
                max_abs_w_diff_vs_eigsh=float(np.abs(w - w_dev).max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--dim", type=int, default=100)
    ap.add_argument("--clusters", default="50,1")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--eigsh-cap", type=float, default=240.0)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    E.require_cuda()
    runs = [(int(n), int(c)) for n in args.sizes.split(",") if n for c in args.clusters.split(",") if c]
    for n, clusters in runs:
        X, _ = synth.gaussian_mixture(n, args.dim, n_clusters=clusters, intrinsic_dim=10, seed=3)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            G = gt.Graph(X, knn=5, decay=40, verbose=0)
        G.diffusion_map(10, random_state=0)                            # warm-up of every shape
        st = eigen.stats()
        e2e = end_to_end(G, args.reps)
        w, _ = G.diffusion_eigs(11, random_state=0)
        r = dict(graph="knn5_decay40_%dx%d_%dclusters" % (n, args.dim, clusters), n=n,
                 clusters=clusters, connected_components=int(connected_components(G.K, directed=False)[0]),
                 nnz=st["nnz"],
                 diffusion_map_components=10, k=11, tol=1e-8, diffusion_map_s=round(e2e, 4), block=st["block"],
                 outer_iterations=st["iterations"], filter_steps=st["filter_steps"], w=w.tolist())
        r.update(kernel_row(G, st["block"], args.launches))
        r.update(eigsh_row(G, w, args.eigsh_cap))
        r["gpu"] = gpu_info()
        print(json.dumps(r), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(r) + "\n")
        del G
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
