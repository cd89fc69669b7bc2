"""Graph-filter measurement: the fused Chebyshev filter step, estimate_lmax and heat_filter on the bench's graph (kNN,
knn=5 decay=40, on the bench's Gaussian mixture: 1M x 100, 50 clusters, intrinsic dimension 10, seed 3).  One JSON
line per measurement, appended to --out (default: a file in the system temporary directory).

* step rows: gtb_spmm_cheb_acc on the combinatorial Laplacian's factor values, (alpha, beta, gamma) = (1, 0, -1),
  rotating two [N, f] buffers as the recurrence does, for f in --widths and F in --banks: CUDA events around
  --launches launches after one warm-up pass.  Byte model nnz (12 + 8f) + 8 N (f (3 + 2F) + 1) (CSR, row gathers,
  the own rows of Y and Z, the write of out, the read and write of every accumulator, indptr); bytes / s over the
  7.7 TB/s HBM3e figure of the B200 data sheet is its share of peak.  The same run times the unfused alternatives:
  gtb_spmm_cheb followed by F accumulations in torch, once as r += c * out (a product and a sum kernel per
  accumulator: numpy's rounding, the result the fused step reproduces) and once as one torch.add(r, out, alpha=c)
  per accumulator (one pass, but fused multiply-add rounding);
* lmax rows: G.estimate_lmax per Laplacian type from a cold cache (host clock and a device synchronise, Laplacian
  assembly included and timed apart), with the Lanczos step count;
* filter row: G.heat_filter(onehot, tau=60, order=50) on one-hot labels of --labels random samples (MELD-style),
  best of --reps on the device, against the numpy / scipy restatement of pygsp's cheby_op on the host with the same
  lmax (tests/gsp_reference.py), and the L1 norm of their difference.
"""
import argparse
import json
import os
import sys
import tempfile
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import graphtools_b200 as gt  # noqa: E402
from graphtools_b200 import _engine as E, gsp, synth  # noqa: E402
from run_shortest_path import HBM_PEAK, gpu_info  # noqa: E402
from tests import gsp_reference as ref  # noqa: E402


def _events(fn, launches):
    fn()                                                           # warm-up
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / launches


def step_row(L, vals, f, F, launches):
    n, nnz = L.shape[0], L.nnz
    gen = torch.Generator(device="cuda").manual_seed(0)
    bufs = [torch.randn((n, f), dtype=torch.float64, device="cuda", generator=gen) * 1e-3 for _ in range(2)]
    R = torch.zeros((F, n, f), dtype=torch.float64, device="cuda")
    coef = torch.full((F,), 1e-3, dtype=torch.float64, device="cuda")
    cf = [1e-3] * F

    def fused():
        cur, old = bufs
        for _ in range(launches):
            E.call("gtb_spmm_cheb_acc", L.indptr, L.indices, vals, n, cur, f, f, 1.0, 0.0, -1.0, old, f, old, f, coef,
                   F, R, f, n * f)
            cur, old = old, cur

    def unfused(exact):
        cur, old = bufs
        for _ in range(launches):
            E.call("gtb_spmm_cheb", L.indptr, L.indices, vals, n, cur, f, f, 1.0, 0.0, -1.0, old, f, old, f)
            for a in range(F):
                if exact:
                    R[a] += cf[a] * old
                else:
                    torch.add(R[a], old, alpha=cf[a], out=R[a])
            cur, old = old, cur

    ms = {}
    for rep in range(2):                                           # alternate, so drift hits both alike
        for name, fn in [("fused", fused), ("unfused_exact", lambda: unfused(True)),
                         ("unfused_add_alpha", lambda: unfused(False))]:
            t = _events(fn, launches)
            ms[name] = t if rep == 0 else min(ms[name], t)
    model = nnz * (12 + 8 * f) + 8 * n * (f * (3 + 2 * F) + 1)
    return dict(kind="step", f=f, F=F, n=n, nnz=nnz, launches=launches, model_bytes=model,
                fused_ms=round(ms["fused"], 4), fused_share_of_hbm_peak=round(model / (ms["fused"] * 1e-3) / HBM_PEAK, 4),
                unfused_exact_ms=round(ms["unfused_exact"], 4), unfused_add_alpha_ms=round(ms["unfused_add_alpha"], 4),
                fused_speedup_vs_exact=round(ms["unfused_exact"] / ms["fused"], 3),
                fused_speedup_vs_add_alpha=round(ms["unfused_add_alpha"] / ms["fused"], 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--d", type=int, default=100)
    ap.add_argument("--clusters", type=int, default=50)
    ap.add_argument("--widths", default="1,8,32")
    ap.add_argument("--banks", default="1,4")
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--labels", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "graph_filter.jsonl"))
    args = ap.parse_args()
    E.require_cuda()
    gpu = gpu_info()
    X, _ = synth.gaussian_mixture(args.n, args.d, n_clusters=args.clusters, intrinsic_dim=10, seed=3)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        G = gt.Graph(X, knn=5, decay=40, verbose=0)
    graph = "knn5_decay40_%dx%d_%dclusters" % (args.n, args.d, args.clusters)
    rows = []

    for lap_type in ("combinatorial", "normalized"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        L, _ = gsp.laplacian_device(G, lap_type)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        lmax = G.estimate_lmax(lap_type)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        st = gsp.stats()
        rows.append(dict(kind="lmax", lap_type=lap_type, n=L.shape[0], nnz_L=L.nnz, laplacian_s=round(t1 - t0, 4),
                         estimate_lmax_s=round(t2 - t1, 4), lanczos_steps=st["lanczos_steps"], stop=st["stop"],
                         theta=st["theta"], residual=st["residual"], lmax=lmax))

    L, _ = gsp.laplacian_device(G, "combinatorial")
    lmax = G.estimate_lmax("combinatorial")
    vals = gsp.factor_values(L, lmax / 2, lmax / 2)
    for f in [int(v) for v in args.widths.split(",")]:
        for F in [int(v) for v in args.banks.split(",")]:
            rows.append(step_row(L, vals, f, F, args.launches))
            torch.cuda.empty_cache()

    labels = np.random.default_rng(0).integers(0, args.labels, size=args.n)
    onehot = np.eye(args.labels)[labels]
    G.heat_filter(onehot, tau=60, order=50)                        # warm-up
    best = None
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        got = G.heat_filter(onehot, tau=60, order=50)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    L_host = G.laplacian("combinatorial")
    t = time.perf_counter()
    want = ref.cheby_op(L_host, ref.cheby_coeff(ref.heat(60, lmax), 50, lmax)[None], onehot, lmax)[0]
    host_s = time.perf_counter() - t
    rows.append(dict(kind="heat_filter", n=args.n, f=args.labels, tau=60, order=50, lmax=lmax, device_s=round(best, 4),
                     host_scipy_s=round(host_s, 3), speedup=round(host_s / best, 1),
                     l1_diff_vs_host=float(np.abs(got - want).sum()), bit_identical=bool(np.array_equal(got, want))))

    with open(args.out, "a") as fh:
        for r in rows:
            r.update(graph=graph, gpu=gpu)
            print(json.dumps(r), flush=True)
            fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
