"""Wide-knn measurement: kNN graphs whose knn is beyond the candidate lists (pipeline.wide_knn), built through the
histogram count sweeps, one JSON line per build, on the bench's Gaussian mixture (N x 100, 50 clusters, intrinsic
dimension 10, seed 3), decay 40.

* end to end: host clock around gt.Graph(X, knn=..., decay=40) with a device synchronise, after one warm-up build;
* per-stage device times of a second build (CUDA events around every entry point, engine timing): coarse count, fine
  count, bound selection, collect sweep, ball refine, CSR, symmetrise;
* each sweep's algorithmic work 2 Nq Nr d over its time, against the sustained bf16 peak DESIGN.md section 4 uses
  (1401.5 TFLOP/s), and the coarse sweep's share of the count time;
* ball length per row (mean / max) next to knn_eff = knn + 1;
* oracle rows: --oracle-rows query rows sampled from the build, their raw kernel rows against the reference's
  kernel_to_data at knn + 1 over the whole reference set (float64, on the host).
The card's name, power limit and clock are read in the same call.
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

import graphtools_b200 as gt  # noqa: E402
from graphtools_b200 import _engine as E, pipeline, synth  # noqa: E402
from run_shortest_path import gpu_info  # noqa: E402

BF16_PEAK = 1401.5e12
STAGES = {"coarse count": ("gtb_knn_count_tc#coarse", "gtb_knn_count_simt#coarse"),
          "fine count": ("gtb_knn_count_tc#fine", "gtb_knn_count_simt#fine"),
          "bound": ("gtb_knn_count_bound",),
          "collect sweep": ("gtb_knn_radius_tc", "gtb_knn_radius_simt", "gtb_knn_radius_simt_l1"),
          "ball refine": ("gtb_scatter_pairs", "gtb_refine_ball"),
          "csr": ("gtb_csr_gather", "gtb_exclusive_scan"),
          "symmetrise": ("gtb_transpose_count", "gtb_transpose_scatter", "gtb_sym_merge_count", "gtb_sym_merge_fill",
                         "gtb_rec_sort_rows")}


def build(X, knn):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gt.Graph(X, knn=knn, decay=40, thresh=1e-4, verbose=0)


def oracle_rows(X, G, knn, rows):
    from oracle import graph_oracle as go
    from tests.parity import compare_sparse
    ref = pipeline.SearchOperand(pipeline.to_device_f32(X))
    qry = pipeline.SearchOperand(pipeline.to_device_f32(X[rows]), mean=ref.mean)
    R, _ = pipeline.knn_kernel(ref, qry, knn=knn + 1, decay=40, thresh=1e-4)
    og = go.KnnOracle(X.astype(np.float64), knn=knn, decay=40, thresh=1e-4)
    R_ref = og.kernel_to_data(X[rows].astype(np.float64), knn=knn + 1)
    r = compare_sparse(R.to_scipy(), R_ref, thresh=1e-4, what="oracle rows")
    return {"rows": len(rows), "n_exempt": r["n_exempt"], "max_rel": r["max_rel"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="200000,1000000")
    ap.add_argument("--knn", default="150,500")
    ap.add_argument("--oracle-rows", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "wide_knn.jsonl"),
                    help="JSON lines are appended here (default: the system temporary directory)")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    card = gpu_info()
    for n in (int(s) for s in a.sizes.split(",")):
        X, _ = synth.gaussian_mixture(n, 100, n_clusters=50, intrinsic_dim=10, seed=3)
        for knn in (int(k) for k in a.knn.split(",")):
            row = {"n": n, "d": 100, "knn": knn, "knn_eff": knn + 1, "decay": 40, "gpu": card}
            try:
                build(X, knn)                                         # warm-up
                torch.cuda.synchronize()
                t = time.perf_counter()
                G = build(X, knn)
                torch.cuda.synchronize()
                row["build_s"] = time.perf_counter() - t
                st = pipeline.stats()
                row.update({k: st.get(k) for k in ("impl", "count_sweeps", "ball_max", "ball_mean", "radius_pairs",
                                                    "nnz_raw", "nnz_sym")})
                E.timing = {}
                del G
                G = build(X, knn)
                tm = E.timings_ms()
                E.timing = None
                stages = {s: round(sum(tm.get(k, (0, 0.0))[1] for k in keys), 3) for s, keys in STAGES.items()}
                row["stage_ms"] = stages
                flop = 2.0 * n * n * 100
                for s in ("coarse count", "fine count", "collect sweep"):
                    if stages[s] > 0:
                        rate = flop / (stages[s] * 1e-3)
                        row[s.replace(" ", "_") + "_tflops"] = round(rate / 1e12, 1)
                        row[s.replace(" ", "_") + "_of_bf16_peak"] = round(rate / BF16_PEAK, 3)
                cnt = stages["coarse count"] + stages["fine count"]
                row["coarse_share_of_count"] = round(stages["coarse count"] / cnt, 3) if cnt else None
                if a.oracle_rows:
                    rows = np.sort(np.random.default_rng(0).choice(n, a.oracle_rows, replace=False))
                    row["oracle"] = oracle_rows(X, G, knn, rows)
                del G
            except pipeline.RowTooLong as e:
                row["row_too_long"] = str(e)
            print(json.dumps(row), flush=True)
            with open(a.out, "a") as f:
                f.write(json.dumps(row) + "\n")
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
