#!/usr/bin/env python
"""Headline benchmark: graph build points/sec (kernel + diff_op), N=1M, d=100, knn=5, decay=40.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --steps K --warmup W    (CPU arm: the reference's path on host cores)
    python bench.py ... --dump-outputs DIR                   (also writes the last timed step's K / P / degree,
                                                              a fixed sample of rows, as DIR/<name>.npy)

One "step" = one full pass of the hot path over the synthetic Gaussian-mixture input: search operand
-> fused distance/top-k -> float64 refine -> CSR -> symmetrise -> diffusion operator.  `value` is
measured with the input already resident in HBM (CUDA events, max over ranks); `e2e` goes through the
public graphtools-style API with HOST buffers (pinned H2D of X, D2H of K and P as scipy CSR).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if "reference" in sys.argv:
    # the CPU arm uses every host thread (torchrun exports OMP_NUM_THREADS=1 to its workers)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KNN, DECAY, THRESH = 5, 40, 1e-4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--d", type=int, default=100)
    ap.add_argument("--clusters", type=int, default=50)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write K, P and the degree vector of the last timed step to DIR/<name>.npy (GPU arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl %s" % a.impl)
    return a


def workload_name(a):
    return "synthetic Gaussian mixture {}x{} ({} clusters, intrinsic dim 10, seed {}), kNNGraph knn=5 decay=40 " \
           "thresh=1e-4, kernel + diff_op".format(a.n, a.d, a.clusters, a.seed)


METRIC = "graph build points/sec (kernel+diff_op)"


def bench_config(a):
    """Identical in both arms (the driver compares them)."""
    return {"workload": workload_name(a), "n": a.n, "d": a.d, "knn": KNN, "decay": DECAY, "thresh": THRESH,
            "l2": "inputs (400 MB operand, 113 MB raw CSR) larger than the 126 MB L2; no explicit flush"}


def make_data(a):
    from graphtools_b200 import synth
    X, _ = synth.gaussian_mixture(a.n, a.d, n_clusters=a.clusters, intrinsic_dim=10, seed=a.seed)
    return X


# ------------------------------------------------------------------------------ CPU arm
REF_SIZES = (25_000, 50_000, 100_000, 200_000)      # BASELINE.md section 3: fit t = a N^2 + b N, quote N = 1M


def load_reference():
    """The UNMODIFIED reference installed under baseline/_ref (baseline/install_ref.sh), float64 path
    (NUMBA_AVAILABLE = False, SURVEY 8c/8d), with the three stand-ins for its uninstalled dependencies
    (tasklogger, future, pygsp) from oracle/shims.  None when the install is missing."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "graphtools")):
        return None
    for p in (os.path.join(ROOT, "oracle", "shims"), ref):
        if p not in sys.path:
            sys.path.insert(0, p)
    import graphtools
    import graphtools.graphs
    graphtools.graphs.NUMBA_AVAILABLE = False
    return graphtools


def _all_threads():
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass


def reference_build_seconds(graphtools, X, n_sub):
    """One run of the reference's own public API on an n_sub-point subsample of the workload (every
    (n / n_sub)-th point, so the mixture proportions are kept): Graph(...) builds the kernel, .diff_op the
    diffusion operator (graphs.py:819-982, base.py:534-646)."""
    rows = np.linspace(0, X.shape[0] - 1, n_sub).astype(np.int64)
    Xs = X[rows].astype(np.float64)
    t0 = time.perf_counter()
    G = graphtools.Graph(Xs, knn=KNN, decay=DECAY, thresh=THRESH, n_jobs=-1, verbose=0)
    K = G.kernel
    P = G.diff_op
    dt = time.perf_counter() - t0
    return dt, int(K.nnz), int(P.nnz)


def fit_quadratic(sizes, times):
    """Least-squares t = a N^2 + b N (relative residuals), as BASELINE.md section 3 prescribes."""
    N = np.asarray(sizes, dtype=np.float64)
    t = np.asarray(times, dtype=np.float64)
    if len(set(sizes)) < 2:
        return float(t.mean() / N.mean() ** 2), 0.0
    A = np.stack([N * N, N], axis=1) / t[:, None]
    (a, b), *_ = np.linalg.lstsq(A, np.ones_like(t), rcond=None)
    if a <= 0 or b < 0:                      # degenerate fit (noise): pure quadratic through the largest size
        i = int(np.argmax(N))
        return float(t[i] / N[i] ** 2), 0.0
    return float(a), float(b)


def cpu_sample_rate(X, seconds, fixed_rows=None):
    """Cross-check leg: the oracle port (restatement of graphs.py:819-982, float64, all host threads) on `m` query
    rows of the workload searched against the FULL reference set; per-row cost = per-point cost of the full job."""
    from oracle import graph_oracle as go
    _all_threads()
    X64 = X.astype(np.float64)
    g = go.KnnOracle(X64, knn=KNN, decay=DECAY, thresh=THRESH, n_jobs=-1)
    g.tree  # fit (brute force: keeps a pointer)
    n = X.shape[0]

    def run(m):
        rows = np.linspace(0, n - 1, m).astype(np.int64)
        t0 = time.perf_counter()
        R = g.kernel_to_data(X64[rows], knn=KNN + 1)
        return time.perf_counter() - t0, rows, R

    if fixed_rows is None:
        m0 = min(n, 512)
        t0, _, _ = run(m0)
        m = int(min(n, max(m0, m0 * seconds / max(t0, 1e-3))))
    else:
        m = fixed_rows
    t, rows, R = run(m)
    return m / t, m, t, rows, R


def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count()


def reference_schedule(steps):
    """Subsample size of each timed step: the four sizes of BASELINE.md section 3, the large ones less often so that
    a 20-step run still ends within a few minutes (200k twice, 100k four times, ...)."""
    out = []
    for i in range(steps):
        if i % 10 == 5:
            out.append(REF_SIZES[3])
        elif i % 5 == 2:
            out.append(REF_SIZES[2])
        elif i % 2 == 1:
            out.append(REF_SIZES[1])
        else:
            out.append(REF_SIZES[0])
    return out


def reference_fit(graphtools, X, sizes, n_target):
    times, nnz = [], []
    for m in sizes:
        dt, nk, _ = reference_build_seconds(graphtools, X, min(m, X.shape[0]))
        times.append(dt); nnz.append(nk)
    a, b = fit_quadratic([min(m, X.shape[0]) for m in sizes], times)
    t_target = a * n_target ** 2 + b * n_target
    return {"a_s_per_point2": a, "b_s_per_point": b, "sizes": [int(min(m, X.shape[0])) for m in sizes],
            "seconds": times, "nnz_K": nnz, "extrapolated_seconds_at_n": t_target, "n": int(n_target)}


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _all_threads()
    X = make_data(a)
    graphtools = load_reference()
    cfg = bench_config(a)
    if graphtools is None:
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is missing (run baseline/install_ref.sh "
                          "in the build container)"}))
        return
    for _ in range(a.warmup):
        reference_build_seconds(graphtools, X, min(a.n, 12_500))
    sched = reference_schedule(a.steps)
    sched = [min(m, a.n) for m in sched]
    times = []
    for m in sched:
        dt, _, _ = reference_build_seconds(graphtools, X, m)
        times.append(dt)
    total_t = sum(times)
    fa, fb = fit_quadratic(sched, times)
    t_full = fa * a.n ** 2 + fb * a.n
    value = a.n / t_full
    per_size = {}
    for m, t in zip(sched, times):
        per_size.setdefault(int(m), []).append(t)
    # port-vs-reference cross-check: the oracle port's per-point rate on rows searched against the full set
    port_rate, port_m, port_t, _, _ = cpu_sample_rate(X, min(a.cpu_seconds, 8.0))
    sample = "unmodified graphtools.Graph(X_sub, knn=5, decay=40, thresh=1e-4, n_jobs=-1).kernel/.diff_op from " \
             "baseline/_ref on subsamples of the workload, one size per step from {}; value = n / (a n^2 + b n) at " \
             "n = {} (extrapolated)".format(sorted(per_size), a.n)
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "points/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * total_t / max(a.steps, 1), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "extrapolated": True,
        "fit": {"model": "t = a N^2 + b N", "a_s_per_point2": fa, "b_s_per_point": fb,
                "seconds_by_size": {str(k): v for k, v in sorted(per_size.items())},
                "points_per_s_by_size": {str(k): k / float(np.mean(v)) for k, v in sorted(per_size.items())},
                "extrapolated_seconds_at_n": t_full},
        "port_check": {"port_points_per_s_full_set_rows": port_rate, "rows": port_m, "seconds": port_t,
                       "reference_over_port": value / port_rate,
                       "note": "oracle port (graphs.py:819-982 restated) on sampled rows against the full 1M set"},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": cpu_threads(), "kind": "reference",
                         "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host": {"cpu_count": os.cpu_count(), "numba": False},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active")
                                                           for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


DUMP_ROWS = 65536          # rows of K / P written by --dump-outputs (halved until the files fit DUMP_BYTES)
DUMP_BYTES = 64 << 20


def dump_outputs(G, out_dir, write):
    """Writes what one build hands its caller -- kernel K (CSR), diffusion operator P (K's structure) and the degree
    vector -- for a fixed seeded sample of rows, as float64 .npy files, so that two builds of the project can be
    compared output for output.  rows.npy holds the sorted row ids; K_indptr / K_indices / K_data / P_data are the
    CSR of those rows, degree.npy their row sums.  Collective when the build is row-sharded over ranks (the first
    access of the full device matrices all-gathers them); only the rank with `write` set writes files."""
    import torch
    K, P, deg = G._dev_kernel, G._dev_P, G._dev_degree
    if not write:
        return None
    n = K.shape[0]
    indptr = K.indptr.cpu().numpy().astype(np.int64)
    perm = np.random.default_rng(0).permutation(n)
    m = min(n, DUMP_ROWS)
    while True:
        rows = np.sort(perm[:m])
        lens = indptr[rows + 1] - indptr[rows]
        nnz = int(lens.sum())
        nbytes = 8 * (3 * nnz + 3 * m + 1) + 128 * 6           # values + one .npy header per file
        if nbytes <= DUMP_BYTES or m == 1:
            break
        m //= 2
    sub_ptr = np.concatenate([[0], np.cumsum(lens)])
    sel = np.arange(nnz, dtype=np.int64) + np.repeat(indptr[rows] - sub_ptr[:-1], lens)
    sel_d = torch.from_numpy(sel).to(K.data.device)
    rows_d = torch.from_numpy(rows).to(K.data.device)
    arrays = {"rows": rows, "K_indptr": sub_ptr, "K_indices": K.indices.index_select(0, sel_d).cpu().numpy(),
              "K_data": K.data.index_select(0, sel_d).cpu().numpy(), "P_data": P.index_select(0, sel_d).cpu().numpy(),
              "degree": deg.reshape(-1).index_select(0, rows_d).cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float64))
    return {"dir": out_dir, "rows": int(m), "of": int(n), "nnz": nnz, "bytes": nbytes}


def run_gpu_arm(a):
    import torch
    import torch.distributed as dist
    import graphtools_b200 as gt
    from graphtools_b200 import _engine as E, distributed as gd, pipeline

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keeps NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    X = make_data(a)
    n, d = X.shape
    Xd = torch.from_numpy(X).cuda()          # `value`: inputs already resident in HBM when the timed region starts
    lo, hi = gd.shard_bounds(n, world, rank)
    bounds = [gd.shard_bounds(n, world, r) for r in range(world)]
    impl = pipeline.default_impl()
    if impl == "auto":
        impl = pipeline.AUTO_TC if d + 1 <= 104 else "simt"
    SEARCH = {"tc": "gtb_knn_topk_tc", "tc16": "gtb_knn_topk_tc", "tch": "gtb_knn_topk_tc",
              "tch1": "gtb_knn_topk_tc_seeded"}.get(impl, "gtb_knn_topk_simt")

    def step():
        """device-resident hot path through the public API: X is already in HBM, nothing is copied back.
        With more than one rank the build shards the query rows, routes edges to their column owner with one NCCL
        all-to-all of packed records and merges / normalises per shard; K and P stay row-sharded in HBM
        (graphtools_b200/knn.py)."""
        G = gt.Graph(Xd, knn=KNN, decay=DECAY, thresh=THRESH, verbose=0)
        sh = G.__dict__.get("_dev_shard")
        if sh is not None:
            return sh["data"], sh["P"], G
        return G._dev_kernel.data, G._dev_P, G

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up steps: every entry point bracketed with CUDA events -> the per-stage breakdown (stage_ms_per_step)
    E.timing = {}
    for _ in range(a.warmup):
        step()
    barrier()
    tm_warm = E.timings_ms()
    E.timing = None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # timed steps: only the dominant kernel is bracketed (two event records per step instead of two per launch: about
    # a hundred launches per build, which a 30 ms step at 8 GPUs feels)
    E.timing = {}
    E.timing_only = {SEARCH}
    launches0 = E.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(a.steps):
        Kv, Pv, G_last = step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    tm_search = E.timings_ms()
    E.timing = None
    E.timing_only = None
    # per-stage times: the warm-up steps' events scaled to a.steps (every consumer below divides by a.steps); the
    # dominant kernel's entry is replaced by the one measured inside the timed region
    tm = {k: (v[0], v[1] * a.steps / max(a.warmup, 1)) for k, v in tm_warm.items()}
    tm[SEARCH] = tm_search[SEARCH]
    launches = E.kernel_launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / a.steps
    value = n / (ms_per_step / 1e3)
    stats = pipeline.stats()
    sums = torch.stack([Kv.sum(), Pv.sum(), torch.tensor(float(Kv.shape[0]), dtype=torch.float64, device="cuda")])
    if world > 1:
        dist.all_reduce(sums)                    # checksums / nnz of the row-sharded result, over all ranks
    checksum_K, checksum_P, nnz_sym = float(sums[0].item()), float(sums[1].item()), int(sums[2].item())
    dumped = dump_outputs(G_last, a.dump_outputs, rank == 0) if a.dump_outputs else None

    # dominant kernel: fused distance/top-k; algorithmic FLOPs = 2 * Nq * Nr * d (SURVEY 8d)
    calls, search_ms = tm[SEARCH]
    per_launch_ms = search_ms / calls
    flop = 2.0 * (hi - lo) * n * d
    achieved = flop / (per_launch_ms / 1e3) / 1e12
    peaks, how = measured_peaks()
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    if impl == "tch1":
        kp = (d + 2 + 15) // 16 * 16
        kname = "search_tc_kernel<TOPK, CL=2, FP16x1, LS=32, QT=2> (%s): tcgen05.mma kind::f16 on float16 operands, ONE " \
                "product A_hi.B_hi, thresholds seeded from a sweep over every 16th reference tile, one candidate list " \
                "of 64 per row, A in TMEM, TMA multicast, persistent, quickselect epilogue" % SEARCH
        issued, ceiling = achieved * 1.0 * kp / d, d / (1.0 * kp)
        note = "the tensor pipe issues that once (float16 operands, 11 bits each; certified bound 2^-10 (|x|^2 + " \
               "|y|^2)) on K padded to %d, so frac <= %.3f by construction; the seed sweep (1/16 of the tiles) is a " \
               "separate launch, timed in stage_ms_per_step" % (kp, ceiling)
    elif impl == "tch":
        kp = (d + 2 + 15) // 16 * 16
        kname = "search_tc_kernel<TOPK, CL=2, FP16x2, LS=16> (%s): tcgen05.mma kind::f16 on float16 hi/lo pairs, two " \
                "products A_hi.B_hi + A_hi.B_lo, A in TMEM, TMA multicast, persistent, quickselect epilogue" % SEARCH
        issued, ceiling = achieved * 2.0 * kp / d, d / (2.0 * kp)
        note = "the tensor pipe issues 2x that (fp16x2 split: the reference operand keeps 22 bits, the query operand " \
               "11; certified bound 2^-11 (|x|^2 + |y|^2)) on K padded to %d, so frac <= %.3f by construction" % (kp, ceiling)
    elif impl == "tc16":
        kp = (d + 1 + 15) // 16 * 16
        kname = "search_tc_kernel<TOPK, CL=2, BF16, LS=16> (%s): tcgen05.mma kind::f16 on bf16 hi/lo pairs " \
                "(bf16x3), A in TMEM, TMA multicast, persistent, quickselect epilogue" % SEARCH
        issued, ceiling = achieved * 3.0 * kp / d, d / (3.0 * kp)
        note = "the tensor pipe issues 3x that (bf16x3 split) on K padded to %d at the bf16 rate, so frac <= %.3f " \
               "by construction" % (kp, ceiling)
    elif impl == "tc":
        kp = (d + 1 + 7) // 8 * 8
        kname = "search_tc_kernel<TOPK, CL=2, TF32> (%s): tcgen05.mma kind::tf32, 3xTF32 split, A in TMEM, TMA " \
                "multicast, persistent" % SEARCH
        issued, ceiling = achieved * 3.0 * kp / d, d / (6.0 * kp)
        note = "the tensor pipe issues 3x that (3xTF32) on K padded to %d at the TF32 rate = half the bf16 peak, " \
               "so frac <= %.3f by construction" % (kp, ceiling)
    else:
        kname, issued, ceiling = "search_simt_kernel<48,false> (%s): fp32 CUDA cores" % SEARCH, achieved, None
        note = "fp32 CUDA-core kernel; tensor peak kept as the denominator"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(impl if world == 1 else "", {}).get("dram_bytes_per_launch")
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": kname, "issued_tflops": issued, "frac_ceiling": ceiling,
                "issued_frac_of_peak": issued / (peak if impl != "tc" else peak / 2.0),
                "launch_ms": per_launch_ms, "share_of_step": per_launch_ms / ms_per_step,
                "peak_source": "%s bf16_tflops_sustained (kernel timed inside a long step). achieved = algorithmic "
                               "2*Nq*Nr*d FLOP/s; %s. traffic = dram read+write bytes of one launch from the ncu "
                               "--set full capture in profiles/ (1-GPU workload)" % (how, note),
                "flops_per_launch": flop}

    # ---- sparse stages against the HBM roofline (SURVEY 8d byte model: float64 values, int32 indices / row pointers),
    # from the same CUDA-event timings; this rank's share of the rows
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    m_rows = hi - lo
    nnz_r = float(stats.get("nnz_raw") or 0)
    nnz_s_loc = float(Kv.shape[0])
    S_cand = float(stats.get("S") or 32)

    def _ms(*names):
        return sum(tm[k][1] for k in names if k in tm) / a.steps

    k4_names = ("gtb_transpose_count", "gtb_transpose_scatter", "gtb_sym_merge_count", "gtb_sym_merge_fill",
                "gtb_rec_sort_rows", "gtb_records_count", "gtb_records_scatter", "gtb_route_count", "gtb_route_fill",
                "gtb_cast_indptr")
    sparse_stages = {}
    for name, ms_, nbytes, what in (
            ("K3 refine (float64 re-evaluation, bandwidth, certification, affinities)", _ms("gtb_refine_topk"),
             m_rows * S_cand * (4.0 + 4.0 * d) + 12.0 * nnz_r + 4.0 * (m_rows + 1),
             "Nq S (4 + 4 d) candidate gather + 12 nnz_r + 4 (Nq + 1) written"),
            ("CSR emission (csr_gather + scans)", _ms("gtb_csr_gather", "gtb_exclusive_scan"),
             12.0 * nnz_r + 4.0 * (m_rows + 1) + 12.0 * nnz_r, "staging read + 12 nnz_r + 4 (Nq + 1) written"),
            ("K4 symmetrise + normalise (transpose, merge, P, degree)", _ms(*k4_names),
             12.0 * nnz_r + 4.0 * (m_rows + 1) + 12.0 * nnz_s_loc + 4.0 * (m_rows + 1) + 16.0 * nnz_s_loc,
             "[12 nnz_r + 4 (N + 1)] read + [12 nnz_s + 4 (N + 1)] written + 8 nnz_s read + 8 nnz_s written (P)")):
        if ms_ > 0:
            gbs = nbytes / (ms_ / 1e3) / 1e9
            sparse_stages[name] = {"ms": ms_, "algorithmic_bytes": nbytes, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm,
                                   "byte_model": what}
    roofline["sparse_stages"] = sparse_stages
    roofline["hbm_peak_gbs"] = hbm

    # ---- end-to-end through the public API with host buffers (rank-sharded builds are not exposed
    # through Graph(); e2e is measured on rank 0's single-GPU API call when world == 1)
    e2e = None
    if not a.no_e2e:
        Xh = torch.from_numpy(X).pin_memory()
        def api_call():
            G = gt.Graph(Xh, knn=KNN, decay=DECAY, thresh=THRESH, verbose=0)
            return G.kernel, G.diff_op
        for _ in range(2):              # warm-up with the loop's own object lifetimes (result memory is pooled)
            Kh, Ph = api_call()
        barrier()
        t0 = time.perf_counter()
        reps = max(1, min(a.steps, 5))
        for _ in range(reps):
            Kh, Ph = api_call()
        barrier()
        dt = (time.perf_counter() - t0) / reps
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        # bytes over PCIe per step, all ranks together: each rank uploads its own row block of X and copies its own
        # rows of K / P / indices / indptr / degree into the shared host result
        d2h = Kh.data.nbytes + Kh.indices.nbytes + Kh.indptr.nbytes + Ph.data.nbytes + 8 * n
        if world == 1:
            d2h = Kh.data.nbytes + Kh.indices.nbytes + Kh.indptr.nbytes + Ph.data.nbytes
        e2e = {"value": n / dt, "unit": "points/s", "h2d_bytes_per_step": int(X.nbytes),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": dt * 1e3,
               "api": "graphtools_b200.Graph(X_host_pinned, knn=5, decay=40).kernel / .diff_op (scipy CSR, K and P "
                      "sharing one structure) called on every rank; with N > 1 each rank uploads its row block of X "
                      "(NCCL all-gather assembles the reference set) and DMAs its rows of the result into one "
                      "page-locked shared-memory segment that all ranks view; result memory is recycled between "
                      "builds (graphtools_b200/hostpool.py)"}
        parity_e2e = {"nnz": int(Kh.nnz), "checksum_K": float(Kh.data.sum()), "checksum_P": float(Ph.data.sum()),
                      "symmetric": bool(abs(Kh[:2000, :2000] - Kh[:2000, :2000].T).max() == 0.0)}
    else:
        parity_e2e = None

    # ---- parity of the headline build, inside the bench: raw kernel rows of sampled queries against the oracle's rows
    # for the same queries searched in the FULL reference set (graphs.py:819-982).  The oracle rows double as the port
    # leg of the CPU baseline (their wall time is the port's per-point cost).
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        from tests.parity import compare_sparse
        port_rate, m, t_port, rows, R_ref = cpu_sample_rate(X, min(a.cpu_seconds, 10.0))
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Gp = gt.Graph(Xd, knn=KNN, decay=DECAY, thresh=THRESH, verbose=0, initialize=False)
            R_gpu = Gp.build_kernel().to_scipy()[rows]
        try:
            r = compare_sparse(R_gpu, R_ref, thresh=THRESH, what="headline raw kernel rows")
            parity = {"rows": int(m), "of": n, "against": "oracle rows vs the full %d-point reference set" % n,
                      "structure_equal": bool(r["n_exempt"] == 0), "n_exempt": int(r["n_exempt"]),
                      "max_rel": r["max_rel"], "nnz_checked": int(R_ref.nnz), "ok": True}
        except AssertionError as ex:
            parity = {"rows": int(m), "ok": False, "error": str(ex)[:300]}
        del Gp, R_gpu
        graphtools = load_reference()
        if graphtools is not None:
            fit = reference_fit(graphtools, X, REF_SIZES[:3], n)
            rate = n / fit["extrapolated_seconds_at_n"]
            cpu = {"value": rate, "unit": "points/s", "cores": cpu_threads(), "kind": "reference",
                   "extrapolated": True, "fit": fit,
                   "sample": "unmodified graphtools.Graph(...).kernel/.diff_op (baseline/_ref) on {} -point subsamples "
                             "of the workload, {:.1f} s in total; value = n / (a n^2 + b n) at n = {}".format(
                                 "/".join(str(x) for x in fit["sizes"]), sum(fit["seconds"]), n),
                   "port_points_per_s": port_rate,
                   "port_sample": "{} of {} query rows vs the full reference set in {:.1f} s (oracle port of "
                                  "graphs.py:819-982)".format(m, n, t_port)}
        else:
            cpu = {"value": port_rate, "unit": "points/s", "cores": cpu_threads(), "kind": "port",
                   "sample": "{} of {} query rows vs the full reference set in {:.1f} s (oracle port of "
                             "graphs.py:819-982: sklearn brute kneighbors + affinity CSR, float64)".format(m, n, t_port)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "points/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "%s tensor-core select (f32 accumulate) / f64 values" % {"tch": "fp16x2", "tc16": "bf16x3",
                                                                                "tc": "3xTF32"}.get(impl, "f32"),
            "data": "synthetic",
            "config": bench_config(a),
            "run": {"sharding": "query rows over %d rank(s); reference set assembled by NCCL all-gather of the ranks' "
                                "row blocks; K / P row-sharded in HBM" % world if world > 1 else
                                "single GPU", "search_impl": impl,
                    "nnz_raw_rank0": stats.get("nnz_raw"), "nnz_sym": nnz_sym, "radius_rows_rank0": stats.get("radius_rows"),
                    "checksum_K": checksum_K, "checksum_P": checksum_P, "e2e_result": parity_e2e},
            "parity": parity,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "stage_ms_per_step": {k: v[1] / a.steps for k, v in sorted(tm.items(), key=lambda kv: -kv[1][1])},
            "stage_ms_source": "CUDA events around every entry point during the warm-up steps; the dominant kernel "
                               "(%s) from the events inside the timed region" % SEARCH,
        }
        if dumped is not None:
            line["dump_outputs"] = dumped
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    # stdout carries exactly ONE line (the JSON): anything libraries print meanwhile (e.g. the NCCL version
    # banner) is diverted to stderr at the file-descriptor level
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(saved, "w")
    py_stdout, sys.stdout = sys.stdout, real_stdout
    try:
        if a.impl == "reference":
            run_reference_arm(a)
        else:
            run_gpu_arm(a)
    finally:
        real_stdout.flush()
        sys.stdout = py_stdout


if __name__ == "__main__":
    main()
