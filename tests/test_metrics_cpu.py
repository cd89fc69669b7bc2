"""Host-side pieces of the cosine / cityblock paths, checked without a GPU: the cosine search copy of data with
all-zero rows, a Python model of the "data" edge lengths of csrc/paths.cu, and the replay of the reference's
search schedule (knn.search_schedule) against the CPU oracle."""
import numpy as np
import pytest
import torch
from sklearn.metrics import pairwise_distances

from graphtools_b200 import pipeline, synth
from graphtools_b200.knn import search_schedule
from oracle import graph_oracle as go


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_cosine_operand_of_zero_rows_is_finite(dtype):
    """sklearn's ``normalize`` leaves an all-zero row at zero; dividing by its norm would give NaN, and the column
    mean would carry that NaN into every row of the search copy."""
    X = np.random.default_rng(0).random((10, 4))
    X[3] = 0
    X[7] = 0
    Xt = torch.from_numpy(X).to(dtype)
    op = pipeline.SearchOperand(Xt, metric="cosine")
    assert torch.isfinite(op.Xs).all() and torch.isfinite(op.mean).all()
    X = Xt.to(torch.float64).numpy()
    Xn = X / np.linalg.norm(X, axis=1, keepdims=True).clip(min=1e-300)
    Xn[[3, 7]] = 0
    assert np.allclose(op.mean.numpy(), Xn.mean(axis=0), rtol=1e-12, atol=0)
    # before centring: zero rows stay zero, the others have unit norm
    rows = op.Xs.to(torch.float64) + op.mean
    assert torch.equal(op.Xs[3], (-op.mean).to(torch.float32))
    assert torch.allclose(rows[[3, 7]], torch.zeros(2, 4, dtype=torch.float64), atol=1e-7)
    norms = rows.norm(dim=1)
    keep = [i for i in range(10) if i not in (3, 7)]
    assert torch.allclose(norms[keep], torch.ones(8, dtype=torch.float64), atol=1e-6)


# --------------------------------------------------------------------------- "data" edge lengths (csrc/paths.cu)
def _sqdist_block(t):
    """sqdist_block: eight interleaved accumulators over blocks of 8, pairwise combination, scalar tail; rows of
    fewer than 8 elements are summed left to right from -0."""
    n = t.shape[0]
    if n < 8:
        r = t.dtype.type(-0.0)
        for v in t:
            r = r + v
        return r
    r = t[:8].copy()
    i = 8
    while i < n - n % 8:
        r = r + t[i:i + 8]
        i += 8
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for v in t[i:]:
        res = res + v
    return res


def _sqdist_pairwise(t):
    """sqdist_pairwise: blocks of <= 128 elements, longer runs split at n / 2 rounded down to a multiple of 8."""
    n = t.shape[0]
    if n <= 128:
        return _sqdist_block(t)
    h = n // 2
    h -= h % 8
    return _sqdist_pairwise(t[:h]) + _sqdist_pairwise(t[h:])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sqdist_model_matches_numpy_pairwise_sum(dtype):
    """The summation order csrc/paths.cu implements is numpy's: a mismatch in the GPU test of the same widths
    then points at the CUDA code, not at the order."""
    rng = np.random.default_rng(11)
    for d in (1, 3, 7, 8, 9, 30, 64, 127, 128, 129, 136, 257, 500, 1000, 1031):
        a = rng.normal(size=(40, d)).astype(dtype)
        b = rng.normal(size=(40, d)).astype(dtype)
        sq = (a - b) ** 2
        want = np.sum(sq, axis=1)
        got = np.array([_sqdist_pairwise(sq[i]) for i in range(40)], dtype=dtype)
        assert got.dtype == want.dtype
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (dtype, d)


# --------------------------------------------------------------------------- search schedule replay
def _counts(X, Y, knn, decay, thresh, metric, bandwidth=None):
    """#{j : d_ij < r_i} with r_i the reference's kernel radius (graphs.py:886-905)."""
    D = pairwise_distances(Y, X, metric=metric)
    if bandwidth is None:
        bw = np.maximum(np.sort(D, axis=1)[:, knn - 1], np.finfo(float).eps)
    else:
        bw = np.maximum(bandwidth, np.finfo(float).eps)
    r = bw * np.power(-np.log(thresh), 1 / decay)
    return (D < np.reshape(r, (-1, 1))).sum(axis=1)


def _check_replay(g, X, Y, knn, knn_max, decay, thresh, metric, bandwidth=None):
    c = _counts(X, Y, knn, decay, thresh, metric, bandwidth)
    if knn_max is not None:
        c = np.minimum(c, knn_max)                      # the device's raw rows are capped at knn_max
    s_todo, s_final, n_todo = search_schedule(lambda s: int((c >= s).sum()), Y.shape[0], X.shape[0], knn, knn_max,
                                              g.search_multiplier)
    sc = g.schedules[-1]
    assert np.array_equal(np.flatnonzero(c >= s_todo), sc["todo"])
    assert n_todo == sc["todo"].size
    assert s_final == sc["search_knn"]
    assert (s_final > X.shape[0] / 2) == sc["fallback"]
    return sc


def test_schedule_replay_matches_oracle():
    """Random configurations around the N / 2 switch: the replay from per-row counts gives the oracle's final todo
    rows and search width in-sample and out of sample.  Every branch (no rows left, radius, knn_max) and both sides
    of the switch occur."""
    rng = np.random.default_rng(5)
    seen = set()
    for trial in range(36):
        metric = ("cosine", "cityblock", "euclidean")[trial % 3]
        n = int(rng.choice([60, 150, 300, 500, 700]))
        d = int(rng.choice([3, 10, 40]))
        knn = int(rng.choice([3, 5, 10]))
        decay = float(rng.choice([2, 5, 10, 40]))
        thresh = float(rng.choice([1e-4, 1e-3, 1e-2]))
        knn_max = None if rng.random() < 0.7 else min(int(knn * rng.choice([2, 8, 30])), n - 2)
        mult = int(rng.choice([3, 6]))
        X, _ = synth.gaussian_mixture(n, d, n_clusters=2, intrinsic_dim=None, seed=trial)
        X = X.astype(np.float64)
        g = go.KnnOracle(X, knn=knn, decay=decay, knn_max=knn_max, thresh=thresh, distance=metric,
                         search_multiplier=mult, n_jobs=1)
        g.kernel()
        kmax = g.knn_max + 1 if g.knn_max else None
        sc = _check_replay(g, X, X, g.knn + 1, kmax, decay, g.thresh, metric)
        seen.add((sc["branch"], sc["fallback"]))
        Y = X[:40] + rng.normal(scale=0.05, size=(40, d))
        g.kernel_to_data(Y)
        sc = _check_replay(g, X, Y, g.knn, None, decay, g.thresh, metric)
        seen.add((sc["branch"], sc["fallback"]))
    assert {(None, False), ("radius", False), ("radius", True), ("kneighbors", True)} <= seen, seen


@pytest.mark.parametrize("metric,n,d,seed,decay,passes", [
    ("cityblock", 400, 10, 3, 10, [(36, 400), ("radius", 17)]),
    ("cosine", 400, 50, 5, 10, [(36, 400), ("radius", 142)]),
    ("cosine", 200, 10, 5, 5, [(36, 200), (200, 3)]),
    ("cosine", 400, 50, 5, 5, [(36, 400), ("radius", 400)]),
    ("cosine", 1000, 50, 0, 5, [(36, 1000), (216, 1000), (1000, 188)]),
])
def test_fallback_cases_take_the_metricless_branch(metric, n, d, seed, decay, passes):
    """The configurations of the GPU fallback tests (tests/test_metrics_gpu.py) do reach the reference's
    metric-less search, and the replay predicts it."""
    X, _ = synth.gaussian_mixture(n, d, n_clusters=2, intrinsic_dim=None, seed=seed)
    X = X.astype(np.float64)
    g = go.KnnOracle(X, knn=5, decay=decay, thresh=1e-3, distance=metric, n_jobs=1)
    g.kernel()
    assert g.passes == passes
    sc = _check_replay(g, X, X, 6, None, decay, 1e-3, metric)
    assert sc["fallback"] and sc["todo"].size > 0
