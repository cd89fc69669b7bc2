"""kNN graphs with knn beyond the candidate lists (pipeline.wide_knn): the histogram count sweeps against float64
distances, parity with the CPU oracle through every entry point, bit identity across the count paths and runs, and the
early RowTooLong."""
import warnings

import numpy as np
import pytest
import torch

import graphtools_b200 as gt
from graphtools_b200 import _engine as E
from graphtools_b200 import pipeline, synth
from tests.parity import compare_dense, compare_sparse
from tests.test_wide_knn_cpu import bound_model, coarse_edge

pytestmark = pytest.mark.gpu


def _graph(X, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gt.Graph(X, verbose=0, **kw)


def _oracle(X, **kw):
    from oracle import graph_oracle as go
    return go.knn_graph(np.asarray(X, dtype=np.float64), **kw)


def _check(G, X, knn, decay=40, thresh=1e-4, what="", **kw):
    K_ref, P_ref = _oracle(X, knn=knn, decay=decay, thresh=thresh, **kw)
    tie = dict(X=X, knn=knn + 1, metric=kw.get("distance", "euclidean")) if decay is None else None
    r = compare_sparse(G.kernel, K_ref, thresh=None if decay is None else thresh, what=what + ".K", tie=tie)
    if r["n_exempt"] == 0:
        compare_sparse(G.diff_op, P_ref, what=what + ".P")
    return K_ref


# ---------------------------------------------------------------- the count kernels
def _exact_search_d2(qry, ref, s2):
    """float64 squared distances between the search copies, in search units, [nq, nr]."""
    a = qry.Xs.to(torch.float64)
    b = ref.Xs.to(torch.float64)
    if ref.metric == "cityblock":
        return torch.cdist(a, b, p=1) * s2
    return ((a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2 * a @ b.T).clamp_min(0) * s2


def _counts_below(d2_sorted, edges):
    """#{d2 < edge} per row and edge: d2_sorted [n, m] ascending, edges [n, e] -> [n, e]."""
    return torch.searchsorted(d2_sorted, edges.contiguous(), right=False)


@pytest.mark.parametrize("impl", ["tch", "simt"])
def test_count_histograms_against_float64(impl, monkeypatch):
    """Every counted cumulative bin lies between the float64 counts at edge - E and at edge + E (E the sweep's bound plus
    the float32 rounding of w); counts are identical from run to run."""
    monkeypatch.setenv("GTB_SEARCH_IMPL", impl)
    X, _ = synth.gaussian_mixture(20_000, 40, n_clusters=8, intrinsic_dim=8, seed=4)
    op = pipeline.SearchOperand(pipeline.to_device_f32(X))
    n, knn = op.n, 150
    flav = pipeline.count_flavour(impl, op.d, "euclidean")
    assert flav == impl
    f = pipeline.FLAVOURS.get(flav)
    scale = pipeline.fp16_scale(op.norm_max()) if f else 1.0
    s2 = scale * scale
    elo = pipeline.count_window(4.04 * op.maxnorm * s2)
    margin = 3

    def run(top=None):
        bins = 64 if top is None else 17
        h = torch.empty((op.n_pad, bins), dtype=torch.int32, device="cuda")
        if f:
            q_hi, q_lo, q_n2 = op.tc(0, 2, scale)
            r_hi, r_lo, _ = op.tc(1, 2, scale)
            E.call("gtb_knn_count_tc", q_hi, q_lo, q_n2 * s2, top, n, op.n_pad, r_hi, r_lo, n, op.n_pad, op.kp(2), 2,
                   2, knn, margin, elo, h, torch.empty((1,), dtype=torch.int32, device="cuda"))
        else:
            E.call("gtb_knn_count_simt", op.XT, op.n2, top, n, op.n_pad, op.XT, op.n2, n, op.n_pad, op.d_pad, knn,
                   margin, elo, h)
        return h[:n]

    hc = run()
    hc2 = run()
    qn2 = (op.tc(0, 2, scale)[2] if f else op.n2)[:n].to(torch.float64)
    eps = f.eps_rel(op.d) if f else pipeline.eps_rel_simt(op.d)
    Eb = ((eps + 2.0 ** -20) * (qn2 + op.maxnorm) * s2)[:, None]
    d2 = torch.sort(_exact_search_d2(op, op, s2), dim=1).values
    cum = torch.cumsum(hc.long(), dim=1)
    edges = torch.tensor([coarse_edge(elo, b) for b in range(63)], dtype=torch.float64, device="cuda")
    bc = torch.searchsorted(cum, torch.full((n, 1), knn, device="cuda", dtype=torch.long)).squeeze(1)
    assert (bc < 63).all()
    lo = _counts_below(d2, (edges[None, :] - Eb))
    hi = _counts_below(d2, (edges[None, :] + Eb))
    full = torch.arange(63, device="cuda")[None, :] <= (bc[:, None] + margin - 1)    # bins counted in full
    c63 = cum[:, :63]
    assert ((c63 >= lo) | ~full).all() and ((c63 <= hi) | ~full).all()
    # the fully counted bins are identical from run to run (above them, where the coarse sweep stopped counting
    # depends on when the two epilogue groups' increments landed; the bound reads none of those bins)
    assert torch.equal(hc[:, :63].masked_fill(~full, 0), hc2[:, :63].masked_fill(~full, 0))
    # fine pass below the coarse crossing edge t
    top = torch.tensor([coarse_edge(elo, int(b)) for b in bc.tolist()], dtype=torch.float32, device="cuda")
    top = torch.cat([top, torch.full((op.n_pad - n,), float("inf"), device="cuda")])
    hf = run(top)
    assert torch.equal(hf, run(top))
    t = top[:n].to(torch.float64)[:, None]
    fedges = torch.cat([0.5 * t, 0.5 * t * (1 + torch.arange(1, 17, device="cuda", dtype=torch.float64) / 16)], 1)
    fcum = torch.cumsum(hf.long(), dim=1)
    assert (fcum >= _counts_below(d2, fedges - Eb)).all() and (fcum <= _counts_below(d2, fedges + Eb)).all()
    # the bound kernel is the numpy model
    lim2 = torch.empty((n,), dtype=torch.float32, device="cuda")
    blo = torch.empty((n,), dtype=torch.int32, device="cuda")
    bhi = torch.empty_like(blo)
    E.call("gtb_knn_count_bound", hc, hf, n, n, elo, margin, s2, qn2.to(torch.float32), op.maxnorm, eps, 0, knn, 0,
           40.0, 1e-4, None, 0, 1.0, None, lim2, blo, bhi)
    hc_h, hf_h, q_h = hc.cpu().numpy(), hf.cpu().numpy(), qn2.cpu().numpy().astype(np.float32)
    lim_h, lo_h, hi_h = lim2.cpu().numpy(), blo.cpu().numpy(), bhi.cpu().numpy()
    for i in range(0, n, 997):
        nrm = float(q_h[i]) + float(np.float32(op.maxnorm))
        _, lim, lo, hi = bound_model(hc_h[i], hf_h[i], elo, margin, s2, nrm, eps, 0, knn, 0, 40.0, 1e-4, 1.0, n)
        up = np.float32(lim)
        if up < lim:
            up = np.nextafter(up, np.float32(np.inf))
        # rounded up to float32 (the kernel's contracted float64 arithmetic may land one float32 step higher)
        assert lim_h[i] == up or lim_h[i] == np.nextafter(up, np.float32(np.inf))
        if lim_h[i] == up:
            assert (lo_h[i], hi_h[i]) == (lo, hi)
    # the lower ball bound counts points whose approximate distance is under the limit: exact distance under limit + E
    ball = torch.searchsorted(d2, lim2.to(torch.float64)[:, None] * s2 + Eb, right=True).squeeze(1)
    assert (blo.long() <= ball).all()


# ---------------------------------------------------------------- parity with the oracle
@pytest.mark.parametrize("knn", [120, 150, 300, 500])
@pytest.mark.parametrize("decay", [40, 10, None])
def test_parity(knn, decay):
    X, _ = synth.gaussian_mixture(6000, 30, n_clusters=4, intrinsic_dim=6, seed=knn)
    G = _graph(X, knn=knn, decay=decay, thresh=1e-4)
    st = pipeline.stats()
    if pipeline.wide_knn(knn + 1, decay is None):                    # binary kNN fits the lists up to knn = 123
        assert st["wide_knn"] and st["count_sweeps"] == 2 and st["impl"] == "tch"
        assert st["ball_max"] <= pipeline.BALL_CAP and st["ball_mean"] >= knn
    else:
        assert not st["wide_knn"] and knn == 120 and decay is None
    _check(G, X, knn, decay, what="knn=%d decay=%s" % (knn, decay))


@pytest.mark.parametrize("opts", [dict(knn_max=200), dict(bandwidth_scale=1.5), dict(bandwidth=3.0),
                                  dict(anisotropy=0.5), dict(knn_max=150, bandwidth_scale=0.7)],
                         ids=["knn_max", "bw_scale", "bw_fixed", "anisotropy", "knn_max_bw_scale"])
def test_parity_options(opts):
    X, _ = synth.gaussian_mixture(5000, 20, n_clusters=3, intrinsic_dim=6, seed=11)
    G = _graph(X, knn=150, decay=20, thresh=1e-4, **opts)
    assert pipeline.stats()["count_sweeps"] == (0 if "bandwidth" in opts else 2)
    _check(G, X, 150, 20, what=str(opts), **opts)


@pytest.mark.parametrize("metric", ["sqeuclidean", "cosine", "correlation", "cityblock"])
def test_parity_metrics(metric):
    X, _ = synth.gaussian_mixture(5000, 24, n_clusters=4, intrinsic_dim=6, seed=12)
    X = X + 3.0                                                     # correlation: no constant rows; cosine: off zero
    G = _graph(X, knn=150, decay=40, thresh=1e-4, distance=metric)
    assert pipeline.stats()["impl"] == ("simt" if metric == "cityblock" else "tch")
    _check(G, X, 150, 40, distance=metric, what=metric)


def test_parity_float64_and_wide_rows():
    rng = np.random.default_rng(5)
    X, _ = synth.gaussian_mixture(5000, 40, n_clusters=4, intrinsic_dim=8, seed=13)
    X = X.astype(np.float64) * (1 + 1e-9 * rng.normal(size=X.shape))
    G = _graph(X, knn=150, decay=40, thresh=1e-4)
    _check(G, X, 150, 40, what="float64")
    X, _ = synth.gaussian_mixture(5000, 600, n_clusters=4, intrinsic_dim=8, seed=14)
    G = _graph(X, knn=150, decay=40, thresh=1e-4)
    assert pipeline.stats()["impl"] == "simt"                       # d > 510: the CUDA-core count path
    _check(G, X, 150, 40, what="d=600")


# ---------------------------------------------------------------- every entry point
def test_out_of_sample_and_interpolate():
    from oracle import graph_oracle as go
    X, _ = synth.gaussian_mixture(6000, 20, n_clusters=4, intrinsic_dim=6, seed=21)
    Y = X[:700] + 0.01
    G = _graph(X, knn=150, decay=40, thresh=1e-4)
    _, _, og = go.knn_graph(X.astype(np.float64), knn=150, decay=40, thresh=1e-4, return_oracle=True)
    Kyx_ref = og.kernel_to_data(Y.astype(np.float64))
    Kyx = G.build_kernel_to_data(Y)
    assert pipeline.stats()["wide_knn"]
    compare_sparse(Kyx, Kyx_ref, thresh=1e-4, what="Kyx")
    ext_ref = go.diff_op(Kyx_ref)
    compare_sparse(G.extend_to_data(Y), ext_ref, thresh=1e-4, what="ext")
    T = np.random.default_rng(0).normal(size=(X.shape[0], 3))
    assert np.allclose(G.interpolate(T, Y=Y), ext_ref.dot(T), rtol=1e-5, atol=1e-12)


def test_mnn_landmark_exact():
    from oracle import graph_oracle as go
    X, idx = synth.batched_mixture(3000, 2, 20, n_clusters=4, intrinsic_dim=6, seed=22)
    R_ref = go.mnn_kernel(X.astype(np.float64), idx, knn=150, decay=40, thresh=1e-4)
    K_ref = go.finish_kernel(R_ref, "mnn", 0.5)
    G = _graph(X, sample_idx=idx, kernel_symm="mnn", theta=0.5, knn=150, decay=40, thresh=1e-4)
    assert type(G).__name__ == "MNNGraph" and pipeline.stats()["wide_knn"]
    compare_sparse(G.kernel, K_ref, thresh=1e-4, what="mnn.K")
    X, _ = synth.gaussian_mixture(6000, 20, n_clusters=4, intrinsic_dim=6, seed=23)
    K_ref, _ = go.knn_graph(X.astype(np.float64), knn=150, decay=40, thresh=1e-4)
    clusters = go.random_landmark_clusters(X.astype(np.float64), 300, 42)
    op_ref, pnm_ref = go.landmark_operator(K_ref, clusters)
    G = _graph(X, knn=150, decay=40, thresh=1e-4, n_landmark=300, random_landmarking=True, random_state=42)
    assert np.array_equal(G.clusters, clusters)
    compare_dense(G.landmark_op, op_ref, what="landmark_op")
    compare_sparse(G.transitions, pnm_ref, what="transitions")
    X, _ = synth.gaussian_mixture(2500, 20, n_clusters=3, intrinsic_dim=6, seed=24)
    G = _graph(X, graphtype="exact", knn=150, decay=40, thresh=1e-4)
    assert pipeline.stats()["wide_knn"]                             # the adaptive bandwidth at knn + 1
    K_ref = go.finish_kernel(go.exact_kernel(X, knn=150, decay=40, thresh=1e-4))
    compare_dense(G.kernel, K_ref, thresh=1e-4, what="exact")


# ---------------------------------------------------------------- bit identity
def _kpd(G):
    return G.kernel.copy(), G.diff_op.copy(), np.asarray(G.kernel_degree).copy()


def _same(a, b):
    return all((x != y).nnz == 0 if hasattr(x, "nnz") else np.array_equal(x, y) for x, y in zip(a, b))


def test_bit_identity_paths_and_runs(monkeypatch):
    X, _ = synth.gaussian_mixture(8000, 30, n_clusters=4, intrinsic_dim=6, seed=31)
    monkeypatch.setenv("GTB_SEARCH_IMPL", "auto")
    a = _kpd(_graph(X, knn=200, decay=40, thresh=1e-4))
    assert pipeline.stats()["impl"] == "tch"
    b = _kpd(_graph(X, knn=200, decay=40, thresh=1e-4))
    monkeypatch.setenv("GTB_SEARCH_IMPL", "simt")
    c = _kpd(_graph(X, knn=200, decay=40, thresh=1e-4))
    assert pipeline.stats()["impl"] == "simt"
    assert _same(a, b) and _same(a, c)


@pytest.mark.parametrize("knn", [119, 120])
def test_switch_at_knn_120(knn):
    X, _ = synth.gaussian_mixture(5000, 20, n_clusters=3, intrinsic_dim=6, seed=32)
    G = _graph(X, knn=knn, decay=40, thresh=1e-4)
    assert pipeline.stats()["wide_knn"] == (knn >= 120)
    _check(G, X, knn, 40, what="knn=%d" % knn)


def test_row_too_long_before_the_collect_sweep():
    X, _ = synth.gaussian_mixture(20_000, 20, n_clusters=2, intrinsic_dim=4, seed=33)
    with pytest.raises(pipeline.RowTooLong, match="neighbours inside the kernel radius"):
        _graph(X, knn=150, decay=1, thresh=1e-4)
    st = pipeline.stats()
    assert st["count_sweeps"] == 2 and st["radius_pairs"] == 0 and st["ball_max"] is None
