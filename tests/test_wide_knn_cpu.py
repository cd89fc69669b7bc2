"""kNN graphs with knn beyond the candidate lists, without a device: the routing predicate, the histogram bin edges and a
numpy model of the bound selection of gtb_knn_count_bound (csrc/refine.cu), which the GPU tests hold the kernel to."""
import math

import numpy as np
import pytest

from graphtools_b200 import pipeline

INF = float("inf")


def coarse_edge(elo, b):
    """Upper edge of coarse bin b: 2^(elo + b - 126), +inf for the overflow bin 63."""
    return INF if b >= 63 else float(np.uint32((elo + b + 1) << 23).view(np.float32))


def coarse_bin(w, elo):
    e = np.asarray(w, dtype=np.float32).view(np.int32) >> 23          # arithmetic: negative values -> bin 0
    return np.clip(e - elo, 0, 63)


def crossing(h, k):
    """(first bin whose cumulative count reaches k or len(h), cumulative count before it)."""
    c = np.cumsum(np.asarray(h, dtype=np.int64))
    b = int(np.searchsorted(c, k))
    return b, (int(c[b - 1]) if b > 0 else 0)


def radius_of_search2(s, metric):
    return math.sqrt(s) if metric == 0 else (0.5 * s if metric in (1, 4) else s)


def search2_of_radius(r, metric):
    return r * r if metric == 0 else (2.0 * r if metric in (1, 4) else r)


def collect_limit(r, metric, E, eps_rel):
    """collect_limit of csrc/refine.cu (before the upward rounding to float32)."""
    l2 = search2_of_radius(r, metric) * (1.0 + 1e-6) + E
    if metric == 2:
        l2 += 2.0 * eps_rel * r
    return l2


def collect_radius(dk, bw, bw_cert, dkmax, decay, rfac):
    if decay < 0:
        return dk
    r = bw * rfac
    return min(r if bw_cert else max(r, dk), dkmax)


def bound_model(hc, hf, elo, margin, s2, nrm, eps_rel, metric, knn, kmax, decay, thresh, bw_scale, nr):
    """One row of count_bound_kernel: (top, lim2 before rounding, ball_lo, ball_hi)."""
    bc, _ = crossing(hc, knn)
    t = coarse_edge(elo, bc) if bc < 64 else INF
    if not t < INF:
        return t, INF, nr, nr

    def fine_edge(k):
        b, _ = crossing(hf, k)
        return 0.5 * t if b == 0 else (0.5 * t * (1 + b / 16.0) if b < 17 else t)

    def upper(e):
        e /= s2
        return e * (1 + eps_rel) + nrm * 2.0 ** -23 if metric == 2 else e + (eps_rel + 2.0 ** -20) * nrm

    rfac = (-math.log(thresh)) ** (1.0 / decay) if decay >= 0 else 0.0
    ek = fine_edge(knn)
    dk = radius_of_search2(upper(ek), metric)
    bw = max(dk * bw_scale, np.finfo(float).eps) if decay >= 0 else 0.0
    dkmax = radius_of_search2(upper(fine_edge(kmax)), metric) if (decay >= 0 and 0 < kmax <= knn) else INF
    r = collect_radius(dk, bw, False, dkmax, decay, rfac)
    E = eps_rel * ek / s2 + nrm * 2.0 ** -23 if metric == 2 else eps_rel * nrm
    lim = collect_limit(r, metric, E, eps_rel)
    lim32 = np.float32(lim)                                             # the kernel rounds the limit up to float32
    if lim32 < lim:
        lim32 = np.nextafter(lim32, np.float32(np.inf))
    ls = np.float32(lim32 * np.float32(s2))
    if ls < 0.5 * t:
        lo, hi = 0, int(hf[0])
    elif ls < t:
        j = int((np.asarray(ls, np.float32).view(np.uint32) >> 19) & 15)
        lo = int(hf[0] + sum(hf[1:1 + j]))
        hi = lo + int(hf[1 + j])
    else:
        bl = int(coarse_bin(ls, elo))
        bmax = bc + margin - 1
        c = np.cumsum(np.asarray(hc, dtype=np.int64))
        top_b = min(bl, bmax)
        lo = int(c[min(bl - 1, top_b)]) if bl >= 1 else 0
        hi = int(c[bl]) if (bl <= bmax and bl < 63) else -1
    return t, lim, min(lo, nr), (-1 if hi < 0 else min(hi, nr))


@pytest.mark.parametrize("binary", [False, True])
def test_wide_knn_is_where_choose_S_raises(binary):
    for knn in range(1, 600):
        try:
            pipeline.choose_S(knn, binary)
            raises = False
        except NotImplementedError:
            raises = True
        assert pipeline.wide_knn(knn, binary) == raises, knn
    assert pipeline.wide_knn(121, False) and not pipeline.wide_knn(120, False)      # knn = 120 in-sample (+1)
    assert pipeline.wide_knn(125, True) and not pipeline.wide_knn(124, True)


def test_count_flavour():
    cf = pipeline.count_flavour
    assert cf("auto", 100, "euclidean") == "tch" and cf("tch1", 100, "cosine") == "tch"
    assert cf("auto", 510, "euclidean") == "tch"                # wide operand rows of the fp16x2 flavour
    assert cf("auto", 600, "euclidean") == "simt" and cf("auto", 100, "cityblock") == "simt"
    assert cf("simt", 100, "euclidean") == "simt" and cf("tc", 50, "euclidean") == "simt"
    with pytest.raises(ValueError):
        cf("bogus", 10, "euclidean")


def test_bin_edges_from_float32_bits():
    rng = np.random.default_rng(0)
    w = np.concatenate([rng.lognormal(0, 6, 200000), [0.0, -1e-3, -5.0, 1e-30, 3e38]]).astype(np.float32)
    for elo in (1, 60, 127, 190):
        b = coarse_bin(w, elo)
        edges = np.array([coarse_edge(elo, k) for k in range(64)])
        assert (w.astype(np.float64) < edges[b]).all()
        inner = b > 0
        assert (w[inner].astype(np.float64) >= edges[b[inner] - 1]).all()
        fin = edges[:63]
        assert np.array_equal(fin.astype(np.float32).astype(np.float64), fin)                 # exact in float64
        assert np.array_equal(np.log2(fin), np.arange(elo - 126, elo - 63, dtype=np.float64))
    # fine sub-bins: the top four mantissa bits split [t/2, t) into 16 steps of t/32; every edge exact in float32
    t = 2.0 ** 5
    v = np.linspace(t / 2, t, 100001, dtype=np.float32)[:-1]
    j = (v.view(np.uint32) >> 19) & 15
    up = t / 2 * (1 + (j + 1) / 16.0)
    assert (v < up).all() and (v >= up - t / 32).all()
    assert np.array_equal(up.astype(np.float32).astype(np.float64), up)


def test_count_window_and_margin():
    for vmax in (1e-20, 3.7, 4 * 8192.0, 1e30):
        elo = pipeline.count_window(vmax)
        assert coarse_bin(np.float32(vmax), elo) <= 62 and coarse_edge(elo, 62) > vmax
    assert pipeline.count_window(0.0) == 1
    assert pipeline.count_margin(1.0) == 2 and pipeline.count_margin(1.117) == 3
    assert pipeline.count_margin(84.8) == 9


def _row(counts_by_bin, nb):
    h = np.zeros(nb, np.int64)
    for b, c in counts_by_bin.items():
        h[b] = c
    return h


def test_bound_model_cumulative_crossing():
    elo, s2 = 120, 1.0
    hc = _row({3: 10, 5: 40, 6: 100, 7: 500}, 64)
    t, *_ = bound_model(hc, np.zeros(17), elo, 2, s2, 0.0, 0.0, 0, 50, 0, 40, 1e-4, 1.0, 10 ** 6)
    assert t == coarse_edge(elo, 5)                                    # 10 + 40 >= 50 at bin 5
    t, *_ = bound_model(hc, np.zeros(17), elo, 2, s2, 0.0, 0.0, 0, 51, 0, 40, 1e-4, 1.0, 10 ** 6)
    assert t == coarse_edge(elo, 6)
    # fine: 10 below the octave, then sub-bins; knn = 30 is reached in sub-bin 4 -> edge t/2 (1 + 5/16)
    t = coarse_edge(elo, 5)
    hf = _row({0: 10, 3: 15, 5: 5, 9: 20}, 17)
    _, lim, _, _ = bound_model(hc, hf, elo, 2, s2, 0.0, 0.0, 0, 30, 0, -1, 1.0, 1.0, 10 ** 6)
    U = 0.5 * t * (1 + 5 / 16.0)
    assert lim == pytest.approx(U * (1 + 1e-6), rel=1e-15)            # binary: radius = sqrt(U), limit = U (1 + 1e-6)
    # fine counts that fall short (a point of the coarse count missed at the octave's top edge): edge t
    _, lim, _, _ = bound_model(hc, _row({0: 10, 3: 15}, 17), elo, 2, s2, 0.0, 0.0, 0, 30, 0, -1, 1.0, 1.0, 10 ** 6)
    assert lim == pytest.approx(t * (1 + 1e-6), rel=1e-15)
    # already reached below the octave: edge t/2
    _, lim, _, _ = bound_model(hc, _row({0: 40}, 17), elo, 2, s2, 0.0, 0.0, 0, 30, 0, -1, 1.0, 1.0, 10 ** 6)
    assert lim == pytest.approx(0.5 * t * (1 + 1e-6), rel=1e-15)


def test_bound_model_rows_that_never_reach_k():
    hc = _row({3: 10, 63: 5}, 64)
    t, lim, lo, hi = bound_model(hc, np.zeros(17), 100, 2, 1.0, 1.0, 1e-3, 0, 20, 0, 40, 1e-4, 1.0, 15)
    assert t == INF and lim == INF and lo == hi == 15                  # every reference row is in the ball
    t, lim, lo, hi = bound_model(hc, np.zeros(17), 100, 2, 1.0, 1.0, 1e-3, 0, 12, 0, 40, 1e-4, 1.0, 15)
    assert t == INF and lim == INF                                      # crossing in the overflow bin


def test_bound_model_kmax_clamp():
    elo = 120
    hc = _row({5: 100}, 64)
    hf = _row({2: 30, 8: 40, 15: 30}, 17)
    args = (elo, 3, 1.0, 0.0, 0.0, 0)
    decay, thresh = 10, 1e-4
    _, lim_free, _, _ = bound_model(hc, hf, *args, 60, 0, decay, thresh, 1.0, 10 ** 6)
    _, lim_k, _, _ = bound_model(hc, hf, *args, 60, 60, decay, thresh, 1.0, 10 ** 6)
    t = coarse_edge(elo, 5)
    U = 0.5 * t * (1 + 8 / 16.0)                                        # 30 + 40 >= 60 in sub-bin 7 (bin 8)
    rfac = (-math.log(thresh)) ** (1 / decay)
    assert lim_free == pytest.approx((math.sqrt(U) * rfac) ** 2 * (1 + 1e-6), rel=1e-14)
    assert lim_k == pytest.approx(U * (1 + 1e-6), rel=1e-14)           # kmax = knn: radius = the knn-th bound
    _, lim_k20, _, _ = bound_model(hc, hf, *args, 60, 20, decay, thresh, 1.0, 10 ** 6)
    assert lim_k20 == pytest.approx(0.5 * t * (1 + 2 / 16.0) * (1 + 1e-6), rel=1e-14)   # 30 >= 20 in sub-bin 1


def test_bound_model_ball_size():
    elo = 120
    hc = _row({4: 7, 5: 100, 6: 300, 7: 1000, 9: 5000}, 64)
    hf = _row({0: 7, 2: 30, 8: 40, 15: 30}, 17)
    t = coarse_edge(elo, 5)
    # binary, knn = 60: limit just above the bound's edge, inside the octave -> its sub-bin brackets the ball
    _, lim, lo, hi = bound_model(hc, hf, elo, 2, 1.0, 0.0, 0.0, 0, 60, 0, -1, 1.0, 1.0, 10 ** 6)
    assert lim < t and lo == 77 and hi == 77
    _, lim, lo, hi = bound_model(hc, hf, elo, 2, 1.0, 0.0, 0.0, 0, 30, 0, -1, 1.0, 1.0, 10 ** 6)
    assert lo == 37 and hi == 37
    # decay 1: the limit is ~85x the bound, four octaves up; counted in full with margin 9, not with margin 2
    _, lim, lo, hi = bound_model(hc, hf, elo, 9, 1.0, 0.0, 0.0, 0, 60, 0, 1, 1e-4, 1.0, 10 ** 6)
    bl = int(coarse_bin(np.float32(lim), elo))
    assert bl == 11 and lo == 6407 and hi == 6407
    _, lim2, lo2, hi2 = bound_model(hc, hf, elo, 2, 1.0, 0.0, 0.0, 0, 60, 0, 1, 1e-4, 1.0, 10 ** 6)
    assert lim2 == lim and hi2 == -1 and lo2 == 407                   # only bins <= crossing + 1 are complete
    _, _, lo3, hi3 = bound_model(hc, hf, elo, 9, 1.0, 0.0, 0.0, 0, 60, 0, 1, 1e-4, 1.0, 500)
    assert lo3 == hi3 == 500                                            # capped at the reference rows


def test_shared_limit_formula_hand_cases():
    """The status-2 rows of refine_topk_kernel: r = max(bw rfac, dk) with bw = dk bw_scale, the (1 + 1e-6) widening,
    + E, the cityblock term; binary rows r = dk."""
    rfac = (-math.log(1e-4)) ** (1 / 40.0)
    dk = 2.0
    r = collect_radius(dk, dk * 1.0, False, INF, 40, rfac)
    assert r == dk * rfac and collect_limit(r, 0, 0.5, 1e-3) == (dk * rfac) ** 2 * (1 + 1e-6) + 0.5
    r = collect_radius(dk, dk * 0.5, False, INF, 40, rfac)             # bandwidth_scale 0.5: bw rfac < dk
    assert r == dk
    assert collect_limit(r, 1, 0.25, 1e-3) == 2 * dk * (1 + 1e-6) + 0.25           # cosine: 2 d
    assert collect_limit(r, 2, 0.25, 1e-3) == dk * (1 + 1e-6) + 0.25 + 2e-3 * dk   # cityblock
    assert collect_limit(r, 3, 0.25, 1e-3) == dk * (1 + 1e-6) + 0.25               # sqeuclidean: distance = search
    assert collect_radius(dk, 0.0, True, INF, -1, 0.0) == dk            # binary
    assert collect_radius(dk, 3.0, True, INF, 40, rfac) == 3.0 * rfac   # certified (fixed) bandwidth: support only
    assert collect_radius(dk, dk, False, 1.5, 40, rfac) == 1.5          # knn_max clamp
