"""Pruned one-product sweep (tile lists over locality-ordered operands): the order, the listed kernel's certification
contract, the skipped tiles, and builds bit-identical to the unpruned sweeps."""
import numpy as np
import pytest
import torch

from graphtools_b200 import _engine as E, pipeline, synth

pytestmark = pytest.mark.gpu


def _dev(X):
    return torch.from_numpy(np.ascontiguousarray(X)).cuda()


def test_order_sort_is_stable_counting_sort():
    rng = np.random.default_rng(1)
    for n, P in ((5000, 256), (70_001, 37), (3, 2)):
        cell = rng.integers(0, P, size=n).astype(np.int32)
        ws = torch.empty((E.lib().gtb_order_ws_elems(n, P),), dtype=torch.int32, device="cuda")
        perm = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        E.call("gtb_order_sort", _dev(cell), n, P, ws, perm)
        assert np.array_equal(perm.cpu().numpy(), np.argsort(cell, kind="stable"))


def test_order_assign_nearest_pivot():
    X, _ = synth.gaussian_mixture(20_000, 30, n_clusters=12, seed=4)
    op = pipeline.SearchOperand(_dev(X))
    P = 64
    cell = torch.empty((op.n,), dtype=torch.int32, device="cuda")
    E.call("gtb_order_assign", op.Xs, op.n, op.d, P, cell)
    c = cell.cpu().numpy()
    piv = X[np.arange(P) * (op.n // P)].astype(np.float64)
    D = ((X.astype(np.float64)[:, None, :] - piv[None]) ** 2).sum(-1)
    best = D.min(1)
    assert ((D[np.arange(op.n), c] - best) <= 1e-4 * (best + (X.astype(np.float64) ** 2).sum(1))).all()


def _one_product_operands(X):
    ref = pipeline.SearchOperand(_dev(X))
    scale = pipeline.fp16_scale(ref.norm_max())
    q_hi, _, q_n2 = ref.tc(0, 3, scale)
    r_hi, _, _ = ref.tc(1, 3, scale)
    return ref, scale, q_hi, q_n2, r_hi


@pytest.mark.parametrize("seeded", [False, True])
def test_listed_sweep_certification(seeded):
    """Hand-made lists: unit 0 sweeps every tile, unit 1 a single tile, the others every third tile, taken in reverse
    order.  Over the listed tiles the contract of the full sweep holds: every listed point that is not a candidate lies
    at exact squared distance >= tau - E, nothing from an unlisted tile becomes a candidate."""
    n, d = 6000, 100
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=8, seed=3)
    ref, scale, q_hi, q_n2, r_hi = _one_product_operands(X)
    s2 = scale * scale
    nt = ref.n_pad // 128
    n_units = -(-ref.n_pad // 512)
    lists = [list(range(nt)), [3]] + [list(range(u % 3, nt, 3)) for u in range(2, n_units)]
    ptr = torch.tensor(np.concatenate([[0], np.cumsum([len(l) for l in lists])]), dtype=torch.int64, device="cuda")
    tiles = torch.tensor(np.concatenate(lists), dtype=torch.int32, device="cuda")
    order = torch.arange(n_units - 1, -1, -1, dtype=torch.int32, device="cuda")
    scratch = torch.zeros((E.lib().gtb_tc_scratch_bytes(ref.n_pad),), dtype=torch.uint8, device="cuda")
    seed = None
    if seeded:
        seed = torch.empty((n, 2), dtype=torch.float32, device="cuda")
        pace = torch.zeros(1, dtype=torch.int32, device="cuda")
        E.call("gtb_knn_seed_tc", q_hi, q_n2 * s2, n, ref.n_pad, r_hi, n, ref.n_pad, ref.kp(3), 2, 2, seed, pace)
    cand = torch.full((n, 64), -7, dtype=torch.int32, device="cuda")
    tau = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    E.call("gtb_knn_topk_tc_seeded", q_hi, q_hi, q_n2 * s2, n, ref.n_pad, r_hi, r_hi, n, ref.n_pad, ref.kp(3), 3, 32, 2,
           2, seed, 1, cand, scratch, tau, None, ptr, tiles, order)
    torch.cuda.synchronize()
    cand = cand.cpu().numpy()
    tau2 = (tau / s2).cpu().numpy()
    assert np.array_equal(tau2[:, 0], tau2[:, 1])
    tau = tau2[:, 0]
    seed_h = None if seed is None else (seed / s2).cpu().numpy()[:, 0]
    X64 = X.astype(np.float64)
    Xc = X64 - X64.mean(0)
    nrm = (Xc ** 2).sum(1)
    eps = pipeline.eps_rel_tch1(d)
    for i in list(range(0, 1024, 7)) + list(range(1024, n, 29)):
        u = i // 512
        listed = np.concatenate([np.arange(t * 128, min(n, t * 128 + 128)) for t in lists[u]])
        assert (cand[i] != -7).all(), "output slot never written"
        c = cand[i][cand[i] >= 0]
        assert len(np.unique(c)) == len(c), "duplicate candidate"
        assert np.isin(c, listed).all(), "candidate from a tile outside the unit's list"
        D2 = ((X64[listed] - X64[i]) ** 2).sum(1)
        bound = eps * (nrm[i] + nrm.max())
        non = ~np.isin(listed, c)
        if non.any():
            assert np.isfinite(tau[i]), i
            assert D2[non].min() >= tau[i] - bound, i
        if seed_h is None:
            assert len(c) == min(64, len(listed))
        elif len(c) < min(64, len(listed)):
            assert tau[i] == seed_h[i] or (np.isinf(tau[i]) and np.isinf(seed_h[i]))
        assert set(listed[D2 < tau[i] - bound]).issubset(set(c))


def test_skipped_tiles_lie_beyond_the_seed(monkeypatch):
    """Every point of a tile missing from a unit's list is, from every row of the unit, at exact squared distance >= the
    row's seed + E: the sweep would not have admitted it."""
    n, d = 100_000, 100
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=10, seed=5)
    ref, scale, q_hi, q_n2, r_hi = _one_product_operands(X)
    s2 = scale * scale
    seed = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    pace = torch.zeros(1, dtype=torch.int32, device="cuda")
    E.call("gtb_knn_seed_tc", q_hi, q_n2 * s2, n, ref.n_pad, r_hi, n, ref.n_pad, ref.kp(3), 2, pipeline.SEED_STRIDE,
           seed, pace)
    eps = pipeline.eps_rel_tch1(d)
    monkeypatch.setattr(pipeline, "PRUNE_MAX_VISITED", 1.0)
    visited, total, lists = pipeline._tile_lists(ref, ref, seed, q_n2, eps, s2, 512)
    assert lists is not None and visited < total, visited / total
    ptr, tiles, order = (t.cpu().numpy() for t in lists)
    assert np.array_equal(np.sort(order), np.arange(len(order)))
    assert (np.diff(ptr)[order][:-1] >= np.diff(ptr)[order][1:]).all(), "longest list first"
    perm = ref.locality_order().long()
    Xp = ref.X.double()[perm]
    qn2 = q_n2[:n].double()[perm]
    thr = seed[:, 0].double()[perm] / s2 + eps * (qn2 + ref.maxnorm)
    nt = ref.n_pad // 128
    units_with_rows = np.arange(len(order)) * 512 < n
    pruned_units = np.flatnonzero((np.diff(ptr) < nt) & units_with_rows)   # lists that leave out at least one tile
    assert len(pruned_units) > 0
    for u in pruned_units[np.linspace(0, len(pruned_units) - 1, 10).astype(int)]:
        rows = torch.arange(u * 512, min(n, u * 512 + 512), device="cuda")
        listed = np.zeros(nt, dtype=bool)
        listed[tiles[ptr[u]:ptr[u + 1]]] = True
        assert np.array_equal(tiles[ptr[u]:ptr[u + 1]], np.sort(tiles[ptr[u]:ptr[u + 1]]))
        skipped = torch.from_numpy(np.flatnonzero(~listed)).cuda()
        cols = (skipped[:, None] * 128 + torch.arange(128, device="cuda")[None]).flatten()
        cols = cols[cols < n]
        D2 = torch.cdist(Xp[rows], Xp[cols]) ** 2
        assert (D2.min(dim=1).values >= thr[rows] * (1 - 1e-9)).all(), u


def _build(X, Y=None):
    """(raw kernel, K, P, degree) as host arrays; Y: out-of-sample rows (raw kernel only)."""
    ref = pipeline.SearchOperand(_dev(X))
    qry = ref if Y is None else pipeline.SearchOperand(_dev(Y), mean=ref.mean)
    R, _ = pipeline.knn_kernel(ref, qry, knn=6, decay=40, thresh=1e-4)
    out = [R.indptr.cpu().numpy(), R.indices.cpu().numpy(), R.data.cpu().numpy()]
    if Y is None:
        K, P, deg, _ = pipeline.symmetrize_normalize(R)
        out += [K.indptr.cpu().numpy(), K.indices.cpu().numpy(), K.data.cpu().numpy(), P.cpu().numpy(),
                deg.cpu().numpy()]
    return out, pipeline.stats()


@pytest.mark.parametrize("n,clusters,oos", [(100_000, 5, False), (200_000, 10, False), (200_000, 50, False),
                                            (150_000, 8, True)])
def test_pruned_build_bit_identical(n, clusters, oos, monkeypatch):
    """K, P and degree of the pruned build equal the plain seeded sweep's and the two-product sweep's bit for bit (the
    lists are used whatever share of the tile pairs they visit)."""
    A, _ = synth.gaussian_mixture(n + (n // 3 if oos else 0), 100, n_clusters=clusters, intrinsic_dim=10, seed=7)
    X, Y = A[:n], (A[n:] if oos else None)
    monkeypatch.setattr(pipeline, "PRUNE_MAX_VISITED", 1.0)
    pruned, st = _build(X, Y)
    assert st["impl"] == "tch1" and st["tile_lists"] and st["tile_pairs_visited"] < 1.0, st
    monkeypatch.setattr(pipeline, "PRUNE_MAX_VISITED", -1.0)
    plain, st2 = _build(X, Y)
    assert not st2["tile_lists"]
    monkeypatch.setenv("GTB_SEARCH_IMPL", "tch")
    two, _ = _build(X, Y)
    for a, b, c in zip(pruned, plain, two):
        assert np.array_equal(a, b)
        assert np.array_equal(a, c)


def test_isotropic_data_takes_the_plain_sweep():
    X = np.random.default_rng(2).normal(size=(100_000, 20)).astype(np.float32)
    pruned, st = _build(X)
    assert st["impl"] == "tch1" and not st["tile_lists"] and st["tile_pairs_visited"] > pipeline.PRUNE_MAX_VISITED
