"""Unit tests of individual C-ABI kernels against numpy (run on the B200 box)."""
import numpy as np
import pytest
import torch

from graphtools_b200 import _engine as E
from graphtools_b200 import pipeline, synth

pytestmark = pytest.mark.gpu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("n", [1, 7, 2048, 2049, 100003, 3000017])
def test_exclusive_scan(n):
    rng = np.random.default_rng(n)
    x = rng.integers(0, 50, size=n).astype(np.int32)
    out = pipeline.exclusive_scan(_dev(x)).cpu().numpy()
    ref = np.concatenate([[0], np.cumsum(x.astype(np.int64))])
    assert np.array_equal(out, ref)


@pytest.mark.parametrize("n,d", [(1797, 64), (1000, 100), (130, 3), (5000, 37)])
def test_prepare_operand(n, d):
    X, _ = synth.gaussian_mixture(n, d, n_clusters=4, intrinsic_dim=min(5, d), seed=1)
    op = pipeline.SearchOperand(_dev(X))
    mean = X.astype(np.float64).mean(0)
    assert np.allclose(op.mean.cpu().numpy(), mean, rtol=1e-6, atol=1e-6)
    Xc = (X - op.mean.cpu().numpy()[None, :]).astype(np.float32)
    XT = op.XT.cpu().numpy()
    assert XT.shape == (op.d_pad, op.n_pad)
    assert np.array_equal(XT[:d, :n], Xc.T)
    assert (XT[d:, :] == 0).all() and (XT[:, n:] == 0).all()
    n2 = op.n2.cpu().numpy()
    ref_n2 = (Xc.astype(np.float64) ** 2).sum(1)
    assert np.allclose(n2[:n], ref_n2, rtol=1e-6)
    assert (n2[:n] >= ref_n2 * (1 - 1e-7)).all()
    assert np.isinf(n2[n:]).all()
    assert np.isclose(op.maxnorm, n2[:n].max())


@pytest.mark.parametrize("n,d,S", [(1797, 64, 48), (3000, 100, 48), (700, 20, 16), (2500, 10, 64), (300, 5, 128),
                                   (40, 3, 48)])
def test_topk_candidates_contain_true_neighbours(n, d, S):
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=min(8, d), seed=3)
    op = pipeline.SearchOperand(_dev(X))
    cand = torch.empty((n, S), dtype=torch.int32, device="cuda")
    tau = torch.empty((n,), dtype=torch.float32, device="cuda")
    E.call("gtb_knn_topk_simt", op.XT, op.n2, n, op.n_pad, op.XT, op.n2, n, op.n_pad, op.d_pad, S, cand, tau)
    cand = cand.cpu().numpy(); tau = tau.cpu().numpy()
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1) if n <= 3000 else None
    k_true = min(S - 8, n)
    order = np.argsort(D2, axis=1, kind="stable")
    for i in range(0, n, max(1, n // 200)):
        c = cand[i][cand[i] >= 0]
        assert len(np.unique(c)) == len(c), "duplicate candidate"
        assert len(c) == min(S, n)
        assert set(order[i, :k_true]).issubset(set(c)), "row %d misses a true neighbour" % i
        if n > S:
            # tau = S-th smallest approximate d2: every non-candidate is at least that far (up to fp32 error)
            non = np.setdiff1d(np.arange(n), c)
            Xc = X64 - X64.mean(0)
            bound = pipeline.eps_rel_simt(d) * ((Xc[i] ** 2).sum() + (Xc ** 2).sum(1).max())
            assert D2[i, non].min() >= tau[i] - bound
        else:
            assert np.isinf(tau[i])


def test_radius_pairs_complete():
    n, d = 2000, 30
    X, _ = synth.gaussian_mixture(n, d, n_clusters=3, intrinsic_dim=6, seed=4)
    op = pipeline.SearchOperand(_dev(X))
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1)
    r2 = np.partition(D2, 40, axis=1)[:, 40]
    lim = _dev((r2 * 1.0001 + 1e-3).astype(np.float32))
    limp = torch.zeros(op.n_pad, dtype=torch.float32, device="cuda"); limp[:n] = lim
    cap = 1 << 20
    pairs = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    rowcnt = torch.zeros(op.n_pad, dtype=torch.int32, device="cuda")
    E.call("gtb_knn_radius_simt", op.XT, op.n2, limp, n, op.n_pad, op.XT, op.n2, n, op.n_pad, op.d_pad, pairs, cap,
           counter, rowcnt)
    m = int(counter.item())
    pr = pairs[:m].cpu().numpy()
    got = set(map(tuple, pr))
    assert len(got) == m
    want = set(zip(*np.nonzero(D2 <= r2[:, None])))
    assert want.issubset(got)
    extra = got - want
    assert len(extra) < 0.05 * len(want) + 50
    assert np.array_equal(np.bincount(pr[:, 0], minlength=n), rowcnt[:n].cpu().numpy())


# ------------------------------------------------------------------ tensor-core (tcgen05) search
def _tc_topk(X, Y=None, dtype=0, ls=32, qtiles=1):
    ref = pipeline.SearchOperand(_dev(X))
    qry = ref if Y is None else pipeline.SearchOperand(_dev(Y), mean=ref.mean)
    scale = pipeline.fp16_scale(max(qry.norm_max(), ref.norm_max())) if dtype == 2 else 1.0
    q_hi, q_lo, q_n2 = qry.tc(0, dtype, scale)
    r_hi, r_lo, _ = ref.tc(1, dtype, scale)
    cand = torch.full((qry.n, 2 * ls), -7, dtype=torch.int32, device="cuda")
    scratch = torch.zeros((E.lib().gtb_tc_scratch_bytes(qry.n_pad),), dtype=torch.uint8, device="cuda")
    tau = torch.empty((qry.n, 2), dtype=torch.float32, device="cuda")
    pace = torch.zeros(1, dtype=torch.int32, device="cuda")
    E.call("gtb_knn_topk_tc", q_hi, q_lo, q_n2 * (scale * scale), qry.n, qry.n_pad, r_hi, r_lo, ref.n, ref.n_pad,
           ref.kp(dtype), dtype, ls, 2, qtiles, cand, scratch, tau, pace)
    torch.cuda.synchronize()
    return cand.cpu().numpy(), (tau / (scale * scale)).cpu().numpy().min(axis=1), qry, ref


def test_tc_operand_split():
    X, _ = synth.gaussian_mixture(300, 100, n_clusters=3, intrinsic_dim=10, seed=2)
    op = pipeline.SearchOperand(_dev(X))
    hi, lo, n2 = [t.cpu().numpy() for t in op.tc(1)]
    assert hi.shape == (384, 104)
    Xc = (X - op.mean.cpu().numpy()[None, :]).astype(np.float32)
    full = hi.astype(np.float64) + lo.astype(np.float64)
    assert np.allclose(full[:300, :100], -2.0 * Xc, rtol=2e-6, atol=1e-9)
    assert (hi.view(np.uint32) & 0x1FFF == 0).all() and (lo.view(np.uint32) & 0x1FFF == 0).all()
    assert np.allclose(full[:300, 100], (Xc.astype(np.float64) ** 2).sum(1), rtol=2e-6)
    assert (full[:300, 101:] == 0).all()
    assert np.allclose(full[300:, 100], 1e30, rtol=1e-3) and (full[300:, :100] == 0).all()
    qhi, qlo, _ = [t.cpu().numpy() for t in op.tc(0)]
    qfull = qhi.astype(np.float64) + qlo.astype(np.float64)
    assert np.allclose(qfull[:300, :100], Xc, rtol=2e-6, atol=1e-9) and (qfull[:300, 100] == 1).all()


@pytest.mark.parametrize("ls", [32, 16])
@pytest.mark.parametrize("dtype", [0, 1, 2])
@pytest.mark.parametrize("n,d", [(1797, 64), (3000, 100), (700, 20), (2500, 10), (300, 5), (40, 3), (1000, 31),
                                 (1000, 55), (777, 103)])
def test_tc_topk_candidates(n, d, dtype, ls):
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=min(8, d), seed=3)
    cand, tau, qry, ref = _tc_topk(X, dtype=dtype, ls=ls)
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1)
    order = np.argsort(D2, axis=1, kind="stable")
    Xc = X64 - X64.mean(0)
    nrm = (Xc ** 2).sum(1)
    eps = (pipeline.eps_rel_tc, pipeline.eps_rel_tc16, pipeline.eps_rel_tch)[dtype](d)
    # two lists of ls: references in even / odd 128-row tiles
    tile_par = (np.arange(n) // 128) % 2
    n_even, n_odd = int((tile_par == 0).sum()), int((tile_par == 1).sum())
    for i in range(0, n, max(1, n // 300)):
        assert (cand[i] != -7).all(), "output slot never written"
        c = cand[i][cand[i] >= 0]
        assert (c < n).all(), "padded reference leaked into the candidates"
        assert len(np.unique(c)) == len(c), "duplicate candidate"
        assert len(c) == min(ls, n_even) + min(ls, n_odd), (i, len(c))
        assert (tile_par[cand[i][:ls][cand[i][:ls] >= 0]] == 0).all() and \
            (tile_par[cand[i][ls:][cand[i][ls:] >= 0]] == 1).all()
        bound = eps * (nrm[i] + nrm.max())
        # the true nearest ls - 8 are present unless the fast pass cannot tell them apart from the ls-th
        sure = [j for j in order[i, :min(ls - 8, n)] if D2[i, j] + 2 * bound < D2[i, order[i, min(ls - 1, n - 1)]]]
        assert set(sure).issubset(set(c)), "row %d misses a true neighbour" % i
        non = np.setdiff1d(np.arange(n), c)
        if len(non):
            assert np.isfinite(tau[i])
            assert D2[i, non].min() >= tau[i] - bound
        if n_even <= ls and n_odd <= ls:
            assert np.isinf(tau[i])


@pytest.mark.parametrize("ls", [32, 16])
@pytest.mark.parametrize("n,d", [(2000, 127), (3000, 129), (1500, 200), (900, 510), (2500, 333)])
def test_tc_topk_wide_rows(n, d, ls):
    """Operand rows beyond 128 float16 elements (d up to 510): the reference tiles stream in chunks of 8 k-steps, the
    accumulator collects the chunks -- same contract as the resident-row kernel."""
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=8, seed=3)
    cand, tau, qry, ref = _tc_topk(X, dtype=2, ls=ls)
    assert ref.kp(2) > 128
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1)
    Xc = X64 - X64.mean(0)
    nrm = (Xc ** 2).sum(1)
    eps = pipeline.eps_rel_tch(d)
    tile_par = (np.arange(n) // 128) % 2
    n_even, n_odd = int((tile_par == 0).sum()), int((tile_par == 1).sum())
    for i in range(0, n, max(1, n // 300)):
        assert (cand[i] != -7).all(), "output slot never written"
        c = cand[i][cand[i] >= 0]
        assert (c < n).all() and len(np.unique(c)) == len(c)
        assert len(c) == min(ls, n_even) + min(ls, n_odd), (i, len(c))
        bound = eps * (nrm[i] + nrm.max())
        non = np.setdiff1d(np.arange(n), c)
        assert np.isfinite(tau[i])
        assert D2[i, non].min() >= tau[i] - bound
        assert set(np.flatnonzero(D2[i] < tau[i] - bound)).issubset(set(c))


@pytest.mark.parametrize("n,d", [(1797, 64), (3000, 100), (300, 5), (40, 3), (1000, 31), (777, 103), (5000, 100)])
def test_tc_topk_two_query_tiles(n, d):
    """fp16x2 with two query tiles per CTA: ONE list of 32 per row over the whole reference set."""
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=min(8, d), seed=3)
    ls = 16
    cand, tau, qry, ref = _tc_topk(X, dtype=2, ls=ls, qtiles=2)
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1)
    order = np.argsort(D2, axis=1, kind="stable")
    Xc = X64 - X64.mean(0)
    nrm = (Xc ** 2).sum(1)
    eps = pipeline.eps_rel_tch(d)
    for i in range(0, n, max(1, n // 400)):
        assert (cand[i] != -7).all(), "output slot never written"
        c = cand[i][cand[i] >= 0]
        assert (c < n).all(), "padded reference leaked into the candidates"
        assert len(np.unique(c)) == len(c), "duplicate candidate"
        assert len(c) == min(2 * ls, n), (i, len(c))
        bound = eps * (nrm[i] + nrm.max())
        sure = [j for j in order[i, :min(2 * ls - 8, n)]
                if D2[i, j] + 2 * bound < D2[i, order[i, min(2 * ls - 1, n - 1)]]]
        assert set(sure).issubset(set(c)), "row %d misses a true neighbour" % i
        non = np.setdiff1d(np.arange(n), c)
        if len(non):
            assert np.isfinite(tau[i])
            assert D2[i, non].min() >= tau[i] - bound
        else:
            assert np.isinf(tau[i])


def _tc_topk_one_product(X, stride):
    """fp16x1 sweep (dtype 3): optional seed pass over every stride-th tile, then the full sweep, one list of 64."""
    ref = pipeline.SearchOperand(_dev(X))
    scale = pipeline.fp16_scale(ref.norm_max())
    q_hi, q_lo, q_n2 = ref.tc(0, 3, scale)
    r_hi, r_lo, _ = ref.tc(1, 3, scale)
    n = ref.n
    scratch = torch.zeros((E.lib().gtb_tc_scratch_bytes(ref.n_pad),), dtype=torch.uint8, device="cuda")
    pace = torch.zeros(1, dtype=torch.int32, device="cuda")
    seed = None
    if stride > 1:
        seed = torch.empty((n, 2), dtype=torch.float32, device="cuda")
        E.call("gtb_knn_seed_tc", q_hi, q_n2 * (scale * scale), n, ref.n_pad, r_hi, n, ref.n_pad, ref.kp(3), 2, stride,
               seed, pace)
    cand = torch.full((n, 64), -7, dtype=torch.int32, device="cuda")
    tau = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    E.call("gtb_knn_topk_tc_seeded", q_hi, q_lo, q_n2 * (scale * scale), n, ref.n_pad, r_hi, r_lo, n, ref.n_pad,
           ref.kp(3), 3, 32, 2, 2, seed, 1, cand, scratch, tau, pace)
    torch.cuda.synchronize()
    seed_h = None if seed is None else (seed / (scale * scale)).cpu().numpy()[:, 0]
    return cand.cpu().numpy(), (tau / (scale * scale)).cpu().numpy(), seed_h


@pytest.mark.parametrize("stride", [1, 2, 5])
@pytest.mark.parametrize("n,d", [(1797, 64), (3000, 100), (300, 5), (40, 3), (1000, 31), (777, 103), (6000, 100),
                                 (2500, 110)])
def test_tc_topk_one_product_seeded(n, d, stride):
    """fp16x1 (one product, dtype 3), cold and with thresholds seeded from a strided sample: every reference point
    that is not a candidate lies at an exact squared distance >= tau - E (the certification contract), the list is
    complete when it is not full, and both tau slots agree."""
    X, _ = synth.gaussian_mixture(n, d, n_clusters=5, intrinsic_dim=min(8, d), seed=3)
    cand, tau2, seed = _tc_topk_one_product(X, stride)
    assert np.array_equal(tau2[:, 0], tau2[:, 1])
    tau = tau2[:, 0]
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1)
    Xc = X64 - X64.mean(0)
    nrm = (Xc ** 2).sum(1)
    eps = pipeline.eps_rel_tch1(d)
    n_full = 0
    for i in range(0, n, max(1, n // 400)):
        assert (cand[i] != -7).all(), "output slot never written"
        c = cand[i][cand[i] >= 0]
        assert (c < n).all(), "padded reference leaked into the candidates"
        assert len(np.unique(c)) == len(c), "duplicate candidate"
        bound = eps * (nrm[i] + nrm.max())
        non = np.setdiff1d(np.arange(n), c)
        if len(non):
            assert np.isfinite(tau[i]), i
            assert D2[i, non].min() >= tau[i] - bound, i
        if stride == 1:
            assert len(c) == min(64, n)
            if n <= 64:
                assert np.isinf(tau[i])
        else:
            # seeded: a list that did not fill reports the seed and holds everything (approximately) under it
            if len(c) < min(64, n):
                assert tau[i] == seed[i] or (np.isinf(tau[i]) and np.isinf(seed[i]))
                assert set(np.flatnonzero(D2[i] < tau[i] - bound)).issubset(set(c))
            else:
                n_full += 1
                assert tau[i] <= seed[i]
        # the nearest neighbours well inside the threshold are present
        assert set(np.flatnonzero(D2[i] < tau[i] - bound)).issubset(set(c))


@pytest.mark.parametrize("stride", [1, 16])
def test_tc_one_product_split_last_round(stride):
    """More query cluster-units than clusters with a short last round (50k queries: 98 units for 74 clusters -> 24 units
    left, split three ways over the reference range and merged by merge_pieces_kernel): the certification contract
    holds for rows of the full rounds and of the split round alike, against exact float64 distances."""
    n, d = 50_000, 32
    X, _ = synth.gaussian_mixture(n, d, n_clusters=8, intrinsic_dim=8, seed=21)
    cand, tau2, seed = _tc_topk_one_product(X, stride)
    assert np.array_equal(tau2[:, 0], tau2[:, 1])
    tau = tau2[:, 0]
    Xd = _dev(X).double()
    Xc = Xd - Xd.mean(0)
    nrm = (Xc * Xc).sum(1)
    eps = pipeline.eps_rel_tch1(d)
    rows = np.unique(np.concatenate([np.arange(0, n, 257), np.arange(37_888, n, 61), [n - 1]]))
    assert (cand != -7).all(), "output slot never written"
    for i in rows.tolist():
        c = cand[i][cand[i] >= 0]
        assert len(np.unique(c)) == len(c) and (c < n).all()
        d2 = ((Xd - Xd[i]) ** 2).sum(1)
        is_c = torch.zeros(n, dtype=torch.bool, device="cuda")
        is_c[torch.from_numpy(c).cuda().long()] = True
        bound = eps * float(nrm[i] + nrm.max())
        assert np.isfinite(tau[i])
        assert float(d2[~is_c].min()) >= tau[i] - bound, i
        inside = torch.nonzero(d2 < tau[i] - bound).flatten()
        assert bool(is_c[inside].all()), i
        if stride == 1:
            assert len(c) == 64


def test_tc_topk_out_of_sample():
    X, _ = synth.gaussian_mixture(5000, 100, n_clusters=6, intrinsic_dim=10, seed=5)
    Y, _ = synth.gaussian_mixture(333, 100, n_clusters=6, intrinsic_dim=10, seed=5)
    Y = Y + np.float32(0.01)
    cand, tau, qry, ref = _tc_topk(X, Y)
    D2 = ((Y.astype(np.float64)[:, None, :] - X.astype(np.float64)[None, :, :]) ** 2).sum(-1)
    order = np.argsort(D2, axis=1, kind="stable")
    for i in range(333):
        assert set(order[i, :24]).issubset(set(cand[i]))


@pytest.mark.parametrize("dtype", [0, 1, 2])
def test_tc_radius_pairs_complete(dtype):
    n, d = 2000, 30
    X, _ = synth.gaussian_mixture(n, d, n_clusters=3, intrinsic_dim=6, seed=4)
    op = pipeline.SearchOperand(_dev(X))
    X64 = X.astype(np.float64)
    D2 = ((X64[:, None, :] - X64[None, :, :]) ** 2).sum(-1)
    r2 = np.partition(D2, 40, axis=1)[:, 40]
    limp = torch.zeros(op.n_pad, dtype=torch.float32, device="cuda")
    Xc = X64 - X64.mean(0)
    slack = (pipeline.eps_rel_tc, pipeline.eps_rel_tc16, pipeline.eps_rel_tch)[dtype](d) * 2 * (Xc ** 2).sum(1).max()
    limp[:n] = _dev((r2 * 1.0001 + slack).astype(np.float32))
    cap = 1 << 20
    pairs = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    rowcnt = torch.zeros(op.n_pad, dtype=torch.int32, device="cuda")
    scale = pipeline.fp16_scale(op.norm_max()) if dtype == 2 else 1.0
    q_hi, q_lo, q_n2 = op.tc(0, dtype, scale)
    r_hi, r_lo, _ = op.tc(1, dtype, scale)
    E.call("gtb_knn_radius_tc", q_hi, q_lo, q_n2 * (scale * scale), limp * (scale * scale), n, op.n_pad, r_hi, r_lo, n,
           op.n_pad, op.kp(dtype), dtype, 2, pairs, cap, counter, rowcnt, None)
    m = int(counter.item())
    pr = pairs[:m].cpu().numpy()
    got = set(map(tuple, pr))
    assert len(got) == m
    want = set(zip(*np.nonzero(D2 <= r2[:, None])))
    assert want.issubset(got)
    assert len(got - want) < (0.05, 0.5, 3.0)[dtype] * len(want) + 50
    assert np.array_equal(np.bincount(pr[:, 0], minlength=n), rowcnt[:n].cpu().numpy())


def _csr_dev(M):
    M = M.tocsr(); M.sort_indices()
    return _dev(M.indptr.astype(np.int64)), _dev(M.indices.astype(np.int32)), _dev(M.data.astype(np.float64))


def _random_kernel(n, density, seed, hub=None):
    """Random non-symmetric sparse matrix with a unit diagonal; ``hub`` = (row, count) adds a long row / column."""
    from scipy import sparse
    rng = np.random.default_rng(seed)
    M = sparse.random(n, n, density=density, random_state=seed, format="lil", dtype=np.float64)
    if hub is not None:
        r, cnt = hub
        cols = rng.choice(n, cnt, replace=False)
        M[r, cols] = rng.uniform(0.1, 1.0, cnt)
        rows = rng.choice(n, cnt, replace=False)
        M[rows, r] = rng.uniform(0.1, 1.0, cnt)
    M.setdiag(1.0)
    M = M.tocsr(); M.sort_indices()
    return M


@pytest.mark.parametrize("n,density,hub", [(500, 0.01, None), (3000, 0.004, (7, 200)), (6000, 0.002, (11, 5000)),
                                            (1, 1.0, None), (33, 0.5, None)])
def test_transpose_and_row_sort(n, density, hub):
    """csrc/symm.cu transpose_count / scan / transpose_scatter / csr_sort_rows against scipy's CSR transpose:
    short rows (register tier), rows of 33..256 (warp shared-memory tier), 257..4096 (block tier) and a 5000-entry
    hub row (global-memory tier)."""
    from scipy import sparse
    M = _random_kernel(n, density, 5, hub)
    R = pipeline.DeviceCSR(*_csr_dev(M), M.shape)
    T = pipeline.transpose_csr(R)
    want = sparse.csr_matrix(M.T); want.sort_indices()
    assert np.array_equal(T.indptr.cpu().numpy(), want.indptr)
    assert np.array_equal(T.indices.cpu().numpy(), want.indices)
    assert np.array_equal(T.data.cpu().numpy(), want.data)


@pytest.mark.parametrize("mode,theta", [("+", None), ("*", None), ("mnn", 0.3), ("mnn", 1.0)])
@pytest.mark.parametrize("n,density,hub", [(800, 0.01, None), (3000, 0.004, (7, 300)), (2000, 0.03, None)])
def test_symmetrize_normalize_matches_scipy(mode, theta, n, density, hub):
    """The whole K4 chain (transpose + merge count / scan / fill) against scipy's own binops (the reference's
    base.py:557-577) and sklearn's normalize: structure and K values bit-exact, P within 1e-15, on rows of every
    length tier; flags report a missing diagonal."""
    from oracle import graph_oracle as go
    M = _random_kernel(n, density, 9, hub)
    K_ref = go.symmetrize(M, mode, theta).tocsr()
    K_ref.eliminate_zeros(); K_ref.sort_indices()
    K, P, deg, flags = pipeline.symmetrize_normalize(pipeline.DeviceCSR(*_csr_dev(M), M.shape), mode, theta, 0.0)
    Kh = K.to_scipy()
    assert np.array_equal(Kh.indptr, K_ref.indptr) and np.array_equal(Kh.indices, K_ref.indices)
    assert np.array_equal(Kh.data, K_ref.data)
    P_ref = go.diff_op(K_ref)
    assert np.allclose(P.cpu().numpy(), P_ref.data, rtol=1e-14, atol=0)
    assert np.allclose(deg.cpu().numpy(), np.asarray(K_ref.sum(1)).ravel(), rtol=1e-14, atol=0)
    assert flags == 0
    M2 = M.tolil(); M2[3, 3] = 0; M2 = M2.tocsr(); M2.eliminate_zeros()
    _, _, _, flags = pipeline.symmetrize_normalize(pipeline.DeviceCSR(*_csr_dev(M2), M2.shape), mode, theta, 0.0)
    assert flags == 2


@pytest.mark.parametrize("mode,theta", [("+", None), ("*", None), ("mnn", 0.0), ("mnn", 0.3), ("mnn", 0.5),
                                        ("mnn", 1.0)])
def test_sharded_symmetrise_merge_matches_global(mode, theta):
    """The multi-GPU path on one device: the rows of two shards are bucketed by route_count / route_fill, the
    records a rank would receive are turned into the transposed rows (records_count / scatter / sort) and merged --
    bit-identical to the single-GPU symmetrise + normalise.  MNN weights from theta = 0 (the larger of the two
    directions) to theta = 1 (the smaller: one-way edges drop out of the merged rows)."""
    from graphtools_b200 import distributed as gd
    X, _ = synth.gaussian_mixture(3000, 20, n_clusters=4, intrinsic_dim=5, seed=9)
    ref = pipeline.SearchOperand(_dev(X))
    R, _ = pipeline.knn_kernel(ref, ref, knn=6, decay=10, thresh=1e-3)
    K, P, deg, _ = pipeline.symmetrize_normalize(R, mode, theta, 0.0)
    Kh, Ph = K.to_scipy(), K.to_scipy(P)
    Rh = R.to_scipy()
    n, world = 3000, 2
    per = gd.rows_per_rank(n, world)
    bounds = [gd.shard_bounds(n, world, r) for r in range(world)]
    smode = pipeline.SYM_MODES[mode]
    sends = []
    for lo, hi in bounds:
        pa, ia, va = _csr_dev(Rh[lo:hi])
        send, counts = gd.cuda_bucket_edges(pa, ia, va, lo, per, world)
        counts = counts.cpu().numpy()
        i, j, w = (t.cpu().numpy() for t in gd.unpack_records(send))
        assert counts.sum() == len(i)
        assert (np.diff(np.minimum(j // per, world - 1)) >= 0).all()       # destination-major
        sends.append((send, np.concatenate([[0], np.cumsum(counts)])))
    for r, (lo, hi) in enumerate(bounds):
        m = hi - lo
        rec = torch.cat([s[o[r]:o[r + 1]] for s, o in sends]).contiguous()   # what rank r receives (rank-major)
        k = rec.shape[0]
        cnt = torch.empty(m, dtype=torch.int32, device="cuda")
        E.call("gtb_records_count", rec, k, lo, cnt, m)
        ptr_t = pipeline.exclusive_scan(cnt)
        t_rec = torch.empty((k, 2), dtype=torch.int64, device="cuda")
        E.call("gtb_records_scatter", rec, k, lo, pipeline.cursor32(ptr_t), t_rec)
        pa, ia, va = _csr_dev(Rh[lo:hi])
        flags = torch.zeros(1, dtype=torch.int32, device="cuda")
        outptr, oi, ov, pv, dg, _ = pipeline.merge_with_transpose(pa, ia, va, ptr_t, t_rec, m, lo, smode,
                                                                  0.0 if theta is None else theta, True, flags)
        Ks, Ps = Kh[lo:hi], Ph[lo:hi]
        assert np.array_equal(outptr.cpu().numpy(), Ks.indptr)
        assert np.array_equal(oi.cpu().numpy(), Ks.indices)
        assert np.array_equal(ov.cpu().numpy(), Ks.data)
        assert np.array_equal(pv.cpu().numpy(), Ps.data)
        assert np.array_equal(dg.cpu().numpy(), deg.cpu().numpy()[lo:hi])
        assert int(flags.item()) == 0


def test_landmark_operator_is_reproducible_and_handles_long_rows():
    """csrc/landmark.cu: fixed-point accumulation makes landmark_op / column sums bit-identical from run to run;
    rows of every tier (<= 32, <= 256, longer) agree with the oracle's C^T K aggregation."""
    from oracle import graph_oracle as go
    from graphtools_b200 import landmark as lm
    n, L = 4000, 300
    M = _random_kernel(n, 0.004, 2, (5, 900))
    K = go.symmetrize(M, "+").tocsr(); K.sort_indices()
    clusters = np.random.default_rng(0).integers(0, L, size=n)
    clusters[:L] = np.arange(L)
    op_ref, pnm_ref = go.landmark_operator(K, clusters)
    labels = _dev(clusters.astype(np.int32))
    Kd = pipeline.DeviceCSR(*_csr_dev(K), K.shape)
    outs = []
    for _ in range(3):
        pnm, pnm_norm, colsum = lm.aggregate_by_cluster(Kd, labels, L, want_colsum=True)
        op = lm.landmark_operator(pnm, pnm_norm, colsum, n, L)
        outs.append((op.cpu().numpy(), colsum.cpu().numpy(), pnm.to_scipy(pnm_norm)))
    for o in outs[1:]:
        assert np.array_equal(o[0], outs[0][0]) and np.array_equal(o[1], outs[0][1])
    assert np.allclose(outs[0][0], op_ref, rtol=1e-10, atol=0)
    T = outs[0][2]
    pnm_ref = pnm_ref.tocsr(); pnm_ref.sort_indices()
    assert np.array_equal(T.indptr, pnm_ref.indptr) and np.array_equal(T.indices, pnm_ref.indices)
    assert np.allclose(T.data, pnm_ref.data, rtol=1e-12, atol=0)
