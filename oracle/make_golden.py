"""Generate tests/golden/*.npz from the UNMODIFIED reference (run in the build container).

    python -m oracle.make_golden

Each file holds the float32 input (except sklearn digits, which ships with sklearn), the
constructor parameters (JSON) and the reference's outputs.  Test infrastructure only.
"""
import json
import os
import sys
import warnings

import numpy as np
from scipy import sparse

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from graphtools_b200 import synth  # noqa: E402
from oracle.refload import load_reference  # noqa: E402
from tests.golden_util import GOLDEN_THREADS  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def pack(prefix, M, out):
    if sparse.issparse(M):
        M = sparse.csr_matrix(M)
        M.sort_indices()
        out[prefix + "_data"] = M.data
        out[prefix + "_indices"] = M.indices
        out[prefix + "_indptr"] = M.indptr
        out[prefix + "_shape"] = np.array(M.shape)
    else:
        out[prefix + "_dense"] = np.asarray(M)


def digits(n=None):
    from sklearn.datasets import load_digits
    return load_digits().data.astype(np.float32)[:n]


def cases():
    iso, _ = synth.gaussian_mixture(1500, 20, n_clusters=3, intrinsic_dim=None, seed=5)
    mix, _ = synth.gaussian_mixture(3000, 100, n_clusters=8, intrinsic_dim=10, seed=0)
    small, _ = synth.gaussian_mixture(600, 50, n_clusters=4, intrinsic_dim=10, seed=1)
    mnnX, mnn_idx = synth.batched_mixture(300, 4, 20, n_clusters=3, intrinsic_dim=5, seed=2)
    # interleave the batches so block placement is non-trivial
    perm = np.random.default_rng(9).permutation(len(mnn_idx))
    mnnX, mnn_idx = np.ascontiguousarray(mnnX[perm]), mnn_idx[perm]
    Yq, _ = synth.gaussian_mixture(257, 100, n_clusters=8, intrinsic_dim=10, seed=0)
    Yq = np.ascontiguousarray(Yq + np.float32(0.01))
    c = {}
    c["digits_knn5_decay40"] = dict(X="digits", params=dict(knn=5, decay=40))
    c["digits_knnmax10"] = dict(X="digits700", params=dict(knn=5, decay=40, knn_max=10))
    c["digits_binary"] = dict(X="digits", params=dict(knn=5, decay=None))
    c["digits_mult"] = dict(X="digits700", params=dict(knn=4, decay=20, kernel_symm="*", thresh=1e-3))
    c["digits_mnnsym"] = dict(X="digits700", params=dict(knn=5, decay=40, kernel_symm="mnn", theta=0.7))
    c["digits_aniso"] = dict(X="digits700", params=dict(knn=5, decay=40, anisotropy=0.5))
    c["digits_fixed_bw"] = dict(X="digits700", params=dict(knn=5, decay=10, bandwidth=18.0,
                                                        bandwidth_scale=1.2))
    c["digits_nosym"] = dict(X="digits700", params=dict(knn=7, decay=15, kernel_symm=None, bandwidth_scale=0.8))
    c["iso_refine"] = dict(X=iso, params=dict(knn=5, decay=40))
    c["iso_knnmax"] = dict(X=iso, params=dict(knn=5, decay=40, knn_max=12))
    c["mix_knn"] = dict(X=mix, params=dict(knn=5, decay=40, thresh=1e-4), Y=Yq)
    c["mix_landmark_random"] = dict(X=mix, X_from="mix_knn", params=dict(knn=5, decay=40, n_landmark=150,
                                                       random_landmarking=True, random_state=42), Y=Yq)
    c["mix_landmark_spectral"] = dict(X=mix, X_from="mix_knn", params=dict(knn=5, decay=40, n_landmark=120, n_svd=50,
                                                         random_state=42))
    c["small_exact"] = dict(X=small, params=dict(knn=5, decay=40, graphtype="exact"), Y=small[:97] + np.float32(0.02))
    c["small_exact_thresh0"] = dict(X=small[:250], params=dict(knn=3, decay=10, thresh=0))
    c["small_exact_fixed_bw"] = dict(X=small, params=dict(knn=5, decay=8, graphtype="exact", bandwidth=6.0,
                                                          kernel_symm="mnn", theta=0.3))
    c["mnn_decay"] = dict(X=mnnX, params=dict(knn=5, decay=40, sample_idx=mnn_idx, kernel_symm="mnn", theta=0.5))
    c["mnn_binary"] = dict(X=mnnX, params=dict(knn=4, decay=None, sample_idx=mnn_idx, kernel_symm="mnn", theta=0.9,
                                                beta=0.5))
    # cosine metric (sklearn brute-force cosine_distances behind knn_tree)
    c["mix_cosine"] = dict(X=mix, X_ref="mix_knn", params=dict(knn=5, decay=40, distance="cosine"), Y=Yq)
    c["digits_cosine_binary"] = dict(X="digits700", params=dict(knn=5, decay=None, distance="cosine"))
    c["iso_cosine_refine"] = dict(X=iso, params=dict(knn=5, decay=20, distance="cosine", thresh=1e-3))
    c["mix_cosine_landmark_random"] = dict(X=mix, X_from="mix_knn", params=dict(
        knn=5, decay=40, distance="cosine", n_landmark=100, random_landmarking=True, random_state=7))
    c["small_exact_cosine"] = dict(X=small, params=dict(knn=5, decay=40, graphtype="exact", distance="cosine"),
                                   Y=small[:97] + np.float32(0.02))
    c["small_exact_cosine_thresh0"] = dict(X=small[:250], params=dict(knn=3, decay=10, thresh=0, distance="cosine",
                                                                      kernel_symm="mnn", theta=0.3))
    # thresh = 0 with a decay: exact (dense) sub-graphs, dense MNN kernel (api.py:207-209, graphs.py:1901-1902)
    c["mnn_thresh0"] = dict(X=mnnX[:480], params=dict(knn=4, decay=12, thresh=0, sample_idx=mnn_idx[:480],
                                                      kernel_symm="mnn", theta=0.6, beta=0.8))
    # cityblock metric (sklearn brute-force manhattan search / scipy pdist "cityblock"; the reference's own landmark
    # tests run it, test/test_landmark.py:195-322)
    c["mix_cityblock"] = dict(X=mix, X_ref="mix_knn", params=dict(knn=5, decay=40, distance="cityblock"), Y=Yq)
    c["mix_cityblock_binary"] = dict(X=mix, X_ref="mix_knn", params=dict(knn=6, decay=None, distance="cityblock"))
    c["iso_cityblock_refine"] = dict(X=iso, params=dict(knn=5, decay=20, distance="cityblock", thresh=1e-3))
    c["mix_cityblock_landmark_random"] = dict(X=mix, X_from="mix_knn", params=dict(
        knn=5, decay=40, distance="cityblock", n_landmark=100, random_landmarking=True, random_state=7))
    c["small_exact_cityblock"] = dict(X=small, params=dict(knn=5, decay=40, graphtype="exact", distance="cityblock"),
                                      Y=small[:97] + np.float32(0.02))
    # float64 input that is NOT float32-exact and carries a large offset: distances must come from the float64 rows
    # on every route (ADVICE r01: the dense route used to round its inputs to float32)
    off = (small.astype(np.float64) * (1.0 + 1e-9) + 1000.0)
    c["small_exact_f64_offset_thresh0"] = dict(X=off[:250], params=dict(knn=3, decay=10, thresh=0), keep64=True)
    c["small_exact_f64_offset"] = dict(X=off, params=dict(knn=5, decay=40, graphtype="exact"), keep64=True,
                                       Y=off[:97] + 0.02)
    return c


def main():
    only = [a for a in sys.argv[1:] if not a.startswith("-")]
    gt = load_reference()
    assert gt is not None, "reference not available"
    import scipy, sklearn
    from threadpoolctl import threadpool_limits
    threadpool_limits(limits=GOLDEN_THREADS, user_api="blas")
    os.makedirs(OUT, exist_ok=True)
    for name, case in cases().items():
        if only and name not in only:
            continue
        X32 = case["X"]
        if isinstance(X32, str):
            X32 = digits(int(X32[6:]) if len(X32) > 6 else None)
        params = dict(case["params"])
        out = {}
        meta = {k: (v if not isinstance(v, np.ndarray) else "array") for k, v in params.items()}
        if "X_from" in case:
            meta["X_from"] = case["X_from"]
        elif "X_ref" in case:
            meta["X_from"] = case["X_ref"]          # same input as another fixture: stored once, outputs stored here
        elif not isinstance(case["X"], str):
            out["X"] = X32
        if "sample_idx" in params:
            out["sample_idx"] = np.asarray(params["sample_idx"])
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            G = gt.Graph(X32.astype(np.float64), n_jobs=GOLDEN_THREADS, verbose=0, **params)   # keep64: already f64
            if "X_from" not in case:
                pack("K", G.kernel, out)
                pack("P", G.diff_op, out)
                # raw (unsymmetrised) kernel
                pack("R", G.build_kernel(), out)
                out["degree"] = np.asarray(G.kernel_degree)
            if "n_landmark" in params:
                out["clusters"] = np.asarray(G.clusters)
                pack("landmark_op", G.landmark_op, out)
                pack("transitions", G.transitions, out)
            if "Y" in case:
                Y32 = np.ascontiguousarray(case["Y"] if case.get("keep64") else case["Y"].astype(np.float32))
                out["Y"] = Y32
                pack("Kyx", G.build_kernel_to_data(Y32.astype(np.float64)), out)
                pack("ext", G.extend_to_data(Y32.astype(np.float64)), out)
        meta["_class"] = type(G).__name__
        meta["_versions"] = dict(numpy=np.__version__, scipy=scipy.__version__, sklearn=sklearn.__version__,
                                 graphtools=gt.__version__)
        out["meta"] = np.array(json.dumps(meta))
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, type(G).__name__, "nnz(K)=%s" % (G.kernel.nnz if sparse.issparse(G.kernel) else G.kernel.size),
              "%.1f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
