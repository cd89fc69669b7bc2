"""Helpers to read tests/golden/*.npz (written by oracle/make_golden.py)."""
import glob
import json
import os

import numpy as np
from scipy import sparse

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# Thread counts of the reference runs stored here: scikit-learn n_jobs and OpenBLAS threads, both 8.  The
# brute-force cosine search splits the distance product over n_jobs workers and OpenBLAS splits each product over
# its threads; either split moves the last bits of the distances, so the golden values hold for these counts and
# not for the defaults of a host with another core count.  The runs used OpenBLAS's AVX-512 ("SkylakeX") kernels;
# other BLAS kernels round some products differently.
GOLDEN_THREADS = 8


def names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))


class Case:
    def __init__(self, name):
        self.name = name
        self.z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
        self.meta = json.loads(str(self.z["meta"]))
        self.cls = self.meta["_class"]
        self.params = {k: v for k, v in self.meta.items() if not k.startswith("_") and k != "X_from"}
        if "sample_idx" in self.params:
            self.params["sample_idx"] = self.z["sample_idx"]

    @property
    def X(self):
        if "X" in self.z.files:
            return self.z["X"]
        if "X_from" in self.meta:
            return Case(self.meta["X_from"]).X
        from sklearn.datasets import load_digits
        n = 700 if self.name != "digits_knn5_decay40" and self.name != "digits_binary" else None
        return load_digits().data.astype(np.float32)[:n]

    def has(self, prefix):
        return (prefix + "_data") in self.z.files or (prefix + "_dense") in self.z.files

    def mat(self, prefix):
        if (prefix + "_dense") in self.z.files:
            return self.z[prefix + "_dense"]
        return sparse.csr_matrix((self.z[prefix + "_data"], self.z[prefix + "_indices"], self.z[prefix + "_indptr"]),
                                 shape=tuple(self.z[prefix + "_shape"]))


def csr_equal(A, B):
    """Bit-exact equality of two sparse matrices in canonical CSR form."""
    A = sparse.csr_matrix(A); B = sparse.csr_matrix(B)
    A.sum_duplicates(); B.sum_duplicates(); A.sort_indices(); B.sort_indices()
    return (A.shape == B.shape and np.array_equal(A.indptr, B.indptr)
            and np.array_equal(A.indices, B.indices) and np.array_equal(A.data, B.data))
