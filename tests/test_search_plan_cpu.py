"""The kNN search plan (pipeline.plan_search): which flavour GTB_SEARCH_IMPL selects for a shape, and the list shapes
it sweeps with.  Pure host logic: no device, no library."""
import pytest

from graphtools_b200 import pipeline

SEEDED, UNSEEDED = 65536, 65408          # padded reference rows: 512 tiles (32 sampled at stride 16) and 511


def plan(want="auto", d=100, n_pad=SEEDED, metric="euclidean", knn=5, kmax=0, binary=False):
    return pipeline.plan_search(want, d, n_pad, metric, knn, kmax, binary)


@pytest.mark.parametrize("want,d,impl", [
    # a flavour fits while its operand row stays within the resident query tile
    ("tc", 103, "tc"), ("tc", 104, "tc16"),
    ("tch1", 126, "tch1"), ("tch1", 127, "tch"),
    ("tc16", 127, "tc16"), ("tc16", 128, "simt"),
    ("tch", 510, "tch"), ("tch", 511, "simt"),
])
def test_fit_boundaries(want, d, impl):
    assert plan(want, d).impl == impl


@pytest.mark.parametrize("want,n_pad,d,knn,impl", [
    ("auto", SEEDED, 100, 5, "tch1"), ("auto", SEEDED, 127, 5, "tch"), ("auto", SEEDED, 511, 5, "simt"),
    ("auto", SEEDED, 127, 25, "simt"), ("auto", SEEDED, 100, 56, "tch1"), ("auto", SEEDED, 100, 57, "simt"),
    # auto without a seed sweep: the one-product flavour only when its list of 64 is needed
    ("auto", UNSEEDED, 100, 5, "tch"), ("auto", UNSEEDED, 100, 24, "tch"), ("auto", UNSEEDED, 100, 25, "tch1"),
    ("auto", UNSEEDED, 511, 5, "simt"),
    ("tch1", UNSEEDED, 100, 5, "tch1"), ("tch1", SEEDED, 127, 5, "tch"), ("tch1", SEEDED, 511, 5, "simt"),
    ("tch1", SEEDED, 127, 25, "simt"), ("tch1", SEEDED, 100, 56, "tch1"), ("tch1", SEEDED, 100, 57, "simt"),
    ("tch", SEEDED, 100, 24, "tch"), ("tch", SEEDED, 100, 25, "simt"), ("tch", SEEDED, 128, 5, "tch"),
    ("tc16", SEEDED, 20, 5, "tc16"), ("tc16", SEEDED, 100, 25, "simt"),
    ("tc", SEEDED, 20, 24, "tc"), ("tc", SEEDED, 20, 25, "simt"), ("tc", SEEDED, 127, 5, "tc16"),
    ("tc", SEEDED, 128, 5, "simt"),
    ("simt", SEEDED, 20, 5, "simt"), ("simt", SEEDED, 100, 56, "simt"),
])
def test_fallback_chain(want, n_pad, d, knn, impl):
    assert plan(want, d, n_pad, knn=knn).impl == impl


@pytest.mark.parametrize("want,n_pad,impl,seeded", [
    ("tch1", UNSEEDED, "tch1", False), ("tch1", SEEDED, "tch1", True),
    ("auto", UNSEEDED, "tch", False), ("auto", SEEDED, "tch1", True),
    ("tch", SEEDED, "tch", False),
])
def test_seed_sweep(want, n_pad, impl, seeded):
    p = plan(want, 100, n_pad)
    assert (p.impl, p.seeded) == (impl, seeded)


@pytest.mark.parametrize("want,d,knn,kmax,binary,expected", [
    # short lists of 16 while knn (and knn_max) + 8 fit them; two lists per row, one threshold each
    ("tc", 100, 8, 0, False, ("tc", 16, 1, 32, 2, False)),
    ("tc", 100, 9, 0, False, ("tc", 32, 1, 64, 2, False)),
    ("tc", 100, 5, 9, False, ("tc", 32, 1, 64, 2, False)),
    ("tc16", 100, 5, 0, True, ("tc16", 16, 1, 32, 2, False)),
    # fp16x2 with rows of 8 k-steps: two query tiles per CTA sharing one list of 32 per row
    ("tch", 100, 5, 0, False, ("tch", 16, 2, 32, 2, False)),
    ("tch", 126, 24, 0, False, ("tch", 16, 2, 32, 2, False)),
    ("tch", 100, 5, 25, False, ("tch", 32, 1, 64, 2, False)),
    # wide rows (Kp > 128): one query tile, the short-list rule of the other flavours
    ("tch", 127, 8, 0, False, ("tch", 16, 1, 32, 2, False)),
    ("tch", 300, 9, 0, False, ("tch", 32, 1, 64, 2, False)),
    # one product: one list of 64 per row, two query tiles, whatever knn
    ("tch1", 100, 5, 0, False, ("tch1", 32, 2, 64, 2, True)),
    ("tch1", 100, 56, 200, True, ("tch1", 32, 2, 64, 2, True)),
    # CUDA cores: choose_S's list, one threshold per row
    ("simt", 100, 5, 0, False, ("simt", None, None, 48, 1, False)),
    ("simt", 100, 5, 0, True, ("simt", None, None, 16, 1, False)),
    ("simt", 100, 41, 0, False, ("simt", None, None, 64, 1, False)),
    ("simt", 100, 120, 0, False, ("simt", None, None, 128, 1, False)),
    ("auto", 600, 124, 200, True, ("simt", None, None, 128, 1, False)),
])
def test_list_shapes(want, d, knn, kmax, binary, expected):
    assert tuple(plan(want, d, knn=knn, kmax=kmax, binary=binary)) == expected


@pytest.mark.parametrize("want", ["auto", "tc", "tch1", "simt", "unknown"])
def test_cityblock_is_simt(want):
    assert tuple(plan(want, 20, metric="cityblock")) == ("simt", None, None, 48, 1, False)


@pytest.mark.parametrize("metric", ["euclidean", "cosine", "sqeuclidean", "correlation"])
def test_gemm_metrics_use_tensor_cores(metric):
    assert plan("auto", 20, metric=metric).impl == "tch1"


def test_unknown_impl():
    with pytest.raises(ValueError, match="GTB_SEARCH_IMPL"):
        plan("tf32")


@pytest.mark.parametrize("knn,binary", [(121, False), (125, True)])
def test_list_longer_than_128(knn, binary):
    with pytest.raises(NotImplementedError, match="longer than 128"):
        plan("auto", 600, knn=knn, binary=binary)
