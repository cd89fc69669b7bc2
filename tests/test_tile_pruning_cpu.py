"""Host logic of the pruned one-product sweep: when it is tried, when its tile lists are used, and the per-unit bound."""
import math

import pytest
import torch

from graphtools_b200 import pipeline


def _plan(want="auto", n_pad=100_000 // 128 * 128 + 128, metric="euclidean", d=100):
    return pipeline.plan_search(want, d, n_pad, metric, 6, 0, False)


@pytest.mark.parametrize("want,n_pad,metric,expect", [
    ("auto", 1_000_064, "euclidean", True),
    ("auto", 1_000_064, "sqeuclidean", True),
    ("auto", 1_000_064, "cosine", False),            # normalised search copy: its rounding is outside the bound
    ("auto", 1_000_064, "correlation", False),
    ("auto", 1_000_064, "cityblock", False),         # no tensor-core sweep
    ("tch", 1_000_064, "euclidean", False),          # two-product flavour: no seeds
    ("tch1", 20_096, "euclidean", False),            # too few tiles for a seed sample: unseeded
])
def test_prunable(want, n_pad, metric, expect):
    assert pipeline.prunable(_plan(want, n_pad, metric), metric) is expect


def test_use_tile_lists():
    assert pipeline.use_tile_lists(10, 100)
    assert pipeline.use_tile_lists(50, 100)
    assert not pipeline.use_tile_lists(51, 100)
    assert not pipeline.use_tile_lists(100, 100)        # every unit lists everything: the plain sweep
    assert not pipeline.use_tile_lists(0, 0)


def test_unit_bounds_hand_case():
    # three rows, units of two rows: unit 0 = rows 0, 1; unit 1 = row 2 and one padding row; unit 2 = padding only
    s2 = 4.0                                              # fp16 scale 2: seeds are in scaled units
    seed = torch.tensor([[8.0, 8.0], [40.0, 40.0], [math.inf, math.inf]])
    qn2 = torch.tensor([1.0, 3.0, 2.0])
    eps, maxnorm = 2.0 ** -10, 5.0
    ub = pipeline.unit_bounds(seed, qn2, eps, maxnorm, s2, 2, 3)
    e = eps + 2.0 ** -20
    assert ub.dtype == torch.float64 and ub.shape == (3,)
    assert ub[0].item() == max(2.0 + e * 6.0, 10.0 + e * 8.0)
    assert ub[1].item() == math.inf                      # a row without a seed reaches every tile
    assert ub[2].item() == -math.inf                     # no rows: nothing to visit


def test_unit_bounds_cover_every_row():
    g = torch.Generator().manual_seed(0)
    seed = torch.rand((1000, 2), generator=g) * 100
    qn2 = torch.rand((1000,), generator=g) * 50
    ub = pipeline.unit_bounds(seed, qn2, 2.0 ** -10, 60.0, 1.0, 128, 8)
    t = seed[:, 0].double() + (2.0 ** -10 + 2.0 ** -20) * (qn2.double() + 60.0)
    for u in range(8):
        assert ub[u].item() == t[u * 128:(u + 1) * 128].max().item()
