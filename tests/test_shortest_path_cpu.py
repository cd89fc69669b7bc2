"""BaseGraph.shortest_path / weighted without a device: argument validation happens before any device work, and
the computation itself raises EngineError (there is no CPU fallback)."""
import numpy as np
import pytest

import graphtools_b200 as gt
from graphtools_b200 import _engine as E


def _X():
    return np.random.default_rng(0).normal(size=(60, 5))


def test_weighted_follows_decay():
    assert gt.Graph(_X(), knn=5, decay=40, initialize=False).weighted
    assert not gt.Graph(_X(), knn=5, decay=None, initialize=False).weighted
    idx = np.arange(60) % 2
    assert gt.Graph(_X(), knn=5, decay=40, sample_idx=idx, initialize=False).weighted
    assert not gt.Graph(_X(), knn=5, decay=None, sample_idx=idx, initialize=False).weighted


def test_distance_validation():
    Gw = gt.Graph(_X(), knn=5, decay=40, initialize=False)
    Gu = gt.Graph(_X(), knn=5, decay=None, initialize=False)
    with pytest.raises(NotImplementedError, match="only implemented for unweighted graphs"):
        Gw.shortest_path(distance="data")
    with pytest.raises(NotImplementedError, match="only implemented for unweighted graphs"):
        Gw.shortest_path(distance="constant")
    with pytest.raises(ValueError, match="only valid for weighted graphs"):
        Gu.shortest_path(distance="affinity")
    for G in (Gw, Gu):
        with pytest.raises(ValueError, match="Expected `distance` in"):
            G.shortest_path(distance="euclidean")
        with pytest.raises(ValueError, match="unrecognized method"):
            G.shortest_path(method="dijkstra")


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    G = gt.Graph(_X(), knn=5, decay=None, initialize=False)
    with pytest.raises(E.EngineError):
        G.shortest_path()
