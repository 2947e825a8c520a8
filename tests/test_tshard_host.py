"""Sample shards without a GPU: the range split of sivo_b200.tshard and the constructor's argument checks, which run after the
prototxt is parsed and before any CUDA call."""
import pytest

from conftest import make_model
from sivo_b200 import BayesianSegNet, BayesianSegNetParams
from sivo_b200 import _lib as L
from sivo_b200.tshard import shard_ranges


@pytest.mark.parametrize("T", [1, 2, 3, 6, 7, 12, 13])
def test_shard_ranges_cover_T_in_balanced_contiguous_order(T):
    for G in range(1, T + 1):
        r = shard_ranges(T, G)
        assert len(r) == G
        assert r[0][0] == 0 and all(a[0] + a[1] == b[0] for a, b in zip(r, r[1:])) and r[-1][0] + r[-1][1] == T
        counts = [c for _, c in r]
        assert min(counts) >= 1 and max(counts) - min(counts) <= 1
        assert counts == sorted(counts, reverse=True)


@pytest.mark.parametrize("T,G", [(6, 0), (6, -1), (6, 7), (1, 2)])
def test_shard_ranges_refuse_empty_shards(T, G):
    with pytest.raises(ValueError):
        shard_ranges(T, G)


def test_shard_ranges_example():
    assert shard_ranges(12, 4) == [(0, 3), (3, 3), (6, 3), (9, 3)]
    assert shard_ranges(6, 4) == [(0, 2), (2, 2), (4, 1), (5, 1)]


@pytest.mark.parametrize("samples", [(-1, 2), (0, 0), (2, -1), (5, 2), (6, 1), (0, 7)])
def test_shard_constructor_refuses_bad_ranges(model_dir, samples):
    _, _, proto, model = make_model(model_dir, "basic", T=6, H=32, W=64, width=8)
    with pytest.raises(ValueError):
        BayesianSegNet(BayesianSegNetParams(proto, model), samples=samples)


def test_shard_constructor_keeps_the_T_rule(model_dir):
    _, _, proto, model = make_model(model_dir, "basic", T=1, H=32, W=64, width=8)
    with pytest.raises(ValueError, match="batch size greater than 1"):
        BayesianSegNet(BayesianSegNetParams(proto, model), samples=(0, 1))


def test_shard_symbols_are_declared():
    syms = L.declared_symbols()
    for s in ("sivo_segnet_create_shard", "sivo_segnet_run_device_partial", "sivo_segnet_finalize_device", "sivo_dbg_mc_partial",
              "sivo_dbg_mc_finalize"):
        assert s in syms
