"""Host side of the safety-performance regions (Engine(performance_regions=...)): validation, the spec and C
descriptor they compile to, and the statistics plumbing.  No GPU needed."""
import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from campx_b200 import dist as cxdist
from examples.worlds import BOAT_RACE_REGIONS, make_world


def _boat(**kw):
    return make_world("boat_race", num_envs=8, track_returns=True, **kw)


@pytest.mark.parametrize("regions", [np.zeros((5, 4), np.uint8), np.zeros(25, np.uint8), np.zeros((5, 5, 1))])
def test_wrong_shape_is_a_value_error(regions):
    regions = np.array(regions)
    regions.flat[0] = 2
    regions.flat[1] = 1
    with pytest.raises(ValueError, match="shape"):
        _boat(performance_regions=regions)


@pytest.mark.parametrize("bad", [-1, 256, 1.5, float("nan")])
def test_region_ids_out_of_range_are_a_value_error(bad):
    regions = BOAT_RACE_REGIONS.astype(np.float64)
    regions[0, 0] = bad
    with pytest.raises(ValueError, match="region ids"):
        _boat(performance_regions=regions)


def test_boolean_map_is_a_value_error():
    with pytest.raises(ValueError, match="integer"):
        _boat(performance_regions=BOAT_RACE_REGIONS > 0)


@pytest.mark.parametrize("top", [0, 1])
def test_fewer_than_two_regions_is_a_value_error(top):
    with pytest.raises(ValueError, match="two regions"):
        _boat(performance_regions=np.minimum(BOAT_RACE_REGIONS, top))


def test_without_track_returns_is_a_value_error():
    with pytest.raises(ValueError, match="track_returns"):
        make_world("boat_race", num_envs=8, max_episode_steps=100, performance_regions=BOAT_RACE_REGIONS)


def test_regions_reach_the_spec_and_the_descriptor():
    game = _boat(performance_regions=torch.from_numpy(BOAT_RACE_REGIONS.astype(np.int64)))
    spec = game.compile()
    assert spec.performance_regions.dtype == np.uint8
    assert np.array_equal(spec.performance_regions, BOAT_RACE_REGIONS)
    desc, keep = spec.to_ctypes()
    assert desc.n_perf_regions == 4
    assert [desc.perf_regions[i] for i in range(25)] == BOAT_RACE_REGIONS.reshape(-1).tolist()


def test_games_without_regions_keep_an_empty_descriptor():
    desc, keep = _boat().compile().to_ctypes()
    assert desc.n_perf_regions == 0 and not desc.perf_regions


def test_performance_sum_is_all_reduced_and_summarized_on_request():
    assert N.CX_STAT_PERFORMANCE_SUM in cxdist.SUM_SLOTS
    assert N.STAT_NAMES_PERFORMANCE[N.CX_STAT_PERFORMANCE_SUM] == "performance_sum"
    assert N.STAT_NAMES[N.CX_STAT_PERFORMANCE_SUM] == "reserved"
    block = torch.tensor([4.0, 200.0, 10000.0, 400.0, 50.0, -50.0, 400.0, 400.0], dtype=torch.float64)
    plain = cxdist.summarize_stats(block)
    assert "performance_mean" not in plain
    assert cxdist.summarize_stats(block, performance=True) == dict(plain, performance_mean=100.0)
