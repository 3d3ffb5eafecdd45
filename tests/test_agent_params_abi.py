"""Per-env tester parameters without a GPU: the C-ABI symbol, its NULL-engine refusal, and the sweep module's point layout
and grouping of drained episode rows (cavgym_b200.sweep)."""
import numpy as np
import pytest

from cavgym_b200 import _abi, _native, sweep

ROW = np.dtype([("env", "<i8"), ("episode", "<i4"), ("timesteps", "<i4"), ("winner", "<i4"), ("liveness_sum", "<i4")])


def test_symbol_is_exported_and_mirrored():
    lib = _native.load()
    assert hasattr(lib, "cavgym_set_agent_params")
    assert "cavgym_set_agent_params" in _abi.PROTOTYPES


def test_null_engine_is_refused():
    lib = _native.load()
    assert lib.cavgym_set_agent_params(None, None, None, None) == -22
    assert b"NULL" in lib.cavgym_last_error()


def test_point_layout_is_contiguous_blocks():
    assert sweep.point_slices(3, 5) == [(0, 5), (5, 10), (10, 15)]
    assert sweep.point_slices(1, 7) == [(0, 7)]


def rows_of(envs, winners, timesteps, liveness):
    rows = np.zeros(len(envs), dtype=ROW)
    rows["env"], rows["winner"], rows["timesteps"], rows["liveness_sum"] = envs, winners, timesteps, liveness
    rows["episode"] = 1
    return rows


@pytest.mark.parametrize("offset", [0, 1 << 20])
def test_rows_are_grouped_by_point_after_the_shard_offset(offset):
    rng = np.random.default_rng(3)
    n_p, k = 6, 3
    envs = rng.permutation(np.repeat(np.arange(k * n_p), 2)) + offset
    rows = rows_of(envs, rng.integers(-1, 3, envs.size), rng.integers(1, 100, envs.size), rng.integers(0, 50, envs.size))
    groups = sweep.group_rows(rows, k, n_p, env_offset=offset)
    assert [g.size for g in groups] == [2 * n_p] * k
    for p, group in enumerate(groups):
        assert np.all((group["env"] - offset) // n_p == p)
        order = np.nonzero((rows["env"] - offset) // n_p == p)[0]
        assert np.array_equal(group, rows[order])     # drain order kept within a point
    with pytest.raises(ValueError):
        sweep.group_rows(rows, k, n_p, env_offset=offset + 1)


def test_point_summary_counts_and_intervals():
    rows = rows_of([0, 1, 2, 3, 4], [1, -1, 2, 0, 1], [10, 900, 20, 30, 40], [5, 0, 7, 0, 9])
    result = sweep.summarise(rows, "epsilon", 0.5, 2.0)
    assert (result.episodes, result.interesting, result.env_steps) == (5, 3, 1000)
    from cavgym_b200 import reporting
    assert tuple(result.confidence_timesteps) == tuple(reporting.confidence_interval([10, 20, 40]))
    assert tuple(result.confidence_score) == tuple(reporting.confidence_interval([-5, -7, -9]))
    assert result.to_data()["device_seconds"] == 2.0
