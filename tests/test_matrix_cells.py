"""The (body count, scenario family) matrix of the thread-per-env kernels on the CPU: the builder gives every cell the family
it claims (engine.cu::convert's homogeneous rule, restated), and the C oracle runs every cell and ends episodes in the
windows the GPU tests use."""
import pytest

from helpers import (FAMILIES, MATRIX_M, compile_from_meta, expect_homogeneous, has_pedestrian, load_golden,
                     matrix_scenario)


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_homogeneous_rule_on_the_stock_scenarios(dtype):
    for name, homogeneous in (("pedestrians_rc_seed0", True), ("pedestrians3_rc_seed2", True),
                              ("crossroads_random_all_seed6", False), ("busstop_random_all_seed8", False),
                              ("pelican_random_all_seed10", False)):
        meta, _ = load_golden(name)
        assert expect_homogeneous(compile_from_meta(meta), dtype) == homogeneous, name


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("mode", ["external", "device"])
def test_every_matrix_cell_is_the_family_it_claims(mode, dtype):
    for family in FAMILIES:
        for m in MATRIX_M:
            comp = matrix_scenario(m, family, mode)
            assert comp.n_bodies == m and len(comp.is_car) == m
            assert expect_homogeneous(comp, dtype) == (family == "homogeneous"), (m, family)
            assert has_pedestrian(m, family) == any("Pedestrian" in c for c in comp.body_classes[1:]), (m, family)


@pytest.mark.parametrize("family", FAMILIES)
def test_the_oracle_runs_every_cell_and_ends_episodes(family):
    """64 envs, max_timesteps 60, 100 auto-reset steps with on-device agents: episodes end and restart inside the window
    (at least one per env), and few steps are flagged."""
    from oracle.oracle import Oracle
    for m in MATRIX_M:
        oracle = Oracle(matrix_scenario(m, family, "device", max_timesteps=60), 64, seed=3, threads=4)
        oracle.reset()
        oracle.rollout(100, auto_reset=True)
        stats = oracle.stats()
        assert stats["env_steps"] == 6400 and stats["episodes"] >= 64, (m, stats)
        assert stats["tangent"] <= 0.01 * stats["env_steps"], (m, stats)
