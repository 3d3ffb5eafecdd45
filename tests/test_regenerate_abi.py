"""Episode regeneration without a GPU: the C-ABI symbol and its ctypes mirror, the NULL-engine refusal, the Python-side
validation of BatchedCAVEnv.regenerate, and the start-step bookkeeping of the sweep and of BatchedSimulation."""
import ctypes as C
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

from cavgym_b200 import _abi, _native, sweep
from cavgym_b200.engine import BatchedCAVEnv
from cavgym_b200.simulation import BatchedSimulation
from helpers import matrix_scenario

ROW = np.dtype([("env", "<i8"), ("episode", "<i4"), ("timesteps", "<i4"), ("winner", "<i4"), ("liveness_sum", "<i4")])
CAV_EINVAL, CAV_ESTATE = -22, -1   # include/cavgym.h
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "cavgym.h")


def test_symbol_is_exported_and_mirrored():
    lib = _native.load()
    assert hasattr(lib, "cavgym_regenerate_episodes")
    restype, argtypes = _abi.PROTOTYPES["cavgym_regenerate_episodes"]
    text = open(HEADER, encoding="utf-8").read()
    decl = re.search(r"int cavgym_regenerate_episodes\(([^)]*)\);", text)
    assert decl is not None
    params = [p.strip() for p in decl.group(1).split(",")]
    assert restype is C.c_int and len(argtypes) == len(params) == 6
    assert params[3].startswith("int ") and argtypes[3] is C.c_int
    assert params[4].startswith("const CavRolloutRecord*") and argtypes[4] == C.POINTER(_abi.CavRolloutRecord)


def test_null_engine_is_refused():
    lib = _native.load()
    assert lib.cavgym_regenerate_episodes(None, None, None, 10, None, None) == CAV_EINVAL
    assert b"NULL" in lib.cavgym_last_error()


def offline_env():
    """A BatchedCAVEnv without an engine: any call into the library would fail, so what raises ValueError is Python's check."""
    env = BatchedCAVEnv.__new__(BatchedCAVEnv)
    env._lib, env._handle = None, None
    env.compiled = matrix_scenario(2, "homogeneous", "device", max_timesteps=23)
    env.num_bodies, env.num_envs = env.compiled.n_bodies, 8
    env._agent_params = (None, None)
    return env


@pytest.mark.parametrize("rows, kwargs", [
    (np.zeros(2, dtype=[("env", "<i8")]), {}),
    (np.zeros(2), {}),
    (np.array([(-1, 1, 0, 0, 0)], dtype=ROW), {}),
    (np.array([(1 << 40, 1, 0, 0, 0)], dtype=ROW), {}),
    (np.array([(3, -1, 0, 0, 0)], dtype=ROW), {}),
    (np.array([(3, 1, 0, 0, 0)], dtype=ROW), {"n_steps": -1}),
    (np.array([(3, 1, 0, 0, 0)], dtype=ROW), {"t_global_start": -5}),
    (np.array([(3, 1, 0, 0, 0)], dtype=ROW), {"record": ("state", "velocity")}),
], ids=["no_episode_field", "not_structured", "negative_env", "env_over_40_bits", "negative_episode", "negative_steps",
        "negative_start", "unknown_field"])
def test_regenerate_validates_before_any_call(rows, kwargs):
    with pytest.raises(ValueError):
        offline_env().regenerate(rows, **kwargs)


def test_sweep_rows_carry_their_round_and_its_start_step():
    rows = np.zeros(5, dtype=ROW)
    rows["env"], rows["winner"] = np.arange(5), [1, -1, 2, 0, 1]
    tagged = sweep.with_round(rows, 3)
    assert tagged.dtype.names == ROW.names + ("round",)
    assert np.array_equal(tagged[list(ROW.names)], rows) and (tagged["round"] == 3).all()
    both = np.concatenate([sweep.with_round(rows, 0), tagged])
    assert sweep.start_steps(both, 23).tolist() == [0] * 5 + [69] * 5
    assert sweep.interesting_rows(both, 4)["env"].tolist() == [0, 2, 4, 0]
    assert sweep.interesting_rows(both, 4)["round"].tolist() == [0, 0, 0, 3]
    grouped = sweep.group_rows(both, 5, 1)
    assert all(g["round"].tolist() == [0, 3] for g in grouped)


def test_auto_reset_runs_start_each_episode_after_the_last_one_ended():
    sim = BatchedSimulation.__new__(BatchedSimulation)
    sim.env = SimpleNamespace(num_envs=3, env_offset=100)
    sim.save_interesting, sim._hits = 10, []

    def drain(*entries):   # (env slot, episode, timesteps, winner), in any order within a drain
        rows = np.zeros(len(entries), dtype=ROW)
        for i, (e, episode, t, w) in enumerate(entries):
            rows[i] = (100 + e, episode, t, w, 0)
        sim._note_interesting(rows, 0)

    drain((1, 2, 4, 1), (0, 1, 5, -1), (1, 1, 7, -1), (2, 1, 3, 2))
    drain((0, 2, 6, 1), (2, 2, 9, -1), (1, 3, 2, 1))
    hits = np.concatenate([h for h, _ in sim._hits])
    starts = np.concatenate([s for _, s in sim._hits])
    found = {(int(r["env"]) - 100, int(r["episode"])): int(s) for r, s in zip(hits, starts)}
    assert found == {(1, 2): 7, (2, 1): 0, (0, 2): 5, (1, 3): 11}
    assert hits["env"].tolist()[:2] == [101, 102]   # drain order is kept
    with pytest.raises(RuntimeError):
        sim._note_interesting(np.zeros(0, dtype=ROW), 1)
