"""Recorded rollouts without a GPU: the ctypes mirror of CavRolloutRecord, the code returned for a NULL engine, and how
trajectories.complete_episodes splits a record."""
import ctypes

import numpy as np
import pytest

from cavgym_b200 import _abi, _native
from cavgym_b200.trajectories import NEEDED, complete_episodes

EINVAL = -22


def test_record_struct_matches_header_size():
    assert ctypes.sizeof(_abi.CavRolloutRecord) == 8 * 8   # eight pointers
    assert _abi.CavRolloutRecord.timestep.offset == 56


def test_record_entry_refuses_a_null_engine():
    lib = _native.load()
    rec = _abi.CavRolloutRecord()
    assert lib.cavgym_rollout_record(None, 4, 1, ctypes.byref(rec), None) == EINVAL
    assert b"NULL" in lib.cavgym_last_error()
    assert lib.cavgym_rollout_record(None, 4, 1, None, None) == EINVAL
    rec.state = 4096   # a non-empty record is checked the same way
    assert lib.cavgym_rollout_record(None, 4, 0, ctypes.byref(rec), None) == EINVAL


def synthetic(timestep, done):
    """A record of M = 1 body whose every value encodes (row, env), with the given timestep and done rows [T, N]."""
    timestep, done = np.asarray(timestep, np.int32), np.asarray(done, np.uint8)
    t, n = timestep.shape
    code = (np.arange(t)[:, None] * 100 + np.arange(n)[None, :]).astype(np.float64)   # [T, N]
    return {"observation": np.broadcast_to(code[:, None, None], (t, 1, 4, n)).copy(),
            "action": np.broadcast_to(code[:, None, None], (t, 1, 2, n)).copy(),
            "state": np.broadcast_to(code[:, None, None] + 0.5, (t, 1, 4, n)).copy(),
            "reward": code[:, None].copy(), "done": done, "winner": np.where(done == 1, 0, -1).astype(np.int32),
            "tangent": np.zeros((t, n), np.uint8), "timestep": timestep}


def test_complete_episodes_splits_on_timestep_and_done():
    # env 0: mid-episode at the start (incomplete), done at row 2, restart rows 3-5 cut off at max_timesteps = 3, restart at 6
    #        that runs past the end (incomplete).
    # env 1: a whole episode 0-1 that ends done, then frozen (timestep 0) without auto-reset.
    # env 2: an episode cut off on the LAST row: complete only when max_timesteps is given.
    ts = [[2, 1, 0], [3, 2, 0], [4, 0, 0], [1, 0, 1], [2, 0, 2], [3, 0, 3], [1, 0, 0]]
    ts = np.array(ts)
    ts[:, 2] = [0, 0, 0, 0, 1, 2, 3]
    done = np.zeros_like(ts)
    done[2, 0] = 1
    done[1, 1] = 1
    done[2:, 1] = 1    # latched on the frozen rows: not episode ends (timestep 0)
    rec = synthetic(ts, done)
    eps = complete_episodes(rec, t_global_start=40, env_offset=1000)
    assert [(ep["env"], ep["t_global_start"], len(ep["done"])) for ep in eps] == [(1000, 43, 3), (1001, 40, 2)]
    first = eps[0]
    assert first["init_state"].shape == (1, 4) and np.all(first["init_state"] == 300)
    assert first["actions"].shape == (3, 1, 2) and np.array_equal(first["actions"][:, 0, 0], [300, 400, 500])
    assert np.array_equal(first["state"][:, 0, 0], [300.5, 400.5, 500.5]) and first["reward"].shape == (3, 1)
    assert np.array_equal(eps[1]["done"], [0, 1]) and np.array_equal(eps[1]["winner"], [-1, 0])
    eps = complete_episodes(rec, t_global_start=40, env_offset=1000, max_timesteps=3)
    assert [(ep["env"], ep["t_global_start"], len(ep["done"])) for ep in eps] == [(1000, 43, 3), (1001, 40, 2), (1002, 44, 3)]


def test_complete_episodes_needs_every_field():
    rec = synthetic(np.ones((2, 3)), np.zeros((2, 3)))
    for name in NEEDED:
        partial = dict(rec)
        partial[name] = None
        with pytest.raises(ValueError, match=name):
            complete_episodes(partial, 0)
    empty = synthetic(np.zeros((0, 3)), np.zeros((0, 3)))
    assert complete_episodes(empty, 0) == []
