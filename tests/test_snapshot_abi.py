"""The snapshot entry points of the C-ABI without a GPU: struct sizes of the ctypes mirror and the codes returned for a NULL
engine (every entry checks its engine before it touches the device)."""
import ctypes

from cavgym_b200 import _abi, _native

EINVAL = -22


def test_snapshot_structs_match_header_sizes():
    # four int32, then int64 / uint64 / double fields only: no padding
    assert ctypes.sizeof(_abi.CavSnapshotLayout) == 16 + 8 * 9
    assert ctypes.sizeof(_abi.CavEngineState) == 16 + 3 * 8 + 2 * 8 + 8 + 8 * _abi.CAV_N_STATS
    assert _abi.CavSnapshotLayout.fingerprint.offset == 80 and _abi.CavEngineState.counters.offset == 64


def test_snapshot_entries_refuse_a_null_engine():
    lib = _native.load()
    layout, state = _abi.CavSnapshotLayout(), _abi.CavEngineState()
    assert lib.cavgym_snapshot_layout(None, 4, ctypes.byref(layout)) == EINVAL
    assert b"NULL" in lib.cavgym_last_error()
    assert lib.cavgym_save_envs(None, None, 0, None, None) == EINVAL
    assert lib.cavgym_load_envs(None, None, 0, None, None) == EINVAL
    assert lib.cavgym_fork_envs(None, None, None, 0, None) == EINVAL
    assert lib.cavgym_save_engine(None, ctypes.byref(state)) == EINVAL
    assert lib.cavgym_load_engine(None, ctypes.byref(state)) == EINVAL
    assert lib.cavgym_load_engine(None, None) == EINVAL
