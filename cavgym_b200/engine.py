"""BatchedCAVEnv — tensor API over N parallel CAV-Gym environments on one B200.

Host side of the drop-in boundary: the same constructor vocabulary as the reference's
`CAVEnv(bodies, constants, env_config, np_random)` (library/environment.py:59) plus
`num_envs / device / dtype / agents`; `reset()` / `step(actions)` exchange torch tensors in the
engine's SoA layout ([M, 4, N] state, [M, 2, N] actions, [M, N] reward, [N] done / winner).
PyTorch is only plumbing here (device memory, streams); every transition runs in the
hand-written CUDA kernels behind the C-ABI of include/cavgym.h, called through ctypes.
"""
import ctypes as C

import numpy as np
import torch

from . import _abi, _native
from .scenario import AgentSpec, compile_scenario

_DTYPES = {"float64": (_abi.CAV_F64, torch.float64), "float32": (_abi.CAV_F32, torch.float32),
           torch.float64: (_abi.CAV_F64, torch.float64), torch.float32: (_abi.CAV_F32, torch.float32)}


class _DeviceArray:
    """Exposes an engine-owned device buffer through __cuda_array_interface__ (zero copy)."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}
        self._owner = owner


def _ptr(tensor):
    return None if tensor is None else C.c_void_p(tensor.data_ptr())


def _is_float32(array):
    return array is not None and (array.dtype == torch.float32 if isinstance(array, torch.Tensor) else getattr(array, "dtype", None) == np.float32)


_REALS = {_abi.CAV_F64: torch.float64, _abi.CAV_F32: torch.float32}
# (name, section, first row, rows per body or None for one row per env) in the order of CavSnapshotLayout's sections
_SECTIONS = (("state", "real", 0, 4), ("action", "real", 4, 2), ("agent", "real", 6, _abi.CAV_AGENT_WORDS),
             ("cs", "real", 6 + _abi.CAV_AGENT_WORDS, 2), ("liveness", "i32", 0, 1), ("t_ep", "i32", 0, None),
             ("episode", "i32", 1, None), ("winner", "i32", 2, None), ("active", "i32", 3, None), ("done", "u8", 0, None),
             ("err", "u8", 1, None))


class EnvSnapshot:
    """Everything the kernels keep for k environments, as one uint8 blob (`data`, on any device) laid out by the engine's
    CavSnapshotLayout (`layout`).  `snap[name]` is a view of one part for inspection: "state" [M,4,K], "action" [M,2,K],
    "agent" [M,5,K], "cs" [M,2,K] (cos/sin of each heading), "liveness" [M,K], "t_ep", "episode", "winner", "active",
    "done", "err" [K].  Loading edited rows is unsupported (the cs rows would no longer match the headings): new states go
    through BatchedCAVEnv.reset(init_state=...)."""

    NAMES = tuple(name for name, *_ in _SECTIONS)

    def __init__(self, data, layout):
        self.data, self.layout = data, layout

    @property
    def k(self):
        return int(self.layout.k)

    @property
    def device(self):
        return self.data.device

    def __getitem__(self, name):
        for key, section, first, per_body in _SECTIONS:
            if key == name:
                break
        else:
            raise KeyError(f"{name!r} is not one of {self.NAMES}")
        lay, m, k = self.layout, int(self.layout.m), self.k
        dtype = {"real": _REALS[lay.dtype], "i32": torch.int32, "u8": torch.uint8}[section]
        offset = {"real": lay.real_offset, "i32": lay.i32_offset, "u8": lay.u8_offset}[section]
        rows = {"real": lay.real_rows, "i32": lay.i32_rows, "u8": lay.u8_rows}[section]
        size = dtype.itemsize
        table = self.data[offset:offset + rows * k * size].view(dtype).view(rows, k)
        if per_body is None:
            return table[first + (m if section == "i32" else 0)]   # the int32 section starts with liveness [M]
        if section == "i32":
            return table[:m]
        return table[first * m:(first + per_body) * m].view(m, per_body, k)

    def to(self, device):
        return EnvSnapshot(self.data.to(device), self.layout)

    def cpu(self):
        return self.to("cpu")


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise RuntimeError("cavgym_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.type != "cuda":
        raise RuntimeError(f"cavgym_b200 runs on CUDA devices only, not {device}")
    return torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())


class BatchedCAVEnv:
    def __init__(self, bodies, constants, env_config, num_envs=1, agents=None, device=None, dtype="float64", seed=0,
                 env_offset=0, compiled=None):
        self._lib = _native.load()
        self.device = _require_cuda(device)
        self.code, self.dtype = _DTYPES[dtype]
        self.bodies, self.constants, self.env_config = bodies, constants, env_config
        self.compiled = compiled if compiled is not None else compile_scenario(bodies, constants, env_config, agents)
        self.num_envs, self.num_bodies = int(num_envs), self.compiled.n_bodies
        self.frequency = 60
        self.time_resolution = 1.0 / self.frequency
        self._handle = C.c_void_p()
        _native.check(self._lib.cavgym_create(self.compiled.pointer(), self.num_envs, self.code, self.device.index,
                                              int(seed), C.byref(self._handle)))
        if env_offset:
            _native.check(self._lib.cavgym_set_shard(self._handle, int(env_offset)))
        self.env_offset = int(env_offset)   # global id of env 0
        n, m = self.num_envs, self.num_bodies
        real = "<f8" if self.code == _abi.CAV_F64 else "<f4"
        self.state = self._view(self._lib.cavgym_state_ptr, (m, 4, n), real)
        self.actions_taken = self._view(self._lib.cavgym_action_ptr, (m, 2, n), real)
        self.agent_state = self._view(self._lib.cavgym_agent_state_ptr, (m, _abi.CAV_AGENT_WORDS, n), real)
        self.episode_liveness = self._view(self._lib.cavgym_liveness_ptr, (m, n), "<i4")
        self.timestep = self._view(self._lib.cavgym_timestep_ptr, (n,), "<i4")
        self.done_latch = self._view(self._lib.cavgym_done_ptr, (n,), "|u1")
        self.winner_latch = self._view(self._lib.cavgym_winner_ptr, (n,), "<i4")
        self.error = self._view(self._lib.cavgym_error_ptr, (n,), "|u1")
        self.reward = torch.zeros((m, n), dtype=self.dtype, device=self.device)
        self.done = torch.zeros(n, dtype=torch.uint8, device=self.device)
        self.winner = torch.full((n,), -1, dtype=torch.int32, device=self.device)
        self.tangent = torch.zeros(n, dtype=torch.uint8, device=self.device)
        self._keep = {}
        self._host_seen = {}
        self._agent_params = (None, None)

    # ---- plumbing ----------------------------------------------------------------------
    def _view(self, getter, shape, typestr):
        return torch.as_tensor(_DeviceArray(getter(self._handle), shape, typestr, self), device=self.device)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _as_real(self, value, shape, name):
        if value is None:
            return None
        tensor = torch.as_tensor(value, dtype=self.dtype, device=self.device).contiguous()
        if tuple(tensor.shape) != tuple(shape):
            raise ValueError(f"{name} must have shape {tuple(shape)}, got {tuple(tensor.shape)}")
        return tensor

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.cavgym_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- reference protocol, batched ------------------------------------------------------
    def reset(self, mask=None, init_state=None):
        """CAVEnv.reset for the envs selected by `mask` (all when None).  `init_state` [M,4,N] replays
        given initial states instead of drawing SpawnPedestrians on the device."""
        n, m = self.num_envs, self.num_bodies
        mask_t = None if mask is None else torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        init_t = self._as_real(init_state, (m, 4, n), "init_state")
        _native.check(self._lib.cavgym_reset(self._handle, _ptr(mask_t), _ptr(init_t), self._stream()))
        return self.state

    def step(self, actions=None, copy_state=None):
        """CAVEnv.step over all envs.  Returns (state, reward, done, winner, tangent) tensors; `state` is the
        engine's own buffer (zero copy) unless `copy_state` is a [M,4,N] tensor to receive a snapshot."""
        n, m = self.num_envs, self.num_bodies
        actions_t = self._as_real(actions, (m, 2, n), "actions")
        if copy_state is not None:   # written by the kernel through a raw pointer: it must be exactly the engine's layout
            if not (isinstance(copy_state, torch.Tensor) and copy_state.device == self.device and copy_state.dtype == self.dtype
                    and tuple(copy_state.shape) == (m, 4, n) and copy_state.is_contiguous()):
                raise ValueError(f"copy_state must be a contiguous {self.dtype} tensor of shape {(m, 4, n)} on {self.device}")
        _native.check(self._lib.cavgym_step(self._handle, _ptr(actions_t), _ptr(copy_state), _ptr(self.reward), _ptr(self.done),
                                            _ptr(self.winner), _ptr(self.tangent), self._stream()))
        return (self.state if copy_state is None else copy_state), self.reward, self.done, self.winner, self.tangent

    # field -> (per-step shape as a function of (M, N), dtype: None = the engine's real type)
    RECORD_FIELDS = {"observation": (lambda m, n: (m, 4, n), None), "action": (lambda m, n: (m, 2, n), None),
                     "state": (lambda m, n: (m, 4, n), None), "reward": (lambda m, n: (m, n), None),
                     "done": (lambda m, n: (n,), torch.uint8), "winner": (lambda m, n: (n,), torch.int32),
                     "tangent": (lambda m, n: (n,), torch.uint8), "timestep": (lambda m, n: (n,), torch.int32)}

    def rollout(self, n_steps, auto_reset=True, record=None):
        """Simulation.run's timestep loop with the on-device agents: n_steps fused transitions per launch.

        record=None returns None.  A tuple of names from RECORD_FIELDS also records those per-step returns and returns them
        as a dict of new device tensors [T, ...] in the engine's layout (see cavgym_rollout_record): "observation" [T,M,4,N]
        (the state the agents saw, after any auto-reset), "action" [T,M,2,N] (the joint action executed), "state" [T,M,4,N]
        (after the step), "reward" [T,M,N], "done" / "tangent" uint8 [T,N], "winner" / "timestep" int32 [T,N].  A row
        where an env did not step has timestep 0.  Recording changes nothing else: the engine state, counters, episode-log
        rows and t_global are those of the same rollout without it.  trajectories.complete_episodes splits a record."""
        n_steps = int(n_steps)
        if record is None:
            _native.check(self._lib.cavgym_rollout(self._handle, n_steps, int(bool(auto_reset)), self._stream()))
            return None
        out, rec = self._record_slabs(n_steps, record)
        _native.check(self._lib.cavgym_rollout_record(self._handle, n_steps, int(bool(auto_reset)), C.byref(rec), self._stream()))
        return out

    def _record_names(self, record):
        names = (record,) if isinstance(record, str) else tuple(record)
        unknown = [name for name in names if name not in self.RECORD_FIELDS]
        if unknown:
            raise ValueError(f"unknown record field(s) {unknown}; choose from {tuple(self.RECORD_FIELDS)}")
        return names

    def _record_slabs(self, n_steps, record):
        """New device slabs [T, ...] for the RECORD_FIELDS named in `record` (checked), and the CavRolloutRecord of them."""
        names = self._record_names(record)
        if n_steps < 0:
            raise ValueError("n_steps must be >= 0")
        m, n = self.num_bodies, self.num_envs
        out = {name: torch.empty((n_steps,) + shape(m, n), dtype=dtype or self.dtype, device=self.device)
               for name, (shape, dtype) in self.RECORD_FIELDS.items() if name in names}
        return out, _abi.CavRolloutRecord(**{name: tensor.data_ptr() for name, tensor in out.items() if tensor.numel()})

    def regenerate_episodes(self, env_ids, episodes, n_steps=None, record=None):
        """cavgym_regenerate_episodes on this engine: slot e becomes episode episodes[e] of global env env_ids[e] (the `env`
        and `episode` of an episode row) and steps n_steps times (default max_timesteps) without auto-reset, drawing from the
        streams of that env and episode, with this engine's per-env tester parameters where set.  The time-out term is
        decided by this engine's t_global (set_global_timestep) at the first step.  `env_ids` / `episodes` hold N values
        each.  Returns what rollout(record=...) returns: None, or a dict of new device slabs [T, ...] whose row 0 is the
        episode's first step.  ValueError, before any call, for a wrong length or an id outside [0, 2^40) or a negative
        episode.  regenerate() is the form that takes drained rows and returns episodes."""
        n = self.num_envs
        ids = torch.as_tensor(np.asarray(env_ids, dtype=np.int64).reshape(-1)).to(self.device).contiguous()
        eps = torch.as_tensor(np.asarray(episodes, dtype=np.int64).reshape(-1)).to(self.device)
        if ids.numel() != n or eps.numel() != n:
            raise ValueError(f"env_ids and episodes must hold {n} values each, got {ids.numel()} and {eps.numel()}")
        if bool(((ids < 0) | (ids >= (1 << 40))).any()) or bool(((eps < 0) | (eps > np.iinfo(np.int32).max)).any()):
            raise ValueError("env ids must be in [0, 2^40) and episode numbers in [0, 2^31)")
        eps = eps.to(torch.int32).contiguous()
        n_steps = self.max_timesteps if n_steps is None else int(n_steps)
        if n_steps < 0:
            raise ValueError("n_steps must be >= 0")
        out, rec = (None, None) if record is None else self._record_slabs(n_steps, record)
        _native.check(self._lib.cavgym_regenerate_episodes(self._handle, _ptr(ids), _ptr(eps), n_steps,
                                                           None if rec is None else C.byref(rec), self._stream()))
        return out

    # share of the free device memory one regenerate() chunk may record into
    REGENERATE_MEMORY_SHARE = 0.25

    def regenerate(self, rows, record=tuple(RECORD_FIELDS), t_global_start=None, n_steps=None):
        """The episodes of `rows` — drained episode rows, or any structured array with `env` and `episode` fields — played
        again on a sibling engine (same compiled scenario, dtype, seed, tau and device, one slot per row) through
        regenerate_episodes, with this engine's per-env tester parameters of each row's slot (env - env_offset) where they are
        set.  This engine is not touched.

        t_global_start: the batch-wide step at each episode's first step (an int, or one per row); only the time-out term
        of the rewards depends on it.  The default, max_timesteps, means "no time-out term", right for every episode that
        started at or after this engine's step max_timesteps.  n_steps (default max_timesteps) bounds each episode.

        Returns one dict per row, in the order of `rows`, in trajectories.complete_episodes' layout for the recorded
        fields: "init_state" [M,4] (from "observation"), "actions" [L,M,2] (from "action"), "state" [L,M,4], "reward" [L,M],
        "done", "winner", "tangent" [L], and "env", "episode", "t_global_start", and "reproduced": whether the regenerated
        (timesteps, winner, liveness_sum) equal the row's (None if `rows` lacks those fields).  An episode not played from a
        reset on the engine's own streams (continued after fork or load_envs, or a salted rollout_until stage) comes back
        with reproduced False; one that has not ended after n_steps has L = n_steps and reproduced False.  Rows are run in
        chunks whose record fits REGENERATE_MEMORY_SHARE of the free device memory."""
        rows = np.asarray(rows)
        if rows.dtype.names is None or "env" not in rows.dtype.names or "episode" not in rows.dtype.names:
            raise ValueError("rows must be a structured array with 'env' and 'episode' fields (drain_episodes())")
        rows = rows.reshape(-1)
        k = rows.size
        env_ids, episodes = rows["env"].astype(np.int64), rows["episode"].astype(np.int64)
        if k and (env_ids.min() < 0 or env_ids.max() >= (1 << 40) or episodes.min() < 0 or episodes.max() > np.iinfo(np.int32).max):
            raise ValueError("rows must have env in [0, 2^40) and episode in [0, 2^31)")
        starts = np.broadcast_to(np.asarray(self.max_timesteps if t_global_start is None else t_global_start, dtype=np.int64), (k,))
        if k and starts.min() < 0:
            raise ValueError("t_global_start must be >= 0")
        n_steps = self.max_timesteps if n_steps is None else int(n_steps)
        if n_steps < 0:
            raise ValueError("n_steps must be >= 0")
        names = self._record_names(record)
        state = self._engine_state()
        slots = env_ids - int(state.shard)
        params = self._agent_params
        if any(p is not None for p in params) and k and (slots.min() < 0 or slots.max() >= self.num_envs):
            raise ValueError(f"per-env tester parameters are set, so every row's env must be one of this engine's "
                             f"[{int(state.shard)}, {int(state.shard) + self.num_envs})")
        check = {"timesteps", "winner", "liveness_sum"} <= set(rows.dtype.names)
        per_step = sum(int(np.prod(shape(self.num_bodies, 1))) * (dtype or self.dtype).itemsize
                       for name, (shape, dtype) in self.RECORD_FIELDS.items() if name in names)
        free = torch.cuda.mem_get_info(self.device)[0]
        chunk = max(1, int(free * self.REGENERATE_MEMORY_SHARE) // max(1, per_step * n_steps))
        episodes_out = [None] * k
        for start in np.unique(starts):
            group = np.flatnonzero(starts == start)
            for lo in range(0, group.size, chunk):
                self._regenerate_chunk(rows, group[lo:lo + chunk], int(start), n_steps, names, state, slots, params, check, episodes_out)
        return episodes_out

    def _regenerate_chunk(self, rows, part, start, n_steps, names, state, slots, params, check, episodes_out):
        sib = BatchedCAVEnv(None, None, None, num_envs=part.size, dtype=self.dtype, compiled=self.compiled, device=self.device,
                            seed=int(state.seed))
        try:
            sib.set_tangent_tolerance(float(state.tau))
            if any(p is not None for p in params):
                index = torch.as_tensor(slots[part], device=self.device)
                sib.set_agent_params(*(None if p is None else p[:, index] for p in params))
            sib.set_episode_log(part.size)
            sib.set_global_timestep(start)
            rec = sib.regenerate_episodes(rows["env"][part], rows["episode"][part], n_steps, names)
            got, _ = sib.drain_episodes()
        finally:
            sib.close()
        rec = {name: tensor.cpu().numpy() for name, tensor in rec.items()}
        found = {(int(r["env"]), int(r["episode"])): r for r in got}
        for slot, i in enumerate(part):
            row = rows[i]
            key = (int(row["env"]), int(row["episode"]))
            mine = found.get(key)
            length = n_steps if mine is None else int(mine["timesteps"])
            episode = {"env": key[0], "episode": key[1], "t_global_start": start}
            if "observation" in rec:
                episode["init_state"] = rec["observation"][0, :, :, slot].copy()
            if "action" in rec:
                episode["actions"] = np.ascontiguousarray(rec["action"][:length, :, :, slot])
            for name in ("state", "reward", "done", "winner", "tangent"):
                if name in rec:
                    episode[name] = np.ascontiguousarray(rec[name][:length, ..., slot])
            episode["reproduced"] = None if not check else (
                mine is not None and all(int(mine[f]) == int(row[f]) for f in ("timesteps", "winner", "liveness_sum")))
            episodes_out[i] = episode

    @property
    def max_timesteps(self):
        """The scenario's episode length (config.json "max_timesteps")."""
        return int(self.compiled.struct.max_timesteps)

    UNTIL_LIVE, UNTIL_PARKED, UNTIL_FINISHED = 0, 1, 2

    def rollout_until(self, n_steps, level, score, salt=0, status=None):
        """rollout(n_steps, auto_reset=False) that parks each env at the first step where its score reaches `level`
        (cavgym_rollout_until): score = running max of the danger (px by which a pedestrian overlaps the ego's reaction
        zone), +inf once a tester wins.  `score` is the caller's contiguous [N] tensor of the engine's dtype on its device,
        read and updated in place.  Returns `status` (uint8 [N], new unless given): UNTIL_LIVE, UNTIL_PARKED (tester wins
        included) or UNTIL_FINISHED.  salt = 0 steps on the engine's random streams; another salt on fresh ones for this call
        only (splitting.py forks envs between calls).  With n_steps = 0 nothing runs and `status` is left as it was."""
        n = self.num_envs
        if not (isinstance(score, torch.Tensor) and score.dtype == self.dtype and tuple(score.shape) == (n,)
                and score.device == self.device and score.is_contiguous()):
            raise ValueError(f"score must be a contiguous {self.dtype} tensor of shape ({n},) on {self.device}")
        if status is None:
            status = torch.zeros(n, dtype=torch.uint8, device=self.device)
        elif not (isinstance(status, torch.Tensor) and status.dtype == torch.uint8 and tuple(status.shape) == (n,)
                  and status.device == self.device and status.is_contiguous()):
            raise ValueError(f"status must be a contiguous uint8 tensor of shape ({n},) on {self.device}")
        _native.check(self._lib.cavgym_rollout_until(self._handle, int(n_steps), float(level), int(salt) % (1 << 64), _ptr(score),
                                                     _ptr(status), self._stream()))
        return status

    # ---- per-env tester parameters -------------------------------------------------------------
    EPSILON_AGENTS = (_abi.CAV_AGENT_RANDOM, _abi.CAV_AGENT_RANDOM_CONSTRAINED)
    THRESHOLD_AGENTS = (_abi.CAV_AGENT_PROXIMITY, _abi.CAV_AGENT_ELECTION)

    def agent_rows(self):
        """(epsilon rows, threshold rows): the bodies whose agent reads row b of set_agent_params' epsilon / threshold."""
        kinds = [int(self.compiled.struct.bodies[b].agent) for b in range(self.num_bodies)]
        return ([b for b, k in enumerate(kinds) if k in self.EPSILON_AGENTS],
                [b for b, k in enumerate(kinds) if k in self.THRESHOLD_AGENTS])

    def set_agent_params(self, epsilon=None, threshold=None):
        """Per-env tester parameters (cavgym_set_agent_params): env e's body b uses epsilon[b, e] instead of its RandomAgent /
        RandomConstrainedAgent epsilon and threshold[b, e] instead of its ProximityAgent / ElectionAgent distance threshold.
        Each is [M, N] of anything convertible (epsilon is kept in float64, threshold in the engine's dtype) or None for the
        scenario's value; both None clears them.  Only the rows of bodies with such an agent are read (agent_rows()); other
        rows may hold anything, NaN included.  ValueError, before any call, for a wrong shape or a read row outside
        epsilon in [0, 1] / threshold > 0 and finite.  The values belong to the env slots: reset, auto-reset, load_envs and
        fork leave them in place.  While they are set, step_host with float32 buffers, rollout_until and the warp-per-env
        path (set_dense_path) refuse to run."""
        m, n = self.num_bodies, self.num_envs
        eps_rows, thr_rows = self.agent_rows()
        eps = None if epsilon is None else torch.as_tensor(epsilon).to(device=self.device, dtype=torch.float64).contiguous()
        thr = None if threshold is None else torch.as_tensor(threshold).to(device=self.device, dtype=self.dtype).contiguous()
        for name, tensor in (("epsilon", eps), ("threshold", thr)):
            if tensor is not None and tuple(tensor.shape) != (m, n):
                raise ValueError(f"{name} must have shape {(m, n)}, got {tuple(tensor.shape)}")
        if eps is not None and eps_rows:
            read = eps[eps_rows]
            if not bool(((read >= 0) & (read <= 1)).all()):
                raise ValueError(f"epsilon must be in [0, 1] in the rows {eps_rows} (bodies with a random agent)")
        if thr is not None and thr_rows:
            read = thr[thr_rows]
            if not bool(((read > 0) & torch.isfinite(read)).all()):
                raise ValueError(f"threshold must be > 0 and finite in the rows {thr_rows} (bodies with a proximity / election agent)")
        _native.check(self._lib.cavgym_set_agent_params(self._handle, _ptr(eps), _ptr(thr), self._stream()))
        self._agent_params = (None if eps is None else eps.clone(), None if thr is None else thr.clone())

    def agent_params(self):
        """(epsilon, threshold) as last set by set_agent_params: [M, N] device tensors, or None where unset."""
        return self._agent_params

    def replay(self, actions, record=("state", "reward", "done", "winner", "tangent")):
        """Replay joint actions [T,M,2,N] in one launch; returns the recorded trajectories as a dict."""
        n, m = self.num_envs, self.num_bodies
        actions_t = torch.as_tensor(actions, dtype=self.dtype, device=self.device).contiguous()
        t = actions_t.shape[0]
        if tuple(actions_t.shape) != (t, m, 2, n):
            raise ValueError(f"actions must have shape (T, {m}, 2, {n})")
        out = {
            "state": torch.empty((t, m, 4, n), dtype=self.dtype, device=self.device) if "state" in record else None,
            "reward": torch.empty((t, m, n), dtype=self.dtype, device=self.device) if "reward" in record else None,
            "done": torch.empty((t, n), dtype=torch.uint8, device=self.device) if "done" in record else None,
            "winner": torch.empty((t, n), dtype=torch.int32, device=self.device) if "winner" in record else None,
            "tangent": torch.empty((t, n), dtype=torch.uint8, device=self.device) if "tangent" in record else None,
        }
        _native.check(self._lib.cavgym_replay(self._handle, t, _ptr(actions_t), _ptr(out["state"]), _ptr(out["reward"]),
                                              _ptr(out["done"]), _ptr(out["winner"]), _ptr(out["tangent"]), self._stream()))
        return out

    _NUMPY = {torch.float64: np.dtype("f8"), torch.float32: np.dtype("f4"), torch.uint8: np.dtype("u1"), torch.int32: np.dtype("i4")}

    def _host_buffer(self, array, shape, dtype, name):
        """Raw host pointer of a numpy array / CPU tensor after checking it is what the kernel will read or write."""
        if array is None:
            return None
        seen = self._host_seen.get(id(array))      # validated before: the cache holds the object, so its id cannot be reused
        if seen is not None and seen[0] is array:
            return seen[1]
        pointer = None
        if isinstance(array, torch.Tensor):
            if array.dtype == dtype and array.shape == shape and array.device.type == "cpu" and array.is_contiguous():
                pointer = array.data_ptr()
        elif isinstance(array, np.ndarray) and array.dtype == self._NUMPY[dtype] and array.shape == shape and array.flags.c_contiguous:
            pointer = array.ctypes.data
        if pointer is not None:
            if len(self._host_seen) > 4096:
                self._host_seen.clear()
            self._host_seen[id(array)] = (array, pointer)
            return pointer
        raise ValueError(f"{name} must be a contiguous host array of shape {tuple(shape)} and dtype {dtype}")

    def replay_host(self, actions, state=None, reward=None, done=None, winner=None, tangent=None, wait=True):
        """cavgym_replay with PINNED HOST tensors: T fused steps in one launch whose kernel reads the joint actions [T,M,2,N]
        from and writes the trajectories ([T,M,4,N] state, [T,M,N] reward, [T,N] done / winner / tangent; each optional) to host
        memory over PCIe — reads of later steps overlap writes of earlier ones, which one cavgym_step_host call per step cannot
        do.  Returns when the results are in the host tensors; with wait=False it returns once the launch is queued on the
        current stream (record an event and wait for that before touching the tensors): consecutive calls then overlap on the
        device tile by tile, the reads of one covering the draining writes of the one before."""
        n, m = self.num_envs, self.num_bodies
        t = int(actions.shape[0])
        wanted = (("actions", actions, (t, m, 2, n), self.dtype), ("state", state, (t, m, 4, n), self.dtype),
                  ("reward", reward, (t, m, n), self.dtype), ("done", done, (t, n), torch.uint8), ("winner", winner, (t, n), torch.int32),
                  ("tangent", tangent, (t, n), torch.uint8))
        pointers = []
        for name, tensor, shape, dtype in wanted:
            if tensor is None:
                pointers.append(None)
                continue
            if not (isinstance(tensor, torch.Tensor) and tensor.device.type == "cpu" and tensor.is_pinned() and tensor.dtype == dtype
                    and tuple(tensor.shape) == shape and tensor.is_contiguous()):
                raise ValueError(f"{name} must be a pinned, contiguous CPU tensor of shape {shape} and dtype {dtype}")
            pointers.append(C.c_void_p(tensor.data_ptr()))
        stream = torch.cuda.current_stream(self.device)
        _native.check(self._lib.cavgym_replay(self._handle, t, *pointers, C.c_void_p(stream.cuda_stream)))
        if wait:
            stream.synchronize()

    def step_host(self, actions, state_out=None, reward_out=None, done_out=None, winner_out=None, tangent_out=None):
        """cavgym_step_host: host buffers in and out (numpy arrays or CPU tensors in the engine's layout).  Pinned buffers
        (tensor.pin_memory()) are read and written by the step kernel itself over PCIe; pageable ones are staged.
        A float64 engine also takes float32 actions / state_out / reward_out (all three the same type): the float32 WIRE
        format of cavgym_step_host_f32 — half the bytes over the link, the engine still steps in double."""
        n, m = self.num_envs, self.num_bodies
        check = self._host_buffer
        real = self.dtype
        if self.dtype == torch.float64 and _is_float32(actions if actions is not None else (state_out if state_out is not None else reward_out)):
            real = torch.float32
        call = self._lib.cavgym_step_host if real == self.dtype else self._lib.cavgym_step_host_f32
        rc = call(self._handle, check(actions, (m, 2, n), real, "actions"), check(state_out, (m, 4, n), real, "state_out"),
                  check(reward_out, (m, n), real, "reward_out"), check(done_out, (n,), torch.uint8, "done_out"),
                  check(winner_out, (n,), torch.int32, "winner_out"), check(tangent_out, (n,), torch.uint8, "tangent_out"))
        if rc:
            _native.check(rc)

    def info(self, polygons=True, road_angles=True):
        """CAVEnv.info() for every env: {'body_polygons': [M, 8, N] (x of the four corners, then y), 'road_angles': [M, N]
        with NaN where the reference returns None}.  Computed on demand by one small kernel."""
        n, m = self.num_envs, self.num_bodies
        out = {"body_polygons": torch.empty((m, 8, n), dtype=self.dtype, device=self.device) if polygons else None,
               "road_angles": torch.empty((m, n), dtype=self.dtype, device=self.device) if road_angles else None}
        _native.check(self._lib.cavgym_info(self._handle, _ptr(out["body_polygons"]), _ptr(out["road_angles"]), self._stream()))
        return out

    # ---- snapshots: save, restore and fork environments; checkpoint the engine ------------------
    # The reference-side equivalent is copy.deepcopy(CAVEnv).  Save, load and fork never touch the counters of stats():
    # an overwritten episode is neither scored nor counted as abandoned, so callers that resample (splitting schemes) keep
    # their own accounting.  An env's random stream is keyed by (global env id, kind, body, episode, t): an env loaded into
    # the slot of the same global id (env_offset + index) continues bit for bit, a copy in another slot continues from the
    # same situation on that slot's own stream.  t_global is batch-wide: a loaded env times out at THIS engine's t_global.
    def _layout(self, k):
        layout = _abi.CavSnapshotLayout()
        _native.check(self._lib.cavgym_snapshot_layout(self._handle, int(k), C.byref(layout)))
        return layout

    def _indices(self, envs, name, unique=False):
        """envs (int, list, array or tensor of env indices) as a contiguous int64 device tensor, checked before any launch."""
        idx = torch.as_tensor(envs, device=self.device)
        if idx.numel() and (idx.dtype == torch.bool or idx.is_floating_point() or idx.is_complex()):   # [] is float32
            raise ValueError(f"{name} must hold integer env indices, not {idx.dtype}")
        idx = idx.reshape(-1).to(torch.int64).contiguous()
        if idx.numel():
            n = self.num_envs
            bad = ((idx < 0) | (idx >= n)).any()
            repeated = torch.zeros((), dtype=torch.bool, device=self.device)
            if unique:   # counted on clamped indices: an out-of-range one is reported as such, never used to index
                counts = torch.zeros(n, dtype=torch.int32, device=self.device)
                counts.index_add_(0, idx.clamp(0, n - 1), torch.ones_like(idx, dtype=torch.int32))
                repeated = counts.max() > 1
            bad, repeated = torch.stack([bad, repeated]).tolist()
            if bad:
                raise ValueError(f"{name}: env index outside [0, {n})")
            if repeated:
                raise ValueError(f"{name}: repeated target env (targets must be unique)")
        return idx

    def save_envs(self, envs=None):
        """EnvSnapshot of the envs listed in `envs` (all, in order, when None) on this engine's device.  Indices may repeat."""
        idx = None if envs is None else self._indices(envs, "envs")
        k = self.num_envs if idx is None else idx.numel()
        layout = self._layout(k)
        data = torch.empty(int(layout.total_bytes), dtype=torch.uint8, device=self.device)
        _native.check(self._lib.cavgym_save_envs(self._handle, _ptr(idx), k, _ptr(data), self._stream()))
        return EnvSnapshot(data, layout)

    def load_envs(self, snapshot, envs=None):
        """Env envs[j] (env j when envs is None) becomes the snapshot's env j.  Targets must be unique.  The snapshot must
        come from an engine of the same scenario, dtype and body count (ValueError otherwise)."""
        if not isinstance(snapshot, EnvSnapshot):
            raise ValueError("snapshot must be an EnvSnapshot (BatchedCAVEnv.save_envs)")
        lay = snapshot.layout
        mine = self._layout(snapshot.k)
        if lay.version != mine.version:
            raise ValueError(f"snapshot of layout version {lay.version}, this engine reads version {mine.version}")
        if lay.fingerprint != mine.fingerprint:
            raise ValueError("snapshot of another scenario (fingerprint differs)")
        if lay.dtype != mine.dtype or lay.m != mine.m:
            raise ValueError(f"snapshot of dtype {_REALS[lay.dtype]} with {lay.m} bodies; this engine: {self.dtype}, {mine.m} bodies")
        if tuple(snapshot.data.shape) != (int(mine.total_bytes),) or snapshot.data.dtype != torch.uint8:
            raise ValueError("snapshot data does not have the size its layout gives")
        idx = None if envs is None else self._indices(envs, "envs", unique=True)
        k = self.num_envs if idx is None else idx.numel()
        if k != snapshot.k:
            raise ValueError(f"snapshot holds {snapshot.k} envs, {k} targets given")
        data = snapshot.data.to(self.device).contiguous()
        if data.data_ptr() % 16:   # the kernels read the snapshot in 8- and 16-byte words
            raise ValueError("snapshot data must start on 16 bytes (a view at an offset is not)")
        _native.check(self._lib.cavgym_load_envs(self._handle, _ptr(idx), k, _ptr(data), self._stream()))

    def fork(self, src, dst):
        """Env dst[j] becomes a copy of env src[j].  Every source is read before any target is written, so src may repeat
        and overlap dst (a population resample); dst must be unique.  A single source is copied into every target.
        All forks of this engine share one staging snapshot: issue them on one stream.  A fork of more envs than any
        before it grows that snapshot and synchronises the device."""
        src_t, dst_t = self._indices(src, "src"), self._indices(dst, "dst", unique=True)
        if src_t.numel() == 1 and dst_t.numel() > 1:
            src_t = src_t.expand(dst_t.numel()).contiguous()
        if src_t.numel() != dst_t.numel():
            raise ValueError(f"src has {src_t.numel()} envs, dst {dst_t.numel()}")
        _native.check(self._lib.cavgym_fork_envs(self._handle, _ptr(src_t), _ptr(dst_t), dst_t.numel(), self._stream()))

    def _engine_state(self):
        state = _abi.CavEngineState()
        _native.check(self._lib.cavgym_save_engine(self._handle, C.byref(state)))
        return state

    def state_dict(self):
        """Checkpoint of the whole engine: every env (as CPU bytes), t_global, the raw counters, seed, shard, tau and the
        scenario fingerprint.  Tensors, ints, floats and strings only (torch.load with weights_only reads it).  The
        episode-log ring is not included: drain it first.  Per-env tester parameters (set_agent_params) are included as
        "agent_epsilon" / "agent_threshold" CPU tensors [M, N] where they are set, and absent otherwise."""
        state = self._engine_state()
        envs = self.save_envs().cpu()
        out = {"version": int(state.version), "dtype": str(self.dtype).replace("torch.", ""), "num_envs": int(state.n),
               "num_bodies": int(state.m), "seed": int(state.seed), "env_offset": int(state.shard), "tau": float(state.tau),
               "t_global": int(state.t_global), "counters": torch.tensor(list(state.counters), dtype=torch.int64),
               "fingerprint": f"{state.fingerprint:016x}", "envs": envs.data}
        for key, value in zip(("agent_epsilon", "agent_threshold"), self._agent_params):
            if value is not None:
                out[key] = value.cpu()
        return out

    def load_state_dict(self, state_dict):
        """Continue a checkpoint of state_dict(): this engine must have the same scenario, dtype, env count, seed and
        env_offset (ValueError otherwise); tau is taken from the checkpoint.  The per-env tester parameters are set from
        the checkpoint's "agent_epsilon" / "agent_threshold", or cleared where it has none, so that it continues bit for bit."""
        sd, mine = state_dict, self._engine_state()
        want = {"version": int(mine.version), "fingerprint": f"{mine.fingerprint:016x}",
                "dtype": str(self.dtype).replace("torch.", ""), "num_envs": int(mine.n), "num_bodies": int(mine.m),
                "seed": int(mine.seed), "env_offset": int(mine.shard)}
        for key, value in want.items():
            if sd.get(key) != value:
                raise ValueError(f"checkpoint {key} is {sd.get(key)!r}, this engine has {value!r}")
        state = _abi.CavEngineState.from_buffer_copy(mine)
        state.t_global, state.tau = int(sd["t_global"]), float(sd["tau"])
        counters = [int(v) for v in torch.as_tensor(sd["counters"]).tolist()]
        if len(counters) != _abi.CAV_N_STATS:
            raise ValueError(f"checkpoint has {len(counters)} counters, not {_abi.CAV_N_STATS}")
        state.counters[:] = counters
        snapshot = EnvSnapshot(torch.as_tensor(sd["envs"]), self._layout(self.num_envs))
        if tuple(snapshot.data.shape) != (int(snapshot.layout.total_bytes),) or snapshot.data.dtype != torch.uint8:
            raise ValueError("checkpoint envs do not have the size this engine's layout gives")
        epsilon, threshold = sd.get("agent_epsilon"), sd.get("agent_threshold")
        self.set_agent_params(epsilon, threshold)   # validated before the engine state is touched
        _native.check(self._lib.cavgym_load_engine(self._handle, C.byref(state)))
        self.load_envs(snapshot)

    # ---- accounting and knobs ------------------------------------------------------------
    def stats(self):
        out = (C.c_int64 * _abi.CAV_N_STATS)()
        _native.check(self._lib.cavgym_stats(self._handle, out))
        return dict(zip(_abi.STAT_NAMES, [int(v) for v in out]))

    def set_episode_log(self, capacity):
        """Keep a device ring of `capacity` per-episode rows (0: off); see drain_episodes."""
        _native.check(self._lib.cavgym_set_episode_log(self._handle, int(capacity)))
        self._episode_capacity = int(capacity)

    def drain_episodes(self):
        """(rows, dropped): the episodes scored since the last drain as a numpy structured array with the fields of
        CavEpisodeRow (env, episode, timesteps, winner, liveness_sum), in the order they finished, and how many rows a
        full ring lost."""
        capacity = getattr(self, "_episode_capacity", 0)
        rows = np.zeros(capacity, dtype=np.dtype([("env", "<i8"), ("episode", "<i4"), ("timesteps", "<i4"), ("winner", "<i4"),
                                                  ("liveness_sum", "<i4")]))
        n_rows, dropped = C.c_int64(), C.c_int64()
        _native.check(self._lib.cavgym_drain_episodes(self._handle, C.c_void_p(rows.ctypes.data), capacity, C.byref(n_rows), C.byref(dropped)))
        return rows[:n_rows.value], int(dropped.value)

    def launch_count(self):
        out = C.c_int64()
        _native.check(self._lib.cavgym_launch_count(self._handle, C.byref(out)))
        return int(out.value)

    def set_global_timestep(self, t):
        _native.check(self._lib.cavgym_set_global_timestep(self._handle, int(t)))

    def set_step_path(self, use_tma=True):
        """False forces the plain thread-per-env step kernel (the TMA-staged kernel is the default where it applies)."""
        _native.check(self._lib.cavgym_set_step_path(self._handle, int(bool(use_tma))))

    def set_dense_path(self, force=True):
        """True runs a small scenario through the warp-per-env kernels that scenarios with > CAV_SMALL_M bodies always use."""
        _native.check(self._lib.cavgym_set_dense_path(self._handle, int(bool(force))))

    def set_host_path(self, zero_copy=True):
        """False makes step_host stage pinned buffers through device copies instead of the zero-copy launch."""
        _native.check(self._lib.cavgym_set_host_path(self._handle, int(zero_copy)))

    def set_tangent_tolerance(self, tau):
        _native.check(self._lib.cavgym_set_tangent_tolerance(self._handle, float(tau)))

    def set_action_logging(self, enabled=True):
        _native.check(self._lib.cavgym_set_action_logging(self._handle, int(bool(enabled))))

    def set_uniform_override(self, uniforms):
        self._keep["uniforms"] = None if uniforms is None else torch.as_tensor(
            uniforms, dtype=torch.float64, device=self.device).contiguous()
        _native.check(self._lib.cavgym_set_uniform_override(self._handle, _ptr(self._keep["uniforms"])))

    def set_spawn_override(self, draws):
        self._keep["spawn"] = None if draws is None else torch.as_tensor(draws, dtype=torch.float64, device=self.device).contiguous()
        _native.check(self._lib.cavgym_set_spawn_override(self._handle, _ptr(self._keep["spawn"])))

    # ---- single-environment helpers for the compat view (library/environment.py) ----------------
    def reset_to(self, rows):
        init = torch.tensor(rows, dtype=self.dtype).reshape(self.num_bodies, 4, 1).expand(-1, -1, self.num_envs)
        self.reset(init_state=init.contiguous())

    def step_single(self, joint_action):
        rows = [[float(a[0]), float(a[1])] if isinstance(a, (list, tuple, np.ndarray)) else [float(int(a)), 0.0] for a in joint_action]
        actions = torch.tensor(rows, dtype=self.dtype).reshape(self.num_bodies, 2, 1)
        state, reward, done, winner, _ = self.step(actions)
        packed = torch.cat([state[:, :, 0].reshape(-1).double(), reward[:, 0].double(), done[:1].double(), winner[:1].double(),
                            self.episode_liveness[:, 0].double()]).cpu().tolist()
        m = self.num_bodies
        state_rows = [packed[4 * b:4 * b + 4] for b in range(m)]
        rewards = packed[4 * m:5 * m]
        done_flag, winner_index = bool(packed[5 * m]), int(packed[5 * m + 1])
        liveness = [int(v) for v in packed[5 * m + 2:6 * m + 2]]
        taken = [[r[0], 0.0 if abs(r[1]) < 0.0000000000001 else r[1]] for r in rows]
        return state_rows, rewards, done_flag, winner_index, liveness, taken


class HostBuffer:
    """A page-locked, device-mapped host array from cavgym_host_alloc, as a numpy array (`.array`).  write_combined=True is for
    buffers the host only writes and the GPU reads — the joint actions of step_host."""

    def __init__(self, shape, dtype, write_combined=False):
        self._lib = _native.load()
        self.array = None
        count = int(np.prod(shape))
        self._ptr = C.c_void_p()
        _native.check(self._lib.cavgym_host_alloc(count * np.dtype(dtype).itemsize, int(bool(write_combined)), C.byref(self._ptr)))
        ctype = np.ctypeslib.as_ctypes_type(np.dtype(dtype))
        self.array = np.ctypeslib.as_array(C.cast(self._ptr, C.POINTER(ctype)), shape=(count,)).reshape(shape)

    def close(self):
        if getattr(self, "_ptr", None) and self._ptr.value:
            self.array = None
            self._lib.cavgym_host_free(self._ptr)
            self._ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bodies_step(constants, states, actions, time_resolution, dtype="float64", device=None):
    """DynamicBody.step (reference library/bodies.py:214-275) for a list of independent bodies of one type,
    run by the stand-alone CUDA kinematics kernel.  states [n][4], actions [n][2] -> new states [n][4]."""
    lib = _native.load()
    device = _require_cuda(device)
    code, tdtype = _DTYPES[dtype]
    state_t = torch.tensor(states, dtype=tdtype, device=device).t().contiguous()
    action_t = torch.tensor(actions, dtype=tdtype, device=device).t().contiguous()
    k = _abi.CavBodyType(*[float(v) for v in (constants.length, constants.width, constants.wheelbase, constants.min_velocity,
                                               constants.max_velocity, constants.min_throttle, constants.max_throttle,
                                               constants.min_steering_angle, constants.max_steering_angle)])
    with torch.cuda.device(device):
        _native.check(lib.cavgym_bodies_step(C.byref(k), _ptr(state_t), _ptr(action_t), state_t.shape[1], float(time_resolution),
                                             code, C.c_void_p(torch.cuda.current_stream(device).cuda_stream)))
    return state_t.t().cpu().tolist()


def zones_probe(constants, states, steering, dtype="float64", device=None):
    """DynamicBody.stopping_zones (reference library/bodies.py:122-135) for n independent bodies of one type, as the step
    kernels represent the zones.  states [n][4], steering [n] -> (zones [n][2][4][2] = braking / reaction corner lists in the
    reference's order, have [n] bool; rows without zones are NaN)."""
    lib = _native.load()
    device = _require_cuda(device)
    code, tdtype = _DTYPES[dtype]
    state_t = torch.tensor(np.asarray(states, dtype=np.float64), dtype=tdtype, device=device).t().contiguous()
    steer_t = torch.tensor(np.asarray(steering, dtype=np.float64), dtype=tdtype, device=device).contiguous()
    n = state_t.shape[1]
    zones = torch.empty((16, n), dtype=tdtype, device=device)
    have = torch.empty(n, dtype=torch.uint8, device=device)
    k = _abi.CavBodyType(*[float(v) for v in (constants.length, constants.width, constants.wheelbase, constants.min_velocity,
                                               constants.max_velocity, constants.min_throttle, constants.max_throttle,
                                               constants.min_steering_angle, constants.max_steering_angle)])
    with torch.cuda.device(device):
        _native.check(lib.cavgym_zones_probe(C.byref(k), _ptr(state_t), _ptr(steer_t), _ptr(zones), _ptr(have), n, code,
                                             C.c_void_p(torch.cuda.current_stream(device).cuda_stream)))
    z = zones.double().cpu().numpy().reshape(2, 2, 4, n)           # [zone][x|y][corner][n]
    return np.transpose(z, (3, 0, 2, 1)), have.cpu().numpy().astype(bool)


def geometry_probe(quads_a, quads_b, dtype="float64", device=None):
    """Shape.intersects / contains / percentage_intersects (reference library/geometry.py:74-87) on n quad pairs,
    run by the CUDA geometry code.  quads [n][4][2] -> array [n][4]: intersects, b.contains(a), share, tangent."""
    lib = _native.load()
    device = _require_cuda(device)
    code, tdtype = _DTYPES[dtype]

    def pack(quads):
        arr = np.asarray(quads, dtype=np.float64)  # [n, 4, 2]
        return torch.tensor(np.concatenate([arr[:, :, 0].T, arr[:, :, 1].T], axis=0), dtype=tdtype, device=device).contiguous()

    a, b = pack(quads_a), pack(quads_b)
    out = torch.empty((4, a.shape[1]), dtype=tdtype, device=device)
    with torch.cuda.device(device):
        _native.check(lib.cavgym_geometry_probe(_ptr(a), _ptr(b), _ptr(out), a.shape[1], code,
                                                C.c_void_p(torch.cuda.current_stream(device).cuda_stream)))
    return out.t().double().cpu().numpy()
