#!/usr/bin/env python
"""bench.py — throughput of the CAV-Gym stepping hot path on B200 (driver contract in the task prompt).

    python bench.py --gpus 1 --steps 1000 --warmup 100             # our arm
    python bench.py --gpus 1 --steps 1000 --warmup 100 --dump-outputs DIR   # also write the last timed step's results
    python bench.py --impl reference --gpus 1 --steps 200 --warmup 10   # CPU arm (oracle port, all host threads)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], "C2"): the stock pedestrians scenario (Car + SpawnPedestrian) batched to
65,536 parallel envs per GPU, replayed joint actions, fp64.  A "step" is one CAVEnv.step over the whole batch.
The joint actions are synthetic: a RandomConstrainedAgent(eps=0.01) trace generated ON DEVICE before the timed
region (untimed) for every env, then replayed.  `value` counts only LIVE env-steps (frozen, finished envs do not
count), inputs resident in HBM, trajectories (state, reward, done, winner, tangent) recorded to HBM slabs larger
than L2.  `e2e` is the same metric through cavgym_step_host with pinned HOST buffers (H2D actions, D2H results
inside the timed region).  `hbm_config` repeats the per-step kernel at 4,194,304 envs, where the working set is
far beyond L2, for the HBM-roofline fraction (SURVEY §8d: do not call the 65,536-env figure an HBM fraction).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_ENVS = 65536          # per GPU (weak scaling)
SEGMENT = 250           # steps replayed from a fresh reset before the whole batch is reset again: a finished env stays frozen
                        # (and uncounted) until then — 3 % of the env-steps at 250, 10 % at 500 (the ego finishes at step 901)
CHUNK = 250             # steps fused per cavgym_replay launch (50: 16.0, 100: 17.9, 250: 20.3, 500: 20.8 G env-steps/s)
HBM_ENVS = 4 * 1024 * 1024
HBM_ADVANCE = 300        # unrecorded steps before the HBM-config trace: envs are mid-episode, pedestrians mid-crossing
EPSILON = 0.01
BYTES_PER_BODY_STEP = {"float64": 88, "float32": 44}   # SURVEY §8d: 4w state in + 2w action + 4w state out + 1w reward
BYTES_PER_ENV_STEP_EXTRA = 5                            # 1 B done + 4 B winner


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(kernel, steps_per_launch=None):
    """(DRAM bytes per launch, note) of `kernel` from the committed ncu captures (profiles/traffic.json).  Entries are
    keyed by launch shape; a shape that was not captured is scaled per fused step from the nearest one, and says so."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as fh:
            entry = json.load(fh).get(kernel, {})
    except (OSError, ValueError):
        return None, "no ncu capture found"
    if steps_per_launch is None:
        return entry.get("dram_bytes_per_launch"), entry.get("launch", "")
    shapes = {int(k): v for k, v in entry.get("per_steps_per_launch", {}).items()}
    if not shapes:
        return None, "no ncu capture found"
    if steps_per_launch in shapes:
        source = entry.get("source_by_shape", {}).get(str(int(steps_per_launch)), entry.get("source", "profiles/"))
        return shapes[int(steps_per_launch)], (f"dram__bytes_read.sum + dram__bytes_write.sum of one {int(steps_per_launch)}-step launch "
                                                f"(ncu --set full, {source}); {entry.get('note', '')}")
    nearest = min(shapes, key=lambda k: abs(k - steps_per_launch))
    return int(shapes[nearest] * steps_per_launch / nearest), (f"scaled per fused step from the ncu capture of a {nearest}-step launch "
                                                               f"({entry.get('source', 'profiles/')}); this shape was not captured")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt, self.ready = threading.Event(), threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM)
            names = {pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            self.ready.set()
            while True:   # at least one sample, even when the timed region lasts a few milliseconds
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                self.reasons.update(name for bit, name in names.items() if mask & bit)
                if self._halt.is_set():
                    break
                time.sleep(0.001)
        except Exception as exc:  # NVML missing: report nothing rather than guess
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")
            self.ready.set()

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        samples = sorted(self.samples)
        return {"sm_mhz": samples[len(samples) // 2] if samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def scenario(mode):
    from helpers import compile_from_meta, load_golden
    meta, _ = load_golden("pedestrians_rc_seed0")   # the stock config.json scenario (ego noop, tester random-constrained)
    meta["config"]["tester_config"]["epsilon"] = EPSILON
    return compile_from_meta(meta, mode=mode)


def make_trace(torch, device, n_envs, n_steps, dtype, env_offset, advance=0):
    """Untimed set-up: run the on-device agents once and log every joint action -> (init_state, actions[T,M,2,N]).
    `advance` first runs that many unrecorded steps (auto-reset on), so the trace starts mid-episode with the
    envs spread over every phase of a crossing."""
    from cavgym_b200 import BatchedCAVEnv
    gen = BatchedCAVEnv(None, None, None, num_envs=n_envs, dtype=dtype, compiled=scenario("device"), device=device, seed=0,
                        env_offset=env_offset)
    gen.set_action_logging(True)
    gen.reset()
    if advance:
        gen.rollout(advance, auto_reset=True)
    init = gen.state.clone()
    actions = torch.empty((n_steps, gen.num_bodies, 2, n_envs), dtype=gen.dtype, device=device)
    for t in range(n_steps):
        gen.step(None)
        actions[t].copy_(gen.actions_taken)
    torch.cuda.synchronize(device)
    gen.close()
    return init, actions


def dump_outputs(directory, arrays):
    """Write what the last timed step returned to its caller (cavgym_replay: state [M, 4, N], reward [M, N], done, winner,
    tangent [N]) as DIR/<name>.npy, so that two builds can be compared output for output: the trace and the initial state
    are generated from fixed seeds, so the same arguments replay the same inputs.  Real arrays keep the run's dtype;
    done / winner / tangent are stored as float64 (exact).  About 7 MB at float64."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, tensor in arrays.items():
        data = tensor.cpu().numpy()
        np.save(os.path.join(directory, f"{name}.npy"), data if data.dtype.kind == "f" else data.astype(np.float64))


def run_ours(args):
    chunk = max(1, min(int(args.chunk), SEGMENT, args.steps))   # steps fused per cavgym_replay launch
    segment = SEGMENT // chunk * chunk                          # whole launches between resets (240 steps at 20 per launch)
    import torch
    import torch.distributed as dist
    from cavgym_b200 import BatchedCAVEnv

    from cavgym_b200 import sharding
    rank, world, local = sharding.rank_world()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    dtype, n, m = args.dtype, N_ENVS, 2
    bytes_env_step = m * BYTES_PER_BODY_STEP[dtype] + BYTES_PER_ENV_STEP_EXTRA
    peak_gbs, peak_src = peaks()

    init, actions = make_trace(torch, device, n, segment, dtype, env_offset=sharding.shard_offset(rank, n))
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=scenario("external"), device=device,
                        env_offset=sharding.shard_offset(rank, n))
    # Trajectory slabs: 5.24 MB per step.  Launches rotate over `slots` slabs so that >= 315 MB (2.5 x the 126 MB L2) are
    # written before a slab is written again: the trajectory stores of the timed region reach HBM, not a warm L2 line.
    slots = max(1, -(-60 // chunk))
    slab_steps = slots * chunk
    slab = {"state": torch.empty((slab_steps, m, 4, n), dtype=env.dtype, device=device),
            "reward": torch.empty((slab_steps, m, n), dtype=env.dtype, device=device),
            "done": torch.empty((slab_steps, n), dtype=torch.uint8, device=device),
            "winner": torch.empty((slab_steps, n), dtype=torch.int32, device=device),
            "tangent": torch.empty((slab_steps, n), dtype=torch.uint8, device=device)}
    lib, handle, stream = env._lib, env._handle, env._stream()
    from cavgym_b200._native import check
    import ctypes as C

    def ptr(t):
        return C.c_void_p(t.data_ptr())

    launch_events, launch_no, last_step = [], [0], [0]

    def advance(n_steps, cursor, timed):
        """Replay n_steps starting at trace position `cursor` (resetting every `segment` steps); returns new cursor."""
        done = 0
        while done < n_steps:
            if cursor == 0:
                env.reset(init_state=init)
            take = min(chunk, n_steps - done, segment - cursor)
            if timed:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
            at = (launch_no[0] % slots) * chunk
            launch_no[0] += 1
            last_step[0] = at + take - 1          # slab row of the results of the last step replayed so far
            check(lib.cavgym_replay(handle, take, ptr(actions[cursor]), ptr(slab["state"][at]), ptr(slab["reward"][at]),
                                    ptr(slab["done"][at]), ptr(slab["winner"][at]), ptr(slab["tangent"][at]), stream))
            if timed:
                b.record()
                launch_events.append((a, b, take))
            done += take
            cursor = (cursor + take) % segment
        return cursor

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- device-resident throughput (value) -------------------------------------------------
    # The timed region is `--steps` steps (resets included).  All its launches are enqueued while a gate kernel keeps the
    # stream busy, so no host launch latency sits between the events: they time the GPU, not the Python loop.
    advance(args.warmup, 0, False)
    cursor = 0   # pass A starts from a fresh reset, pass B where pass A ended
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    sampler.ready.wait(timeout=10)    # NVML initialised before the timed region starts
    launches_per_region = -(-args.steps // chunk) + args.steps // segment + 2
    barrier()
    if args.profile_region:      # ncu --profile-from-start off: capture exactly the timed region
        torch.cuda.profiler.start()
    torch.cuda._sleep(int((4e-3 + 4e-5 * launches_per_region) * 1.9e9))
    # Pass A (per-launch statistics, untimed for `value`): a CUDA event before and after every launch.  An event between two
    # launches also serialises them, so this pass shows each launch in isolation (no programmatic dependent launch overlap).
    cursor = advance(args.steps, cursor, True)
    queued_ahead = not launch_events[0][0].query()   # the GPU had not reached the first event when the host finished enqueuing
    barrier()
    region_ms = launch_events[0][0].elapsed_time(launch_events[-1][1])
    mid, launches_mid = env.stats(), env.launch_count()
    # Pass B (the measurement): the next `--steps` steps of the trace, launched back to back as a caller issues them —
    # nothing between them — with ONE event pair around them: consecutive replay launches overlap head and tail
    # (launch_replay_tma).
    torch.cuda._sleep(int((4e-3 + 4e-5 * launches_per_region) * 1.9e9))
    start_b, stop_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start_b.record()
    advance(args.steps, cursor, False)
    stop_b.record()
    queued_ahead = queued_ahead and not start_b.query()
    barrier()
    if args.profile_region:
        torch.cuda.profiler.stop()
    clocks = sampler.stop()
    elapsed_ms = start_b.elapsed_time(stop_b)
    after, launches_after = env.stats(), env.launch_count()
    live_env_steps = after["env_steps"] - mid["env_steps"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {name: slab[name][last_step[0]] for name in slab})
    # stats() itself launches one reduction kernel per call: not part of the timed region
    gpu_launches = launches_after - launches_mid - 1
    isolated_ms = sum(a.elapsed_time(b) for a, b, _ in launch_events) / len(launch_events)
    kernel_steps = sum(k for _, _, k in launch_events)
    replay_launches = len(launch_events)          # pass B issues exactly the launches of pass A again
    steps_per_launch = kernel_steps / replay_launches
    kernel_ms = elapsed_ms                         # back-to-back: the launches tile the timed region

    elapsed_ms, total_env_steps = sharding.reduce_timing(elapsed_ms, live_env_steps, device)   # MAX time, SUM units
    value = total_env_steps / (elapsed_ms * 1e-3)

    # roofline of the dominant kernel: algorithmic bytes per launch / mean launch duration (CUDA events around each launch)
    live_fraction = live_env_steps / float(n * args.steps)
    bytes_per_launch = bytes_env_step * n * steps_per_launch * live_fraction
    achieved = bytes_per_launch / (kernel_ms / replay_launches * 1e-3) / 1e9
    kernel_name = f"replay_tma_kernel<{'double' if dtype == 'float64' else 'float'},2,false>"
    traffic, traffic_note = measured_traffic(kernel_name, steps_per_launch)
    roofline = {"bound": "hbm", "kernel": kernel_name,
                "achieved": round(achieved, 1), "peak": peak_gbs, "peak_source": peak_src, "unit": "GB/s",
                "frac": round(achieved / peak_gbs, 4), "traffic": traffic, "traffic_note": traffic_note,
                "algorithmic_bytes_per_launch": int(bytes_per_launch),
                "algorithmic_bytes_per_env_step": bytes_env_step, "launches": replay_launches,
                "steps_per_launch": steps_per_launch, "avg_launch_ms": round(kernel_ms / replay_launches, 5),
                "isolated_launch_ms": round(isolated_ms, 5),
                "frac_isolated": round(bytes_per_launch / (isolated_ms * 1e-3) / 1e9 / peak_gbs, 4),
                "launch_chaining": "consecutive cavgym_replay launches chain tile by tile (a CTA waits for its own tile's sequence "
                                   "number, not for the whole previous grid: kernels_tma.cuh), so back-to-back launches OVERLAP on the "
                                   "device — ramp, tail and drain of one launch are covered by its neighbours",
                "timing": "avg_launch_ms = device time of the timed region (one CUDA event pair around all launches, issued back to "
                          "back) / launches, i.e. the time per launch at which the train advances; isolated_launch_ms = mean of "
                          "per-launch event pairs in a separate pass (an event between two launches serialises them: the duration "
                          "of one launch alone, what ncu's serialised launch list also shows); frac is from the first, "
                          "frac_isolated from the second",
                "note": "65,536 envs: the state (4 MiB) stays in registers for the whole launch; actions stream in and "
                        "trajectories stream out through HBM (slabs larger than L2)"}

    out = {"metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64" if dtype == "float64" else "f32", "data": "synthetic",
           "body_steps_per_sec": value * m,
           "timed_region": {"steps": args.steps, "total_ms": elapsed_ms, "region_ms_per_launch_events": region_ms,
                            "launches_queued_before_first_event": bool(queued_ahead),
                            "note": "value = live env-steps / device time between ONE event pair around the --steps steps, launches "
                                    "issued back to back behind a gate kernel (max over ranks); region_ms_per_launch_events is from a "
                                    "separate pass over as many steps with an event pair around every launch (which serialises them)"},
           "config": {"workload": "C2: pedestrians scenario (Car + SpawnPedestrian) x 65,536 envs per GPU, replayed joint "
                                  f"actions (on-device RandomConstrained eps=0.01 trace), cavgym_replay {steps_per_launch:g} steps/launch, "
                                  f"trajectories recorded, {args.steps} timed steps",
                      "envs_per_gpu": n, "bodies": m, "segment": segment,
                      "l2": f"{slots} rotating trajectory slabs ({slab_steps * 5.24e6 / 1e9:.2f} GB) and the action trace (1 GB) exceed L2; state is register resident",
                      "live_fraction": round(live_fraction, 4)},
           "roofline": roofline, "gpu_launches": int(gpu_launches), "clocks": clocks}

    if rank == 0 or world > 1:
        # ---- end to end through the host-buffer API (every rank; max over ranks) -------------
        e2e_steps = max(3, min(args.e2e_steps, segment - 3))   # its own length: 20 calls of 0.15 ms would be a 3 ms measurement
        np_dtype = "float64" if dtype == "float64" else "float32"
        import numpy as np
        h_actions = torch.empty((segment, m, 2, n), dtype=env.dtype).pin_memory()
        h_actions.copy_(actions)
        h_state = torch.empty((m, 4, n), dtype=env.dtype).pin_memory()
        h_reward = torch.empty((m, n), dtype=env.dtype).pin_memory()
        h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
        h_winner = torch.empty(n, dtype=torch.int32).pin_memory()
        h_tangent = torch.empty(n, dtype=torch.uint8).pin_memory()
        # (a) the call that matches `value`: cavgym_replay, `chunk` fused steps per call, on pinned HOST tensors — the kernel reads
        #     every step's joint actions from and writes every step's results to host memory over PCIe inside the launch; the
        #     call returns when the results are in host memory and the next call is issued after that.
        call = min(chunk, 50)                       # steps per replay_host call (50 steps of results are 0.28 GB of pinned memory)
        e2e_steps = e2e_steps // call * call or call
        t_out = {"state": torch.empty((call, m, 4, n), dtype=env.dtype).pin_memory(), "reward": torch.empty((call, m, n), dtype=env.dtype).pin_memory(),
                 "done": torch.empty((call, n), dtype=torch.uint8).pin_memory(), "winner": torch.empty((call, n), dtype=torch.int32).pin_memory(),
                 "tangent": torch.empty((call, n), dtype=torch.uint8).pin_memory()}
        windows = [h_actions[at:at + call] for at in range(0, min(e2e_steps, segment // call * call), call)]
        env.reset(init_state=init)
        env.replay_host(windows[0], **t_out)
        env.reset(init_state=init)
        barrier()
        s0 = env.stats()
        t0 = time.perf_counter()
        for window in windows:
            env.replay_host(window, **t_out)
        e2e_s = time.perf_counter() - t0
        s1 = env.stats()
        e2e_time, e2e_units = sharding.reduce_timing(e2e_s, s1["env_steps"] - s0["env_steps"], device)
        rs = 8 if dtype == "float64" else 4
        out["e2e"] = {"value": e2e_units / e2e_time, "unit": "env-steps/s",
                      "h2d_bytes_per_step": m * 2 * n * rs, "d2h_bytes_per_step": m * 4 * n * rs + m * n * rs + n * 6,
                      "steps": len(windows) * call, "steps_per_call": call,
                      "api": "BatchedCAVEnv.replay_host = cavgym_replay on pinned host tensors: one launch per call reads the joint actions of "
                             "its steps from and writes state/reward/done/winner/tangent of every step to host memory over PCIe; the caller "
                             "waits for each call's results before issuing the next"}
        # (a2) the same calls with TWO in flight (double-buffered results): the caller issues call k + 1 before it consumes the
        #      results of call k, which a replayed-action workload allows; back-to-back launches overlap on the device, so the
        #      PCIe reads of one call cover the draining writes of the one before.  Reported beside the synchronous figure.
        t_out2 = {k_: torch.empty_like(v_).pin_memory() for k_, v_ in t_out.items()}
        results, ready = [t_out, t_out2], [torch.cuda.Event(), torch.cuda.Event()]
        env.reset(init_state=init)
        torch.cuda.synchronize(device)
        barrier()
        s0 = env.stats()
        t0 = time.perf_counter()
        for i, window in enumerate(windows):
            if i >= 2:
                ready[i % 2].synchronize()          # the results of call i - 2 are in host memory and consumed: its buffers are free
            env.replay_host(window, wait=False, **results[i % 2])
            ready[i % 2].record(torch.cuda.current_stream(device))
        torch.cuda.synchronize(device)
        pipe_s = time.perf_counter() - t0
        s1 = env.stats()
        pipe_time, pipe_units = sharding.reduce_timing(pipe_s, s1["env_steps"] - s0["env_steps"], device)
        out["e2e"]["two_calls_in_flight"] = {"value": pipe_units / pipe_time, "unit": "env-steps/s", "steps": len(windows) * call,
                                             "steps_per_call": call,
                                             "api": "the same replay_host calls, the next one issued before the previous one's results are "
                                                    "consumed (two result buffers, one CUDA event per call)"}
        del t_out2, results
        # (b) the per-step API: one cavgym_step_host call per step (what a host-side agent that needs every observation uses)
        e2e_steps = max(3, min(args.e2e_steps, segment - 3))
        env.reset(init_state=init)
        joint = [h_actions[t_] for t_ in range(3 + e2e_steps)]
        for t_ in range(3):
            env.step_host(joint[t_], h_state, h_reward, h_done, h_winner, h_tangent)
        barrier()
        s0 = env.stats()
        t0 = time.perf_counter()
        for t_ in range(e2e_steps):
            env.step_host(joint[3 + t_], h_state, h_reward, h_done, h_winner, h_tangent)
        torch.cuda.synchronize(device)
        step_s = time.perf_counter() - t0
        s1 = env.stats()
        step_time, step_units = sharding.reduce_timing(step_s, s1["env_steps"] - s0["env_steps"], device)
        out["e2e"]["per_step_api"] = {"value": step_units / step_time, "unit": "env-steps/s", "steps": e2e_steps,
                                      "api": "cavgym_step_host, pinned host buffers, zero copy: one launch per step reads the actions from and "
                                             "writes state/reward/done/winner/tangent to host memory over PCIe"}
        if dtype == "float64":   # side number: the same call with the float32 wire format (half the PCIe bytes; not the headline)
            w_actions = h_actions.float().pin_memory()
            w_state, w_reward = h_state.float().pin_memory(), h_reward.float().pin_memory()
            w_joint = [w_actions[t_] for t_ in range(3 + e2e_steps)]
            env.reset(init_state=init)
            for t_ in range(3):
                env.step_host(w_joint[t_], w_state, w_reward, h_done, h_winner, h_tangent)
            torch.cuda.synchronize(device)
            s0, t0 = env.stats(), time.perf_counter()
            for t_ in range(e2e_steps):
                env.step_host(w_joint[3 + t_], w_state, w_reward, h_done, h_winner, h_tangent)
            torch.cuda.synchronize(device)
            wire_s = time.perf_counter() - t0
            out["e2e"]["float32_wire"] = {"value": (env.stats()["env_steps"] - s0["env_steps"]) / wire_s, "unit": "env-steps/s (this rank)",
                                          "h2d_bytes_per_step": m * 2 * n * 4, "d2h_bytes_per_step": m * 4 * n * 4 + m * n * 4 + n * 6,
                                          "api": "cavgym_step_host_f32: fp64 engine, float32 actions / state / rewards on the wire"}

    # ---- episode statistics: the single NCCL reduce over NVLink (SURVEY §8e) ---------------------
    out["episode_stats"] = sharding.reduce_stats(env.stats(), device)
    env.close()

    if not args.skip_configs:   # C3 and C5 are sharded over every rank (BASELINE configs[2], [4]); rank 0 reports
        c3 = scenario_configs(torch, device, dtype, rank, world)
        c5 = sweep_config(torch, device, dtype, rank, world)
        if rank == 0:
            out["scenario_configs"], out["sweep_config"] = c3, c5
    if rank == 0:
        if not args.skip_hbm:
            out["hbm_config"] = hbm_config(torch, device, dtype, peak_gbs)
        if not args.skip_configs:   # C4 on this one GPU: reported beside the headline, not as it
            out["dense_config"] = dense_config(torch, device, dtype, skip_cpu=args.skip_cpu)
        if not args.skip_cpu:
            out["cpu_baseline"] = cpu_baseline(budget_s=args.cpu_seconds)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def hbm_config(torch, device, dtype, peak_gbs):
    """The per-step kernel (cavgym_step) at 4,194,304 envs: 268 MB of state, 0.77 GB algorithmic bytes per launch."""
    from cavgym_b200 import BatchedCAVEnv
    n, m, t_len = HBM_ENVS, 2, 6
    init, actions = make_trace(torch, device, n, t_len, dtype, env_offset=0, advance=HBM_ADVANCE)
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=scenario("external"), device=device)
    env.reset(init_state=init)
    for t in range(3):
        env.step(actions[t])
    torch.cuda.synchronize(device)
    times = []
    for rep in range(5):
        for t in range(t_len):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            env.step(actions[t])
            b.record()
            times.append((a, b))
    torch.cuda.synchronize(device)
    ms = sorted(a.elapsed_time(b) for a, b in times)
    mean_ms = sum(ms) / len(ms)
    bytes_launch = n * (m * BYTES_PER_BODY_STEP[dtype] + BYTES_PER_ENV_STEP_EXTRA)
    achieved = bytes_launch / (mean_ms * 1e-3) / 1e9
    env.close()
    return {"workload": "pedestrians x 4,194,304 envs, 300 steps into their episodes, cavgym_step (one launch per step), "
                        "replayed actions, working set >> L2",
            "kernel": (kernel := f"step_tma_kernel<{'double' if dtype == 'float64' else 'float'},2,false>"), "envs": n,
            "traffic": measured_traffic(kernel)[0], "traffic_note": measured_traffic(kernel)[1],
            "env_steps_per_sec": n / (mean_ms * 1e-3), "body_steps_per_sec": n * m / (mean_ms * 1e-3),
            "avg_launch_ms": round(mean_ms, 4), "min_launch_ms": round(ms[0], 4), "algorithmic_bytes_per_launch": bytes_launch,
            "achieved_gbs": round(achieved, 1), "peak_gbs": peak_gbs, "frac": round(achieved / peak_gbs, 4)}


def timed(torch, fn, repeats):
    """Mean milliseconds of fn() over `repeats` calls, CUDA events on the current stream."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(repeats):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / repeats


C3_ENVS = 1048576       # BASELINE configs[2]: each scenario at 1M envs, env-sharded over the GPUs of the run
BYTES_PER_BODY_STEP_AGENTS = {"float64": {"noop": 72, "random": 88, "random-constrained": 152}, "float32": {"noop": 36, "random": 44, "random-constrained": 76}}


def timed_all_ranks(torch, device, fn, repeats):
    """Device milliseconds of `repeats` calls of fn() on this rank, bracketed by barriers; MAX over ranks."""
    import torch.distributed as dist
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    torch.cuda.synchronize(device)
    if multi:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(repeats):
        fn()
    b.record()
    torch.cuda.synchronize(device)
    ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=device)
    if multi:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def scenario_configs(torch, device, dtype, rank=0, world=1, total_envs=C3_ENVS, steps=1000, chunk=100):
    """BASELINE config C3: each of the four examples/environments scenarios at 1,048,576 envs, sharded over the ranks of
    this run (sharding.split_envs; 131,072 per GPU at 8 GPUs), with the on-device agents Config.setup would build (ego noop;
    tester random-constrained on the pedestrians scenario, random elsewhere — config.py:358-396), auto-reset, cavgym_rollout.
    Every rank runs its shard; time = max over ranks, counters summed with one all-reduce."""
    from helpers import compile_from_meta, load_golden
    from cavgym_b200 import BatchedCAVEnv, sharding
    offset, n = sharding.split_envs(total_envs, world)[rank]
    peak_gbs, _ = peaks()
    out = {}
    for name, golden in (("pedestrians", "pedestrians_rc_seed0"), ("crossroads", "crossroads_random_all_seed6"),
                         ("bus-stop", "busstop_random_all_seed8"), ("pelican-crossing", "pelican_random_all_seed10")):
        meta, _ = load_golden(golden)
        meta["config"]["tester_config"]["epsilon"] = EPSILON
        env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compile_from_meta(meta, mode="device"), device=device, seed=0,
                            env_offset=offset)
        env.reset()
        env.rollout(chunk, auto_reset=True)
        torch.cuda.synchronize(device)
        before = sharding.reduce_stats(env.stats(), device)
        ms = timed_all_ranks(torch, device, lambda: env.rollout(chunk, auto_reset=True), steps // chunk)
        after = sharding.reduce_stats(env.stats(), device)
        live = after["env_steps"] - before["env_steps"]
        m = env.num_bodies
        # algorithmic bytes of one env-step with on-device agents (SURVEY 8d): ego 9 words, a tester 9 (noop) / 11 (random) /
        # 19 (crossing agent) words, + 4 B liveness r/w per tester
        tester = meta["config"]["tester_config"]["option"]
        per_env_step = BYTES_PER_BODY_STEP_AGENTS[dtype]["noop"] + (m - 1) * (BYTES_PER_BODY_STEP_AGENTS[dtype][tester] + 8) + BYTES_PER_ENV_STEP_EXTRA
        rate = live / (ms * 1e-3)
        out[name] = {"bodies": m, "envs": total_envs, "envs_per_rank": n, "steps": steps, "env_steps_per_sec": rate,
                     "body_steps_per_sec": rate * m, "episodes": after["episodes"] - before["episodes"],
                     "collisions": meta["config"]["terminate_collisions"],
                     "algorithmic_bytes_per_env_step": per_env_step,
                     "algorithmic_gbs_per_gpu": round(rate * per_env_step / 1e9 / world, 1),
                     "frac_of_hbm_peak_if_every_step_streamed": round(rate * per_env_step / 1e9 / world / peak_gbs, 4)}
        env.close()
    return {"workload": f"C3: {total_envs} envs per scenario over {world} GPU(s) ({n} on rank 0), on-device Philox agents (eps={EPSILON}), "
                        f"auto-reset, cavgym_rollout {chunk} steps/launch, {steps} steps timed",
            "note": "cavgym_rollout keeps the state in registers for the whole launch, so its DRAM traffic is 1/chunk of the per-step "
                    "algorithmic figure; the fraction says how far the kernel is from the rate at which a per-step API could stream",
            "scenarios": out}


def dense_config(torch, device, dtype, n=100000, steps=100, chunk=50, skip_cpu=False):
    """BASELINE config C4: 64 cars + 256 spawned pedestrians per env (51,040 box pairs per env-step), 100,000 envs,
    terminate_collisions = all; warp-per-env kernels (kernels_dense.cuh), on-device agents, auto-reset."""
    from types import SimpleNamespace
    import numpy as np
    from cavgym_b200 import BatchedCAVEnv
    from cavgym_b200.examples.environments import dense_traffic
    from cavgym_b200.library.bodies import Pedestrian
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    road_map, constants = dense_traffic.make_world()
    bodies = dense_traffic.make_bodies(np_random=np.random.RandomState(0), road_map=road_map)
    cfg = SimpleNamespace(terminate_collisions="all", terminate_ego_zones=True, terminate_ego_offroad=False, max_timesteps=1000,
                          reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)
    m = len(bodies)

    def measure(epsilon):
        specs = [AgentSpec("random-constrained", epsilon=epsilon) if isinstance(b, Pedestrian) else AgentSpec("noop") for b in bodies]
        env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compile_scenario(bodies, constants, cfg, specs), device=device, seed=1)
        env.reset()
        for _ in range(2):
            env.rollout(chunk, auto_reset=True)
        torch.cuda.synchronize(device)
        before = env.stats()
        ms = timed(torch, lambda: env.rollout(chunk, auto_reset=True), steps // chunk) * (steps // chunk)
        after = env.stats()
        env.close()
        return specs, ms, before, after

    # the pedestrians' crossing rate decides how many of the 256 are mid-crossing (turning, off the pavement) at any time:
    # eps = 2e-4 keeps ~5 % of them crossing, the reference's config.json value 0.01 nearly all of them
    _, ms_ref, before_ref, after_ref = measure(EPSILON)
    specs, ms, before, after = measure(2e-4)
    live = after["env_steps"] - before["env_steps"]
    rate = live / (ms * 1e-3)
    real = 8 if dtype == "float64" else 4
    cpu = None
    if not skip_cpu:   # the oracle port on the same scenario, all host threads, a bounded sample (cpu_baseline leg)
        from oracle.oracle import Oracle
        threads = os.cpu_count() or 1
        sim = Oracle(compile_scenario(bodies, constants, cfg, specs), 4 * threads, seed=1, threads=threads)
        sim.reset()
        sim.rollout(5, auto_reset=True)
        t0 = time.perf_counter()
        sim.rollout(40, auto_reset=True)
        cpu = {"env_steps_per_sec": 4 * threads * 40 / (time.perf_counter() - t0), "cores": threads, "kind": "port",
               "sample": f"{4 * threads} envs x 40 steps, oracle/cavgym_oracle.c"}
        sim.close()
    return {"workload": f"C4: 64 cars + 256 spawned pedestrians x {n} envs, terminate_collisions=all, on-device agents "
                        f"(noop cars, random-constrained pedestrians eps=2e-4), auto-reset, {chunk} steps/launch",
            "kernel": f"dense_kernel<{'double' if dtype == 'float64' else 'float'},true>", "envs": n, "bodies": m,
            "env_steps_per_sec": rate, "body_steps_per_sec": rate * m, "pair_tests_per_sec": rate * (m * (m - 1) // 2),
            "ms_per_batch_step": ms / steps, "episodes": after["episodes"] - before["episodes"], "tangent": after["tangent"] - before["tangent"],
            "algorithmic_gbs": rate * m * 11 * real / 1e9, "bound": "instruction fetch / latency (DESIGN.md 4.4, 4.5), not HBM",
            "at_reference_epsilon": {"epsilon": EPSILON, "env_steps_per_sec": (after_ref["env_steps"] - before_ref["env_steps"]) / (ms_ref * 1e-3),
                                     "episodes": after_ref["episodes"] - before_ref["episodes"]},
            "cpu_baseline": cpu}


C5_ENVS = 1048576          # concurrent envs of the seed sweep (global; split over the ranks of the run)
C5_EPISODES = 10_000_000   # BASELINE configs[4]


def sweep_config(torch, device, dtype, rank=0, world=1, total_envs=C5_ENVS, episodes=C5_EPISODES, chunk=500):
    """BASELINE config C5 (experiments.py:95-122 as one batch): RandomConstrained testers searching for 'interesting'
    episodes; 1,048,576 concurrent envs (global ids 0..2^20-1, split over the ranks) roll forward with auto-reset in
    launches of `chunk` steps until the all-reduced episode count reaches 10 M.  Philox is keyed by the global env id and the
    stop rule only looks at global counts, so every total below is identical for any number of GPUs
    (tests/test_gpu_replay.py::test_sweep_totals_do_not_depend_on_the_split).  Mean +- 95 % CI as reporting.analyse_run."""
    from helpers import compile_from_meta, load_golden
    from cavgym_b200 import BatchedCAVEnv, sharding
    from cavgym_b200.reporting import RunSummary
    offset, n = sharding.split_envs(total_envs, world)[rank]
    out = {}
    for eps in (0.5, 0.01):
        meta, _ = load_golden("pedestrians_rc_seed0")
        meta["config"]["tester_config"]["epsilon"] = eps
        env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compile_from_meta(meta, mode="device"), device=device, seed=0,
                            env_offset=offset)
        env.reset()
        ms, steps, stats = 0.0, 0, sharding.reduce_stats(env.stats(), device)
        while stats["episodes"] < episodes and steps < 40000:
            ms += timed_all_ranks(torch, device, lambda: env.rollout(chunk, auto_reset=True), 1)
            steps += chunk
            stats = sharding.reduce_stats(env.stats(), device)       # the single all-reduce of the counters (untimed)
        summary = RunSummary.from_stats(stats, ms, env.time_resolution)
        out[f"epsilon={eps}"] = {"episodes": stats["episodes"], "interesting": stats["interesting"], "steps_per_env": steps,
                                 "env_steps": stats["env_steps"], "seconds": ms * 1e-3,
                                 "env_steps_per_sec": stats["env_steps"] / (ms * 1e-3), "body_steps_per_sec": 2 * stats["env_steps"] / (ms * 1e-3),
                                 "episodes_per_sec": stats["episodes"] / (ms * 1e-3),
                                 "timesteps_interesting": {"mean": summary.confidence_timesteps.value, "ci95": summary.confidence_timesteps.error},
                                 "score_interesting": {"mean": summary.confidence_score.value, "ci95": summary.confidence_score.error},
                                 "totals": {k: stats[k] for k in ("episodes", "interesting", "sum_t", "sum_t2", "sum_score", "sum_score2",
                                                                  "sum_t_interesting", "sum_t2_interesting")}}
        env.close()
    return {"workload": f"C5: pedestrians scenario, {total_envs} concurrent envs over {world} GPU(s), on-device RandomConstrained testers, "
                        f"auto-reset, cavgym_rollout {chunk} steps/launch, run until >= {episodes} episodes have finished", "runs": out}


def oracle_trace(n_envs, n_steps, threads):
    """Joint-action trace for the CPU arm, produced by the oracle's own RandomConstrained agents (untimed)."""
    import numpy as np
    from oracle.oracle import Oracle
    gen = Oracle(scenario("device"), n_envs, seed=0, threads=threads)
    gen.reset()
    init = gen.state.copy()
    actions = np.empty((n_steps, 2, 2, n_envs))
    for t in range(n_steps):
        gen.step(None)
        actions[t] = gen.actions_taken
    gen.close()
    return init, actions


def cpu_baseline(budget_s=15.0, threads=None):
    """The oracle port of the reference's step timed on this host's cores, on a bounded sample of the C2 workload."""
    from oracle.oracle import Oracle
    threads = threads or os.cpu_count() or 1
    n, t_len = 8192, 100
    init, actions = oracle_trace(n, t_len, threads)
    results = {}
    for label, nt in (("all", threads), ("one", 1)):
        sim = Oracle(scenario("external"), n, threads=nt)
        sim.reset(init_state=init)
        sim.replay(actions[:5], outputs=False)
        steps, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < budget_s / 2 and steps + 5 < t_len:
            take = min(10 if nt > 1 else 2, t_len - 5 - steps)
            sim.replay(actions[5 + steps:5 + steps + take], outputs=True)
            steps += take
        results[label] = n * steps / (time.perf_counter() - t0)
        sim.close()
    return {"value": results["all"], "unit": "env-steps/s", "cores": threads, "kind": "port",
            "single_thread_value": results["one"],
            "sample": f"{n} envs of the C2 scenario, replayed joint actions, oracle/cavgym_oracle.c (exact predicates), "
                      f"~{budget_s:.0f} s of CPU work",
            "note": "the reference itself is Python (README.md:27: 2,557 env-steps/s with real Shapely/GEOS); the port is C"}


def run_reference(args):
    """--impl reference: the CPU implementation of the path (oracle port; the Python reference cannot travel to the
    GPU box and has no compiled form), all host threads, same workload / metric / unit."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle.oracle import Oracle
    threads = os.cpu_count() or 1
    n = N_ENVS
    t_len = min(SEGMENT, args.warmup + args.steps)
    init, actions = oracle_trace(n, t_len, threads)
    sim = Oracle(scenario("external"), n, threads=threads)
    sim.reset(init_state=init)
    cursor = 0

    def advance(k, cursor):
        while k > 0:
            if cursor == 0:
                sim.reset(init_state=init)
            take = min(k, t_len - cursor, 10)
            sim.replay(actions[cursor:cursor + take], outputs=True)
            cursor = (cursor + take) % t_len
            k -= take
        return cursor

    cursor = advance(args.warmup, cursor)
    before = sim.stats()["env_steps"]
    t0 = time.perf_counter()
    cursor = advance(args.steps, cursor)
    elapsed = time.perf_counter() - t0
    live = sim.stats()["env_steps"] - before
    value = live / elapsed
    print(json.dumps({
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed * 1e3 / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "body_steps_per_sec": value * 2,
        "config": {"workload": "C2: pedestrians scenario x 65,536 envs, replayed joint actions, CPU", "envs": n, "bodies": 2},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps of the full 65,536-env batch, oracle/cavgym_oracle.c on {threads} threads"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=1000)
    parser.add_argument("--warmup", type=int, default=100)
    parser.add_argument("--impl", default="ours", choices=["ours", "reference"])
    parser.add_argument("--dtype", default="float64", choices=["float64", "float32"])
    parser.add_argument("--e2e-steps", type=int, default=200)
    parser.add_argument("--cpu-seconds", type=float, default=15.0)
    parser.add_argument("--chunk", type=int, default=CHUNK, help="steps fused per cavgym_replay launch (at most --steps)")
    parser.add_argument("--skip-hbm", action="store_true")
    parser.add_argument("--skip-cpu", action="store_true")
    parser.add_argument("--skip-configs", action="store_true", help="skip the C3 / C4 / C5 side measurements")
    parser.add_argument("--profile-region", action="store_true", help="cudaProfilerStart/Stop around the timed region (ncu --profile-from-start off)")
    parser.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step (rank 0's envs) as DIR/<name>.npy")
    args = parser.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if args.steps > 200:
            args.steps = 200   # bounded: 200 steps of 65,536 envs is ~13 M env-steps of CPU work
        args.warmup = min(args.warmup, 10)
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
