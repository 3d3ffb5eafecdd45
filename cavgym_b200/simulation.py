"""Episode loops over the engine.

  Simulation          the reference's driver (simulation.py:9-118) on the single-environment compat view: host-side agents
                      choose the joint action, `env.step` is one CUDA launch on a batch of one.  Same console / log lines.
  BatchedSimulation   the same experiment at batch scale: N concurrent copies of the config's scenario, on-device agents,
                      scoring and auto-reset inside the rollout kernel (cavgym_rollout); the run summary comes from the
                      device counters (cavgym_stats), optionally summed over ranks with one all-reduce; with an
                      `episode_log` the per-episode rows come from the device ring (cavgym_drain_episodes), one per
                      finished episode, in the reference's episode.log format.  With `save_interesting` = K the first K
                      interesting episodes are regenerated after the run (BatchedCAVEnv.regenerate) and kept in
                      `interesting`.
"""
import timeit

import numpy as np

from . import reporting
from .config import AgentType, Mode


class Simulation:
    def __init__(self, env, agents, config, keyboard_agent=None):
        assert len(env.bodies) == len(agents), "each body must be assigned an agent and vice versa"
        if keyboard_agent is not None:
            raise NotImplementedError("keyboard agents need the reference's pyglet viewer")
        self.env, self.agents, self.config = env, agents, config
        self.election = None
        if config.tester_config.agent is AgentType.ELECTION:   # simulation.py:20-23
            from .examples.election import Election
            self.election = Election(env, agents)
        self.console = reporting.get_console(config.verbosity)
        self.episode_file = reporting.get_episode_file_logger(config.episode_log) if config.episode_log is not None else None
        self.run_file = reporting.get_run_file_logger(config.run_log) if config.run_log is not None else None

    def run(self):
        """Runs config.episodes episodes (each cut off at config.max_timesteps); returns (episode_results, run_summary)."""
        env, agents, config = self.env, self.agents, self.config
        episode_data = []
        run_start = timeit.default_timer()
        for episode in range(1, config.episodes + 1):
            episode_start = timeit.default_timer()
            state = env.reset()
            info = env.info()
            self.console.debug(f"state={state}")
            for agent in agents:
                agent.reset()
            final_timestep = config.max_timesteps
            for timestep in range(1, config.max_timesteps + 1):
                joint_action = [agent.choose_action(state, space, info) for agent, space in zip(agents, env.action_space)]
                if self.election:
                    joint_action = self.election.result(state, joint_action)
                previous_state = state
                state, joint_reward, done, info = env.step(joint_action)
                self.console.debug(f"timestep={timestep}")
                self.console.debug(f"action={joint_action}")
                self.console.debug(f"state={state}")
                self.console.debug(f"reward={joint_reward}")
                self.console.debug(f"done={done}")
                for agent, action, reward in zip(agents, joint_action, joint_reward):
                    agent.process_feedback(previous_state, action, state, reward)
                if done:
                    final_timestep = timestep
                    break
            results = reporting.analyse_episode(episode, episode_start, timeit.default_timer(), final_timestep, info, config, env)
            episode_data.append(results)
            self.console.info(results.console_message())
            if self.episode_file:
                self.episode_file.info(results.file_message())
        summary = reporting.RunSummary.from_episodes(episode_data, run_start, timeit.default_timer(), env.time_resolution)
        self.console.info(summary.console_message())
        if self.run_file:
            self.run_file.info(summary.file_message())
        env.close()
        return episode_data, summary


class BatchedSimulation:
    def __init__(self, config, num_envs, device=None, dtype="float64", env_offset=0, chunk=100):
        self.config, self.chunk = config, int(chunk)
        self.env = config.batched(num_envs, device=device, dtype=dtype, env_offset=env_offset)
        self.console = reporting.get_console(config.verbosity)
        self.run_file = reporting.get_run_file_logger(config.run_log) if config.run_log is not None else None
        self.episode_file = reporting.get_episode_file_logger(config.episode_log) if config.episode_log is not None else None
        self.episode_rows = []      # EpisodeResults of every drained episode when an episode log is kept (keep_rows / episode_log)
        self.keep_rows = False
        self.dropped_rows = 0
        self.save_interesting = 0   # K: regenerate the first K interesting episodes after run() into `interesting`
        self.interesting = []

    def _drain(self, resolution):
        """Per-episode rows from the device ring -> reporting.EpisodeResults, numbered in finishing order (the reference
        numbers episodes in running order, simulation.py:40); written to episode.log in the reference's row format
        (reporting.py:157-158) with NaN for the per-episode wall-clock, which concurrent environments do not have."""
        rows, dropped = self.env.drain_episodes()
        self.dropped_rows += dropped
        if self.save_interesting:
            self._note_interesting(rows, dropped)
        if not (self.keep_rows or self.episode_file):
            return
        nan = float("nan")
        for row in rows:
            index = self._episodes_logged = getattr(self, "_episodes_logged", 0) + 1
            interesting = int(row["winner"]) > 0
            result = reporting.EpisodeResults(index, reporting.TimeResults(int(row["timesteps"]), nan, nan, resolution),
                                              completed=int(row["timesteps"]) == self.config.max_timesteps, interesting=interesting,
                                              score=-int(row["liveness_sum"]) if interesting else nan)
            if self.keep_rows:
                self.episode_rows.append((int(row["env"]), int(row["episode"]), result))
            if self.episode_file:
                self.episode_file.info(result.file_message())

    def _note_interesting(self, rows, dropped):
        """Keep the first save_interesting rows of tester wins with the t_global of their first step.  With auto-reset an env's
        next episode starts at the step after its last one ends, so episode j of an env starts at the sum of the lengths of its
        episodes before j since the run's reset (at t_global 0): every row of the env is needed, so none may be dropped."""
        if dropped:
            raise RuntimeError("episode rows were dropped from the device ring: the start steps of later episodes are unknown")
        env = self.env
        if not hasattr(self, "_next_start"):
            self._next_start = np.zeros(env.num_envs, dtype=np.int64)
        order = np.lexsort((rows["episode"], rows["env"]))
        slot = rows["env"][order].astype(np.int64) - env.env_offset
        length = rows["timesteps"][order].astype(np.int64)
        before = np.cumsum(length) - length                   # within this drain, per env in episode order
        first = np.r_[True, slot[1:] != slot[:-1]]
        start = self._next_start[slot] + before - np.maximum.accumulate(np.where(first, before, 0))
        np.add.at(self._next_start, slot, length)
        wins = order[rows["winner"][order] > 0]
        starts = start[rows["winner"][order] > 0]
        keep = np.argsort(wins, kind="stable")[:max(0, self.save_interesting - sum(len(r) for r, _ in self._hits))]
        self._hits.append((rows[wins[keep]], starts[keep]))

    def _regenerate_interesting(self):
        hits = [r for r, _ in self._hits]
        if not hits or not sum(len(r) for r in hits):
            return []
        return self.env.regenerate(np.concatenate(hits), t_global_start=np.concatenate([s for _, s in self._hits]))

    def _learner(self):
        """The Q-learning ego on the tensor API (config.json's stock ego option), or None when every agent is on the device."""
        if self.config.ego_config.agent is not AgentType.Q_LEARNING:
            return None
        from .examples.agents.ego import BatchedQLearningEgoAgent
        env = self.env
        self.learner = BatchedQLearningEgoAgent(self.config.ego_config, env.bodies[0].constants, env.time_resolution, env.num_bodies - 1,
                                                env.constants.viewer_width, env.constants.viewer_height, env.num_envs, env.device,
                                                dtype=env.dtype, seed=self.config.seed or 0)
        return self.learner

    def _learning_steps(self, learner, n_steps):
        """Simulation.run's timestep loop (simulation.py:69-93) with the ego's action chosen by the learner: choose on the
        pre-step state, one cavgym_step (testers act on the device), TD update on the transition, reset of the envs that
        finished (their episode was scored by the step kernel)."""
        import torch
        env = self.env
        if not hasattr(self, "_joint"):
            self._joint = torch.zeros((env.num_bodies, 2, env.num_envs), dtype=env.dtype, device=env.device)
            self._previous = torch.empty_like(env.state)
        for _ in range(n_steps):
            self._previous.copy_(env.state)
            index, rows = learner.choose_action(self._previous)
            self._joint[0] = rows
            state, reward, _, _, _ = env.step(self._joint)
            learner.process_feedback(self._previous, index, state, reward[0])
            env.reset(mask=env.done_latch != 0)

    def run(self, episodes=None, reduce=True):
        """Rolls every env forward (auto-reset) until at least `episodes` (default: config.episodes) episodes have finished
        on this rank; returns the RunSummary of everything finished so far (summed over ranks when a process group is up)."""
        import torch
        from . import sharding
        target = self.config.episodes if episodes is None else int(episodes)
        env = self.env
        logging_rows = self.episode_file is not None or self.keep_rows or self.save_interesting > 0
        if self.save_interesting and self.config.ego_config.agent is AgentType.Q_LEARNING:
            raise ValueError("save_interesting regenerates episodes on the device: the Q-learning ego chooses its actions on the host")
        self._hits = []
        if logging_rows:   # an episode lasts tens of steps at least: room for every env to finish chunk/16 times between drains
            env.set_episode_log(env.num_envs * max(1, self.chunk // 16) + 1024)
        env.reset()
        self.steps_run = 0
        start = timeit.default_timer()
        learner = self._learner()
        while True:
            if learner is None:
                env.rollout(self.chunk, auto_reset=True)
            else:
                self._learning_steps(learner, self.chunk)
            self.steps_run += self.chunk
            stats = env.stats()          # synchronises
            if logging_rows:
                self._drain(env.time_resolution)
            if stats["episodes"] >= target:
                break
        if self.dropped_rows:
            self.console.warning(f"{self.dropped_rows} episode row(s) did not fit the device ring and are missing from the episode log")
        torch.cuda.synchronize(env.device)
        runtime_ms = (timeit.default_timer() - start) * 1000
        if reduce:
            stats = sharding.reduce_stats(stats, env.device)
        summary = reporting.RunSummary.from_stats(stats, runtime_ms, env.time_resolution)
        self.console.info(summary.console_message())
        if self.run_file:
            self.run_file.info(summary.file_message())
        if self.save_interesting:
            self.interesting = self._regenerate_interesting()
        return summary
