"""`python -m cavgym_b200 [config.json] [--envs N]` — the reference's entry point (cavgym.py:1-40: read a config, set the
scenario up, run the simulation).  Without --envs: the reference's own loop on one environment (host-side agents, one
CUDA launch per transition).  With --envs N: N concurrent copies with the on-device agents (BatchedSimulation);
--save-interesting K then also writes the full trajectories of the first K interesting episodes (a tester won) to
interesting.npz beside the config's episode / run log (trajectories.save_episodes)."""
import json
import os
import sys

from .config import AgentType, ConfigParser, make_config
from .simulation import BatchedSimulation, Simulation


def main(argv=None):
    parser = ConfigParser()
    parser.add_argument("--envs", type=int, default=0, help="run this many concurrent environments on the GPU (0: single environment)")
    parser.add_argument("--dtype", default="float64", choices=["float64", "float32"])
    parser.add_argument("--save-interesting", type=int, default=0, metavar="K",
                        help="with --envs: write the trajectories of the first K interesting episodes to interesting.npz")
    args = parser.parse_args(argv)
    config = make_config(json.load(args.input))
    if args.save_interesting:
        if args.envs <= 0 or args.save_interesting < 0:
            parser.error("--save-interesting takes K > 0 and needs --envs")
        if config.ego_config.agent is AgentType.Q_LEARNING:
            parser.error("--save-interesting regenerates episodes on the device: the Q-learning ego chooses its actions on the host")
    if args.envs > 0:
        simulation = BatchedSimulation(config, args.envs, dtype=args.dtype)
        simulation.save_interesting = args.save_interesting
        simulation.run()
        if args.save_interesting:
            from . import trajectories
            log = config.episode_log or config.run_log
            path = os.path.join(os.path.dirname(log) if log else ".", "interesting.npz")
            trajectories.save_episodes(path, simulation.interesting,
                                       {"config": config.to_data(), "dtype": args.dtype, "seed": config.seed or 0})
    else:
        _, env, agents, keyboard_agent = config.setup()
        Simulation(env, agents, config, keyboard_agent).run()


if __name__ == "__main__":
    sys.exit(main())
