"""cavgym_b200 — B200-native batched stepping engine behind CAV-Gym's multi-agent Gym API.

Public entry points:
  BatchedCAVEnv          tensor API over N environments (engine.py)
  EnvSnapshot            saved per-env state of some of its environments (BatchedCAVEnv.save_envs)
  library.environment.CAVEnv   single-environment compat view (reference protocol)
  make / register        env-id registry ('Pedestrians-v0', ... as the reference's examples/__init__.py)
  Config / make_config   config.json scenarios (config.py)
The CUDA extension is loaded on first use and its absence is an error — there is no CPU path.
"""
__version__ = "0.1.0"


def __getattr__(name):
    if name in ("BatchedCAVEnv", "EnvSnapshot"):
        from . import engine
        return getattr(engine, name)
    if name in ("make", "register"):
        from . import examples
        return getattr(examples, name)
    if name in ("Config", "make_config"):
        from . import config
        return getattr(config, name)
    raise AttributeError(name)
