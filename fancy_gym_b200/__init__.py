"""fancy_gym_b200 — B200-native movement-primitive black-box rollouts with fancy_gym's API.

    import fancy_gym_b200 as fancy_gym
    env = fancy_gym.make('fancy_ProMP/HoleReacher-v0', num_envs=65536, device='cuda:0')
    obs, _ = env.reset(seed=0)
    obs, ret, terminated, truncated, infos = env.step(params)      # params [65536, 25]

Importing this package loads the CUDA library; it raises if the library has not been built
(there is no CPU fallback).
"""
from . import _lib  # noqa: F401  (fails loudly when the CUDA library is missing)
from .envs.registry import (ALL_MOVEMENT_PRIMITIVE_ENVIRONMENTS, MOVEMENT_PRIMITIVE_ENVIRONMENTS_FOR_NS,  # noqa: F401
                            register, upgrade)
from . import envs  # noqa: F401,E402  (runs the registrations)
from .utils.gym_compat import make, registry  # noqa: F401,E402
from .utils.make_env_helpers import make_bb  # noqa: F401,E402
from .vector import BlackBoxVectorEnv, StepVectorEnv, make_vec  # noqa: F401,E402
from .graph import EpisodePipeline, GraphedEpisode  # noqa: F401,E402

__version__ = "0.1.0"
ALL_FANCY_MOVEMENT_PRIMITIVE_ENVIRONMENTS = MOVEMENT_PRIMITIVE_ENVIRONMENTS_FOR_NS.get('fancy', {})
