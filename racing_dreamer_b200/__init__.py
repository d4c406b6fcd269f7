"""racing_dreamer_b200 -- B200-native batched racing-environment step.

Drop-in for the env path that CPS-TUWien/racing_dreamer's ``dreamer/wrappers.py`` drives
(SURVEY.md §8): dynamics -> 1080-beam LiDAR -> observation transforms -> progress/lap/collision
reward and termination, as hand-written sm_100a CUDA kernels behind a C ABI (``include/rd_env.h``).
"""
from .maps import TrackMap, load_track, available_tracks, TRACK_FILES  # noqa: F401

__version__ = "0.1.0"


def __getattr__(name):
    # the CUDA-backed classes import torch + the native library; keep `import racing_dreamer_b200` light
    if name in ("BatchedRaceEnv", "EnvConfig"):
        from . import env as _env
        return getattr(_env, name)
    if name in ("RaceCarGymCompat", "ReferenceEnv", "SingleAgentRaceCompat", "BaselinesEnv", "make_reference_env",
                "load_scenario"):
        from . import compat as _compat
        return getattr(_compat, name)
    if name in ("GapFollowerPolicy", "DreamerPolicy", "DreamerAgents", "load_dreamer_checkpoint", "save_dreamer_checkpoint"):
        from . import policy as _policy
        return getattr(_policy, name)
    raise AttributeError(name)
