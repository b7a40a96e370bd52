"""sand_crate_b200 - the SandCrate per-timestep particle step as hand-written sm_100a CUDA kernels behind the
reference's own step API (`Crate(world_config).physics_tick()`, `config/*.yaml`).

    from sand_crate_b200 import Crate, load_config
    crate = Crate(load_config("config/stirring_cup.yaml").world_config)
    crate.physics_tick()

Layout: `csrc/` CUDA kernels + the C ABI of `include/sandcrate.h`; `_lib.py` ctypes binding; `crate.py`,
`load_config.py`, `rigid_body.py`, `particle_source.py` the host-side mirror of the reference interface;
`ensemble.py` many variants of one scene (a sweep, seed replicas) stepped in one context;
`scenes.py` synthetic benchmark scenes.  Nothing here imports `oracle/`.
"""
from .load_config import Config, PlaybackConfig, WorldConfig, config_from_dict, load_config  # noqa: F401
from .crate import Crate  # noqa: F401
from .ensemble import Ensemble  # noqa: F401
from ._lib import Context, SandCrateError  # noqa: F401

__all__ = ["Crate", "Ensemble", "Context", "SandCrateError", "load_config", "config_from_dict", "Config", "WorldConfig",
           "PlaybackConfig"]
