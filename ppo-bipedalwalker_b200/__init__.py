"""walker_b200: B200-native (sm_100a) hot path of De-Rosa/PPO-BipedalWalker behind the reference's own
Environment / Walker / IMaterial / PPOAgent method surface.  Imported as `ppo_bipedalwalker_b200`
(see __graft_entry__.load_package); the compute lives in lib/libwalker_b200.so (csrc/), never in Python."""
from ._lib import Hyperparams, WalkerB200Error, declared_symbols, lib  # noqa: F401
from .env import (DT_FRAME, MATERIALS, Carpet, EnvBatch, Environment, Ice, IMaterial, Metal, Paper, Rubber,  # noqa: F401
                  SuperRubber, Titanium, Walker, Wood, default_hyperparams, init, pin_host, unpin_host, JOINT_TRACE_DTYPE,
                  PAIR_TRACE_DTYPE)

from . import dist  # noqa: F401
from .ppo import *  # noqa: F401,F403
from .loop import VectorPPO  # noqa: F401
from .population import PBT, IndependentPPO, PPOPopulation, default_seeds  # noqa: F401
from .scene import (CreateCreature, CreateFloor, CreateRoughFloor, Hexagon, Hull, IObject, Joint, Pole, Scene, Square,  # noqa: F401
                    TerrainEnvBatch, Triangle)
from .settings import DeserializeJson, SerializeJson, Settings  # noqa: F401
