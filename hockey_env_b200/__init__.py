"""hockey_env_b200 -- B200-native batched HockeyEnv (drop-in for hockey.hockey_env of julilili42/hockey-env).

The hot path (HockeyEnv.step/reset incl. the Box2D world step, contact sensing, rewards, observations,
BasicOpponent and auto-reset) runs in hand-written sm_100a CUDA kernels behind the C ABI declared in
include/hockey_b200.h; this package is the thin host-side mirror of the reference's Python surface.
"""
from ._lib import HockeyLibraryError, load as load_library  # noqa: F401
from .env import (  # noqa: F401
    BasicOpponent, HockeyEnv, HockeyEnv_BasicOpponent, HockeyVecEnv, Mode, PolicyOpponent, REGISTRY, make, make_vec, spec,
    FPS, SCALE, VIEWPORT_W, VIEWPORT_H, W, H, CENTER_X, CENTER_Y, ZONE, MAX_ANGLE, MAX_TIME_KEEP_PUCK, GOAL_SIZE,
    RACKETPOLY, RACKETFACTOR, FORCEMULTIPLIER, SHOOTFORCEMULTIPLIER, TORQUEMULTIPLIER, MAX_PUCK_SPEED,
)

from .vector import HockeyGymVectorEnv  # noqa: F401
from .actor import ActorNetwork, ExplorationNoise, FusedActor, FusedActorPool, actor_rollout, load_td3_actor  # noqa: F401
from .training import DeviceReplayBuffer, OpponentPool, collect, cross_play, evaluate, evaluate_model  # noqa: F401
from .td3 import (  # noqa: F401
    DevicePrioritizedReplayBuffer, DeviceTD3Learner, FusedTD3Learner, FusedTD3Population, PopulationReplayBuffer, TD3Config,
    TwinQNetwork, train_population,
)

__all__ = ["make", "make_vec", "spec", "REGISTRY", "OpponentPool", "DeviceReplayBuffer", "collect", "cross_play", "evaluate", "evaluate_model", "DevicePrioritizedReplayBuffer", "DeviceTD3Learner", "FusedTD3Learner", "FusedTD3Population", "PopulationReplayBuffer", "train_population", "TD3Config", "TwinQNetwork", "HockeyGymVectorEnv", "ActorNetwork", "ExplorationNoise", "FusedActor", "FusedActorPool", "actor_rollout", "load_td3_actor", "HockeyVecEnv", "HockeyEnv", "HockeyEnv_BasicOpponent", "BasicOpponent", "PolicyOpponent", "Mode",
           "HockeyLibraryError", "load_library"]
