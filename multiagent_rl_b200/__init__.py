"""B200-native batched particle-environment rollouts for yjpark1/multiagent_rl.

The hot path (MPE ``World.step`` + observation + reward, and the rls actor forward + hard
Gumbel sampling) runs as hand-written sm_100a CUDA kernels in ``libmpe_b200.so`` behind the C ABI of
``include/mpe_b200.h``; this package is the thin host mirror of the reference's surfaces:

    make_env(...)            experiments/scenarios.py:124-192
    env.reset() / env.step() upstream MultiAgentEnv (called at experiments/run.py:28,44,60)
    FusedActingMixin /
    ActingTrainer            rls/agent/multiagent/ddpg_gumbel_fix.py:86-107 get_exploration_action
    FusedActorNetwork /
    FusedCriticNetwork       the reference's ActorNetwork / CriticNetwork, trained through the kernels
"""
from .env import BatchedMultiAgentEnv, make_env  # noqa: F401
from .actor import ActingTrainer, FusedActingMixin, FusedActor, FusedActorNetwork  # noqa: F401
from .networks import ActorNetwork  # noqa: F401
from .critic import FusedCritic, FusedCriticNetwork  # noqa: F401
from .replay import DeviceReplayBuffer  # noqa: F401
from .history import EpisodeHistory  # noqa: F401
from .hostpipe import HostRollout  # noqa: F401
from . import distributed  # noqa: F401

__all__ = ['make_env', 'BatchedMultiAgentEnv', 'FusedActor', 'FusedActorNetwork', 'FusedActingMixin', 'ActingTrainer',
           'ActorNetwork', 'FusedCritic', 'FusedCriticNetwork', 'DeviceReplayBuffer', 'EpisodeHistory', 'HostRollout', 'distributed']
