"""ma_league_b200: B200 (sm_100a) implementation of ma-league's value-decomposition hot path behind the reference's
Python API.  Sub-packages mirror the reference's `marl.*` layout:

    marl.components.episode_batch / replay_buffers / action_selectors / transforms / epsilon_schedules
    marl.controllers (BasicMAC)   marl.learners (QLearner)   marl.modules.agents / mixers
"""
from . import _native
from .components.episode_batch import EpisodeBatch
from .components.replay_buffers import ReplayBuffer, PrioritizedReplayBuffer
from .components.transforms import OneHot
from .components.action_selectors import EpsilonGreedyActionSelector, REGISTRY as action_REGISTRY
from .controllers import BasicMAC, EnsembleMAC, REGISTRY as mac_REGISTRY
from .learners import QLearner, REGISTRY as learner_REGISTRY
from .modules.agents import DRQNAgentNetwork, DQNAgentNetwork, REGISTRY as agent_REGISTRY
from .modules.mixers import QMixer, VDNMixer

__all__ = ["EpisodeBatch", "ReplayBuffer", "PrioritizedReplayBuffer", "OneHot", "EpsilonGreedyActionSelector", "BasicMAC", "QLearner",
           "EnsembleMAC", "DRQNAgentNetwork", "DQNAgentNetwork", "QMixer", "VDNMixer", "mac_REGISTRY", "learner_REGISTRY", "agent_REGISTRY",
           "action_REGISTRY"]
