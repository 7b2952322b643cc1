"""prism_b200 -- B200-native learner hot path of AechPro/Prism (PER buffer + IQN/IDS update).

Product code only: every compute path calls hand-written sm_100a CUDA in lib/libprism_b200.so
through the C ABI of include/prism_b200.h.  There is no CPU fallback; the CPU oracle lives in
oracle/ and is never imported from here.
"""
from . import _lib
from .config import Config, minatar_ids_iqn_config, minatar_dqn_per_config, atari_iqn_ids_config
from .experience import (Batch, DevicePrioritizedReplayBuffer, PrioritizedTree, Timestep, TimestepBuffer,
                         TransitionRing, UniformSampler)
from .agents import Agent, FlatAdam, FlatOptimizer, FlatRMSprop, FlatSGD, action_selectors
from .agents.models import CompositeModel, FFNNModel, IQNModel, MinAtarModel, NatureAtariCnn, QEnsemble
from .factory import build_agent, build_exp_buffer, create_model

__all__ = ["Config", "minatar_ids_iqn_config", "minatar_dqn_per_config", "atari_iqn_ids_config", "Batch", "DevicePrioritizedReplayBuffer", "PrioritizedTree", "Timestep", "TimestepBuffer",
           "TransitionRing", "Agent", "FlatAdam", "FlatOptimizer", "FlatRMSprop", "FlatSGD", "action_selectors", "CompositeModel", "FFNNModel", "IQNModel",
           "MinAtarModel", "NatureAtariCnn", "QEnsemble", "UniformSampler", "build_agent", "build_exp_buffer", "create_model"]
