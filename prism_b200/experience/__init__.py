from .timestep import Timestep
from .batch import Batch
from .per import PrioritizedTree
from .ring import TransitionRing
from .timestep_buffer import TimestepBuffer, DevicePrioritizedReplayBuffer
from .uniform import UniformSampler
