from .agent import Agent
from . import action_selectors
from .optim import FlatAdam, FlatOptimizer, FlatRMSprop, FlatSGD, flatten_parameters
