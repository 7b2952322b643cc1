"""Action selectors with the reference's interface (prism/agents/action_selectors.py):
``generate_action_probs(z, q) -> one-hot (N, A)`` and ``select_action(probs) -> int64 (N,)``.
IDS and greedy selection are single fused kernels (pb_ids_select / pb_greedy_select)."""
import numpy as np
import torch

from . import ops
from .squish_functions import unsquash_kind


class ActionSelector(object):
    def __init__(self, logger=None):
        self.logger = logger
        self.loggables = {}

    def generate_action_probs(self, *args, **kwargs):
        raise NotImplementedError

    def select_action(self, action_probs):
        raise NotImplementedError

    def save(self, path):
        pass

    def load(self, path):
        pass

    def log(self, logger, action_value_distribution, q_estimates):
        pass


def _head_major(q_estimates):
    """(N, A, K) -> contiguous (K, N, A).  QEnsemble.forward returns a permuted view of a head-major
    tensor, so this is normally free."""
    return q_estimates.permute(2, 0, 1)


class GreedyActionSelector(ActionSelector):
    """argmax_a mean_k q (action_selectors.py:70-82)."""

    def generate_action_probs(self, action_value_distribution, q_estimates):
        action = ops.greedy_select(_head_major(q_estimates))
        return torch.nn.functional.one_hot(action, q_estimates.shape[1])

    def select_action(self, action_probs):
        return torch.argmax(action_probs, dim=-1).long().view(-1)


class LinearAnneal(object):
    """Linear schedule advanced by the number of rows seen (prism/util/annealing_strategies.py:22-33):
    value = start*(1-a) + stop*a with a = step/max_steps, pinned to `stop` once step >= max_steps."""

    def __init__(self, start_value, stop_value, max_steps):
        self.start, self.stop, self.max_steps = start_value, stop_value, max_steps
        self.current_step = 0

    def get_value(self):
        if self.max_steps == 0 or self.current_step >= self.max_steps:
            return self.stop
        a = min(1, self.current_step / self.max_steps)
        return self.start * (1 - a) + self.stop * a

    def update(self, n_steps):
        self.current_step += n_steps
        return self.get_value()

    def get_state(self):
        return self.current_step

    def set_state(self, state):
        self.current_step = state


class EGreedyActionSelector(ActionSelector):
    """One host coin flip per *call* (not per row), numpy RandomState(seed) (action_selectors.py:25-67)."""

    def __init__(self, e_start, e_stop, anneal_time, seed=123):
        super().__init__()
        self.epsilon = LinearAnneal(start_value=e_start, stop_value=e_stop, max_steps=anneal_time)
        self.greedy = GreedyActionSelector()
        self.rng = np.random.RandomState(seed)

    def generate_action_probs(self, action_value_distribution, q_estimates):
        n_timesteps, n_actions, _ = q_estimates.shape
        if self.rng.uniform(0, 1) < self.epsilon.update(n_timesteps):
            action = torch.as_tensor(self.rng.randint(n_actions, size=(n_timesteps,)), dtype=torch.long)
            return torch.nn.functional.one_hot(action, n_actions).to(q_estimates.device)
        return self.greedy.generate_action_probs(action_value_distribution, q_estimates)

    def select_action(self, action_probs):
        return torch.argmax(action_probs, dim=-1)

    def save(self, path):
        import os
        with open(os.path.join(path, "epsilon.txt"), "w") as f:
            f.write(str(self.epsilon.get_state()) + "\n")

    def load(self, path):
        import os
        eps_path = os.path.join(path, "epsilon.txt")
        if os.path.exists(eps_path):
            with open(eps_path) as f:
                self.epsilon.set_state(int(f.readlines()[0]))

    def log(self, logger, action_value_distribution, q_estimates):
        logger.log_data(data=self.epsilon.get_value(), group_name="Report/Action Selector", var_name="Epsilon")


class IDSActionSelector(ActionSelector):
    """Information-directed sampling, deterministic branch (action_selectors.py:114-176).

    Reproduces the reference's naming quirk: the ensemble "variance" is torch.std and its "std"
    is sqrt(std) (SURVEY appendix Q1).  With an unsquish function (squish_functions.py) every q and z value is read
    through it, inside the selection kernel."""

    squash = 0              # PB_SQUASH_NONE; also what a selector pickled before value squashing existed reads

    def __init__(self, lmbda, random_sample, epsilon, ids_rho_lower_bound, beta, unsquish_function=None):
        super().__init__()
        if random_sample:
            raise NotImplementedError("ids_use_random_samples=True is not used by any reference config")
        # every q and z value is unsquashed inside the selection kernel: the function is recognised, not called
        self.squash = unsquash_kind(unsquish_function)
        self.unsquish_function = unsquish_function
        self.random_sample = random_sample
        self.beta = beta
        self.lmbda = lmbda
        self.epsilon = epsilon
        self.ids_rho_lower_bound = ids_rho_lower_bound

    def generate_action_probs(self, action_value_distribution, q_estimates, for_log=False):
        out = ops.ids_select(_head_major(q_estimates), action_value_distribution, self.lmbda, self.epsilon,
                             self.ids_rho_lower_bound, return_scores=for_log, squash=self.squash)
        action, scores = out if for_log else (out, None)
        probs = torch.nn.functional.one_hot(action, q_estimates.shape[1])
        if for_log:
            self.loggables["IDS Scores"] = scores
            self.loggables["Action Probs"] = probs
        return probs

    def select_action(self, action_probs):
        return action_probs.argmax(dim=-1).long().view(-1)

    def log(self, logger, action_value_distribution, q_estimates):
        self.generate_action_probs(action_value_distribution, q_estimates, for_log=True)
        for key, value in self.loggables.items():
            if isinstance(value, torch.Tensor):
                value = [[round(v, 4) for v in row] for row in value.float().tolist()]
                if len(value) == 1:
                    value = value[0]
            logger.log_data(data=value, group_name="Debug/IDS", var_name=key)
