"""build_agent(config, obs_shape, n_actions) -> Agent: the seam of prism/factory/agent_factory.py:7-61.

Same decisions from the same config fields (target network, IDS / e-greedy / greedy acting policy, Adam / RMSprop / SGD);
what differs is what gets built: on CUDA the optimizer is a flat one (``FlatAdam`` / ``FlatRMSprop`` / ``FlatSGD``: clip +
update fused over one flat arena), and the online and target parameters are laid out in identical arenas so the target
sync is a single copy.
"""
from ..agents import Agent, action_selectors
from ..agents.optim import FlatAdam, FlatOptimizer, FlatRMSprop, FlatSGD, flatten_parameters
from . import model_factory


def _acting_policy(cfg):
    """agent_factory.py:20-38.  IDS gets the config's unsquish function; greedy and e-greedy get none (as upstream)."""
    if cfg.use_ids:
        return action_selectors.IDSActionSelector(cfg.ids_lambda, cfg.ids_use_random_samples, cfg.ids_epsilon,
                                                  cfg.ids_rho_lower_bound, cfg.ids_beta,
                                                  model_factory.squish_functions(cfg)[1])
    if cfg.use_e_greedy:
        return action_selectors.EGreedyActionSelector(cfg.e_greedy_initial_epsilon, cfg.e_greedy_final_epsilon,
                                                      cfg.e_greedy_decay_timesteps, cfg.seed)
    return action_selectors.GreedyActionSelector()


def _optimizer(cfg, model, arena):
    """agent_factory.py:40-58."""
    params = model.parameters()
    if cfg.use_adam:
        return FlatAdam(params, lr=cfg.learning_rate, betas=(cfg.adam_beta1, cfg.adam_beta2), eps=cfg.adam_epsilon,
                        max_grad_norm=cfg.max_grad_norm, arena=arena)
    if cfg.use_rmsprop:
        return FlatRMSprop(params, lr=cfg.learning_rate, alpha=cfg.rmsprop_alpha, eps=cfg.rmsprop_epsilon, centered=True,
                           max_grad_norm=cfg.max_grad_norm, arena=arena)
    return FlatSGD(params, lr=cfg.learning_rate, max_grad_norm=cfg.max_grad_norm, arena=arena)


def build_agent(config, obs_shape, n_actions):
    shape, n_actions = [int(d) for d in obs_shape], int(n_actions)
    on_cuda = "cuda" in config.device
    graphed = bool(config.use_cuda_graph) and on_cuda

    online = model_factory.create_model(shape, n_actions, config)
    arena = flatten_parameters(online) if on_cuda else None

    target = None
    if config.use_target_network:                      # a frozen twin, same arena layout as the online network
        target = model_factory.create_model(shape, n_actions, config)
        target.load_state_dict(online.state_dict())
        if on_cuda:
            flatten_parameters(target)
            for p in target.parameters():
                p.requires_grad_(False)

    optimizer = _optimizer(config, online, arena)
    if isinstance(optimizer, FlatOptimizer):
        optimizer.layout_model = online        # checkpoints in torch.optim's formats, reference parameter order
    return Agent(online, _acting_policy(config), action_selectors.GreedyActionSelector(), optimizer, target, graphed,
                 config.max_grad_norm)
