"""create_model(env_state_shape, env_n_actions, config) -> CompositeModel.

The seam of prism/factory/model_factory.py:49-153: an embedding network chosen by ``embedding_model_type``, an IQN
distribution head when ``use_iqn``, and a Q ensemble (K heads under IDS, one head under plain DQN), all reading the
reference's Config field names.  ``loss_squish_fn_id`` selects the (squish, unsquish) pair of
agents/squish_functions.py that both heads receive (model_factory.py passes it the same way).
"""
import torch.nn as nn

from ..agents.models import CompositeModel, FFNNModel, IQNModel, MinAtarModel, NatureAtariCnn, QEnsemble
from ..agents.squish_functions import get_squish_functions

_ACTIVATIONS = {"tanh": nn.Tanh, "gelu": nn.GELU, "sigmoid": nn.Sigmoid, "swish": nn.SiLU}     # anything else: ReLU


def _squish_id(cfg):
    sq = getattr(cfg, "loss_squish_fn_id", "none")
    # two reference configs carry a trailing comma and hold the 1-tuple ("none",) (SURVEY appendix Q9)
    return sq[0] if isinstance(sq, tuple) else sq


def squish_functions(cfg):
    """(squish, unsquish) for the config's loss_squish_fn_id; (None, None) for "none" and any unknown id."""
    return get_squish_functions(_squish_id(cfg))


def _embedding(cfg, state_shape, act):
    """model_factory.py:54-83.  The CNNs fix their own output width, which is written back into the config."""
    kind = cfg.embedding_model_type
    shared = dict(act_fn=act, device=cfg.device, sparse_init_p=cfg.sparse_init_p, use_layer_norm=cfg.use_layer_norm)
    if "ffnn" in kind:
        return FFNNModel(n_input_features=state_shape[-1], n_output_features=cfg.embedding_model_final_dim,
                         n_layers=cfg.embedding_model_num_layers, layer_width=cfg.embedding_model_layer_sizes,
                         apply_layer_norm_first_layer=False, output_act_fn=act, **shared)
    if kind == "nature_atari_cnn":
        net = NatureAtariCnn(frame_stack=cfg.frame_stack_size, feature_dim=cfg.embedding_model_final_dim, **shared)
    elif kind == "minatar_cnn":
        net = MinAtarModel(in_channels=state_shape[-1], **shared)
    else:
        return None
    cfg.embedding_model_final_dim = net.output_dim
    return net


def _q_ensemble(cfg, head_args, heads, layers, width, variation_coef):
    # q_loss_fn "huber" falls through to MSE upstream as well (model_factory.py:43-46, SURVEY appendix Q2)
    return QEnsemble(n_heads=heads, n_model_layers=layers, model_layer_size=width, q_loss_weight=cfg.q_loss_weight,
                     q_loss_function=nn.MSELoss(reduction="none"), ensemble_variation_coef=variation_coef, **head_args)


def create_model(env_state_shape, env_n_actions, config):
    cfg = config
    squish, unsquish = squish_functions(cfg)
    act = _ACTIVATIONS.get(cfg.embedding_model_act_fn_id, nn.ReLU)
    embedding = _embedding(cfg, env_state_shape, act)
    # what every head on top of the embedding shares
    head_args = dict(n_input_features=cfg.embedding_model_final_dim, n_actions=env_n_actions, model_activation=act,
                     use_layer_norm=cfg.use_layer_norm, sparse_init_p=cfg.sparse_init_p,
                     use_double_q_learning=cfg.use_double_q_learning, squish_function=squish,
                     unsquish_function=unsquish, device=cfg.device)

    distribution = None
    if cfg.use_iqn:
        # under IDS the distributional loss may be cut off from the embedding (model_factory.py:87)
        grads_reach_embedding = (not cfg.use_ids) or bool(cfg.ids_allow_distributional_gradients)
        distribution = IQNModel(n_basis_elements=cfg.iqn_n_basis_elements, n_model_layers=cfg.iqn_quantile_model_layers,
                                model_layer_size=cfg.iqn_quantile_model_feature_dim, huber_k=cfg.iqn_huber_loss_kappa,
                                distributional_loss_weight=cfg.distributional_loss_weight,
                                n_current_quantile_samples=cfg.iqn_n_current_state_quantile_samples,
                                n_next_quantile_samples=cfg.iqn_n_next_state_quantile_samples,
                                n_quantile_samples_per_action=cfg.iqn_quantile_samples_per_action,
                                propagate_grad=grads_reach_embedding, **head_args)

    q_function = None
    if cfg.use_ids:
        q_function = _q_ensemble(cfg, head_args, cfg.ids_n_q_heads, cfg.ids_n_q_head_model_layers,
                                 cfg.ids_q_head_feature_dim, cfg.ids_ensemble_variation_coef)
    elif cfg.use_dqn:
        q_function = _q_ensemble(cfg, head_args, 1, cfg.dqn_n_model_layers, cfg.dqn_n_model_feature_dim, 0)

    return CompositeModel(embedding_model=embedding, distribution_model=distribution, q_function_model=q_function,
                          device=cfg.device, use_cuda_graph=bool(cfg.use_cuda_graph) and "cuda" in cfg.device)
