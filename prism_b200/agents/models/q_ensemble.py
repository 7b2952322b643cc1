"""QEnsemble -- K independent Q heads evaluated as ONE batched GEMM chain.

Same constructor and ``forward`` / ``get_loss`` contract as the reference
(prism/agents/models/q_ensemble.py:6-95); ``forward`` still returns (B, A, K).  The reference
loops over K ``nn.Sequential`` heads in Python (:48); here the heads' weights are stacked
parameters (K, out, in) and each layer is a single ``baddbmm`` with K as the batch dimension.
``state_dict`` stays in the reference's per-head naming (``q_heads.<k>.model.<i>.weight``) via
load/save hooks, so checkpoints are interchangeable.  The per-head double-Q target, the MSE and
its gradient are one fused kernel (pb_ens_q_loss).
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from ..squish_functions import squash_kind
from .ffnn_model import FFNNModel


class QEnsemble(nn.Module):
    def __init__(self, n_input_features, n_actions, n_heads=10, use_layer_norm=True,
                 n_model_layers=0, model_layer_size=0, model_activation=nn.ReLU,
                 q_loss_function=None, ensemble_variation_coef=0, q_loss_weight=1,
                 squish_function=None, unsquish_function=None,
                 use_double_q_learning=True, sparse_init_p=0.0, device="cpu"):
        super().__init__()
        if q_loss_function is not None and not isinstance(q_loss_function, nn.MSELoss):
            # the reference's "huber" option silently falls back to MSE (model_factory.py:43-46)
            raise NotImplementedError("only the MSE Q loss exists in the reference")
        # value squashing of the targets happens inside the loss kernel: the pair is recognised, not called
        self.squash = squash_kind(squish_function, unsquish_function)
        self.squish_function, self.unsquish_function = squish_function, unsquish_function
        self.device = device
        self.q_loss_weight = q_loss_weight
        self.use_double_q_learning = use_double_q_learning
        self.ensemble_variation_coef = ensemble_variation_coef
        self.theil = torch.tensor(0.0, device=device)
        self.n_heads = n_heads
        self.n_actions = n_actions
        self.use_layer_norm = use_layer_norm
        self.act = model_activation()

        # build K reference-shaped heads once (same init stream as the reference), then stack them
        heads = []
        for _ in range(n_heads):
            if n_model_layers > 0:
                heads.append(FFNNModel(n_input_features=n_input_features, n_output_features=n_actions,
                                       n_layers=n_model_layers, layer_width=model_layer_size,
                                       use_layer_norm=use_layer_norm, sparse_init_p=sparse_init_p,
                                       output_act_fn=None, act_fn=model_activation, device="cpu").model)
            elif use_layer_norm:
                heads.append(nn.Sequential(nn.LayerNorm(n_input_features), nn.Linear(n_input_features, n_actions)))
            else:
                heads.append(nn.Sequential(nn.Linear(n_input_features, n_actions)))
        self._bare_linear_heads = n_model_layers == 0 and not use_layer_norm
        self._ffnn_heads = n_model_layers > 0
        # layer plan: list of ("ln" | "linear" | "act", index in the head's Sequential)
        self._plan = []
        self.stacked = nn.ParameterList()
        self._slot = {}  # (seq_index, "weight"|"bias") -> position in self.stacked
        for i, mod in enumerate(heads[0]):
            if isinstance(mod, (nn.LayerNorm, nn.Linear)):
                self._plan.append(("ln" if isinstance(mod, nn.LayerNorm) else "linear", i))
                for pname in ("weight", "bias"):
                    stacked = torch.stack([getattr(h[i], pname).detach() for h in heads], dim=0)
                    self._slot[(i, pname)] = len(self.stacked)
                    self.stacked.append(nn.Parameter(stacked.to(device)))
            else:
                self._plan.append(("act", i))
        self._register_load_state_dict_pre_hook(self._from_reference_keys)
        self._register_state_dict_hook(self._to_reference_keys)

    # ---- reference-compatible state_dict ------------------------------------------------
    def _ref_key(self, k, seq_idx, pname):
        if self._ffnn_heads:
            return "q_heads.%d.model.%d.%s" % (k, seq_idx, pname)
        if self._bare_linear_heads:
            return "q_heads.%d.%s" % (k, pname)
        return "q_heads.%d.%d.%s" % (k, seq_idx, pname)

    @staticmethod
    def _to_reference_keys(module, state_dict, prefix, local_metadata):
        # head-major, each head's parameters in Sequential order: the order the reference's ModuleList of K heads
        # yields (q_ensemble.py:26-42).  Agent.serialize_model / deserialize_model and the optimizer checkpoint walk
        # state_dict order, so a reference process on the other end reads the heads in this order.
        stacked = {key: state_dict.pop("%sstacked.%d" % (prefix, pos)) for key, pos in module._slot.items()}
        for k in range(module.n_heads):
            for (seq_idx, pname), t in stacked.items():
                state_dict[prefix + module._ref_key(k, seq_idx, pname)] = t[k]
        return state_dict

    def _from_reference_keys(self, state_dict, prefix, *args):
        if (prefix + self._ref_key(0, self._plan[0][1] if self._plan[0][0] != "act" else 0, "weight")) not in state_dict:
            return
        for (seq_idx, pname), pos in self._slot.items():
            parts = [state_dict.pop(prefix + self._ref_key(k, seq_idx, pname)) for k in range(self.n_heads)]
            state_dict["%sstacked.%d" % (prefix, pos)] = torch.stack(parts, dim=0)

    def _p(self, seq_idx, pname):
        return self.stacked[self._slot[(seq_idx, pname)]]

    # ---- forward ------------------------------------------------------------------------
    def forward_heads(self, x):
        """(B, F) -> (K, B, A), head-major: what the fused loss / IDS kernels consume."""
        if not isinstance(x, torch.Tensor):
            x = torch.as_tensor(x, dtype=torch.float32, device=self.device)
        x = x.view(x.shape[0], -1)
        h = None  # (K, B, width) once the heads have diverged; x is shared before that
        plan, n, i = self._plan, len(self._plan), 0
        while i < n:
            kind, si = plan[i]
            if kind == "ln":
                w, b = self._p(si, "weight"), self._p(si, "bias")
                h = ops.layer_norm_heads(x if h is None else h, w, b)   # K heads, one launch (shared x: stats per row)
            elif kind == "linear":
                w, b = self._p(si, "weight"), self._p(si, "bias")        # (K, out, in), (K, out)
                fuse = i + 1 < n and plan[i + 1][0] == "act" and isinstance(self.act, nn.ReLU)
                h = ops.linear_heads(x if h is None else h, w, b, relu=fuse)   # one launch for all K heads
                if fuse:
                    i += 1
            else:
                h = self.act(h)
            i += 1
        return h

    def forward(self, x):
        return self.forward_heads(x).permute(1, 2, 0)                    # (B, A, K) like torch.stack(..., dim=-1)

    # ---- loss ---------------------------------------------------------------------------
    def q_tables(self, embedded_obs, embedded_next_obs, target_model=None):
        """(q_cur, q_next_online, q_next_target), head-major (K, B, A)  (:60-68)."""
        if target_model is None:
            target_model = self
        q_cur = self.forward_heads(embedded_obs)
        with torch.no_grad():
            if target_model is self:
                q_next_online = q_next_target = self.forward_heads(embedded_next_obs)
            elif self.use_double_q_learning:
                q_next_online = self.forward_heads(embedded_next_obs)
                q_next_target = target_model.forward_heads(embedded_next_obs)
            else:
                q_next_target = q_next_online = target_model.forward_heads(embedded_next_obs)
        return q_cur, q_next_online, q_next_target

    def theil_index(self):
        """Theil index of the heads' parameter L2 norms (:86-90); stacked params make it one reduction per
        tensor.  Returns None when the regulariser is off."""
        if self.ensemble_variation_coef == 0:
            return None
        params = list(self.stacked)
        if params[0].is_cuda and all(p.is_contiguous() and p.dtype == torch.float32 for p in params) and self.n_heads <= 64:
            theil = ops.theil_index(params, self.__dict__.setdefault("_theil_cache", {}))   # 3 launches incl. backward
        else:
            sq = sum(p.square().flatten(1).sum(dim=1) for p in params)
            l2_set = sq.sqrt()
            ratio = l2_set / l2_set.mean()
            theil = (ratio * torch.log(ratio)).mean()
        self.theil = theil.detach()              # logged value only: never keep an autograd graph on the module
        return theil

    def get_loss(self, embedded_obs, embedded_next_obs, batch_acts, batch_returns, dones_and_gamma, target_model=None):
        q_cur, q_next_online, q_next_target = self.q_tables(embedded_obs, embedded_next_obs, target_model)
        q_loss = ops.ensemble_q_loss(q_cur, q_next_online, q_next_target, batch_acts.view(-1), batch_returns,
                                     dones_and_gamma, loss_weight=1.0, squash=self.squash)
        theil = self.theil_index()
        if theil is None:
            return q_loss if self.q_loss_weight == 1 else self.q_loss_weight * q_loss
        return self.q_loss_weight * (q_loss - theil * self.ensemble_variation_coef)

    def log(self, logger):
        logger.log_data(data=self.theil.item(), group_name="Debug/Q Ensemble", var_name="Variation Loss")
