"""IQNModel -- implicit quantile network head, device-native.

Constructor, ``forward`` / ``get_loss`` signatures, parameter names and the order of the
random tau draws follow the reference (prism/agents/models/iqn_model.py:6-201), so weights
and seeds carry over.  Differences underneath:
  * the cos(pi*i*tau) basis comes from one kernel (pb_iqn_cos_basis) instead of tile+mul+cos;
  * phi(tau) (.) x is a broadcast over the quantile axis, the (n*B, F) tiled copy of the state
    embedding the reference materialises with torch.tile (:70) never exists;
  * target construction, the pairwise tau x tau' quantile-Huber loss and its gradient are one
    fused warp-per-row kernel (pb_iqn_qh_loss) instead of ~30 ATen kernels and 6 B*T'*T temporaries.
Dense layers go through ops.linear / ops.phi_times_x: tcgen05 3xTF32 GEMMs for the (T*B)-row layers (the
phi(tau) (.) x product fused into the GEMM epilogue), the fp32 FFMA cluster kernel for small ones.
"""
import numpy as np
import torch
import torch.nn as nn

from .. import ops
from ..squish_functions import squash_kind
from .ffnn_model import FFNNModel


class IQNModel(nn.Module):
    def __init__(self, n_input_features, n_actions, n_basis_elements, use_layer_norm,
                 n_model_layers=0, model_layer_size=0, model_activation=nn.ReLU,
                 squish_function=None, unsquish_function=None, huber_k=1.0,
                 n_current_quantile_samples=8, n_next_quantile_samples=8,
                 n_quantile_samples_per_action=200, use_double_q_learning=True,
                 distributional_loss_weight=1, sparse_init_p=0.0,
                 propagate_grad=True, risk_policy=None, device="cpu"):
        super().__init__()
        if risk_policy is not None:
            # every BASELINE config runs the neutral risk policy (SURVEY 2 row 9)
            raise NotImplementedError("risk policies are outside the hot-path scope")
        # value squashing of the targets happens inside the loss kernel: the pair is recognised, not called
        self.squash = squash_kind(squish_function, unsquish_function)
        self.squish_function, self.unsquish_function = squish_function, unsquish_function
        self.device = device
        self.n_actions = n_actions
        self.n_basis_elements = n_basis_elements
        self.distributional_loss_weight = distributional_loss_weight
        self.propagate_grad = propagate_grad
        self.n_current_quantile_samples = n_current_quantile_samples
        self.n_next_quantile_samples = n_next_quantile_samples
        self.n_quantile_samples_per_action = n_quantile_samples_per_action
        self.huber_k = huber_k
        self.use_double_q_learning = use_double_q_learning

        self.phi = nn.Sequential(nn.Linear(n_basis_elements, n_input_features), nn.ReLU()).to(device)
        self.model = None
        width = n_input_features
        if n_model_layers > 0:
            self.model = FFNNModel(n_input_features=n_input_features, n_output_features=model_layer_size,
                                   n_layers=n_model_layers, layer_width=model_layer_size,
                                   use_layer_norm=use_layer_norm, output_act_fn=model_activation,
                                   act_fn=model_activation, device=device, sparse_init_p=sparse_init_p)
            width = model_layer_size
        if use_layer_norm:
            self.embedding_to_quantile_layer = nn.Sequential(nn.LayerNorm(width), nn.Linear(width, n_actions)).to(device)
        else:
            self.embedding_to_quantile_layer = nn.Linear(width, n_actions, device=device)
        # injected quantile draws, consumed in call order (parity tests replay the reference's torch.rand
        # stream through this; production draws from the device Philox generator)
        self.tau_queue = []
        # static quantile buffers (set_static_taus): device tensors every learning forward reads, in call order --
        # how a CAPTURED update graph is fed chosen draws (a Python queue cannot be popped per replay)
        self._static_taus = []
        self._static_call = 0

    def set_static_taus(self, taus):
        """Pin the quantile draws of the learning forwards to these device tensors, consumed cyclically in call order
        (current, next-online | next-target: iqn_model.py:104-126).  Calling it again with the same shapes copies IN
        PLACE, so a captured graph sees the new values on its next replay.  ``None`` / [] returns to random draws."""
        taus = [] if taus is None else [t.to(self.device).float().reshape(-1, 1) for t in taus]
        if len(taus) == len(self._static_taus) and all(a.shape == b.shape for a, b in zip(taus, self._static_taus)):
            for dst, src in zip(self._static_taus, taus):
                dst.copy_(src)
        else:
            self._static_taus = [t.clone() for t in taus]
        self._static_call = 0

    # ------------------------------------------------------------------
    def forward(self, x, n_quantile_samples=None, for_action=False, static_quantiles=None):
        if not isinstance(x, torch.Tensor):
            x = torch.from_numpy(np.asarray(x, dtype=np.float32))
        x = x.float().to(self.device)
        if not self.propagate_grad:
            x = x.detach()
        x = x.view(x.shape[0], -1)
        n_rows = x.shape[0]
        if for_action:
            n_quantile_samples = self.n_quantile_samples_per_action
        n = int(n_quantile_samples)

        if static_quantiles is not None:
            quantiles = static_quantiles
        elif self.tau_queue:
            quantiles = self.tau_queue.pop(0).to(self.device).float().view(n * n_rows, 1)
        elif self._static_taus and not for_action:
            quantiles = self._static_taus[self._static_call % len(self._static_taus)]
            self._static_call += 1
            if quantiles.numel() != n * n_rows:
                raise ValueError("static quantiles hold %d draws, this forward needs %d" % (quantiles.numel(), n * n_rows))
        else:
            quantiles = None

        if quantiles is None:
            # same shape and dtype as the reference draw (:64-66), drawn by this library's Philox generator in the
            # same launch that builds the cosine basis (seeded from torch's seed at first use)
            quantiles, basis = ops.draw_cos_basis(n * n_rows, self.n_basis_elements, self._rng_state())
        else:
            basis = ops.cos_basis(quantiles, self.n_basis_elements)        # (n*rows, n_basis)
        # phi(tau) (.) x with quantile-major rows (r = q*rows + b): the state embedding is broadcast over q inside
        # the phi GEMM's epilogue (large layers) or by a broadcasting multiply (small ones)
        h = ops.phi_times_x(self.phi, basis, x, n)
        if self.model is not None:
            h = self.model(h)
        head = self.embedding_to_quantile_layer
        z = ops.run_sequential(head, h) if isinstance(head, nn.Sequential) else ops.linear(h, head.weight, head.bias)
        if for_action:
            return z.view(n, -1, self.n_actions)
        return z, quantiles

    def _rng_state(self):
        rng = getattr(self, "_rng", None)
        if rng is None or rng.device != torch.device(self.device):
            IQNModel._n_generators = getattr(IQNModel, "_n_generators", 0) + 1
            seed = (torch.initial_seed() * 2654435761 + IQNModel._n_generators * 40503) & 0x7FFFFFFF
            rng = self._rng = torch.tensor([seed, 0, 0, 0], dtype=torch.int64, device=self.device)
        return rng

    def _embed_quantiles(self, quantiles):
        return ops.run_sequential(self.phi, ops.cos_basis(quantiles, self.n_basis_elements))

    # ------------------------------------------------------------------
    def quantile_tables(self, embedded_obs, embedded_next_obs, target_model=None):
        """(z_cur, tau, z_next_online, z_next_target): the three forward passes of get_loss, in the
        reference's draw order -- tau (current), tau' (online next), tau' (target next)  (:104-126)."""
        if not self.propagate_grad:
            embedded_obs = embedded_obs.detach()
            embedded_next_obs = embedded_next_obs.detach()
        if target_model is None:
            target_model = self
        T, Tp = self.n_current_quantile_samples, self.n_next_quantile_samples
        z_cur, tau = self.forward(embedded_obs, n_quantile_samples=T)
        with torch.no_grad():
            if target_model is self:
                z_next_online = self.forward(embedded_next_obs, n_quantile_samples=Tp)[0]
                z_next_target = z_next_online
            elif self.use_double_q_learning:
                z_next_online = self.forward(embedded_next_obs, n_quantile_samples=Tp)[0]
                z_next_target = target_model.forward(embedded_next_obs, n_quantile_samples=Tp)[0]
            else:
                z_next_target = target_model.forward(embedded_next_obs, n_quantile_samples=Tp)[0]
                z_next_online = z_next_target
        return z_cur, tau, z_next_online, z_next_target

    def get_loss(self, embedded_obs, embedded_next_obs, batch_acts, batch_returns, dones_and_gamma, target_model=None):
        z_cur, tau, z_next_online, z_next_target = self.quantile_tables(embedded_obs, embedded_next_obs, target_model)
        return ops.quantile_huber_loss(z_cur, tau, z_next_online, z_next_target, batch_acts, batch_returns,
                                       dones_and_gamma, self.n_current_quantile_samples,
                                       self.n_next_quantile_samples, kappa=self.huber_k,
                                       loss_weight=self.distributional_loss_weight, squash=self.squash)

    def log(self, logger):
        pass
