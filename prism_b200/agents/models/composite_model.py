"""CompositeModel -- embedding -> {IQN head, Q ensemble}; builds the per-row losses and the new
PER priorities.  Same surface as the reference (prism/agents/models/composite_model.py:7-154):
``forward(x, for_action=True) -> (q (N,A,K), z (Nq,N,A))``, ``get_losses(batch, target_model) ->
(dist (B,), q (B,), td (B,))``, attributes ``embedding_model / distribution_model /
q_function_model / device / should_build_forward_cuda_graph``.
"""
import numpy as np
import torch
import torch.nn as nn

from .. import ops
from .iqn_model import IQNModel


class CompositeModel(nn.Module):
    def __init__(self, embedding_model, distribution_model, q_function_model, device="cpu", use_cuda_graph=False):
        super().__init__()
        self.embedding_model = embedding_model
        self.distribution_model = distribution_model
        self.q_function_model = q_function_model
        self.device = device
        self.use_cuda_graph = use_cuda_graph
        self.should_build_forward_cuda_graph = use_cuda_graph
        self._forward_cuda_graph = None
        self._static_input = None
        self._static_q = None
        self._static_z = None
        self.loggables = {}

    # ---- acting ---------------------------------------------------------------------
    def forward(self, x, for_action=True):
        if not isinstance(x, torch.Tensor):
            x = torch.from_numpy(np.asarray(x, dtype=np.float32))
        x = x.float().to(self.device)
        if for_action and self.use_cuda_graph:
            return self._forward_with_cuda_graph(x)
        return self._forward_without_cuda_graph(x, for_action=for_action)

    def _forward_without_cuda_graph(self, x, for_action=True):
        emb = self.embedding_model(x) if self.embedding_model is not None else x
        z = self.distribution_model(emb, for_action=for_action) if self.distribution_model is not None else None
        if self.q_function_model is not None:
            q = self.q_function_model(emb)
        elif for_action and type(self.distribution_model) is IQNModel:
            q = z.mean(dim=0).unsqueeze(-1)
        else:
            q = None
        return q, z

    @torch.no_grad()
    def _forward_with_cuda_graph(self, x):
        if self._forward_cuda_graph is None or self._static_input.shape != x.shape:
            if not self.should_build_forward_cuda_graph:
                return self._forward_without_cuda_graph(x)
            self._build_forward_cuda_graph(x)
        self._static_input.copy_(x)
        self._forward_cuda_graph.replay()
        q = None if self._static_q is None else self._static_q.clone()
        z = None if self._static_z is None else self._static_z.clone()
        return q, z

    @torch.no_grad()
    def _build_forward_cuda_graph(self, x):
        self._static_input = x.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                self._forward_without_cuda_graph(self._static_input, for_action=True)
        torch.cuda.current_stream().wait_stream(side)
        self._forward_cuda_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._forward_cuda_graph):
            self._static_q, self._static_z = self._forward_without_cuda_graph(self._static_input, for_action=True)

    # ---- learning -------------------------------------------------------------------
    def get_losses(self, batch, target_model):
        obs = batch["observation"]
        next_obs = batch["next"]["observation"]
        if obs.shape[1] == 1:                      # frame_stack == 1: drop the stack axis (:97-99)
            obs = obs.squeeze(1)
            next_obs = next_obs.squeeze(1)
        returns = batch["next"]["reward"].flatten()
        nonterminal = batch["nonterminal"].flatten().float()
        gammas = batch["gamma"].flatten().float()
        act = batch["action"]
        if act.dim() == 2 and act.shape[-1] != 1:
            act = act.argmax(dim=-1)
        acts = act.flatten().long()
        dones_and_gamma = gammas * nonterminal

        emb = self.embedding_model(obs)
        with torch.no_grad():
            if target_model is not None:
                emb_next = target_model.embedding_model(next_obs)
                dist_target, q_target = target_model.distribution_model, target_model.q_function_model
            else:
                emb_next = self.embedding_model(next_obs)
                dist_target = q_target = None

        dist_loss = q_loss = td = None
        if self.distribution_model is not None:
            dist_loss = self.distribution_model.get_loss(emb, emb_next, acts, returns, dones_and_gamma,
                                                         target_model=dist_target)
        if self.q_function_model is not None:
            q_loss = self.q_function_model.get_loss(emb, emb_next, acts, returns, dones_and_gamma,
                                                    target_model=q_target)
        if dist_loss is not None or q_loss is not None:
            with torch.no_grad():
                _, td = ops.loss_combine(None if dist_loss is None else dist_loss.detach(),
                                         None if q_loss is None else q_loss.detach(), None)
        return dist_loss, q_loss, td

    def _side_streams(self, device):
        return ops.fork_stream(device, "boot1"), ops.fork_stream(device, "boot2")

    def losses_total(self, batch, target_model, per_weights=None):
        """get_losses + the PER-weighted total of Agent.update (agent.py:58-64) as one fused head:
        returns (dist_loss, q_loss, total, td).  Same math as get_losses followed by
        mean(dist*w) + mean(q*w); the bootstrap factor gamma^k * nonterminal, both loss heads, the TD mix
        and the gradients w.r.t. the network outputs come out of three launches."""
        obs = batch["observation"]
        next_obs = batch["next"]["observation"]
        if obs.shape[1] == 1:
            obs, next_obs = obs.squeeze(1), next_obs.squeeze(1)
        returns = batch["next"]["reward"].flatten()
        gamma = batch["gamma"].flatten()
        nonterm = batch["nonterminal"].flatten()
        act = batch["action"]
        if act.dim() == 2 and act.shape[-1] != 1:
            act = act.argmax(dim=-1)
        acts = act.flatten()
        if nonterm.dtype != torch.bool:
            gamma, nonterm = gamma.float() * nonterm.float(), None

        iqn, ens = self.distribution_model, self.q_function_model
        if iqn is None and ens is None:
            return None, None, None, None
        tgt = target_model if target_model is not None else self
        iqn_t, ens_t = tgt.distribution_model, tgt.q_function_model
        z_cur = tau = z_on = z_tg = q_cur = q_on = q_tg = None
        T = Tp = 0
        kappa = dist_w = q_w = 1.0
        if iqn is not None:
            T, Tp, kappa, dist_w = (iqn.n_current_quantile_samples, iqn.n_next_quantile_samples, iqn.huber_k,
                                    iqn.distributional_loss_weight)
        # which next-state passes exist (iqn_model.py:110-126, q_ensemble.py:62-68)
        iqn_online_next = iqn is not None and (tgt is self or iqn.use_double_q_learning)
        ens_online_next = ens is not None and (tgt is self or ens.use_double_q_learning)

        # The bootstrap passes (no_grad) are independent of the online pass on the current observations:
        # they run on side streams -- parallel branches of the captured graph -- and join before the loss.
        cur = torch.cuda.current_stream(obs.device)
        s1, s2 = self._side_streams(obs.device)
        self._keepalive = keep = []          # side-stream tensors stay referenced until the next call
        s1.wait_stream(cur)
        with torch.cuda.stream(s1), torch.no_grad():
            emb_next = tgt.embedding_model(next_obs)
            emb_ready = torch.cuda.Event()
            emb_ready.record(s1)
            if tgt is not self:
                if iqn is not None:
                    z_tg = iqn_t.forward(emb_next, n_quantile_samples=Tp)[0]
                if ens is not None:
                    q_tg = ens_t.forward_heads(emb_next)
            ops.trace_mark("boot:target_next_done")
        emb = self.embedding_model(obs)
        ops.trace_mark("fwd:embedded")
        if iqn is not None:
            z_cur, tau = iqn.forward(emb, n_quantile_samples=T)
        if ens is not None:
            q_cur = ens.forward_heads(emb)
        ops.trace_mark("fwd:heads_done")
        if iqn_online_next or ens_online_next:
            s2.wait_event(emb_ready)
            with torch.cuda.stream(s2), torch.no_grad():
                if iqn_online_next:
                    z_on = iqn.forward(emb_next, n_quantile_samples=Tp)[0]
                if ens_online_next:
                    q_on = ens.forward_heads(emb_next)
                ops.trace_mark("boot:online_next_done")
            cur.wait_stream(s2)
        cur.wait_stream(s1)
        if iqn is not None:
            z_tg = z_on if z_tg is None else z_tg
            z_on = z_tg if z_on is None else z_on
        if ens is not None:
            q_tg = q_on if q_tg is None else q_tg
            q_on = q_tg if q_on is None else q_on
        keep.extend(t for t in (emb_next, z_on, z_tg, q_on, q_tg) if t is not None)
        theil = None
        if ens is not None:
            q_w = ens.q_loss_weight
            theil = ens.theil_index()
        w = per_weights if isinstance(per_weights, torch.Tensor) else None
        off = None if theil is None else (theil.detach() * ens.ensemble_variation_coef).float()
        total, dist, mse, td = ops.fused_total_loss(z_cur, q_cur, tau, z_on, z_tg, q_on, q_tg, acts, returns, gamma,
                                                    nonterm, w, off, T, Tp, kappa, dist_w, q_w,
                                                    dist_squash=iqn.squash if iqn is not None else 0,
                                                    q_squash=ens.squash if ens is not None else 0)
        if theil is not None:
            # the regulariser's own gradient: d total / d theil = -q_w * coef * mean(w)
            mean_w = w.mean() if w is not None else 1.0
            total = total + (theil - theil.detach()) * (-(q_w * ens.ensemble_variation_coef) * mean_w)
        if w is None and not isinstance(per_weights, torch.Tensor) and per_weights not in (None, 1):
            total = total * per_weights
        return (dist if iqn is not None else None), (mse if ens is not None else None), total, td

    def log(self, logger):
        for m in (self.embedding_model, self.distribution_model, self.q_function_model):
            if m is not None:
                m.log(logger)
