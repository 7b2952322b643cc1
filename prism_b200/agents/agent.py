"""Agent -- acting forward, the learner update step, target sync, (de)serialisation.

Same constructor and methods as the reference (prism/agents/agent.py:7-264).  The update step is
    get_losses -> PER-weighted total -> backward -> clip_grad_norm_ -> Adam / RMSprop / SGD
with the loss heads, the loss combine and clip + update running as fused libprism_b200 kernels, and
the whole step captured in ONE CUDA graph when ``use_cuda_graph`` is set.

Deliberate deviations from the reference (SURVEY appendix Q3):
  * the captured graph bootstraps from the *target* network like the eager path does (the
    reference's capture passes ``self.model`` as the target, agent.py:135-136, silently disabling
    the target net on GPU);
  * graph warm-up iterations do not mutate the weights or the optimiser state (the reference's
    three warm-up iterations are real optimiser steps on the first batch, agent.py:111-127).
"""
import os
import pickle

import numpy as np
import torch

from . import ops
from .action_selectors import GreedyActionSelector, IDSActionSelector
from .optim import FlatOptimizer


class Agent(object):
    def __init__(self, model, action_selector, eval_action_selector, optimizer, target_model,
                 use_cuda_graph, max_grad_norm):
        self.model, self.target_model, self.optimizer = model, target_model, optimizer
        self.action_selector, self.eval_action_selector = action_selector, eval_action_selector
        self.max_grad_norm, self.use_cuda_graph = max_grad_norm, use_cuda_graph
        self.n_updates, self._is_eval = 0, False
        if isinstance(optimizer, FlatOptimizer):
            optimizer.max_grad_norm = float(max_grad_norm) if max_grad_norm else 0.0
        # static tensors of the captured update (names as upstream: learner.py and the logger read them)
        for name in ("per_weights", "distribution_loss", "q_loss", "total_loss", "new_per_weights", "batch"):
            setattr(self, "_static_" + name, None)
        self._learn_cuda_graph = None
        self.model.train()

    # ---- acting -------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, obs):
        selector = self.eval_action_selector if self._is_eval else self.action_selector
        if self.use_cuda_graph and type(selector) in (IDSActionSelector, GreedyActionSelector):
            act = self._forward_acting_graph(obs, selector)
            if act is not None:
                return act
        q, z = self.model(obs, for_action=True)
        return selector.select_action(selector.generate_action_probs(z, q))

    @torch.no_grad()
    def _forward_acting_graph(self, obs, selector):
        """The whole acting path of prism/agents/agent.py:31-41 -- embedding, IQN with Nq quantile samples, K Q heads and
        the IDS / greedy selection kernel -- as ONE CUDA graph per (selector, input shape): one staging copy in, one
        replay, the action vector out.  Only selectors that live entirely on the device are captured (epsilon-greedy
        flips a host coin per call and stays eager)."""
        model = self.model
        dev = torch.device(getattr(model, "device", "cpu"))
        if dev.type != "cuda" or not hasattr(model, "_forward_without_cuda_graph"):
            return None
        if not isinstance(obs, torch.Tensor):
            obs = torch.from_numpy(np.asarray(obs, dtype=np.float32))
        key = (id(selector), tuple(obs.shape))
        graphs = self.__dict__.setdefault("_acting_graphs", {})
        entry = graphs.get(key)
        if entry is None:
            if len(graphs) >= 8:                       # a handful of inference batch shapes at most
                return None
            static_in = torch.zeros(obs.shape, dtype=torch.float32, device=dev)
            static_in.copy_(obs)

            def body():
                q, z = model._forward_without_cuda_graph(static_in, for_action=True)
                return selector.select_action(selector.generate_action_probs(z, q))
            d = getattr(model, "distribution_model", None)
            if d is not None and hasattr(d, "_rng_state"):
                d._rng_state()
            q_rng = self.quantile_rng_snapshot()               # warm-up and capture must not consume quantile draws
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    body()
            torch.cuda.current_stream(dev).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                static_out = body()
            self.quantile_rng_restore(q_rng)
            entry = graphs[key] = (g, static_in, static_out)
        g, static_in, static_out = entry
        static_in.copy_(obs, non_blocking=True)
        g.replay()
        return static_out.clone()

    # ---- device generators of the IQN heads (quantile draws): graph warm-ups must not advance them --------------
    def quantile_rng_snapshot(self):
        out = []
        for m in (self.model, self.target_model):
            d = getattr(m, "distribution_model", None) if m is not None else None
            rng = getattr(d, "_rng", None) if d is not None else None
            if rng is not None:
                out.append((rng, rng.clone()))
        return out

    @staticmethod
    def quantile_rng_restore(snap):
        for rng, saved in snap:
            rng.copy_(saved)

    # ---- learning -----------------------------------------------------------------------
    def update(self, batch, per_weights=1):
        self.train()
        step = self._update_with_cuda_graph if self.use_cuda_graph else self._update_without_cuda_graph
        td = step(batch, per_weights)
        self.n_updates += 1
        return td

    def _loss_and_backward(self, batch, per_weights, target_model, after_loss=None):
        """``after_loss(td)``: called once the losses / new priorities exist and before the backward pass starts
        (LearnerStep forks the priority write-back onto a parallel graph branch there)."""
        if hasattr(self.model, "losses_total"):
            # fused head: loss kernels emit PER-weighted gradients directly (agent.py:58-64 folded in)
            dist_loss, q_loss, total, td = self.model.losses_total(batch, target_model, per_weights)
            if total is None:
                return None, None, None, 0
        else:
            dist_loss, q_loss, td = self.model.get_losses(batch, target_model)
            if dist_loss is None and q_loss is None:
                return None, None, None, 0
            w = per_weights if isinstance(per_weights, torch.Tensor) else None
            total, _ = ops.loss_combine(dist_loss, q_loss, w)   # mean(dist*w) + mean(q*w)  (agent.py:58-64)
            if w is None and per_weights != 1:
                total = total * per_weights
        if after_loss is not None:
            after_loss(td)
        self.optimizer.zero_grad(set_to_none=True)
        if total.is_cuda and total.dim() == 0 and total.dtype == torch.float32:
            ops.UNIT_TOTAL_GRAD = True          # the fused loss head then hands its saved gradients through unscaled
            try:
                total.backward(gradient=ops.unit_gradient(total.device))
            finally:
                ops.UNIT_TOTAL_GRAD = False
        else:
            total.backward()
        return dist_loss, q_loss, total, td

    def _optimizer_step(self, refresh_table=True):
        if isinstance(self.optimizer, FlatOptimizer):
            self.optimizer.step(refresh_table=refresh_table)     # clip + update fused
        else:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.max_grad_norm)
            self.optimizer.step()

    def _update_without_cuda_graph(self, batch, per_weights=1):
        dist_loss, q_loss, total, td = self._loss_and_backward(batch, per_weights, self.target_model)
        if total is None:
            return 0
        self._static_distribution_loss, self._static_q_loss, self._static_total_loss = dist_loss, q_loss, total
        self._optimizer_step()
        return td

    def _update_with_cuda_graph(self, batch, per_weights=1):
        if self._learn_cuda_graph is None:
            self._build_update_cuda_graph(batch, per_weights)
        if batch is not self._static_batch:
            sb = self._static_batch
            sb["observation"].copy_(batch["observation"])
            sb["next"]["observation"].copy_(batch["next"]["observation"])
            sb["next"]["reward"].copy_(batch["next"]["reward"])
            sb["action"].copy_(batch["action"])
            sb["nonterminal"].copy_(batch["nonterminal"])
            sb["gamma"].copy_(batch["gamma"])
        if isinstance(per_weights, torch.Tensor) and per_weights.data_ptr() != self._static_per_weights.data_ptr():
            self._static_per_weights.copy_(per_weights)
        self._learn_cuda_graph.replay()
        return self._static_new_per_weights

    def _build_update_cuda_graph(self, batch, per_weights=1):
        self._static_batch = batch
        dev = batch.device if hasattr(batch, "device") else batch["observation"].device
        B = batch["observation"].shape[0]
        if isinstance(per_weights, torch.Tensor):
            self._static_per_weights = per_weights.clone()
        else:
            self._static_per_weights = torch.full((B,), float(per_weights), dtype=torch.float32, device=dev)

        flat = isinstance(self.optimizer, FlatOptimizer)
        snap = self.optimizer.snapshot() if flat else None
        # no autograd graph from an earlier (eager, other-stream) update may stay alive across the capture
        self._static_total_loss = self._static_distribution_loss = self._static_q_loss = None
        self.optimizer.zero_grad(set_to_none=True)
        rng_state = torch.cuda.get_rng_state(dev)
        for m in (self.model, self.target_model):              # make the IQN generators exist before they are snapshotted
            d = getattr(m, "distribution_model", None) if m is not None else None
            if d is not None and hasattr(d, "_rng_state"):
                d._rng_state()
        q_rng = self.quantile_rng_snapshot()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                self._loss_and_backward(self._static_batch, self._static_per_weights, self.target_model)
                self._optimizer_step()
        torch.cuda.current_stream().wait_stream(side)
        if flat:
            self.optimizer.restore(snap)                         # warm-up must not train
        torch.cuda.set_rng_state(rng_state, dev)
        self.quantile_rng_restore(q_rng)

        self._learn_cuda_graph = torch.cuda.CUDAGraph()
        self.optimizer.zero_grad(set_to_none=True)
        with torch.cuda.graph(self._learn_cuda_graph):
            dl, ql, total, td = self._loss_and_backward(self._static_batch, self._static_per_weights,
                                                        self.target_model)
            self._static_distribution_loss, self._static_q_loss = dl, ql
            self._static_total_loss, self._static_new_per_weights = total, td
            self._optimizer_step(refresh_table=False)
        if flat:
            self.optimizer.refresh_grad_table()                  # gradient addresses are static from here on

    @torch.no_grad()
    def sync_target_model(self):
        src, dst = self.model, self.target_model
        fa, fb = getattr(src, "_flat_arena", None), getattr(dst, "_flat_arena", None)
        if fa is not None and fb is not None and fa.numel() == fb.numel():
            fb.copy_(fa)                                         # one device copy (agent.py:149-152 loops)
            return
        for p1, p2 in zip(src.parameters(), dst.parameters()):
            p2.data.copy_(p1.data)

    def set_static_batch(self, batch):
        self._static_batch = batch

    def get_static_batch(self):
        return self._static_batch

    # ---- (de)serialisation ---------------------------------------------------------------
    def serialize_model(self):
        out = []
        for value in self.model.state_dict().values():
            out += value.flatten().tolist()
        return out

    def deserialize_model(self, serialized_state_dict):
        state_dict, restored, idx = self.model.state_dict(), {}, 0
        for key, value in state_dict.items():
            n = value.numel()
            restored[key] = torch.as_tensor(serialized_state_dict[idx:idx + n]).view_as(value)
            idx += n
        self.model.load_state_dict(restored)

    def save(self, directory):
        path = os.path.join(directory, "agent")
        os.makedirs(path, exist_ok=True)
        torch.save(self.model.state_dict(), os.path.join(path, "model.pt"))
        torch.save(self.optimizer.state_dict(), os.path.join(path, "optimizer.pt"))
        if self.target_model is not None:
            torch.save(self.target_model.state_dict(), os.path.join(path, "target_model.pt"))
        state = {"action_selector": self.action_selector, "n_updates": self.n_updates,
                 "eval_action_selector": self.eval_action_selector, "max_grad_norm": self.max_grad_norm,
                 "use_cuda_graph": self.use_cuda_graph}
        with open(os.path.join(path, "state.pkl"), "wb") as f:
            pickle.dump(state, f)

    def load(self, directory):
        path = os.path.join(directory, "agent")
        dev = self.model.device
        self.model.load_state_dict(torch.load(os.path.join(path, "model.pt"), map_location=dev))
        self.optimizer.load_state_dict(torch.load(os.path.join(path, "optimizer.pt"), map_location=dev))
        if self.target_model is not None:
            self.target_model.load_state_dict(torch.load(os.path.join(path, "target_model.pt"), map_location=dev))
        with open(os.path.join(path, "state.pkl"), "rb") as f:
            state = pickle.load(f)
        self.action_selector = state["action_selector"]
        self.eval_action_selector = state["eval_action_selector"]
        self.max_grad_norm = state["max_grad_norm"]
        self.use_cuda_graph = state["use_cuda_graph"]
        self.n_updates = state["n_updates"]
        self.train()

    def eval(self):
        self.model.eval()
        self._is_eval = True

    def train(self):
        self.model.train()
        self._is_eval = False

    @torch.no_grad()
    def log(self, logger):
        logger.log_data(data=self._static_total_loss.detach().item(), group_name="Report/Losses",
                        var_name="Total Loss")
        if self._static_distribution_loss is not None:
            logger.log_data(data=self._static_distribution_loss.detach().mean().item(),
                            group_name="Report/Losses", var_name="Distribution Loss")
        if self._static_q_loss is not None:
            logger.log_data(data=self._static_q_loss.detach().mean().item(), group_name="Report/Losses",
                            var_name="Q Loss")
        if getattr(logger, "holdout_data", None) is not None:
            idx = np.random.randint(0, logger.holdout_data["observation"].shape[0])
            obs = logger.holdout_data["observation"][idx]
            if obs.shape[0] != 1:
                obs = obs.unsqueeze(0)
            q, z = self.model._forward_without_cuda_graph(obs)
            self.action_selector.log(logger, z, q)
        self.model.log(logger)
