"""CPU fp32 restatement of value squashing (Config.loss_squish_fn_id) -- TEST INFRASTRUCTURE ONLY.

The reference's prism/agents/squish_functions.py is not in this tree: these are the published definitions,
    "obs_look_further" (Pohlen et al. 2018): h(x) = sign(x) (sqrt(|x| + 1) - 1) + eps x, eps = 1e-2, h^-1 its inverse
    "symlog": h = symlog, h^-1 = symexp
in the same cancellation-free fp32 forms as prism_b200/csrc/common.cuh (each op rounded once), and the IQN / ensemble
losses of oracle/agent_oracle.py with their targets built as h(R + gdn * h^-1(Z_target)) (the reference's IQNModel and
QEnsemble with a (squish, unsquish) pair).  ``squash_oracle_agent`` turns an OracleAgent's heads into these.
"""
import numpy as np
import torch

from oracle.agent_oracle import OracleEnsemble, OracleIQN, ids_actions

OBS_LOOK_FURTHER_EPS = 1e-2
SQUISH_IDS = ("obs_look_further", "symlog")


def squish_id(cfg):
    """Config.loss_squish_fn_id -> "obs_look_further" | "symlog" | "none" (the 1-tuple ("none",) and unknown ids: none)."""
    sq = getattr(cfg, "loss_squish_fn_id", "none")
    sq = sq[0] if isinstance(sq, tuple) else sq
    return sq if sq in SQUISH_IDS else "none"


def _f32(v):
    return torch.tensor(np.float32(v), dtype=torch.float32)


def squash(x, kind):
    """h(x) in fp32.  obs_look_further: sign(x) (sqrt(|x| + 1) - 1) + eps x with sqrt(a + 1) - 1 = a / (sqrt(a + 1) + 1);
    symlog: sign(x) log1p(|x|)."""
    if kind == "obs_look_further":
        a = x.abs()
        r = a / ((a + _f32(1)).sqrt() + _f32(1))
        return torch.copysign(r, x) + _f32(OBS_LOOK_FURTHER_EPS) * x
    if kind == "symlog":
        return torch.copysign(torch.log1p(x.abs()), x)
    return x


def unsquash(x, kind):
    """h^-1(x) in fp32.  obs_look_further: sign(x) (t - 1) ((t - 1) + 2) with s = sqrt(1 + 4 eps (|x| + 1 + eps)) and
    t - 1 = 2 |x| / (s + 1 + 2 eps) (the closed form ((s - 1) / (2 eps))^2 - 1 without its cancellation); symlog:
    symexp = sign(x) expm1(|x|)."""
    if kind == "obs_look_further":
        e = np.float32(OBS_LOOK_FURTHER_EPS)
        a = x.abs()
        s = (_f32(1) + _f32(np.float32(4) * e) * (a + _f32(np.float32(1) + e))).sqrt()
        tm1 = (_f32(2) * a) / (s + _f32(np.float32(1) + np.float32(2) * e))
        return torch.copysign(tm1 * (tm1 + _f32(2)), x)
    if kind == "symlog":
        return torch.copysign(torch.expm1(x.abs()), x)
    return x


class SquashOracleIQN(OracleIQN):
    """OracleIQN.get_loss with squashed targets (iqn_model.py:136-145 with the (squish, unsquish) pair)."""
    squish = "none"

    def get_loss(self, emb, emb_next, acts, returns, gdn, target=None):
        if not self.propagate_grad:
            emb, emb_next = emb.detach(), emb_next.detach()
        target = self if target is None else target
        B, T, Tp, k = acts.shape[0], self.T, self.Tp, self.kappa
        z_cur, tau = self.forward(emb, T)
        with torch.no_grad():
            if target is self:
                z_on = self.forward(emb_next, Tp)[0]
                z_tg = z_on
            elif self.double_q:
                z_on = self.forward(emb_next, Tp)[0]
                z_tg = target.forward(emb_next, Tp)[0]
            else:
                z_tg = target.forward(emb_next, Tp)[0]
                z_on = z_tg
            best = z_on.view(Tp, B, -1).mean(dim=0).argmax(dim=-1)                 # raw quantiles decide a*
            z_sel = torch.gather(z_tg, 1, torch.tile(best.view(-1, 1), [Tp, 1]))
            y = torch.tile(returns.view(-1, 1), [Tp, 1]) + unsquash(z_sel, self.squish) * torch.tile(gdn.view(-1, 1), [Tp, 1])
            y = squash(y, self.squish).view(Tp, B, 1).transpose(1, 0)              # (B, T', 1)
        theta = torch.gather(z_cur, 1, torch.tile(acts.view(-1, 1), [T, 1])).view(T, B, 1).transpose(1, 0)
        delta = y[:, :, None] - theta[:, None, :]                                  # (B, T', T, 1)
        small = (delta.abs() <= k).float()
        huber = small * 0.5 * delta.square() + (1 - small) * k * (delta.abs() - 0.5 * k)
        tq = tau.view(T, B, 1).transpose(1, 0)[:, None, :, :]
        rho = (tq - (delta < 0).float().detach()).abs() * huber / k
        return rho.sum(dim=2).mean(dim=1).view(-1) * self.loss_weight


class SquashOracleEnsemble(OracleEnsemble):
    """OracleEnsemble.get_loss with squashed per-head double-Q targets."""
    squish = "none"

    def get_loss(self, emb, emb_next, acts, returns, gdn, target=None):
        target = self if target is None else target
        B = acts.shape[0]
        q_cur = self.forward(emb)
        with torch.no_grad():
            if target is self:
                q_on = q_tg = self.forward(emb_next)
            elif self.double_q:
                q_on, q_tg = self.forward(emb_next), target.forward(emb_next)
            else:
                q_tg = q_on = target.forward(emb_next)
            best = q_on.argmax(dim=-2)                                            # (B, K)
            rows = torch.arange(B)[:, None]
            q_sel = q_tg[rows, best, torch.arange(q_tg.shape[-1])[None, :]]
            y = squash(returns.view(-1, 1) + unsquash(q_sel, self.squish) * gdn.view(-1, 1), self.squish)
        loss = (q_cur[torch.arange(B), acts.view(-1), :] - y).square().mean(dim=-1)
        if self.theil_coef != 0:
            l2 = torch.stack([torch.nn.utils.parameters_to_vector(h.parameters()).norm() for h in self.q_heads])
            ratio = l2 / l2.mean()
            self.theil = (ratio * torch.log(ratio)).mean()
        return self.loss_weight * (loss - self.theil * self.theil_coef)


def squash_oracle_agent(agent, kind):
    """Give every IQN / ensemble head of an OracleAgent (online and target) squashed targets of ``kind``."""
    for model in (agent.model, agent.target):
        if model is None:
            continue
        for head, cls in ((model.distribution_model, SquashOracleIQN), (model.q_function_model, SquashOracleEnsemble)):
            if head is not None:
                head.__class__ = cls
                head.squish = kind
    return agent


def squash_ids_actions(q, z, kind, *args, **kwargs):
    """IDSActionSelector with an unsquish function: ids_actions on h^-1(q), h^-1(z)."""
    return ids_actions(unsquash(q, kind), unsquash(z, kind), *args, **kwargs)
