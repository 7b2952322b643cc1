"""Bisect a parity gap at a BASELINE config's shapes: per-parameter gradient errors of the product update vs the CPU
oracle, in network order, with the fast routes switched off one at a time.
    python profiles/diag_parity.py configs0 40 50"""
import sys
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_gpu_config_shapes as T  # noqa: E402
from helpers import rel_err  # noqa: E402
from prism_b200.agents import ops  # noqa: E402

name, bseed, tseed = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])


def run(label, setup=None):
    undo = setup() if setup else None
    try:
        cfg, agent, oracle, obs_shape, A, B, fs = T._build_pair(name)
        cpu_batch, dev_batch, w = T._make_batch(obs_shape, A, B, fs, seed=bseed)
        taus = T._taus(cfg, B, seed=tseed)
        oracle.inject_taus([t.clone() for t in taus])
        out = oracle.update(cpu_batch, w)
        T._inject(cfg, agent, taus)
        ops.route_counts(reset=True)
        td = agent.update(dev_batch, w.to(T.DEV))
        torch.cuda.synchronize()
        coef = float(agent.optimizer.norm_out[1])
        ograds = {k: p.grad for k, p in oracle.model.named_parameters()}
        print("== %s: routes %s; clip coef %.6f (oracle norm %.5f)" % (label, ops.route_counts(), coef, float(out["grad_norm"])))
        print("   loss total err %.2e  td err %.2e" % (rel_err(agent._static_total_loss.detach().cpu().numpy(), out["total"].numpy()),
                                                       rel_err(td.cpu().numpy(), out["td"].numpy())))
        for k, g in T._named_grads(agent).items():
            if "q_heads" in k and not k.split("q_heads.")[1].startswith("0."):
                continue
            e = rel_err(g.cpu().numpy() * coef, ograds[k].numpy())
            a, b = g.cpu().numpy() * coef, ograds[k].numpy()
            bad = np.abs(a - b) > 1e-4 * np.abs(b).max()
            print("   %-62s err %.2e  off elements %d / %d" % (k, e, int(bad.sum()), bad.size))
    finally:
        if undo:
            undo()


def no_tc():
    old = ops.TC_MIN_FLOPS
    ops.TC_MIN_FLOPS = float("inf")
    return lambda: setattr(ops, "TC_MIN_FLOPS", old)


def no_narrow():
    old = ops._narrow_eligible
    ops._narrow_eligible = lambda x, w: False
    return lambda: setattr(ops, "_narrow_eligible", old)


def no_ln():
    old = ops._ln_supported
    ops._ln_supported = lambda x, F_: False
    return lambda: setattr(ops, "_ln_supported", old)


run("all fast routes")
run("narrow output layer off", no_narrow)
run("fused LayerNorm off", no_ln)
run("tensor-core GEMMs off", no_tc)
