#!/usr/bin/env python
"""Value squashing (loss_squish_fn_id none / obs_look_further / symlog) on two learner paths, alternating in one process
on one GPU.

    python profiles/bench_squash.py [--steps K] [--rounds R] [--warmup W]

Two workloads, three arms each:
  step     bench.py's resident configs[1] leg through LearnerStep (1M-capacity PER shard filled with the synthetic
           collector trace, raw priorities ~ Exp(1), batch 256, 4 new steps per iteration planned ahead and fused into
           the step graph, prefetch on): the squash kind changes the target of the ensemble loss kernel only
  update   Agent.update at configs[0] (MinAtar IDS + IQN, batch 64, T = T' = 32, K = 10 heads) captured as one CUDA
           graph on a fixed batch: the squash kind changes the targets of the quantile-Huber and ensemble loss kernels
The arms of a workload alternate: R rounds of K timed calls each (CUDA events).  Prints one JSON line: us per call
(median of the rounds, min and max) per workload and arm, the step graph's library launches, and the card's name and
power limit read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import BATCH, CAPACITY, N_ACTIONS, N_STREAMS, OBS_SHAPE, STEPS_PER_ITER, Trace  # noqa: E402
from profiles.bench_optimizers import card  # noqa: E402

ARMS = ("none", "obs_look_further", "symlog")


def build_step(arm, device, n_blocks, seed_u):
    import torch
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    cfg = prism_b200.minatar_dqn_per_config(device=device, experience_replay_capacity=CAPACITY, batch_size=BATCH,
                                            per_sampling="stratified", replay_max_streams=N_STREAMS,
                                            replay_staging_rows=65536, use_cuda_graph=False, loss_squish_fn_id=arm)
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, OBS_SHAPE, N_ACTIONS)
    assert agent.model.q_function_model.squash == ARMS.index(arm)
    buf = prism_b200.build_exp_buffer(cfg)
    trace = Trace(4, int(np.prod(OBS_SHAPE)), N_ACTIONS, N_STREAMS)
    done = 0
    while done < CAPACITY:
        n = min(65536, CAPACITY - done)
        c = trace.chunk(n)
        buf.extend_batch(c["stream"], c["obs"].reshape((n,) + OBS_SHAPE), c["action"], c["reward"], c["done"],
                         c["trunc"], c["next_obs"].reshape((n,) + OBS_SHAPE))
        done += n
    buf._flush()
    g = torch.Generator(device=device)
    g.manual_seed(1)
    prio = torch.empty(CAPACITY, device=device).exponential_(1.0, generator=g)
    buf.buffer._sampler.update_priority(torch.arange(CAPACITY, device=device), prio, sorted=True)
    step = LearnerStep(buf, agent, batch_size=BATCH, use_cuda_graph=True, prefetch=True)
    pre = trace.chunk(n_blocks * STEPS_PER_ITER)
    pre_u = np.random.default_rng(seed_u).random((n_blocks, step.B_global))
    pool = torch.stack([step.plan_ingest(tuple(pre[k][i * STEPS_PER_ITER:(i + 1) * STEPS_PER_ITER] for k in
                                               ("stream", "obs", "action", "reward", "done", "trunc", "next_obs")),
                                         u=pre_u[i]) for i in range(n_blocks)]).to(device)
    state = {"next": 0}

    def call():
        step.step(ingest_block=pool[state["next"]])
        state["next"] += 1
    return call, step


def build_update(arm, device):
    import torch
    import prism_b200
    from prism_b200.experience.batch import Batch
    cfg = prism_b200.minatar_ids_iqn_config(device=device, use_cuda_graph=True, loss_squish_fn_id=arm)
    obs_shape, A, B = (10, 10, 4), 3, cfg.batch_size
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, obs_shape, A)
    assert agent.model.distribution_model.squash == ARMS.index(arm)
    g = torch.Generator().manual_seed(7)
    k = torch.randint(1, 4, (B, 1), generator=g)
    raw = {"observation": (torch.rand((B, 1) + obs_shape, generator=g) < 0.1).float(),
           "next": {"observation": (torch.rand((B, 1) + obs_shape, generator=g) < 0.1).float(),
                    "reward": torch.randn(B, 1, generator=g)},
           "nonterminal": torch.rand(B, 1, generator=g) > 0.1, "gamma": 0.99 ** k.float(),
           "action": torch.randint(0, A, (B, 1), generator=g)}
    to = lambda d: Batch({key: (to(v) if isinstance(v, dict) else v.to(device)) for key, v in d.items()})
    batch, w = to(raw), (torch.rand(B, generator=g) * 0.7 + 0.3).to(device)

    def call():
        agent.update(batch, w)
    return call, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300, help="timed calls per arm and round")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    import torch
    device = "cuda:0"
    torch.cuda.set_device(0)
    n_blocks = args.warmup + args.rounds * args.steps
    work = {"step": {a: build_step(a, device, n_blocks, 2) for a in ARMS},
            "update": {a: build_update(a, device) for a in ARMS}}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out_us = {w: {a: [] for a in ARMS} for w in work}
    for wname, arms in work.items():
        for call, _ in arms.values():
            for _ in range(args.warmup):
                call()
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for a, (call, _) in arms.items():
                torch.cuda.synchronize()
                ev0.record()
                for _ in range(args.steps):
                    call()
                ev1.record()
                torch.cuda.synchronize()
                out_us[wname][a].append(ev0.elapsed_time(ev1) * 1e3 / args.steps)
    name, watts = card(0)
    out = {"bench": "value squashing arms alternating in one process: configs[1] resident LearnerStep (1M filled PER "
                    "shard, batch 256, 4 new steps fused, prefetch on) and configs[0] Agent.update as one CUDA graph",
           "calls_per_round": args.steps, "rounds": args.rounds, "gpu": name, "power_limit_w": watts}
    for wname in work:
        out[wname] = {}
        for a in ARMS:
            us = np.asarray(out_us[wname][a])
            step = work[wname][a][1]
            out[wname][a] = {"us_per_call": round(float(np.median(us)), 2), "us_per_call_min": round(float(us.min()), 2),
                             "us_per_call_max": round(float(us.max()), 2)}
            if step is not None:
                out[wname][a]["library_launches_per_step"] = step.launches_per_step
    print(json.dumps(out))


if __name__ == "__main__":
    main()
