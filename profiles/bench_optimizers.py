#!/usr/bin/env python
"""clip + Adam / RMSprop / SGD on bench.py's resident configs[1] step, alternating in one process on one GPU.

    python profiles/bench_optimizers.py [--steps K] [--rounds R] [--warmup W]

Four arms, each bench.py's resident leg through LearnerStep (1M-capacity PER shard filled with the synthetic collector
trace, raw priorities ~ Exp(1), batch 256, 4 new steps per iteration planned ahead, parked in HBM and fused into the
step graph, prefetch on):
  adam           FlatAdam (use_adam, what bench.py runs)
  rmsprop        FlatRMSprop, centered (use_rmsprop)
  sgd            FlatSGD (neither)
  rmsprop_torch  the path use_rmsprop took before FlatRMSprop: the same agent with torch.optim.RMSprop(centered=True,
                 capturable=True) after clip_grad_norm_ (Agent's generic optimizer branch), captured in the same graph
The arms alternate: R rounds of K timed steps each (CUDA events), so all see the same clocks and neighbours.  Prints one
JSON line per run: us/step (median of the rounds, min and max), the launches of each arm's step graph (all CUDA kernels
of one replay, counted by torch.profiler after the timed rounds, and those of libprism_b200 alone), and the card's name
and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import BATCH, CAPACITY, N_ACTIONS, N_STREAMS, OBS_SHAPE, STEPS_PER_ITER, Trace  # noqa: E402

PROFILED = 20                # replays per arm counted by the profiler


def card(local):
    """(name, power limit in W) of this rank's GPU: nvidia-smi, read-only query."""
    import torch
    name = torch.cuda.get_device_name(local)
    vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
    phys = vis[local] if local < len(vis) else str(local)
    try:
        out = subprocess.run(["nvidia-smi", "-i", phys, "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        watts = float(out.splitlines()[0])
    except Exception:
        watts = None
    return name, watts


def build(arm, device, fill):
    import torch
    import prism_b200
    cfg = prism_b200.minatar_dqn_per_config(device=device, experience_replay_capacity=CAPACITY, batch_size=BATCH,
                                            per_sampling="stratified", replay_max_streams=N_STREAMS,
                                            replay_staging_rows=65536, use_cuda_graph=False, use_adam=arm == "adam",
                                            use_rmsprop=arm.startswith("rmsprop"))
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, OBS_SHAPE, N_ACTIONS)
    if arm == "rmsprop_torch":
        agent.optimizer = torch.optim.RMSprop(agent.model.parameters(), lr=cfg.learning_rate, alpha=cfg.rmsprop_alpha,
                                              eps=cfg.rmsprop_epsilon, centered=True, capturable=True)
    buf = prism_b200.build_exp_buffer(cfg)
    trace = Trace(4, int(np.prod(OBS_SHAPE)), N_ACTIONS, N_STREAMS)
    done = 0
    while done < fill:
        n = min(65536, fill - done)
        c = trace.chunk(n)
        buf.extend_batch(c["stream"], c["obs"].reshape((n,) + OBS_SHAPE), c["action"], c["reward"], c["done"],
                         c["trunc"], c["next_obs"].reshape((n,) + OBS_SHAPE))
        done += n
    buf._flush()
    g = torch.Generator(device=device)
    g.manual_seed(1)
    prio = torch.empty(fill, device=device).exponential_(1.0, generator=g)
    buf.buffer._sampler.update_priority(torch.arange(fill, device=device), prio, sorted=True)
    torch.cuda.synchronize()
    return agent, buf, trace


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=500, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    import torch
    device = "cuda:0"
    torch.cuda.set_device(0)
    from prism_b200.learner_step import LearnerStep

    arms = {}
    for name in ("adam", "rmsprop", "sgd", "rmsprop_torch"):
        agent, buf, trace = build(name, device, CAPACITY)
        step = LearnerStep(buf, agent, batch_size=BATCH, use_cuda_graph=True, prefetch=True)
        n_blocks = args.warmup + args.rounds * args.steps + PROFILED
        pre = trace.chunk(n_blocks * STEPS_PER_ITER)
        pre_u = np.random.default_rng(2).random((n_blocks, step.B_global))
        pool = torch.stack([step.plan_ingest(tuple(pre[k][i * STEPS_PER_ITER:(i + 1) * STEPS_PER_ITER] for k in
                                                   ("stream", "obs", "action", "reward", "done", "trunc", "next_obs")),
                                             u=pre_u[i]) for i in range(n_blocks)]).to(device)
        arms[name] = {"step": step, "pool": pool, "next": 0, "us": []}

    def run(arm, n):
        st, pool = arm["step"], arm["pool"]
        for _ in range(n):
            st.step(ingest_block=pool[arm["next"]])
            arm["next"] += 1

    for arm in arms.values():
        run(arm, args.warmup)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for arm in arms.values():
            torch.cuda.synchronize()
            ev0.record()
            run(arm, args.steps)
            ev1.record()
            torch.cuda.synchronize()
            sec = ev0.elapsed_time(ev1) * 1e-3
            arm["us"].append(sec / args.steps * 1e6)
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    for arm in arms.values():                                     # after the timed rounds: tracing slows the host
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(arm, PROFILED)
            torch.cuda.synchronize()
        kernels = [e for e in prof.events() if e.device_type == DeviceType.CUDA
                   and not e.name.startswith(("Memcpy", "Memset", "cudaGraph"))]
        arm["kernels"] = len(kernels) / PROFILED
    name, watts = card(0)
    out = {"bench": "clip + Adam / RMSprop / SGD, configs[1] resident step (1M filled PER shard, batch 256, 4 new steps "
                    "per iteration fused, prefetch on), arms alternating in one process",
           "steps_per_round": args.steps, "rounds": args.rounds, "gpu": name, "power_limit_w": watts}
    for key, arm in arms.items():
        us = np.asarray(arm["us"])
        out[key] = {"us_per_step": round(float(np.median(us)), 2), "us_per_step_min": round(float(us.min()), 2),
                    "us_per_step_max": round(float(us.max()), 2), "us_per_step_rounds": [round(float(x), 2) for x in us],
                    "kernels_per_step": arm["kernels"], "library_launches_per_step": arm["step"].launches_per_step}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
