#!/usr/bin/env python
"""Uniform replay (use_per=False) against PER on bench.py's resident configs[1] step, alternating in one process.

    python profiles/bench_uniform.py [--steps K] [--rounds R] [--warmup W]
    torchrun --nproc-per-node N profiles/bench_uniform.py ...        # N = 2 / 4 / 8: data parallel, weak scaling

Both arms run bench.py's resident leg: a 1M-capacity shard filled with the synthetic collector trace (bench.Trace),
batch 256 per GPU, 4 new steps per iteration planned on the host ahead of the timed region, parked in HBM and fused
into the step graph (step(ingest_block=...)), prefetch on.  The PER arm sets raw priorities ~ Exp(1) as bench.py does.
The arms alternate: R rounds of K timed steps each (CUDA events; under torchrun the slowest rank's time), so both see
the same clocks and neighbours.  Prints one JSON line: us/step (median of the rounds, min and max), transitions/s,
launches per step of each arm, and the card's name and power limit read in the same run.
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


def build(use_per, rank, device, fill):
    import torch
    import prism_b200
    cfg = prism_b200.minatar_dqn_per_config(device=device, experience_replay_capacity=CAPACITY, batch_size=BATCH,
                                            use_per=use_per, per_sampling="stratified", replay_max_streams=N_STREAMS,
                                            replay_staging_rows=65536, use_cuda_graph=False)
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, OBS_SHAPE, N_ACTIONS)
    buf = prism_b200.build_exp_buffer(cfg)
    trace = Trace(4 + 1000 * rank, int(np.prod(OBS_SHAPE)), N_ACTIONS, N_STREAMS)
    done = 0
    while done < fill:
        n = min(65536, fill - done)
        c = trace.chunk(n)
        buf.extend_batch(c["stream"], c["obs"].reshape((n,) + OBS_SHAPE), c["action"], c["reward"], c["done"],
                         c["trunc"], c["next_obs"].reshape((n,) + OBS_SHAPE))
        done += n
    buf._flush()
    if use_per:
        g = torch.Generator(device=device)
        g.manual_seed(1 + rank)
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
    import torch.distributed as dist
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    device = "cuda:%d" % local
    torch.cuda.set_device(local)
    pg = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device(device))
        pg = dist.group.WORLD
    from prism_b200.learner_step import LearnerStep

    arms = {}
    for name, use_per in (("uniform", False), ("per", True)):
        agent, buf, trace = build(use_per, rank, device, CAPACITY)
        if world > 1:
            dist.broadcast(agent.optimizer.arena, src=0)
            if agent.target_model is not None:
                dist.broadcast(agent.target_model._flat_arena, src=0)
        step = LearnerStep(buf, agent, batch_size=BATCH, use_cuda_graph=True, process_group=pg, rank=rank,
                           world_size=world, prefetch=True)
        n_blocks = args.warmup + args.rounds * args.steps
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

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for arm in arms.values():
        run(arm, args.warmup)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for arm in arms.values():
            barrier()
            ev0.record()
            run(arm, args.steps)
            ev1.record()
            barrier()
            sec = ev0.elapsed_time(ev1) * 1e-3
            if world > 1:
                t = torch.tensor([sec], device=device, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                sec = float(t.item())
            arm["us"].append(sec / args.steps * 1e6)
    for arm in arms.values():
        if arm["step"].peer is not None:
            arm["step"].peer.check()
    name, watts = card(local)
    if rank == 0:
        out = {"bench": "uniform replay vs PER, configs[1] resident step (1M filled, batch 256 per GPU, 4 new steps "
                        "per iteration fused, prefetch on), arms alternating in one process",
               "n_gpus": world, "steps_per_round": args.steps, "rounds": args.rounds, "gpu": name,
               "power_limit_w": watts}
        for key, arm in arms.items():
            us = np.asarray(arm["us"])
            med = float(np.median(us))
            out[key] = {"us_per_step": round(med, 2), "us_per_step_min": round(float(us.min()), 2),
                        "us_per_step_max": round(float(us.max()), 2), "us_per_step_rounds": [round(float(x), 2) for x in us],
                        "transitions_per_s": round(BATCH * world / (med * 1e-6), 1),
                        "launches_per_step": arm["step"].launches_per_step,
                        "exchange": getattr(arm["step"], "exchange", None) if world > 1 else None}
        print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == "__main__":
    main()
