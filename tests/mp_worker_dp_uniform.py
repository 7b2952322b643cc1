"""Worker of tests/test_gpu_uniform_replay.py: one rank of a data-parallel LearnerStep run with uniform replay
(use_per=False, torchrun), or the single-rank run on the UNION buffer (world 1).  Same shards, constants and uniforms as
mp_worker_dp.py.  Writes losses, the parameter arena and every step's sampled rows (as indices into the union) to --out."""
import argparse
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from mp_worker_dp import A, B, C, OBS, S, shard_trace  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--union", type=int, default=0, help="single rank holding the concatenation of this many shards")
    ap.add_argument("--prefetch", type=int, default=0)
    args = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    dev = "cuda:%d" % local
    torch.cuda.set_device(local)
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    pg = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device(dev))
        pg = dist.group.WORLD
    n_shards = args.union if args.union else 1
    shards = list(range(n_shards)) if args.union else [rank]
    # the union's single sampler is stratified, like the global sampling of the ranks
    cfg = prism_b200.minatar_dqn_per_config(device=dev, experience_replay_capacity=C * n_shards, use_per=False,
                                            batch_size=B * n_shards, per_sampling="stratified",
                                            replay_max_streams=S * n_shards, replay_staging_rows=C, use_cuda_graph=False)
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, OBS, A)
    buf = prism_b200.build_exp_buffer(cfg)
    for j, r in enumerate(shards):
        t = shard_trace(r)
        buf.extend_batch(t["stream"] + S * j, t["obs"], t["action"], t["reward"], t["done"], t["trunc"], t["next_obs"])
        buf._flush()
    step = LearnerStep(buf, agent, batch_size=B * n_shards if args.union else B, use_cuda_graph=True, process_group=pg,
                       rank=rank, world_size=world, prefetch=bool(args.prefetch))
    assert step.uniform
    Bg = step.B_global
    offset = 0 if args.union else rank * C
    rng = np.random.default_rng(7)
    losses, rows = [], []
    for it in range(args.steps):
        u = torch.from_numpy(rng.random(Bg)).to(dev)
        losses.append(float(step.step(u=u).detach()))
        idx = step.idx[:step.B_pad].cpu()
        rows.append(idx[idx >= 0] + offset)                # live rows first, padding rows (-1) after
    torch.cuda.synchronize()
    if step.peer is not None:
        step.peer.check()
    torch.save({"losses": losses, "arena": agent.optimizer.arena.cpu(), "rows": rows,
                "exchange": getattr(step, "exchange", None), "B_pad": step.B_pad}, args.out + ".rank%d" % rank)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
