"""Worker of tests/test_gpu_value_squash.py: mp_worker_dp.py's data-parallel LearnerStep run (torchrun, or the single rank
on the UNION buffer) with Config.loss_squish_fn_id = --squish.  Writes losses, the parameter arena and the leaves to
--out."""
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
    ap.add_argument("--squish", required=True)
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
    cfg = prism_b200.minatar_dqn_per_config(device=dev, experience_replay_capacity=C * n_shards,
                                            batch_size=B * n_shards, per_sampling="stratified",
                                            replay_max_streams=S * n_shards, replay_staging_rows=C, use_cuda_graph=False,
                                            loss_squish_fn_id=args.squish)
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, OBS, A)
    buf = prism_b200.build_exp_buffer(cfg)
    for j, r in enumerate(shards):
        t = shard_trace(r)
        buf.extend_batch(t["stream"] + S * j, t["obs"], t["action"], t["reward"], t["done"], t["trunc"], t["next_obs"])
        buf._flush()
    prio = np.concatenate([shard_trace(r)["prio"] for r in shards])
    buf.buffer._sampler.update_priority(torch.arange(C * n_shards, device=dev), torch.from_numpy(prio).to(dev), sorted=True)
    step = LearnerStep(buf, agent, batch_size=B * n_shards if args.union else B, use_cuda_graph=True, process_group=pg,
                       rank=rank, world_size=world)
    Bg = step.B_global
    rng = np.random.default_rng(7)
    losses = []
    for it in range(args.steps):
        u = torch.from_numpy(rng.random(Bg)).to(dev)
        losses.append(float(step.step(u=u).detach()))
    torch.cuda.synchronize()
    if step.peer is not None:
        step.peer.check()
    tree = buf.buffer._sampler
    torch.save({"losses": losses, "arena": agent.optimizer.arena.cpu(), "leaves": tree.leaves().cpu(),
                "squash": agent.model.q_function_model.squash, "B_pad": step.B_pad}, args.out + ".rank%d" % rank)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
