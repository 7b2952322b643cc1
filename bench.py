#!/usr/bin/env python
"""bench.py -- PER sampled transitions/s + learner updates/s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (hand-written sm_100a CUDA)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: oracle port on the host cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy

Workload at every N: BASELINE.json configs[1] per GPU -- MinAtar Space-Invaders shaped transitions
(10x10x6), DQN + double-Q + PER, 1M-capacity shard, batch 256, 3-step returns.  One "step" is one
iteration of the reference's hot loop (prism/learner.py:95-125): sample -> gather(+n-step) ->
update (loss, backward, clip, Adam) -> priority write-back.  N > 1 is weak scaling: every rank
holds its own 1M shard and trains on the strata of a global stratified sample (batch 256*N) that
land in its shard (one 64-byte all-gather + one flat gradient all-reduce per step).

`value`  : sampled transitions/s, whole job, everything resident in HBM (one CUDA graph per step).
`e2e`    : same metric through the public buffer/agent API with HOST inputs: every step stages 4
           new transitions + 256 uniforms in pinned host memory, copies them H2D, and reads the
           loss back D2H -- all inside the timed region.
`roofline`: the dominant kernel of OUR library inside the step, timed live with CUDA events.
`extras.per_microbench`: BASELINE configs[2] (16M-leaf tree, batch 4096 sample + priority update)
           and the streaming kernels (bulk build, Atari-shaped gather), each with its own roofline.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = ("PER sampled transitions/s (4 new steps ingested -> sample -> 3-step gather -> DQN update -> priority "
          "write-back, per learner iteration)")
OBS_SHAPE = (10, 10, 6)
N_ACTIONS = 4
CAPACITY = 1_000_000
BATCH = 256
N_STREAMS = 32
STEPS_PER_ITER = 4            # timesteps_per_iteration of every reference config
L2_BYTES = 126e6


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# synthetic collector trace (SURVEY 8d: MinAtar-shaped, seed 4)
# ------------------------------------------------------------------------------------------------
class Trace:
    """Round-robin interleaving of N_STREAMS collector streams; obs ~ Bernoulli(0.1), reward
    Bernoulli(0.05), done 1/200, truncated 1/2000, uniform actions."""

    def __init__(self, seed, obs_elems, n_actions, n_streams):
        self.rng = np.random.default_rng(seed)
        self.E, self.A, self.S = obs_elems, n_actions, n_streams
        self.carry = self._obs(n_streams)
        self.t = 0

    def _obs(self, n):
        return (self.rng.random((n, self.E), dtype=np.float32) < 0.1).astype(np.float32)

    def chunk(self, n):
        S = self.S
        fresh = self._obs(n)
        allobs = np.concatenate([self.carry, fresh], axis=0)           # step j: obs = allobs[j], successor = allobs[j+S]
        self.carry = allobs[n:]
        out = {
            "stream": ((self.t + np.arange(n)) % S).astype(np.int32),
            "obs": allobs[:n], "next_obs": allobs[S:S + n],
            "action": self.rng.integers(0, self.A, n).astype(np.int32),
            "reward": (self.rng.random(n) < 0.05).astype(np.float32),
            "done": self.rng.random(n) < (1 / 200),
        }
        out["trunc"] = (~out["done"]) & (self.rng.random(n) < (1 / 2000))
        self.t += n
        return out


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed regions: NVML polled from a thread every 5 ms
    (the timed regions last a fraction of a second -- nvidia-smi -lms starts too slowly for that); falls back
    to an nvidia-smi loop when the NVML binding is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
            "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc, self.nvml, self.stop_flag = gpu_index, [], None, None, False
        self.sm, self.mask, self.sm_max, self.source = [], 0, None, None
        self.active = True       # window(False) pauses sampling between the timed regions

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v for v in vis.split(",") if v.strip()]
        if ids and all(v.strip().isdigit() for v in ids) and self.idx < len(ids):
            return int(ids[self.idx])
        return self.idx

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml"
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            if not self.active:
                time.sleep(0.002)
                continue
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(0.005)

    def window(self, on):
        self.active = bool(on)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.th.join(timeout=1.0)
            reasons = sorted(n for n, bit in self.BITS.items() if self.mask & bit)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                    "reasons": reasons, "samples": len(self.sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def build_ours(rank, world, device, capacity, fill, seed):
    import torch
    import prism_b200
    cfg = prism_b200.minatar_dqn_per_config(device=device, experience_replay_capacity=capacity, batch_size=BATCH,
                                            per_sampling="stratified", replay_max_streams=N_STREAMS,
                                            replay_staging_rows=65536, use_cuda_graph=False)
    torch.manual_seed(123)                                   # default_config.py:97
    agent = prism_b200.build_agent(cfg, OBS_SHAPE, N_ACTIONS)
    buf = prism_b200.build_exp_buffer(cfg)
    trace = Trace(4 + 1000 * rank, int(np.prod(OBS_SHAPE)), N_ACTIONS, N_STREAMS)
    t0 = time.perf_counter()
    done = 0
    while done < fill:
        n = min(65536, fill - done)
        c = trace.chunk(n)
        buf.extend_batch(c["stream"], c["obs"].reshape((n,) + OBS_SHAPE), c["action"], c["reward"], c["done"],
                         c["trunc"], c["next_obs"].reshape((n,) + OBS_SHAPE))
        done += n
    buf._flush()
    torch.cuda.synchronize()
    ingest_s = time.perf_counter() - t0
    # priorities (SURVEY 8d seed 1): raw p ~ Exp(1) for every slot
    g = torch.Generator(device=device)
    g.manual_seed(1 + rank)
    prio = torch.empty(fill, device=device).exponential_(1.0, generator=g)
    buf.buffer._sampler.update_priority(torch.arange(fill, device=device), prio, sorted=True)
    torch.cuda.synchronize()
    return cfg, agent, buf, trace, ingest_s


DUMP_MAX_BYTES = 64 << 20


def step_outputs(step, prefix=""):
    """What the last LearnerStep iteration computed, on the host: its loss and TD errors, the batch it sampled and
    gathered, the parameters after its optimizer step and every priority leaf after its write-back.  Integer and fp64
    arrays come back as float64, the rest as float32."""
    import torch
    torch.cuda.synchronize()
    b = step.batch
    out = {"loss": step.agent._static_total_loss, "td": step.td, "index": step.idx[:step.B_pad],
           "weight": step.weight[:step.B_pad], "observation": b["observation"],
           "next_observation": b["next"]["observation"], "reward": b["next"]["reward"], "gamma": b["gamma"],
           "nonterminal": b["nonterminal"], "action": b["action"], "params": step.agent.optimizer.arena,
           "priorities": step.tree.leaves()}
    wide = (torch.int64, torch.int32, torch.float64)
    return {prefix + k: v.detach().cpu().numpy().astype(np.float64 if v.dtype in wide else np.float32)
            for k, v in out.items()}


def dump_outputs(path, arrays):
    """DIR/<name>.npy for every array (--dump-outputs)."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("outputs to dump take %d bytes, more than %d" % (total, DUMP_MAX_BYTES))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def time_kernel(fn, reps, torch):
    """Average duration (s) of one call of fn, CUDA events on the launching stream."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3 / reps


def time_kernel_graph(fn, reps, torch):
    """Average device time (s) of one call of fn: `reps` back-to-back calls captured in a CUDA graph (no host launch
    overhead between them), replayed, CUDA events on the launching stream."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3 / (5 * reps)


def kernel_rooflines(step, buf, agent, torch, hbm_gbs, peak_src):
    """Per-C-ABI-op timing of our kernels at the step's shapes + algorithmic bytes (SURVEY 8d)."""
    tree, ring = buf.buffer._sampler, buf.buffer._storage
    B = step.B_pad
    L = int(np.log2(tree.capacity))
    D = ring.obs_elems * ring.obs.element_size() * ring.frame_stack
    Dout = ring.obs_elems * 4 * ring.frame_stack
    u = torch.rand(B, dtype=torch.float64, device=buf.device)
    idx = torch.empty(B, dtype=torch.int64, device=buf.device)
    w = torch.empty(B, dtype=torch.float32, device=buf.device)
    tree.sample(B, u=u, idx_out=idx, weight_out=w)
    prio = torch.rand(B, device=buf.device)
    opt = agent.optimizer
    saved_allreduce, opt.allreduce = opt.allreduce, None      # rank-0-only timing: no collective in here
    saved_peer, opt.peer = opt.peer, None
    rows = {}
    time_kernel = time_kernel_graph          # device time per call, launch overhead excluded (shadows the eager timer)
    rows["per_sample (tree_sample_kernel)"] = (time_kernel(lambda: tree.sample(B, u=u, idx_out=idx, weight_out=w), 50, torch),
                                               B * (4 * L + 24))
    rows["per_gather (store_gather_kernel)"] = (time_kernel(lambda: ring.gather(idx, buf._obs, buf._next_obs, buf._reward,
                                                                                 buf._gamma, buf._nonterminal, buf._action), 50, torch),
                                                B * (2 * D + 2 * Dout + 43))
    rows["per_update (upd_lines_sorted_kernel + tree_rebuild_kernel)"] = (time_kernel(lambda: tree.update_priority(idx, prio, sorted=True), 50, torch),
                                                     B * (16 * L + 20))
    snap = opt.snapshot()
    rows["gather+clip+adam (adam_fused_kernel, one launch)"] = (time_kernel(lambda: opt.step(refresh_table=False), 50, torch),
                                                  opt.numel * 4 * (2 + 1 + 2 + 2 + 2))   # pack r/w, sumsq fused, p/m/v r+w, g read
    opt.restore(snap)
    opt.allreduce = saved_allreduce
    opt.peer = saved_peer
    # the dense layers of the Q head at the step's shapes (embedding 1024 -> hidden 256, fused bias + ReLU)
    from prism_b200.agents import ops
    F_, H_ = 1024, 256
    xg = torch.randn(B, F_, device=buf.device)
    wg = torch.randn(1, H_, F_, device=buf.device) / 32.0
    bg = torch.zeros(1, H_, device=buf.device)
    with torch.no_grad():
        t_fc = time_kernel(lambda: ops.linear_heads(xg, wg, bg, relu=True), 50, torch)
    fc_flops = 2.0 * B * H_ * F_
    fc_bytes = 4 * (B * F_ + H_ * F_ + H_ + B * H_)
    out = {}
    for k, (sec, nbytes) in rows.items():
        gbs = nbytes / sec / 1e9
        out[k] = {"us": round(sec * 1e6, 2), "algorithmic_bytes": int(nbytes), "achieved_gbs": round(gbs, 2),
                  "frac": round(gbs / hbm_gbs, 5)}
    bf16 = tensor_peak()
    out["q_head_fc1_fwd (gemm_async_kernel, %dx%dx%d 3xTF32 mma.sync, cluster split-K)" % (B, H_, F_)] = {
        "us": round(t_fc * 1e6, 2), "algorithmic_flops": int(fc_flops), "algorithmic_bytes": int(fc_bytes),
        "achieved_tflops": round(fc_flops / t_fc / 1e12, 3), "achieved_gbs": round(fc_bytes / t_fc / 1e9, 2),
        "frac_of_bf16_tensor_peak": round(fc_flops / t_fc / 1e12 / bf16, 5), "frac": round(fc_bytes / t_fc / 1e9 / hbm_gbs, 5)}
    dom = max(out, key=lambda k: out[k]["us"])
    d = out[dom]
    if "algorithmic_flops" in d:
        # GEMM-shaped work: the tensor / FMA pipes bound it; 3 forward + 2x2 backward launches of this family are ~45 %
        # of the step (profiles/launches_r01d_step.txt).  traffic: dram__bytes_read+write of one launch, ncu --set full
        # (profiles/ncu_full_step_r02b.txt, gemm_async_kernel<1,1,0,4> grid (4,4,8); before the cp.async kernel:
        # ncu_full_step_r02.txt, gemm_kernel<1,1,0>).
        traffic, traffic_file = ncu_traffic("gemm_async_kernel<1, 1, 0,")
        if traffic is None:
            traffic, traffic_file = ncu_traffic("gemm_kernel<1, 1, 0,")
        roof = {"bound": "tensor", "kernel": dom, "achieved": d["achieved_tflops"], "peak": bf16, "unit": "TFLOP/s",
                "frac": d["frac_of_bf16_tensor_peak"], "traffic": traffic, "traffic_source": traffic_file,
                "peak_source": peak_src,
                "note": "batch-256 fp32 layer (134 MFLOP, 2.3 MB): latency-bound by construction -- 128 CTAs in clusters of 8, "
                        "each fetching its whole K slice by cp.async at entry; the reference computes it in fp32, so the "
                        "products are 3xTF32 on the legacy mma.sync path (3 MMAs per product) and the bf16 tensor peak is "
                        "only the nominal denominator.  Layers from 2e8 FLOP up run on tcgen05 (3xTF32): "
                        "see extras.tc_gemm for their tensor-pipe roofline and extras.per_microbench for the HBM-bound "
                        "PER kernels"}
    else:
        traffic, traffic_file = ncu_traffic(dom.split("(")[-1].split(",")[0].split(")")[0].strip())
        roof = {"bound": "hbm", "kernel": dom, "achieved": d["achieved_gbs"], "peak": hbm_gbs, "unit": "GB/s",
                "frac": d["frac"], "traffic": traffic, "traffic_source": traffic_file, "peak_source": peak_src,
                "note": "batch-256 launches move KBs-MBs: latency-bound by construction; see extras.per_microbench "
                        "for the saturated PER kernels"}
    return roof, out


def sharded_per_microbench(step, rank, world, device, torch, dist, hbm_gbs):
    """BASELINE configs[3]: sharded PER, 8M (2^23) leaves per GPU, global batch 4096: exchange of the shard states +
    global stratified sampling (owner-computes) + priority update of the owned strata, captured as one CUDA graph per
    rank and replayed in lock-step; max over ranks.  Collective: the peer-memory all-gather of LearnerStep (or NCCL)."""
    from prism_b200 import PrioritizedTree
    N, Bg = 1 << 23, 4096
    tree = PrioritizedTree(N, device=device, mode="stratified")
    g = torch.Generator(device=device)
    g.manual_seed(100 + rank)
    tree.build(torch.empty(N, device=device).exponential_(1.0, generator=g))
    tree.seed(7)                                       # same Philox key on every rank
    idx = torch.zeros(Bg, dtype=torch.int64, device=device)
    w = torch.zeros(Bg, dtype=torch.float32, device=device)
    stratum = torch.zeros(Bg, dtype=torch.int64, device=device)
    pad = Bg // world + int(4 * (Bg / world) ** 0.5)
    prio = torch.rand(pad, device=device)
    peer = step.peer
    all_state = peer.all_state if peer is not None else torch.zeros(world, 64, dtype=torch.uint8, device=device)

    def one():
        if peer is not None:
            # every rank puts its 64-byte state to every rank; the sampling kernel itself waits for the puts
            peer.state_put(tree.state)
            tree.sample_global_peer(peer, Bg, None, idx_out=idx, weight_out=w, stratum_out=stratum)
        else:
            dist.all_gather_into_tensor(all_state.view(-1), tree.state)
            tree.sample_global(world, rank, all_state, Bg, None, idx_out=idx, weight_out=w, stratum_out=stratum)
        tree.update_priority(idx[:pad], prio, sorted=True)
    reps = 20
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            one()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    dist.barrier()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(reps):
            one()
    gr.replay()
    torch.cuda.synchronize()
    dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        gr.replay()
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) * 1e-3 / (10 * reps)], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item())
    L = 23
    nbytes = Bg * (4 * L + 24) + Bg * (16 * L + 20)          # SURVEY 8d per-transition figures, whole job
    del gr
    return {"leaves_per_gpu": N, "global_batch": Bg, "us_per_iteration": round(sec * 1e6, 2),
            "transitions_per_s": round(Bg / sec, 1), "algorithmic_bytes": int(nbytes),
            "achieved_gbs": round(nbytes / sec / 1e9, 2), "frac_of_one_gpu_hbm": round(nbytes / sec / 1e9 / hbm_gbs, 5),
            "exchange": "peer" if peer is not None else "nccl",
            "note": "latency-bound: one cross-GPU state exchange (put + in-kernel wait) + 1 sampling launch + 2 update "
                    "launches per iteration"}


def ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, read from the committed `ncu --set full`
    summaries of this round (profiles/ncu_full_*_r02*.txt, written by profiles/summarize_ncu.py).  Returns
    (bytes or None, file name or None)."""
    import glob
    best = (None, None)
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_full_*_r02*.txt"))):
        try:
            lines = open(path).read().splitlines()
        except OSError:
            continue
        vals = []
        for ln in lines[1:]:
            if kernel_substr not in ln:
                continue
            m = __import__("re").search(r"\(\d+,\d+,\d+\)\s+\(\d+,\d+,\d+\)\s+([0-9.]+)\s+(\d+)\s+(\d+)", ln)
            if m:
                vals.append(float(m.group(2)) + float(m.group(3)))
        if vals:
            best = (int(sum(vals) / len(vals)), os.path.basename(path))
    return best


def ncu_per_traffic():
    """{K: DRAM bytes (read + written) of ONE sample + write-back iteration at K batches in flight}, from the committed
    `ncu --set full` capture of profiles/per_ncu.py (profiles/ncu_full_per_r02.txt: after the bulk build the kernels of
    K = 1, 16, 64 follow, two repetitions each; the second one is read).  {} when the file is absent."""
    path = os.path.join(ROOT, "profiles", "ncu_full_per_r02.txt")
    try:
        lines = open(path).read().splitlines()[1:]
    except OSError:
        return {}
    import re
    rows = []
    for ln in lines:
        m = re.match(r"\s*(\d+)\s+(\S+)\s.*?\(\d+,\d+,\d+\)\s+\(\d+,\d+,\d+\)\s+([0-9.]+)\s+(\d+)\s+(\d+)", ln)
        if m:
            rows.append((m.group(2), float(m.group(4)) + float(m.group(5))))
    # an iteration starts at every sampling kernel; iterations come in pairs (two repetitions per K)
    iters, cur = [], None
    for name, b in rows:
        if "tree_sample" in name:
            cur = [b]
            iters.append(cur)
        elif cur is not None and ("upd_" in name or "tree_rebuild" in name):
            cur.append(b)
            if "tree_rebuild" in name:
                cur = None
    out = {}
    for K, i in zip((1, 16, 64), (1, 3, 5)):
        if i < len(iters):
            out[K] = int(sum(iters[i]))
    return out


def measure_tf32_peak(device, torch):
    """Dense TF32 TFLOP/s of this GPU: the library GEMM on 8192^3 fp32 operands with TF32 allowed (best of 5) -- the
    denominator of the 3xTF32 kernels' roofline, measured instead of assumed (bf16 / 2)."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=device)
        b = torch.randn(n, n, device=device)
        for _ in range(2):
            a @ b
        torch.cuda.synchronize()
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        del a, b
        return best
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def torch_gpu_baseline(device, torch):
    """BASELINE leg (not the product): the reference-equivalent update step in STOCK PyTorch on this GPU, captured as a
    CUDA graph -- the stand-in for the reference's best GPU path (prism/agents/agent.py:102-147; the reference itself
    needs torchrl to run).  Same models (oracle/agent_oracle.py restates the reference's modules with the reference's
    parameter names), same shapes, ATen / cuBLAS / cuDNN kernels, torch.optim.Adam(capturable).  Update only: the
    reference samples and writes priorities back on the CPU."""
    import dataclasses
    import prism_b200
    from oracle.agent_oracle import OracleAgent
    out = {}
    specs = {"configs[1] dqn_B256": (prism_b200.minatar_dqn_per_config, OBS_SHAPE, N_ACTIONS, 256, 1, 200),
             "configs[0] minatar_ids_iqn_B64": (prism_b200.minatar_ids_iqn_config, (10, 10, 4), 3, 64, 1, 100),
             "configs[4] atari_iqn64x64_ids_B512": (prism_b200.atari_iqn_ids_config, (4, 84, 84), 18, 512, 4, 10)}
    for name, (make, obs_shape, A, B, fs, reps) in specs.items():
        try:
            cfg = dataclasses.replace(make(), device=device, use_cuda_graph=False)
            torch.manual_seed(123)
            with torch.device(device):
                oracle = OracleAgent(cfg, obs_shape, A)
                oracle.opt = torch.optim.Adam(oracle.model.parameters(), lr=cfg.learning_rate,
                                              betas=(cfg.adam_beta1, cfg.adam_beta2), eps=cfg.adam_epsilon, capturable=True)
                shape = (B,) + tuple(obs_shape) if fs > 1 else (B, 1) + tuple(obs_shape)
                batch = {"observation": torch.rand(shape), "next": {"observation": torch.rand(shape), "reward": torch.randn(B, 1)},
                         "nonterminal": torch.rand(B, 1) > 0.1, "gamma": torch.full((B, 1), 0.97),
                         "action": torch.randint(0, A, (B, 1))}
                w = torch.rand(B)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(3):
                        oracle.update(batch, w)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    oracle.update(batch, w)
                sec = time_kernel(g.replay, reps, torch)
            out[name] = {"ms_per_update": round(sec * 1e3, 4), "updates_per_s": round(1.0 / sec, 2), "batch": B,
                         "what": "stock PyTorch (ATen/cuBLAS/cuDNN, TF32 matmul off) update step under one CUDA graph"}
            del g, oracle, batch
        except Exception as e:
            out[name] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()
    return out


def config_rooflines(extras, hbm_gbs, tf32_peak):
    """One roofline object per BASELINE config, from the live measurements already in `extras`."""
    out = {}
    pm = extras.get("per_microbench", {})
    tc = extras.get("tc_gemm", {})
    oc = extras.get("other_configs", {})

    def tc_row(key, label):
        r = tc.get(key)
        if not isinstance(r, dict) or "us" not in r:
            return None
        return {"kernel": label, "bound": "tensor", "achieved": r["achieved_tf32_tflops"], "peak": round(tf32_peak, 1),
                "unit": "TFLOP/s (TF32; 3 TF32 FLOP per fp32-equivalent FLOP)", "frac": round(r["achieved_tf32_tflops"] / tf32_peak, 4),
                "us": r["us"], "peak_source": "measured here: library TF32 GEMM 8192^3"}
    r = tc_row("iqn_hidden_cfg0_2048x256x1024_fwd", "tc_gemm_kernel (IQN hidden layer 2048x256x1024)")
    if r:
        r["step_ms"] = oc.get("configs[0] minatar_ids_iqn_B64", {}).get("ms_per_update")
        out["configs[0]"] = r
    k = pm.get("sample+update_16M_B4096_x64_in_flight") or pm.get("sample+update_16M_B4096")
    if k:
        out["configs[2]"] = {"kernel": "tree_sample_kernel + priority write-back, 64 batches of 4096 in flight (see per_microbench for K = 1, 4, 16)",
                             "bound": "hbm", "achieved": k["achieved_gbs"], "peak": hbm_gbs, "unit": "GB/s", "frac": k["frac"],
                             "us": k["us"], "single_batch_us": pm.get("sample+update_16M_B4096", {}).get("us")}
    k = extras.get("sharded_per_configs3") or pm.get("shard_8M_global_sample+update_B4096")
    if k and "us_per_iteration" in k:
        out["configs[3]"] = {"kernel": "global_sample_kernel + upd_lines_sorted_kernel + tree_rebuild_kernel per 2^23-leaf shard", "bound": "hbm",
                             "achieved": k["achieved_gbs"], "peak": hbm_gbs, "unit": "GB/s",
                             "frac": k.get("frac_of_one_gpu_hbm"), "us": k["us_per_iteration"]}
    r = tc_row("iqn_hidden_32768x512x3136_fwd", "tc_gemm_kernel (IQN hidden layer 32768x512x3136)")
    if r:
        r["step_ms"] = oc.get("configs[4] atari_iqn64x64_ids_B512", {}).get("ms_per_update")
        out["configs[4]"] = r
    return out


def tensor_peak():
    """Measured dense bf16 TFLOP/s (MEASURED_PEAKS.json, burst: kernels timed alone), else the nominal 2250."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["bf16_tflops"])
    except Exception:
        return 2250.0


def tc_gemm_microbench(device, torch):
    """The tcgen05 3xTF32 GEMMs of the configs[4] IQN hidden layer (32768 rows = 64 quantiles x 512, 3136 -> 512) and
    K-head ensemble: forward, input gradient, weight gradient.  TF32 peak = half the measured bf16 peak; every
    fp32-equivalent FLOP costs three TF32 FLOPs."""
    from prism_b200.agents import ops
    tf32 = measure_tf32_peak(device, torch)
    out = {"tf32_peak_tflops": round(tf32, 1), "bf16_peak_tflops": tensor_peak(),
           "note": "achieved_tf32 = 3 x fp32-equivalent (3xTF32 split keeps the reference's fp32 accuracy); frac = "
                   "achieved_tf32 / the TF32 peak MEASURED here (library TF32 GEMM, 8192^3)"}
    for name, (K, M, N, J) in {"iqn_hidden_32768x512x3136": (1, 32768, 512, 3136), "ensemble_10x512x512x3136": (10, 512, 512, 3136),
                               "iqn_hidden_cfg0_2048x256x1024": (1, 2048, 256, 1024)}.items():
        x = torch.randn(K, M, J, device=device)
        w = torch.randn(K, N, J, device=device)
        b = torch.randn(K, N, device=device)
        dz = torch.randn(K, M, N, device=device)
        y, dx, dw = torch.empty(K, M, N, device=device), torch.empty(K, M, J, device=device), torch.empty(K, N, J, device=device)
        fl = 2.0 * K * M * N * J
        for kind, fn in (("fwd", lambda: ops.tc_gemm(y, x, 0, J, M * J, w, 0, J, N * J, K, M, N, J, bias=b, bias_bs=N, act=1)),
                         ("dgrad", lambda: ops.tc_gemm(dx, dz, 0, N, M * N, w, 1, J, N * J, K, M, J, N)),
                         ("wgrad", lambda: ops.tc_gemm(dw, dz, 1, N, M * N, x, 1, J, M * J, K, N, J, M))):
            t = time_kernel(fn, 10, torch)
            eq = fl / t / 1e12
            out["%s_%s" % (name, kind)] = {"us": round(t * 1e6, 1), "algorithmic_flops": int(fl), "fp32_equivalent_tflops": round(eq, 1),
                                            "achieved_tf32_tflops": round(3 * eq, 1), "frac": round(3 * eq / tf32, 3)}
        del x, w, b, dz, y, dx, dw
        torch.cuda.empty_cache()
    return out


def per_microbench(device, torch, hbm_gbs):
    """BASELINE configs[2]: 16M-leaf tree, batch 4096 sample + priority update; plus the streaming kernels."""
    from prism_b200 import PrioritizedTree, TransitionRing
    out = {}
    N = 1 << 24
    L = 24
    tree = PrioritizedTree(N, device=device, mode="stratified")
    g = torch.Generator(device=device)
    g.manual_seed(1)
    leaves = torch.empty(N, device=device).exponential_(1.0, generator=g).add_(1e-8).sqrt_()
    sec = time_kernel_graph(lambda: tree.build(leaves), 10, torch)
    nbytes = 2 * (4 * N + 4 * 2 * N)                     # SURVEY 8d: read leaves once per tree, write 2N nodes per tree
    out["bulk_build_16M"] = {"ms": round(sec * 1e3, 4), "algorithmic_bytes": nbytes,
                             "achieved_gbs": round(nbytes / sec / 1e9, 1), "frac": round(nbytes / sec / 1e9 / hbm_gbs, 4)}
    nbytes_per = 4 * L + 24 + 16 * L + 20                  # 524 B / transition at L = 24 (SURVEY 8d)
    # K batches of 4096 in flight: ONE sampling launch draws K stratified batches against the current tree, ONE
    # write-back call applies the K*4096 priorities (later batches win, like K successive reference calls)
    B = 4096
    traffic = ncu_per_traffic()
    for K in (1, 4, 16, 64):
        n = K * B
        u = torch.rand(n, dtype=torch.float64, device=device, generator=g)
        idx = torch.empty(n, dtype=torch.int64, device=device)
        w = torch.empty(n, dtype=torch.float32, device=device)
        prio = torch.rand(n, device=device, generator=g)
        srt = (K == 1)

        def both():
            tree.sample(B, u=u, idx_out=idx, weight_out=w, n_batches=K)
            tree.update_priority(idx, prio, sorted=srt)
        reps = 40 if K <= 16 else 10                        # back-to-back iterations inside one captured graph
        sec = time_kernel_graph(both, reps, torch)
        s_sec = time_kernel_graph(lambda: tree.sample(B, u=u, idx_out=idx, weight_out=w, n_batches=K), reps, torch)
        u_sec = time_kernel_graph(lambda: tree.update_priority(idx, prio, sorted=srt), reps, torch)
        nbytes = n * nbytes_per
        key = "sample+update_16M_B4096" if K == 1 else "sample+update_16M_B4096_x%d_in_flight" % K
        out[key] = {
            "batches_in_flight": K, "us": round(sec * 1e6, 2), "transitions_per_s": round(n / sec, 1),
            "algorithmic_bytes": nbytes, "achieved_gbs": round(nbytes / sec / 1e9, 2),
            "frac": round(nbytes / sec / 1e9 / hbm_gbs, 5), "sample_us": round(s_sec * 1e6, 2),
            "update_us": round(u_sec * 1e6, 2),
            "traffic": traffic.get(K), "traffic_source": "profiles/ncu_full_per_r02.txt" if K in traffic else None}
    for B in (65536, 1 << 20):                              # one large stratified (sorted) batch
        u = torch.rand(B, dtype=torch.float64, device=device, generator=g)
        idx = torch.empty(B, dtype=torch.int64, device=device)
        w = torch.empty(B, dtype=torch.float32, device=device)
        prio = torch.rand(B, device=device, generator=g)

        def both():
            tree.sample(B, u=u, idx_out=idx, weight_out=w)
            tree.update_priority(idx, prio, sorted=True)
        reps = 40 if B <= 65536 else 10
        sec = time_kernel_graph(both, reps, torch)
        s_sec = time_kernel_graph(lambda: tree.sample(B, u=u, idx_out=idx, weight_out=w), reps, torch)
        u_sec = time_kernel_graph(lambda: tree.update_priority(idx, prio, sorted=True), reps, torch)
        nbytes = B * nbytes_per
        out["sample+update_16M_B%d" % B] = {
            "us": round(sec * 1e6, 2), "transitions_per_s": round(B / sec, 1), "algorithmic_bytes": nbytes,
            "achieved_gbs": round(nbytes / sec / 1e9, 2), "frac": round(nbytes / sec / 1e9 / hbm_gbs, 5),
            "sample_us": round(s_sec * 1e6, 2), "update_us": round(u_sec * 1e6, 2)}
    del tree, leaves
    torch.cuda.empty_cache()
    # configs[3] on one GPU: ONE 2^23-leaf shard doing its part of a global batch of 4096 (the sharded sampling kernel
    # with a single-rank virtual top; the multi-GPU run adds the peer state exchange: extras.sharded_per_configs3)
    Ns, Bs, Ls = 1 << 23, 4096, 23
    shard = PrioritizedTree(Ns, device=device, mode="stratified")
    shard.build(torch.empty(Ns, device=device).exponential_(1.0, generator=g))
    idx = torch.empty(Bs, dtype=torch.int64, device=device)
    w = torch.empty(Bs, dtype=torch.float32, device=device)
    prio = torch.rand(Bs, device=device, generator=g)
    all_state = torch.zeros(1, 64, dtype=torch.uint8, device=device)

    def shard_iter():
        all_state.copy_(shard.state.view(1, 64))
        shard.sample_global(1, 0, all_state, Bs, None, idx_out=idx, weight_out=w)
        shard.update_priority(idx, prio, sorted=True)
    sec = time_kernel_graph(shard_iter, 40, torch)
    nbytes = Bs * (4 * Ls + 24 + 16 * Ls + 20)
    out["shard_8M_global_sample+update_B4096"] = {
        "leaves": Ns, "us_per_iteration": round(sec * 1e6, 2), "transitions_per_s": round(Bs / sec, 1),
        "algorithmic_bytes": nbytes, "achieved_gbs": round(nbytes / sec / 1e9, 2),
        "frac_of_one_gpu_hbm": round(nbytes / sec / 1e9 / hbm_gbs, 5)}
    del shard
    torch.cuda.empty_cache()
    # Atari-shaped gather: uint8 frames 84x84, frame_stack 4, batch 512 (configs[4] shapes)
    cap, Bg = 1 << 17, 512
    ring = TransitionRing(cap, (84, 84), frame_stack=4, n_step=3, gamma=0.99, storage_dtype=torch.uint8,
                          obs_scale=True, max_streams=8, staging_rows=64, device=device)
    ring.obs.random_(0, 256, generator=g)
    seq = torch.arange(cap, device=device)
    ring.slot_seq.copy_(seq); ring.prev_link.copy_(seq - 1); ring.next_link.copy_(seq + 1)
    ring.next_link[-1] = -1
    ring.seq = cap
    idx = torch.randint(8, cap - 8, (Bg,), device=device, generator=g)
    o = torch.empty(Bg, 4, 84, 84, device=device); no = torch.empty_like(o)
    r = torch.empty(Bg, 1, device=device); gm = torch.empty(Bg, 1, device=device)
    nt = torch.empty(Bg, 1, dtype=torch.bool, device=device); ac = torch.empty(Bg, 1, dtype=torch.int64, device=device)
    sec = time_kernel_graph(lambda: ring.gather(idx, o, no, r, gm, nt, ac), 40, torch)
    nbytes = Bg * (2 * 4 * 7056 + 2 * 4 * 7056 * 4 + 43)
    out["gather_atari_u8_B512"] = {"us": round(sec * 1e6, 2), "algorithmic_bytes": nbytes,
                                   "achieved_gbs": round(nbytes / sec / 1e9, 1),
                                   "frac": round(nbytes / sec / 1e9 / hbm_gbs, 4)}
    return out


def config_extras(device, torch):
    """The other BASELINE model configurations as learner steps (same LearnerStep graph), short runs:
    configs[0] MinAtar Breakout IDS+IQN+LayerNorm+3-step+target+PER (B=64) and configs[4] IQN 64x64 + IDS on
    Atari-shaped 84x84x4 transitions (B=512, uint8 frame storage)."""
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    out = {}
    specs = {
        "configs[0] minatar_ids_iqn_B64": (prism_b200.minatar_ids_iqn_config(
            device=device, experience_replay_capacity=1 << 18, per_sampling="stratified", replay_max_streams=32,
            replay_staging_rows=32768, use_cuda_graph=False), (10, 10, 4), 3, 1 << 17, 200, np.float32),
        "configs[4] atari_iqn64x64_ids_B512": (prism_b200.atari_iqn_ids_config(
            device=device, experience_replay_capacity=1 << 16, per_sampling="stratified", replay_max_streams=32,
            replay_staging_rows=8192, replay_storage_dtype="uint8", replay_obs_scale_255=True, use_cuda_graph=False),
            (84, 84), 18, 1 << 15, 10, np.uint8),
    }
    for name, (cfg, obs_shape, A, fill, steps, dt) in specs.items():
        torch.manual_seed(123)
        agent = prism_b200.build_agent(cfg, obs_shape if len(obs_shape) == 3 else (cfg.frame_stack_size,) + obs_shape, A)
        buf = prism_b200.build_exp_buffer(cfg)
        rng = np.random.default_rng(5)
        E = int(np.prod(obs_shape))
        done_n = 0
        while done_n < fill:
            n = min(8192, fill - done_n)
            if dt == np.uint8:
                frames = rng.integers(0, 256, (n + 32, E), dtype=np.uint8)
            else:
                frames = (rng.random((n + 32, E), dtype=np.float32) < 0.1).astype(np.float32)
            sid = ((done_n + np.arange(n)) % 32).astype(np.int32)
            buf.extend_batch(sid, frames[:n].reshape((n,) + obs_shape), rng.integers(0, A, n).astype(np.int32),
                             (rng.random(n) < 0.05).astype(np.float32), rng.random(n) < (1 / 500), np.zeros(n, bool),
                             frames[32:32 + n].reshape((n,) + obs_shape))
            done_n += n
        buf._flush()
        step = LearnerStep(buf, agent, batch_size=cfg.batch_size, use_cuda_graph=True)
        for _ in range(3):
            step.step()
        sec = time_kernel(step.step, steps, torch)
        n_params = agent.optimizer.numel
        out[name] = {"ms_per_update": round(sec * 1e3, 4), "updates_per_s": round(1.0 / sec, 2),
                     "transitions_per_s": round(cfg.batch_size / sec, 1), "batch": cfg.batch_size,
                     "parameters": int(n_params), "launches_per_step_ours": step.launches_per_step}
        del step, agent, buf
        torch.cuda.empty_cache()
    return out


def configs4_dp(rank, world, device, pg, torch, dist):
    """BASELINE configs[4] data parallel: IQN 64x64 + IDS on Atari-shaped 84x84x4 transitions, batch 512 PER GPU, one
    shard per rank, global stratified sampling, 73 MB gradient arena through the reduce-scatter-by-pull + fused
    clip/Adam exchange (csrc/peer.cu).  Every rank runs it; returns the max-over-ranks step time."""
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    cfg = prism_b200.atari_iqn_ids_config(device=device, experience_replay_capacity=1 << 15, per_sampling="stratified",
                                          replay_max_streams=32, replay_staging_rows=8192, replay_storage_dtype="uint8",
                                          replay_obs_scale_255=True, use_cuda_graph=False)
    torch.manual_seed(123)
    agent = prism_b200.build_agent(cfg, (cfg.frame_stack_size, 84, 84), 18)
    buf = prism_b200.build_exp_buffer(cfg)
    rng = np.random.default_rng(50 + rank)
    fill, done_n, E = 1 << 14, 0, 84 * 84
    while done_n < fill:
        n = min(8192, fill - done_n)
        frames = rng.integers(0, 256, (n + 32, E), dtype=np.uint8)
        sid = ((done_n + np.arange(n)) % 32).astype(np.int32)
        buf.extend_batch(sid, frames[:n].reshape((n, 84, 84)), rng.integers(0, 18, n).astype(np.int32),
                         (rng.random(n) < 0.05).astype(np.float32), rng.random(n) < (1 / 500), np.zeros(n, bool),
                         frames[32:32 + n].reshape((n, 84, 84)))
        done_n += n
    buf._flush()
    if world > 1:
        dist.broadcast(agent.optimizer.arena, src=0)
    step = LearnerStep(buf, agent, batch_size=cfg.batch_size, use_cuda_graph=True, process_group=pg, rank=rank,
                       world_size=world, prefetch=True)
    for _ in range(3):
        step.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    reps = 10
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        step.step()
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) * 1e-3 / reps], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item())
    if step.peer is not None:
        step.peer.check()
    out = {"ms_per_update": round(sec * 1e3, 4), "updates_per_s": round(1.0 / sec, 2), "batch_per_gpu": cfg.batch_size,
           "global_batch": cfg.batch_size * world, "transitions_per_s": round(cfg.batch_size * world / sec, 1),
           "parameters": int(agent.optimizer.numel), "exchange": getattr(step, "exchange", None),
           "launches_per_step_ours": step.launches_per_step}
    del step, agent, buf
    torch.cuda.empty_cache()
    return out


def cpu_baseline(steps, fill, budget_s=25.0, batch=BATCH, warmup=3):
    """The oracle port (reference algorithm restated for the CPU) on the host cores: Python linked-list
    buffer + C sum-tree (1 thread, like torchrl) + PyTorch CPU agent (all intra-op threads)."""
    import torch
    from oracle.agent_oracle import OracleAgent
    from oracle.buffer_oracle import OracleTimestepBuffer, Step, StreamLinker
    import prism_b200
    BATCH = int(batch)                                       # noqa: N806 (shadows the module constant on purpose)
    cfg = prism_b200.minatar_dqn_per_config(device="cpu", batch_size=BATCH)
    torch.manual_seed(123)
    agent = OracleAgent(cfg, OBS_SHAPE, N_ACTIONS)
    buf = OracleTimestepBuffer(CAPACITY, BATCH, frame_stack=1, n_step=3, gamma=0.99)
    trace = Trace(4, int(np.prod(OBS_SHAPE)), N_ACTIONS, N_STREAMS)
    ids = [0]

    def make_step():
        ids[0] += 1
        return Step(ids[0])

    linkers = {}

    def feed(n):
        c = trace.chunk(n)
        for j in range(n):
            s = int(c["stream"][j])
            if s not in linkers:
                linkers[s] = StreamLinker(c["obs"][j].reshape(OBS_SHAPE), make_step)
            buf.extend(linkers[s].step(int(c["action"][j]), float(c["reward"][j]), bool(c["done"][j]), bool(c["trunc"][j]),
                                       c["next_obs"][j].reshape(OBS_SHAPE), c["next_obs"][j].reshape(OBS_SHAPE)))

    feed(fill)
    rng = np.random.default_rng(1)
    buf.tree.update_priority(np.arange(fill), rng.exponential(1.0, fill).astype(np.float32))

    def one():
        feed(STEPS_PER_ITER)
        batch, info = buf.sample(u=rng.random(BATCH), mode=1)
        tb = {"observation": torch.from_numpy(batch["observation"]),
              "next": {"observation": torch.from_numpy(batch["next"]["observation"]),
                       "reward": torch.from_numpy(batch["next"]["reward"])},
              "nonterminal": torch.from_numpy(batch["nonterminal"]), "gamma": torch.from_numpy(batch["gamma"]),
              "action": torch.from_numpy(batch["action"])}
        out = agent.update(tb, torch.from_numpy(info["_weight"]))
        buf.update_priority(info["index"], out["td"].numpy())

    for _ in range(max(3, warmup)):
        one()
    t0 = time.perf_counter()
    n = 0
    while n < steps and (budget_s is None or time.perf_counter() - t0 < budget_s):
        one()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": BATCH * n / dt, "unit": "transitions/s", "updates_per_s": n / dt, "cores": torch.get_num_threads(),
            "kind": "port",
            "sample": "%d hot-loop iterations after %d warm-ups (4 new steps, sample %d, DQN update, priority "
                      "write-back) on a 1M-capacity buffer holding %d transitions; Python linked-list store + "
                      "single-thread C tree + torch CPU agent" % (n, max(3, warmup), BATCH, fill),
            "ms_per_step": dt / max(n, 1) * 1e3, "host_cpus": os.cpu_count(), "batch": BATCH, "fill": fill}


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    device = "cuda:%d" % local
    torch.cuda.set_device(local)
    pg = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")             # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device(device))
        pg = dist.group.WORLD
    hbm_gbs, peak_src = peaks()
    from prism_b200 import _lib
    from prism_b200.learner_step import LearnerStep

    cfg, agent, buf, trace, ingest_s = build_ours(rank, world, device, CAPACITY, CAPACITY, seed=4)
    if world > 1:                                            # identical weights on every rank
        dist.broadcast(agent.optimizer.arena, src=0)
        if agent.target_model is not None:
            dist.broadcast(agent.target_model._flat_arena, src=0)
    # prefetch of the next batch: on the tail branch at 1 GPU; at N > 1 beside the gradient pulls + optimizer sweep,
    # right after the step's single cross-GPU handshake (which carries the shard states the sampling needs)
    prefetch = os.environ.get("PB_PREFETCH", "1") != "0"
    step = LearnerStep(buf, agent, batch_size=BATCH, use_cuda_graph=True, process_group=pg, rank=rank, world_size=world,
                       prefetch=prefetch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident metric: W warm-up + K timed graph replays -----------------
    # Every iteration ingests STEPS_PER_ITER new transitions (like the reference loop and like the CPU arm), samples,
    # gathers, updates and writes the priorities back.  Here the new steps' staged blocks (rows + link records + the
    # iteration's uniforms) are planned on the host BEFORE the timed region and parked in HBM: the timed loop only
    # copies a block device-to-device into the staging slot and replays the step graph.
    # clocks are sampled (NVML, every 5 ms) only inside the two timed regions (device-resident and e2e)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        clocks.window(False)
    n_warm = max(3, args.warmup)
    rng_u = np.random.default_rng(2)               # global stratified sampling: every rank must see the SAME uniforms
    n_res = n_warm + args.steps
    pre = trace.chunk(n_res * STEPS_PER_ITER)
    pre_u = rng_u.random((n_res, step.B_global))

    def ingest_slice(src, i):
        sl = slice(i * STEPS_PER_ITER, (i + 1) * STEPS_PER_ITER)
        return (src["stream"][sl], src["obs"][sl], src["action"][sl], src["reward"][sl], src["done"][sl], src["trunc"][sl],
                src["next_obs"][sl])

    pool = torch.stack([step.plan_ingest(ingest_slice(pre, i), u=pre_u[i]) for i in range(n_res)]).to(device)
    torch.cuda.synchronize()
    graph_ok = True
    try:
        for i in range(n_warm):
            step.step(ingest_block=pool[i])
        torch.cuda.synchronize()
    except Exception as e:                                    # e.g. capture refused: fall back to eager launches
        graph_ok = False
        sys.stderr.write("graph capture failed (%r); running the step eagerly\n" % (e,))
        step.use_cuda_graph = False
        for i in range(n_warm):
            step.step(ingest_block=pool[i])
    barrier()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.window(True)
    ev0.record()
    for i in range(args.steps):
        step.step(ingest_block=pool[n_warm + i])
    ev1.record()
    barrier()
    clocks.window(False)
    sec = ev0.elapsed_time(ev1) * 1e-3
    if world > 1:
        t = torch.tensor([sec], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    lp = step.launches_per_step if graph_ok else None
    exchange = getattr(step, "exchange", None) if world > 1 else None
    gpu_launches = (lp * args.steps) if lp is not None else (_lib.launch_count() - launches0)
    value = BATCH * world * args.steps / sec
    del pool
    dump = args.dump_outputs is not None and rank == 0
    outputs = step_outputs(step) if dump else None

    # ---------------- end-to-end through the public API with host buffers ----------------------
    # synthetic host inputs are generated BEFORE the timed region; the timed loop copies them through pinned
    # staging (H2D), runs the step, and reads the loss back (D2H)
    e2e_steps = args.steps
    n_pre = max(3, args.warmup) + e2e_steps
    pre = trace.chunk(n_pre * STEPS_PER_ITER)
    pre_u = rng_u.random((n_pre, step.B_global))
    u_hosts = [torch.empty(step.B_global, dtype=torch.float64).pin_memory() for _ in range(2)]
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    tick = [0]

    def e2e_one():
        # one call of the public API per iteration: the new steps (host arrays) are staged in pinned memory, copied and
        # scattered inside the step graph (FusedIngest); uniforms go up, the loss comes back
        i = tick[0]
        tick[0] += 1
        sl = slice(i * STEPS_PER_ITER, (i + 1) * STEPS_PER_ITER)
        u_host = u_hosts[i & 1]             # double-buffered: the previous step's async H2D may still be queued
        u_host.numpy()[:] = pre_u[i]
        step.step(u=u_host, ingest=(pre["stream"][sl], pre["obs"][sl], pre["action"][sl], pre["reward"][sl],
                                    pre["done"][sl], pre["trunc"][sl], pre["next_obs"][sl]))
        # the loss read-back (D2H, 4 bytes into a pinned scalar) is a node of the step graph: step.loss_host
    loss_host = step.enable_loss_readback()
    for _ in range(max(3, args.warmup)):
        e2e_one()
    barrier()
    t0 = time.perf_counter()
    clocks.window(True)
    ev0.record()
    for _ in range(e2e_steps):
        e2e_one()
    ev1.record()
    barrier()
    clocks.window(False)
    e2e_sec = max(ev0.elapsed_time(ev1) * 1e-3, 0.0)
    wall = time.perf_counter() - t0
    clk = clocks.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([e2e_sec], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_sec = float(t.item())
    h2d = step.ingest.h2d_bytes                       # staged steps + the fp64 uniforms, one block per iteration
    e2e = {"value": BATCH * world * e2e_steps / e2e_sec, "unit": "transitions/s", "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": 4, "updates_per_s": e2e_steps / e2e_sec,
           "host_wall_s": round(wall, 4), "loss": float(loss_host)}
    if dump:
        outputs.update(step_outputs(step, prefix="e2e_"))
        dump_outputs(args.dump_outputs, outputs)

    sharded = cfg4 = None
    if world > 1 and not args.quick:
        try:
            sharded = sharded_per_microbench(step, rank, world, device, torch, dist, hbm_gbs)
        except Exception as e:
            sharded = {"error": repr(e)[:300]}
        try:
            if step.peer is not None:
                step.peer.check()
            cfg4 = configs4_dp(rank, world, device, pg, torch, dist)
        except Exception as e:
            cfg4 = {"error": repr(e)[:300]}
    if rank != 0:
        _finish(world, dist)
        return
    # ---------------- roofline + extras + CPU baseline (rank 0) ---------------------------------
    roof, ktable = kernel_rooflines(step, buf, agent, torch, hbm_gbs, peak_src)
    extras = {"kernels_at_step_shapes": ktable, "ingest_transitions_per_s": round(CAPACITY / ingest_s, 1),
              "launches_per_step_ours": lp, "graph": graph_ok}
    if sharded is not None:
        extras["sharded_per_configs3"] = sharded
    if cfg4 is not None:
        extras["configs4_data_parallel"] = cfg4
    cpu = None
    if world == 1 and not args.quick:
        del step
        extras["per_microbench"] = per_microbench(device, torch, hbm_gbs)
        try:
            extras["tc_gemm"] = tc_gemm_microbench(device, torch)
        except Exception as e:
            extras["tc_gemm"] = {"error": repr(e)[:300]}
        del agent, buf
        torch.cuda.empty_cache()
        try:
            extras["other_configs"] = config_extras(device, torch)
        except Exception as e:                       # never lose the headline line to an extra
            extras["other_configs"] = {"error": repr(e)[:300]}
        try:
            extras["torch_gpu_baseline"] = torch_gpu_baseline(device, torch)
        except Exception as e:
            extras["torch_gpu_baseline"] = {"error": repr(e)[:300]}
        try:
            extras["rooflines"] = config_rooflines(extras, hbm_gbs, extras["tc_gemm"].get("tf32_peak_tflops", tensor_peak() / 2))
        except Exception as e:
            extras["rooflines"] = {"error": repr(e)[:300]}
        from prism_b200.agents import ops as _ops
        extras["routes"] = _ops.route_counts()
        extras["library_fallthroughs"] = _ops.fallthrough_count()
        # same buffer fill and batch as our arm; bounded to ~25 s of timed CPU work (the fill itself takes about as long)
        cpu = cpu_baseline(steps=400, fill=CAPACITY, budget_s=25.0, warmup=20)
    line = {
        "metric": METRIC,
        "value": value, "unit": "transitions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "learner_updates_per_s": args.steps / sec,
        "config": {"workload": "configs[1]: MinAtar SpaceInvaders-shaped (10x10x6) DQN + double-Q + PER, 1M-capacity "
                               "shard per GPU, batch 256 per GPU, 3-step returns, stratified sampling",
                   "capacity_per_gpu": CAPACITY, "batch_per_gpu": BATCH, "global_batch": BATCH * world,
                   "obs_shape": list(OBS_SHAPE), "n_step": 3, "parallelism": "dp%d (buffer sharded by collector)" % world,
                   "exchange": ("NVLink peer-memory kernels (csrc/peer.cu): state all-gather + one-shot gradient all-reduce fused "
                                "with clip+Adam" if exchange == "peer" else ("NCCL all-gather + all-reduce" if exchange else None)),
                   "l2": "inputs larger than L2: each step gathers random rows of a 2.4 GB ring; the 16 MB "
                         "sum/min trees are L2-resident by design"},
        "clocks": clk, "e2e": e2e, "gpu_launches": int(gpu_launches), "roofline": roof, "cpu_baseline": cpu,
        "extras": extras,
    }
    print(json.dumps(line))
    _finish(world, dist)


def _finish(world, dist):
    """Leave together.  The captured graph holds NCCL work: tearing the process group down under it
    can block, so ranks synchronise once more and exit without the teardown."""
    sys.stdout.flush()
    if world > 1:
        import torch
        dist.barrier()
        torch.cuda.synchronize()
        sys.stderr.flush()
        os._exit(0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    # like for like with our arm at N GPUs: the global batch (256 per GPU) on the host and a 1M-filled buffer.  Exactly
    # --steps timed iterations; short cold runs overstate the GPU/CPU ratio, so compare at a few hundred steps
    steps, warmup = args.steps, max(3, args.warmup)
    fill = int(os.environ.get("PB_REF_FILL", CAPACITY))      # tests shrink the fill; the driver's run uses the full 1M
    cpu = cpu_baseline(steps=steps, fill=fill, budget_s=None, batch=BATCH * world, warmup=warmup)
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": cpu["value"], "unit": "transitions/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": cpu["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "learner_updates_per_s": cpu["updates_per_s"],
        "config": {"workload": "configs[1]: MinAtar SpaceInvaders-shaped (10x10x6) DQN + double-Q + PER, 1M-capacity "
                               "buffer (filled), global batch %d (256 per GPU of the other arm), 3-step returns, 4 new "
                               "steps ingested per iteration -- reference algorithm on the host CPU" % (BATCH * world),
                   "global_batch": BATCH * world,
                   "note": "the reference is pure Python + torchrl (absent): this arm times the oracle port of its "
                           "algorithm (oracle/buffer_oracle.py, oracle/per_oracle.c, oracle/agent_oracle.py); "
                           "single process, rank 0 only"},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="skip extras and the CPU baseline (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, TD errors, batch, parameters, priorities; "
                         "e2e_* for the end-to-end leg) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU arm's step; the reference arm has none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
