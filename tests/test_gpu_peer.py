"""Peer-memory exchange kernels (csrc/peer.cu) driven in LOOPBACK: `world` ranks inside one process on one GPU,
each on its own stream with plain pointers to the other ranks' blocks -- same kernels, same flag protocol as the
multi-process CUDA-IPC set-up of LearnerStep (SURVEY 8e)."""

import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


class _Opt:
    """The fields PeerGroup.allreduce_adam reads from FlatAdam."""

    def __init__(self, n, p0, lr=1e-3, max_grad_norm=10.0):
        self.arena = p0.clone()
        self.exp_avg = torch.zeros(n, device=DEV)
        self.exp_avg_sq = torch.zeros(n, device=DEV)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=DEV)
        self.partials = torch.zeros(4096, device=DEV)
        self.norm_out = torch.zeros(2, device=DEV)
        self.lr, self.betas, self.eps, self.max_grad_norm = lr, (0.9, 0.999), 1.5e-4, max_grad_norm


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("n,one_shot", [(4096, True), (1_000_004, True), (1_000_004, False)])
def test_peer_allreduce_adam_matches_single_rank_step(world, n, one_shot, monkeypatch):
    """Both exchange schedules: one-shot (every rank pulls everything, one barrier) and two-shot (reduce-scatter by
    pull + the all-gather fused into the Adam sweep, two barriers)."""
    from prism_b200 import _lib, peer as peer_mod
    from prism_b200.peer import PeerGroup
    monkeypatch.setattr(peer_mod, "ONE_SHOT_MAX_BYTES", (1 << 40) if one_shot else 0)
    monkeypatch.setattr(peer_mod, "FUSED_EXCHANGE", False)     # the multi-launch schedules; the fused one: next test
    _run_allreduce_adam(world, n)


@pytest.mark.parametrize("world,n", [(2, 4096), (4, 4096), (8, 4096), (8, 40_000), (4, 40_000), (2, 100_000),
                                     (4, 100_000), (2, 400_004)])
def test_peer_fused_allreduce_adam_matches_single_rank_step(world, n, monkeypatch):
    """Small arenas: handshake + pulls + global norm + clip + Adam as ONE launch per rank (peer_allreduce_adam_kernel),
    every rank pulling every other rank's whole arena.
    Sizes are bounded here because the loopback ranks share one GPU: every rank's CTAs must be resident at once (in the
    multi-process set-up each rank has its own GPU; tests/test_gpu_multiprocess.py runs that)."""
    from prism_b200 import peer as peer_mod
    monkeypatch.setattr(peer_mod, "FUSED_EXCHANGE", True)
    _run_allreduce_adam(world, n)


def _run_allreduce_adam(world, n):
    from prism_b200 import _lib
    from prism_b200.peer import PeerGroup
    lib = _lib.load()
    groups = PeerGroup.loopback(world, n, DEV)
    g = torch.Generator(device=DEV).manual_seed(n + world)
    p0 = torch.randn(n, device=DEV, generator=g)
    grads = [torch.randn(n, device=DEV, generator=g) * (3.0 if r == 0 else 1.0) for r in range(world)]
    opts = [_Opt(n, p0) for _ in range(world)]
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    # every tensor exists before the first barrier kernel spins: a cudaMalloc (device-wide sync) issued by this single
    # host thread while one loopback rank waits for a rank that is not launched yet would deadlock the test
    staged = [[grads[r] * (1.0 + it) for r in range(world)] for it in range(3)]
    torch.cuda.synchronize()
    for it in range(3):                                       # three steps: epochs, ticket and step counter carry over
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                groups[r].grad_in_flight().copy_(staged[it][r])     # the half this step's exchange reads
                groups[r].allreduce_adam(opts[r])
    torch.cuda.synchronize()
    # reference: the single-rank fused step on the rank-order fp32 sum
    ref = _Opt(n, p0)
    for it in range(3):
        total = grads[0] * (1.0 + it)
        for r in range(1, world):
            total = total + grads[r] * (1.0 + it)
        _lib.check(lib.pb_adam_clip_step(n, ref.arena.data_ptr(), total.data_ptr(), ref.exp_avg.data_ptr(),
                                         ref.exp_avg_sq.data_ptr(), ref.step_count.data_ptr(), ref.lr, 0.9, 0.999, ref.eps,
                                         ref.max_grad_norm, ref.norm_out.data_ptr(), ref.partials.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream), "pb_adam_clip_step")
    torch.cuda.synchronize()
    for r in range(world):
        assert int(opts[r].step_count) == 3
        assert torch.equal(opts[r].arena, opts[0].arena), "replicas must stay bit-identical"
        assert torch.equal(opts[r].exp_avg_sq, opts[0].exp_avg_sq)
    assert rel_err(opts[0].norm_out.cpu().numpy(), ref.norm_out.cpu().numpy()) < 1e-6
    assert rel_err(opts[0].arena.cpu().numpy(), ref.arena.cpu().numpy()) < 1e-6
    assert rel_err(opts[0].exp_avg.cpu().numpy(), ref.exp_avg.cpu().numpy()) < 1e-6


def test_peer_state_allgather_and_barrier():
    from prism_b200.peer import PeerGroup
    world = 4
    groups = PeerGroup.loopback(world, 1024, DEV)
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    for it in range(5):
        states = [torch.randint(0, 256, (64,), dtype=torch.uint8, device=DEV) for _ in range(world)]
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                groups[r].state_allgather(states[r])
                groups[r].barrier()
        torch.cuda.synchronize()
        want = torch.stack(states)
        for r in range(world):
            assert torch.equal(groups[r].all_state, want)


def test_state_put_and_in_kernel_wait_equal_the_gathered_states():
    """The put-based shard-state exchange of LearnerStep: every rank PUTS its state block to every rank (nobody waits),
    the global sampling kernel waits for the puts itself.  4 loopback shards, three rounds with priority updates in
    between: indices / weights / owned strata identical to sample_global on the stacked states."""
    import numpy as np
    from prism_b200 import PrioritizedTree
    from prism_b200.peer import PeerGroup
    world, C, B = 4, 4096, 256
    groups = PeerGroup.loopback(world, 1024, DEV)
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    rng = np.random.default_rng(5)
    shards = []
    for r in range(world):
        t = PrioritizedTree(C, device=DEV, mode="stratified")
        t.build(torch.from_numpy(np.sqrt(rng.exponential(1.0 + r, C).astype(np.float32) + 1e-8)).to(DEV))
        shards.append(t)
    out = [(torch.empty(B, dtype=torch.int64, device=DEV), torch.empty(B, device=DEV),
            torch.empty(B, dtype=torch.int64, device=DEV)) for _ in range(world)]
    ref = [(torch.empty(B, dtype=torch.int64, device=DEV), torch.empty(B, device=DEV),
            torch.empty(B, dtype=torch.int64, device=DEV)) for _ in range(world)]
    for it in range(3):
        u = torch.from_numpy(rng.random(B)).to(DEV)
        prio = [torch.from_numpy(rng.exponential(2.0, B).astype(np.float32)).to(DEV) for _ in range(world)]
        torch.cuda.synchronize()
        all_state = torch.stack([t.state for t in shards]).contiguous()
        for r in range(world):
            shards[r].sample_global(world, r, all_state, B, u, idx_out=ref[r][0], weight_out=ref[r][1], stratum_out=ref[r][2])
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                groups[r].state_put(shards[r].state)
                shards[r].sample_global_peer(groups[r], B, u, idx_out=out[r][0], weight_out=out[r][1], stratum_out=out[r][2])
        torch.cuda.synchronize()
        for r in range(world):
            groups[r].check()
            for a, b in zip(out[r], ref[r]):
                assert torch.equal(a, b), (it, r)
            n = shards[r].state_host()["owned_n"]
            shards[r].update_priority(out[r][0][:n], prio[r][:n], sorted=True)


def test_a_missing_rank_times_out_instead_of_hanging(monkeypatch):
    """Verdict r1 #8: the flag wait is bounded.  Rank 1 of a 2-rank loopback group never launches; rank 0's barrier
    gives up after the timeout, sets its status word, and PeerGroup.check() raises."""
    from prism_b200 import _lib, peer as peer_mod
    from prism_b200.peer import PeerGroup
    monkeypatch.setattr(peer_mod, "WAIT_TIMEOUT_S", 0.2)
    groups = PeerGroup.loopback(2, 1024, DEV)
    groups[0].check()
    groups[0].barrier()
    torch.cuda.synchronize()                                  # returns: the kernel gave up after ~0.2 s
    with pytest.raises(_lib.PbError):
        groups[0].check()
