"""Uniform replay (use_per=False, the reference's default config): the device sampler of csrc/uniform.cu against a float64
numpy oracle and the eager TimestepBuffer.sample path, the one-graph LearnerStep against the eager update loop, the
length bookkeeping of the fused ingest, and sharded global sampling (loopback peers, two processes)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rel_err

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
SEED = 0x5EED
gpu = pytest.mark.gpu


# ---- oracle: the same IEEE operations in the same order, float64 numpy ------------------------------------------------
def oracle_index(u, length, mode):
    u = np.asarray(u, np.float64)
    k = np.arange(u.size, dtype=np.float64)
    x = u * np.float64(length) if mode == 0 else ((k + u) / np.float64(u.size)) * np.float64(length)
    return np.minimum(x.astype(np.int64), length - 1)


def oracle_philox(seed, call, n):
    """philox_uniform of csrc/common.cuh: Philox4x32-10, counter (k, call), 53 bits -> [0, 1)."""
    m = np.uint64(0xFFFFFFFF)
    k = np.arange(n, dtype=np.uint64)
    c0, c1 = k & m, k >> np.uint64(32)
    c2, c3 = np.full(n, call, np.uint64), np.full(n, 0x50455221, np.uint64)
    k0, k1 = np.uint64(seed), np.uint64(0x9E3779B9 ^ seed)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return ((c0 >> np.uint64(5)).astype(np.float64) * 67108864.0 + (c1 >> np.uint64(6)).astype(np.float64)) \
        * (1.0 / 9007199254740992.0)


# ---- CPU: argument checks before any launch ---------------------------------------------------------------------------
def test_null_state_and_pointers_are_rejected_without_a_launch():
    from prism_b200 import _lib
    lib = _lib.load()
    before = lib.pb_launch_count()
    buf = (C.c_longlong * 8)()
    w = (C.c_float * 8)()
    st = (C.c_ubyte * 128)()
    group = _lib.pb_peer_group(world=2, rank=0)
    E = -1
    assert lib.pb_uniform_init(None, 16, 0, SEED, None) == E
    assert lib.pb_uniform_extend(None, 16, 4, None) == E
    assert lib.pb_uniform_sample(None, 8, None, 0, buf, w, None) == E
    assert lib.pb_uniform_sample(st, 8, None, 0, None, w, None) == E
    assert lib.pb_uniform_sample(st, 8, None, 2, buf, w, None) == E
    assert lib.pb_uniform_sample_global(None, 2, 0, st, 8, None, buf, w, None, None) == E
    assert lib.pb_uniform_sample_global(st, 2, 0, None, 8, None, buf, w, None, None) == E
    assert lib.pb_uniform_sample_global(st, 2, 2, st, 8, None, buf, w, None, None) == E
    assert lib.pb_uniform_sample_global_peer(None, C.byref(group), 8, None, buf, w, None, None) == E
    assert lib.pb_uniform_sample_global_peer(st, None, 8, None, buf, w, None, None) == E
    assert lib.pb_uniform_sample_global_peer(st, C.byref(group), 8, None, buf, w, None, None) == E   # no pads mapped
    assert lib.pb_launch_count() == before


def test_uniform_sampler_refuses_a_cpu_device():
    from prism_b200 import UniformSampler, _lib
    with pytest.raises(_lib.PbError):
        UniformSampler(16, device="cpu")


# ---- 1. the sampler against the oracle --------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_sampler_matches_float64_oracle(mode):
    from prism_b200 import UniformSampler
    size, B = 1000, 512
    s = UniformSampler(size, mode=mode, device=DEV)
    rng = np.random.default_rng(3 + mode)
    edge = np.array([0.0, np.nextafter(1.0, 0.0), 0.5, np.nextafter(0.5, 1.0)])
    for seq in (1, 7, 999, 1000, 1000 + 37, 5 * 1000 + 3):               # len < size, full, after wrap
        s.reset(seq)
        length = min(seq, size)
        u = np.concatenate([edge, rng.random(B - edge.size)])
        idx, w = s.sample(B, u=torch.from_numpy(u).to(DEV))
        assert np.array_equal(idx.cpu().numpy(), oracle_index(u, length, mode)), seq
        assert bool((w == 1.0).all())
        st = s.state_host()
        assert (st["len"], st["seq"], st["status"]) == (length, seq, 0)
    s.reset(990)
    s.extend(4)
    s.extend(40)
    st = s.state_host()
    assert (st["len"], st["seq"]) == (1000, 1034)
    # device draws: Philox keyed by the seed, one call number per launch
    for call in range(3):
        idx, w = s.sample(B)
        assert np.array_equal(idx.cpu().numpy(), oracle_index(oracle_philox(SEED, call, B), 1000, mode))
    assert s.state_host()["call"] == 3
    s.reset(0)
    idx, w = s.sample(8)
    assert s.state_host()["status"] == 1 and float(w.sum()) == 0.0          # PB_ST_EMPTY


# ---- 2. the eager uniform path of TimestepBuffer.sample -----------------------------------------------------------------
def _script(seed, n, obs_shape=(10, 10, 6), A=4):
    """n collector steps as the tuple extend_batch / step(ingest=...) take."""
    from oracle.gen_golden import make_script
    S = make_script(seed, n_streams=4, n_steps=n, obs_shape=obs_shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])
    shp = (-1,) + obs_shape
    return (S["stream"], S["obs"].reshape(shp), S["action"], S["reward"], S["done"], S["trunc"], succ.reshape(shp))


def _chunk(rows, a, b):
    return tuple(x[a:b] for x in rows)


def _uniform_cfg(cap, B, **kw):
    import prism_b200
    return prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=cap, batch_size=B, use_per=False,
                                             replay_max_streams=4, replay_staging_rows=64, use_cuda_graph=False, **kw)


@gpu
def test_kernel_equals_the_eager_uniform_path():
    import prism_b200
    from prism_b200 import UniformSampler
    cap, B = 256, 64
    buf = prism_b200.build_exp_buffer(_uniform_cfg(cap, B))
    assert buf.buffer._sampler is None
    rows = _script(21, 700)
    s = UniformSampler(cap, device=DEV)
    rng = np.random.default_rng(8)
    for a, b in ((0, 100), (100, 300), (300, 700)):                        # len < size, then after wraps
        buf.extend_batch(*_chunk(rows, a, b))
        buf._flush()
        s.reset(buf.buffer._storage.seq)
        u = rng.random(B)
        u[0] = np.nextafter(1.0, 0.0)
        buf.inject_uniforms(torch.from_numpy(u.copy()))
        buf.sample()
        want = buf._idx.clone()
        idx, _ = s.sample(B, u=torch.from_numpy(u).to(DEV), mode="iid")
        assert torch.equal(idx, want), b


# ---- 3. LearnerStep == the eager update loop ----------------------------------------------------------------------------
def _setup(cap, B, rows, n0, seed=0):
    import prism_b200
    cfg = _uniform_cfg(cap, B)
    torch.manual_seed(seed)
    agent = prism_b200.build_agent(cfg, (10, 10, 6), 4)
    buf = prism_b200.build_exp_buffer(cfg)
    buf.extend_batch(*_chunk(rows, 0, n0))
    buf._flush()
    return agent, buf


def _batch_of(b, idx):
    return (idx.clone(), b["observation"].clone(), b["next"]["observation"].clone(), b["next"]["reward"].clone(),
            b["gamma"].clone(), b["nonterminal"].clone(), b["action"].clone())


def _eager_loop(rows, n0, batch_u, between=None):
    """buf.inject_uniforms(u); agent.update(buf.sample()) with ``between(i, buf)`` before update i."""
    cap, B = 256, 16
    agent, buf = _setup(cap, B, rows, n0)
    losses, batches = [], []
    for i, u in enumerate(batch_u):
        if between is not None:
            between(i, buf)
        buf.inject_uniforms(torch.from_numpy(np.ascontiguousarray(u)))
        b = buf.sample()
        batches.append(_batch_of(b, buf._idx))
        agent.update(b)
        losses.append(float(agent._static_total_loss))
    torch.cuda.synchronize()
    return losses, batches, agent.optimizer.arena.clone()


def _assert_same_training(a, b):
    la, ba, pa = a
    lb, bb, pb = b
    assert len(ba) == len(bb)
    for i, (x, y) in enumerate(zip(ba, bb)):
        for p, q in zip(x, y):
            assert torch.equal(p, q), i
    assert np.allclose(la, lb, rtol=1e-5, atol=1e-7), (la, lb)
    assert rel_err(pa.cpu().numpy(), pb.cpu().numpy()) < 1e-5


@gpu
@pytest.mark.parametrize("host_u", [True, False])
@pytest.mark.parametrize("prefetch", [False, True])
@pytest.mark.parametrize("use_graph", [True, False])
def test_step_equals_the_eager_update_loop(use_graph, prefetch, host_u):
    from prism_b200.learner_step import LearnerStep
    B, n0, iters = 16, 200, 8
    rows = _script(5, n0)
    us = np.random.default_rng(11).random((iters, B))
    agent, buf = _setup(256, B, rows, n0)
    step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=use_graph, prefetch=prefetch)
    assert step.uniform and step.launches_per_step is None
    losses, batches = [], []
    for i in range(iters):
        total = step.step(u=torch.from_numpy(us[i].copy()) if host_u else None)
        losses.append(float(total))
        batches.append(_batch_of(step.batch, step.idx[:B]))
    torch.cuda.synchronize()
    got = (losses, batches, agent.optimizer.arena.clone())
    if use_graph:
        assert step.launches_per_step > 0
    # the uniforms each batch was drawn with: host uniforms drive the NEXT batch under prefetch (the first one is
    # primed from the device generator); device draws take one call number per batch
    if host_u:
        batch_u = [oracle_philox(SEED, 0, B)] + list(us[:-1]) if prefetch else list(us)
    else:
        batch_u = [oracle_philox(SEED, c, B) for c in range(iters)]
    _assert_same_training(got, _eager_loop(rows, n0, batch_u))


# ---- 4. fused ingest and the device length ------------------------------------------------------------------------------
def _fused_run(rows, n0, us, n_new, mode, use_graph=True, prefetch=False):
    """mode: "fused" step(u, ingest=...), "push" step(u) then an ingest_graph push, "planned" plan_ingest ahead +
    step(ingest_block=...)."""
    from prism_b200.learner_step import LearnerStep
    B = us.shape[1]
    agent, buf = _setup(256, B, rows, n0)
    step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=use_graph, prefetch=prefetch)
    iters = us.shape[0]
    new = [_chunk(rows, n0 + i * n_new, n0 + (i + 1) * n_new) for i in range(iters)]
    push = buf.ingest_graph(n_new) if mode == "push" else None
    pool = None
    if mode == "planned":
        pool = torch.stack([step.plan_ingest(new[i], u=us[i]) for i in range(iters)]).to(DEV)
        torch.cuda.synchronize()
    losses = []
    for i in range(iters):
        if mode == "fused":
            losses.append(float(step.step(u=torch.from_numpy(us[i].copy()), ingest=new[i])))
        elif mode == "push":
            losses.append(float(step.step(u=torch.from_numpy(us[i]).to(DEV))))
            push(*new[i])
        else:
            losses.append(float(step.step(ingest_block=pool[i])))
    torch.cuda.synchronize()
    ring = buf.buffer._storage
    st = step.tree.state_host()
    return losses, agent.optimizer.arena.clone(), ring.obs.clone(), ring.next_link.clone(), (st["len"], st["seq"]), ring.seq


@gpu
@pytest.mark.parametrize("use_graph", [True, False])
def test_fused_ingest_step_equals_step_then_push(use_graph):
    n0, n_new, iters, B = 200, 4, 9, 16
    rows = _script(5, n0 + n_new * iters)
    us = np.random.default_rng(12).random((iters, B))
    a = _fused_run(rows, n0, us, n_new, "fused", use_graph)
    b = _fused_run(rows, n0, us, n_new, "push", use_graph)
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    # the fused run's device length counts every consumed block; the push run's was set from the ring at each step
    assert a[4] == (min(a[5], 256), a[5]) and b[5] == a[5]


@gpu
@pytest.mark.parametrize("prefetch", [False, True])
def test_blocks_planned_ahead_keep_the_device_length(prefetch):
    """bench.py's resident leg plans its whole pool of ingest blocks before the first step: the host ring.seq runs many
    blocks ahead of what the device has consumed.  Training must equal feeding the same steps one call at a time."""
    n0, n_new, iters, B = 200, 4, 9, 16
    rows = _script(6, n0 + n_new * iters)
    us = np.random.default_rng(13).random((iters, B))
    a = _fused_run(rows, n0, us, n_new, "planned", prefetch=prefetch)
    b = _fused_run(rows, n0, us, n_new, "fused", prefetch=prefetch)
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert a[4] == b[4] == (min(n0 + n_new * iters, 256), n0 + n_new * iters)


@gpu
@pytest.mark.parametrize("host_u", [True, False])
@pytest.mark.parametrize("use_graph", [True, False])
def test_outside_extend_and_empty_refill_between_steps(use_graph, host_u):
    """extend_batch, then empty() + a refill, between steps: the step re-reads the ring's length (and keeps the
    device generator's position) and trains exactly like the eager loop doing the same."""
    from prism_b200.learner_step import LearnerStep
    B, n0, iters = 16, 120, 8
    rows = _script(7, n0 + 60)
    refill = _script(8, 90)
    us = np.random.default_rng(14).random((iters, B))

    def between(i, buf):
        if i == 3:
            buf.extend_batch(*_chunk(rows, n0, n0 + 60))
        if i == 5:
            buf.empty()
            buf.extend_batch(*refill)

    agent, buf = _setup(256, B, rows, n0)
    step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=use_graph)
    losses, batches, lens = [], [], []
    for i in range(iters):
        between(i, buf)
        losses.append(float(step.step(u=torch.from_numpy(us[i].copy()) if host_u else None)))
        batches.append(_batch_of(step.batch, step.idx[:B]))
        lens.append(step.tree.state_host()["len"])
    torch.cuda.synchronize()
    assert lens == [120] * 3 + [180] * 2 + [90] * 3
    batch_u = list(us) if host_u else [oracle_philox(SEED, c, B) for c in range(iters)]
    _assert_same_training((losses, batches, agent.optimizer.arena.clone()), _eager_loop(rows, n0, batch_u, between))


# ---- 5. sharded global sampling: loopback peers --------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("device_u", [False, True])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_peer_global_sampling_equals_gathered_and_the_concatenation(world, device_u):
    from prism_b200 import UniformSampler
    from prism_b200.peer import PeerGroup
    C_, B = 4096, 512
    rng = np.random.default_rng(40 + world)
    groups = PeerGroup.loopback(world, 1024, DEV)
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    seqs = [int(x) for x in rng.integers(1, 3 * C_, world)]
    seqs[1] = 17                                                         # unequal, one almost empty
    if world >= 4:
        seqs[2] = 0                                                      # an empty shard owns no stratum
    peer_s = [UniformSampler(C_, seq=q, device=DEV) for q in seqs]
    ref_s = [UniformSampler(C_, seq=q, device=DEV) for q in seqs]
    lens = [min(q, C_) for q in seqs]
    prefix = np.concatenate([[0], np.cumsum(lens)])
    total = int(prefix[-1])
    one = UniformSampler(total, mode="stratified", seq=total, device=DEV)
    out = [[torch.empty(B, dtype=torch.int64, device=DEV), torch.empty(B, device=DEV),
            torch.empty(B, dtype=torch.int64, device=DEV)] for _ in range(world)]
    ref = [[torch.empty(B, dtype=torch.int64, device=DEV), torch.empty(B, device=DEV),
            torch.empty(B, dtype=torch.int64, device=DEV)] for _ in range(world)]
    for it in range(3):
        u = None if device_u else torch.from_numpy(rng.random(B)).to(DEV)
        torch.cuda.synchronize()
        all_state = torch.stack([s.state for s in ref_s]).contiguous()
        for r in range(world):
            ref_s[r].sample_global(world, r, all_state, B, u, idx_out=ref[r][0], weight_out=ref[r][1], stratum_out=ref[r][2])
        want, _ = one.sample(B, u=u)
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                groups[r].state_put(peer_s[r].state)
                peer_s[r].sample_global_peer(groups[r], B, u, idx_out=out[r][0], weight_out=out[r][1],
                                             stratum_out=out[r][2])
        torch.cuda.synchronize()
        got = np.full(B, -1, np.int64)
        for r in range(world):
            groups[r].check()
            for a, b in zip(out[r], ref[r]):
                assert torch.equal(a, b), (it, r)
            st = peer_s[r].state_host()
            lo, n = st["owned_lo"], st["owned_n"]
            assert (lo, n) == (ref_s[r].state_host()["owned_lo"], ref_s[r].state_host()["owned_n"])
            assert np.array_equal(out[r][2][:n].cpu().numpy(), np.arange(lo, lo + n))
            assert bool((out[r][1][:n] == 1.0).all()) and float(out[r][1][n:].abs().sum()) == 0.0
            assert bool((out[r][0][n:] == -1).all()) and bool((out[r][2][n:] == -1).all())
            idx = out[r][0][:n].cpu().numpy()
            assert n == 0 or (idx.min() >= 0 and idx.max() < lens[r])
            got[lo:lo + n] = idx + prefix[r]
        assert np.array_equal(got, want.cpu().numpy()), it               # every stratum once, as one big sampler
        calls = {s.state_host()["call"] for s in peer_s + ref_s + [one]}
        assert calls == {it + 1 if device_u else 0}
    if device_u:
        assert np.array_equal(oracle_index(oracle_philox(SEED, 2, B), total, 1), want.cpu().numpy())


# ---- 6. two processes on two GPUs ----------------------------------------------------------------------------------------
def _run(cmd):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=540)
    assert p.returncode == 0, p.stdout[-3000:]


@gpu
@pytest.mark.parametrize("prefetch", [0, 1])
def test_two_ranks_equal_one_rank_on_the_union_buffer(tmp_path, prefetch):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = os.path.join(HERE, "mp_worker_dp_uniform.py")
    out2, out1 = str(tmp_path / "dp2"), str(tmp_path / "one")
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
          "127.0.0.1", "--master-port", str(29720 + prefetch), worker, "--out", out2, "--prefetch", str(prefetch)])
    _run([sys.executable, worker, "--out", out1, "--union", "2", "--prefetch", str(prefetch)])
    one = torch.load(out1 + ".rank0", weights_only=False)
    r0, r1 = (torch.load(out2 + ".rank%d" % r, weights_only=False) for r in (0, 1))
    assert r0["exchange"] == "peer", "the ranks could not map each other's memory: peer path not exercised"
    assert torch.equal(r0["arena"], r1["arena"]), "replicas diverged"
    # every step, the two ranks' batches together are the union's batch, row for row
    for a, b, want in zip(r0["rows"], r1["rows"], one["rows"]):
        assert torch.equal(torch.cat([a, b]), want)
    B_pad, B_global = r0["B_pad"], one["B_pad"]
    both = (np.asarray(r0["losses"]) + np.asarray(r1["losses"])) * (B_pad / B_global)
    assert np.allclose(both, one["losses"], rtol=2e-5, atol=1e-7), (r0["losses"], r1["losses"], one["losses"])
    err = float((r0["arena"] - one["arena"]).abs().max() / one["arena"].abs().max())
    assert err < 2e-5, err
