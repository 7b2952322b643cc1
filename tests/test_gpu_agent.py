"""GPU parity of the agent-side kernels and of the drop-in Agent update against the REFERENCE
outputs frozen in tests/golden/agent_*.npz / ids.npz and against the CPU oracle.
Bar (north star): loss and gradients within 1e-4 relative; IDS / greedy actions identical."""

import numpy as np
import pytest
import torch

from helpers import (cfg_from_fixture, fixture_batch, fixture_state_dict, fixture_taus, load_golden, rel_err,
                     target_transform)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CASES = ["agent_ids_iqn_ln_target", "agent_ids_iqn_double", "agent_dqn_double", "agent_iqn_self"]


def build_product_agent(fx, use_cuda_graph=False):
    import prism_b200
    cfg = cfg_from_fixture(fx, DEV)
    cfg.use_cuda_graph = use_cuda_graph
    agent = prism_b200.build_agent(cfg, tuple(fx["obs_shape"].tolist()), int(fx["n_actions"]))
    sd = fixture_state_dict(fx)
    agent.model.load_state_dict(sd, strict=True)
    if agent.target_model is not None:
        agent.target_model.load_state_dict({k: target_transform(v) for k, v in sd.items()}, strict=True)
    return cfg, agent


def inject_taus(cfg, agent, taus):
    taus = [torch.as_tensor(t, dtype=torch.float32) for t in taus]
    d = agent.model.distribution_model
    if d is None:
        return
    if agent.target_model is None:
        d.tau_queue = list(taus)
    elif cfg.use_double_q_learning:
        d.tau_queue = [taus[0], taus[1]]
        agent.target_model.distribution_model.tau_queue = [taus[2]]
    else:
        d.tau_queue = [taus[0]]
        agent.target_model.distribution_model.tau_queue = [taus[1]]


def reference_named_grads(agent):
    """Gradients keyed like the reference's named_parameters (un-stacking the ensemble heads)."""
    out = {}
    for name, p in agent.model.named_parameters():
        if ".stacked." in name:
            prefix, pos = name.split(".stacked.")
            ens = agent.model.q_function_model
            (seq_idx, pname), = [k for k, v in ens._slot.items() if v == int(pos)]
            for k in range(ens.n_heads):
                out[prefix + "." + ens._ref_key(k, seq_idx, pname)] = p.grad[k]
        else:
            out[name] = p.grad
    return out


@pytest.mark.parametrize("name", CASES)
def test_update_matches_reference_golden(name):
    fx = load_golden(name)
    cfg, agent = build_product_agent(fx)
    inject_taus(cfg, agent, fixture_taus(fx))
    td = agent.update(fixture_batch(fx, DEV), torch.from_numpy(fx["per_weights"]).to(DEV))
    torch.cuda.synchronize()
    if "out.dist" in fx:
        assert rel_err(agent._static_distribution_loss.detach().cpu().numpy(), fx["out.dist"]) < 1e-4
    if "out.q" in fx:
        assert rel_err(agent._static_q_loss.detach().cpu().numpy(), fx["out.q"]) < 1e-4
    assert rel_err(td.cpu().numpy(), fx["out.td"]) < 1e-4
    assert rel_err(agent._static_total_loss.detach().cpu().numpy(), fx["out.total"]) < 1e-4
    coef = float(agent.optimizer.norm_out[1])
    for k, g in reference_named_grads(agent).items():
        assert rel_err(g.cpu().numpy() * coef, fx["grad_clipped." + k]) < 1e-4, k
    after = agent.model.state_dict()
    for k, v in after.items():
        assert rel_err(v.cpu().numpy(), fx["param_after." + k]) < 1e-4, k


@pytest.mark.parametrize("name", [c for c in CASES if "iqn" in c])
def test_acting_matches_reference_golden(name):
    fx = load_golden(name)
    cfg, agent = build_product_agent(fx)
    agent.model.load_state_dict(fixture_state_dict(fx, "param_after."))
    obs = torch.from_numpy(fx["batch.observation"][:, 0]).to(DEV)
    agent.model.distribution_model.tau_queue = [torch.from_numpy(fx["act.tau_model"])]
    with torch.no_grad():
        q, z = agent.model(obs, for_action=True)
    assert rel_err(z.cpu().numpy(), fx["act.z"]) < 1e-4
    if "act.q" in fx:
        assert tuple(q.shape) == fx["act.q"].shape
        assert rel_err(q.cpu().numpy(), fx["act.q"]) < 1e-4
    agent.model.distribution_model.tau_queue = [torch.from_numpy(fx["act.tau_agent"])]
    act = agent.forward(obs)
    assert act.dtype == torch.int64
    assert np.array_equal(act.cpu().numpy(), fx["act.action"])


def test_ids_and_greedy_kernels_match_reference_golden():
    from prism_b200.agents import ops
    fx = load_golden("ids")
    for tag in "abc":
        q = torch.from_numpy(fx[tag + ".q"]).to(DEV)      # (N, A, K)
        z = torch.from_numpy(fx[tag + ".z"]).to(DEV)      # (Nq, N, A)
        act, scores = ops.ids_select(q.permute(2, 0, 1), z, 0.1, 1e-10, 0.25, return_scores=True)
        assert np.array_equal(act.cpu().numpy(), fx[tag + ".action"]), tag
        assert np.allclose(scores.cpu().numpy(), fx[tag + ".scores"], rtol=2e-4, equal_nan=True)
        assert np.array_equal(ops.greedy_select(q.permute(2, 0, 1)).cpu().numpy(), fx[tag + ".greedy"])


@pytest.mark.parametrize("B,T,Tp,A", [(64, 32, 32, 3), (512, 64, 64, 18), (7, 8, 12, 5), (33, 200, 8, 6)])
def test_quantile_huber_kernel_vs_oracle_math(B, T, Tp, A):
    """pb_iqn_qh_loss (loss + gradient in one pass) against the oracle's broadcasted formula + autograd."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(B * 31 + T)
    z_cur = torch.randn(T * B, A, generator=g) * 2
    tau = torch.rand(T * B, 1, generator=g)
    z_on, z_tg = torch.randn(Tp * B, A, generator=g), torch.randn(Tp * B, A, generator=g) * 3
    act = torch.randint(0, A, (B,), generator=g)
    ret, gdn = torch.randn(B, generator=g), torch.rand(B, generator=g)
    gdn[::5] = 0.0
    w = torch.rand(B, generator=g)
    # oracle math (iqn_model.py:129-201) on the CPU
    zc = z_cur.clone().requires_grad_(True)
    best = z_on.view(Tp, B, A).mean(0).argmax(-1)
    y = (torch.tile(ret.view(-1, 1), [Tp, 1]) + torch.gather(z_tg, 1, torch.tile(best.view(-1, 1), [Tp, 1])) *
         torch.tile(gdn.view(-1, 1), [Tp, 1])).view(Tp, B, 1).transpose(1, 0)
    theta = torch.gather(zc, 1, torch.tile(act.view(-1, 1), [T, 1])).view(T, B, 1).transpose(1, 0)
    d = y[:, :, None] - theta[:, None, :]
    small = (d.abs() <= 1.0).float()
    hub = small * 0.5 * d.square() + (1 - small) * (d.abs() - 0.5)
    rho = (tau.view(T, B, 1).transpose(1, 0)[:, None] - (d < 0).float()).abs() * hub
    loss_ref = rho.sum(2).mean(1).view(-1)
    (loss_ref * w).mean().backward()
    zg = z_cur.to(DEV).requires_grad_(True)
    loss = ops.quantile_huber_loss(zg, tau.to(DEV), z_on.to(DEV), z_tg.to(DEV), act.to(DEV), ret.to(DEV), gdn.to(DEV),
                                   T, Tp, kappa=1.0)
    (loss * w.to(DEV)).mean().backward()
    assert rel_err(loss.detach().cpu().numpy(), loss_ref.detach().numpy()) < 1e-4
    assert rel_err(zg.grad.cpu().numpy(), zc.grad.numpy()) < 1e-4


@pytest.mark.parametrize("B,A,K", [(256, 4, 1), (64, 3, 10), (9, 18, 10)])
def test_ensemble_loss_kernel_vs_oracle_math(B, A, K):
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(B + K)
    qc, qo, qt = (torch.randn(K, B, A, generator=g) for _ in range(3))
    act = torch.randint(0, A, (B,), generator=g)
    ret, gdn, w = torch.randn(B, generator=g), torch.rand(B, generator=g), torch.rand(B, generator=g)
    q = qc.clone().requires_grad_(True)
    best = qo.argmax(-1)                                          # (K, B)
    y = ret.view(1, B) + torch.gather(qt, 2, best.unsqueeze(-1)).squeeze(-1) * gdn.view(1, B)
    loss_ref = (torch.gather(q, 2, act.view(1, B, 1).expand(K, B, 1)).squeeze(-1) - y).square().mean(0)
    (loss_ref * w).mean().backward()
    qg = qc.to(DEV).requires_grad_(True)
    loss = ops.ensemble_q_loss(qg, qo.to(DEV), qt.to(DEV), act.to(DEV), ret.to(DEV), gdn.to(DEV))
    (loss * w.to(DEV)).mean().backward()
    assert rel_err(loss.detach().cpu().numpy(), loss_ref.detach().numpy()) < 1e-5
    assert rel_err(qg.grad.cpu().numpy(), q.grad.numpy()) < 1e-5


def test_cos_basis_kernel():
    """cos(fl32(fl32(tau * i) * pi)) (iqn_model.py:89-92).  The argument is built exactly like torch builds it (checked
    bit for bit); the cosine is judged against float64 math on that fp32 argument, so the host's libm plays no role.
    Seeded: the draw used to come from the global generator, i.e. from whatever ran before."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(0)
    tau = torch.rand(4096, 1, generator=g)
    arg = torch.tile(tau, [1, 64]) * torch.arange(1, 65) * np.pi               # fp32, as the reference computes it
    arg_np = (tau.numpy() * np.arange(1, 65, dtype=np.float32)).astype(np.float32) * np.float32(np.pi)
    assert np.array_equal(arg.numpy(), arg_np)
    want = np.cos(arg_np.astype(np.float64))
    got = ops.cos_basis(tau.to(DEV), 64).cpu().numpy().astype(np.float64)
    assert float(np.abs(got - want).max()) < 2e-6
    assert float(np.abs(torch.cos(arg).numpy() - want).max()) < 2e-6             # and so does torch on this host


def test_flat_adam_matches_torch_adam_over_steps():
    """clip_grad_norm_ + torch.optim.Adam (agent.py:73-74) vs the fused flat kernels, 20 steps."""
    from prism_b200.agents.optim import FlatAdam
    torch.manual_seed(0)
    shapes = [(64, 33), (33,), (7, 5, 3), (1,), (130,)]
    ref_p = [torch.randn(s, dtype=torch.float32).requires_grad_(True) for s in shapes]
    dev_p = [p.detach().clone().to(DEV).requires_grad_(True) for p in ref_p]
    ref_opt = torch.optim.Adam(ref_p, lr=1e-3, betas=(0.9, 0.999), eps=1.5e-4)
    opt = FlatAdam(dev_p, lr=1e-3, betas=(0.9, 0.999), eps=1.5e-4, max_grad_norm=2.0)
    for step in range(20):
        grads = [torch.randn(s) * (3.0 if step % 3 == 0 else 0.05) for s in shapes]
        for p, g in zip(ref_p, grads):
            p.grad = g.clone()
        total = torch.nn.utils.clip_grad_norm_(ref_p, 2.0)
        ref_opt.step()
        for p, g in zip(dev_p, grads):
            p.grad = g.to(DEV)
        opt.step()
        assert abs(float(opt.norm_out[0]) - float(total)) / float(total) < 1e-5
    for a, b in zip(dev_p, ref_p):
        assert rel_err(a.detach().cpu().numpy(), b.detach().numpy()) < 1e-5


@pytest.mark.parametrize("name", ["agent_ids_iqn_ln_target", "agent_dqn_double"])
def test_cuda_graph_update_equals_eager(name):
    """The captured update (agent.py:81-147) must give the eager result and, unlike the reference,
    keep bootstrapping from the TARGET network (SURVEY appendix Q3)."""
    fx = load_golden(name)
    batch = fixture_batch(fx, DEV)
    w = torch.from_numpy(fx["per_weights"]).to(DEV)
    taus = fixture_taus(fx)
    results = []
    for graph in (False, True):
        cfg, agent = build_product_agent(fx, use_cuda_graph=graph)
        d = agent.model.distribution_model
        if d is not None:
            # pin the quantiles for every call so eager and replayed draws coincide
            fixed = [torch.as_tensor(t, dtype=torch.float32, device=DEV).view(-1, 1) for t in taus]
            calls = {"n": 0}
            models = [agent.model.distribution_model] + ([agent.target_model.distribution_model]
                                                         if agent.target_model is not None else [])
            for m in models:
                orig = m.forward

                def fwd(x, n_quantile_samples=None, for_action=False, static_quantiles=None, _o=orig, _m=m):
                    rows = (n_quantile_samples or 0) * x.shape[0]
                    sq = next((t for t in fixed if t.numel() == rows), None)
                    return _o(x, n_quantile_samples=n_quantile_samples, for_action=for_action, static_quantiles=sq)
                m.forward = fwd
        outs = []
        for _ in range(3):
            outs.append(agent.update(batch, w).clone())
        torch.cuda.synchronize()
        results.append((outs, {k: v.clone() for k, v in agent.model.state_dict().items()}))
    for a, b in zip(results[0][0], results[1][0]):
        assert rel_err(b.cpu().numpy(), a.cpu().numpy()) < 1e-5
    for k in results[0][1]:
        assert rel_err(results[1][1][k].cpu().numpy(), results[0][1][k].cpu().numpy()) < 1e-5, k


def test_target_sync_is_one_copy():
    fx = load_golden("agent_dqn_double")
    cfg, agent = build_product_agent(fx)
    agent.sync_target_model()
    for (k, a), (_, b) in zip(agent.model.state_dict().items(), agent.target_model.state_dict().items()):
        assert torch.equal(a, b), k


def test_learner_step_graph_after_eager_update():
    """An eager update on the default stream followed by a captured LearnerStep (what smoke() does):
    capture must not inherit autograd state from the default stream, and the graph must train."""
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    from oracle.gen_golden import make_script
    cap, B, obs_shape, A = 256, 16, (10, 10, 4), 3
    cfg = prism_b200.minatar_ids_iqn_config(device=DEV, experience_replay_capacity=cap, batch_size=B,
                                            iqn_n_current_state_quantile_samples=8,
                                            iqn_n_next_state_quantile_samples=8, iqn_quantile_samples_per_action=8,
                                            iqn_quantile_model_feature_dim=32, ids_q_head_feature_dim=16,
                                            ids_n_q_heads=3, use_cuda_graph=False, replay_max_streams=4,
                                            replay_staging_rows=32)
    torch.manual_seed(0)
    agent = prism_b200.build_agent(cfg, obs_shape, A)
    buf = prism_b200.build_exp_buffer(cfg)
    S = make_script(3, n_streams=4, n_steps=300, obs_shape=obs_shape, p_done=0.05, p_trunc=0.02, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])
    buf.extend_batch(S["stream"], S["obs"].reshape((-1,) + obs_shape), S["action"], S["reward"], S["done"],
                     S["trunc"], succ.reshape((-1,) + obs_shape))
    batch, info = buf.sample(return_info=True)
    td = agent.update(batch, info["_weight"])                       # eager, default stream
    buf.update_priority(info["index"], td.abs())
    before = agent.optimizer.arena.clone()
    step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=True)
    losses = [float(step.step()) for _ in range(5)]
    torch.cuda.synchronize()
    assert all(np.isfinite(losses))
    assert int(agent.optimizer.step_count) == 1 + 5                  # warm-up iterations did not train
    assert not torch.equal(before, agent.optimizer.arena)
    assert step.launches_per_step is not None and step.launches_per_step > 0
    st = buf.buffer._sampler.state_host()
    assert st["status"] == 0 and st["len"] == cap


FUSED_LINEAR_CASES = [
    (1, 256, 256, 1024, True, True, "linear:ffma"), (1, 256, 4, 256, False, False, "linear:narrow"),
    (10, 64, 256, 1024, True, True, "linear:ffma"), (10, 64, 3, 256, False, False, "linear:narrow"),
    (3, 37, 19, 50, False, True, "linear:ffma"), (1, 2048, 256, 1024, True, True, "linear:tc_gemm"),
    (4, 5, 7, 3, True, False, "linear:ffma"), (1, 512, 512, 3136, True, True, "linear:tc_gemm"),
    # 2 * 272 * 2 * 200 * 1000 = 2.2e8 FLOP reaches TC_MIN_FLOPS: tcgen05, not linear.cu
    (2, 272, 200, 1000, False, True, "linear:tc_gemm"),
    # 16-byte aligned operands with ragged tiles: the cp.async kernel's zero-filled row / column / k tails;
    # (3, 37, 19, 50) and (4, 5, 7, 3) above are unaligned: the register-staged kernel
    (1, 100, 36, 68, True, True, "linear:ffma"), (3, 64, 64, 36, False, False, "linear:ffma"),
    # the data-parallel layer (272 rows = the padded batch): 16 live rows in the last M tile, an empty split in dW
    (1, 272, 256, 1024, True, True, "linear:ffma")]


@pytest.mark.parametrize("K,M,N,J,shared,relu,route", FUSED_LINEAR_CASES,
                         ids=["-".join(map(str, c[:6])) for c in FUSED_LINEAR_CASES])     # the route is not part of the id
def test_fused_linear_matches_torch(K, M, N, J, shared, relu, route):
    """A dense layer through ops.linear_heads against torch fp64 math, on the route the test names: linear:ffma is
    pb_linear_{fwd,bwd_input,bwd_weight} (cluster split-K GEMM, 3xTF32 products, fused bias/ReLU/mask/bias-grad;
    cp.async operand tiles when aligned, register-staged otherwise; every path of it: tests/test_gpu_linear.py),
    linear:tc_gemm the tcgen05 GEMM, linear:narrow the narrow output-layer kernels.  Tolerance 2e-5 relative of the
    tensor's max (fp32 accumulation order)."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(K * 1000 + M + N + J)
    x = torch.randn((M, J) if shared else (K, M, J), generator=g)
    w = torch.randn(K, N, J, generator=g) / J ** 0.5
    b = torch.randn(K, N, generator=g)
    gy = torch.randn(K, M, N, generator=g)
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    xe = xr.unsqueeze(0).expand(K, M, J) if shared else xr
    yr = torch.baddbmm(br.unsqueeze(1), xe, wr.transpose(1, 2))
    if relu:
        # a ReLU mask is a step function: a pre-activation within rounding of 0 may legitimately come out on the other
        # side on the GPU (3xTF32 products, fp32 sums) and that unit's whole gradient row moves.  Gradients are judged
        # away from the kinks: units that close to 0 receive no upstream gradient.
        gy = gy * (yr.detach().abs() > 1e-4).float()
        yr = yr.relu()
    yr.backward(gy.double())
    xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
    ops.route_counts(reset=True)
    y = ops.linear_heads(xd, wd, bd, relu=relu)
    assert ops.route_counts() == {route: 1}, ops.route_counts()
    y.backward(gy.to(DEV))
    torch.cuda.synchronize()
    assert rel_err(y.detach().cpu().numpy(), yr.detach().numpy()) < 2e-5
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) < 2e-5
    assert rel_err(wd.grad.cpu().numpy(), wr.grad.numpy()) < 2e-5
    assert rel_err(bd.grad.cpu().numpy(), br.grad.numpy()) < 2e-5


@pytest.mark.parametrize("split_mode", [0, 1])
@pytest.mark.parametrize("batch,kbatches,M,N,K,a_major,b_major,act", [
    (1, 1, 128, 64, 32, 0, 0, 0),            # one tile, one K block
    (1, 1, 128, 64, 32, 1, 0, 0),            # MN-major A
    (1, 1, 128, 64, 32, 0, 1, 0),            # MN-major B
    (1, 1, 300, 72, 100, 0, 0, 1),           # ragged M / N / K (TMA zero fill), bias + ReLU
    (1, 1, 300, 72, 100, 1, 1, 0),           # weight-gradient form, ragged
    (3, 1, 260, 200, 96, 0, 1, 0),           # batched input-gradient form
    (1, 4, 256, 320, 64, 0, 1, 0),           # K loop over 4 operand batches (shared-input gradient)
    (1, 1, 512, 3136, 64, 0, 0, 1),          # cos-embedding layer shape (config 5 columns)
    (1, 1, 256, 512, 8192, 1, 1, 0),         # long K: split-K partials + reduction
    (2, 1, 1024, 256, 1024, 0, 0, 1),        # persistent loop: several tiles per CTA, both accumulators
])
def test_tc_gemm_matches_fp64(batch, kbatches, M, N, K, a_major, b_major, act, split_mode):
    """pb_tc_gemm (tcgen05 3xTF32, TMA-fed, TMEM accumulators) against fp64 math, every operand orientation:
    2e-5 of the output's max (single-pass TF32 sits at ~1e-3)."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(batch * 7 + M + N + K + a_major * 3 + b_major * 5)
    nb = kbatches if kbatches > 1 else batch
    a = torch.randn((nb, K, M) if a_major else (nb, M, K), generator=g)
    b = torch.randn((nb, K, N) if b_major else (nb, N, K), generator=g) / K ** 0.5
    bias = torch.randn(batch, N, generator=g) if act else None
    ad, bd = a.to(DEV), b.to(DEV)
    out = torch.full((batch, M, N), float("nan"), device=DEV)
    old = ops.TC_SPLIT_MODE
    ops.TC_SPLIT_MODE = split_mode
    try:
        ops.tc_gemm(out, ad, a_major, M if a_major else K, M * K, bd, b_major, N if b_major else K, N * K, batch, M, N, K,
                    bias=None if bias is None else bias.to(DEV), bias_bs=N, act=act, kbatches=kbatches)
        torch.cuda.synchronize()
    finally:
        ops.TC_SPLIT_MODE = old
    al = (a.transpose(1, 2) if a_major else a).double()
    bl = (b.transpose(1, 2) if b_major else b).double()
    ref = torch.bmm(al, bl.transpose(1, 2))
    if kbatches > 1:
        ref = ref.sum(dim=0, keepdim=True)
    if bias is not None:
        ref = ref + bias.double().unsqueeze(1)
    if act:
        ref = torch.relu(ref)
    got = out.cpu().double()
    assert torch.isfinite(got).all()
    assert rel_err(got.numpy(), ref.numpy()) < 2e-5


@pytest.mark.parametrize("M,N,K,a_major,b_major", [
    (512, 3136, 32768, 1, 1),                # configs[4] weight gradient: stream-K segments, each several chunks
    (256, 256, 16384, 1, 1),                 # 4 tiles on 148 SMs: stream-K ranges shorter than a chunk and longer
    (4736, 256, 8192, 0, 0),                 # 74 whole tiles per CTA-wave: whole tiles accumulated in chunks (slot 2)
])
def test_tc_gemm_long_k_chains_do_not_drift(M, N, K, a_major, b_major):
    """The tensor core accumulates with truncation: one chain of K / 8 * 3 MMAs over same-signed products drifts by
    ~7e-4 at K = 32768 (the configs[4] weight gradient: dW = dZ^T X over 32768 rows) -- measured -4.2e-5 per 2048 floats
    of K.  pb_tc_gemm caps a chain at 2048 floats of K (once K >= 4096) and adds the chunks in round-to-nearest fp32
    (csrc/tc_gemm.cu, SegIter): 6e-5 on operands whose products all have the same sign, the worst case for a truncating
    adder (mixed signs, as in the layers' real operands, sit below the 2e-5 of the short-K tests)."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn((1, K, M) if a_major else (1, M, K), generator=g).abs_()
    b = torch.randn((1, K, N) if b_major else (1, N, K), generator=g).abs_() / K
    out = torch.full((1, M, N), float("nan"), device=DEV)
    ops.tc_gemm(out, a.to(DEV), a_major, M if a_major else K, M * K, b.to(DEV), b_major, N if b_major else K, N * K, 1, M, N, K)
    torch.cuda.synchronize()
    al = (a.transpose(1, 2) if a_major else a).double()
    bl = (b.transpose(1, 2) if b_major else b).double()
    ref = torch.bmm(al, bl.transpose(1, 2))
    err = (out.cpu().double() - ref) / ref.abs().max()
    print("long-K chain: max |err| %.2e, mean signed err %.2e" % (float(err.abs().max()), float(err.mean())))
    assert float(err.abs().max()) < 6e-5


@pytest.mark.parametrize("M,N,K,rows", [(2048, 1024, 64, 64), (640, 328, 64, 10), (384, 18, 512, 384)])
def test_tc_gemm_fused_multiplier_and_unaligned_output(M, N, K, rows):
    """Epilogue fusion of iqn_model.py:70-71: out = relu(A B^T + bias) * x[row % rows] (x broadcast over the
    quantile-major rows).  N = 18 (row stride not 16-byte aligned) exercises the direct-store epilogue."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(M + N + K)
    a, b = torch.randn(1, M, K, generator=g), torch.randn(1, N, K, generator=g) / K ** 0.5
    bias, x = torch.randn(1, N, generator=g), torch.randn(rows, N, generator=g)
    out = torch.full((1, M, N), float("nan"), device=DEV)
    ops.tc_gemm(out, a.to(DEV), 0, K, M * K, b.to(DEV), 0, K, N * K, 1, M, N, K, bias=bias.to(DEV), bias_bs=N, act=1,
                mul=x.to(DEV))
    torch.cuda.synchronize()
    ref = torch.relu(torch.bmm(a.double(), b.double().transpose(1, 2)) + bias.double().unsqueeze(1))
    ref = ref * x.double().repeat(M // rows, 1).unsqueeze(0)
    assert rel_err(out.cpu().numpy(), ref.numpy()) < 2e-5


@pytest.mark.parametrize("K,M,N,J,shared,relu", [
    (1, 2048, 256, 1024, True, True), (1, 2048, 1024, 64, True, True), (1, 300, 64, 32, True, False),
    (10, 512, 512, 3136, False, True), (2, 1000, 128, 96, True, False)])
def test_tensor_core_linear_matches_fp64(K, M, N, J, shared, relu):
    """pb_linear_fwd_tc (tcgen05 3xTF32, TMEM accumulator) must hold fp32-level accuracy: 2e-5 of the
    tensor's max against fp64 math (single-pass TF32 would sit at ~1e-3)."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(K * 7 + M + N + J)
    x = torch.randn((M, J) if shared else (K, M, J), generator=g)
    w = torch.randn(K, N, J, generator=g) / J ** 0.5
    b = torch.randn(K, N, generator=g)
    gy = torch.randn(K, M, N, generator=g)
    xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
    y = ops._LinearTC.apply(xd, wd, bd, 1 if relu else 0)
    y.backward(gy.to(DEV))
    torch.cuda.synchronize()
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    xe = xr.unsqueeze(0).expand(K, M, J) if shared else xr
    yr = torch.baddbmm(br.unsqueeze(1), xe, wr.transpose(1, 2))
    if relu:
        # the ReLU gate is discontinuous: outputs within rounding of 0 may gate differently in fp32 and fp64.
        # Judge the gradients with the gate the kernel actually produced.
        yr = yr * (y.detach().cpu() > 0)
    yr.backward(gy.double())
    assert rel_err(y.detach().cpu().numpy(), yr.detach().numpy()) < 2e-5
    assert rel_err(wd.grad.cpu().numpy(), wr.grad.numpy()) < 1e-4
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) < 1e-4
    assert rel_err(bd.grad.cpu().numpy(), br.grad.numpy()) < 1e-4


@pytest.mark.parametrize("n,B,F_,J", [(8, 64, 1024, 64), (7, 48, 3136, 64)])
def test_phi_times_x_matches_fp64(n, B, F_, J):
    """relu(basis W^T + b) (.) x with x broadcast over quantile-major rows (iqn_model.py:70-71, 89-93): fused
    GEMM epilogue forward, fused element-wise backward + tensor-core weight gradient, against fp64 autograd."""
    import torch.nn as nn
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(n * 100 + B)
    basis = torch.randn(n * B, J, generator=g)
    w, b = torch.randn(F_, J, generator=g) / J ** 0.5, torch.randn(F_, generator=g) * 0.1
    x = torch.relu(torch.randn(B, F_, generator=g))               # conv embedding after ReLU: exact zeros
    gh = torch.randn(n * B, F_, generator=g)
    seq = nn.Sequential(nn.Linear(J, F_), nn.ReLU()).to(DEV)
    with torch.no_grad():
        seq[0].weight.copy_(w)
        seq[0].bias.copy_(b)
    xd = x.to(DEV).requires_grad_(True)
    old = ops.TC_MIN_FLOPS
    ops.TC_MIN_FLOPS = 0.0
    try:
        h = ops.phi_times_x(seq, basis.to(DEV), xd, n)
        assert h.grad_fn is not None and "PhiTimesX" in type(h.grad_fn).__name__
        h.backward(gh.to(DEV))
        with torch.no_grad():
            h_nograd = ops.phi_times_x(seq, basis.to(DEV), xd, n)
    finally:
        ops.TC_MIN_FLOPS = old
    torch.cuda.synchronize()
    wr, br, xr = w.double().requires_grad_(True), b.double().requires_grad_(True), x.double().requires_grad_(True)
    pre = basis.double() @ wr.t() + br
    # the ReLU gate is discontinuous: judge with the gate the kernel's fp32 pre-activation produced
    gate = (torch.relu(basis @ w.t() + b) > 0).double()
    href = (pre * gate).view(n, B, F_) * xr.unsqueeze(0)
    href.view(n * B, F_).backward(gh.double())
    assert rel_err(h.detach().cpu().numpy(), href.detach().view(n * B, F_).numpy()) < 2e-5
    assert torch.equal(h_nograd, h.detach())
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) < 1e-4
    assert rel_err(seq[0].weight.grad.cpu().numpy(), wr.grad.numpy()) < 1e-4
    assert rel_err(seq[0].bias.grad.cpu().numpy(), br.grad.numpy()) < 1e-4


@pytest.mark.parametrize("rows,F_", [(2048, 3136), (4100, 512), (1111, 1024), (513, 2052)])
def test_fused_layer_norm_matches_fp64(rows, F_):
    """csrc/ln.cu forward + single-pass backward against fp64 autograd of nn.LayerNorm (ffnn_model.py:17-18)."""
    import torch.nn as nn
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(rows + F_)
    x = torch.randn(rows, F_, generator=g) * 2.0 + 0.7
    gy = torch.randn(rows, F_, generator=g)
    ln = nn.LayerNorm(F_).to(DEV)
    with torch.no_grad():
        ln.weight.copy_(torch.randn(F_, generator=g))
        ln.bias.copy_(torch.randn(F_, generator=g))
    xd = x.to(DEV).requires_grad_(True)
    y = ops.layer_norm(xd, ln)
    assert "LayerNorm" in type(y.grad_fn).__name__ and "Native" not in type(y.grad_fn).__name__
    y.backward(gy.to(DEV))
    ref = nn.LayerNorm(F_).double()
    with torch.no_grad():
        ref.weight.copy_(ln.weight.cpu().double())
        ref.bias.copy_(ln.bias.cpu().double())
    xr = x.double().requires_grad_(True)
    yr = ref(xr)
    yr.backward(gy.double())
    assert rel_err(y.detach().cpu().numpy(), yr.detach().numpy()) < 1e-5
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) < 1e-5
    assert rel_err(ln.weight.grad.cpu().numpy(), ref.weight.grad.numpy()) < 1e-5
    assert rel_err(ln.bias.grad.cpu().numpy(), ref.bias.grad.numpy()) < 1e-5


@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("host_u", [False, True])
@pytest.mark.parametrize("use_graph", [True, False])
def test_fused_ingest_step_equals_separate_push_then_step(use_graph, host_u, native, monkeypatch):
    """LearnerStep.step(ingest=...) scatters the new steps inside the step graph (after the priority write-back,
    concurrently with backward) from double-buffered staging blocks.  Same uniforms, same data: it must produce the
    same losses, parameters, ring and trees as `step(); push(new steps)` run one after the other.  Both host stagings:
    one C call (pb_store_stage_block, the default) and the numpy assignments."""
    import prism_b200
    from prism_b200.experience import ring as ring_mod
    from prism_b200.learner_step import LearnerStep
    from oracle.gen_golden import make_script
    monkeypatch.setattr(ring_mod, "NATIVE_STAGE", native)
    taken = []
    orig = ring_mod.IngestSlot._fill_native
    monkeypatch.setattr(ring_mod.IngestSlot, "_fill_native",
                        lambda self, *a: taken.append(orig(self, *a)) or taken[-1])
    cap, B, obs_shape, A, n_new, iters = 256, 16, (10, 10, 6), 4, 4, 9
    S = make_script(5, n_streams=4, n_steps=200 + n_new * iters, obs_shape=obs_shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])
    rng = np.random.default_rng(11)
    us = rng.random((iters, B))

    def run(fused):
        cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=cap, batch_size=B,
                                                per_sampling="stratified", replay_max_streams=4, replay_staging_rows=64,
                                                use_cuda_graph=False)
        torch.manual_seed(0)
        agent = prism_b200.build_agent(cfg, obs_shape, A)
        buf = prism_b200.build_exp_buffer(cfg)
        buf.extend_batch(S["stream"][:200], S["obs"][:200].reshape((-1,) + obs_shape), S["action"][:200], S["reward"][:200],
                         S["done"][:200], S["trunc"][:200], succ[:200].reshape((-1,) + obs_shape))
        step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=use_graph)
        push = None if fused else buf.ingest_graph(n_new)
        losses = []
        for i in range(iters):
            sl = slice(200 + i * n_new, 200 + (i + 1) * n_new)
            new = (S["stream"][sl], S["obs"][sl], S["action"][sl], S["reward"][sl], S["done"][sl], S["trunc"][sl], succ[sl])
            u = torch.from_numpy(us[i]).to(DEV)
            if fused:
                if host_u:                       # host uniforms ride in the ingest's staging block
                    u = torch.from_numpy(us[i].copy())
                losses.append(float(step.step(u=u, ingest=new)))
            else:
                losses.append(float(step.step(u=u)))
                push(*new)
        torch.cuda.synchronize()
        tree, ring = buf.buffer._sampler, buf.buffer._storage
        return (losses, agent.optimizer.arena.clone(), tree.sum.clone(), tree.min.clone(), tree.state_host(),
                ring.obs.clone(), ring.next_link.clone())

    a, b = run(True), run(False)
    assert (len(taken) > 0 and all(taken)) if native else not taken     # the staging path under test really ran
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1])
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert a[4] == b[4]
    assert torch.equal(a[5], b[5]) and torch.equal(a[6], b[6])


@pytest.mark.parametrize("use_graph", [True, False])
def test_prefetched_batches_equal_in_order_sampling(use_graph):
    """LearnerStep(prefetch=True) samples + gathers the next batch on the tail branch of the current iteration (after
    the priority write-back, concurrently with backward / Adam).  The tree it sees and the order of the generator's
    draws are the same as when the batch is sampled at the head of the next iteration: identical training."""
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    from oracle.gen_golden import make_script
    cap, B, obs_shape, A, iters = 256, 16, (10, 10, 6), 4, 8
    S = make_script(9, n_streams=4, n_steps=240, obs_shape=obs_shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])

    def run(prefetch):
        cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=cap, batch_size=B,
                                                per_sampling="stratified", replay_max_streams=4, replay_staging_rows=64,
                                                use_cuda_graph=False)
        torch.manual_seed(0)
        agent = prism_b200.build_agent(cfg, obs_shape, A)
        buf = prism_b200.build_exp_buffer(cfg)
        buf.extend_batch(S["stream"], S["obs"].reshape((-1,) + obs_shape), S["action"], S["reward"], S["done"], S["trunc"],
                         succ.reshape((-1,) + obs_shape))
        buf._flush()
        buf.buffer._sampler.seed(1234)
        step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=use_graph, prefetch=prefetch)
        losses = [float(step.step()) for _ in range(iters)]
        torch.cuda.synchronize()
        tree = buf.buffer._sampler
        return losses, agent.optimizer.arena.clone(), tree.sum.clone(), tree.min.clone()

    a, b = run(True), run(False)
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1])
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])


@pytest.mark.parametrize("kind", ["ids_iqn", "dqn_greedy"])
def test_acting_graph_equals_eager_acting(kind, monkeypatch):
    """Agent.forward as one CUDA graph (embedding -> IQN(Nq) -> K heads -> IDS / greedy kernel) picks the same actions
    as the eager path (prism/agents/agent.py:31-41).  The quantile draw is pinned on both sides."""
    import prism_b200
    obs_shape, A, N = ((10, 10, 4), 3, 14) if kind == "ids_iqn" else ((10, 10, 6), 4, 9)
    if kind == "ids_iqn":
        cfg = prism_b200.minatar_ids_iqn_config(device=DEV, experience_replay_capacity=64, batch_size=8,
                                                iqn_quantile_samples_per_action=16, iqn_quantile_model_feature_dim=32,
                                                ids_q_head_feature_dim=16, ids_n_q_heads=3, use_cuda_graph=True,
                                                replay_max_streams=2, replay_staging_rows=8)
    else:
        cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=64, batch_size=8,
                                                use_cuda_graph=True, replay_max_streams=2, replay_staging_rows=8)
    torch.manual_seed(0)
    agent = prism_b200.build_agent(cfg, obs_shape, A)
    agent.eval() if kind == "dqn_greedy" else agent.train()
    real_rand = torch.rand
    iqn = agent.model.distribution_model

    def pin_draw(call):
        # the quantiles come from the library's own Philox generator (counter = call number): the same call number on
        # both sides gives the same draws, under graph replay as well as eagerly
        if iqn is not None:
            iqn._rng_state()[1:3] = torch.tensor([call, 0], device=DEV)
    g = torch.Generator().manual_seed(3)
    for trial in range(3):
        obs = (real_rand((N,) + obs_shape, generator=g) < 0.15).float()
        pin_draw(100 + trial)
        got = agent.forward(obs)                                   # graph (captured on the first trial)
        agent.use_cuda_graph, saved = False, agent.use_cuda_graph
        agent.model.use_cuda_graph, saved_m = False, getattr(agent.model, "use_cuda_graph", False)
        pin_draw(100 + trial)
        want = agent.forward(obs)                                  # eager
        agent.use_cuda_graph, agent.model.use_cuda_graph = saved, saved_m
        assert got.dtype == torch.int64 and got.shape == (N,)
        assert torch.equal(got.cpu(), want.cpu())
    assert len(agent._acting_graphs) == 1


def test_fused_theil_index_matches_autograd():
    """csrc/theil.cu against the ATen formulation of q_ensemble.py:86-92 (value and gradient w.r.t. every stacked
    parameter), K = 10 heads."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(4)
    shapes = [(10, 256, 64), (10, 256), (10, 64), (10, 3, 256), (10, 3)]
    base = [torch.randn(s, generator=g) * (0.5 + 0.1 * torch.arange(10.0).view(10, *([1] * (len(s) - 1)))) for s in shapes]
    dev_p = [b.to(DEV).requires_grad_(True) for b in base]
    T = ops.theil_index(dev_p, {})
    (T * 3.0).backward()
    ref_p = [b.double().requires_grad_(True) for b in base]
    sq = sum(p.square().flatten(1).sum(dim=1) for p in ref_p)
    l2 = sq.sqrt()
    ratio = l2 / l2.mean()
    Tr = (ratio * torch.log(ratio)).mean()
    (Tr * 3.0).backward()
    assert abs(float(T) - float(Tr)) < 1e-6 * max(1.0, abs(float(Tr)))
    for d, r in zip(dev_p, ref_p):
        assert rel_err(d.grad.cpu().numpy(), r.grad.numpy()) < 1e-4


def test_prefetch_toggle_and_loss_readback_keep_training_identical():
    """set_prefetch(True) in the middle of a run and the in-graph loss read-back change scheduling only: losses,
    parameters and trees stay bit-identical to the plain in-order loop, and loss_host mirrors the returned loss."""
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    from oracle.gen_golden import make_script
    cap, B, obs_shape, A = 256, 16, (10, 10, 6), 4
    S = make_script(13, n_streams=4, n_steps=240, obs_shape=obs_shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])

    def run(toggle):
        cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=cap, batch_size=B,
                                                per_sampling="stratified", replay_max_streams=4, replay_staging_rows=64,
                                                use_cuda_graph=False)
        torch.manual_seed(0)
        agent = prism_b200.build_agent(cfg, obs_shape, A)
        buf = prism_b200.build_exp_buffer(cfg)
        buf.extend_batch(S["stream"], S["obs"].reshape((-1,) + obs_shape), S["action"], S["reward"], S["done"], S["trunc"],
                         succ.reshape((-1,) + obs_shape))
        buf._flush()
        buf.buffer._sampler.seed(77)
        step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=True)
        losses, mirrored = [], []
        for i in range(7):
            if toggle and i == 3:
                step.set_prefetch(True)
                host = step.enable_loss_readback()
            total = step.step()
            losses.append(float(total))
            if toggle and i >= 3:
                torch.cuda.synchronize()
                mirrored.append(float(host))
        torch.cuda.synchronize()
        tree = buf.buffer._sampler
        return losses, mirrored, agent.optimizer.arena.clone(), tree.sum.clone()

    a, b = run(True), run(False)
    assert a[0] == b[0]
    assert a[1] == a[0][3:]
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])


def test_step_trace_marks_are_ordered_and_do_not_change_training():
    """LearnerStep.enable_trace(): the in-graph %globaltimer marks come out in phase order on the main branch, the tail
    branches start after the loss exists, and a traced run trains bit-identically to an untraced one."""
    import prism_b200
    from prism_b200.learner_step import LearnerStep
    from oracle.gen_golden import make_script
    cap, B, obs_shape, A = 256, 16, (10, 10, 6), 4
    S = make_script(13, n_streams=4, n_steps=240, obs_shape=obs_shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])

    def run(traced):
        cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=cap, batch_size=B,
                                                per_sampling="stratified", replay_max_streams=4, replay_staging_rows=64,
                                                use_cuda_graph=False)
        torch.manual_seed(0)
        agent = prism_b200.build_agent(cfg, obs_shape, A)
        buf = prism_b200.build_exp_buffer(cfg)
        buf.extend_batch(S["stream"], S["obs"].reshape((-1,) + obs_shape), S["action"], S["reward"], S["done"], S["trunc"],
                         succ.reshape((-1,) + obs_shape))
        buf._flush()
        buf.buffer._sampler.seed(77)
        step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=True, prefetch=True)
        report = None
        if traced:
            step.enable_trace()
        losses = [float(step.step()) for _ in range(5)]
        if traced:
            report = step.trace_report()
        # disable_trace() re-captures the step, and a re-capture re-primes the prefetched batch: the untraced run goes
        # through the same re-capture so that both runs train on the same batches
        step.disable_trace()
        losses += [float(step.step()) for _ in range(2)]
        torch.cuda.synchronize()
        return losses, agent.optimizer.arena.clone(), report

    (la, pa, rep), (lb, pb, _) = run(True), run(False)
    assert la == lb and torch.equal(pa, pb)
    main = ["start", "batch_ready", "fwd:embedded", "fwd:heads_done", "loss_ready", "backward_done", "opt:packed",
            "optimizer_done", "end"]
    assert all(m in rep for m in main), sorted(rep)
    times = [rep[m] for m in main]
    assert times[0] == 0 and times == sorted(times) and times[-1] < 5_000_000        # one small step: well under 5 ms
    for tail in ("tail:priorities_written", "tail:sampled", "tail:next_batch_ready"):
        assert rep["loss_ready"] <= rep[tail] <= rep["end"]


def test_optimizer_checkpoint_is_a_torch_adam_state_dict():
    """Agent.save writes ``optimizer.state_dict()`` (prism/agents/agent.py:231-236) and the reference reads it back into
    torch.optim.Adam (:244-252).  After the same two updates, the product's checkpoint must load (strict) into a
    torch.optim.Adam over the oracle model (reference parameter names / order) and equal the oracle's own Adam state;
    and the oracle's checkpoint must load into the product."""
    from oracle.agent_oracle import OracleAgent
    fx = load_golden("agent_ids_iqn_ln_target")
    cfg, agent = build_product_agent(fx)
    import dataclasses
    oracle = OracleAgent(dataclasses.replace(cfg, device="cpu"), tuple(fx["obs_shape"].tolist()), int(fx["n_actions"]))
    sd = fixture_state_dict(fx)
    oracle.model.load_state_dict(sd, strict=True)
    oracle.target.load_state_dict({k: target_transform(v) for k, v in sd.items()})
    w = torch.from_numpy(fx["per_weights"])
    for _ in range(2):
        taus = fixture_taus(fx)
        oracle.inject_taus(taus)
        oracle.update(fixture_batch(fx), w)
        inject_taus(cfg, agent, taus)
        agent.update(fixture_batch(fx, DEV), w.to(DEV))
    torch.cuda.synchronize()
    mine, ref = agent.optimizer.state_dict(), oracle.opt.state_dict()
    assert set(mine["param_groups"][0].keys()) == set(ref["param_groups"][0].keys())
    assert mine["param_groups"][0]["params"] == ref["param_groups"][0]["params"]
    assert len(mine["state"]) == len(ref["state"])
    for i, st in ref["state"].items():
        assert float(mine["state"][i]["step"]) == float(st["step"]) == 2.0
        assert mine["state"][i]["exp_avg"].shape == st["exp_avg"].shape
        assert rel_err(mine["state"][i]["exp_avg"].numpy(), st["exp_avg"].numpy()) < 1e-4, i
        assert rel_err(mine["state"][i]["exp_avg_sq"].numpy(), st["exp_avg_sq"].numpy()) < 2e-4, i
    fresh = torch.optim.Adam(oracle.model.parameters(), lr=cfg.learning_rate)
    fresh.load_state_dict(mine)                               # what the reference's Agent.load does
    # and the other direction: a reference checkpoint into the product's arena
    m_before = agent.optimizer.exp_avg.clone()
    agent.optimizer.exp_avg.zero_(); agent.optimizer.step_count.zero_()
    agent.optimizer.load_state_dict(ref)
    assert int(agent.optimizer.step_count.item()) == 2
    live = m_before != 0
    assert rel_err(agent.optimizer.exp_avg[live].cpu().numpy(), m_before[live].cpu().numpy()) < 1e-4


def test_static_batch_overflow_is_refused_and_ring_growth_recaptures():
    """ADVICE r1: sample(batch_size > static batch rows) must not write out of bounds; a grown aux pool must not leave a
    captured graph holding the freed descriptor."""
    import prism_b200
    cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=4096, batch_size=16,
                                            replay_max_streams=4, replay_staging_rows=64, use_cuda_graph=False)
    buf = prism_b200.build_exp_buffer(cfg)
    rng = np.random.default_rng(0)
    n = 512
    obs = (rng.random((n + 4, 10, 10, 6)) < 0.1).astype(np.float32)
    sid = (np.arange(n) % 4).astype(np.int32)
    buf.extend_batch(sid, obs[:n], rng.integers(0, 4, n).astype(np.int32), np.zeros(n, np.float32), np.zeros(n, bool),
                     np.zeros(n, bool), obs[4:n + 4])
    buf.sample(batch_size=16)
    buf.sample(batch_size=32)                                  # own static batch: grows
    assert buf._obs.shape[0] == 32
    buf.set_static_batch(buf.get_static_batch())               # now "owned by the agent" (learner.py:96-97)
    with pytest.raises(ValueError):
        buf.sample(batch_size=64)
    ring = buf.buffer._storage
    gen = ring.generation
    ring._grow_trunc_pool()
    assert ring.generation == gen + 1
    with pytest.raises(ValueError):
        ring.gather(torch.zeros(64, dtype=torch.int64, device=DEV), buf._obs, buf._next_obs, buf._reward, buf._gamma,
                    buf._nonterminal, buf._action)


@pytest.mark.parametrize("M,N,J", [(32768, 18, 512), (2048, 3, 256), (1000, 6, 64), (777, 32, 1024), (4100, 4, 320),
                                   (2048, 9, 512), (600, 16, 128)])     # N 9..16: narrow_*_kernel<16>
def test_narrow_linear_matches_fp64(M, N, J):
    """pb_narrow_linear_fwd / _bwd (the n_actions-wide output layer of the IQN head) against fp64 math + autograd."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(M + N)
    x = torch.randn(M, J, generator=g)
    w = torch.randn(N, J, generator=g) / J ** 0.5
    b = torch.randn(N, generator=g)
    dy = torch.randn(M, N, generator=g)
    xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
    ops.route_counts(reset=True)
    y = ops.linear(xd, wd, bd)
    assert ops.route_counts().get("linear:narrow", 0) == 1, ops.route_counts()
    y.backward(dy.to(DEV))
    torch.cuda.synchronize()
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
    y64 = x64 @ w64.t() + b64
    y64.backward(dy.double())
    assert rel_err(y.detach().cpu().numpy(), y64.detach().numpy()) < 2e-6
    assert rel_err(xd.grad.cpu().numpy(), x64.grad.numpy()) < 2e-6
    assert rel_err(wd.grad.cpu().numpy(), w64.grad.numpy()) < 2e-5
    assert rel_err(bd.grad.cpu().numpy(), b64.grad.numpy()) < 2e-5


@pytest.mark.parametrize("K,B,F_,shared", [(10, 512, 3136, True), (10, 64, 1024, True), (10, 64, 256, False),
                                           (4, 33, 512, False), (3, 7, 64, True), (1, 256, 256, True)])
def test_grouped_layer_norm_matches_fp64(K, B, F_, shared):
    """LayerNorm with per-head affine parameters (K ensemble heads; shared or per-head input) against fp64 autograd."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(K * 100 + B)
    x = torch.randn((B, F_) if shared else (K, B, F_), generator=g) * 2 + 0.5
    w = torch.rand(K, F_, generator=g) + 0.5
    b = torch.randn(K, F_, generator=g)
    dy = torch.randn(K, B, F_, generator=g)
    xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
    ops.route_counts(reset=True)
    y = ops.layer_norm_heads(xd, wd, bd)
    assert ops.route_counts().get("ln:fused_heads", 0) == 1
    y.backward(dy.to(DEV))
    torch.cuda.synchronize()
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
    n64 = torch.nn.functional.layer_norm(x64, (F_,))
    y64 = (n64 if not shared else n64.unsqueeze(0)) * w64.unsqueeze(1) + b64.unsqueeze(1)
    y64.backward(dy.double())
    assert rel_err(y.detach().cpu().numpy(), y64.detach().numpy()) < 1e-5
    assert rel_err(xd.grad.cpu().numpy(), x64.grad.numpy()) < 2e-5
    assert rel_err(wd.grad.cpu().numpy(), w64.grad.numpy()) < 2e-5
    assert rel_err(bd.grad.cpu().numpy(), b64.grad.numpy()) < 2e-5


def test_small_layer_norm_goes_through_the_fused_kernel():
    from prism_b200.agents import ops
    ln = torch.nn.LayerNorm(256).to(DEV)
    with torch.no_grad():
        ln.weight.uniform_(0.5, 1.5)
        ln.bias.uniform_(-0.5, 0.5)
    x = torch.randn(64, 256, device=DEV, requires_grad=True)
    # a generic upstream gradient: sum(y^2) would make dx the O(eps) residual of an exact cancellation (dy = 2 y is
    # collinear with xhat), which no two fp32 implementations agree on
    gy = torch.randn(64, 256, device=DEV)
    ops.route_counts(reset=True)
    y = ops.layer_norm(x, ln)
    assert ops.route_counts() == {"ln:fused": 1}
    y.backward(gy)
    got_w, got_b = ln.weight.grad.clone(), ln.bias.grad.clone()
    ln.weight.grad = ln.bias.grad = None
    xr = x.detach().clone().requires_grad_(True)
    yr = ln(xr)
    yr.backward(gy)
    assert rel_err(y.detach().cpu().numpy(), yr.detach().cpu().numpy()) < 1e-5
    assert rel_err(x.grad.cpu().numpy(), xr.grad.cpu().numpy()) < 1e-4
    assert rel_err(got_w.cpu().numpy(), ln.weight.grad.cpu().numpy()) < 1e-4
    assert rel_err(got_b.cpu().numpy(), ln.bias.grad.cpu().numpy()) < 1e-4


def test_device_quantile_draws():
    """pb_iqn_draw_cos_basis: uniforms in [0, 1) from the library's Philox generator, fresh per launch (also under graph
    replay), equal for equal seeds, and the basis is cos(pi i tau) of exactly those draws."""
    from prism_b200.agents import ops
    rng_a = torch.tensor([1234, 0, 0, 0], dtype=torch.int64, device=DEV)
    rng_b = rng_a.clone()
    t1, b1 = ops.draw_cos_basis(4096, 64, rng_a)
    t2, _ = ops.draw_cos_basis(4096, 64, rng_a)
    t3, _ = ops.draw_cos_basis(4096, 64, rng_b)
    torch.cuda.synchronize()
    assert torch.equal(t1, t3) and not torch.equal(t1, t2)
    assert float(t1.min()) >= 0.0 and float(t1.max()) < 1.0
    assert 0.47 < float(t1.mean()) < 0.53 and 0.27 < float(t1.std()) < 0.31
    assert rng_a.cpu().tolist()[:3] == [1234, 2, 0]
    assert torch.equal(b1, ops.cos_basis(t1, 64))
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        ops.draw_cos_basis(512, 64, rng_a)
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(graph):
        tg, _ = ops.draw_cos_basis(512, 64, rng_a)
    graph.replay()
    first = tg.clone()
    graph.replay()
    torch.cuda.synchronize()
    assert not torch.equal(first, tg)


def test_sum_leading_matches_torch():
    from prism_b200.agents import ops
    x = torch.randn(10, 512, 3136, device=DEV)
    assert rel_err(ops.sum_leading(x).cpu().numpy(), x.double().sum(0).cpu().numpy()) < 1e-6


@pytest.mark.parametrize("K,M,N,J,shared", [(10, 64, 3, 256, False), (10, 512, 18, 512, False), (1, 256, 4, 256, False),
                                            (4, 100, 6, 128, True), (10, 64, 9, 256, False), (4, 300, 16, 512, True)])
def test_narrow_linear_heads_matches_fp64(K, M, N, J, shared):
    """The n_actions-wide last layer of the K ensemble heads through the narrow kernels (batched over heads)."""
    from prism_b200.agents import ops
    g = torch.Generator().manual_seed(K * 7 + M)
    x = torch.randn((M, J) if shared else (K, M, J), generator=g)
    w = torch.randn(K, N, J, generator=g) / J ** 0.5
    b = torch.randn(K, N, generator=g)
    dy = torch.randn(K, M, N, generator=g)
    xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
    ops.route_counts(reset=True)
    y = ops.linear_heads(xd, wd, bd)
    assert ops.route_counts().get("linear:narrow", 0) == 1, ops.route_counts()
    y.backward(dy.to(DEV))
    torch.cuda.synchronize()
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
    xe = x64.unsqueeze(0).expand(K, -1, -1) if shared else x64
    y64 = torch.baddbmm(b64.unsqueeze(1), xe, w64.transpose(1, 2))
    y64.backward(dy.double())
    assert rel_err(y.detach().cpu().numpy(), y64.detach().numpy()) < 2e-6
    assert rel_err(xd.grad.cpu().numpy(), x64.grad.numpy()) < 2e-6
    assert rel_err(wd.grad.cpu().numpy(), w64.grad.numpy()) < 2e-5
    assert rel_err(bd.grad.cpu().numpy(), b64.grad.numpy()) < 2e-5


@pytest.mark.parametrize("K,M,N,J,shared", [(10, 256, 9, 256, False), (4, 4100, 16, 320, True)])
def test_narrow_linear_split_reduce_equals_one_call(K, M, N, J, shared):
    """pb_narrow_linear_bwd with dW = db = NULL, then pb_narrow_linear_bwd_reduce on a second stream ordered after it
    (as the learner step's graph runs it) gives the same bits as the one-call form."""
    from prism_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(K * 13 + M + N)
    x = torch.randn((M, J) if shared else (K, M, J), generator=g).to(DEV)
    w = (torch.randn(K, N, J, generator=g) / J ** 0.5).to(DEV)
    dy = torch.randn(K, M, N, generator=g).to(DEV)
    xhs = 0 if shared else M * J
    nb = lib.pb_narrow_linear_bwd_blocks(M)
    nan = lambda *shape: torch.full(shape, float("nan"), device=DEV)
    cur = torch.cuda.current_stream()
    dx1, dw1, db1, part1 = nan(K, M, J), nan(K, N, J), nan(K, N), nan(K * nb * (N * J + N))
    _lib.check(lib.pb_narrow_linear_bwd(K, M, N, J, x.data_ptr(), xhs, w.data_ptr(), dy.data_ptr(), dx1.data_ptr(),
                                        dw1.data_ptr(), db1.data_ptr(), part1.data_ptr(), cur.cuda_stream))
    dx2, dw2, db2, part2 = nan(K, M, J), nan(K, N, J), nan(K, N), nan(K * nb * (N * J + N))
    _lib.check(lib.pb_narrow_linear_bwd(K, M, N, J, x.data_ptr(), xhs, w.data_ptr(), dy.data_ptr(), dx2.data_ptr(),
                                        None, None, part2.data_ptr(), cur.cuda_stream))
    side = torch.cuda.Stream()
    side.wait_stream(cur)
    _lib.check(lib.pb_narrow_linear_bwd_reduce(K, M, N, J, part2.data_ptr(), dw2.data_ptr(), db2.data_ptr(),
                                               side.cuda_stream))
    cur.wait_stream(side)
    torch.cuda.synchronize()
    for a, b in ((dx1, dx2), (dw1, dw2), (db1, db2)):
        assert not torch.isnan(a).any() and torch.equal(a, b)
    xe = x.double().cpu().expand(K, M, J) if shared else x.double().cpu()
    assert rel_err(dw2.cpu().numpy(), (dy.double().cpu().transpose(1, 2) @ xe).numpy()) < 2e-5
    assert rel_err(db2.cpu().numpy(), dy.double().cpu().sum(1).numpy()) < 2e-5
