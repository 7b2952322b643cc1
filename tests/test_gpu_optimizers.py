"""clip_grad_norm_ + RMSprop / SGD over the flat parameter arena (FlatRMSprop, FlatSGD; the PB_OPT_* instantiations of
the optimizer kernels in csrc/agent_kernels.cu and csrc/peer.cu): the kernels against a float64 oracle on every path
they dispatch to, against torch.optim itself, at agent level, through LearnerStep, under loopback and two-process data
parallelism, and their checkpoints in torch's formats."""
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
gpu = pytest.mark.gpu
RULES = ("rmsprop_centered", "rmsprop", "sgd")


def _rule(name):
    from prism_b200 import _lib
    return {"adam": _lib.PB_OPT_ADAM, "rmsprop": _lib.PB_OPT_RMSPROP, "rmsprop_centered": _lib.PB_OPT_RMSPROP_CENTERED,
            "sgd": _lib.PB_OPT_SGD}[name]


def _make_opt(name, params, lr=1e-3, alpha=0.95, eps=0.01, max_grad_norm=10.0, arena=None):
    from prism_b200 import FlatRMSprop, FlatSGD
    if name == "sgd":
        return FlatSGD(params, lr=lr, max_grad_norm=max_grad_norm, arena=arena)
    return FlatRMSprop(params, lr=lr, alpha=alpha, eps=eps, centered=name == "rmsprop_centered",
                       max_grad_norm=max_grad_norm, arena=arena)


# ---- float64 oracle of clip + rule, written from torch's op order -----------------------------------------------------
def oracle_step(name, p, m, v, g, lr, alpha, eps, max_norm):
    """One step in float64 on float64 copies; hyper-parameters as the kernel sees them (fp32-rounded)."""
    f = lambda x: float(np.float32(x))
    lr, alpha, eps = f(lr), f(alpha), f(eps)
    norm = float(np.sqrt(np.sum(g * g)))
    coef = min(1.0, f(max_norm) / (norm + 1e-6)) if max_norm > 0 else 1.0
    g = g * coef
    if name == "sgd":
        return p - lr * g, m, v, (norm, coef)
    v = v * alpha + (1.0 - alpha) * g * g
    if name == "rmsprop_centered":
        m = m + (1.0 - alpha) * (g - m)
        avg = np.sqrt(v - m * m) + eps
    else:
        avg = np.sqrt(v) + eps
    return p - lr * g / avg, m, v, (norm, coef)


# ---- CPU: argument checks before any launch ---------------------------------------------------------------------------
def test_new_entries_reject_bad_arguments_without_a_launch():
    from prism_b200 import _lib
    lib = _lib.load()
    before = lib.pb_launch_count()
    P = 16                                           # any 16-byte aligned non-null "pointer": nothing may be launched
    A, R, RC, S = _lib.PB_OPT_ADAM, _lib.PB_OPT_RMSPROP, _lib.PB_OPT_RMSPROP_CENTERED, _lib.PB_OPT_SGD
    g = _lib.pb_peer_group(world=2, rank=0)          # no pads mapped
    for bad in (-1, 4, 99):                          # unknown rule
        assert lib.pb_opt_fused_max_n(bad) == 0 and lib.pb_peer_allreduce_opt_max_n(bad) == 0
        assert lib.pb_opt_fused_step(bad, 1, P, 1.0, 64, P, P, P, P, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_opt_clip_apply(bad, 64, P, P, P, P, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 4, None, None) == -1
        assert lib.pb_peer_allreduce_opt(bad, C.byref(g), 64, P, P, P, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_peer_opt(bad, C.byref(g), 64, P, P, P, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, None, None, None) == -1
    # a null state array the rule reads
    for rule, m, v in ((A, None, P), (A, P, None), (RC, None, P), (RC, P, None), (R, P, None)):
        assert lib.pb_opt_fused_step(rule, 1, P, 1.0, 64, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_opt_clip_apply(rule, 64, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 4, None, None) == -1
        assert lib.pb_peer_allreduce_opt(rule, C.byref(g), 64, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_peer_opt(rule, C.byref(g), 64, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, None, None, None) == -1
    # what the Adam entries refuse, every rule refuses (SGD with its null state arrays)
    for rule in (A, R, RC, S):
        m = None if rule in (R, S) else P
        v = None if rule == S else P
        assert lib.pb_opt_fused_step(rule, 1, P, 1.0, 66, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_opt_fused_step(rule, 1, None, 1.0, 64, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_opt_fused_step(rule, 65, P, 1.0, 64, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -3
        assert lib.pb_opt_fused_step(rule, 1, P, 1.0, 64, P, P, m, v, None, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_opt_clip_apply(rule, 0, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 4, None, None) == -1
        assert lib.pb_opt_clip_apply(rule, 64, None, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 4, None, None) == -1
        assert lib.pb_opt_clip_apply(rule, 64, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 0, None, None) == -1
        assert lib.pb_opt_clip_apply(rule, 64, P, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 4097, None, None) == -1
        assert lib.pb_opt_clip_apply(rule, 64, 18, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, 4, None, None) == -1
        assert lib.pb_peer_allreduce_opt(rule, C.byref(g), 64, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_peer_allreduce_opt(rule, None, 64, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, P, None, None) == -1
        assert lib.pb_peer_opt(rule, C.byref(g), 64, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, None, None, None) == -1
        assert lib.pb_peer_opt(rule, None, 64, P, m, v, P, 1e-3, 0.9, 0.9, 1e-8, 1.0, None, None, None) == -1
    assert lib.pb_launch_count() == before


def test_new_entries_are_in_the_header_and_the_ctypes_mirror():
    from prism_b200 import _lib
    from test_boundary import header_functions
    fns = header_functions()
    for name in ("pb_opt_fused_max_n", "pb_opt_fused_step", "pb_opt_clip_apply", "pb_peer_allreduce_opt_max_n",
                 "pb_peer_allreduce_opt", "pb_peer_opt"):
        assert name in fns and len(fns[name]) == len(_lib.SIGNATURES[name]), name
    src = open(os.path.join(os.path.dirname(HERE), "include", "prism_b200.h")).read()
    for k in ("PB_OPT_ADAM", "PB_OPT_RMSPROP", "PB_OPT_RMSPROP_CENTERED", "PB_OPT_SGD"):
        assert "#define %s %d" % (k, getattr(_lib, k)) in src


def test_flat_rmsprop_and_sgd_reject_what_the_reference_never_sets():
    from prism_b200 import FlatRMSprop, FlatSGD
    p = [torch.zeros(4, requires_grad=True)]
    with pytest.raises(ValueError):
        FlatRMSprop(p, lr=1e-3, momentum=0.9)
    with pytest.raises(ValueError):
        FlatRMSprop(p, lr=1e-3, weight_decay=1e-4)
    with pytest.raises(ValueError):
        FlatSGD(p, lr=1e-3, momentum=0.9)
    with pytest.raises(ValueError):
        FlatSGD(p, lr=1e-3, weight_decay=1e-4)
    with pytest.raises(ValueError):
        FlatSGD(p, lr=1e-3, nesterov=True)


# ---- 1. the kernels against the float64 oracle, every path ------------------------------------------------------------
def _oracle_run(name, shapes, max_norm, steps=5, seed=0, path="fused"):
    from prism_b200 import _lib
    from prism_b200.agents import optim
    gen = torch.Generator().manual_seed(seed)
    # parameters of the size of the update they receive: the parameter is stored in fp32 after every step, and one
    # rounding of |p| ~ 4 (2.4e-7) alone is more than 1e-5 of an accumulated update of ~1e-2 -- at this scale the bar on
    # p_5 - p_0 measures the update arithmetic, not the storage format
    p0 = [torch.randn(s, generator=gen) * 1e-4 for s in shapes]
    params = [t.to(DEV).requires_grad_(True) for t in p0]
    opt = _make_opt(name, params, max_grad_norm=max_norm)
    assert (opt.numel > opt._fused_max_n()) == (path == "large"), (opt.numel, opt._fused_max_n())
    old = optim.FUSED_STEP
    optim.FUSED_STEP = path == "fused"
    try:
        P = opt.arena.double().cpu().numpy()
        start = P.copy()
        M, V = np.zeros_like(P), np.zeros_like(P)
        for it in range(steps):
            grads = [torch.randn(s, generator=gen) * (3.0 if it % 2 == 0 else 0.2) for s in shapes]
            for q, g in zip(params, grads):
                q.grad = g.to(DEV)
            params[1].grad = None                         # a parameter without a gradient this step: zero slice
            flat = np.zeros_like(P)
            for k, (g, o) in enumerate(zip(grads, opt.offsets)):
                if k != 1:
                    flat[o:o + g.numel()] = g.double().numpy().reshape(-1)
            torch.cuda.synchronize()
            before = _lib.launch_count()
            opt.step()
            torch.cuda.synchronize()
            assert _lib.launch_count() - before == (1 if path == "fused" else 2)
            P, M, V, norm = oracle_step(name, P, M, V, flat, opt.lr, getattr(opt, "alpha", 0.0), opt.eps, max_norm)
            # stored as the kernel stores them: fp32
            P, M, V = (x.astype(np.float32).astype(np.float64) for x in (P, M, V))
            assert rel_err(opt.norm_out.cpu().numpy(), np.array(norm)) < 1e-6, (it, opt.norm_out, norm)
            assert rel_err(opt.arena.cpu().numpy(), P) < 1e-6, it
            if opt.exp_avg_sq is not None:
                assert rel_err(opt.exp_avg_sq.cpu().numpy(), V) < 1e-6, it
            if opt.exp_avg is not None:
                assert rel_err(opt.exp_avg.cpu().numpy(), M) < 1e-6, it
        d_got = opt.arena.double().cpu().numpy() - start
        d_want = P - start
        assert np.abs(d_got - d_want).max() <= 1e-5 * np.abs(d_want).max()
        assert int(opt.step_count) == steps
        if name == "sgd":
            assert opt.exp_avg is None and opt.exp_avg_sq is None
        elif name == "rmsprop":
            assert opt.exp_avg is None
    finally:
        optim.FUSED_STEP = old


SMALL = [(64, 33), (33,), (7, 5, 3), (1,), (130,), (256, 256)]


@gpu
@pytest.mark.parametrize("clip", ["active", "inactive", "zero"])
@pytest.mark.parametrize("path", ["fused", "two_launch"])
@pytest.mark.parametrize("name", RULES)
def test_kernels_match_float64_oracle(name, path, clip):
    max_norm = {"active": 1.0, "inactive": 1e6, "zero": 0.0}[clip]
    _oracle_run(name, SMALL, max_norm, path=path)


@gpu
@pytest.mark.parametrize("name", RULES)
def test_kernels_match_float64_oracle_above_the_fused_limit(name):
    from prism_b200 import _lib
    n_max = int(_lib.load().pb_opt_fused_max_n(_rule(name)))
    assert n_max > 0
    _oracle_run(name, [(n_max // 2 + 5,), (33,), (n_max // 2 + 4,)], 1.0, path="large")


@gpu
def test_sgd_leaves_state_arrays_untouched_and_accepts_null_ones():
    from prism_b200 import _lib
    lib = _lib.load()
    n = 4096
    p = torch.randn(n, device=DEV)
    g = torch.randn(n, device=DEV)
    sentinel = torch.full((n,), 7.0, device=DEV)
    m, v = sentinel.clone(), sentinel.clone()
    step = torch.zeros(1, dtype=torch.int64, device=DEV)
    parts = torch.zeros(4096, device=DEV)
    norm = torch.zeros(2, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    n_part = C.c_int(0)
    ref = p.clone()
    for ptrs in ((m.data_ptr(), v.data_ptr()), (None, None)):
        _lib.check(lib.pb_grad_sumsq(n, g.data_ptr(), parts.data_ptr(), step.data_ptr(), C.byref(n_part), st))
        _lib.check(lib.pb_opt_clip_apply(_lib.PB_OPT_SGD, n, p.data_ptr(), g.data_ptr(), ptrs[0], ptrs[1], step.data_ptr(),
                                         1e-2, 0.0, 0.0, 0.0, 0.0, parts.data_ptr(), n_part.value, norm.data_ptr(), st))
    torch.cuda.synchronize()
    assert torch.equal(m, sentinel) and torch.equal(v, sentinel)
    assert int(step) == 2
    assert rel_err(p.cpu().numpy(), (ref - 2e-2 * g).cpu().numpy()) < 1e-6


# ---- 2. against torch.optim itself -------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("max_norm", [1.0, 1e6])
@pytest.mark.parametrize("name", RULES)
def test_matches_torch_optim_over_steps(name, max_norm):
    torch.manual_seed(1)
    shapes = [(64, 33), (33,), (7, 5, 3), (1,), (130,)]
    ref_p = [torch.randn(s, device=DEV).requires_grad_(True) for s in shapes]
    dev_p = [p.detach().clone().requires_grad_(True) for p in ref_p]
    lr, alpha, eps = 1e-3, 0.95, 0.01
    if name == "sgd":
        ref_opt = torch.optim.SGD(ref_p, lr=lr)
    else:
        ref_opt = torch.optim.RMSprop(ref_p, lr=lr, alpha=alpha, eps=eps, centered=name == "rmsprop_centered")
    opt = _make_opt(name, dev_p, lr=lr, alpha=alpha, eps=eps, max_grad_norm=max_norm)
    for it in range(5):
        grads = [torch.randn(s, device=DEV) * (3.0 if it % 2 == 0 else 0.2) for s in shapes]
        for p, g in zip(ref_p, grads):
            p.grad = g.clone()
        total = torch.nn.utils.clip_grad_norm_(ref_p, max_norm)
        ref_opt.step()
        for p, g in zip(dev_p, grads):
            p.grad = g.clone()
        opt.step()
        torch.cuda.synchronize()
        assert abs(float(opt.norm_out[0]) - float(total)) <= 1e-6 * float(total)
        for a, b in zip(dev_p, ref_p):
            assert rel_err(a.detach().cpu().numpy(), b.detach().cpu().numpy()) < 1e-6, it
        if name != "sgd":
            for k, (p, o) in enumerate(zip(ref_p, opt.offsets)):
                st = ref_opt.state[p]
                got = opt.square_avg[o:o + p.numel()].view_as(p)
                assert rel_err(got.cpu().numpy(), st["square_avg"].cpu().numpy()) < 1e-6, (it, k)
                if name == "rmsprop_centered":
                    got = opt.grad_avg[o:o + p.numel()].view_as(p)
                    assert rel_err(got.cpu().numpy(), st["grad_avg"].cpu().numpy()) < 1e-6, (it, k)
                assert float(st["step"]) == float(opt.step_count)


# ---- 3. agent level ---------------------------------------------------------------------------------------------------
def _agent_setup(kind, name, graph, seed=0):
    """An agent at configs[1] (DQN, 0.27 M parameters) or configs[0] (IDS + IQN, 3 M parameters) shapes, and one fixed
    batch + per-row weights from a filled buffer."""
    import prism_b200
    from oracle.gen_golden import make_script
    kw = dict(use_adam=False, use_rmsprop=name == "rmsprop", device=DEV, experience_replay_capacity=1024,
              use_cuda_graph=graph, replay_max_streams=4, replay_staging_rows=64)
    if kind == "configs1":
        cfg, shape, A = prism_b200.minatar_dqn_per_config(batch_size=64, **kw), (10, 10, 6), 4
    else:
        cfg, shape, A = prism_b200.minatar_ids_iqn_config(batch_size=32, **kw), (10, 10, 4), 3
    torch.manual_seed(seed)
    agent = prism_b200.build_agent(cfg, shape, A)
    buf = prism_b200.build_exp_buffer(cfg)
    S = make_script(seed + 3, n_streams=4, n_steps=300, obs_shape=shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"]).reshape((-1,) + shape)
    buf.extend_batch(S["stream"], S["obs"].reshape((-1,) + shape), S["action"], S["reward"], S["done"], S["trunc"], succ)
    buf._flush()
    buf.inject_uniforms(torch.from_numpy(np.random.default_rng(seed).random(cfg.batch_size)))
    b = buf.sample()
    batch = prism_b200.Batch({"observation": b["observation"].clone(),
                              "next": {"observation": b["next"]["observation"].clone(),
                                       "reward": b["next"]["reward"].clone()},
                              "nonterminal": b["nonterminal"].clone(), "gamma": b["gamma"].clone(),
                              "action": b["action"].clone()})
    w = torch.from_numpy(np.random.default_rng(seed + 1).uniform(0.2, 1.0, cfg.batch_size).astype(np.float32)).to(DEV)
    return cfg, agent, batch, w


def _pin_quantile_draws(src, dst):
    """The IQN heads draw their quantiles from device generators of their own: give ``dst`` the state of ``src``'s."""
    for ag in (src, dst):
        for m in (ag.model, ag.target_model):
            d = getattr(m, "distribution_model", None) if m is not None else None
            if d is not None and hasattr(d, "_rng_state"):
                d._rng_state()
    for (rng, _), (_, saved) in zip(dst.quantile_rng_snapshot(), src.quantile_rng_snapshot()):
        rng.copy_(saved)


def _torch_state_flat(agent, ref_opt, key):
    """torch.optim's per-parameter state laid out like the flat arena."""
    arena = agent.model._flat_arena
    out = torch.zeros_like(arena)
    base = arena.data_ptr()
    for p in agent.model.parameters():
        st = ref_opt.state.get(p)
        if st is not None and key in st:
            o = (p.data_ptr() - base) // 4
            out[o:o + p.numel()] = st[key].reshape(-1)
    return out


def _updates(agent, batch, w, n):
    losses, tds = [], []
    for _ in range(n):
        td = agent.update(batch, w)
        losses.append(float(agent._static_total_loss))
        tds.append(td.clone())
    torch.cuda.synchronize()
    return losses, tds


AGENT_CASES = [("configs1", "rmsprop"), ("configs0", "rmsprop"), ("configs1", "sgd")]


@gpu
@pytest.mark.parametrize("kind,name", AGENT_CASES)
def test_agent_builds_a_flat_optimizer_and_graph_equals_eager(kind, name):
    from prism_b200 import FlatOptimizer, FlatRMSprop, FlatSGD
    cfg, a_eager, batch, w = _agent_setup(kind, name, graph=False)
    _, a_graph, _, _ = _agent_setup(kind, name, graph=True)
    _pin_quantile_draws(a_eager, a_graph)
    assert isinstance(a_eager.optimizer, FlatRMSprop if name == "rmsprop" else FlatSGD)
    assert isinstance(a_eager.optimizer, FlatOptimizer)
    if name == "rmsprop":
        opt = a_eager.optimizer
        assert opt.centered and (opt.alpha, opt.eps) == (cfg.rmsprop_alpha, cfg.rmsprop_epsilon)
    if kind == "configs1":
        assert a_eager.optimizer.numel <= a_eager.optimizer._fused_max_n()       # the one-launch path
    le, te = _updates(a_eager, batch, w, 3)
    lg, tg = _updates(a_graph, batch, w, 3)
    assert np.allclose(le, lg, rtol=1e-5, atol=1e-8), (le, lg)
    for x, y in zip(te, tg):
        assert rel_err(y.cpu().numpy(), x.cpu().numpy()) < 1e-5
    assert rel_err(a_graph.optimizer.arena.cpu().numpy(), a_eager.optimizer.arena.cpu().numpy()) < 1e-5
    for s_e, s_g in ((a_eager.optimizer.exp_avg, a_graph.optimizer.exp_avg),
                     (a_eager.optimizer.exp_avg_sq, a_graph.optimizer.exp_avg_sq)):
        if s_e is not None:
            assert rel_err(s_g.cpu().numpy(), s_e.cpu().numpy()) < 1e-5


@gpu
@pytest.mark.parametrize("kind,name", AGENT_CASES)
def test_graph_warm_up_does_not_train(kind, name):
    """After the capture (three warm-up iterations) and ONE replay, the parameters equal ONE eager step."""
    _, a_eager, batch, w = _agent_setup(kind, name, graph=False)
    _, a_graph, _, _ = _agent_setup(kind, name, graph=True)
    _pin_quantile_draws(a_eager, a_graph)
    start = a_graph.optimizer.arena.clone()
    _updates(a_eager, batch, w, 1)
    _updates(a_graph, batch, w, 1)
    assert int(a_graph.optimizer.step_count) == 1
    assert float((a_eager.optimizer.arena - start).abs().max()) > 0
    assert rel_err(a_graph.optimizer.arena.cpu().numpy(), a_eager.optimizer.arena.cpu().numpy()) < 1e-6


@gpu
@pytest.mark.parametrize("kind,name", AGENT_CASES)
def test_agent_matches_torch_optim_with_clip_grad_norm(kind, name):
    """Same weights, same batch: the flat optimizer vs ``clip_grad_norm_`` + ``torch.optim.RMSprop(centered=True)`` /
    ``torch.optim.SGD`` on an agent built the same way (Agent's generic optimizer branch)."""
    cfg, mine, batch, w = _agent_setup(kind, name, graph=False)
    _, ref, _, _ = _agent_setup(kind, name, graph=False)
    _pin_quantile_draws(mine, ref)
    params = list(ref.model.parameters())
    if name == "rmsprop":
        ref.optimizer = torch.optim.RMSprop(params, lr=cfg.learning_rate, alpha=cfg.rmsprop_alpha, eps=cfg.rmsprop_epsilon,
                                            centered=True)
    else:
        ref.optimizer = torch.optim.SGD(params, lr=cfg.learning_rate)
    lm, tm = _updates(mine, batch, w, 3)
    lr_, tr = _updates(ref, batch, w, 3)
    assert np.allclose(lm, lr_, rtol=1e-4, atol=1e-7), (lm, lr_)
    for x, y in zip(tm, tr):
        assert rel_err(x.cpu().numpy(), y.cpu().numpy()) < 1e-4
    assert rel_err(mine.optimizer.arena.cpu().numpy(), ref.model._flat_arena.cpu().numpy()) < 1e-4
    if name == "rmsprop":
        for key, flat in (("square_avg", mine.optimizer.square_avg), ("grad_avg", mine.optimizer.grad_avg)):
            want = _torch_state_flat(ref, ref.optimizer, key)
            assert rel_err(flat.cpu().numpy(), want.cpu().numpy()) < 1e-4, key


# ---- 4. LearnerStep on one GPU ----------------------------------------------------------------------------------------
def _script(seed, n, obs_shape=(10, 10, 6), A=4):
    from oracle.gen_golden import make_script
    S = make_script(seed, n_streams=4, n_steps=n, obs_shape=obs_shape, p_done=0.05, p_trunc=0.03, n_actions=A)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])
    shp = (-1,) + obs_shape
    return (S["stream"], S["obs"].reshape(shp), S["action"], S["reward"], S["done"], S["trunc"], succ.reshape(shp))


def _step_setup(name, use_per, B=16, n0=200, seed=0):
    import prism_b200
    cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=256, batch_size=B, use_per=use_per,
                                            replay_max_streams=4, replay_staging_rows=64, use_cuda_graph=False,
                                            use_adam=False, use_rmsprop=name == "rmsprop")
    torch.manual_seed(seed)
    agent = prism_b200.build_agent(cfg, (10, 10, 6), 4)
    buf = prism_b200.build_exp_buffer(cfg)
    buf.extend_batch(*_script(5, n0))
    buf._flush()
    return agent, buf


def _step_run(name, use_per, use_graph, prefetch, us):
    from prism_b200.learner_step import LearnerStep
    B = us.shape[1]
    agent, buf = _step_setup(name, use_per, B)
    step = LearnerStep(buf, agent, batch_size=B, use_cuda_graph=use_graph, prefetch=prefetch)
    losses = [float(step.step(u=torch.from_numpy(u.copy()))) for u in us]
    torch.cuda.synchronize()
    if use_graph:
        assert step.launches_per_step > 0
    opt = agent.optimizer
    return losses, opt.arena.clone(), [None if t is None else t.clone() for t in (opt.exp_avg, opt.exp_avg_sq)]


def _same(a, b, tol=1e-5):
    assert np.allclose(a[0], b[0], rtol=tol, atol=1e-7), (a[0], b[0])
    assert rel_err(a[1].cpu().numpy(), b[1].cpu().numpy()) < tol
    for x, y in zip(a[2], b[2]):
        assert (x is None) == (y is None)
        if x is not None:
            assert rel_err(x.cpu().numpy(), y.cpu().numpy()) < tol


@gpu
@pytest.mark.parametrize("prefetch", [False, True])
@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("name", ["rmsprop", "sgd"])
def test_learner_step_uniform_replay_equals_the_eager_update_loop(name, use_graph, prefetch):
    """Uniform replay: the step against ``buf.inject_uniforms(u); agent.update(buf.sample())`` (host uniforms; with
    prefetch they drive the NEXT batch, the first one comes from the device generator)."""
    from test_gpu_uniform_replay import SEED, oracle_philox
    B, iters = 16, 6
    us = np.random.default_rng(11).random((iters, B))
    got = _step_run(name, False, use_graph, prefetch, us)
    batch_u = [oracle_philox(SEED, 0, B)] + list(us[:-1]) if prefetch else list(us)
    agent, buf = _step_setup(name, False, B)
    losses = []
    for u in batch_u:
        buf.inject_uniforms(torch.from_numpy(np.ascontiguousarray(u)))
        agent.update(buf.sample())
        losses.append(float(agent._static_total_loss))
    torch.cuda.synchronize()
    opt = agent.optimizer
    _same(got, (losses, opt.arena.clone(), [None if t is None else t.clone() for t in (opt.exp_avg, opt.exp_avg_sq)]))


@gpu
@pytest.mark.parametrize("name", ["rmsprop", "sgd"])
def test_learner_step_per_replay_graph_prefetch_and_eager_agree(name):
    """PER: the one-graph step, with and without prefetch, equals the eager step (same host uniforms, same priorities
    written back); and the optimizer really trained."""
    B, iters = 16, 6
    us = np.random.default_rng(12).random((iters, B))
    ref = _step_run(name, True, False, False, us)
    for use_graph, prefetch in ((True, False), (False, True), (True, True)):
        if prefetch:
            # under prefetch host uniforms drive the NEXT batch: compare prefetch runs with each other
            ref_p = _step_run(name, True, False, True, us)
            _same(_step_run(name, True, use_graph, True, us), ref_p)
        else:
            _same(_step_run(name, True, use_graph, prefetch, us), ref)
    agent, _ = _step_setup(name, True, B)
    assert float((ref[1] - agent.optimizer.arena).abs().max()) > 0


# ---- 5. loopback data parallelism ---------------------------------------------------------------------------------------
class _Opt:
    """The fields PeerGroup.allreduce_adam reads from a flat optimizer, for one update rule."""

    def __init__(self, name, n, p0, lr=1e-3, alpha=0.95, eps=0.01, max_grad_norm=10.0):
        self.rule = _rule(name)
        self.arena = p0.clone()
        self.exp_avg = torch.zeros(n, device=DEV) if name == "rmsprop_centered" else None
        self.exp_avg_sq = None if name == "sgd" else torch.zeros(n, device=DEV)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=DEV)
        self.partials = torch.zeros(4096, device=DEV)
        self.norm_out = torch.zeros(2, device=DEV)
        self.lr, self.alpha, self.eps, self.max_grad_norm = lr, alpha, eps, max_grad_norm

    def _hyper(self):
        return self.alpha, 0.0


def _run_allreduce(name, world, n):
    from prism_b200 import _lib
    from prism_b200.peer import PeerGroup
    lib = _lib.load()
    groups = PeerGroup.loopback(world, n, DEV)
    g = torch.Generator(device=DEV).manual_seed(n + world)
    p0 = torch.randn(n, device=DEV, generator=g)
    grads = [torch.randn(n, device=DEV, generator=g) * (3.0 if r == 0 else 1.0) for r in range(world)]
    opts = [_Opt(name, n, p0) for _ in range(world)]
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    # every tensor exists before the first exchange kernel spins (see tests/test_gpu_peer.py)
    staged = [[grads[r] * (1.0 + it) for r in range(world)] for it in range(3)]
    torch.cuda.synchronize()
    for it in range(3):
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                groups[r].grad_in_flight().copy_(staged[it][r])
                groups[r].allreduce_adam(opts[r])
    torch.cuda.synchronize()
    # reference: the single-rank two-launch step on the rank-order fp32 sum
    ref = _Opt(name, n, p0)
    st = torch.cuda.current_stream().cuda_stream
    for it in range(3):
        total = grads[0] * (1.0 + it)
        for r in range(1, world):
            total = total + grads[r] * (1.0 + it)
        n_part = C.c_int(0)
        _lib.check(lib.pb_grad_sumsq(n, total.data_ptr(), ref.partials.data_ptr(), ref.step_count.data_ptr(),
                                     C.byref(n_part), st), "pb_grad_sumsq")
        _lib.check(lib.pb_opt_clip_apply(ref.rule, n, ref.arena.data_ptr(), total.data_ptr(), _lib.ptr(ref.exp_avg),
                                         _lib.ptr(ref.exp_avg_sq), ref.step_count.data_ptr(), ref.lr, ref.alpha, 0.0,
                                         ref.eps, ref.max_grad_norm, ref.partials.data_ptr(), n_part.value,
                                         ref.norm_out.data_ptr(), st), "pb_opt_clip_apply")
    torch.cuda.synchronize()
    for r in range(world):
        groups[r].check()
        assert int(opts[r].step_count) == 3
        assert torch.equal(opts[r].arena, opts[0].arena), "replicas must stay bit-identical"
        for a, b in ((opts[r].exp_avg, opts[0].exp_avg), (opts[r].exp_avg_sq, opts[0].exp_avg_sq)):
            assert a is None or torch.equal(a, b)
    assert rel_err(opts[0].norm_out.cpu().numpy(), ref.norm_out.cpu().numpy()) < 1e-6
    assert rel_err(opts[0].arena.cpu().numpy(), ref.arena.cpu().numpy()) < 1e-6
    for a, b in ((opts[0].exp_avg, ref.exp_avg), (opts[0].exp_avg_sq, ref.exp_avg_sq)):
        if a is not None:
            assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-6


@gpu
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("n,one_shot", [(4096, True), (1_000_004, True), (1_000_004, False)])
@pytest.mark.parametrize("name", RULES)
def test_peer_exchange_multi_launch_matches_single_rank_step(name, world, n, one_shot, monkeypatch):
    from prism_b200 import peer as peer_mod
    monkeypatch.setattr(peer_mod, "ONE_SHOT_MAX_BYTES", (1 << 40) if one_shot else 0)
    monkeypatch.setattr(peer_mod, "FUSED_EXCHANGE", False)
    _run_allreduce(name, world, n)


@gpu
@pytest.mark.parametrize("world,n", [(2, 4096), (4, 4096), (8, 4096), (8, 40_000), (4, 40_000), (2, 100_000),
                                     (4, 100_000), (2, 400_004)])
@pytest.mark.parametrize("name", RULES)
def test_peer_fused_exchange_matches_single_rank_step(name, world, n, monkeypatch):
    from prism_b200 import _lib, peer as peer_mod
    monkeypatch.setattr(peer_mod, "FUSED_EXCHANGE", True)
    assert n <= int(_lib.load().pb_peer_allreduce_opt_max_n(_rule(name)))
    _run_allreduce(name, world, n)


# ---- 6. two processes on two GPUs -----------------------------------------------------------------------------------------
def _run(cmd, env=None):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=540, env=env)
    assert p.returncode == 0, p.stdout[-3000:]


@gpu
@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_ranks_with_rmsprop_equal_one_rank_on_the_union_batch(tmp_path, exchange):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = os.path.join(HERE, "mp_worker_dp_optim.py")
    out2, out1 = str(tmp_path / "dp2"), str(tmp_path / "one")
    env = dict(os.environ, PB_DP_EXCHANGE=exchange)
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
          "127.0.0.1", "--master-port", str(29740 + (exchange == "nccl")), worker, "--out", out2], env=env)
    _run([sys.executable, worker, "--out", out1, "--union", "2"])
    one = torch.load(out1 + ".rank0", weights_only=False)
    r0, r1 = (torch.load(out2 + ".rank%d" % r, weights_only=False) for r in (0, 1))
    assert r0["exchange"] == exchange
    assert torch.equal(r0["arena"], r1["arena"]), "replicas diverged"
    B_pad, B_global = r0["B_pad"], one["B_pad"]
    both = (np.asarray(r0["losses"]) + np.asarray(r1["losses"])) * (B_pad / B_global)
    assert np.allclose(both, one["losses"], rtol=2e-5, atol=1e-7), (r0["losses"], r1["losses"], one["losses"])
    assert rel_err(r0["arena"].numpy(), one["arena"].numpy()) < 2e-5
    for a, b in zip(r0["state"], one["state"]):
        assert (a is None) == (b is None)
        if a is not None:
            assert rel_err(a.numpy(), b.numpy()) < 2e-5
    leaves = torch.cat([r0["leaves"], r1["leaves"]])
    assert np.allclose(leaves.numpy(), one["leaves"].numpy(), rtol=1e-4, atol=1e-7)


# ---- 7. checkpoints -------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["rmsprop", "sgd"])
def test_agent_save_load_continues_bit_exact(name, tmp_path):
    _, a, batch, w = _agent_setup("configs1", name, graph=False)
    _updates(a, batch, w, 2)
    a.save(str(tmp_path))
    _updates(a, batch, w, 3)
    _, b, _, _ = _agent_setup("configs1", name, graph=False, seed=5)          # different initial weights
    b.load(str(tmp_path))
    _updates(b, batch, w, 3)
    assert torch.equal(a.optimizer.arena, b.optimizer.arena)
    for x, y in ((a.optimizer.exp_avg, b.optimizer.exp_avg), (a.optimizer.exp_avg_sq, b.optimizer.exp_avg_sq)):
        assert (x is None) == (y is None) and (x is None or torch.equal(x, y))
    if name == "rmsprop":
        assert int(b.optimizer.step_count) == 5


@gpu
@pytest.mark.parametrize("name", ["rmsprop_centered", "rmsprop", "sgd"])
def test_checkpoints_cross_load_with_torch_optim(name):
    """``torch.optim.X.load_state_dict(flat.state_dict())`` and the reverse; continuing steps agree."""
    torch.manual_seed(2)
    shapes = [(64, 33), (33,), (7, 5, 3), (130,)]
    lr, alpha, eps = 1e-3, 0.95, 0.01

    def torch_opt(params):
        if name == "sgd":
            return torch.optim.SGD(params, lr=lr)
        return torch.optim.RMSprop(params, lr=lr, alpha=alpha, eps=eps, centered=name == "rmsprop_centered")

    grads = [[torch.randn(s, device=DEV) for s in shapes] for _ in range(6)]

    def run(opt, params, its):
        for it in its:
            for p, g in zip(params, grads[it]):
                p.grad = g.clone()
            if not hasattr(opt, "rule"):
                torch.nn.utils.clip_grad_norm_(params, 5.0)
            opt.step()
        torch.cuda.synchronize()

    p0 = [torch.randn(s, device=DEV) for s in shapes]
    # flat -> torch
    fp = [t.clone().requires_grad_(True) for t in p0]
    flat = _make_opt(name, fp, lr=lr, alpha=alpha, eps=eps, max_grad_norm=5.0)
    run(flat, fp, range(3))
    sd = flat.state_dict()
    tp = [p.detach().clone().requires_grad_(True) for p in fp]
    top = torch_opt(tp)
    top.load_state_dict(sd)
    if name != "sgd":
        assert set(top.state_dict()["state"][0]) == set(sd["state"][0])
        assert set(top.state_dict()["param_groups"][0]) == set(sd["param_groups"][0])
    run(flat, fp, range(3, 6))
    run(top, tp, range(3, 6))
    for a, b in zip(fp, tp):
        assert rel_err(a.detach().cpu().numpy(), b.detach().cpu().numpy()) < 1e-6
    # torch -> flat
    tp = [t.clone().requires_grad_(True) for t in p0]
    top = torch_opt(tp)
    run(top, tp, range(3))
    fp = [p.detach().clone().requires_grad_(True) for p in tp]
    flat = _make_opt(name, fp, lr=0.5, alpha=0.5, eps=0.5, max_grad_norm=5.0)
    flat.load_state_dict(top.state_dict())
    assert flat.lr == lr and (name == "sgd" or (flat.alpha, flat.eps) == (alpha, eps))
    if name != "sgd":
        assert int(flat.step_count) == 3
    run(top, tp, range(3, 6))
    run(flat, fp, range(3, 6))
    for a, b in zip(fp, tp):
        assert rel_err(a.detach().cpu().numpy(), b.detach().cpu().numpy()) < 1e-6
    if name != "sgd":
        for k, (p, o) in enumerate(zip(tp, flat.offsets)):
            got = flat.square_avg[o:o + p.numel()].view_as(p)
            assert rel_err(got.cpu().numpy(), top.state[p]["square_avg"].cpu().numpy()) < 1e-6, k
