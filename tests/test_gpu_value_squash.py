"""Value squashing on the GPU (Config.loss_squish_fn_id = "obs_look_further" / "symlog").

1. pb_value_squash, both kinds and both directions, against fp64 of the definitions.
2. The four *_sq entries at every kind against fp64 oracles written here; at PB_SQUASH_NONE bit-identical to the entries
   without the suffix.
3. Agent.update at the configs[0] / [1] / [4] shapes with each id against oracle/agent_oracle.py's agent with the
   squashed heads of tests/squash_oracle.py (eager, graph, three consecutive steps), with the routes asserted.
4. LearnerStep (PER, prefetch, fused ingest) with squashing against the eager sample -> update -> write-back loop;
   two ranks against one rank on the union buffer.
5. The acting graph (IDS with the unsquish function) against eager acting."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rel_err
from test_value_squash import fp64_squash, log_grid

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
KINDS = {"none": 0, "obs_look_further": 1, "symlog": 2}
IDS = ["obs_look_further", "symlog"]


def _lib():
    from prism_b200 import _lib as L
    return L, L.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _h(x, kind, inverse):
    return x if kind == "none" else fp64_squash(x, kind, inverse)


# ---- 1. pb_value_squash ----------------------------------------------------------------------------------------------
def _dev_squash(x, kind, inverse):
    L, lib = _lib()
    xd = torch.as_tensor(np.ascontiguousarray(x, np.float32)).to(DEV)
    y = torch.empty_like(xd)
    L.check(lib.pb_value_squash(xd.numel(), xd.data_ptr(), y.data_ptr(), KINDS[kind], int(inverse), _stream()),
            "pb_value_squash")
    return y.cpu().numpy()


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("kind", IDS)
def test_value_squash_matches_fp64(kind, inverse):
    x = log_grid(1e-30, 80.0 if (kind == "symlog" and inverse) else 1e30)
    got = _dev_squash(x, kind, inverse).astype(np.float64)
    want = fp64_squash(x, kind, inverse)
    rel = np.abs(got - want) / np.abs(want)
    assert rel.max() < 1e-6, (float(rel.max()), float(x[rel.argmax()]))
    # the signed zeros keep their sign, NaN propagates
    z = _dev_squash(np.array([0.0, -0.0, np.nan], np.float32), kind, inverse)
    assert z[0] == 0 and not np.signbit(z[0]) and z[1] == 0 and np.signbit(z[1]) and np.isnan(z[2])


@pytest.mark.parametrize("kind", IDS)
def test_squash_of_unsquash_round_trips(kind):
    x = log_grid(1e-30, 80.0 if kind == "symlog" else 1e30)
    back = _dev_squash(_dev_squash(x, kind, True), kind, False).astype(np.float64)
    err = np.abs(back - x) / np.maximum(1.0, np.abs(x))
    assert err.max() < 2e-6, (float(err.max()), float(x[err.argmax()]))


def test_squish_functions_run_the_kernel_and_refuse_unknown_kinds():
    from prism_b200.agents import squish_functions as sf
    L, lib = _lib()
    x = torch.linspace(-50, 50, 1001, device=DEV)
    for name, (h, hinv) in sf.SQUISH_FUNCTIONS.items():
        assert np.array_equal(h(x).cpu().numpy(), _dev_squash(x.cpu().numpy(), name, False))
        assert np.array_equal(hinv(x.view(11, 91)).view(-1).cpu().numpy(), _dev_squash(x.cpu().numpy(), name, True))
    assert lib.pb_value_squash(4, 16, 16, 3, 0, None) == -3          # unknown kind: PB_E_UNSUPPORTED, nothing launched
    assert lib.pb_value_squash(4, 16, 16, 1, 2, None) == -1
    assert lib.pb_ids_select_sq(4, 4, 2, 2, 16, 16, 0.1, 1e-10, 0.25, 16, None, None, -1) == -3
    assert lib.pb_iqn_qh_loss_sq(4, 2, 2, 3, 16, 16, 16, 16, 16, 16, 16, None, 1.0, 1.0, None, 1.0, 16, 16, None, 3) == -3
    assert lib.pb_ens_q_loss_sq(4, 3, 2, 16, 16, 16, 16, 16, 16, None, 1.0, None, 1.0, 16, 16, None, 7) == -3
    assert lib.pb_ens_q_loss_total_sq(4, 3, 2, 16, 16, 16, 16, 16, 16, None, 1.0, None, 1.0, 16, 16, None, 1.0, None,
                                      16, None, 16, None, 9) == -3
    with pytest.raises(RuntimeError, match="no backward"):
        sf.symlog(x.clone().requires_grad_(True))


# ---- 2. the loss and selection entries against fp64 ---------------------------------------------------------------------
def _offsets(rng, rows, A, spread=0.6):
    """Per-row action offsets with a clear winner, so the argmax over actions is never decided by rounding."""
    base = np.linspace(-spread, spread, A)
    return np.stack([rng.permutation(base) for _ in range(rows)])


def _iqn_inputs(B, T, Tp, A, seed):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    off = _offsets(rng, B, A).astype(np.float32)
    return dict(z_cur=f(T, B, A) * 0.8, tau=rng.random((T, B)).astype(np.float32),
                z_on=(f(Tp, B, A) * 0.2 + off[None]).astype(np.float32), z_tg=f(Tp, B, A) * 0.9 + 0.3,
                action=rng.integers(0, A, B), ret=f(B) * 2.0, gdn=(0.99 ** rng.integers(1, 4, B)).astype(np.float32),
                nonterm=rng.random(B) > 0.2, w=(rng.random(B) * 0.7 + 0.3).astype(np.float32))


def iqn_fp64(d, kind, kappa, loss_weight, use_nonterm, use_w, grad_scale):
    T, B, A = d["z_cur"].shape
    zc, zon, ztg, tau = (d[k].astype(np.float64) for k in ("z_cur", "z_on", "z_tg", "tau"))
    Tp = zon.shape[0]
    rows = np.arange(B)
    best = zon.mean(axis=0).argmax(axis=1)
    g = d["gdn"].astype(np.float64) * (d["nonterm"] if use_nonterm else 1.0)
    y = _h(d["ret"].astype(np.float64)[None] + g[None] * _h(ztg[:, rows, best], kind, True), kind, False)   # (Tp, B)
    theta = zc[:, rows, d["action"]]                                                                       # (T, B)
    delta = y[None, :, :] - theta[:, None, :]                                                              # (T, Tp, B)
    ad = np.abs(delta)
    quad = ad <= kappa
    hub = np.where(quad, 0.5 * delta * delta, kappa * (ad - 0.5 * kappa))
    dh = np.where(quad, delta, np.sign(delta) * kappa)
    wq = np.abs(tau[:, None, :] - (delta < 0))
    loss = (wq * hub).sum(axis=(0, 1)) / kappa / Tp * loss_weight
    w = d["w"].astype(np.float64) if use_w else 1.0
    gi = -(wq * dh).sum(axis=1) / kappa * (w * grad_scale * loss_weight / Tp)                             # (T, B)
    grad = np.zeros((T, B, A))
    grad[:, rows, d["action"]] = gi
    return loss, grad


def _t(x, dtype=None):
    return torch.as_tensor(np.ascontiguousarray(x) if dtype is None else np.ascontiguousarray(x, dtype)).to(DEV)


def _run_iqn(lib, d, kind, kappa, loss_weight, use_nonterm, use_w, grad_scale, entry):
    T, B, A = d["z_cur"].shape
    Tp = d["z_on"].shape[0]
    t = {k: _t(v) for k, v in d.items() if k not in ("action", "nonterm")}
    act, nt = _t(d["action"], np.int64), _t(d["nonterm"])
    loss = torch.full((B,), float("nan"), device=DEV)
    grad = torch.full((T, B, A), float("nan"), device=DEV)
    args = (B, T, Tp, A, t["z_cur"].data_ptr(), t["tau"].data_ptr(), t["z_on"].data_ptr(), t["z_tg"].data_ptr(),
            act.data_ptr(), t["ret"].data_ptr(), t["gdn"].data_ptr(), nt.data_ptr() if use_nonterm else None, kappa,
            loss_weight, t["w"].data_ptr() if use_w else None, grad_scale, loss.data_ptr(), grad.data_ptr(), _stream())
    rc = lib.pb_iqn_qh_loss(*args) if entry == "plain" else lib.pb_iqn_qh_loss_sq(*args, KINDS[kind])
    assert rc == 0
    torch.cuda.synchronize()
    return loss.cpu().numpy(), grad.cpu().numpy()


@pytest.mark.parametrize("A", [3, 7, 18])
@pytest.mark.parametrize("B,use_nonterm,use_w", [(13, True, True), (64, False, False), (30, True, False)])
@pytest.mark.parametrize("kind", ["none"] + IDS)
def test_iqn_qh_loss_sq_matches_fp64(kind, B, use_nonterm, use_w, A):
    L, lib = _lib()
    T, Tp, kappa, loss_weight, grad_scale = 8, 12, 1.0, 0.7, (1.0 / B if use_w else 1.0)
    d = _iqn_inputs(B, T, Tp, A, seed=B * 100 + A)
    loss, grad = _run_iqn(lib, d, kind, kappa, loss_weight, use_nonterm, use_w, grad_scale, "sq")
    want_l, want_g = iqn_fp64(d, kind, kappa, loss_weight, use_nonterm, use_w, grad_scale)
    assert rel_err(loss, want_l) < 1e-5 and rel_err(grad, want_g) < 1e-5, (rel_err(loss, want_l), rel_err(grad, want_g))
    if kind == "none":
        plain = _run_iqn(lib, d, kind, kappa, loss_weight, use_nonterm, use_w, grad_scale, "plain")
        assert np.array_equal(loss, plain[0]) and np.array_equal(grad, plain[1])
    else:                                             # squashing really changed the targets
        assert rel_err(loss, iqn_fp64(d, "none", kappa, loss_weight, use_nonterm, use_w, grad_scale)[0]) > 1e-3


def _ens_inputs(B, K, A, seed):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    off = np.stack([_offsets(rng, B, A) for _ in range(K)]).astype(np.float32)                     # (K, B, A)
    return dict(q_cur=f(K, B, A), q_on=(f(K, B, A) * 0.05 + off).astype(np.float32), q_tg=f(K, B, A) * 1.5 + 0.2,
                action=rng.integers(0, A, B), ret=f(B) * 2.0, gdn=(0.99 ** rng.integers(1, 4, B)).astype(np.float32),
                nonterm=rng.random(B) > 0.2, w=(rng.random(B) * 0.7 + 0.3).astype(np.float32), dist=rng.random(B) * 2,
                q_off=np.float32(0.05))


def ens_fp64(d, kind, loss_weight, use_nonterm, use_w, grad_scale, q_scale=1.0, use_dist=False, use_off=False):
    K, B, A = d["q_cur"].shape
    qc, qon, qtg = (d[k].astype(np.float64) for k in ("q_cur", "q_on", "q_tg"))
    rows = np.arange(B)
    best = qon.argmax(axis=2)                                                                         # (K, B)
    g = d["gdn"].astype(np.float64) * (d["nonterm"] if use_nonterm else 1.0)
    sel = np.take_along_axis(qtg, best[..., None], axis=2)[..., 0]
    y = _h(d["ret"].astype(np.float64)[None] + g[None] * _h(sel, kind, True), kind, False)            # (K, B)
    diff = qc[:, rows, d["action"]] - y
    loss = (diff * diff).mean(axis=0) * loss_weight
    w = d["w"].astype(np.float64) if use_w else np.ones(B)
    grad = np.zeros((K, B, A))
    grad[:, rows, d["action"]] = (w * grad_scale * loss_weight * 2.0 / K)[None] * diff
    qq = q_scale * (loss - (float(d["q_off"]) if use_off else 0.0))
    dist = d["dist"] if use_dist else np.zeros(B)
    total = ((dist * w).sum() + (qq * w).sum()) / B
    td = 0.5 * dist + 0.5 * qq if use_dist else np.abs(qq)
    return loss, grad, total, td


def _run_ens(lib, d, kind, loss_weight, use_nonterm, use_w, grad_scale, entry, q_scale=1.0, use_dist=False,
             use_off=False):
    K, B, A = d["q_cur"].shape
    t = {k: _t(d[k]) for k in ("q_cur", "q_on", "q_tg", "ret", "gdn", "w")}
    act, nt = _t(d["action"], np.int64), _t(d["nonterm"])
    dist, off = _t(d["dist"], np.float32), _t(np.array([d["q_off"]], np.float32))
    loss = torch.full((B,), float("nan"), device=DEV)
    grad = torch.full((K, B, A), float("nan"), device=DEV)
    total = torch.full((1,), float("nan"), device=DEV)
    td = torch.full((B,), float("nan"), device=DEV)
    ticket = torch.zeros(1, dtype=torch.int32, device=DEV)
    head = (B, A, K, t["q_cur"].data_ptr(), t["q_on"].data_ptr(), t["q_tg"].data_ptr(), act.data_ptr(),
            t["ret"].data_ptr(), t["gdn"].data_ptr(), nt.data_ptr() if use_nonterm else None, loss_weight,
            t["w"].data_ptr() if use_w else None, grad_scale, loss.data_ptr(), grad.data_ptr())
    tail = (dist.data_ptr() if use_dist else None, q_scale, off.data_ptr() if use_off else None, total.data_ptr(),
            td.data_ptr(), ticket.data_ptr())
    if entry == "plain":
        rc = lib.pb_ens_q_loss(*head, _stream())
    elif entry == "sq":
        rc = lib.pb_ens_q_loss_sq(*head, _stream(), KINDS[kind])
    elif entry == "total":
        rc = lib.pb_ens_q_loss_total(*head, *tail, _stream())
    else:
        rc = lib.pb_ens_q_loss_total_sq(*head, *tail, _stream(), KINDS[kind])
    assert rc == 0
    torch.cuda.synchronize()
    assert int(ticket) == 0
    return loss.cpu().numpy(), grad.cpu().numpy(), float(total), td.cpu().numpy()


@pytest.mark.parametrize("A", [3, 7, 18])
@pytest.mark.parametrize("B,K,use_nonterm,use_w", [(13, 10, True, True), (256, 1, False, False), (61, 5, True, False)])
@pytest.mark.parametrize("kind", ["none"] + IDS)
def test_ens_q_loss_sq_matches_fp64(kind, B, K, use_nonterm, use_w, A):
    L, lib = _lib()
    loss_weight, grad_scale = 0.8, (0.5 / B if use_w else 1.0)
    d = _ens_inputs(B, K, A, seed=B * 31 + K * 7 + A)
    loss, grad, _, _ = _run_ens(lib, d, kind, loss_weight, use_nonterm, use_w, grad_scale, "sq")
    want = ens_fp64(d, kind, loss_weight, use_nonterm, use_w, grad_scale)
    assert rel_err(loss, want[0]) < 1e-5 and rel_err(grad, want[1]) < 1e-5, (rel_err(loss, want[0]), rel_err(grad, want[1]))
    # the _total variant: loss head + PER-weighted total + TD mix in one launch
    for use_dist, use_off, q_scale in ((True, True, 0.6), (False, False, 1.0), (False, True, 2.0)):
        got = _run_ens(lib, d, kind, loss_weight, use_nonterm, use_w, grad_scale, "total_sq", q_scale, use_dist, use_off)
        want = ens_fp64(d, kind, loss_weight, use_nonterm, use_w, grad_scale, q_scale, use_dist, use_off)
        assert rel_err(got[0], want[0]) < 1e-5 and rel_err(got[1], want[1]) < 1e-5
        assert abs(got[2] - want[2]) <= 1e-5 * abs(want[2]) and rel_err(got[3], want[3]) < 1e-5
        if kind == "none":
            plain = _run_ens(lib, d, kind, loss_weight, use_nonterm, use_w, grad_scale, "total", q_scale, use_dist,
                             use_off)
            assert all(np.array_equal(a, b) for a, b in zip(got, plain))
    if kind == "none":
        plain = _run_ens(lib, d, kind, loss_weight, use_nonterm, use_w, grad_scale, "plain")
        assert np.array_equal(loss, plain[0]) and np.array_equal(grad, plain[1])
    else:
        assert rel_err(loss, ens_fp64(d, "none", loss_weight, use_nonterm, use_w, grad_scale)[0]) > 1e-3


def ids_fp64(q, z, kind, lmbda, eps, rho_lb):
    """IDS scores in fp64 (action_selectors.py:125-176 with the std / sqrt(std) quirk).  q (K, N, A), z (Nq, N, A)."""
    q, z = _h(q.astype(np.float64), kind, True), _h(z.astype(np.float64), kind, True)
    mean, var = q.mean(axis=0), q.std(axis=0, ddof=1)
    std = np.sqrt(var)
    regret = (mean + lmbda * std).max(axis=1, keepdims=True) - (mean - lmbda * std)
    var_z = z.var(axis=0, ddof=1)
    rho = np.maximum(var_z / (eps + var_z.mean(axis=1, keepdims=True)), rho_lb)
    return regret * regret / (np.log(1 + var / rho) + eps)


def ids_inputs(N, K, Nq, A, seed):
    rng = np.random.default_rng(seed)
    off = _offsets(rng, N, A, spread=1.5)
    q = (off[None] + rng.standard_normal((K, N, A)) * rng.uniform(0.05, 0.6, (1, N, A))).astype(np.float32)
    z = (off[None] + rng.standard_normal((Nq, N, A)) * rng.uniform(0.1, 1.0, (1, N, A))).astype(np.float32)
    return q, z


def ids_margin(scores):
    """(second smallest - smallest) / |second smallest| per row: how far a rounding of the scores is from flipping the
    argmin (the kernel's scores hold 1e-4 of fp64)."""
    s = np.sort(scores, axis=1)
    return (s[:, 1] - s[:, 0]) / np.maximum(np.abs(s[:, 1]), 1e-30)


@pytest.mark.parametrize("A", [3, 7, 18, 32])
@pytest.mark.parametrize("N,K,Nq", [(13, 10, 32), (256, 4, 8), (1, 3, 200)])
@pytest.mark.parametrize("kind", ["none"] + IDS)
def test_ids_select_sq_matches_fp64(kind, N, K, Nq, A):
    L, lib = _lib()
    lmbda, eps, rho_lb = 0.1, 1e-10, 0.25
    q, z = ids_inputs(N, K, Nq, A, seed=N * 11 + K + A)
    want = ids_fp64(q, z, kind, lmbda, eps, rho_lb)
    margin = ids_margin(want)
    keep = margin > 1e-3                            # rows whose argmin no fp32 rounding can flip
    assert keep.mean() >= 0.9, "inputs do not separate the IDS scores: %d of %d rows" % (keep.sum(), N)

    def run(entry):
        qd, zd = _t(q), _t(z)
        act = torch.full((N,), -1, dtype=torch.int64, device=DEV)
        sc = torch.full((N, A), float("nan"), device=DEV)
        args = (N, A, K, Nq, qd.data_ptr(), zd.data_ptr(), lmbda, eps, rho_lb, act.data_ptr(), sc.data_ptr(), _stream())
        assert (lib.pb_ids_select(*args) if entry == "plain" else lib.pb_ids_select_sq(*args, KINDS[kind])) == 0
        torch.cuda.synchronize()
        return act.cpu().numpy(), sc.cpu().numpy()

    act, sc = run("sq")
    assert np.array_equal(act[keep], want.argmin(axis=1)[keep])
    assert np.all(np.abs(sc - want) <= 1e-4 * np.abs(want).max(axis=1, keepdims=True) + 1e-30)
    if kind == "none":
        plain = run("plain")
        assert np.array_equal(act, plain[0]) and np.array_equal(sc, plain[1])


# ---- 3. Agent.update at the BASELINE shapes against the oracle ------------------------------------------------------------
def _build_pair(name, squish_id, use_cuda_graph=False, dekink_with=None):
    """test_gpu_config_shapes._build_pair with the config's loss_squish_fn_id set on both sides (the oracle's heads
    get squashed targets: squash_oracle.py)."""
    import test_gpu_config_shapes as cs
    from squash_oracle import squash_oracle_agent
    make, obs_shape, A, B, fs = cs._spec(name)
    orig = cs._spec
    cs._spec = lambda n: (lambda **kw: make(loss_squish_fn_id=squish_id, **kw),) + orig(n)[1:]
    try:
        out = cs._build_pair(name, use_cuda_graph=use_cuda_graph, dekink_with=dekink_with)
    finally:
        cs._spec = orig
    cfg = out[0]
    assert cfg.loss_squish_fn_id == squish_id
    squash_oracle_agent(out[2], squish_id)
    heads = [m for m in (out[1].model.distribution_model, out[1].model.q_function_model) if m is not None]
    assert heads and all(m.squash == KINDS[squish_id] for m in heads)
    assert all(m.squish == squish_id for m in (out[2].model.distribution_model, out[2].model.q_function_model)
               if m is not None)
    return out


@pytest.mark.parametrize("squish_id", IDS)
@pytest.mark.parametrize("name", ["configs0", "configs1", "configs4"])
def test_update_with_squashing_matches_oracle(name, squish_id):
    import test_gpu_config_shapes as cs
    from prism_b200.agents import ops
    make, obs_shape, A, B, fs = cs._spec(name)
    cpu_batch, dev_batch, w = cs._make_batch(obs_shape, A, B, fs, seed=7)
    taus = cs._taus(make(), B, seed=11)
    cfg, agent, oracle, obs_shape, A, B, fs = _build_pair(name, squish_id, dekink_with=(cpu_batch, taus))
    oracle.inject_taus([t.clone() for t in taus])
    out = oracle.update(cpu_batch, w)
    cs._inject(cfg, agent, taus)
    ops.route_counts(reset=True)
    td = agent.update(dev_batch, w.to(DEV))
    torch.cuda.synchronize()
    routes = ops.route_counts()
    cs._compare(agent, oracle, out, td, "%s %s" % (name, squish_id))
    assert ops.fallthrough_count() == 0, routes
    if name in ("configs0", "configs4"):
        assert routes.get("linear:tc_gemm", 0) >= 2 and routes.get("phi_x:tc_gemm", 0) >= 2, routes


@pytest.mark.parametrize("squish_id", IDS)
@pytest.mark.parametrize("name", ["configs0", "configs1"])
def test_graph_update_with_squashing_matches_oracle(name, squish_id):
    import test_gpu_config_shapes as cs
    make, obs_shape, A, B, fs = cs._spec(name)
    probe = (cs._make_batch(obs_shape, A, B, fs, seed=20)[0], cs._taus(make(), B, seed=30))
    cfg, agent, oracle, obs_shape, A, B, fs = _build_pair(name, squish_id, use_cuda_graph=True, dekink_with=probe)
    for it in range(2):
        cpu_batch, dev_batch, w = cs._make_batch(obs_shape, A, B, fs, seed=20 + it)
        taus = cs._taus(cfg, B, seed=30 + it)
        oracle.inject_taus([t.clone() for t in taus])
        out = oracle.update(cpu_batch, w)
        if cfg.use_iqn:
            cs._set_static_taus(cfg, agent, taus)
        td = agent.update(dev_batch, w.to(DEV))
        torch.cuda.synchronize()
        cs._compare(agent, oracle, out, td, "%s %s graph step %d" % (name, squish_id, it))
    assert agent._learn_cuda_graph is not None


@pytest.mark.parametrize("squish_id", IDS)
def test_configs0_squashing_parity_over_consecutive_steps(squish_id):
    import test_gpu_config_shapes as cs
    make, obs_shape, A, B, fs = cs._spec("configs0")
    probe = (cs._make_batch(obs_shape, A, B, fs, seed=40)[0], cs._taus(make(), B, seed=50))
    cfg, agent, oracle, obs_shape, A, B, fs = _build_pair("configs0", squish_id, dekink_with=probe)
    for it in range(3):
        cpu_batch, dev_batch, w = cs._make_batch(obs_shape, A, B, fs, seed=40 + it)
        taus = cs._taus(cfg, B, seed=50 + it)
        oracle.inject_taus([t.clone() for t in taus])
        out = oracle.update(cpu_batch, w)
        cs._inject(cfg, agent, taus)
        td = agent.update(dev_batch, w.to(DEV))
        torch.cuda.synchronize()
        cs._compare(agent, oracle, out, td, "configs0 %s step %d" % (squish_id, it), tol=2e-4)


# ---- 4. LearnerStep and data parallelism ----------------------------------------------------------------------------------
CAP, B_STEP, OBS, A_STEP, N_NEW, ITERS = 256, 32, (10, 10, 6), 4, 4, 6


def _step_script():
    from oracle.gen_golden import make_script
    S = make_script(5, n_streams=4, n_steps=200 + N_NEW * ITERS, obs_shape=OBS, p_done=0.05, p_trunc=0.03,
                    n_actions=A_STEP)
    succ = np.where(S["trunc"][:, None], S["final_obs"], S["next_obs"])
    return S, succ


def _step_agent(squish_id):
    import prism_b200
    S, succ = _step_script()
    cfg = prism_b200.minatar_dqn_per_config(device=DEV, experience_replay_capacity=CAP, batch_size=B_STEP,
                                            per_sampling="stratified", replay_max_streams=4, replay_staging_rows=64,
                                            use_cuda_graph=False, loss_squish_fn_id=squish_id)
    torch.manual_seed(0)
    agent = prism_b200.build_agent(cfg, OBS, A_STEP)
    buf = prism_b200.build_exp_buffer(cfg)
    buf.extend_batch(S["stream"][:200], S["obs"][:200].reshape((-1,) + OBS), S["action"][:200], S["reward"][:200],
                     S["done"][:200], S["trunc"][:200], succ[:200].reshape((-1,) + OBS))
    buf._flush()
    assert agent.model.q_function_model.squash == KINDS[squish_id]
    return agent, buf, S, succ


def _new_steps(S, succ, i):
    sl = slice(200 + i * N_NEW, 200 + (i + 1) * N_NEW)
    return (S["stream"][sl], S["obs"][sl].reshape((-1,) + OBS), S["action"][sl], S["reward"][sl], S["done"][sl],
            S["trunc"][sl], succ[sl].reshape((-1,) + OBS))


def _state(agent, buf, losses):
    tree = buf.buffer._sampler
    return losses, agent.optimizer.arena.clone(), tree.sum.clone(), tree.min.clone()


def _step_run(squish_id, us, use_graph, prefetch):
    from prism_b200.learner_step import LearnerStep
    agent, buf, S, succ = _step_agent(squish_id)
    step = LearnerStep(buf, agent, batch_size=B_STEP, use_cuda_graph=use_graph, prefetch=prefetch)
    losses = [float(step.step(u=torch.from_numpy(us[i].copy()), ingest=_new_steps(S, succ, i))) for i in range(ITERS)]
    torch.cuda.synchronize()
    if use_graph:
        assert step.launches_per_step > 0
    return _state(agent, buf, losses)


def _eager_run(squish_id, us):
    agent, buf, S, succ = _step_agent(squish_id)
    losses = []
    for i in range(ITERS):
        buf.inject_uniforms(torch.from_numpy(us[i]).to(DEV))
        batch, info = buf.sample(return_info=True)
        td = agent.update(batch, info["_weight"])
        buf.update_priority(info["index"], td.abs())
        losses.append(float(agent._static_total_loss.detach()))
        buf.extend_batch(*_new_steps(S, succ, i))
        buf._flush()
    torch.cuda.synchronize()
    return _state(agent, buf, losses)


def _same(a, b, tol=1e-5):
    assert np.allclose(a[0], b[0], rtol=tol, atol=1e-7), (a[0], b[0])
    assert rel_err(a[1].cpu().numpy(), b[1].cpu().numpy()) < tol
    assert np.allclose(a[2].cpu().numpy(), b[2].cpu().numpy(), rtol=1e-4, atol=1e-7)
    assert np.allclose(a[3].cpu().numpy(), b[3].cpu().numpy(), rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("squish_id", IDS)
def test_learner_step_with_squashing_equals_the_eager_loop(squish_id):
    """The one-graph step with PER and the fused ingest against sample -> update -> write-back -> push on the same host
    uniforms; with prefetch (host uniforms then drive the NEXT batch) the graph against the step without a graph."""
    us = np.random.default_rng(21).random((ITERS, B_STEP))
    eager = _eager_run(squish_id, us)
    _same(_step_run(squish_id, us, True, False), eager)
    _same(_step_run(squish_id, us, True, True), _step_run(squish_id, us, False, True))
    assert not np.allclose(eager[0], _eager_run("none", us)[0], rtol=1e-3), "squashing changed nothing"


def _run(cmd):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=540)
    assert p.returncode == 0, p.stdout[-3000:]


@pytest.mark.parametrize("squish_id", IDS)
def test_two_ranks_with_squashing_equal_one_rank_on_the_union_buffer(tmp_path, squish_id):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = os.path.join(HERE, "mp_worker_dp_squash.py")
    out2, out1 = str(tmp_path / "dp2"), str(tmp_path / "one")
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
          "127.0.0.1", "--master-port", str(29760 + KINDS[squish_id]), worker, "--out", out2, "--squish", squish_id])
    _run([sys.executable, worker, "--out", out1, "--union", "2", "--squish", squish_id])
    one = torch.load(out1 + ".rank0", weights_only=False)
    r0, r1 = (torch.load(out2 + ".rank%d" % r, weights_only=False) for r in (0, 1))
    assert r0["squash"] == r1["squash"] == one["squash"] == KINDS[squish_id]
    assert torch.equal(r0["arena"], r1["arena"]), "replicas diverged"
    B_pad, B_global = r0["B_pad"], one["B_pad"]
    both = (np.asarray(r0["losses"]) + np.asarray(r1["losses"])) * (B_pad / B_global)
    assert np.allclose(both, one["losses"], rtol=2e-5, atol=1e-7), (r0["losses"], r1["losses"], one["losses"])
    assert rel_err(r0["arena"].numpy(), one["arena"].numpy()) < 2e-5
    leaves = torch.cat([r0["leaves"], r1["leaves"]])
    assert np.allclose(leaves.numpy(), one["leaves"].numpy(), rtol=1e-4, atol=1e-7)


# ---- 5. acting ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("squish_id", IDS)
def test_acting_graph_with_unsquash_equals_eager(squish_id):
    """Agent.forward as one CUDA graph (embedding -> IQN(Nq) -> K heads -> IDS kernel reading through h^-1) picks the
    actions of the eager path, and those of the oracle's IDS on the same q and z."""
    import prism_b200
    from squash_oracle import squash_ids_actions
    obs_shape, A, N = (10, 10, 4), 3, 14
    cfg = prism_b200.minatar_ids_iqn_config(device=DEV, experience_replay_capacity=64, batch_size=8,
                                            iqn_quantile_samples_per_action=16, iqn_quantile_model_feature_dim=32,
                                            ids_q_head_feature_dim=16, ids_n_q_heads=3, use_cuda_graph=True,
                                            replay_max_streams=2, replay_staging_rows=8, loss_squish_fn_id=squish_id)
    torch.manual_seed(0)
    agent = prism_b200.build_agent(cfg, obs_shape, A)
    assert agent.action_selector.squash == KINDS[squish_id]
    iqn = agent.model.distribution_model
    g = torch.Generator().manual_seed(3)
    for trial in range(3):
        obs = (torch.rand((N,) + obs_shape, generator=g) < 0.15).float()
        iqn._rng_state()[1:3] = torch.tensor([100 + trial, 0], device=DEV)
        got = agent.forward(obs)                                   # graph (captured on the first trial)
        agent.use_cuda_graph, agent.model.use_cuda_graph = False, False
        iqn._rng_state()[1:3] = torch.tensor([100 + trial, 0], device=DEV)
        want = agent.forward(obs)                                  # eager
        iqn._rng_state()[1:3] = torch.tensor([100 + trial, 0], device=DEV)
        with torch.no_grad():
            q, z = agent.model(obs.to(DEV), for_action=True)
        agent.use_cuda_graph = agent.model.use_cuda_graph = True
        assert torch.equal(got.cpu(), want.cpu())
        ref, scores = squash_ids_actions(q.cpu(), z.cpu(), squish_id, cfg.ids_lambda, cfg.ids_epsilon,
                                         cfg.ids_rho_lower_bound, return_scores=True)
        keep = torch.from_numpy(ids_margin(scores.double().numpy()) > 1e-3)
        assert keep.float().mean() >= 0.5
        assert torch.equal(want.cpu()[keep], ref[keep])
    assert len(agent._acting_graphs) == 1
