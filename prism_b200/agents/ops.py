"""torch.autograd bridges to the fused CUDA kernels of libprism_b200 (csrc/agent_kernels.cu).

Every function here launches hand-written sm_100a kernels through the C ABI on the current
torch stream; inputs must be CUDA tensors (no CPU path -- the CPU restatement lives in
oracle/ and is only ever used by tests and the bench's cpu_baseline leg).
"""
import collections

import torch

from .. import _lib

# How every dense layer / LayerNorm call was executed, by route name.  "fallthrough:*" routes leave this library
# (ATen / cuBLAS); the bench line prints the counter and the config-shape parity tests assert on it.
ROUTES = collections.Counter()


def route_counts(reset=False):
    out = dict(ROUTES)
    if reset:
        ROUTES.clear()
    return out


def fallthrough_count():
    return sum(v for k, v in ROUTES.items() if k.startswith("fallthrough"))


def _c(t, dtype=torch.float32):
    if t.dtype != dtype:
        t = t.to(dtype)
    return t if t.is_contiguous() else t.contiguous()


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def cos_basis(tau, n_basis):
    """cos(pi * i * tau), i = 1..n_basis  ->  (rows, n_basis).  tau carries no gradient
    (prism/agents/models/iqn_model.py:89-92)."""
    _lib.require_cuda(tau, "tau")
    tau = _c(tau.detach()).view(-1)
    out = torch.empty(tau.numel(), n_basis, dtype=torch.float32, device=tau.device)
    _lib.check(_lib.load().pb_iqn_cos_basis(tau.numel(), int(n_basis), tau.data_ptr(), out.data_ptr(), _stream(tau)),
               "pb_iqn_cos_basis")
    return out


def draw_cos_basis(n_rows, n_basis, rng):
    """tau ~ U[0,1) drawn on the device + its cosine basis, one launch (pb_iqn_draw_cos_basis).  ``rng``: int64[4]
    device tensor {seed, call number, ticket, -}.  Returns (tau (n_rows, 1), basis (n_rows, n_basis))."""
    _lib.require_cuda(rng, "rng")
    tau = torch.empty(n_rows, 1, dtype=torch.float32, device=rng.device)
    out = torch.empty(n_rows, n_basis, dtype=torch.float32, device=rng.device)
    _lib.check(_lib.load().pb_iqn_draw_cos_basis(int(n_rows), int(n_basis), rng.data_ptr(), tau.data_ptr(), out.data_ptr(),
                                                 _stream(rng)), "pb_iqn_draw_cos_basis")
    return tau, out


def sum_leading(x):
    """x (K, ...) -> sum over the leading axis, fixed order (pb_sum_heads)."""
    K = x.shape[0]
    n = x[0].numel()
    if K == 1:
        return x[0]
    if n % 4 != 0 or not x.is_contiguous():
        ROUTES["fallthrough:sum"] += 1
        return x.sum(dim=0)
    out = torch.empty(x.shape[1:], dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().pb_sum_heads(int(K), int(n), x.data_ptr(), out.data_ptr(), _stream(x)), "pb_sum_heads")
    return out


class _QuantileHuberLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z_cur, tau, z_next_online, z_next_target, action, ret, gdn, B, T, Tp, kappa, loss_weight):
        _lib.require_cuda(z_cur, "z_cur")
        A = z_cur.shape[-1]
        z_cur_c, tau_c = _c(z_cur), _c(tau).view(-1)
        zo, zt = _c(z_next_online), _c(z_next_target)
        action_c, ret_c, gdn_c = _c(action, torch.int64).view(-1), _c(ret).view(-1), _c(gdn).view(-1)
        loss = torch.empty(B, dtype=torch.float32, device=z_cur.device)
        grad = torch.empty_like(z_cur_c)
        _lib.check(_lib.load().pb_iqn_qh_loss(
            B, T, Tp, A, z_cur_c.data_ptr(), tau_c.data_ptr(), zo.data_ptr(), zt.data_ptr(), action_c.data_ptr(),
            ret_c.data_ptr(), gdn_c.data_ptr(), None, float(kappa), float(loss_weight), None, 1.0, loss.data_ptr(),
            grad.data_ptr(), _stream(z_cur)), "pb_iqn_qh_loss")
        ctx.save_for_backward(grad)
        ctx.dims = (B, T, A)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        (grad,) = ctx.saved_tensors
        B, T, A = ctx.dims
        # rows are quantile-major (r = i*B + b): scale row b of every quantile by dL/dloss_b
        gz = (grad.view(T, B, A) * grad_loss.view(1, B, 1)).view(T * B, A)
        return (gz,) + (None,) * 11


def quantile_huber_loss(z_cur, tau, z_next_online, z_next_target, action, ret, gdn, n_cur, n_next, kappa=1.0,
                        loss_weight=1.0):
    """IQN loss per batch row, (B,) -- target build, pairwise quantile-Huber and its gradient in
    one kernel (prism/agents/models/iqn_model.py:110-201)."""
    B = action.numel()
    return _QuantileHuberLoss.apply(z_cur, tau, z_next_online, z_next_target, action, ret, gdn, B, int(n_cur),
                                    int(n_next), kappa, loss_weight)


class _EnsembleQLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q_cur, q_next_online, q_next_target, action, ret, gdn, loss_weight):
        _lib.require_cuda(q_cur, "q_cur")
        K, B, A = q_cur.shape
        qc, qo, qt = _c(q_cur), _c(q_next_online), _c(q_next_target)
        action_c, ret_c, gdn_c = _c(action, torch.int64).view(-1), _c(ret).view(-1), _c(gdn).view(-1)
        loss = torch.empty(B, dtype=torch.float32, device=q_cur.device)
        grad = torch.empty_like(qc)
        _lib.check(_lib.load().pb_ens_q_loss(
            B, A, K, qc.data_ptr(), qo.data_ptr(), qt.data_ptr(), action_c.data_ptr(), ret_c.data_ptr(),
            gdn_c.data_ptr(), None, float(loss_weight), None, 1.0, loss.data_ptr(), grad.data_ptr(), _stream(q_cur)),
            "pb_ens_q_loss")
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        (grad,) = ctx.saved_tensors
        return (grad * grad_loss.view(1, -1, 1),) + (None,) * 6


def ensemble_q_loss(q_cur, q_next_online, q_next_target, action, ret, gdn, loss_weight=1.0):
    """Mean-over-heads MSE with per-head double-Q targets, (B,).  Tables are head-major (K, B, A)
    (prism/agents/models/q_ensemble.py:62-84)."""
    return _EnsembleQLoss.apply(q_cur, q_next_online, q_next_target, action, ret, gdn, loss_weight)


def ids_select(q_kna, z_qna, lmbda, eps, rho_lower_bound, return_scores=False):
    """IDS information-ratio argmin (prism/agents/action_selectors.py:125-176).
    q_kna: (K, N, A) head-major ensemble values; z_qna: (Nq, N, A)."""
    _lib.require_cuda(q_kna, "q")
    K, N, A = q_kna.shape
    Nq = z_qna.shape[0]
    q, z = _c(q_kna), _c(z_qna)
    act = torch.empty(N, dtype=torch.int64, device=q.device)
    scores = torch.empty(N, A, dtype=torch.float32, device=q.device) if return_scores else None
    _lib.check(_lib.load().pb_ids_select(N, A, K, Nq, q.data_ptr(), z.data_ptr(), float(lmbda), float(eps),
                                         float(rho_lower_bound), act.data_ptr(), _lib.ptr(scores), _stream(q)),
               "pb_ids_select")
    return (act, scores) if return_scores else act


def greedy_select(q_kna):
    _lib.require_cuda(q_kna, "q")
    K, N, A = q_kna.shape
    q = _c(q_kna)
    act = torch.empty(N, dtype=torch.int64, device=q.device)
    _lib.check(_lib.load().pb_greedy_select(N, A, K, q.data_ptr(), act.data_ptr(), _stream(q)), "pb_greedy_select")
    return act


class _LossCombine(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dist, q, w):
        ref = dist if dist is not None else q
        _lib.require_cuda(ref, "loss")
        B = ref.numel()
        total = torch.empty((), dtype=torch.float32, device=ref.device)
        td = torch.empty(B, dtype=torch.float32, device=ref.device)
        dist_c = None if dist is None else _c(dist)
        q_c = None if q is None else _c(q)
        w_c = None if w is None else _c(w).view(-1)
        _lib.check(_lib.load().pb_loss_combine(B, _lib.ptr(dist_c), _lib.ptr(q_c), _lib.ptr(w_c), 1.0, None,
                                               total.data_ptr(), td.data_ptr(), _stream(ref)), "pb_loss_combine")
        ctx.B = B
        ctx.has = (dist is not None, q is not None)
        ctx.save_for_backward(w_c if w_c is not None else torch.empty(0, device=ref.device))
        ctx.mark_non_differentiable(td)
        return total, td

    @staticmethod
    def backward(ctx, g_total, _g_td):
        (w,) = ctx.saved_tensors
        row = (w / ctx.B) * g_total if w.numel() else torch.full((ctx.B,), 1.0 / ctx.B, device=g_total.device) * g_total
        return (row if ctx.has[0] else None, row if ctx.has[1] else None, None)


def loss_combine(dist_loss, q_loss, per_weights):
    """total = mean(dist*w) + mean(q*w); td = 0.5 dist + 0.5 q | dist | |q|
    (prism/agents/agent.py:58-64, prism/agents/models/composite_model.py:135-142)."""
    return _LossCombine.apply(dist_loss, q_loss, per_weights)


# LearnerStep.enable_trace() points this at its timeline-mark function (measurement runs only); None otherwise
TRACE_MARK = None


def trace_mark(name):
    if TRACE_MARK is not None:
        TRACE_MARK(name)
_SIDE_STREAMS = {}


def fork_stream(device, key="bwd"):
    """A cached side stream (a parallel branch under CUDA-graph capture)."""
    device = torch.device(device)
    s = _SIDE_STREAMS.get((device, key))
    if s is None:
        s = _SIDE_STREAMS[(device, key)] = torch.cuda.Stream(device=device)
    return s


# Weight-gradient branches and their joins.  A layer's dW (and db) feed nothing but the optimizer, so inside the captured
# learner step the branch that computes them does not have to rejoin the backward pass before the next layer starts:
# LearnerStep defers the joins to just before the optimizer step (mode 2).  That is only sound when autograd hands the
# very tensor the branch writes to the parameter as its .grad (no accumulation kernel on the main stream), so the step's
# first warm-up iteration runs in mode 1: joins stay where they are, the gradient addresses are recorded, and
# LearnerStep checks them against the parameters' .grad before it turns mode 2 on.  Mode 0 (default): join in place.
_JOINS = {"mode": 0, "streams": [], "ptrs": []}


def defer_joins(mode):
    _JOINS["mode"], _JOINS["streams"], _JOINS["ptrs"] = int(mode), [], []


def finish_deferred(device):
    """Join every deferred branch into the current stream; returns the recorded gradient addresses."""
    cur = torch.cuda.current_stream(device)
    seen = set()
    for s in _JOINS["streams"]:
        if s.cuda_stream not in seen and s.cuda_stream != cur.cuda_stream:
            seen.add(s.cuda_stream)
            cur.wait_stream(s)
    ptrs = _JOINS["ptrs"]
    defer_joins(0)
    return ptrs


def _join_or_defer(side, device, *grads):
    mode = _JOINS["mode"]
    if mode:
        _JOINS["ptrs"].extend(g.data_ptr() for g in grads if g is not None)     # addresses: a reference would block the steal
    if mode == 2:
        _JOINS["streams"].append(side)
    else:
        torch.cuda.current_stream(device).wait_stream(side)


class _Linear(torch.autograd.Function):
    """Y = act(X W^T + b), batched over heads.  X: (M, J) shared or (K, M, J); W: (K, N, J); b: (K, N)."""

    @staticmethod
    def forward(ctx, x, w, b, act):
        _lib.require_cuda(x, "x")
        K, N, J = w.shape
        shared = x.dim() == 2
        M = x.shape[-2]
        xc, wc, bc = _c(x), _c(w), (None if b is None else _c(b))
        y = torch.empty(K, M, N, dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().pb_linear_fwd(K, M, N, J, xc.data_ptr(), 0 if shared else M * J, wc.data_ptr(),
                                             _lib.ptr(bc), int(act), y.data_ptr(), _stream(x)), "pb_linear_fwd")
        ctx.act, ctx.shared, ctx.dims, ctx.has_bias = int(act), shared, (K, M, N, J), b is not None
        ctx.save_for_backward(xc, wc, y if act else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        xc, wc, y = ctx.saved_tensors
        K, M, N, J = ctx.dims
        dy = _c(dy)
        lib, stream = _lib.load(), _stream(dy)
        mask = _lib.ptr(y) if ctx.act else None
        dx = dw = db = None
        want_dx = ctx.needs_input_grad[0]
        want_dw = ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2])
        if want_dx:
            dx = torch.empty((M, J) if ctx.shared else (K, M, J), dtype=torch.float32, device=dy.device)
        if want_dw:
            dw = torch.empty(K, N, J, dtype=torch.float32, device=dy.device)
            db = torch.empty(K, N, dtype=torch.float32, device=dy.device) if ctx.has_bias else None
        # the two gradient GEMMs are independent and each is too small to fill the chip: the weight gradient goes to a
        # second stream (a parallel branch under CUDA-graph capture) and is joined before the function returns
        side = fork_stream(dy.device) if (want_dx and want_dw) else None
        if want_dw:
            if side is not None:
                cur = torch.cuda.current_stream(dy.device)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    _lib.check(lib.pb_linear_bwd_weight(K, M, N, J, dy.data_ptr(), mask, xc.data_ptr(),
                                                        0 if ctx.shared else M * J, dw.data_ptr(), _lib.ptr(db),
                                                        side.cuda_stream), "pb_linear_bwd_weight")
            else:
                _lib.check(lib.pb_linear_bwd_weight(K, M, N, J, dy.data_ptr(), mask, xc.data_ptr(),
                                                    0 if ctx.shared else M * J, dw.data_ptr(), _lib.ptr(db), stream),
                           "pb_linear_bwd_weight")
        if want_dx:
            _lib.check(lib.pb_linear_bwd_input(K, M, N, J, dy.data_ptr(), mask, wc.data_ptr(), int(ctx.shared),
                                               dx.data_ptr(), stream), "pb_linear_bwd_input")
        if side is not None:
            _join_or_defer(side, dy.device, dw, db)
        if TRACE_MARK is not None:
            TRACE_MARK("bwd:linear K%d M%d N%d J%d" % (K, M, N, J))
        return dx, dw, db, None


# Dispatch of a dense layer (DESIGN.md sections 4 and 4.1):
#   * >= TC_MIN_FLOPS and >= TC_MIN_ROWS rows: tcgen05 3xTF32 GEMM (csrc/tc_gemm.cu), forward and both gradients;
#   * up to FUSED_LINEAR_MAX_ROWS rows: fp32 FFMA cluster split-K kernel (csrc/linear.cu) -- learner-batch-sized Q heads;
#   * anything else (e.g. the 18-action output layer of the (T*B)-row IQN head, whose rows are not 16-byte
#     aligned): library SGEMM.
FUSED_LINEAR_MAX_ROWS = 512
NARROW_OUT, NARROW_MAX_ROWS = 32, 4096


_TC_WORKSPACE = {}
# partial tiles: at most 3 per CTA of 128 x 256 floats (two stream-K cut tiles + the running sum of a tile accumulated
# in chunks) -> 3 * 148 * 128 * 256 floats (58 MB).  One workspace
# PER STREAM: GEMMs on parallel graph branches (bootstrap passes, weight gradients) may overlap at their tails, and a
# GEMM's fix-up must never read partial tiles of another one.
TC_WORKSPACE_FLOATS = 15 * 1024 * 1024
TC_SPLIT_MODE = 0                           # 0: hi = raw fp32 word (hardware reads its top 19 bits); 1: cvt.rna hi


def _tc_workspace(device, stream):
    key = (device, stream)
    ws = _TC_WORKSPACE.get(key)
    if ws is None:
        ws = _TC_WORKSPACE[key] = torch.empty(TC_WORKSPACE_FLOATS, dtype=torch.float32, device=device)
    return ws


def tc_gemm(out, a, a_major, lda, a_bs, b, b_major, ldb, b_bs, batch, M, N, K, bias=None, bias_bs=0, act=0,
            kbatches=1, ldc=None, c_bs=None, mul=None):
    """out[b] (M x N) = act(A[b] . B[b]^T + bias[b]) on the tensor cores (pb_tc_gemm, 3xTF32).  See
    include/prism_b200.h for the operand conventions (major 1 = the transposed view)."""
    _lib.require_cuda(out, "out")
    stream = _stream(out)
    ws = _tc_workspace(out.device, stream)
    _lib.check(_lib.load().pb_tc_gemm(int(batch), int(kbatches), int(M), int(N), int(K),
                                      a.data_ptr(), int(a_major), int(lda), int(a_bs),
                                      b.data_ptr(), int(b_major), int(ldb), int(b_bs),
                                      _lib.ptr(bias), int(bias_bs), int(act),
                                      _lib.ptr(mul), 0 if mul is None else int(mul.shape[0]),
                                      0 if mul is None else int(mul.stride(0)),
                                      out.data_ptr(), int(N if ldc is None else ldc), int(M * N if c_bs is None else c_bs),
                                      ws.data_ptr(), ws.numel(), int(TC_SPLIT_MODE), stream), "pb_tc_gemm")
    return out


class _LinearTC(torch.autograd.Function):
    """Y = act(X W^T + b) with forward, input-gradient and weight-gradient GEMMs all on the tensor cores
    (tcgen05 3xTF32, csrc/tc_gemm.cu).  X: (M, J) shared by the heads or (K, M, J); W: (K, N, J); b: (K, N)."""

    @staticmethod
    def forward(ctx, x, w, b, act):
        K, N, J = w.shape
        shared = x.dim() == 2
        M = x.shape[-2]
        xc, wc, bc = _c(x), _c(w), (None if b is None else _c(b))
        y = torch.empty(K, M, N, dtype=torch.float32, device=x.device)
        tc_gemm(y, xc, 0, J, 0 if shared else M * J, wc, 0, J, N * J, K, M, N, J, bias=bc, bias_bs=N, act=int(act))
        ctx.act, ctx.shared, ctx.has_bias, ctx.dims = int(act), shared, b is not None, (K, M, N, J)
        ctx.save_for_backward(xc, wc, y if act else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        xc, wc, y = ctx.saved_tensors
        K, M, N, J = ctx.dims
        dy = _c(dy)
        lib = _lib.load()
        want_db = ctx.has_bias and ctx.needs_input_grad[2]
        dz, db = dy, None
        if ctx.act or want_db:
            # ReLU mask + bias gradient in one pass (pb_relu_bwd_bias) instead of compare + multiply + sum(dim)
            strips = lib.pb_relu_bwd_bias_strips(M)
            partials = torch.empty(K * strips * N, dtype=torch.float32, device=dy.device)
            dz = torch.empty_like(dy) if ctx.act else dy
            db = torch.empty(K, N, dtype=torch.float32, device=dy.device) if want_db else None
            _lib.check(lib.pb_relu_bwd_bias(K, M, N, dy.data_ptr(), _lib.ptr(y) if ctx.act else None,
                                            dz.data_ptr() if ctx.act else None, _lib.ptr(db), partials.data_ptr(),
                                            _stream(dy)), "pb_relu_bwd_bias")
        dx = dw = None
        if ctx.needs_input_grad[0]:
            # dX (M x J) = dZ (M x N) . W (N x J): B operand is W read as its transpose (b_major 1)
            if ctx.shared:
                dx = torch.empty(M, J, dtype=torch.float32, device=dz.device)
                tc_gemm(dx, dz, 0, N, M * N, wc, 1, J, N * J, 1, M, J, N, kbatches=K)
            else:
                dx = torch.empty(K, M, J, dtype=torch.float32, device=dz.device)
                tc_gemm(dx, dz, 0, N, M * N, wc, 1, J, N * J, K, M, J, N)
        if ctx.needs_input_grad[1]:
            # dW (N x J) = dZ^T (N x M) . X (M x J): both operands read as transposes
            dw = torch.empty(K, N, J, dtype=torch.float32, device=dz.device)
            tc_gemm(dw, dz, 1, N, M * N, xc, 1, J, 0 if ctx.shared else M * J, K, N, J, M)
        return dx, dw, db, None


class _NarrowLinear(torch.autograd.Function):
    """y = x W^T + b for a handful of outputs (the n_actions-wide layers of the IQN head and of the K ensemble heads):
    one streaming pass forward, one backward (csrc/narrow.cu) instead of library SGEMMs with 64-wide tiles.
    x: (M, J) shared by the heads or (K, M, J); W: (K, N, J); b: (K, N) or None -> (K, M, N)."""

    @staticmethod
    def forward(ctx, x, w, b):
        K, N, J = w.shape
        shared = x.dim() == 2
        M = x.shape[-2]
        xc, wc, bc = _c(x), _c(w), (None if b is None else _c(b))
        y = torch.empty(K, M, N, dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().pb_narrow_linear_fwd(K, M, N, J, xc.data_ptr(), 0 if shared else M * J, wc.data_ptr(),
                                                    _lib.ptr(bc), y.data_ptr(), _stream(x)), "pb_narrow_linear_fwd")
        ctx.save_for_backward(xc, wc)
        ctx.has_bias, ctx.shared = b is not None, shared
        return y

    @staticmethod
    def backward(ctx, dy):
        xc, wc = ctx.saved_tensors
        K, N, J = wc.shape
        M = xc.shape[-2]
        dy = _c(dy)
        lib = _lib.load()
        want_dx, want_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        want_db = ctx.has_bias and ctx.needs_input_grad[2]
        dx = torch.empty(K, M, J, dtype=torch.float32, device=dy.device) if want_dx else None
        dw = torch.empty_like(wc) if want_dw else None
        db = torch.empty(K, N, dtype=torch.float32, device=dy.device) if want_db else None
        partials = None
        if want_dw or want_db:
            partials = torch.empty(K * lib.pb_narrow_linear_bwd_blocks(M) * (N * J + N), dtype=torch.float32, device=dy.device)
        # inside the learner step graph the dW / db reduction goes to the weight-gradient branch (see _JOINS)
        split = partials is not None and want_dx and _JOINS["mode"]
        _lib.check(lib.pb_narrow_linear_bwd(K, M, N, J, xc.data_ptr(), 0 if ctx.shared else M * J, wc.data_ptr(), dy.data_ptr(),
                                            _lib.ptr(dx), None if split else _lib.ptr(dw), None if split else _lib.ptr(db),
                                            _lib.ptr(partials), _stream(dy)), "pb_narrow_linear_bwd")
        if split:
            side = fork_stream(dy.device)
            side.wait_stream(torch.cuda.current_stream(dy.device))
            with torch.cuda.stream(side):
                _lib.check(lib.pb_narrow_linear_bwd_reduce(K, M, N, J, partials.data_ptr(), _lib.ptr(dw), _lib.ptr(db),
                                                           side.cuda_stream), "pb_narrow_linear_bwd_reduce")
            _join_or_defer(side, dy.device, dw, db)
        if want_dx and ctx.shared:
            dx = sum_leading(dx)                                   # the heads share their input
        return dx, dw, db


NARROW_MIN_ROWS = 32


def _narrow_eligible(x, weight):
    """weight: (N, J) or (K, N, J)."""
    N, J = weight.shape[-2], weight.shape[-1]
    return (x.is_cuda and x.dtype == torch.float32 and x.shape[-2] >= NARROW_MIN_ROWS
            and _lib.load().pb_narrow_linear_supported(x.shape[-2], N, J) == 1)


TC_MIN_ROWS = 256              # an M = 128 tile needs rows to fill it
TC_MIN_FLOPS = 2.0e8           # below this a layer is launch-bound and stays on the fused SIMT kernel / library


def _tc_eligible(x, M, Kh, N, J):
    return (x.is_cuda and (J % 4) == 0 and (N % 4) == 0 and M >= TC_MIN_ROWS
            and 2.0 * M * Kh * N * J >= TC_MIN_FLOPS)


class _PhiTimesX(torch.autograd.Function):
    """h[q*B + b, :] = relu(basis[q*B + b, :] W^T + bias) * x[b, :]   (iqn_model.py:70-71, 89-93).

    Forward: the broadcast product is fused into the tensor-core GEMM's epilogue, so the (n*B, F) tensor phi is
    only materialised when a gradient is needed (a second pass of the K = 64 GEMM is cheaper than an element-wise
    kernel reading and writing (n*B, F)).  Backward: one fused element-wise pass (pb_iqn_phi_bwd) + the
    weight-gradient GEMM."""

    @staticmethod
    def forward(ctx, basis, w, b, x):
        M, J = basis.shape
        F_ = w.shape[0]
        B = x.shape[0]
        basis_c, wc, bc, xc = _c(basis), _c(w), _c(b), _c(x)
        h = torch.empty(M, F_, dtype=torch.float32, device=x.device)
        tc_gemm(h, basis_c, 0, J, 0, wc, 0, J, 0, 1, M, F_, J, bias=bc, bias_bs=0, act=1, mul=xc)
        if any(ctx.needs_input_grad[1:]):
            phi = torch.empty(M, F_, dtype=torch.float32, device=x.device)
            tc_gemm(phi, basis_c, 0, J, 0, wc, 0, J, 0, 1, M, F_, J, bias=bc, bias_bs=0, act=1)
            ctx.save_for_backward(basis_c, phi, xc)
            ctx.dims = (M, J, F_, B)
        return h

    @staticmethod
    def backward(ctx, dh):
        basis_c, phi, xc = ctx.saved_tensors
        M, J, F_, B = ctx.dims
        n = M // B
        dh = _c(dh)
        dpre = torch.empty_like(phi)
        dx = torch.empty_like(xc) if ctx.needs_input_grad[3] else None
        dbp = torch.empty_like(xc)
        _lib.check(_lib.load().pb_iqn_phi_bwd(n, B, F_, dh.data_ptr(), phi.data_ptr(), xc.data_ptr(), dpre.data_ptr(),
                                              _lib.ptr(dx), dbp.data_ptr(), _stream(dh)), "pb_iqn_phi_bwd")
        dw = None
        if ctx.needs_input_grad[1]:
            dw = torch.empty(F_, J, dtype=torch.float32, device=dh.device)
            # dW (F x J) = dpre^T (F x M) . basis (M x J): both operands read as transposes
            tc_gemm(dw, dpre, 1, F_, 0, basis_c, 1, J, 0, 1, F_, J, M)
        db = sum_leading(dbp) if ctx.needs_input_grad[2] else None
        return None, dw, db, dx


def phi_times_x(phi_seq, basis, x, n):
    """IQN quantile embedding times the state embedding: (n*B, n_basis), (B, F) -> (n*B, F)."""
    import torch.nn as nn
    lin = phi_seq[0]
    M, J = basis.shape
    F_ = lin.weight.shape[0]
    if (len(phi_seq) == 2 and isinstance(lin, nn.Linear) and isinstance(phi_seq[1], nn.ReLU) and lin.bias is not None
            and x.dim() == 2 and x.shape[1] == F_ and (F_ % 4) == 0 and _tc_eligible(x, M, 1, F_, J)):
        ROUTES["phi_x:tc_gemm"] += 1
        return _PhiTimesX.apply(basis, lin.weight, lin.bias, x)
    ROUTES["fallthrough:phi_x_mul"] += 1                      # small layers (the reference-golden shapes): ATen broadcast multiply
    phi = run_sequential(phi_seq, basis)
    return (phi.view(n, x.shape[0], -1) * x.unsqueeze(0)).view(n * x.shape[0], -1)


def linear_heads(x, w, b, relu=False):
    """Stacked-head dense layer: x (M, J) shared by all heads or (K, M, J); w (K, N, J); b (K, N) -> (K, M, N)."""
    M, (Kh, N, J) = x.shape[-2], w.shape
    if _tc_eligible(x, M, Kh, N, J):
        ROUTES["linear:tc_gemm"] += 1
        return _LinearTC.apply(x, w, b, 1 if relu else 0)
    if not relu and N <= NARROW_OUT and _narrow_eligible(x, w):
        ROUTES["linear:narrow"] += 1
        return _NarrowLinear.apply(x, w, b)
    if x.shape[-2] > FUSED_LINEAR_MAX_ROWS:
        ROUTES["fallthrough:baddbmm"] += 1
        xe = x.unsqueeze(0).expand(w.shape[0], -1, -1) if x.dim() == 2 else x
        y = torch.baddbmm(b.unsqueeze(1), xe, w.transpose(1, 2)) if b is not None else torch.bmm(xe, w.transpose(1, 2))
        return torch.relu(y) if relu else y
    ROUTES["linear:ffma"] += 1
    return _Linear.apply(x, w, b, 1 if relu else 0)


def linear(x, weight, bias, relu=False):
    """nn.Linear (+ optional fused ReLU) on a 2-D input through the fused kernel."""
    # narrow output layers (a handful of actions) of a few thousand rows stay on the fused FFMA kernel: the library picks
    # 64-wide tiles for them (25 us for the 3 x 256 weight gradient of configs[0])
    if not relu and x.dim() == 2 and weight.shape[0] <= NARROW_OUT and _narrow_eligible(x, weight):
        ROUTES["linear:narrow"] += 1
        return _NarrowLinear.apply(x, weight.unsqueeze(0), None if bias is None else bias.unsqueeze(0)).squeeze(0)
    narrow = weight.shape[0] <= NARROW_OUT and x.shape[0] <= NARROW_MAX_ROWS
    if x.shape[0] > FUSED_LINEAR_MAX_ROWS and not narrow:
        if _tc_eligible(x, x.shape[0], 1, *weight.shape):
            ROUTES["linear:tc_gemm"] += 1
            b = None if bias is None else bias.unsqueeze(0)
            return _LinearTC.apply(x, weight.unsqueeze(0), b, 1 if relu else 0).squeeze(0)
        ROUTES["fallthrough:F.linear"] += 1
        y = torch.nn.functional.linear(x, weight, bias)
        return torch.relu(y) if relu else y
    ROUTES["linear:ffma"] += 1
    b = None if bias is None else bias.unsqueeze(0)
    return _Linear.apply(x, weight.unsqueeze(0), b, 1 if relu else 0).squeeze(0)


class _LayerNorm(torch.autograd.Function):
    """nn.LayerNorm over the last dimension: one streaming pass forward, ONE pass backward (csrc/ln.cu) instead of
    ATen's grad_input + GammaBeta kernels.  Grouped form: ``groups`` affine pairs (weight / bias (groups, F)); output row
    r of groups * rows_per_group rows normalises input row r % x_rows -- the K ensemble heads, each starting with its own
    LayerNorm on the SHARED embedding (q_ensemble.py:26-48), are one launch instead of F.layer_norm + addcmul."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, groups, heads=False):
        xc = _c(x)
        F_ = xc.shape[-1]
        x_rows = xc.numel() // F_
        shared = heads and xc.dim() == 2                         # (B, F) shared by the heads -> (K, B, F)
        rpg = x_rows if (not heads or shared) else x_rows // groups
        rows = groups * rpg
        need = any(ctx.needs_input_grad[:3])
        y = torch.empty((groups, rpg, F_) if heads else xc.shape, dtype=torch.float32, device=x.device)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device) if need else None
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device) if need else None
        wc = None if weight is None else _c(weight)
        bc = None if bias is None else _c(bias)
        _lib.check(_lib.load().pb_layer_norm_grouped_fwd(int(groups), int(rpg), int(x_rows), F_, float(eps), xc.data_ptr(),
                                                         _lib.ptr(wc), _lib.ptr(bc), y.data_ptr(), _lib.ptr(mean),
                                                         _lib.ptr(rstd), _stream(x)), "pb_layer_norm_grouped_fwd")
        if need:
            ctx.save_for_backward(xc, wc, mean, rstd)
            ctx.has_affine = (weight is not None, bias is not None)
            ctx.meta = (int(groups), int(rpg), int(x_rows), F_, shared, bool(heads))
        return y

    @staticmethod
    def backward(ctx, dy):
        xc, wc, mean, rstd = ctx.saved_tensors
        groups, rpg, x_rows, F_, shared, heads = ctx.meta
        dy = _c(dy)
        lib = _lib.load()
        nb = lib.pb_layer_norm_grouped_bwd_blocks(groups, rpg, F_)
        partials = torch.empty(2 * groups * nb * F_, dtype=torch.float32, device=dy.device)
        dx = torch.empty((groups, rpg, F_) if heads else xc.shape, dtype=torch.float32, device=dy.device)
        shape_p = (groups, F_) if heads else (F_,)
        dg = torch.empty(shape_p, dtype=torch.float32, device=dy.device) if ctx.has_affine[0] else None
        db = torch.empty(shape_p, dtype=torch.float32, device=dy.device) if ctx.has_affine[1] else None
        _lib.check(lib.pb_layer_norm_grouped_bwd(groups, rpg, x_rows, F_, xc.data_ptr(), dy.data_ptr(), _lib.ptr(wc),
                                                 mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(), _lib.ptr(dg), _lib.ptr(db),
                                                 partials.data_ptr(), _stream(dy)), "pb_layer_norm_grouped_bwd")
        if not ctx.needs_input_grad[0]:
            dx = None
        elif shared:
            dx = sum_leading(dx)                                  # the heads share their input
        return dx, dg, db, None, None, None


def _ln_supported(x, F_):
    return (x.is_cuda and x.dtype == torch.float32 and x.numel() > 0
            and _lib.load().pb_layer_norm_supported(x.numel() // F_, F_) == 1)


def layer_norm(x, module):
    """nn.LayerNorm module applied through the fused kernels (any number of rows)."""
    if x.dim() == 2 and len(module.normalized_shape) == 1 and _ln_supported(x, x.shape[1]):
        ROUTES["ln:fused"] += 1
        return _LayerNorm.apply(x, module.weight, module.bias, module.eps, 1, False)
    ROUTES["fallthrough:nn.LayerNorm"] += 1
    return module(x)


def layer_norm_heads(x, weight, bias, eps=1e-5):
    """LayerNorm with per-head affine parameters weight / bias (K, F): x (B, F) shared by the heads or (K, B, F)
    -> (K, B, F)."""
    K, F_ = weight.shape
    if _ln_supported(x, F_) and (x.dim() == 2 or (x.dim() == 3 and x.shape[0] == K)):
        ROUTES["ln:fused_heads"] += 1
        return _LayerNorm.apply(x, weight, bias, eps, K, True)
    ROUTES["fallthrough:F.layer_norm+addcmul"] += 1
    normed = torch.nn.functional.layer_norm(x, (F_,), eps=eps)
    return torch.addcmul(bias.unsqueeze(1), normed if x.dim() == 3 else normed.unsqueeze(0), weight.unsqueeze(1))


def run_sequential(seq, x):
    """Evaluate an nn.Sequential of Linear / ReLU / LayerNorm / ... modules, routing every Linear (with a
    directly following ReLU fused in) through the fused kernel.  Other modules run as they are."""
    import torch.nn as nn
    mods = list(seq)
    i = 0
    while i < len(mods):
        m = mods[i]
        if isinstance(m, nn.Linear) and x.dim() == 2 and x.is_cuda:
            fuse = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
            x = linear(x, m.weight, m.bias, relu=fuse)
            i += 2 if fuse else 1
        elif isinstance(m, nn.LayerNorm):
            x = layer_norm(x, m)
            i += 1
        else:
            if not isinstance(m, (nn.ReLU, nn.Flatten, nn.Identity)):
                ROUTES["fallthrough:module:%s" % type(m).__name__] += 1
            x = m(x)
            i += 1
    return x


class _TheilIndex(torch.autograd.Function):
    """Theil index of the heads' parameter norms over stacked (K, ...) tensors: 2 launches forward, 1 backward
    (csrc/theil.cu) instead of ~100 ATen launches (q_ensemble.py:86-92)."""

    @staticmethod
    def forward(ctx, table, total_numel, *stacked):
        K = stacked[0].shape[0]
        dev = stacked[0].device
        lib = _lib.load()
        chunks = lib.pb_theil_chunks(max(p[0].numel() for p in stacked))
        partial = torch.empty(len(stacked) * K * chunks, dtype=torch.float32, device=dev)
        theil = torch.empty((), dtype=torch.float32, device=dev)
        coef = torch.empty(K, dtype=torch.float32, device=dev)
        _lib.check(lib.pb_theil_fwd(len(stacked), K, chunks, table.data_ptr(), partial.data_ptr(), theil.data_ptr(),
                                    coef.data_ptr(), _stream(stacked[0])), "pb_theil_fwd")
        ctx.save_for_backward(table, coef)
        ctx.meta = (len(stacked), K, int(total_numel), [tuple(p.shape) for p in stacked], chunks)
        return theil

    @staticmethod
    def backward(ctx, g):
        table, coef = ctx.saved_tensors
        n, K, total, shapes, chunks = ctx.meta
        g = _c(g)
        out = torch.empty(total, dtype=torch.float32, device=g.device)
        _lib.check(_lib.load().pb_theil_bwd(n, K, chunks, table.data_ptr(), coef.data_ptr(), g.data_ptr(), out.data_ptr(),
                                            _stream(g)), "pb_theil_bwd")
        grads, off = [], 0
        for shp in shapes:
            cnt = 1
            for d in shp:
                cnt *= d
            grads.append(out[off:off + cnt].view(shp))
            off += cnt
        return (None, None) + tuple(grads)


def theil_index(stacked, cache):
    """stacked: list of contiguous CUDA parameters of shape (K, ...).  ``cache``: dict owned by the module (the address
    table is rebuilt when a parameter moves)."""
    key = tuple(p.data_ptr() for p in stacked)
    if cache.get("key") != key:
        rows, off = [], 0
        for p in stacked:
            per = p[0].numel()
            rows += [p.data_ptr(), per, off]
            off += p.numel()
        cache["key"], cache["total"] = key, off
        cache["table"] = torch.tensor(rows, dtype=torch.int64, device=stacked[0].device)
    return _TheilIndex.apply(cache["table"], cache["total"], *stacked)


UNIT_TOTAL_GRAD = False        # set by Agent._loss_and_backward while it runs total.backward() with the implicit gradient 1
_ONES = {}


def unit_gradient(device):
    """A cached scalar 1.0 on ``device`` (saves autograd's ones_like fill launch per backward)."""
    t = _ONES.get(device)
    if t is None:
        t = _ONES[device] = torch.ones((), dtype=torch.float32, device=device)
    return t


_LOSS_TICKET = {}


def _loss_ticket(device):
    t = _LOSS_TICKET.get(device)
    if t is None:
        t = _LOSS_TICKET[device] = torch.zeros(1, dtype=torch.int32, device=device)
    return t


class _FusedTotalLoss(torch.autograd.Function):
    """total = mean(dist*w) + mean(q'*w) straight from the quantile / ensemble tables: loss heads, PER
    weighting, TD mix and the gradients w.r.t. z_cur / q_cur (already scaled by w_b/B) in 3 launches;
    backward is one scalar multiply per table.  q' = q_weight * (mse - q_offset)."""

    @staticmethod
    def forward(ctx, z_cur, q_cur, tau, z_on, z_tg, q_on, q_tg, action, ret, gamma, nonterm, w, q_offset, T, Tp,
                kappa, dist_weight, q_weight):
        ref = z_cur if z_cur is not None else q_cur
        _lib.require_cuda(ref, "tables")
        lib, stream, dev = _lib.load(), _stream(ref), ref.device
        B = action.numel()
        action_c, ret_c, gamma_c = _c(action, torch.int64).view(-1), _c(ret).view(-1), _c(gamma).view(-1)
        nt = None if nonterm is None else nonterm.contiguous().view(-1).view(torch.uint8)
        w_c = None if w is None else _c(w).view(-1)
        dist = mse = gz = gq = None
        if z_cur is not None:
            zc = _c(z_cur)
            dist = torch.empty(B, dtype=torch.float32, device=dev)
            gz = torch.empty_like(zc)
            _lib.check(lib.pb_iqn_qh_loss(B, T, Tp, zc.shape[-1], zc.data_ptr(), _c(tau).view(-1).data_ptr(),
                                          _c(z_on).data_ptr(), _c(z_tg).data_ptr(), action_c.data_ptr(),
                                          ret_c.data_ptr(), gamma_c.data_ptr(), _lib.ptr(nt), float(kappa),
                                          float(dist_weight), _lib.ptr(w_c), 1.0 / B, dist.data_ptr(), gz.data_ptr(),
                                          stream), "pb_iqn_qh_loss")
        total = torch.empty((), dtype=torch.float32, device=dev)
        td = torch.empty(B, dtype=torch.float32, device=dev)
        if q_cur is not None:
            qc = _c(q_cur)
            K, _, A = qc.shape
            mse = torch.empty(B, dtype=torch.float32, device=dev)
            gq = torch.empty_like(qc)
            # the ensemble loss kernel's last CTA also combines the heads' losses into the PER-weighted total and the TD
            # mix (agent.py:58-64): one launch less on the step's critical path
            _lib.check(lib.pb_ens_q_loss_total(B, A, K, qc.data_ptr(), _c(q_on).data_ptr(), _c(q_tg).data_ptr(),
                                               action_c.data_ptr(), ret_c.data_ptr(), gamma_c.data_ptr(), _lib.ptr(nt), 1.0,
                                               _lib.ptr(w_c), float(q_weight) / B, mse.data_ptr(), gq.data_ptr(),
                                               _lib.ptr(dist), float(q_weight), _lib.ptr(q_offset), total.data_ptr(),
                                               td.data_ptr(), _loss_ticket(dev).data_ptr(), stream), "pb_ens_q_loss_total")
        else:
            _lib.check(lib.pb_loss_combine(B, _lib.ptr(dist), None, _lib.ptr(w_c), float(q_weight),
                                           _lib.ptr(q_offset), total.data_ptr(), td.data_ptr(), stream), "pb_loss_combine")
        ctx.save_for_backward(gz, gq)
        ctx.set_materialize_grads(False)      # no zero-fill launches for the non-differentiable outputs
        outs = (total, dist if dist is not None else td.new_empty(0), mse if mse is not None else td.new_empty(0), td)
        ctx.mark_non_differentiable(*outs[1:])
        return outs

    @staticmethod
    def backward(ctx, g_total, *_):
        gz, gq = ctx.saved_tensors
        if g_total is None:
            return (None,) * 18
        if UNIT_TOTAL_GRAD:
            # Agent._loss_and_backward differentiates the scalar total itself: d total / d total = 1 exactly
            return (gz, gq) + (None,) * 16
        return (None if gz is None else gz * g_total, None if gq is None else gq * g_total) + (None,) * 16


def fused_total_loss(z_cur, q_cur, tau, z_on, z_tg, q_on, q_tg, action, ret, gamma, nonterm, w, q_offset, T, Tp,
                     kappa, dist_weight, q_weight):
    return _FusedTotalLoss.apply(z_cur, q_cur, tau, z_on, z_tg, q_on, q_tg, action, ret, gamma, nonterm, w, q_offset,
                                 T, Tp, kappa, dist_weight, q_weight)


class _ConvEmbed(torch.autograd.Function):
    """MinAtar embedding: channels-last obs -> conv3x3 + bias + ReLU -> NCHW flatten, one launch
    (prism/agents/models/minatar_cnn_model.py:13-18,41-44); backward = dW, db only."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _lib.require_cuda(x, "x")
        B, H, W, C = x.shape
        OC = weight.shape[0]
        xc, wc, bc = _c(x), _c(weight), (None if bias is None else _c(bias))
        out = torch.empty(B, OC * (H - 2) * (W - 2), dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().pb_conv3x3_relu_fwd(B, H, W, C, OC, xc.data_ptr(), wc.data_ptr(), _lib.ptr(bc),
                                                   out.data_ptr(), _stream(x)), "pb_conv3x3_relu_fwd")
        ctx.dims = (B, H, W, C, OC)
        ctx.has_bias = bias is not None
        ctx.save_for_backward(xc, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        xc, out = ctx.saved_tensors
        B, H, W, C, OC = ctx.dims
        lib = _lib.load()
        dout = _c(dout)
        groups = lib.pb_conv3x3_relu_bwd_groups(B)
        scratch = torch.empty(groups * (OC * C * 9 + OC), dtype=torch.float32, device=dout.device)
        dw = torch.empty(OC, C, 3, 3, dtype=torch.float32, device=dout.device)
        db = torch.empty(OC, dtype=torch.float32, device=dout.device) if ctx.has_bias else None
        _lib.check(lib.pb_conv3x3_relu_bwd(B, H, W, C, OC, xc.data_ptr(), out.data_ptr(), dout.data_ptr(),
                                           scratch.data_ptr(), dw.data_ptr(), _lib.ptr(db), _stream(dout)),
                   "pb_conv3x3_relu_bwd")
        if TRACE_MARK is not None:
            TRACE_MARK("bwd:conv3x3")
        return None, dw, db


def conv3x3_relu_flatten(x, weight, bias):
    return _ConvEmbed.apply(x, weight, bias)
