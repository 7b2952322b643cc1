"""FlatAdam -- clip_grad_norm_ + Adam over one flat fp32 parameter arena.

Replaces ``torch.nn.utils.clip_grad_norm_`` + ``torch.optim.Adam.step`` of the reference update
(prism/agents/agent.py:73-74; optimiser built at prism/factory/agent_factory.py:44-47) with two
launches per step (csrc/agent_kernels.cu): a multi-tensor gather of autograd's gradients into the
arena with the squared norm folded in, and one fused clip+Adam sweep.  All model parameters are
re-pointed at views of the arena at construction, so
  * the target-network sync is one device copy,
  * the data-parallel gradient all-reduce is ONE NCCL call on the flat gradient.
The step counter lives on the device: the whole step is CUDA-graph capturable.
"""
import torch

from .. import _lib


def flatten_parameters(module):
    """Re-point every parameter of ``module`` at a view of one flat fp32 arena (16-byte aligned
    slices, registration order).  Returns (arena, offsets); also stored as ``module._flat_arena`` /
    ``module._flat_offsets``.  Two modules of the same architecture get identical layouts, which
    makes the target-network sync a single copy."""
    params = [p for p in module.parameters()]
    dev = params[0].device
    offsets, off = [], 0
    for p in params:
        offsets.append(off)
        off += (p.numel() + 3) // 4 * 4
    arena = torch.zeros(off, dtype=torch.float32, device=dev)
    with torch.no_grad():
        for p, o in zip(params, offsets):
            view = arena[o:o + p.numel()].view_as(p)
            view.copy_(p.data)
            p.data = view
    module._flat_arena, module._flat_offsets = arena, offsets
    return arena, offsets


FUSED_STEP = __import__("os").environ.get("PB_ADAM_FUSED", "1") != "0"   # one-launch gather + clip + Adam for small arenas


class FlatAdam(object):
    def __init__(self, params, lr, betas=(0.9, 0.999), eps=1e-8, max_grad_norm=0.0, arena=None):
        self._lib = _lib.load()
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("no parameters")
        dev = self.params[0].device
        if dev.type != "cuda":
            raise _lib.PbError("FlatAdam needs CUDA parameters (no CPU path)")
        self.device = dev
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.max_grad_norm = float(max_grad_norm) if max_grad_norm else 0.0
        if arena is not None:
            # parameters were already flattened (flatten_parameters): adopt that arena
            self.arena, self.offsets = arena
            off = self.arena.numel()
            for p, o in zip(self.params, self.offsets):
                if p.data_ptr() != self.arena.data_ptr() + 4 * o:
                    raise _lib.PbError("parameter is not a view of the given arena")
        else:
            # arena layout: every tensor starts on a 16-byte boundary
            self.offsets, off = [], 0
            for p in self.params:
                self.offsets.append(off)
                off += (p.numel() + 3) // 4 * 4
            self.arena = torch.zeros(off, dtype=torch.float32, device=dev)
            with torch.no_grad():
                for p, o in zip(self.params, self.offsets):
                    view = self.arena[o:o + p.numel()].view_as(p)
                    view.copy_(p.data)
                    p.data = view
        self.numel = off
        self.grad = torch.zeros(off, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(off, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(off, dtype=torch.float32, device=dev)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=dev)
        self.partials = torch.zeros(4096, dtype=torch.float32, device=dev)
        self.norm_out = torch.zeros(2, dtype=torch.float32, device=dev)
        self.table = torch.zeros(len(self.params) * 3, dtype=torch.int64, device=dev)
        self._table_host = torch.zeros(len(self.params) * 3, dtype=torch.int64).pin_memory()
        self._table_key = None
        self.grad_scale = 1.0           # 1/world_size under data parallelism
        self.allreduce = None           # callable(flat_grad) inserted between gather and Adam (library collective)
        self.peer = None                # PeerGroup: gradient exchange fused with clip + Adam over peer memory

    def _fused_max_n(self):
        m = getattr(self, "_fused_max", None)
        if m is None:
            m = self._fused_max = int(self._lib.pb_adam_fused_max_n())
        return m

    def attach_peer_group(self, peer):
        """Route the data-parallel gradient exchange through csrc/peer.cu: the flat gradient arena moves into the
        rank's peer-mapped block and ``step`` becomes pack -> barrier -> reduce-scatter -> barrier -> fused Adam."""
        if peer.n != self.numel:
            raise _lib.PbError("peer group sized for %d parameters, optimizer has %d" % (peer.n, self.numel))
        self.grad = peer.grad
        self.peer = peer
        self.allreduce = None

    # ---- torch.optim-like surface ------------------------------------------------------
    def zero_grad(self, set_to_none=True):
        for p in self.params:
            if set_to_none:
                p.grad = None
            elif p.grad is not None:
                p.grad.zero_()

    def refresh_grad_table(self):
        """Re-read the addresses of autograd's gradient tensors (static under a CUDA graph)."""
        key = tuple(0 if p.grad is None else p.grad.data_ptr() for p in self.params)
        if key == self._table_key:
            return
        t = self._table_host
        for i, (p, o) in enumerate(zip(self.params, self.offsets)):
            g = p.grad
            if g is not None and (g.dtype != torch.float32 or not g.is_contiguous()):
                raise _lib.PbError("gradients must be contiguous fp32")
            t[3 * i + 0] = 0 if g is None else g.data_ptr()
            t[3 * i + 1] = o
            t[3 * i + 2] = p.numel()
        self.table.copy_(t, non_blocking=True)
        self._table_key = key

    def step(self, refresh_table=True):
        if refresh_table:
            self.refresh_grad_table()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        import ctypes
        n_part = ctypes.c_int(0)
        mark = getattr(self, "_mark", None) or (lambda name: None)      # LearnerStep.enable_trace()
        if self.peer is not None:
            # into the half of the double-buffered peer arena this step's exchange will read (device-side parity)
            _lib.check(self._lib.pb_pack_grads_parity(len(self.params), self.table.data_ptr(), self.grad_scale,
                                                      self.grad.data_ptr(), self.peer.epoch_gather_ptr,
                                                      self.peer.grad_stride, None, None, None, stream),
                       "pb_pack_grads_parity")
            mark("opt:packed")
            self.peer.allreduce_adam(self, mark=mark)
            return
        if self.allreduce is None and FUSED_STEP and len(self.params) <= 64 and self.numel <= self._fused_max_n():
            # small arena: gather + norm + clip + Adam in ONE launch (the gradient stays in registers)
            _lib.check(self._lib.pb_adam_fused_step(len(self.params), self.table.data_ptr(), self.grad_scale, self.numel,
                                                    self.arena.data_ptr(), self.grad.data_ptr(), self.exp_avg.data_ptr(),
                                                    self.exp_avg_sq.data_ptr(), self.step_count.data_ptr(), self.lr,
                                                    self.betas[0], self.betas[1], self.eps, self.max_grad_norm,
                                                    self.partials.data_ptr(), self.norm_out.data_ptr(), stream),
                       "pb_adam_fused_step")
            mark("opt:packed")
            return
        if self.allreduce is None:
            _lib.check(self._lib.pb_pack_grads(len(self.params), self.table.data_ptr(), self.grad_scale,
                                               self.grad.data_ptr(), self.partials.data_ptr(),
                                               self.step_count.data_ptr(), ctypes.byref(n_part), stream),
                       "pb_pack_grads")
            mark("opt:packed")
        else:
            _lib.check(self._lib.pb_pack_grads(len(self.params), self.table.data_ptr(), self.grad_scale,
                                               self.grad.data_ptr(), None, None, None, stream), "pb_pack_grads")
            self.allreduce(self.grad)
            _lib.check(self._lib.pb_grad_sumsq(self.numel, self.grad.data_ptr(), self.partials.data_ptr(),
                                               self.step_count.data_ptr(), ctypes.byref(n_part), stream),
                       "pb_grad_sumsq")
        _lib.check(self._lib.pb_adam_clip_apply(self.numel, self.arena.data_ptr(), self.grad.data_ptr(),
                                                self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                                                self.step_count.data_ptr(), self.lr, self.betas[0], self.betas[1],
                                                self.eps, self.max_grad_norm, self.partials.data_ptr(), n_part.value,
                                                self.norm_out.data_ptr(), stream), "pb_adam_clip_apply")

    # ---- checkpoint format: torch.optim.Adam's own (prism/agents/agent.py:231-252 saves optimizer.state_dict()) ------
    def reference_layout(self):
        """[(arena offset, shape)] in the order the REFERENCE's ``model.parameters()`` yields its tensors: the order of
        ``model.state_dict()`` (reference key names; the stacked (K, ...) ensemble tensors un-stacked head by head).
        Needs ``layout_model`` (set by build_agent); the entries are views of the parameter arena, so their addresses
        give the offsets."""
        model = getattr(self, "layout_model", None)
        if model is None:
            return [(o, tuple(p.shape)) for p, o in zip(self.params, self.offsets)]
        base, out = self.arena.data_ptr(), []
        for _, v in model.state_dict().items():
            off = (v.data_ptr() - base) // 4
            if not (0 <= off and off + v.numel() <= self.numel and v.is_contiguous()):
                raise _lib.PbError("state_dict entry is not a contiguous view of the parameter arena")
            out.append((off, tuple(v.shape)))
        return out

    def state_dict(self):
        """A ``torch.optim.Adam.state_dict()``: per-parameter ``step`` / ``exp_avg`` / ``exp_avg_sq`` keyed by the
        index of the parameter in the reference's ``model.parameters()``, plus ``param_groups`` -- what the reference
        reads back with ``optimizer.load_state_dict`` (agent.py:244-252), and vice versa."""
        layout = self.reference_layout()
        template = torch.optim.Adam([torch.zeros(1)], lr=self.lr, betas=self.betas, eps=self.eps)
        group = dict(template.state_dict()["param_groups"][0])
        group["params"] = list(range(len(layout)))
        state = {}
        steps = int(self.step_count.item())
        if steps > 0:
            m, v = self.exp_avg.cpu(), self.exp_avg_sq.cpu()
            for i, (off, shape) in enumerate(layout):
                n = 1
                for d in shape:
                    n *= d
                state[i] = {"step": torch.tensor(float(steps)), "exp_avg": m[off:off + n].view(shape).clone(),
                            "exp_avg_sq": v[off:off + n].view(shape).clone()}
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, sd):
        if "param_groups" not in sd:
            # the flat layout written by earlier versions of this class
            self.exp_avg.copy_(sd["exp_avg"]); self.exp_avg_sq.copy_(sd["exp_avg_sq"]); self.step_count.copy_(sd["step"])
            self.lr, self.betas, self.eps = sd["lr"], tuple(sd["betas"]), sd["eps"]
            return
        layout = self.reference_layout()
        group = sd["param_groups"][0]
        if len(group["params"]) != len(layout):
            raise ValueError("optimizer checkpoint holds %d parameters, the model has %d" %
                             (len(group["params"]), len(layout)))
        self.lr, self.betas, self.eps = float(group["lr"]), tuple(float(b) for b in group["betas"]), float(group["eps"])
        m, v = torch.zeros(self.numel), torch.zeros(self.numel)
        steps = 0
        for i, (off, shape) in enumerate(layout):
            st = sd["state"].get(group["params"][i], sd["state"].get(i))
            if st is None:
                continue
            n = st["exp_avg"].numel()
            if tuple(st["exp_avg"].shape) != shape:
                raise ValueError("optimizer state %d has shape %s, expected %s" % (i, tuple(st["exp_avg"].shape), shape))
            m[off:off + n] = st["exp_avg"].detach().float().cpu().reshape(-1)
            v[off:off + n] = st["exp_avg_sq"].detach().float().cpu().reshape(-1)
            steps = max(steps, int(float(st["step"])))
        self.exp_avg.copy_(m); self.exp_avg_sq.copy_(v); self.step_count.fill_(steps)

    # ---- helpers -------------------------------------------------------------------------
    def snapshot(self):
        return (self.arena.clone(), self.exp_avg.clone(), self.exp_avg_sq.clone(), self.step_count.clone())

    def restore(self, snap):
        self.arena.copy_(snap[0]); self.exp_avg.copy_(snap[1]); self.exp_avg_sq.copy_(snap[2])
        self.step_count.copy_(snap[3])
