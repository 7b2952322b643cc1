"""PeerGroup -- the host side of csrc/peer.cu: one peer-mapped block per rank (NVLink / NVSwitch, CUDA IPC).

Layout of a rank's block (bytes):  grad [2 x n floats, double-buffered] | reduced [n floats] | flags [64 u64] |
norm_parts [8 f64] | state [4 x 8 x 64 B] | epochs [3 x u64] | status [u32].  ``torch.distributed`` is only used once, to exchange the 64-byte IPC handles; no
collective library call remains on the per-step path (SURVEY 8e, DESIGN.md section 5).

``PeerGroup.loopback(world, n, device)`` builds ``world`` groups inside ONE process on one GPU (plain pointers to
each other's blocks): the tests drive them on separate streams, which exercises the same kernels and flag protocol
without a second GPU.
"""
import ctypes as C

import torch

from . import _lib


FUSED_EXCHANGE = __import__("os").environ.get("PB_PEER_FUSED", "1") != "0"   # one-launch exchange + update for small arenas
ONE_SHOT_MAX_BYTES = 32 * 1024 * 1024      # n * 4 * world up to which the one-shot (single barrier) all-reduce is used
WAIT_TIMEOUT_S = float(__import__("os").environ.get("PB_PEER_TIMEOUT_S", "20"))   # bound of every cross-GPU flag wait


class _RawCuda:
    """Expose a raw device allocation to torch through __cuda_array_interface__."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def _layout(n):
    n_bytes = ((int(n) * 4 + 255) // 256) * 256
    off = {"grad": 0, "grad_stride_bytes": n_bytes, "reduced": 2 * n_bytes, "flags": 3 * n_bytes}
    off["norm_parts"] = off["flags"] + 64 * 8
    off["state"] = off["norm_parts"] + 64
    off["epoch"] = off["state"] + 4 * _lib.PB_PEER_MAX * 64      # slots 0-1: state_allgather, 2-3: state_put
    off["status"] = off["epoch"] + 64
    off["total"] = off["epoch"] + 256
    return off


class PeerGroup:
    def __init__(self, rank, world, n, device, bases, own_ptr, opened=()):
        self.rank, self.world, self.n, self.device = int(rank), int(world), int(n), torch.device(device)
        self._own_ptr, self._opened = own_ptr, list(opened)
        self.off = _layout(n)
        _lib.check(_lib.load().pb_peer_preload(), "pb_peer_preload")
        _lib.check(_lib.load().pb_optimizer_preload(), "pb_optimizer_preload")
        g = _lib.pb_peer_group()
        g.world, g.rank = self.world, self.rank
        for p in range(self.world):
            b = bases[p]
            g.grad[p], g.reduced[p] = b + self.off["grad"], b + self.off["reduced"]
            g.flags[p], g.norm_parts[p], g.state[p] = b + self.off["flags"], b + self.off["norm_parts"], b + self.off["state"]
        g.epoch = bases[self.rank] + self.off["epoch"]
        g.status = bases[self.rank] + self.off["status"]
        g.timeout_ns = int(WAIT_TIMEOUT_S * 1e9)
        g.grad_stride = self.off["grad_stride_bytes"] // 4
        self.c = g
        self.grad_stride = self.off["grad_stride_bytes"] // 4
        self.epoch_gather_ptr = bases[self.rank] + self.off["epoch"] + 8        # channel 1: completed state gathers
        self._n_gathers = 0                                                     # host mirror of that count (eager calls)
        self._block = torch.as_tensor(_RawCuda(own_ptr, self.off["total"]), device=self.device)
        # both halves of the double-buffered gradient arena; the pack of a step writes half (completed gathers & 1)
        self.grad = self._block[self.off["grad"]:self.off["grad"] + 4 * self.n].view(torch.float32)
        self.grad_halves = [self._block[self.off["grad"] + h * self.off["grad_stride_bytes"]:
                                        self.off["grad"] + h * self.off["grad_stride_bytes"] + 4 * self.n].view(torch.float32)
                            for h in (0, 1)]
        self._status = self._block[self.off["status"]:self.off["status"] + 4].view(torch.int32)
        self._dummy_state = torch.zeros(64, dtype=torch.uint8, device=self.device)
        self.reduced = self._block[self.off["reduced"]:self.off["reduced"] + 4 * self.n].view(torch.float32)
        self.all_state = torch.zeros(self.world, 64, dtype=torch.uint8, device=self.device)     # local copy of the gather

    # ---- construction -------------------------------------------------------------------------------------
    @classmethod
    def create(cls, process_group, rank, world, n, device):
        """One block per rank, handles exchanged through ``torch.distributed`` (any backend)."""
        import torch.distributed as dist
        if world > _lib.PB_PEER_MAX:
            raise _lib.PbError("peer exchange supports up to %d ranks on one box" % _lib.PB_PEER_MAX)
        lib = _lib.load()
        torch.cuda.set_device(device)
        own = C.c_void_p()
        _lib.check(lib.pb_peer_alloc(_layout(n)["total"], C.byref(own)), "pb_peer_alloc")
        handle = (C.c_ubyte * 64)()
        _lib.check(lib.pb_peer_export(own, handle), "pb_peer_export")
        handles = [None] * world
        dist.all_gather_object(handles, bytes(handle), group=process_group)
        bases, opened = [], []
        for p in range(world):
            if p == rank:
                bases.append(own.value)
                continue
            ptr = C.c_void_p()
            buf = (C.c_ubyte * 64).from_buffer_copy(handles[p])
            _lib.check(lib.pb_peer_open(buf, C.byref(ptr)), "pb_peer_open")
            bases.append(ptr.value)
            opened.append(ptr.value)
        dist.barrier(group=process_group)
        return cls(rank, world, n, device, bases, own.value, opened)

    @classmethod
    def loopback(cls, world, n, device):
        lib = _lib.load()
        torch.cuda.set_device(device)
        ptrs = []
        for _ in range(world):
            own = C.c_void_p()
            _lib.check(lib.pb_peer_alloc(_layout(n)["total"], C.byref(own)), "pb_peer_alloc")
            ptrs.append(own.value)
        return [cls(r, world, n, device, ptrs, ptrs[r]) for r in range(world)]

    # ---- stream-ordered operations --------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def barrier(self):
        _lib.check(_lib.load().pb_peer_barrier(C.byref(self.c), self._stream()), "pb_peer_barrier")

    def state_allgather(self, state):
        """state: this rank's 64-byte tree state block (uint8 tensor).  Returns the (world, 64) gathered view.
        A full handshake of all ranks: it is also THE barrier of the gradient exchange (allreduce_adam)."""
        _lib.check(_lib.load().pb_peer_state_allgather(C.byref(self.c), state.data_ptr(), self.all_state.data_ptr(),
                                                       self._stream()),
                   "pb_peer_state_allgather")
        self._n_gathers += 1
        return self.all_state

    def state_put(self, state):
        """Non-blocking half of the shard-state exchange: this rank's 64-byte tree state goes to every rank; the wait
        happens inside the next ``PrioritizedTree.sample_global_peer`` (every rank must call both, in the same order)."""
        _lib.check(_lib.load().pb_peer_state_put(C.byref(self.c), state.data_ptr(), self._stream()), "pb_peer_state_put")

    def grad_in_flight(self):
        """The half of the gradient arena the next exchange reads (eager calls only: under graph replay the device
        counter decides, see pb_pack_grads_parity)."""
        return self.grad_halves[self._n_gathers & 1]

    def check(self):
        """Raise if a cross-GPU wait timed out (synchronises; call it off the hot path)."""
        st = int(self._status.item())
        if st:
            raise _lib.PbError("peer exchange: a rank did not arrive within %.0f s (status 0x%x, rank %d of %d)"
                               % (WAIT_TIMEOUT_S, st, self.rank, self.world))

    def allreduce_adam(self, opt, mark=None):
        """Sum the gradient arenas over the ranks and apply clip + the optimizer's update on every replica
        (csrc/peer.cu).  ``opt.rule`` (a ``_lib.PB_OPT_*``) selects Adam, RMSprop or SGD; an optimizer without one is
        Adam, read through ``betas``.

        ONE cross-GPU handshake per step for small arenas: it tells every rank all gradients are packed (the fused
        launch signals on channel 1 itself; the multi-launch schedules run ``state_allgather`` of a dummy block).  The
        arena is double-buffered by the parity of the handshake count, so a fast rank packing its next gradient never
        overwrites what a slower rank still pulls -- no trailing barrier."""
        lib, st = _lib.load(), self._stream()
        mark = mark or (lambda name: None)                        # timeline marks of LearnerStep.enable_trace()
        rule = getattr(opt, "rule", _lib.PB_OPT_ADAM)
        h1, h2 = opt._hyper() if hasattr(opt, "_hyper") else opt.betas
        m, v = _lib.ptr(opt.exp_avg), _lib.ptr(opt.exp_avg_sq)
        if (FUSED_EXCHANGE and self.n <= int(lib.pb_peer_allreduce_opt_max_n(rule))
                and self.n * 4 * self.world <= ONE_SHOT_MAX_BYTES):
            # small arena: handshake + pulls + global norm + clip + update in ONE launch
            _lib.check(lib.pb_peer_allreduce_opt(rule, C.byref(self.c), self.n, opt.arena.data_ptr(), m, v,
                                                 opt.step_count.data_ptr(), opt.lr, h1, h2, opt.eps, opt.max_grad_norm,
                                                 opt.partials.data_ptr(), opt.norm_out.data_ptr(), st),
                       "pb_peer_allreduce_opt")
            self._n_gathers += 1                                  # channel 1 advanced: the other half of the arena is next
            mark("opt:applied")
            return
        self.state_allgather(self._dummy_state)                   # every rank packed its gradient
        mark("opt:exchanged")
        if self.n * 4 * self.world <= ONE_SHOT_MAX_BYTES:
            # small arena: pulling every rank's gradient whole costs less than a second cross-GPU barrier
            n_part = C.c_int(0)
            _lib.check(lib.pb_peer_pull_sum(C.byref(self.c), self.n, opt.partials.data_ptr(), opt.step_count.data_ptr(),
                                            C.byref(n_part), st), "pb_peer_pull_sum")
            mark("opt:summed")
            _lib.check(lib.pb_opt_clip_apply(rule, self.n, opt.arena.data_ptr(), self.reduced.data_ptr(), m, v,
                                             opt.step_count.data_ptr(), opt.lr, h1, h2, opt.eps, opt.max_grad_norm,
                                             opt.partials.data_ptr(), n_part.value, opt.norm_out.data_ptr(), st),
                       "pb_opt_clip_apply")
            mark("opt:applied")
            return
        _lib.check(lib.pb_peer_reduce_scatter(C.byref(self.c), self.n, opt.partials.data_ptr(), opt.step_count.data_ptr(), st),
                   "pb_peer_reduce_scatter")
        mark("opt:slice_reduced")
        _lib.check(lib.pb_peer_barrier(C.byref(self.c), st), "pb_peer_barrier")            # every slice reduced + norms published
        mark("opt:all_reduced")
        _lib.check(lib.pb_peer_opt(rule, C.byref(self.c), self.n, opt.arena.data_ptr(), m, v, opt.step_count.data_ptr(),
                                   opt.lr, h1, h2, opt.eps, opt.max_grad_norm, opt.norm_out.data_ptr(), None, st),
                   "pb_peer_opt")

    def close(self):
        """Unmap the peers' blocks and free this rank's own.  Every rank must have finished its last exchange (the
        caller synchronises and, across processes, barriers first); ``grad`` / ``reduced`` are dead afterwards."""
        lib = _lib.load()
        for p in self._opened:
            lib.pb_peer_close(C.c_void_p(p))
        self._opened = []
        if self._own_ptr:
            torch.cuda.synchronize(self.device)
            self.grad = self.reduced = self._block = self.grad_halves = self._status = None
            lib.pb_peer_free(C.c_void_p(self._own_ptr))
            self._own_ptr = None
