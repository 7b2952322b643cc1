"""Device-resident uniform replay sampler.

Stands in for the sampler of torchrl's uniform ``ReplayBuffer`` that the reference builds when ``use_per`` is off
(prism/factory/exp_buffer_factory.py:29-33; ``use_per=False`` is its DEFAULT_CONFIG).  The whole sampler is the same
64-byte state block the prioritized store keeps (len / seq / rng words), so ``LearnerStep`` drives it through the
calls it makes on a ``PrioritizedTree`` -- one-graph step, fused ingest, prefetch, and the peer exchange of data
parallelism, which carries the block unchanged.  All arithmetic runs in libprism_b200 (csrc/uniform.cu); this class
only owns the state tensor and forwards raw pointers.  There is no CPU path and no priority write-back.
"""
import ctypes as C

import torch

from .. import _lib


class UniformSampler:
    MODE_IID = 0          # idx = floor(u * len): TimestepBuffer.sample's eager uniform path
    MODE_STRATIFIED = 1   # idx = floor((k + u_k) / n * len)

    def __init__(self, size, mode="iid", seq=0, seed=0x5EED, device="cuda:0"):
        self._lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.PbError("UniformSampler needs a CUDA device (no CPU fallback); got %s" % device)
        self.size = int(size)
        if self.size <= 0:
            raise ValueError("size must be positive")
        self.mode = self.MODE_STRATIFIED if mode in ("stratified", 1) else self.MODE_IID
        self.state = torch.zeros(64, dtype=torch.uint8, device=self.device)
        self._seed = int(seed) & 0x7FFFFFFF                 # the tree's default: ranks draw identical strata
        self.reset(seq)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _st(self):
        return self.state.data_ptr()

    # -- mutation ----------------------------------------------------------------
    def reset(self, seq=0):
        """seq = ``seq``, len = min(seq, size), call number 0 (stream-ordered, no sync)."""
        _lib.check(self._lib.pb_uniform_init(self._st(), self.size, int(seq), self._seed, self._stream()),
                   "pb_uniform_init")

    def resync(self, seq):
        """Like ``reset`` but the device generator keeps its position: after the ring changed outside a learner step,
        the step's draws continue their sequence instead of repeating it (and ranks stay in step with each other)."""
        call = self.state[52:56].clone()                    # pad[2], the call number
        self.reset(seq)
        self.state[52:56].copy_(call)

    def extend(self, n):
        """n new transitions at the ring cursor: seq += n, len = min(seq, size) on the device (capturable)."""
        _lib.check(self._lib.pb_uniform_extend(self._st(), self.size, int(n), self._stream()), "pb_uniform_extend")

    def seed(self, seed, call=0):
        """Key of the in-kernel Philox generator (all ranks of a sharded buffer must share it)."""
        self._seed = int(seed) & 0x7FFFFFFF
        words = self.state.view(torch.int32)
        words[13] = int(call) & 0x7FFFFFFF
        words[14] = self._seed

    # -- sampling ----------------------------------------------------------------
    def _u(self, u):
        if u is None:
            return None
        u = torch.as_tensor(u)
        if u.device != self.device or u.dtype != torch.float64 or not u.is_contiguous():
            u = u.to(device=self.device, dtype=torch.float64, non_blocking=True).contiguous()
        return u

    def _outs(self, n, idx_out, weight_out):
        if idx_out is None:
            idx_out = torch.empty(n, dtype=torch.int64, device=self.device)
        if weight_out is None:
            weight_out = torch.empty(n, dtype=torch.float32, device=self.device)
        return idx_out, weight_out

    def sample(self, n, u=None, mode=None, idx_out=None, weight_out=None):
        """n indices in [0, len) and weights 1.  ``u``: fp64 uniforms in [0,1) (device); drawn inside the kernel
        (Philox4x32-10 keyed by ``seed()``) when omitted."""
        n = int(n)
        u = self._u(u)
        idx_out, weight_out = self._outs(n, idx_out, weight_out)
        mode = self.mode if mode is None else (self.MODE_STRATIFIED if mode in ("stratified", 1) else self.MODE_IID)
        _lib.check(self._lib.pb_uniform_sample(self._st(), n, _lib.ptr(u), mode, idx_out.data_ptr(),
                                               weight_out.data_ptr(), self._stream()), "pb_uniform_sample")
        return idx_out, weight_out

    def sample_global(self, n_ranks, rank, all_state, n_global, u, idx_out=None, weight_out=None, stratum_out=None):
        """Sharded global stratified sampling over the concatenated shards: every rank evaluates all strata and keeps
        its run.  ``all_state``: (n_ranks, 64) uint8, the all-gathered shard state blocks."""
        n_global = int(n_global)
        idx_out, weight_out = self._outs(n_global, idx_out, weight_out)
        assert all_state.dtype == torch.uint8 and all_state.numel() == 64 * n_ranks and all_state.is_contiguous()
        assert u is None or (u.dtype == torch.float64 and u.is_cuda)
        _lib.check(self._lib.pb_uniform_sample_global(self._st(), int(n_ranks), int(rank), all_state.data_ptr(),
                                                      n_global, _lib.ptr(u), idx_out.data_ptr(), weight_out.data_ptr(),
                                                      _lib.ptr(stratum_out), self._stream()),
                   "pb_uniform_sample_global")
        return idx_out, weight_out

    def sample_global_peer(self, peer, n_global, u, idx_out=None, weight_out=None, stratum_out=None):
        """``sample_global`` on the shard states of the latest ``PeerGroup.state_put`` exchange: the kernel itself waits
        (bounded) until every rank's put has landed in this rank's peer-mapped slot."""
        n_global = int(n_global)
        idx_out, weight_out = self._outs(n_global, idx_out, weight_out)
        assert u is None or (u.dtype == torch.float64 and u.is_cuda)
        _lib.check(self._lib.pb_uniform_sample_global_peer(self._st(), C.byref(peer.c), n_global, _lib.ptr(u),
                                                           idx_out.data_ptr(), weight_out.data_ptr(),
                                                           _lib.ptr(stratum_out), self._stream()),
                   "pb_uniform_sample_global_peer")
        return idx_out, weight_out

    # -- host-visible state (synchronises; not on the hot path) -------------------
    def state_host(self):
        raw = self.state.cpu().numpy().tobytes()
        s = _lib.pb_per_state.from_buffer_copy(raw)
        return {"len": s.len, "seq": s.seq, "status": s.status, "owned_lo": s.owned_lo, "owned_n": s.owned_n,
                "call": s.pad[2], "seed": s.pad[3]}

    def snapshot(self):
        """Device copy of everything a call mutates (graph warm-ups that must not advance the sampler)."""
        return (self.state.clone(),)

    def restore(self, snap):
        self.state.copy_(snap[0])
