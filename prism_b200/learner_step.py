"""LearnerStep -- one iteration of the reference's hot loop as ONE CUDA graph.

The reference learner (prism/learner.py:95-125) runs, strictly serially and with a device->host
sync in the middle:
    batch, info = buffer.sample(return_info=True)            # CPU tree + Python batch loop + H2D
    td = agent.update(batch, info['_weight'].to(device))     # CUDA graph of ~100 small kernels
    buffer.update_priority(info['index'], td.abs())          # D2H sync + CPU tree
Here the same three calls never leave the device: sample (Philox uniforms -> tree descent -> fused
n-step/gather into the agent's static batch), update (fused loss heads, clip+Adam) and the
priority write-back are captured into a single graph, replayed once per iteration.

Data parallel (SURVEY 8e): every rank owns a shard (ring + trees) fed by its own collectors.
Per iteration: every rank puts its 64-byte shard state block into every rank's slot after its
priority write-back, the next batch's global stratified sampling waits for those puts itself and
places each stratum on its owner (no transition crosses NVLink), and one all-reduce of the flat
gradient arena is fused with clip + Adam.  Both exchanges run as our own kernels over NVLink peer
memory (csrc/peer.cu); PB_DP_EXCHANGE=nccl (or ranks that cannot map each other) falls back to
NCCL, which all-gathers the states right before the sampling.

Software pipelining (``prefetch``, ``step(ingest=...)``): the priority write-back, the fused ingest
of new collector steps and the NEXT iteration's sample + gather run on parallel branches of the
same graph while backward / exchange / Adam proceed (DESIGN.md section 6).
"""
import torch

from . import _lib
from .agents.optim import FlatAdam
from .experience.per import PrioritizedTree


class LearnerStep:
    def __init__(self, buffer, agent, batch_size=None, use_cuda_graph=True, process_group=None,
                 rank=0, world_size=1, pad_slack=None, exchange=None, prefetch=False):
        self.buffer, self.agent = buffer, agent
        self._lib = _lib.load()
        self.tree = buffer.buffer._sampler
        self.ring = buffer.buffer._storage
        if self.ring is None or self.tree is None:
            raise _lib.PbError("LearnerStep needs a prioritized buffer that already holds transitions")
        self.device = torch.device(buffer.device)
        self.B = int(batch_size or buffer.buffer._batch_size)
        self.world_size, self.rank, self.pg = int(world_size), int(rank), process_group
        self.use_cuda_graph = use_cuda_graph
        self.graph = None
        self._graph_key = None
        self.ingest = None
        d = self.device
        if self.world_size > 1:
            if self.world_size & (self.world_size - 1):
                raise ValueError("sharded sampling needs a power-of-two number of ranks")
            self.B_global = self.B * self.world_size
            # owner-computes placement: a rank trains on the strata that land in its shard.  With STRATIFIED masses that
            # count is B_global * (shard mass / total mass) +- 1, so the slack only has to cover the imbalance of the
            # shards' priority mass, not sampling noise (strata beyond B_pad are dropped for that step)
            slack = pad_slack if pad_slack is not None else max(8, self.B // 16)
            self.B_pad = self.B + slack                      # static rows per rank (zero-weight padding)
            self.all_state = torch.zeros(self.world_size, 64, dtype=torch.uint8, device=d)
            self.stratum = torch.empty(self.B_global, dtype=torch.int64, device=d)
            n_rows = self.B_global
        else:
            self.B_global = self.B_pad = self.B
            n_rows = self.B
        self.u = torch.empty(self.B_global, dtype=torch.float64, device=d)
        self.td = None
        self.sorted = self.world_size > 1 or self.tree.mode == PrioritizedTree.MODE_STRATIFIED
        self.prefetch = bool(prefetch)
        self._primed, self._seen_mutations = False, None
        self.loss_host = None            # enable_loss_readback(): pinned fp32 scalar written by every step
        # static batch, shared by the buffer (writes) and the agent (reads)
        buffer._flush()
        self._n_rows = n_rows
        self._live = None
        if self.prefetch:
            self._setup_prefetch()
        else:
            self.idx = torch.zeros(n_rows, dtype=torch.int64, device=d)
            self.weight = torch.zeros(n_rows, dtype=torch.float32, device=d)
            if buffer._batch is None or buffer._obs.shape[0] != self.B_pad:
                buffer._batch = None
                buffer._alloc_static_batch(self.B_pad, self.ring)
        self.batch = buffer.get_static_batch()
        agent.set_static_batch(self.batch)
        opt = agent.optimizer
        self.peer = None
        if self.world_size > 1:
            if not isinstance(opt, FlatAdam):
                raise _lib.PbError("data parallel needs the FlatAdam arena (one exchange per step)")
            import os
            import sys
            import torch.distributed as dist
            opt.grad_scale = float(self.B_pad) / float(self.B_global)   # local mean over B_pad -> global mean
            mode = (exchange or os.environ.get("PB_DP_EXCHANGE", "peer")).lower()
            if mode == "peer":
                # NVLink / NVSwitch peer memory (csrc/peer.cu): state all-gather and gradient all-reduce + Adam as our
                # own kernels; torch.distributed only exchanges the IPC handles, once
                try:
                    from .peer import PeerGroup
                    self.peer = PeerGroup.create(self.pg, self.rank, self.world_size, opt.numel, d)
                    opt.attach_peer_group(self.peer)
                    # The shard states travel by PUT right after the priority write-back (no rank waits there) and the
                    # global sampling kernel waits for them itself: the exchange hides behind the backward pass, and the
                    # gradient exchange + clip + Adam is one launch whose CTAs wait on the signal pad themselves.
                    self.all_state = self.peer.all_state
                    self._states_synced = False
                except Exception as e:                                   # e.g. ranks on different boxes
                    sys.stderr.write("peer-memory exchange unavailable (%r): using the library collectives\n" % (e,))
                    self.peer = None
            if self.peer is None:
                opt.allreduce = lambda flat: dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.pg)
            self.exchange = "peer" if self.peer is not None else "nccl"
        self.launches_per_step = None
        self._side = None
        self._trace = None               # enable_trace(): device buffer of timeline marks
        self._u_in_block = False         # the step's host uniforms ride in the fused ingest's staging block
        self._defer_mode, self._defer_ok = 0, False             # weight-gradient joins: see _capture / ops._JOINS

    # ------------------------------------------------------------------------------------
    def _setup_prefetch(self):
        """Software pipelining: the NEXT iteration's batch is sampled and gathered on the tail branch of this
        iteration (after the priority write-back and the fused ingest, i.e. exactly where the reference order puts it)
        into a shadow copy of the static batch, while backward / exchange / Adam run; the next replay starts with one
        copy shadow -> live.  Live and shadow are two flat arenas of identical layout."""
        from .experience.batch import Batch
        d = self.device
        self._live, self._live_arena = self._carve(self._n_rows)
        self._shadow, self._shadow_arena = self._carve(self._n_rows)
        lv = self._live
        batch = Batch({"observation": lv["obs"],
                       "next": Batch({"observation": lv["next_obs"], "reward": lv["reward"]},
                                     batch_size=self.B_pad, device=d),
                       "nonterminal": lv["nonterminal"], "gamma": lv["gamma"], "action": lv["action"]},
                      batch_size=self.B_pad, device=d)
        self.buffer.set_static_batch(batch)
        self.idx, self.weight = lv["idx"], lv["weight"]

    def set_prefetch(self, flag):
        """Switch the tail-branch prefetch on or off (the step graph is re-captured on the next call)."""
        flag = bool(flag)
        if flag == self.prefetch:
            return
        self.prefetch = flag
        if flag and self._live is None:
            self._setup_prefetch()
            self.batch = self.buffer.get_static_batch()
            self.agent.set_static_batch(self.batch)
        self.graph, self._primed = None, False

    def _carve(self, n_rows):
        """One flat arena holding a static batch + the sampled indices / weights; returns (views, arena)."""
        import numpy as np
        d, B = self.device, self.B_pad
        E = self.buffer.frame_stack * int(np.prod(self.ring.obs_shape))
        spec = [("obs", B * E, torch.float32), ("next_obs", B * E, torch.float32), ("reward", B, torch.float32),
                ("gamma", B, torch.float32), ("nonterminal", B, torch.bool), ("action", B, torch.int64),
                ("idx", n_rows, torch.int64), ("weight", n_rows, torch.float32)]
        offs, off = {}, 0
        for name, n, dt in spec:
            offs[name] = off
            off += (n * torch.empty(0, dtype=dt).element_size() + 255) // 256 * 256
        arena = torch.zeros(off, dtype=torch.uint8, device=d)
        v = {}
        for name, n, dt in spec:
            nbytes = n * torch.empty(0, dtype=dt).element_size()
            v[name] = arena[offs[name]:offs[name] + nbytes].view(dt)
        fs, shp = self.buffer.frame_stack, tuple(self.ring.obs_shape)
        v["obs"], v["next_obs"] = v["obs"].view(B, fs, *shp), v["next_obs"].view(B, fs, *shp)
        for k in ("reward", "gamma", "nonterminal", "action"):
            v[k] = v[k].view(B, 1)
        v["gamma"].fill_(1.0)
        return v, arena

    def sync_shard_states(self):
        """Collective (every rank, same stream order): put this shard's state block to every rank NOW.  The step graph
        puts it after its priority write-back for the next batch's sampling; this primes the first step and
        re-synchronises after anything outside the step changed a tree (ingest, a manual priority update)."""
        if self.peer is not None:
            self.peer.state_put(self.tree.state)
            self._states_synced = True

    def _sample_gather(self, u, out, tag=""):
        """(shard states of all ranks ->) sample + fused n-step gather into ``out`` (live or shadow views)."""
        tree, ring = self.tree, self.ring
        if self.world_size > 1:
            if self.peer is not None:
                # the kernel waits for the latest put of every rank (this step's tail, or sync_shard_states)
                tree.sample_global_peer(self.peer, self.B_global, u, idx_out=out["idx"], weight_out=out["weight"],
                                        stratum_out=self.stratum)
            else:
                import torch.distributed as dist
                dist.all_gather_into_tensor(self.all_state.view(-1), tree.state, group=self.pg)
                self._mark(tag + "shard_states_gathered")
                tree.sample_global(self.world_size, self.rank, self.all_state, self.B_global, u,
                                   idx_out=out["idx"], weight_out=out["weight"], stratum_out=self.stratum)
        else:
            tree.sample(self.B, u=u, idx_out=out["idx"], weight_out=out["weight"])
        self._mark(tag + "sampled")
        # rows past the strata this rank owns have idx -1 / weight 0: skipped by gather and update
        ring.gather(out["idx"][:self.B_pad], out["obs"], out["next_obs"], out["reward"], out["gamma"],
                    out["nonterminal"], out["action"])

    def _prime(self):
        """Fill the shadow batch eagerly (first iteration, or after anything outside this object touched the
        buffer): uniforms from the in-kernel generator."""
        trace, self._trace = self._trace, None          # eager: not part of the replayed timeline
        try:
            self.sync_shard_states()
            self._sample_gather(None, self._shadow)
        finally:
            self._trace = trace
        self._primed = True
        self._seen_mutations = getattr(self.buffer, "_mutations", 0)

    def _body(self, refresh_table, draw, consume=False):
        tree, ring, agent, b = self.tree, self.ring, self.agent, self.buffer
        u = None if draw else self.u            # None: uniforms are drawn inside the sampling kernel
        u_sel = consume and self._u_in_block
        mark = self._mark
        mark("start")
        if self.prefetch:
            self._live_arena.copy_(self._shadow_arena)          # batch sampled on the previous iteration's tail
        else:
            if u_sel:
                self.ingest.select_uniforms(self.u, after_counter_inc=False)
            self._sample_gather(u, {"idx": self.idx, "weight": self.weight, "obs": b._obs, "next_obs": b._next_obs,
                                    "reward": b._reward, "gamma": b._gamma, "nonterminal": b._nonterminal,
                                    "action": b._action})
        mark("batch_ready")
        idx, w = self.idx[:self.B_pad], self.weight[:self.B_pad]
        # The priority write-back (learner.py:120) needs the new TD errors only, not the optimizer step: it runs on
        # a second stream -- a parallel branch of the captured graph -- while backward / (exchange) / Adam proceed.
        cur = torch.cuda.current_stream(self.device)
        from .agents import ops as _ops
        self._side = _ops.fork_stream(self.device, "writeback")

        def write_back(td):
            self.td = td
            mark("loss_ready")
            self._side.wait_stream(cur)
            side2 = _ops.fork_stream(self.device, "ingest") if consume else None
            if consume:
                # the ring scatter touches no tree array: a third branch, beside the priority write-back
                side2.wait_stream(cur)
                with torch.cuda.stream(side2):
                    self.ingest.consume_ring()
                    mark("tail:ring_ingested")
            with torch.cuda.stream(self._side):
                tree.update_priority(idx, td, sorted=self.sorted)      # |td| is taken inside the kernel
                mark("tail:priorities_written")
                if consume:
                    self.ingest.consume_tree()         # default priorities of the new steps, after the write-back
                    self._side.wait_stream(side2)
                if self.peer is not None:
                    self.peer.state_put(tree.state)            # this shard's new state -> every rank; nobody waits here
                    mark("tail:state_put")
                if self.prefetch:
                    if u_sel:
                        self.ingest.select_uniforms(self.u, after_counter_inc=True)
                    self._sample_gather(u, self._shadow, tag="tail:")      # next iteration's batch
                    mark("tail:next_batch_ready")

        # weight-gradient branches rejoin before the optimizer, not inside backward (agents/ops.py: _JOINS)
        _ops.defer_joins(self._defer_mode)
        try:
            dl, ql, total, td = agent._loss_and_backward(self.batch, w, agent.target_model, after_loss=write_back)
        finally:
            wgrad_ptrs = _ops.finish_deferred(self.device)
        if self._defer_mode == 1:
            opt = agent.optimizer
            params = opt.params if hasattr(opt, "params") else [p for g in opt.param_groups for p in g["params"]]
            held = {p.grad.data_ptr() for p in params if p.grad is not None}
            self._defer_ok = all(q in held for q in wgrad_ptrs)
        agent._static_distribution_loss, agent._static_q_loss, agent._static_total_loss = dl, ql, total
        mark("backward_done")
        agent._optimizer_step(refresh_table=refresh_table)
        mark("optimizer_done")
        if self.loss_host is not None and total is not None:
            # device -> host read of the step's result as a node of the same graph (pinned scalar)
            self.loss_host.copy_(total.detach(), non_blocking=True)
        cur.wait_stream(self._side)
        mark("end")
        return total

    # ---- timeline marks (measurement only; nsys is not available on the boxes) ---------------------------------------
    def enable_trace(self, max_marks=64):
        """Insert device timestamps (pb_stamp_time: one single-thread launch each) at the phase boundaries of the
        step, on whichever graph branch reaches them; the graph is re-captured.  ``trace_report()`` reads them."""
        self._trace = {"buf": torch.zeros(max_marks, dtype=torch.int64, device=self.device), "names": {}}
        from .agents import ops as _ops
        opt = self.agent.optimizer
        if isinstance(opt, FlatAdam):
            opt._mark = self._mark
        _ops.TRACE_MARK = self._mark                  # forward / backward phases inside the agent
        self.graph, self._primed = None, False

    def disable_trace(self):
        from .agents import ops as _ops
        self._trace = None
        if isinstance(self.agent.optimizer, FlatAdam):
            self.agent.optimizer._mark = None
        _ops.TRACE_MARK = None
        self.graph, self._primed = None, False

    def _mark(self, name):
        tr = self._trace
        if tr is None:
            return
        names = tr["names"]
        i = names.setdefault(name, len(names))
        if i >= tr["buf"].numel():
            raise _lib.PbError("more timeline marks than enable_trace(max_marks=%d)" % tr["buf"].numel())
        _lib.check(self._lib.pb_stamp_time(tr["buf"].data_ptr() + 8 * i,
                                           torch.cuda.current_stream(self.device).cuda_stream), "pb_stamp_time")

    def trace_report(self):
        """{mark: nanoseconds since "start"} of the LAST replay (synchronises)."""
        tr = self._trace
        if tr is None:
            raise _lib.PbError("enable_trace() first")
        torch.cuda.synchronize(self.device)
        t = tr["buf"].cpu().tolist()
        t0 = t[tr["names"]["start"]]
        return {name: t[i] - t0 for name, i in sorted(tr["names"].items(), key=lambda kv: kv[1])}

    def plan_ingest(self, ingest, u=None):
        """Host half of a fused ingest without the copy: plans the links of the next ``len(ingest[0])`` steps and returns
        the staged block (pinned uint8 tensor; the fp64 uniforms ``u`` of that iteration ride in it).  Blocks must be fed
        back IN ORDER through ``step(ingest_block=...)`` -- e.g. after parking them in HBM (bench.py's resident leg)."""
        n = len(ingest[0])
        if self.ingest is None or self.ingest.n != n:
            from .experience.ring import FusedIngest
            self.ingest = FusedIngest(self.ring, self.tree, n, n_uniforms=self.u.numel())
        return self.ingest.plan_block(*ingest, u=None if u is None else u.numpy() if isinstance(u, torch.Tensor) else u)

    def step(self, u=None, ingest=None, ingest_block=None):
        """Run one iteration.  ``u`` (optional): fp64 uniforms (device or pinned-host tensor, B_global
        values) used instead of the device Philox generator (with ``prefetch`` they drive the sampling that happens
        during this call, i.e. the NEXT iteration's batch).  ``ingest`` (optional): a tuple
        (stream_ids, obs, action, reward, done, trunc, next_obs) of a FIXED number of new steps per call; their
        scatter into the ring and default priorities run inside the step graph, after the priority write-back and
        concurrently with backward / Adam (FusedIngest); they are sampleable from the next iteration on."""
        self.buffer._flush()
        main = torch.cuda.current_stream(self.device).cuda_stream
        if ingest_block is not None:
            # a block planned by plan_ingest (uniforms inside), resident on the device: D2D into the staging slot
            if self.ingest is None:
                raise _lib.PbError("plan_ingest() first")
            parity = self.ingest.stage_device(ingest_block, main)
            draw, consume, self._u_in_block = False, True, True
        else:
            draw = u is None
            # host uniforms + fused ingest: the uniforms ride in the ingest's staging block (one H2D copy per iteration)
            # and are picked inside the graph by the replay counter
            u_in_block = (not draw) and ingest is not None and isinstance(u, torch.Tensor) and u.device.type == "cpu" \
                and u.dtype == torch.float64 and u.numel() == self.u.numel()
            if not draw and not u_in_block:
                if u.device.type == "cpu" and u.dtype == torch.float64 and u.is_contiguous() and u.numel() == self.u.numel():
                    # host uniforms (pinned): one raw async copy on the step's stream
                    _lib.check(self._lib.pb_copy_h2d_async(self.u.data_ptr(), u.data_ptr(), 8 * self.u.numel(), main),
                               "pb_copy_h2d_async")
                else:
                    self.u.copy_(u, non_blocking=True)
            consume, parity = ingest is not None, None
            if consume:
                n = len(ingest[0])
                if self.ingest is None or self.ingest.n != n:
                    from .experience.ring import FusedIngest
                    self.ingest = FusedIngest(self.ring, self.tree, n, n_uniforms=self.u.numel())
                parity = self.ingest.stage(*ingest, main_stream=main, u=u.numpy() if u_in_block else None)
            self._u_in_block = u_in_block
        # the captured kernels hold the ring descriptor and beta BY VALUE: a grown aux pool (ring.generation) or a
        # new beta (learner.py:105-107 writes _sampler._beta every iteration) re-captures
        key = (draw, consume, self._u_in_block, self.ring.generation, float(self.tree._beta))
        if self.use_cuda_graph and (self.graph is None or key != self._graph_key):
            if self.graph is not None and key[3] != self._graph_key[3]:
                torch.cuda.synchronize(self.device)
            self._capture(draw, consume)
            self._primed = False                            # the warm-up iterations sampled into the shadow batch
        if self.prefetch and (not self._primed or getattr(self.buffer, "_mutations", 0) != self._seen_mutations):
            self._prime()
        elif self.peer is not None and (not self._states_synced
                                        or getattr(self.buffer, "_mutations", 0) != self._seen_mutations):
            self.sync_shard_states()
            self._seen_mutations = getattr(self.buffer, "_mutations", 0)
        if not self.use_cuda_graph:
            total = self._body(refresh_table=True, draw=draw, consume=consume)
        else:
            self.graph.replay()
            total = self.agent._static_total_loss
        if consume:
            self.ingest.mark_consumed(parity, main)
        self.agent.n_updates += 1
        return total

    def enable_loss_readback(self):
        """Every following step also copies its total loss into ``self.loss_host`` (pinned fp32 scalar): the
        device -> host read is part of the step graph; synchronise before reading it on the host."""
        if self.loss_host is None:
            self.loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
            self.graph = None                      # recapture with the copy node
        return self.loss_host

    def copy_loss_to(self, host_scalar):
        """Asynchronous device -> host read of the last step's total loss into a pinned fp32 scalar."""
        t = self.agent._static_total_loss
        _lib.check(self._lib.pb_copy_d2h_async(host_scalar.data_ptr(), t.data_ptr(), 4,
                                               torch.cuda.current_stream(self.device).cuda_stream), "pb_copy_d2h_async")

    def _capture(self, draw, consume=False):
        opt = self.agent.optimizer
        flat = isinstance(opt, FlatAdam)
        # drop every reference to autograd graphs built on another stream (an eager update leaves its
        # loss tensors on the agent): their AccumulateGrad nodes would tie the capture to that stream
        ag = self.agent
        ag._static_total_loss = ag._static_distribution_loss = ag._static_q_loss = None
        self.td = None
        opt.zero_grad(set_to_none=True)
        # warm-up on a side stream; it must neither train nor disturb the priorities
        snap = opt.snapshot() if flat else None
        tree_snap = self.tree.snapshot()
        u_snap = self.u.clone()
        rng = torch.cuda.get_rng_state(self.device)
        for m in (ag.model, ag.target_model):                   # the IQN heads' own generators (quantile draws)
            d = getattr(m, "distribution_model", None) if m is not None else None
            if d is not None and hasattr(d, "_rng_state"):
                d._rng_state()
        q_rng = ag.quantile_rng_snapshot()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for it in range(3):
                # first iteration: probe whether the weight-gradient joins can move to the optimizer (ops._JOINS)
                self._defer_mode = 1 if it == 0 else (2 if self._defer_ok else 0)
                self._body(refresh_table=True, draw=draw)
        torch.cuda.current_stream(self.device).wait_stream(side)
        if flat:
            opt.restore(snap)
        self.tree.restore(tree_snap)
        self.u.copy_(u_snap)
        torch.cuda.set_rng_state(rng, self.device)
        ag.quantile_rng_restore(q_rng)
        self._states_synced = False                         # the warm-up's exchanges carried warm-up tree states
        self._graph_key = (draw, consume, self._u_in_block, self.ring.generation, float(self.tree._beta))
        opt.zero_grad(set_to_none=True)
        self.graph = None                                   # release the previous graph's pool before capturing anew
        self.graph = torch.cuda.CUDAGraph()
        before = _lib.launch_count()
        try:
            with torch.cuda.graph(self.graph):
                self._body(refresh_table=False, draw=draw, consume=consume)
        finally:
            self._defer_mode = 0                                # eager steps join in place
        self.launches_per_step = _lib.launch_count() - before
        if flat:
            opt.refresh_grad_table()
