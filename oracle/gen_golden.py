"""Generate tests/golden/*.npz by running the REFERENCE's own code (imported from /root/reference).

Run here (the build container), never on the GPU box -- /root/reference does not travel:
    python -m oracle.gen_golden
What is frozen:
  agent_*.npz        reference CompositeModel.get_losses + Agent._update_without_cuda_graph
                     (prism/agents/*) on seeded weights / batches / injected taus
  ids.npz            reference IDSActionSelector / GreedyActionSelector on random + tie cases
  nstep_gather_*.npz reference TimestepBuffer._timesteps_to_batch (prism/experience/timestep_buffer.py)
                     driven through a stub `tensordict` and a fake torchrl ring, on scripted
                     multi-stream trajectories (done / truncated / in-flight tail / ring wrap)
  wire.npz           reference Timestep.serialize / deserialize_linked_list (prism/experience/timestep.py), the
                     MessageSerializer envelope with the "NONE" compressor (async_components/compression_methods.py;
                     lz4, msgpack_numpy and redis are absent here and stubbed at import) and the batch flat-list
                     format (async_components/async_experience_buffer.py) on a scripted multi-stream trace
  ref_checkpoint/    reference TimestepBuffer.save (prism/experience/timestep_buffer.py:259-302) of a wrapped 48-slot
                     ring over the same kind of trace: experience_buffer/timesteps.pkl (+ ref_checkpoint.npz: the
                     script and the stored ids) -- input of the checkpoint reader test
  per_tree.npz       ORACLE-generated (parity unpinned: torchrl is absent) -- freezes the restated
                     tree/sampler arithmetic so the C oracle and the CUDA path cannot drift apart
"""
import io
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, "tests", "golden")
MAX_FILE_BYTES = 1 << 20          # no file in the repository is larger: bigger fixtures are stored in parts
REF = "/root/reference"


def _import_reference():
    if not os.path.isdir(REF):
        raise SystemExit("reference tree not present; golden vectors can only be generated in the build container")
    td = types.ModuleType("tensordict")

    class TensorDict(dict):
        def __init__(self, data=None, batch_size=None, device=None):
            super().__init__(data or {})

    td.TensorDict = TensorDict
    sys.modules.setdefault("tensordict", td)
    if REF not in sys.path:
        sys.path.insert(0, REF)


# --------------------------------------------------------------------------------------------
# agent fixtures
# --------------------------------------------------------------------------------------------
AGENT_CASES = {
    # name: (config overrides on the reference DEFAULT_CONFIG, obs_shape, n_actions, B)
    "agent_ids_iqn_ln_target": (dict(
        embedding_model_type="minatar_cnn", frame_stack_size=1, use_iqn=True, use_ids=True, use_layer_norm=True,
        use_target_network=True, use_double_q_learning=False, iqn_n_current_state_quantile_samples=8,
        iqn_n_next_state_quantile_samples=8, iqn_quantile_samples_per_action=8, iqn_quantile_model_feature_dim=32,
        iqn_quantile_model_layers=1, ids_n_q_heads=3, ids_q_head_feature_dim=16, ids_n_q_head_model_layers=2,
        learning_rate=1e-3, adam_epsilon=0.0003125), (10, 10, 4), 3, 6),
    "agent_ids_iqn_double": (dict(
        embedding_model_type="ffnn", embedding_model_num_layers=1, embedding_model_final_dim=24,
        embedding_model_layer_sizes=24, frame_stack_size=1, use_iqn=True, use_ids=True, use_layer_norm=True,
        use_target_network=True, use_double_q_learning=True, iqn_n_current_state_quantile_samples=16,
        iqn_n_next_state_quantile_samples=12, iqn_quantile_samples_per_action=20, iqn_quantile_model_feature_dim=32,
        iqn_quantile_model_layers=1, ids_n_q_heads=10, ids_q_head_feature_dim=16, ids_n_q_head_model_layers=2,
        learning_rate=1e-3), (12,), 5, 9),
    "agent_dqn_double": (dict(
        embedding_model_type="minatar_cnn", frame_stack_size=1, use_iqn=False, use_ids=False, use_dqn=True,
        use_e_greedy=True, use_layer_norm=False, use_target_network=True, use_double_q_learning=True,
        dqn_n_model_layers=2, dqn_n_model_feature_dim=16, learning_rate=2.5e-4, adam_epsilon=0.0003125),
        (10, 10, 6), 4, 8),
    "agent_iqn_self": (dict(
        embedding_model_type="ffnn", embedding_model_num_layers=2, embedding_model_final_dim=20,
        embedding_model_layer_sizes=28, frame_stack_size=1, use_iqn=True, use_ids=False, use_dqn=False,
        use_layer_norm=False, use_target_network=False, use_double_q_learning=False,
        iqn_n_current_state_quantile_samples=8, iqn_n_next_state_quantile_samples=8,
        iqn_quantile_samples_per_action=8, iqn_quantile_model_feature_dim=16, iqn_quantile_model_layers=0,
        learning_rate=1e-3), (7,), 4, 5),
}


def target_transform(t):
    """Deterministic perturbation that makes the target network differ from the online one."""
    return t * 0.97 + 0.003


def make_batch(rng, B, obs_shape, n_actions, binary_obs):
    if binary_obs:
        obs = (rng.random((B, 1) + tuple(obs_shape)) < 0.2).astype(np.float32)
        nobs = (rng.random((B, 1) + tuple(obs_shape)) < 0.2).astype(np.float32)
    else:
        obs = rng.standard_normal((B, 1) + tuple(obs_shape)).astype(np.float32)
        nobs = rng.standard_normal((B, 1) + tuple(obs_shape)).astype(np.float32)
    return {
        "observation": obs, "next_observation": nobs,
        "reward": rng.standard_normal((B, 1)).astype(np.float32) * 2.0,
        "nonterminal": (rng.random((B, 1)) < 0.8),
        "gamma": np.where(rng.random((B, 1)) < 0.7, 0.99 ** 3, 0.99 ** 2).astype(np.float32),
        "action": rng.integers(0, n_actions, (B, 1)).astype(np.int64),
    }


def save_parts(name, out, groups):
    """GOLD/<name>.npz; when that would exceed MAX_FILE_BYTES, the keys "<group>.*" of each group go to
    GOLD/<name>.<group>.npz instead (tests/helpers.py load_golden merges the parts back)."""
    whole = io.BytesIO()
    np.savez_compressed(whole, **out)
    if whole.tell() > MAX_FILE_BYTES:
        for g in groups:
            part = {k: out.pop(k) for k in list(out) if k.startswith(g + ".")}
            np.savez_compressed(os.path.join(GOLD, "%s.%s.npz" % (name, g)), **part)
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)


def to_torch_batch(b):
    return {"observation": torch.from_numpy(b["observation"]),
            "next": {"observation": torch.from_numpy(b["next_observation"]), "reward": torch.from_numpy(b["reward"])},
            "nonterminal": torch.from_numpy(b["nonterminal"]), "gamma": torch.from_numpy(b["gamma"]),
            "action": torch.from_numpy(b["action"])}


def gen_agent_case(name, overrides, obs_shape, n_actions, B):
    from prism.config import DEFAULT_CONFIG, Config
    from prism.factory import agent_factory
    cfg = Config(**DEFAULT_CONFIG.__dict__)
    cfg.device = "cpu"
    cfg.use_cuda_graph = False
    for k, v in overrides.items():
        setattr(cfg, k, v)
    torch.manual_seed(1234)
    agent = agent_factory.build_agent(cfg, obs_shape, n_actions)
    if agent.target_model is not None:
        with torch.no_grad():
            for p in agent.target_model.parameters():
                p.copy_(target_transform(p))
    rng = np.random.default_rng(abs(hash(name)) % (2 ** 31))
    rng = np.random.default_rng(sum(ord(c) for c in name))
    batch = make_batch(rng, B, obs_shape, n_actions, binary_obs=(cfg.embedding_model_type == "minatar_cnn"))
    per_w = (rng.random(B) * 0.9 + 0.1).astype(np.float32)
    out = {"cfg_keys": np.array(list(overrides.keys())),
           "cfg_vals": np.array([repr(v) for v in overrides.values()]),
           "obs_shape": np.array(obs_shape), "n_actions": np.array(n_actions), "per_weights": per_w}
    for k, v in batch.items():
        out["batch." + k] = v
    for k, v in agent.model.state_dict().items():
        out["param." + k] = v.numpy().copy()

    # record the reference's own torch.rand draws so the other side can replay them
    draws = []
    real_rand = torch.rand

    def recording_rand(*a, **kw):
        t = real_rand(*a, **kw)
        draws.append(t.clone())
        return t

    torch.manual_seed(77)
    torch.rand = recording_rand
    try:
        td = agent._update_without_cuda_graph(to_torch_batch(batch), torch.from_numpy(per_w))
    finally:
        torch.rand = real_rand
    for i, t in enumerate(draws):
        out["tau.%d" % i] = t.numpy().reshape(-1)
    out["n_taus"] = np.array(len(draws))
    if agent._static_distribution_loss is not None:
        out["out.dist"] = agent._static_distribution_loss.detach().numpy()
    if agent._static_q_loss is not None:
        out["out.q"] = agent._static_q_loss.detach().numpy()
    out["out.td"] = td.detach().numpy()
    out["out.total"] = agent._static_total_loss.detach().numpy()
    gsq = 0.0
    for k, p in agent.model.named_parameters():
        # after clip_grad_norm_ the stored grads are already clipped: store them plus the clip-free norm
        out["grad_clipped." + k] = p.grad.numpy().copy()
        gsq += float(p.grad.double().square().sum())
    out["out.clipped_grad_norm"] = np.array(np.sqrt(gsq))
    for k, v in agent.model.state_dict().items():
        out["param_after." + k] = v.numpy().copy()

    # acting: IDS / greedy forward on fresh observations with recorded quantile draws
    if cfg.use_iqn:
        obs_act = batch["observation"][:, 0]
        draws.clear()
        torch.rand = recording_rand
        try:
            with torch.no_grad():
                q, z = agent.model(torch.from_numpy(obs_act), for_action=True)
                act = agent.forward(torch.from_numpy(obs_act))
        finally:
            torch.rand = real_rand
        # two forwards were run (model(...) then agent.forward): keep the draw of each
        out["act.tau_model"] = draws[0].numpy().reshape(-1)
        out["act.tau_agent"] = draws[1].numpy().reshape(-1)
        out["act.z"] = z.numpy()
        if q is not None:
            out["act.q"] = q.numpy()
        out["act.action"] = act.numpy()
    save_parts(name, out, ("grad_clipped", "param_after"))
    print("wrote", name, "params", sum(v.size for k, v in out.items() if k.startswith("param.")))


# --------------------------------------------------------------------------------------------
# IDS fixture
# --------------------------------------------------------------------------------------------
def gen_ids():
    from prism.agents.action_selectors import GreedyActionSelector, IDSActionSelector
    rng = np.random.default_rng(5)
    out = {}
    for tag, (N, A, K, Nq) in {"a": (64, 6, 10, 32), "b": (14, 18, 10, 200), "c": (33, 3, 10, 32)}.items():
        q = rng.standard_normal((N, A, K)).astype(np.float32)
        z = (rng.standard_normal((Nq, N, A)) * rng.random((1, N, A)) * 3).astype(np.float32)
        if tag == "c":
            q[0] = q[0, :1]            # every action identical -> exact tie, first index must win
            z[:, 0] = z[:, 0, :1]
        sel = IDSActionSelector(0.1, False, 1e-10, 0.25, 1.0, None)
        probs = sel.generate_action_probs(torch.from_numpy(z), torch.from_numpy(q), for_log=True)
        out[tag + ".q"], out[tag + ".z"] = q, z
        out[tag + ".action"] = sel.select_action(probs).numpy()
        out[tag + ".scores"] = sel.loggables["IDS Scores"].numpy()
        g = GreedyActionSelector()
        out[tag + ".greedy"] = g.select_action(g.generate_action_probs(None, torch.from_numpy(q))).numpy()
    np.savez_compressed(os.path.join(GOLD, "ids.npz"), **out)
    print("wrote ids")


# --------------------------------------------------------------------------------------------
# n-step / gather fixtures through the reference TimestepBuffer
# --------------------------------------------------------------------------------------------
def make_script(seed, n_streams, n_steps, obs_shape, p_done, p_trunc, n_actions=5):
    """A collector trace: for every completed step its stream, observation, action, reward, done,
    truncated, the observation that follows (next step's / reset) and the truncated final observation."""
    rng = np.random.default_rng(seed)
    sid = rng.integers(0, n_streams, n_steps).astype(np.int32)
    obs_elems = int(np.prod(obs_shape))
    cur_obs = rng.standard_normal((n_streams, obs_elems)).astype(np.float32)
    S = {"stream": sid, "obs": np.zeros((n_steps, obs_elems), np.float32),
         "next_obs": np.zeros((n_steps, obs_elems), np.float32),
         "final_obs": np.zeros((n_steps, obs_elems), np.float32),
         "action": rng.integers(0, n_actions, n_steps).astype(np.int32),
         "reward": np.round(rng.standard_normal(n_steps), 3).astype(np.float32),
         "done": (rng.random(n_steps) < p_done), "trunc": np.zeros(n_steps, bool)}
    S["trunc"] = (~S["done"]) & (rng.random(n_steps) < p_trunc)
    for t in range(n_steps):
        s = sid[t]
        S["obs"][t] = cur_obs[s]
        nxt = rng.standard_normal(obs_elems).astype(np.float32)
        S["next_obs"][t] = nxt
        S["final_obs"][t] = rng.standard_normal(obs_elems).astype(np.float32)
        cur_obs[s] = nxt
    return S


def gen_nstep_gather(name, frame_stack, capacity, n_steps, checkpoints, seed):
    from prism.experience.timestep import Timestep
    from prism.experience.timestep_buffer import TimestepBuffer
    from oracle.buffer_oracle import StreamLinker
    obs_shape = (3, 2)
    script = make_script(seed, n_streams=4, n_steps=n_steps, obs_shape=obs_shape, p_done=0.08, p_trunc=0.05)

    class FakeRing:
        """torchrl stand-in: list ring + caller-chosen indices."""

        def __init__(self, cap):
            self.cap, self.items, self.cursor, self._batch_size, self.next_indices = cap, [], 0, None, None

        def extend(self, lst):
            for it in lst:
                if self.cursor < len(self.items):
                    self.items[self.cursor] = it
                else:
                    self.items.append(it)
                self.cursor = (self.cursor + 1) % self.cap

        def sample(self, batch_size=None, return_info=False):
            ts = [self.items[i] for i in self.next_indices]
            return (ts, {"index": self.next_indices}) if return_info else ts

    ring = FakeRing(capacity)
    tb = TimestepBuffer(ring, frame_stack=frame_stack, device="cpu", n_step=3, gamma=0.99)
    ids = [0]

    def make_step():
        ids[0] += 1
        return Timestep(ids[0])

    linkers = {}
    out = {"capacity": np.array(capacity), "frame_stack": np.array(frame_stack), "obs_shape": np.array(obs_shape),
           "n_step": np.array(3), "gamma": np.array(0.99), "checkpoints": np.array(checkpoints)}
    for k, v in script.items():
        out["script." + k] = v
    for t in range(n_steps):
        s = int(script["stream"][t])
        obs = torch.from_numpy(script["obs"][t].reshape(obs_shape).copy())
        if s not in linkers:
            linkers[s] = StreamLinker(obs, make_step)
        done, trunc = bool(script["done"][t]), bool(script["trunc"][t])
        step = linkers[s].step(int(script["action"][t]), float(script["reward"][t]), done, trunc,
                               torch.from_numpy(script["next_obs"][t].reshape(obs_shape).copy()),
                               torch.from_numpy(script["final_obs"][t].reshape(obs_shape).copy()))
        tb.extend(step)
        if (t + 1) in checkpoints:
            n = len(ring.items)
            idx = list(range(n))
            ring.next_indices = idx
            tb._batch = None                   # fresh zeroed static batch: unfilled frame rows stay 0
            tb._cpu_obs_buffer = None
            batch = tb.sample(batch_size=n)
            tag = "cp%d." % (t + 1)
            out[tag + "index"] = np.array(idx)
            out[tag + "observation"] = batch["observation"].numpy().copy()
            out[tag + "next_observation"] = batch["next"]["observation"].numpy().copy()
            out[tag + "reward"] = batch["next"]["reward"].numpy().copy()
            out[tag + "nonterminal"] = batch["nonterminal"].numpy().copy()
            out[tag + "gamma"] = batch["gamma"].numpy().copy()
            out[tag + "action"] = batch["action"].numpy().copy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name)


# --------------------------------------------------------------------------------------------
# wire formats of the Redis transport, through the reference's own serializers
# --------------------------------------------------------------------------------------------
def _stub_wire_deps():
    """Modules the reference's async components import at module level but that are absent here.  Only code paths
    that never touch them are exercised (the "NONE" compressor; unbound tensor (de)serializers)."""
    class _Anything(types.ModuleType):
        def __getattr__(self, name):
            if name.startswith("__"):
                raise AttributeError(name)
            return type(name, (), {})

    for name in ("lz4", "lz4.frame", "redis", "torchrl", "torchrl.data", "torchrl.envs"):
        mod = _Anything(name)
        mod.__path__ = []
        sys.modules.setdefault(name, mod)
    mn = types.ModuleType("msgpack_numpy")
    mn.patch = lambda: None
    sys.modules.setdefault("msgpack_numpy", mn)


def gen_wire():
    import contextlib
    import io
    _stub_wire_deps()
    from prism.async_components.compression_methods import MessageSerializer
    from prism.async_components.async_experience_buffer import AsyncExperienceBuffer, AsyncExperienceBufferInterface
    from prism.experience.timestep import Timestep
    from oracle.buffer_oracle import StreamLinker
    obs_shape = (3, 2)
    n_steps, block = 90, 7
    script = make_script(21, n_streams=3, n_steps=n_steps, obs_shape=obs_shape, p_done=0.08, p_trunc=0.06)
    ser = MessageSerializer(compression_type="NONE")
    ids = [0]

    def make_step():
        ids[0] += 1
        return Timestep(ids[0])

    out = {"obs_shape": np.array(obs_shape), "block": np.array(block)}
    for k, v in script.items():
        out["script." + k] = v
    linkers, keep, pending, step_ids = {}, [], [], []
    waiting, n_blocks = {}, 0
    for t in range(n_steps):
        s = int(script["stream"][t])
        if s not in linkers:
            linkers[s] = StreamLinker(torch.from_numpy(script["obs"][t].reshape(obs_shape).copy()), make_step)
        step = linkers[s].step(int(script["action"][t]), float(script["reward"][t]), bool(script["done"][t]),
                               bool(script["trunc"][t]),
                               torch.from_numpy(script["next_obs"][t].reshape(obs_shape).copy()),
                               torch.from_numpy(script["final_obs"][t].reshape(obs_shape).copy()))
        keep.append(step)                      # the collector side keeps its steps alive (weak links)
        step_ids.append(step.id)
        pending.append(step)
        if len(pending) == block or t == n_steps - 1:
            serialized = []
            for ts in pending:
                serialized += ts.serialize()                               # redis_interface.py:113-116
            packed = ser.pack(serialized)
            tag = "block%d." % n_blocks
            out[tag + "packed"] = np.frombuffer(packed, dtype=np.uint8).copy()
            with contextlib.redirect_stdout(io.StringIO()):                # the reference prints per element
                complete, waiting = Timestep.deserialize_linked_list(ser.unpack(packed), waiting)
            out[tag + "released"] = np.array([ts.id for ts in complete], dtype=np.int64)
            out[tag + "waiting"] = np.array(sorted(waiting.keys()), dtype=np.int64)
            pending, n_blocks = [], n_blocks + 1
    out["n_blocks"] = np.array(n_blocks)
    out["step_ids"] = np.array(step_ids, dtype=np.int64)
    # a training batch through the reference's tensor (de)serializers (async_experience_buffer.py:76-96, 148-184)
    rng = np.random.default_rng(22)
    B = 5
    tensors = [torch.from_numpy(rng.standard_normal((B, 2, 3, 2)).astype(np.float32)),
               torch.from_numpy(rng.standard_normal((B, 2, 3, 2)).astype(np.float32)),
               torch.from_numpy(rng.standard_normal((B, 1)).astype(np.float32)),
               torch.from_numpy(rng.random((B, 1)) < 0.7),
               torch.from_numpy(np.full((B, 1), 0.99 ** 3, np.float32)),
               torch.from_numpy(rng.integers(0, 5, (B, 1)).astype(np.int64))]
    serialized = []
    for x in tensors:
        serialized += AsyncExperienceBuffer._serialize_tensor(None, x)
    out["batch.packed"] = np.frombuffer(ser.pack(serialized), dtype=np.uint8).copy()
    idx, flat = 0, ser.unpack(ser.pack(serialized))
    for k, x in enumerate(tensors):
        out["batch.in%d" % k] = x.numpy()
        back, idx = AsyncExperienceBufferInterface._deserialize_tensor(None, flat, idx)
        out["batch.out%d" % k] = back.numpy()
    np.savez_compressed(os.path.join(GOLD, "wire.npz"), **out)
    print("wrote wire")


def gen_ref_checkpoint():
    """The reference's own buffer checkpoint (timesteps.pkl) for the reader in prism_b200 (SURVEY 8f-3)."""
    from prism.experience.timestep import Timestep
    from prism.experience.timestep_buffer import TimestepBuffer
    from oracle.buffer_oracle import StreamLinker
    obs_shape, capacity, n_steps = (3, 2), 48, 70
    script = make_script(31, n_streams=3, n_steps=n_steps, obs_shape=obs_shape, p_done=0.08, p_trunc=0.06)

    class Dumps:
        def dumps(self, path):
            pass

    class FakeRing:
        """torchrl stand-in: ListStorage semantics of `_storage[i]` (a one-element list per slot)."""

        def __init__(self, cap):
            self.cap, self._storage, self.cursor, self._batch_size = cap, [], 0, None
            self._sampler, self._writer = Dumps(), Dumps()

        def extend(self, lst):
            for it in lst:
                if self.cursor < len(self._storage):
                    self._storage[self.cursor] = [it]
                else:
                    self._storage.append([it])
                self.cursor = (self.cursor + 1) % self.cap

    ring = FakeRing(capacity)
    tb = TimestepBuffer(ring, frame_stack=1, device="cpu", n_step=3, gamma=0.99)
    ids = [0]

    def make_step():
        ids[0] += 1
        return Timestep(ids[0])

    linkers, step_ids = {}, []
    for t in range(n_steps):
        s = int(script["stream"][t])
        if s not in linkers:
            linkers[s] = StreamLinker(torch.from_numpy(script["obs"][t].reshape(obs_shape).copy()), make_step)
        step = linkers[s].step(int(script["action"][t]), float(script["reward"][t]), bool(script["done"][t]),
                               bool(script["trunc"][t]),
                               torch.from_numpy(script["next_obs"][t].reshape(obs_shape).copy()),
                               torch.from_numpy(script["final_obs"][t].reshape(obs_shape).copy()))
        step_ids.append(step.id)
        tb.extend(step)
    out_dir = os.path.join(GOLD, "ref_checkpoint")
    tb.save(out_dir)
    out = {"obs_shape": np.array(obs_shape), "capacity": np.array(capacity), "step_ids": np.array(step_ids, dtype=np.int64),
           "stored_ids": np.array([slot[0].id for slot in ring._storage], dtype=np.int64)}
    for k, v in script.items():
        out["script." + k] = v
    np.savez_compressed(os.path.join(GOLD, "ref_checkpoint.npz"), **out)
    print("wrote ref_checkpoint")


# --------------------------------------------------------------------------------------------
# PER tree fixture (oracle-generated, parity unpinned)
# --------------------------------------------------------------------------------------------
def gen_per_tree():
    from oracle.per_oracle import OracleTree
    rng = np.random.default_rng(1)
    N = 1000
    t = OracleTree(N)
    t.extend(N)
    p0 = rng.exponential(1.0, N).astype(np.float32)
    t.update_priority(np.arange(N), p0)
    out = {"N": np.array(N), "p0": p0}
    u = rng.random((4, 64))
    for r in range(4):
        idx, w, mass, ps, pm = t.sample(u[r], 0.5, mode=r % 2)
        newp = rng.exponential(1.0, 64).astype(np.float32)
        out["r%d.u" % r], out["r%d.idx" % r], out["r%d.w" % r], out["r%d.mass" % r] = u[r], idx, w, mass
        out["r%d.psum" % r], out["r%d.pmin" % r], out["r%d.newp" % r] = np.float32(ps), np.float32(pm), newp
        t.update_priority(idx, newp)
        out["r%d.root" % r] = t.sum[1].copy()
        out["r%d.maxp" % r] = np.array(t.max_priority)
    out["final.sum"] = t.sum.copy()
    out["final.min"] = t.min.copy()
    np.savez_compressed(os.path.join(GOLD, "per_tree.npz"), **out)
    print("wrote per_tree")


def main():
    os.makedirs(GOLD, exist_ok=True)
    _import_reference()
    for name, (ov, shape, A, B) in AGENT_CASES.items():
        gen_agent_case(name, ov, shape, A, B)
    gen_ids()
    gen_nstep_gather("nstep_gather_fs1", 1, 64, 200, [10, 64, 130, 200], seed=11)
    gen_nstep_gather("nstep_gather_fs4", 4, 48, 160, [7, 48, 100, 160], seed=12)
    gen_per_tree()
    gen_wire()
    gen_ref_checkpoint()


if __name__ == "__main__":
    main()
