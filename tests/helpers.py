"""Shared test plumbing: golden fixtures, config reconstruction, script replay."""
import ast
import glob
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    """golden/<name>.npz merged with its parts golden/<name>.<group>.npz (a fixture over 1 MB is stored split)."""
    out = {}
    for path in [os.path.join(GOLD, name + ".npz")] + sorted(glob.glob(os.path.join(GOLD, name + ".*.npz"))):
        out.update(np.load(path, allow_pickle=False))
    return out


def cfg_from_fixture(fx, device):
    """prism_b200.Config with the reference DEFAULT_CONFIG defaults + the fixture's overrides."""
    from prism_b200.config import Config
    kw = {k: ast.literal_eval(v) for k, v in zip(fx["cfg_keys"].tolist(), fx["cfg_vals"].tolist())}
    cfg = Config(**kw)
    cfg.device = device
    cfg.use_cuda_graph = False
    return cfg


def fixture_state_dict(fx, prefix="param."):
    return {k[len(prefix):]: torch.from_numpy(v.copy()) for k, v in fx.items() if k.startswith(prefix)}


def fixture_batch(fx, device="cpu"):
    from prism_b200.experience.batch import Batch
    t = lambda k: torch.from_numpy(fx["batch." + k].copy()).to(device)
    return Batch({"observation": t("observation"),
                  "next": {"observation": t("next_observation"), "reward": t("reward")},
                  "nonterminal": t("nonterminal"), "gamma": t("gamma"), "action": t("action")})


def fixture_taus(fx):
    return [fx["tau.%d" % i] for i in range(int(fx["n_taus"]))]


def target_transform(t):
    return t * 0.97 + 0.003


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    denom = max(np.abs(b).max(), 1e-12)
    return float(np.abs(a - b).max() / denom)


def script_from_fixture(fx):
    return {k[len("script."):]: v for k, v in fx.items() if k.startswith("script.")}


def replay_script_oracle(fx, upto=None, buf=None, linkers=None, start=0):
    """Feed the fixture's collector trace into the oracle buffer (linked Step objects)."""
    from oracle.buffer_oracle import OracleTimestepBuffer, Step, StreamLinker
    S = script_from_fixture(fx)
    obs_shape = tuple(fx["obs_shape"].tolist())
    if buf is None:
        buf = OracleTimestepBuffer(int(fx["capacity"]), batch_size=4, frame_stack=int(fx["frame_stack"]),
                                   n_step=int(fx["n_step"]), gamma=float(fx["gamma"]))
        linkers = {}
    n = len(S["stream"]) if upto is None else upto
    ids = [0]

    def make_step():
        ids[0] += 1
        return Step(ids[0])

    for t in range(start, n):
        s = int(S["stream"][t])
        if s not in linkers:
            linkers[s] = StreamLinker(S["obs"][t].reshape(obs_shape).copy(), make_step)
        step = linkers[s].step(int(S["action"][t]), float(S["reward"][t]), bool(S["done"][t]), bool(S["trunc"][t]),
                               S["next_obs"][t].reshape(obs_shape).copy(), S["final_obs"][t].reshape(obs_shape).copy())
        buf.extend(step)
    return buf, linkers


def script_successor_obs(S, t):
    """Observation that follows step t of the trace: truncated -> final observation, else next/reset obs."""
    return S["final_obs"][t] if S["trunc"][t] else S["next_obs"][t]


class FakeRedis(object):
    """The redis-py calls RedisInterface uses, in memory."""

    def __init__(self):
        self.kv, self.lists = {}, {}

    def get(self, k):
        return self.kv.get(k)

    def set(self, k, v):
        self.kv[k] = v.encode() if isinstance(v, str) else (str(v).encode() if isinstance(v, (int, float)) else v)

    def lpush(self, k, v):
        self.lists.setdefault(k, []).insert(0, v)

    def lrange(self, k, a, b):
        lst = self.lists.get(k, [])
        return lst[a:] if b == -1 else lst[a:b + 1]

    def ltrim(self, k, a, b):
        lst = self.lists.get(k, [])
        self.lists[k] = lst[a:] if b == -1 else lst[a:b + 1]

    def delete(self, k):
        self.lists.pop(k, None)
        self.kv.pop(k, None)

    def incrby(self, k, n):
        self.kv[k] = str(int(self.kv.get(k, b"0")) + n).encode()

    def flushall(self):
        self.kv, self.lists = {}, {}

    def pipeline(self):
        outer = self

        class Pipe(object):
            def __init__(self):
                self.calls = []

            def __getattr__(self, name):
                return lambda *a: self.calls.append((name, a))

            def execute(self):
                return [getattr(outer, name)(*a) for name, a in self.calls]

        return Pipe()
