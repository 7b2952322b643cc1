"""Value squashing (Config.loss_squish_fn_id) without a GPU: the factories hand the right (squish, unsquish) pair to the
IQN head, the Q ensemble and the IDS selector, unknown ids stay unsquashed, foreign callables are refused, and the
oracle's fp32 forms of h / h^-1 hold 1e-6 relative against fp64."""
import dataclasses
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(squish_id, **kw):
    import prism_b200
    return dataclasses.replace(prism_b200.minatar_ids_iqn_config(device="cpu", iqn_quantile_model_feature_dim=16,
                                                                 ids_q_head_feature_dim=16, ids_n_q_heads=2, **kw),
                               loss_squish_fn_id=squish_id)


@pytest.mark.parametrize("squish_id,kind,pair", [("obs_look_further", 1, ("obs_look_further_squish", "obs_look_further_unsquish")),
                                                 ("symlog", 2, ("symlog", "symexp")),
                                                 (("symlog",), 2, ("symlog", "symexp"))])
def test_factories_wire_the_pair(squish_id, kind, pair):
    from prism_b200.agents import squish_functions as sf
    from prism_b200.factory import agent_factory, model_factory
    cfg = _cfg(squish_id)
    model = model_factory.create_model([10, 10, 4], 3, cfg)
    squish, unsquish = getattr(sf, pair[0]), getattr(sf, pair[1])
    for head in (model.distribution_model, model.q_function_model):
        assert head.squash == kind
        assert head.squish_function is squish and head.unsquish_function is unsquish
    ids = agent_factory._acting_policy(cfg)
    assert ids.squash == kind and ids.unsquish_function is unsquish


def test_dqn_heads_get_the_pair_and_greedy_selectors_do_not():
    import prism_b200
    from prism_b200.agents import action_selectors
    from prism_b200.factory import agent_factory, model_factory
    cfg = dataclasses.replace(prism_b200.minatar_dqn_per_config(device="cpu"), loss_squish_fn_id="symlog")
    model = model_factory.create_model([10, 10, 6], 4, cfg)
    assert model.distribution_model is None and model.q_function_model.squash == 2
    assert type(agent_factory._acting_policy(cfg)) in (action_selectors.EGreedyActionSelector,
                                                       action_selectors.GreedyActionSelector)


@pytest.mark.parametrize("squish_id", ["none", ("none",), "identity", "symlog2", "huber"])
def test_unknown_ids_stay_unsquashed(squish_id):
    from prism_b200.factory import agent_factory, model_factory
    cfg = _cfg(squish_id)
    model = model_factory.create_model([10, 10, 4], 3, cfg)
    for head in (model.distribution_model, model.q_function_model):
        assert head.squash == 0 and head.squish_function is None and head.unsquish_function is None
    ids = agent_factory._acting_policy(cfg)
    assert ids.squash == 0 and ids.unsquish_function is None


def test_foreign_callables_are_refused():
    import torch.nn as nn
    from prism_b200.agents import action_selectors, squish_functions as sf
    from prism_b200.agents.models import IQNModel, QEnsemble
    foreign = (torch.tanh, torch.atanh)
    mixed = (sf.symlog, sf.obs_look_further_unsquish)
    for pair in (foreign, mixed, (sf.symlog, None), (None, sf.symexp)):
        with pytest.raises(NotImplementedError, match="obs_look_further.*symlog"):
            IQNModel(8, 3, 16, False, squish_function=pair[0], unsquish_function=pair[1])
        with pytest.raises(NotImplementedError, match="obs_look_further.*symlog"):
            QEnsemble(8, 3, n_heads=2, use_layer_norm=False, q_loss_function=nn.MSELoss(reduction="none"),
                      squish_function=pair[0], unsquish_function=pair[1])
    with pytest.raises(NotImplementedError, match="obs_look_further.*symlog"):
        action_selectors.IDSActionSelector(0.1, False, 1e-10, 0.25, 0.0, unsquish_function=lambda x: x)
    with pytest.raises(NotImplementedError):                     # risk policies stay out of scope
        IQNModel(8, 3, 16, False, risk_policy=object())


def test_epsilon_is_the_same_on_both_sides_of_the_abi():
    import squash_oracle
    from prism_b200 import _lib
    header = open(os.path.join(ROOT, "include", "prism_b200.h")).read()
    m = re.search(r"#define PB_SQUASH_OLF_EPS\s+([0-9.eE+-]+)f", header)
    assert m and float(m.group(1)) == _lib.PB_SQUASH_OLF_EPS == squash_oracle.OBS_LOOK_FURTHER_EPS
    kinds = {k: int(v) for k, v in re.findall(r"#define (PB_SQUASH_[A-Z_]+)\s+(\d+)\n", header)}
    assert kinds == {"PB_SQUASH_NONE": _lib.PB_SQUASH_NONE, "PB_SQUASH_OBS_LOOK_FURTHER": _lib.PB_SQUASH_OBS_LOOK_FURTHER,
                     "PB_SQUASH_SYMLOG": _lib.PB_SQUASH_SYMLOG}


def fp64_squash(x, kind, inverse):
    """The definitions in fp64 (stable forms; fp64 has 29 bits to spare over the fp32 results they judge)."""
    x = np.asarray(x, np.float64)
    a, e = np.abs(x), 1e-2
    if kind == "obs_look_further":
        if not inverse:
            return np.sign(x) * a / (np.sqrt(a + 1) + 1) + e * x
        s = np.sqrt(1 + 4 * e * (a + 1 + e))
        tm1 = 2 * a / (s + 1 + 2 * e)
        return np.sign(x) * tm1 * (tm1 + 2)
    return np.sign(x) * (np.expm1(a) if inverse else np.log1p(a))


def log_grid(lo, hi, n=4001):
    mag = np.logspace(np.log10(lo), np.log10(hi), n).astype(np.float32)
    return np.concatenate([-mag[::-1], mag])


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("kind", ["obs_look_further", "symlog"])
def test_oracle_fp32_forms_hold_1e6_against_fp64(kind, inverse):
    from squash_oracle import squash, unsquash
    x = log_grid(1e-30, 80.0 if (kind == "symlog" and inverse) else 1e30)
    got = (unsquash if inverse else squash)(torch.from_numpy(x), kind).numpy()
    want = fp64_squash(x, kind, inverse)
    rel = np.abs(got.astype(np.float64) - want) / np.abs(want)
    assert rel.max() < 1e-6, (kind, inverse, float(rel.max()), float(x[rel.argmax()]))
