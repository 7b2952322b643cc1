"""Value squashing pairs (squish h, unsquish h^-1), at the reference's module path (prism/agents/squish_functions.py).

``Config.loss_squish_fn_id`` selects a pair: "obs_look_further" (Pohlen et al. 2018, "Observe and Look Further":
h(x) = sign(x) (sqrt(|x| + 1) - 1) + eps x, eps = 1e-2) or "symlog" (h = symlog, h^-1 = symexp); any other id means no
squashing.  The functions themselves are one elementwise kernel each (pb_value_squash); the models never call them:
IQNModel, QEnsemble and IDSActionSelector recognise a pair by identity and pass its kind (PB_SQUASH_*) to their fused
kernels, which apply h / h^-1 where the targets are built and where IDS reads its inputs.  A callable that is not one of
these functions is refused: there is no per-element fallback.
"""
from .. import _lib
from . import ops


def obs_look_further_squish(x):
    return ops.value_squash(x, _lib.PB_SQUASH_OBS_LOOK_FURTHER)


def obs_look_further_unsquish(x):
    return ops.value_squash(x, _lib.PB_SQUASH_OBS_LOOK_FURTHER, inverse=True)


def symlog(x):
    return ops.value_squash(x, _lib.PB_SQUASH_SYMLOG)


def symexp(x):
    return ops.value_squash(x, _lib.PB_SQUASH_SYMLOG, inverse=True)


SQUISH_FUNCTIONS = {
    "obs_look_further": (obs_look_further_squish, obs_look_further_unsquish),
    "symlog": (symlog, symexp),
}
_KIND = {"obs_look_further": _lib.PB_SQUASH_OBS_LOOK_FURTHER, "symlog": _lib.PB_SQUASH_SYMLOG}


def get_squish_functions(squish_fn_id):
    """(squish, unsquish) of a ``loss_squish_fn_id``; (None, None) for "none" and any id that is not a squashing."""
    return SQUISH_FUNCTIONS.get(squish_fn_id, (None, None))


def _refuse(fn):
    raise NotImplementedError("value squashing function %r is not supported: the fused kernels implement %s"
                              % (fn, " and ".join('"%s"' % k for k in SQUISH_FUNCTIONS)))


def squash_kind(squish_function, unsquish_function):
    """PB_SQUASH_* of a (squish, unsquish) pair; (None, None) is PB_SQUASH_NONE."""
    if squish_function is None and unsquish_function is None:
        return _lib.PB_SQUASH_NONE
    for name, pair in SQUISH_FUNCTIONS.items():
        if (squish_function, unsquish_function) == pair:
            return _KIND[name]
    _refuse((squish_function, unsquish_function))


def unsquash_kind(unsquish_function):
    """PB_SQUASH_* of an unsquish function alone (IDSActionSelector); None is PB_SQUASH_NONE."""
    if unsquish_function is None:
        return _lib.PB_SQUASH_NONE
    for name, (_, unsquish) in SQUISH_FUNCTIONS.items():
        if unsquish_function is unsquish:
            return _KIND[name]
    _refuse(unsquish_function)
