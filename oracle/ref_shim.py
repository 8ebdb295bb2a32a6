"""Import shim for the LIVE reference learner classes of a marlbase checkout (the directory that holds `marlbase/`, named by the
MARLBASE_SRC environment variable).

TEST INFRASTRUCTURE ONLY.  The reference's learner half imports cleanly once `gymnasium.spaces.flatdim`
(its only gymnasium use: marlbase/dqn/model.py:4, marlbase/ac/model.py:4) and stub `hydra` / `omegaconf` /
`imageio` modules exist (imports at marlbase/dqn/train.py:6,8,11).  The test suite never needs it: the fixture
generators (tests/golden/make_golden.py and the `make_*` functions of the test modules) use it to record what the
reference computes into the committed files under tests/golden/.
"""
from __future__ import annotations

import os
import sys
import types

REF_ROOT = os.environ.get("MARLBASE_SRC", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isdir(os.path.join(REF_ROOT, "marlbase"))


class Space:
    """Duck-typed stand-in for gymnasium Box / Discrete: `.shape` or `.n`."""

    def __init__(self, shape=None, n=None):
        self.shape, self.n = shape, n


def _flatdim(space):
    if getattr(space, "n", None) is not None:
        return int(space.n)
    if isinstance(space, (list, tuple)):
        return sum(_flatdim(s) for s in space)
    out = 1
    for d in space.shape:
        out *= int(d)
    return out


def load():
    """Returns a namespace with the reference modules: dqn_model, dqn_train, ac_model, utils, models."""
    if not available():
        raise RuntimeError("set MARLBASE_SRC to a directory that contains the marlbase package")
    if "gymnasium" not in sys.modules:
        gym = types.ModuleType("gymnasium")
        spaces = types.ModuleType("gymnasium.spaces")
        spaces.flatdim = _flatdim
        gym.spaces = spaces
        sys.modules["gymnasium"], sys.modules["gymnasium.spaces"] = gym, spaces
    if "hydra" not in sys.modules:
        sys.modules["hydra"] = types.ModuleType("hydra")
    if "omegaconf" not in sys.modules:
        oc = types.ModuleType("omegaconf")
        oc.DictConfig = dict
        oc.OmegaConf = object
        sys.modules["omegaconf"] = oc
    if "imageio" not in sys.modules:
        sys.modules["imageio"] = types.ModuleType("imageio")
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import importlib

    ns = types.SimpleNamespace()
    ns.dqn_model = importlib.import_module("marlbase.dqn.model")
    ns.dqn_train = importlib.import_module("marlbase.dqn.train")
    ns.ac_model = importlib.import_module("marlbase.ac.model")
    ns.utils = importlib.import_module("marlbase.utils.utils")
    ns.models = importlib.import_module("marlbase.utils.models")
    return ns


def dqn_cfg(**kw):
    d = dict(optimizer="Adam", lr=3e-4, gamma=0.99, grad_clip=1.0, target_update_interval_or_tau=200, double_q=True,
             standardise_returns=False)
    d.update(kw)
    return types.SimpleNamespace(**d)


def a2c_cfg(**kw):
    d = dict(optimizer="Adam", lr=3e-4, gamma=0.99, grad_clip=False, target_update_interval_or_tau=200, n_steps=5,
             entropy_coef=0.001, value_loss_coef=0.5, standardise_returns=False)
    d.update(kw)
    return types.SimpleNamespace(**d)


def net_cfg(parameter_sharing=False, layers=(128, 128), centralised=False):
    return types.SimpleNamespace(layers=list(layers), parameter_sharing=parameter_sharing, use_rnn=False,
                                 use_orthogonal_init=True, centralised=centralised)
