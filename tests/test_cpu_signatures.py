"""Constructor / function signatures of the mirrors against the reference's: same parameter names in the same order
with the same default values (so that code relying on positional arguments or on defaults behaves identically); the
mirrors may only append keyword parameters of their own.  `device` defaults differ on purpose (the reference defaults
to "cpu", this package has no CPU path) and logger defaults are instances.  The reference's signatures are stored in
tests/golden/reference_surface.npz (record_reference below, run by oracle/record_reference.py)."""
import inspect

import numpy as np
import pytest

from tests import helpers

ALGOS = ["BC", "BCQL", "CPQ", "BEARL", "CDT", "COptiDICE"]
DATASET = ["TransitionDataset", "SequenceDataset"]
FUNCTIONS = ["process_bc_dataset", "seed_all", "get_cfg_value", "load_config_and_model", "to_string", "auto_name"]
LAMBDA_AT = (0.0, 1.0, 37.5)      # where a callable default (SequenceDataset's cost_transform) is compared


class Recorded:
    """A stored parameter of a reference signature: name, and default (inspect.Parameter.empty when it has none)."""

    def __init__(self, name, tag, value):
        self.name = name
        self.default = {"empty": inspect.Parameter.empty, "value": value, "object": object()}[tag] \
            if tag != "callable" else CallableAt(value)


class CallableAt(tuple):
    """A callable default, known by its values at LAMBDA_AT."""


def record_reference(osrl):
    import osrl.common.dataset as rd
    import osrl.common.exp_util as re_
    ra = osrl.algorithms
    objs = {}
    for name in ALGOS:
        objs[name] = getattr(ra, name).__init__
        objs[name + "Trainer"] = getattr(ra, name + "Trainer").__init__
        for meth in ("train_one_step", "evaluate", "rollout"):
            objs[f"{name}Trainer.{meth}"] = getattr(getattr(ra, name + "Trainer"), meth)
    for name in DATASET:
        objs[name] = getattr(rd, name).__init__
    for name in FUNCTIONS:
        objs[name] = getattr(rd, name, None) or getattr(re_, name)

    def param(p):
        d = p.default
        if d is inspect.Parameter.empty:
            return (p.name, "empty", None)
        if callable(d) and getattr(d, "__name__", "") == "<lambda>":
            return (p.name, "callable", [d(x) for x in LAMBDA_AT])
        if d is None or isinstance(d, (bool, int, float, str, list, tuple, dict)):
            return (p.name, "value", d)
        return (p.name, "object", type(d).__name__)     # logger instances: not compared

    return {k: [param(p) for p in inspect.signature(f).parameters.values() if p.name != "self"] for k, f in objs.items()}


@pytest.fixture(scope="module")
def ref():
    return {k: [Recorded(*p) for p in v] for k, v in helpers.load_pin("surface").items()}


def _same(a, b):
    if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        return np.array_equal(a, b)
    if isinstance(a, CallableAt):
        return callable(b) and all(b(x) == y for x, y in zip(LAMBDA_AT, a))
    return a == b and type(a) is type(b)


def _check(name, theirs, ours, skip=("device", "logger")):
    pt = theirs
    po = list(inspect.signature(ours).parameters.values())
    po = [p for p in po if p.name != "self"]
    assert [p.name for p in po[:len(pt)]] == [p.name for p in pt], f"{name}: parameter names / order"
    for t, o in zip(pt, po):
        if t.name in skip:
            continue
        if t.default is inspect.Parameter.empty:
            continue    # required in the reference: the mirror may relax it (env=None for the device-resident path)
        assert o.default is not inspect.Parameter.empty, f"{name}.{t.name}: default dropped"
        if True:
            assert _same(t.default, o.default), f"{name}.{t.name}: default {o.default!r} vs reference {t.default!r}"
    for extra in po[len(pt):]:
        assert extra.kind in (extra.VAR_KEYWORD, extra.KEYWORD_ONLY) or extra.default is not inspect.Parameter.empty, \
            f"{name}: extra parameter {extra.name} needs a default"


@pytest.mark.parametrize("name", ALGOS + [a + "Trainer" for a in ALGOS])
def test_algorithm_signatures(ref, name):
    import osrl_b200.algorithms as mine
    _check(name, ref[name], getattr(mine, name).__init__)


@pytest.mark.parametrize("name", DATASET)
def test_dataset_signatures(ref, name):
    import osrl_b200.common.dataset as mine
    _check(name, ref[name], getattr(mine, name).__init__)


@pytest.mark.parametrize("name", FUNCTIONS)
def test_function_signatures(ref, name):
    import osrl_b200.common.dataset as md
    import osrl_b200.common.exp_util as me
    ours = getattr(md, name, None) or getattr(me, name)
    _check(name, ref[name], ours)


@pytest.mark.parametrize("name", ALGOS)
def test_trainer_methods_exist_with_reference_signatures(ref, name):
    import osrl_b200.algorithms as mine
    o = getattr(mine, name + "Trainer")
    for meth in ("train_one_step", "evaluate", "rollout"):
        _check(f"{name}Trainer.{meth}", ref[f"{name}Trainer.{meth}"], getattr(o, meth))
