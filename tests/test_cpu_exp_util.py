"""osrl_b200.common.exp_util against the UNMODIFIED reference module (osrl/common/exp_util.py) on the same inputs: run
naming (auto_name / to_string incl. abbreviations, skip keys, prefix / suffix, the "default" fallback), the depth-first
config lookup with its quirk (a nested dict that lacks the key answers the string "None" and ends the search), and the
generator streams seed_all leaves behind.  The reference's answers are stored in tests/golden/reference_exp_util.npz
(record_reference below, run by oracle/record_reference.py)."""
import os
import random
import uuid

import numpy as np
import pytest
import torch

from tests import helpers


@pytest.fixture(scope="module")
def ref():
    return helpers.load_pin("exp_util")


CASES = [
    (dict(a=1, b=[1, 2], task="x", cost_limit=10), dict(a=2, b=[1, 2], task="y", cost_limit=20), "BCQL", ""),
    (dict(a=1, b=[1, 2]), dict(a=1, b=[1, 2]), "", ""),
    (dict(a=1, b=[1, 2]), dict(a=1, b=[1, 2]), "", "tail"),
    (dict(a=1, b=[1, [2, 3]], c={"z": 1, "y": (2, 3)}), dict(a=1, b=[4, [5, 6]], c={"z": 7, "y": (8, 9)}), "P", "S"),
    (dict(update_per_step=1, seed=0, device="cpu"), dict(update_per_step=4, seed=3, device="cuda"), "", ""),
]
TO_STRING = (3, "s", [1, [2, "x"], (3, 4)], {"b": 1, "a": [2, 3]}, [], {})
CFG = {"a": 1, "l": [1, 2, 3], "n1": {"x": 5}, "n2": {"y": {"deep": [7, 8]}, "x": 6}}
CFG_KEYS = ("a", "l", "x", "deep", "y", "missing")


class Env:
    def seed(self, s):
        self.s = s


def draw(seed_all):
    e = Env()
    seed_all(123, others=[e])
    return random.random(), np.random.rand(3).tolist(), torch.rand(3).tolist(), e.s


def write_run_dir(path):
    """A run directory as the reference's training scripts leave it (config.yaml, checkpoint/model[_best].pt)."""
    import yaml
    os.makedirs(os.path.join(path, "checkpoint"), exist_ok=True)
    with open(os.path.join(path, "config.yaml"), "w") as f:
        yaml.dump({"task": "t", "seed": 3}, f)
    torch.save({"model_state": {"w": torch.arange(3.0)}}, os.path.join(path, "checkpoint", "model.pt"))
    torch.save({"model_state": {"w": torch.arange(4.0)}}, os.path.join(path, "checkpoint", "model_best.pt"))


def record_reference(osrl):
    import tempfile
    from unittest import mock
    r = osrl.common.exp_util
    with mock.patch.object(uuid, "uuid4", lambda: "abcd-ef"):
        names = [r.auto_name(*c) for c in CASES]
    e = Env()
    ret = r.seed_all(5, others=e)
    with tempfile.TemporaryDirectory() as d:
        write_run_dir(d)
        loaded = []
        for best in (False, True):
            c, m = r.load_config_and_model(d, best)
            loaded.append({"config": c, "w": m["model_state"]["w"].numpy()})
    return {"auto_name": names, "DEFAULT_SKIP_KEY": r.DEFAULT_SKIP_KEY, "DEFAULT_KEY_ABBRE": r.DEFAULT_KEY_ABBRE,
            "to_string": [r.to_string(v) for v in TO_STRING], "get_cfg_value": [r.get_cfg_value(CFG, k) for k in CFG_KEYS],
            "draw": draw(r.seed_all), "seed_all_5": {"returns": ret, "env_seed": e.s}, "load": loaded}


@pytest.mark.parametrize("default,current,prefix,suffix", CASES)
def test_auto_name(ref, monkeypatch, default, current, prefix, suffix):
    from osrl_b200.common import exp_util as mine
    monkeypatch.setattr(uuid, "uuid4", lambda: "abcd-ef")
    want = ref["auto_name"][CASES.index((default, current, prefix, suffix))]
    assert mine.auto_name(default, current, prefix, suffix) == want
    assert mine.DEFAULT_SKIP_KEY == ref["DEFAULT_SKIP_KEY"] and mine.DEFAULT_KEY_ABBRE == ref["DEFAULT_KEY_ABBRE"]


def test_to_string_and_get_cfg_value(ref):
    from osrl_b200.common import exp_util as mine
    for v, want in zip(TO_STRING, ref["to_string"]):
        assert mine.to_string(v) == want
    for key, want in zip(CFG_KEYS, ref["get_cfg_value"]):
        assert mine.get_cfg_value(CFG, key) == want, key


def test_seed_all_streams(ref):
    from osrl_b200.common import exp_util as mine
    assert draw(mine.seed_all) == ref["draw"]
    e1 = Env()
    assert mine.seed_all(5, others=e1) == ref["seed_all_5"]["returns"] and e1.s == ref["seed_all_5"]["env_seed"] == 5


def test_load_config_and_model_roundtrip(ref, tmp_path):
    from osrl_b200.common import exp_util as mine
    write_run_dir(str(tmp_path))
    for best, want in zip((False, True), ref["load"]):
        c1, m1 = mine.load_config_and_model(str(tmp_path), best)
        assert c1 == want["config"] and torch.equal(m1["model_state"]["w"], torch.tensor(want["w"]))
    with pytest.raises(ValueError):
        mine.load_config_and_model(str(tmp_path / "nope"))
