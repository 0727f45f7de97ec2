"""Record what the UNMODIFIED reference computes for the CPU comparison tests: tests/golden/reference_<name>.npz.

Needs the reference tree (ref_shim.REFERENCE_ROOT); the tests read these pins and never the reference itself:
    python -m oracle.record_reference [name ...]

Each test module below defines record_reference(osrl): the reference's side of its comparisons, on the same inputs
its tests use.  Test infrastructure only.
"""
from __future__ import annotations

import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "stubs"))

from oracle import ref_shim  # noqa: E402
from tests import helpers  # noqa: E402

MODULES = {
    "surface": "tests.test_cpu_signatures",          # also read by tests/test_cpu_config_plumbing.py
    "scripts": "tests.test_cpu_dropin_surface",
    "exp_util": "tests.test_cpu_exp_util",
    "models": "tests.test_cpu_models_vs_reference",
    "dataset": "tests.test_cpu_dataset_preproc",
    "hparams": "tests.test_cpu_oracle_hparams",
}


def main():
    import oapackage  # the stub: the reference's dataset module imports it
    import torch
    torch.set_num_threads(8)
    osrl = ref_shim.import_reference()
    import osrl.common.dataset as rd
    import osrl.common.exp_util  # noqa: F401
    if not hasattr(rd, "oapackage"):
        rd.oapackage = oapackage
    only = sys.argv[1:]
    for name, mod in MODULES.items():
        if only and name not in only:
            continue
        helpers.save_pin(name, importlib.import_module(mod).record_reference(osrl))
        size = os.path.getsize(os.path.join(helpers.GOLDEN, f"reference_{name}.npz"))
        print(f"[pin] reference_{name}.npz: {size} bytes")


if __name__ == "__main__":
    main()
