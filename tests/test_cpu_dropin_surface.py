"""Drop-in surface (SURVEY.md section 8b): every name the reference's example scripts import from `osrl.*` exists in the
alias package (compat/osrl), and every keyword they pass to those classes / functions is accepted by the mirrors.

The scripts are parsed, not executed (they need a GPU for our models): for each `examples/train/*.py` and
`examples/eval/*.py` of the reference, record_reference collects `from osrl... import X` and the calls `X(...)` /
`trainer.method(...)` / `model.method(...)` into tests/golden/reference_scripts.npz, and the test checks them against
`inspect.signature` of the mirror; the executable counterpart is tests/test_gpu_dropin_loop.py."""
import ast
import glob
import inspect
import os
import sys

import pytest

from tests import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPTS = [f"{kind}_{algo}.py" for kind in ("eval", "train") for algo in ("bc", "bcql", "bearl", "cdt", "coptidice", "cpq")]


def record_reference(osrl):
    """{script: {"imports": [(module, name, asname)], "calls": [(receiver or None, function, keywords, n_positional)]}}"""
    from oracle import ref_shim
    ref = ref_shim.REFERENCE_ROOT
    out = {}
    for path in sorted(glob.glob(os.path.join(ref, "examples", "train", "train_*.py")) +
                       glob.glob(os.path.join(ref, "examples", "eval", "eval_*.py"))):
        tree = ast.parse(open(path).read())
        imports, calls = [], []
        for node in ast.walk(tree):
            if isinstance(node, ast.ImportFrom) and node.module and node.module.startswith("osrl"):
                imports += [(node.module, a.name, a.asname) for a in node.names]
        names = {asname or name for _, name, asname in imports}
        for node in ast.walk(tree):
            if not isinstance(node, ast.Call):
                continue
            kwargs = [k.arg for k in node.keywords if k.arg]
            if isinstance(node.func, ast.Name) and node.func.id in names:
                calls.append((None, node.func.id, kwargs, len(node.args)))
            elif isinstance(node.func, ast.Attribute) and isinstance(node.func.value, ast.Name) and \
                    node.func.value.id in ("trainer", "model"):
                calls.append((node.func.value.id, node.func.attr, kwargs, len(node.args)))
        out[os.path.basename(path)] = {"imports": imports, "calls": calls}
    assert sorted(out) == SCRIPTS, sorted(out)
    return out


@pytest.fixture(scope="module")
def alias():
    for m in [m for m in sys.modules if m == "osrl" or m.startswith("osrl.")]:
        del sys.modules[m]
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    try:
        import osrl.algorithms  # noqa: F401
        import osrl.common  # noqa: F401
        import osrl.common.dataset  # noqa: F401
        import osrl.common.exp_util  # noqa: F401
        import osrl
        assert "compat" in osrl.__file__
        yield osrl
    finally:
        sys.path.remove(os.path.join(ROOT, "compat"))
        for m in [m for m in sys.modules if m == "osrl" or m.startswith("osrl.")]:
            del sys.modules[m]


def _accepts(fn, kwargs, n_pos):
    sig = inspect.signature(fn)
    params = sig.parameters
    if any(p.kind == p.VAR_KEYWORD for p in params.values()):
        names_ok = True
    else:
        names_ok = all(k in params for k in kwargs)
    positional = [p for p in params.values() if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD) and p.name != "self"]
    return names_ok and (n_pos <= len(positional) or any(p.kind == p.VAR_POSITIONAL for p in params.values()))


@pytest.fixture(scope="module")
def scripts():
    return helpers.load_pin("scripts")


@pytest.mark.parametrize("script", SCRIPTS)
def test_script_surface(alias, scripts, script):
    import importlib
    rec = scripts[script]
    imported = {}
    for module, name, asname in rec["imports"]:
        mod = importlib.import_module(module)
        assert hasattr(mod, name), f"{script}: {module}.{name} missing"
        imported[asname or name] = getattr(mod, name)
    assert imported, "script imports nothing from osrl?"
    trainer_cls = [v for k, v in imported.items() if k.endswith("Trainer")]
    checked = 0
    for receiver, func, kwargs, n_args in rec["calls"]:
        if receiver is None and func in imported:
            target = imported[func]
            fn = target.__init__ if inspect.isclass(target) else target
            assert _accepts(fn, kwargs, n_args), f"{script}: {func}({', '.join(kwargs)}) not accepted by {fn}"
            checked += 1
        elif receiver == "trainer" and trainer_cls:
            assert hasattr(trainer_cls[0], func), f"{script}: trainer.{func} missing"
            assert _accepts(getattr(trainer_cls[0], func), kwargs, n_args), f"{script}: trainer.{func} call not accepted"
            checked += 1
        elif receiver == "model" and func in ("load_state_dict", "state_dict", "to", "eval", "parameters"):
            checked += 1   # nn.Module API: the mirrors are nn.Modules
    assert checked >= 3, f"{script}: only {checked} calls recognised"
