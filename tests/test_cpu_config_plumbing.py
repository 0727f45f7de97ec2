"""Every hyper-parameter of the reference's model and trainer constructors must reach the C ABI's osrl_config with the
value the caller passed: the mirrors are built with DISTINCT non-default values for every parameter the reference's
signature has, and the struct `make_config(algo, **model._hyper(), **trainer._lrs)` produces is checked field by field.
(The GPU parity fixtures mostly run the default values, where a parameter that never leaves Python would go
unnoticed -- CPQ's KL weight did, once.)  The reference's signatures come from tests/golden/reference_surface.npz
(tests/test_cpu_signatures.py: record_reference)."""
import numpy as np
import pytest

from tests import helpers

O, A = 8, 2
# reference parameter -> osrl_config field(s); None = not a step hyper-parameter of the engine (says why)
FIELD = {"state_dim": "obs_dim", "action_dim": "act_dim", "vae_hidden_sizes": "vae_hidden", "kernel": "mmd_kernel",
         "PID": ("pid_kp", "pid_ki", "pid_kd"), "betas": ("adam_beta1", "adam_beta2"),
         "a_hidden_sizes": ("n_a_hidden", "a_hidden"), "c_hidden_sizes": ("n_c_hidden", "c_hidden")}
NOT_CONFIG = {
    "device": "placement", "env": "evaluation only", "logger": "host side", "model": "the model itself",
    "reward_scale": "applied when the dataset is packed (dataset.py:836-837, :762-763)", "cost_scale": "same",
    "cost_reverse": "dataset option (process_sequence_dataset)", "no_entropy": "not built: the mirror raises",
    "bc_mode": "dataset filter (process_bc_dataset)", "observations_std": "pointer, checked separately",
    "actions_std": "pointer, checked separately",
    # CDT switches: only the configured mode is built, anything else raises in the mirror's constructor
    "time_emb": "fixed", "use_rew": "fixed", "use_cost": "fixed", "cost_transform": "fixed", "stochastic": "fixed",
    "add_cost_feat": "fixed", "mul_cost_feat": "fixed", "cat_cost_feat": "fixed", "action_head_layers": "fixed",
    "cost_prefix": "fixed",
}
FIXED = {"time_emb": True, "use_rew": True, "use_cost": True, "cost_transform": True, "stochastic": True,
         "f_type": "kl", "kernel": "laplacian", "init_state_propotion": 0.25, "observations_std": np.full(O, 2.0, np.float32),
         "actions_std": np.full(A, 3.0, np.float32), "state_dim": O, "action_dim": A, "bc_mode": "all",
         "num_heads": 4, "embedding_dim": 64, "betas": (0.85, 0.97), "PID": [0.21, 0.0043, 0.0017],
         "a_hidden_sizes": [48, 40], "c_hidden_sizes": [56, 24], "target_entropy": -3.5, "max_action": 1.7,
         "vae_hidden_sizes": 72, "action_head_layers": 1}


@pytest.fixture(scope="module")
def ref_algos():
    from tests.test_cpu_signatures import Recorded
    return {k: [Recorded(*p) for p in v] for k, v in helpers.load_pin("surface").items()}


def _distinct(name, default, salt):
    if name in FIXED:
        return FIXED[name]
    if isinstance(default, bool):
        return default
    if isinstance(default, int):
        return default + 1 + salt % 3
    if isinstance(default, float):
        return round(default * (0.61 + 0.07 * (salt % 4)) + 0.0113, 6)
    raise AssertionError(f"no distinct value rule for {name}={default!r}")


def _check_field(cfg, name, value):
    f = FIELD.get(name, name)
    if name in ("a_hidden_sizes", "c_hidden_sizes"):
        assert getattr(cfg, f[0]) == len(value) and list(getattr(cfg, f[1]))[:len(value)] == list(value), name
    elif name == "PID" or name == "betas":
        for fld, v in zip(f, value):
            assert getattr(cfg, fld) == pytest.approx(v, rel=1e-6), name
    elif name == "kernel":
        assert cfg.mmd_kernel == {"gaussian": 0, "laplacian": 1}[value]
    elif name == "f_type":
        assert cfg.f_type == {"chi2": 0, "softchi": 1, "kl": 2}[value]
    else:
        assert hasattr(cfg, f), f"osrl_config has no field for {name}"
        got = getattr(cfg, f)
        assert got == pytest.approx(value, rel=1e-6), f"{name}: config holds {got}, caller passed {value}"


@pytest.mark.parametrize("name", ["BC", "BCQL", "CPQ", "BEARL", "CDT", "COptiDICE"])
def test_every_reference_hyperparameter_reaches_the_config(ref_algos, name):
    import osrl_b200.algorithms as mine
    from osrl_b200.engine import make_config
    kw, salt = {}, 0
    for p in ref_algos[name]:
        if p.name == "device":
            continue
        salt += 1
        kw[p.name] = _distinct(p.name, p.default, salt)
    model = getattr(mine, name)(device="cpu", **kw)
    tkw = {}
    for p in ref_algos[name + "Trainer"]:
        if p.name in NOT_CONFIG and p.name not in FIXED:
            continue
        salt += 1
        tkw[p.name] = _distinct(p.name, p.default, salt)
    tkw.pop("bc_mode", None)
    trainer = getattr(mine, name + "Trainer")(model, None, None, device="cpu", **tkw)
    algo = {"BC": "bc", "BCQL": "bcql", "CPQ": "cpq", "BEARL": "bearl", "CDT": "cdt", "COptiDICE": "coptidice"}[name]
    cfg = make_config(algo, batch_size=4, **model._hyper(), **trainer._lrs)
    for k, v in {**kw, **tkw}.items():
        if k in NOT_CONFIG or (name == "BC" and k in ("episode_len", "cost_limit")):   # (BC: roll-out settings only)
            continue
        _check_field(cfg, k, v)
    if name == "COptiDICE":
        import ctypes as C
        got = np.ctypeslib.as_array(C.cast(cfg.observations_std, C.POINTER(C.c_float)), shape=(O,))
        assert np.array_equal(got, kw["observations_std"])
        got = np.ctypeslib.as_array(C.cast(cfg.actions_std, C.POINTER(C.c_float)), shape=(A,))
        assert np.array_equal(got, kw["actions_std"])
