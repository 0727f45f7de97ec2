"""The model mirrors (osrl_b200.algorithms.*) against the UNMODIFIED reference classes on the CPU, before any engine
is bound: constructed under the same seed_all(s) they must hold the same state_dict (keys, order, shapes, bits -- the
modules are built in the reference's order, so the same generator stream initialises them) and `act()` -- the
evaluation path of evaluate()/rollout() -- must return the same actions for the same observation and generator state.
What the reference classes hold and return is stored in tests/golden/reference_models.npz (record_reference below, run
by oracle/record_reference.py; parameters as sha256 digests of their bits)."""
import os
import sys

import numpy as np
import pytest
import torch

from tests import helpers

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "stubs"))
from synthetic_env import SyntheticOfflineEnv  # noqa: E402

O, A = 8, 2
COP = dict(f_type="softchi", init_state_propotion=1.0, observations_std=np.ones(O, np.float32), actions_std=np.ones(A, np.float32))
CASES = {
    "BC": (dict(a_hidden_sizes=[32, 32]), [()]),
    "BCQL": (dict(a_hidden_sizes=[32, 32], c_hidden_sizes=[32, 32], vae_hidden_sizes=48), [()]),
    # (the reference's CPQ / BEAR-Lag / COptiDICE act() needs with_logprob=True: it dereferences the log-probability)
    "CPQ": (dict(a_hidden_sizes=[32, 32], c_hidden_sizes=[32, 32], vae_hidden_sizes=48), [(True, True), (False, True)]),
    "BEARL": (dict(a_hidden_sizes=[32, 32], c_hidden_sizes=[32, 32], vae_hidden_sizes=48), [(True, True), (False, True)]),
    "COptiDICE": (dict(a_hidden_sizes=[32, 32], c_hidden_sizes=[32, 32], **COP), [(True, True), (False, True)]),
}


CDT_KW = dict(seq_len=5, episode_len=12, embedding_dim=32, num_layers=2, num_heads=4, use_rew=True, use_cost=True,
              cost_transform=True, stochastic=True, time_emb=True)


def state_digests(model):
    return [(k, helpers.digest(v.float())) for k, v in model.state_dict().items()]


def act_draws(model, act_args):
    """act() on three seeded observations per argument set, under the same generator state."""
    rng = np.random.default_rng(0)
    out = []
    for args in act_args:
        for _ in range(3):
            obs = rng.standard_normal(O).astype(np.float32)
            torch.manual_seed(11)
            r = model.act(obs, *args)
            out.append([None if x is None else np.asarray(x) for x in (r if isinstance(r, tuple) else (r,))])
    return out


def evaluate_run(mod, name, kw):
    from osrl_b200.common.exp_util import seed_all
    seed_all(3)
    model = getattr(mod, name)(O, A, 1.0, device="cpu", episode_len=12, **kw)
    env = SyntheticOfflineEnv(O, A, episode_len=12, seed=5)
    scales = {} if name == "BC" else dict(reward_scale=0.5, cost_scale=2.0)
    tr = getattr(mod, name + "Trainer")(model, env, device="cpu", **scales)
    torch.manual_seed(1)
    return np.asarray(tr.evaluate(3), dtype=np.float64)


def cdt_inputs():
    g = torch.Generator().manual_seed(0)
    B, T = 3, 5
    st, ac = torch.randn(B, T, O, generator=g), torch.randn(B, T, A, generator=g)
    rtg, ctg = torch.rand(B, T, generator=g) * 10, torch.rand(B, T, generator=g) * 5
    ts = torch.arange(T).repeat(B, 1)
    pad = torch.zeros(B, T, dtype=torch.bool)
    pad[1, 3:] = True          # windows are zero-padded at the END (dataset.py:757-775)
    return st, ac, rtg, ctg, ts, pad


def cdt_forward(model):
    model.eval()
    with torch.no_grad():
        a, c, s = model(*cdt_inputs())
    return [x.numpy() for x in (a.mean, a.stddev, c, s)]


def cdt_evaluate(mod, model):
    env = SyntheticOfflineEnv(O, A, episode_len=12, seed=5)
    tr = mod.CDTTrainer(model, env, reward_scale=0.5, cost_scale=2.0, device="cpu")
    torch.manual_seed(1)
    return np.asarray(tr.evaluate(2, 6.0, 3.0), dtype=np.float64)


def record_reference(osrl):
    from osrl_b200.common.exp_util import seed_all
    ra = osrl.algorithms
    out = {}
    for name, (kw, act_args) in CASES.items():
        seed_all(7)
        model = getattr(ra, name)(O, A, 1.0, device="cpu", **kw)
        out[name] = {"state": state_digests(model), "act": act_draws(model, act_args),
                     "evaluate": evaluate_run(ra, name, kw)}
    seed_all(9)
    model = ra.CDT(O, A, 1.0, **CDT_KW)
    out["CDT"] = {"state": [(k, helpers.digest(v)) for k, v in model.state_dict().items()], "forward": cdt_forward(model),
                  "evaluate": cdt_evaluate(ra, model)}
    return out


@pytest.fixture(scope="module")
def ref_algos():
    return helpers.load_pin("models")


@pytest.mark.parametrize("name", list(CASES))
def test_same_init_and_same_actions(ref_algos, name):
    import osrl_b200.algorithms as mine
    from osrl_b200.common.exp_util import seed_all
    kw, act_args = CASES[name]
    want = ref_algos[name]
    seed_all(7)
    ours = getattr(mine, name)(O, A, 1.0, device="cpu", **kw)
    got = state_digests(ours)
    assert [k for k, _ in got] == [k for k, _ in want["state"]]
    for (k, g), (_, w) in zip(got, want["state"]):
        assert g == w, k
    for w_draw, g_draw in zip(want["act"], act_draws(ours, act_args), strict=True):
        assert len(w_draw) == len(g_draw)
        for w, g in zip(w_draw, g_draw):
            if w is None:
                assert g is None
            else:
                np.testing.assert_allclose(g, w, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("name", list(CASES))
def test_evaluate_rolls_out_like_the_reference(ref_algos, name):
    """<Algo>Trainer.evaluate on a seeded synthetic environment: same episodes, same returns -- in particular CPQ,
    BEAR-Lag and COptiDICE roll out the deterministic policy (act(obs, True, True)), BCQ-Lag the sampled one."""
    import osrl_b200.algorithms as mine
    kw, _ = CASES[name]
    np.testing.assert_allclose(evaluate_run(mine, name, kw), ref_algos[name]["evaluate"], rtol=1e-6, atol=1e-7)


def test_cdt_same_init_forward_and_evaluate(ref_algos):
    """CDT in the configured mode (time_emb, use_rew, use_cost, cost_transform, stochastic head): same state_dict under
    the same seed (construction order + _init_weights), same evaluation-time forward (action distribution, cost
    log-probabilities, state prediction) and the same target-conditioned roll-outs (cdt.py:436-518)."""
    import osrl_b200.algorithms as mine
    from osrl_b200.common.exp_util import seed_all
    want = ref_algos["CDT"]
    seed_all(9)
    ours = mine.CDT(O, A, 1.0, device="cpu", **CDT_KW)
    got = [(k, helpers.digest(v)) for k, v in ours.state_dict().items()]
    assert [k for k, _ in got] == [k for k, _ in want["state"]]
    for (k, g), (_, w) in zip(got, want["state"]):
        assert g == w, k
    for y, x in zip(cdt_forward(ours), want["forward"], strict=True):
        torch.testing.assert_close(torch.tensor(y), torch.tensor(x), rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(cdt_evaluate(mine, ours), want["evaluate"], rtol=1e-5, atol=1e-6)
