"""The checker itself, away from the fixture configurations: oracle/algos.py against the UNMODIFIED reference
(oracle/make_golden.py: run_case asserts stats and final parameters within 2e-6 relative) with every hyper-parameter
moved off its default -- discount, Polyak rate, perturbation range, the two lambdas, KL weight, ensemble sizes 1 and 3,
sample counts, episode length, cost limits on both sides of the batch's Qc, PID gains, CPQ's threshold scalar, BEAR's
Laplacian kernel / sigma / MMD threshold / delayed policy start -- so that a GPU parity run at such a configuration
compares against something that was itself compared.  The reference's runs are stored in
tests/golden/reference_hparams.npz (record_reference below, run by oracle/record_reference.py: stats in full, initial
parameters as digests, each final tensor as its max |x|, checksum and a fixed sample of entries)."""
import pytest

from oracle import algos, make_golden
from tests import helpers

TWISTED = {
    "bc_t": ("bc", algos.BCConfig(9, 3, 2.0, [24, 40], 3e-3), 12, 3),
    "bcql_t1": ("bcql", algos.BCQLConfig(7, 3, 1.5, [24, 40], [40, 24], 56, 7, gamma=0.97, tau=0.02, phi=0.11, lmbda=0.6,
                                         beta=0.8, PID=[0.7, 0.05, 0.2], num_q=3, num_qc=1, cost_limit=3, episode_len=150,
                                         actor_lr=3e-4, critic_lr=2e-3, vae_lr=5e-4), 12, 3),
    "bcql_t2": ("bcql", algos.BCQLConfig(5, 2, 1.0, [32, 32], [32, 32], 40, 4, gamma=0.9, tau=0.3, phi=0.3, lmbda=1.0,
                                         beta=0.1, PID=[2.0, 0.5, 1.0], num_q=1, num_qc=3, cost_limit=-2, episode_len=40,
                                         actor_lr=1e-3, critic_lr=1e-3, vae_lr=1e-3), 10, 4),
    "cpq_t1": ("cpq", algos.CPQConfig(7, 3, 1.5, [24, 40], [40, 24], 56, 6, gamma=0.95, tau=0.05, beta=0.9, num_q=3,
                                      num_qc=2, qc_scalar=1.2, cost_limit=4, episode_len=80, actor_lr=2e-4, critic_lr=2e-3,
                                      alpha_lr=5e-3, vae_lr=7e-4), 12, 3),
    "cpq_t2": ("cpq", algos.CPQConfig(6, 2, 1.0, [32, 32], [32, 32], 40, 3, gamma=0.99, tau=0.005, beta=2.5, num_q=1,
                                      num_qc=1, qc_scalar=3.0, cost_limit=0.01, episode_len=500, actor_lr=1e-3,
                                      critic_lr=1e-3, alpha_lr=1e-2, vae_lr=1e-3), 10, 3),
    "bearl_t1": ("bearl", algos.BEARLConfig(7, 3, 1.5, [24, 40], [40, 24], 56, 6, gamma=0.96, tau=0.03, beta=0.7,
                                            lmbda=0.4, mmd_sigma=20.0, target_mmd_thresh=0.09, num_samples_mmd_match=6,
                                            PID=[0.9, 0.1, 0.3], kernel="laplacian", num_q=3, num_qc=2, cost_limit=2,
                                            episode_len=120, start_update_policy_step=0, actor_lr=4e-4, critic_lr=2e-3,
                                            vae_lr=6e-4, alpha_lr=3e-3), 12, 3),
    "bearl_t2": ("bearl", algos.BEARLConfig(5, 2, 1.0, [32, 32], [32, 32], 40, 4, gamma=0.99, tau=0.005, beta=0.5,
                                            lmbda=0.9, mmd_sigma=5.0, target_mmd_thresh=0.2, num_samples_mmd_match=3,
                                            PID=[1.0, 0.3, 0.5], kernel="gaussian", num_q=1, num_qc=1, cost_limit=-1,
                                            episode_len=60, start_update_policy_step=2, actor_lr=1e-3, critic_lr=1e-3,
                                            vae_lr=1e-3, alpha_lr=1e-3), 10, 4),   # policy loss switches form at step 2
}


@pytest.fixture(scope="module")
def osrl_ref():
    return helpers.load_pin("hparams")


@pytest.mark.parametrize("name", list(TWISTED))
def test_oracle_equals_reference_off_the_defaults(osrl_ref, name):
    algo, cfg, B, steps = TWISTED[name]
    make_golden.check_run(name, osrl_ref[name], make_golden.oracle_run(algo, cfg, B, steps), 2e-6, 1e-12, 2e-6)


CDT_TWISTED = {
    "cdt_t1": (dict(state_dim=6, action_dim=2, max_action=2.0, seq_len=6, episode_len=950, embedding_dim=48, num_layers=1,
                    num_heads=3, init_temperature=0.3, learning_rate=2e-3, weight_decay=1e-2, betas=(0.8, 0.95),
                    clip_grad=0.1, lr_warmup_steps=3, loss_cost_weight=0.5, loss_state_weight=0.3), 6, 4),
    "cdt_t2": (dict(state_dim=4, action_dim=3, max_action=1.0, seq_len=4, episode_len=1200, embedding_dim=32, num_layers=2,
                    num_heads=2, init_temperature=0.05, learning_rate=5e-4, weight_decay=0.0, betas=(0.9, 0.999),
                    clip_grad=5.0, lr_warmup_steps=1, loss_cost_weight=0.0, loss_state_weight=1.0,
                    attention_dropout=0.2, residual_dropout=0.1, embedding_dropout=0.05), 5, 3),
}


@pytest.mark.parametrize("name", list(CDT_TWISTED))
def test_cdt_oracle_equals_reference_off_the_defaults(osrl_ref, name):
    """oracle/cdt.py against the unmodified CDT / CDTTrainer (check_cdt_run asserts stats and parameters): other window
    length, width, head count, temperature, AdamW betas / decay, clip threshold on both sides of the gradient norm,
    warm-up, both auxiliary loss weights, and replayed dropout at three different rates."""
    kw, B, steps = CDT_TWISTED[name]
    make_golden.check_cdt_run(name, osrl_ref[name], make_golden.oracle_cdt_run(_cdt(**kw), B, steps))


def _cdt(**kw):
    from oracle import cdt as ocdt
    return ocdt.CDTConfig(**kw)


def _cop(**kw):
    from oracle import coptidice as oc
    return oc.COptiDICEConfig(**kw)


COP_TWISTED = {
    "cop_chi2": (dict(state_dim=7, action_dim=3, max_action=1.5, f_type="chi2", init_state_propotion=0.4,
                      a_hidden_sizes=[24, 40], c_hidden_sizes=[40, 24], gamma=0.95, alpha=0.8, cost_ub_epsilon=0.05,
                      num_nu=3, num_chi=1, cost_limit=4, episode_len=120, actor_lr=3e-4, critic_lr=2e-3, scalar_lr=5e-3), 20, 3),
    "cop_kl": (dict(state_dim=6, action_dim=2, max_action=1.0, f_type="kl", init_state_propotion=1.0,
                    a_hidden_sizes=[32, 32], c_hidden_sizes=[32, 32], gamma=0.99, alpha=0.2, cost_ub_epsilon=0.0,
                    num_nu=1, num_chi=3, cost_limit=25, episode_len=500, actor_lr=1e-3, critic_lr=5e-4, scalar_lr=1e-2), 16, 3),
    "cop_softchi": (dict(state_dim=5, action_dim=2, max_action=2.0, f_type="softchi", init_state_propotion=0.1,
                         a_hidden_sizes=[16, 48], c_hidden_sizes=[48, 16], gamma=0.9, alpha=1.5, cost_ub_epsilon=0.2,
                         num_nu=2, num_chi=2, cost_limit=1, episode_len=40, actor_lr=2e-3, critic_lr=2e-3, scalar_lr=2e-3), 24, 4),
}


@pytest.mark.parametrize("name", list(COP_TWISTED))
def test_coptidice_oracle_equals_reference_off_the_defaults(osrl_ref, name):
    """oracle/coptidice.py against the unmodified COptiDICE.update (check_coptidice_run asserts stats, parameters, tau
    and lambda): all three f-divergences (the committed fixture is softchi only), ensemble sizes 1..3, discount, alpha,
    the cost upper-bound epsilon incl. 0, initial-state proportion, cost limits and the three learning rates."""
    kw, B, steps = COP_TWISTED[name]
    make_golden.check_coptidice_run(name, osrl_ref[name], make_golden.oracle_coptidice_run(_cop(**kw), B, steps))


def record_reference(osrl):
    out = {}
    for name, (algo, cfg, B, steps) in TWISTED.items():
        run = make_golden.reference_run(osrl, algo, cfg, B, steps)
        make_golden.check_run(name, run, make_golden.oracle_run(algo, cfg, B, steps), 2e-6, 1e-12, 2e-6)
        out[name] = make_golden.pin_run(run)
    for name, (kw, B, steps) in CDT_TWISTED.items():
        run = make_golden.reference_cdt_run(osrl, _cdt(**kw), B, steps)
        make_golden.check_cdt_run(name, run, make_golden.oracle_cdt_run(_cdt(**kw), B, steps))
        out[name] = make_golden.pin_run(run)
    for name, (kw, B, steps) in COP_TWISTED.items():
        run = make_golden.reference_coptidice_run(osrl, _cop(**kw), B, steps)
        make_golden.check_coptidice_run(name, run, make_golden.oracle_coptidice_run(_cop(**kw), B, steps))
        out[name] = make_golden.pin_run(run)
    return out
