"""Pin the oracle against the live reference and write tests/golden/*.npz.

Run in the build container only (needs /root/reference):
    python -m oracle.make_golden

For every algorithm it (1) seeds torch, builds the UNMODIFIED reference model+trainer
and the oracle, checks the initial parameters are bit-identical; (2) feeds both the
same seeded minibatches with torch's global generator re-seeded identically, so both
consume the same noise stream; (3) asserts per-step stats and final parameters agree;
(4) writes the batches, the consumed noise, the stats and the parameters (small
configs: full tensors; full-size configs: checksums) as fixtures.  Test
infrastructure only.
"""
from __future__ import annotations

import dataclasses
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import algos, ref_shim, synth  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = {
    # name: (algo, oracle cfg, batch, steps, store_full)
    "bc_small": ("bc", algos.BCConfig(28, 2, 1.0, [32, 32], 1e-3), 16, 3, True),
    "bcql_small": ("bcql", algos.BCQLConfig(8, 2, 1.0, [32, 32], [32, 32], 48, 10, num_q=2, num_qc=2,
                                            actor_lr=1e-3, critic_lr=1e-3, vae_lr=1e-3), 16, 3, True),
    "cpq_small": ("cpq", algos.CPQConfig(11, 3, 1.0, [32, 32], [32, 32], 40, 10, beta=0.5, num_q=2, num_qc=2,
                                         episode_len=200, actor_lr=1e-4, critic_lr=1e-3, alpha_lr=1e-4,
                                         vae_lr=1e-3), 16, 3, True),
    "bearl_small": ("bearl", algos.BEARLConfig(8, 2, 1.0, [32, 32], [32, 32], 48, 10, num_q=2, num_qc=2,
                                               start_update_policy_step=0, actor_lr=1e-3, critic_lr=1e-3,
                                               vae_lr=1e-3), 16, 3, True),
    # active constraint branch: qc_thres < 0 and O(1) PID gains -> lambda = O(0.1..1), qc_penalty != 0 (net.py:376-387,
    # bcql.py:189-198, bearl.py:233-260); the default configs keep lambda ~ 1e-5 over the first steps
    "bcql_pid_small": ("bcql", algos.BCQLConfig(8, 2, 1.0, [32, 32], [32, 32], 48, 10, num_q=2, num_qc=2,
                                                PID=[1.0, 0.3, 0.5], cost_limit=-1, actor_lr=1e-3, critic_lr=1e-3,
                                                vae_lr=1e-3), 16, 4, True),
    "bearl_pid_small": ("bearl", algos.BEARLConfig(8, 2, 1.0, [32, 32], [32, 32], 48, 10, num_q=2, num_qc=2,
                                                   PID=[1.0, 0.3, 0.5], cost_limit=-1, start_update_policy_step=0,
                                                   actor_lr=1e-3, critic_lr=1e-3, vae_lr=1e-3), 16, 4, True),
    # BASELINE.json configs[0..2,4] at full layer sizes (checksums only)
    "bc_full": ("bc", algos.BCConfig(28, 2, 1.0, [256, 256], 1e-3), 256, 3, False),
    "bcql_full": ("bcql", algos.BCQLConfig(8, 2, 1.0, [256, 256], [256, 256], 400, 10, num_q=2, num_qc=2,
                                           actor_lr=1e-3, critic_lr=1e-3, vae_lr=1e-3), 256, 3, False),
    "cpq_full": ("cpq", algos.CPQConfig(33, 8, 1.0, [256, 256], [256, 256], 400, 10, beta=0.5, num_q=2, num_qc=2,
                                        episode_len=200, actor_lr=1e-4, critic_lr=1e-3, alpha_lr=1e-4,
                                        vae_lr=1e-3), 512, 2, False),
    "bearl_full": ("bearl", algos.BEARLConfig(8, 2, 1.0, [256, 256], [256, 256], 400, 10, num_q=2, num_qc=2,
                                              start_update_policy_step=0, actor_lr=1e-3, critic_lr=1e-3,
                                              vae_lr=1e-3), 512, 2, False),
    "bcql_pid_full": ("bcql", algos.BCQLConfig(8, 2, 1.0, [256, 256], [256, 256], 400, 10, num_q=2, num_qc=2,
                                               PID=[1.0, 0.3, 0.5], cost_limit=-1, actor_lr=1e-3, critic_lr=1e-3,
                                               vae_lr=1e-3), 256, 3, False),
    "bearl_pid_full": ("bearl", algos.BEARLConfig(8, 2, 1.0, [256, 256], [256, 256], 400, 10, num_q=2, num_qc=2,
                                                  PID=[1.0, 0.3, 0.5], cost_limit=-1, start_update_policy_step=0,
                                                  actor_lr=1e-3, critic_lr=1e-3, vae_lr=1e-3), 512, 2, False),
}

ORACLES = {"bc": algos.BCOracle, "bcql": algos.BCQLOracle, "cpq": algos.CPQOracle, "bearl": algos.BEARLOracle}
LR_KEYS = ("actor_lr", "critic_lr", "vae_lr", "alpha_lr")


def build_reference(osrl, algo: str, cfg):
    kw = {k: v for k, v in dataclasses.asdict(cfg).items() if k not in LR_KEYS}
    lrs = {k: v for k, v in dataclasses.asdict(cfg).items() if k in LR_KEYS}
    A = osrl.algorithms
    if algo == "bc":
        model = A.BC(**kw, device="cpu")
        trainer = A.BCTrainer(model, None, logger=ref_shim.NullLogger(), actor_lr=lrs["actor_lr"], device="cpu")
    elif algo == "bcql":
        model = A.BCQL(**kw, device="cpu")
        trainer = A.BCQLTrainer(model, None, logger=ref_shim.NullLogger(), **lrs, device="cpu")
    elif algo == "cpq":
        model = A.CPQ(**kw, device="cpu")
        trainer = A.CPQTrainer(model, None, logger=ref_shim.NullLogger(), **lrs, device="cpu")
    elif algo == "bearl":
        model = A.BEARL(**kw, device="cpu")
        trainer = A.BEARLTrainer(model, None, logger=ref_shim.NullLogger(), **lrs, device="cpu")
    else:
        raise ValueError(algo)
    return model, trainer


def batch_args(algo, b):
    t = {k: torch.from_numpy(v) for k, v in b.items()}
    if algo == "bc":
        return (t["observations"], t["actions"])
    return (t["observations"], t["next_observations"], t["actions"], t["rewards"], t["costs"], t["done"])


def checksum(t: torch.Tensor):
    d = t.double()
    return [float(d.sum()), float(d.abs().sum()), float((d * d).sum())]


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    den = float(b.abs().max()) + 1e-30
    return float((a - b).abs().max()) / den


# ---- reference results kept small: tests/test_cpu_oracle_hparams.py holds the oracle to what the reference computed at
# configurations away from the fixtures; it stores each final tensor's max |x|, checksum and a fixed sample of entries
PIN_SAMPLE = 8


def pin_tensor(t: torch.Tensor) -> dict:
    a = t.detach().double().reshape(-1).numpy()
    idx = np.sort(np.random.default_rng(0).choice(a.size, min(PIN_SAMPLE, a.size), replace=False)).astype(np.int32)
    return {"max": float(np.abs(a).max()), "checksum": checksum(t), "idx": idx, "val": a[idx].astype(np.float32)}


def pin_run(run: dict) -> dict:
    """What check_run needs of a reference run: initial parameters as digests, final parameters pinned, the rest (stats,
    scalars) as is."""
    from tests.helpers import digest
    return dict(run, init={k: digest(v) for k, v in run["init"].items()},
                stats=[{k: float(v) for k, v in r.items()} for r in run["stats"]],
                final={k: pin_tensor(v) for k, v in run["final"].items()})


def _param_err(got: torch.Tensor, want) -> float:
    """max |got - want| / max |want| for a full tensor; for a pinned one, the largest ratio among the bounds that
    max |got - want| <= tol max |want| implies (max |x|, the sampled entries, the checksums)."""
    if isinstance(want, torch.Tensor):
        return rel_err(got, want)
    a = got.detach().double().reshape(-1)
    m, n = want["max"], a.numel()
    den = m + 1e-30
    sampled = a[torch.tensor(want["idx"], dtype=torch.long)] - torch.tensor(want["val"], dtype=torch.float64)
    errs = [abs(float(a.abs().max()) - m) / den, float(sampled.abs().max()) / den]
    got_sum = checksum(got)
    for i, (g, w) in enumerate(zip(got_sum, want["checksum"])):
        scale = n * den * ((2 * m + 1e-30) if i == 2 else 1.0)   # sum(a^2 - b^2) <= sum |a - b| |a + b|
        errs.append(abs(g - w) / scale)
    return max(errs)


def check_run(name, want, got, stat_tol, stat_den, param_tol, skip_params=()):
    """got (an oracle run) against want (a reference run, full or pinned): same initial parameters bit for bit,
    per-step stats within stat_tol relative, final parameters within param_tol of each tensor's max |x|."""
    from tests.helpers import digest
    assert list(want["init"]) == list(got["init"]), (name, "state_dict keys differ")
    for k, v in want["init"].items():
        same = torch.equal(v, got["init"][k]) if isinstance(v, torch.Tensor) else v == digest(got["init"][k])
        assert same, (name, "init differs", k)
    worst = 0.0
    assert len(want["stats"]) == len(got["stats"])
    for s, (r, o) in enumerate(zip(want["stats"], got["stats"])):
        assert set(r) == set(o), (name, s, set(r) ^ set(o))
        for k in r:
            e = abs(r[k] - o[k]) / (abs(r[k]) + stat_den)
            worst = max(worst, e)
            assert e < stat_tol, (name, s, k, r[k], o[k])
    perr = 0.0
    for k, v in want["final"].items():
        if any(x in k for x in skip_params):
            continue
        perr = max(perr, _param_err(got["final"][k], v))
    assert perr < param_tol, (name, "final params differ", perr)
    return worst, perr


def make_batches(cfg, B, steps, data_seed=1234):
    rng = np.random.default_rng(data_seed)
    return [synth.make_batch(rng, B, cfg.state_dim, cfg.action_dim) for _ in range(steps)]


def reference_run(osrl, algo, cfg, B, steps, init_seed=0, noise_seed=4321):
    """The unmodified reference: initial parameters, per-step logged stats, final parameters."""
    torch.manual_seed(init_seed)
    ref_model, ref_trainer = build_reference(osrl, algo, cfg)
    init = {k: v.clone() for k, v in ref_model.state_dict().items()}
    torch.manual_seed(noise_seed)
    stats = []
    for b in make_batches(cfg, B, steps):
        n0 = len(ref_trainer.logger.rows)
        ref_trainer.train_one_step(*batch_args(algo, b))
        row = {}
        for r in ref_trainer.logger.rows[n0:]:
            row.update(r)
        stats.append(row)
    return {"init": init, "stats": stats, "final": ref_model.state_dict()}


def oracle_run(algo, cfg, B, steps, init_seed=0, noise_seed=4321):
    """The oracle on the same seeds, batches and noise stream as reference_run (plus the batches and the noise)."""
    torch.manual_seed(init_seed)
    orc = ORACLES[algo](cfg)
    init = {k: v.clone() for k, v in orc.params.items()}
    batches = make_batches(cfg, B, steps)
    torch.manual_seed(noise_seed)
    stats, noises = [], []
    for b in batches:
        stats.append(orc.step(*batch_args(algo, b)))
        noises.append({k: v.clone() for k, v in orc.last_noise.items()})
    return {"init": init, "stats": stats, "final": orc.params, "batches": batches, "noises": noises}


def run_case(osrl, name, algo, cfg, B, steps, full):
    init_seed, data_seed, noise_seed = 0, 1234, 4321
    ref = reference_run(osrl, algo, cfg, B, steps, init_seed, noise_seed)
    orc = oracle_run(algo, cfg, B, steps, init_seed, noise_seed)
    worst, perr = check_run(name, ref, orc, 2e-6, 1e-12, 2e-6)
    print(f"[golden] {name}: oracle == reference over {steps} steps (stat rel err {worst:.2e}, param rel err {perr:.2e})")

    init, ref_stats, batches, noises = orc["init"], ref["stats"], orc["batches"], orc["noises"]
    out = {"meta": json.dumps({"algo": algo, "cfg": dataclasses.asdict(cfg), "B": B, "steps": steps,
                               "init_seed": init_seed, "data_seed": data_seed, "noise_seed": noise_seed,
                               "full": full, "torch": torch.__version__, "keys": list(init.keys()),
                               "stat_keys": sorted(ref_stats[0].keys())})}
    out["stats"] = np.array([[r[k] for k in sorted(r)] for r in ref_stats], dtype=np.float64)
    if full:
        for k, v in init.items():
            out["init/" + k] = v.numpy()
        for k, v in ref["final"].items():
            out["final/" + k] = v.numpy()
        for s, (b, nz) in enumerate(zip(batches, noises)):
            for k, v in b.items():
                out[f"batch{s}/{k}"] = v
            for k, v in nz.items():
                out[f"noise{s}/{k}"] = v.numpy()
    else:
        out["init_checksum"] = np.array([checksum(v) for v in init.values()])
        out["final_checksum"] = np.array([checksum(v) for v in ref["final"].values()])
        out["noise_checksum"] = np.array([[checksum(v) for v in nz.values()] for nz in noises])
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    osrl = ref_shim.import_reference()
    only = sys.argv[1:]
    for name, (algo, cfg, B, steps, full) in CASES.items():
        if only and name not in only:
            continue
        run_case(osrl, name, algo, cfg, B, steps, full)


if __name__ == "__main__" and not ({"cdt", "coptidice"} & set(sys.argv[1:])):
    main()


# =========================================================================== CDT
def make_seq_batch(rng, B, T, o, a):
    """A collated SequenceDataset batch (dtypes as the reference yields them: float64 mask, int64 time_steps)."""
    lens = rng.integers(1, T + 1, B)
    lens[: B // 2] = T
    mask = (np.arange(T)[None, :] < lens[:, None]).astype(np.float64)
    m32 = mask.astype(np.float32)
    start = rng.integers(0, 900, B)
    return {
        "states": rng.standard_normal((B, T, o), dtype=np.float32) * m32[..., None],
        "actions": rng.uniform(-1, 1, (B, T, a)).astype(np.float32) * m32[..., None],
        "returns": (rng.uniform(0, 40, (B, T)).astype(np.float32)) * m32,
        "costs_return": (rng.uniform(0, 30, (B, T)).astype(np.float32)) * m32,
        "time_steps": (start[:, None] + np.arange(T)[None, :]).astype(np.int64),
        "mask": mask,
        "episode_cost": rng.uniform(0, 30, B).astype(np.float32),
        "costs": (rng.random((B, T)) < 0.2).astype(np.float32) * m32,
    }


CDT_KEYS = ("states", "actions", "returns", "costs_return", "time_steps", "mask", "episode_cost", "costs")


class DropReplay:
    """Run the UNMODIFIED reference modules on prescribed dropout multipliers: torch.nn.functional.dropout (what
    nn.Dropout calls) and torch.nn.functional.scaled_dot_product_attention (what nn.MultiheadAttention's training path
    calls with dropout_p) are swapped for versions that multiply by the next tensor of the queue.  The reference's
    call order per step is emb_drop (cdt.py:222), then per block: attention weights, self.drop(attention_out),
    the mlp's trailing nn.Dropout (net.py:428-440)."""

    def __init__(self, masks):
        self.q = list(masks)

    def __enter__(self):
        import math
        import torch.nn.functional as F
        self.F, self.old = F, (F.dropout, F.scaled_dot_product_attention)
        q = self.q

        def dropout(input, p=0.5, training=True, inplace=False):
            if not training or p == 0.0:
                return input
            m = q.pop(0)
            assert m.shape == input.shape, (m.shape, input.shape)
            return input * m

        def sdpa(query, key, value, attn_mask=None, dropout_p=0.0, is_causal=False, scale=None, **kw):
            sc = (query @ key.transpose(-1, -2)) * (scale if scale is not None else 1.0 / math.sqrt(query.shape[-1]))
            if attn_mask is not None:
                sc = sc.masked_fill(~attn_mask, float("-inf")) if attn_mask.dtype == torch.bool else sc + attn_mask
            pw = torch.softmax(sc, dim=-1)
            if dropout_p > 0.0:
                pw = pw * q.pop(0).reshape(pw.shape)
            return pw @ value

        F.dropout, F.scaled_dot_product_attention = dropout, sdpa
        return self

    def __exit__(self, *a):
        self.F.dropout, self.F.scaled_dot_product_attention = self.old
        assert not self.q, f"{len(self.q)} dropout tensors were not consumed by the reference"


def reference_cdt_run(osrl, cfg, B, steps):
    """The unmodified CDT / CDTTrainer on replayed dropout multipliers: initial parameters, stats, final parameters,
    log-temperature."""
    from oracle import cdt as ocdt
    torch.manual_seed(0)
    ref = osrl.algorithms.CDT(state_dim=cfg.state_dim, action_dim=cfg.action_dim, max_action=cfg.max_action,
                              seq_len=cfg.seq_len, episode_len=cfg.episode_len, embedding_dim=cfg.embedding_dim,
                              num_layers=cfg.num_layers, num_heads=cfg.num_heads,
                              attention_dropout=cfg.attention_dropout, residual_dropout=cfg.residual_dropout,
                              embedding_dropout=cfg.embedding_dropout, time_emb=True, use_rew=True, use_cost=True,
                              cost_transform=True, stochastic=True, init_temperature=cfg.init_temperature,
                              target_entropy=-cfg.action_dim)
    trainer = osrl.algorithms.CDTTrainer(ref, None, logger=ref_shim.NullLogger(), learning_rate=cfg.learning_rate,
                                         weight_decay=cfg.weight_decay, betas=cfg.betas, clip_grad=cfg.clip_grad,
                                         lr_warmup_steps=cfg.lr_warmup_steps, loss_cost_weight=cfg.loss_cost_weight,
                                         loss_state_weight=cfg.loss_state_weight, device="cpu")
    init = {k: v.clone() for k, v in ref.state_dict().items() if "causal_mask" not in k}
    torch.manual_seed(0)
    masker = ocdt.CDTOracle(cfg)          # draws the multipliers (and leaves torch's generator where the oracle does)
    mgen = torch.Generator().manual_seed(4242)
    ref.train()
    stats = []
    for b in make_cdt_batches(cfg, B, steps):
        n0 = len(trainer.logger.rows)
        with DropReplay(masker.draw_masks(B, generator=mgen).values()):
            trainer.train_one_step(*[torch.from_numpy(b[k]) for k in CDT_KEYS])
        row = {}
        for r in trainer.logger.rows[n0:]:
            row.update(r)
        stats.append(row)
    return {"init": init, "stats": stats, "log_temperature": float(ref.log_temperature.detach()),
            "final": {k: v for k, v in ref.state_dict().items() if "causal_mask" not in k}}


def make_cdt_batches(cfg, B, steps):
    rng = np.random.default_rng(77)
    return [make_seq_batch(rng, B, cfg.seq_len, cfg.state_dim, cfg.action_dim) for _ in range(steps)]


def oracle_cdt_run(cfg, B, steps):
    """oracle/cdt.py on the batches and dropout multipliers of reference_cdt_run (plus the batches and multipliers)."""
    from oracle import cdt as ocdt
    torch.manual_seed(0)
    orc = ocdt.CDTOracle(cfg)
    init = {k: v.clone() for k, v in orc.params.items()}
    batches = make_cdt_batches(cfg, B, steps)
    mgen = torch.Generator().manual_seed(4242)
    stats, all_masks = [], []
    for b in batches:
        masks = orc.draw_masks(B, generator=mgen)       # empty when every dropout is 0
        all_masks.append(masks)
        stats.append(orc.step(*[torch.from_numpy(b[k]) for k in CDT_KEYS], noise=masks))
    return {"init": init, "stats": stats, "final": orc.params, "log_temperature": float(orc.log_temperature),
            "batches": batches, "masks": all_masks}


def check_cdt_run(name, want, got):
    # in_proj_bias: the key-bias slice has an exactly-zero true gradient (softmax shift invariance); what
    # Adam sees there is rounding noise, so its sign-like update is not reproducible even by the reference
    worst, perr = check_run(name, want, got, 2e-5, 1e-9, 2e-5, skip_params=("in_proj_bias",))
    lt = abs(want["log_temperature"] - got["log_temperature"])
    assert lt < 1e-9, lt
    return worst, perr


def run_cdt_case(osrl, name, cfg, B, steps, full):
    ref = reference_cdt_run(osrl, cfg, B, steps)
    orc = oracle_cdt_run(cfg, B, steps)
    worst, perr = check_cdt_run(name, ref, orc)
    print(f"[golden] {name}: oracle == reference over {steps} steps (stat rel err {worst:.2e}, param rel err {perr:.2e})")
    init, ref_stats, batches, all_masks = orc["init"], ref["stats"], orc["batches"], orc["masks"]
    cfgd = dataclasses.asdict(cfg)
    cfgd["betas"] = list(cfgd["betas"])
    out = {"meta": json.dumps({"algo": "cdt", "cfg": cfgd, "B": B, "steps": steps, "full": full,
                               "keys": list(init.keys()), "stat_keys": sorted(ref_stats[0].keys()),
                               "torch": torch.__version__})}
    out["stats"] = np.array([[r[k] for k in sorted(r)] for r in ref_stats], dtype=np.float64)
    if full:
        for k, v in init.items():
            out["init/" + k] = v.numpy()
        for k, v in ref["final"].items():
            out["final/" + k] = v.numpy()
        for s, b in enumerate(batches):
            for k, v in b.items():
                out[f"batch{s}/{k}"] = v
            for k, v in all_masks[s].items():          # keep bits; the multiplier is bit / (1 - p)
                out[f"drop{s}/{k}"] = np.packbits((v.numpy() > 0).reshape(-1))
        out["log_temperature"] = np.array(ref["log_temperature"])
    else:
        out["init_checksum"] = np.array([checksum(v) for v in init.values()])
        out["final_checksum"] = np.array([checksum(v) for v in ref["final"].values()])
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)


def main_cdt():
    from oracle import cdt as ocdt
    osrl = ref_shim.import_reference()
    if "cdt_b2048" in sys.argv[1:]:
        # BASELINE.json configs[3] at its own size: B=2048, seq_len 10, 3 layers, E=128, dropout 0.1 at all three
        # sites (cdt_configs.py:22-44,498-511).  81,920 tokens -> the split-K weight-gradient path.  Checksums and
        # stats only; the GPU test re-draws the same multipliers from the same torch CPU generator (seed 4242).
        run_cdt_case(osrl, "cdt_b2048", ocdt.CDTConfig(17, 6, 1.0, seq_len=10, episode_len=1000, embedding_dim=128,
                                                       num_layers=3, num_heads=8, attention_dropout=0.1,
                                                       residual_dropout=0.1, embedding_dropout=0.1), 2048, 2, False)
        return
    run_cdt_case(osrl, "cdt_small", ocdt.CDTConfig(5, 3, 1.0, seq_len=10, episode_len=1000, embedding_dim=32,
                                                   num_layers=2, num_heads=4, learning_rate=1e-3, lr_warmup_steps=4), 8, 3, True)
    run_cdt_case(osrl, "cdt_full", ocdt.CDTConfig(17, 6, 1.0, seq_len=10, episode_len=1000, embedding_dim=128,
                                                  num_layers=3, num_heads=8), 64, 2, False)
    # the reference's configured dropouts (cdt_configs.py: 0.1 at all three sites), replayed multipliers
    run_cdt_case(osrl, "cdt_drop_small", ocdt.CDTConfig(5, 3, 1.0, seq_len=10, episode_len=1000, embedding_dim=32,
                                                        num_layers=2, num_heads=4, learning_rate=1e-3, lr_warmup_steps=4,
                                                        attention_dropout=0.1, residual_dropout=0.1,
                                                        embedding_dropout=0.1), 8, 3, True)


if __name__ == "__main__" and "cdt" in sys.argv[1:]:
    main_cdt()


def check_sequence_sampler():
    """Pin oracle.cdt.sequence_sample / split_trajectories against the reference's SequenceDataset
    (dataset.py:668-775) on a seeded synthetic dataset, including the cost-based sample_prob."""
    from oracle import cdt as ocdt
    osrl = ref_shim.import_reference()
    d = synth.make_dataset(6, 3, 41, 13, seed=9)
    d["timeouts"][-7:] = False          # trailing unfinished episode must be dropped
    ct = lambda x: 70 - x
    ref = osrl.common.dataset.SequenceDataset({k: v.copy() for k, v in d.items()}, seq_len=10, reward_scale=0.1,
                                              cost_scale=1.0, augment_percent=0, cost_sample=True, cost_transform=ct)
    tr = ocdt.split_trajectories(d)
    assert len(tr) == len(ref.dataset)
    p = np.array([ct(t["cost_returns"][0]) for t in tr])     # float32, like dataset.py:452-458
    p[p < 0] = 0
    p /= np.sum(p)
    assert p.dtype == ref.sample_prob.dtype and np.array_equal(p, ref.sample_prob)
    rng = np.random.default_rng(0)
    for _ in range(200):
        t = int(rng.integers(0, len(tr)))
        s = int(rng.integers(0, tr[t]["rewards"].shape[0]))
        a = ref._SequenceDataset__prepare_sample(t, s)
        b = ocdt.sequence_sample(tr, t, s, 10, 0.1, 1.0)
        for x, y in zip(a, b):
            assert np.array_equal(np.asarray(x), np.asarray(y)) and np.asarray(x).dtype == np.asarray(y).dtype, (t, s)
    print("[golden] sequence sampler: oracle == reference on 200 (trajectory, start) pairs")


if __name__ == "__main__" and "cdt" in sys.argv[1:]:
    check_sequence_sampler()


# =========================================================================== COptiDICE (SURVEY 8f rank 1: next row)
def main_coptidice():
    """Pin oracle.coptidice against the unmodified reference (coptidice.py:125-227) and write the fixture the CUDA
    implementation will be held to.  Both consume torch's global generator in the same order (obs noise, action
    noise, the actor's unused rsample), re-seeded identically before each step."""
    from oracle import coptidice as oc
    osrl = ref_shim.import_reference()
    cfg = oc.COptiDICEConfig(8, 2, 1.0, f_type="softchi", init_state_propotion=0.25, a_hidden_sizes=[32, 32],
                             c_hidden_sizes=[32, 32], num_nu=2, num_chi=2, actor_lr=1e-3, critic_lr=1e-3, scalar_lr=1e-3)
    run_coptidice_case(osrl, "coptidice_small", cfg, 32, 4)


COP_KEYS = ("observations", "next_observations", "actions", "rewards", "costs", "done")


def coptidice_inputs(cfg, B, steps):
    """observations_std, actions_std and the batches (with is_init) of a COptiDICE case, seeded"""
    rng = np.random.default_rng(21)
    obs_std = rng.uniform(0.5, 1.5, (1, cfg.state_dim)).astype(np.float32)
    act_std = rng.uniform(0.3, 0.8, (1, cfg.action_dim)).astype(np.float32)
    batches = []
    for _ in range(steps):
        b = synth.make_batch(rng, B, cfg.state_dim, cfg.action_dim)
        b["is_init"] = (rng.random(B) < 0.25).astype(np.float32)
        batches.append(b)
    return obs_std, act_std, batches


def _cop_args(b):
    return [torch.from_numpy(b[k]) for k in COP_KEYS] + [torch.from_numpy(b["is_init"])]


def reference_coptidice_run(osrl, cfg, B, steps):
    """The unmodified COptiDICE / COptiDICETrainer: initial parameters, stats, final parameters, tau and lambda."""
    obs_std, act_std, batches = coptidice_inputs(cfg, B, steps)
    torch.manual_seed(0)
    ref = osrl.algorithms.COptiDICE(cfg.state_dim, cfg.action_dim, cfg.max_action, cfg.f_type, cfg.init_state_propotion,
                                    obs_std, act_std, cfg.a_hidden_sizes, cfg.c_hidden_sizes, cfg.gamma, cfg.alpha,
                                    cfg.cost_ub_epsilon, cfg.num_nu, cfg.num_chi, cfg.cost_limit, cfg.episode_len, "cpu")
    trainer = osrl.algorithms.COptiDICETrainer(ref, None, logger=ref_shim.NullLogger(), actor_lr=cfg.actor_lr,
                                               critic_lr=cfg.critic_lr, scalar_lr=cfg.scalar_lr, device="cpu")
    scalars = {"tau": ref.tau, "lmbda": ref.lmbda}           # (parameters outside the state_dict)
    init = {k: v.detach().clone() for k, v in {**ref.state_dict(), **scalars}.items()}
    stats = []
    for s, b in enumerate(batches):
        n0 = len(trainer.logger.rows)
        torch.manual_seed(1000 + s)
        trainer.train_one_step(_cop_args(b))
        row = {}
        for r in trainer.logger.rows[n0:]:
            row.update(r)
        stats.append(row)
    return {"init": init, "stats": stats, "final": {k: v.detach() for k, v in {**ref.state_dict(), **scalars}.items()},
            "tau": float(ref.tau.detach()), "lmbda": float(ref.lmbda.detach())}


def oracle_coptidice_run(cfg, B, steps):
    """oracle/coptidice.py on the inputs of reference_coptidice_run (plus the inputs and the noise)."""
    from oracle import coptidice as oc
    obs_std, act_std, batches = coptidice_inputs(cfg, B, steps)
    torch.manual_seed(0)
    orc = oc.COptiDICEOracle(cfg, obs_std, act_std)
    init = {k: v.clone() for k, v in orc.params.items()}
    stats, noises = [], []
    for s, b in enumerate(batches):
        torch.manual_seed(1000 + s)
        stats.append(orc.step(*_cop_args(b)))
        noises.append({k: v.clone() for k, v in orc.last_noise.items()})
    return {"init": init, "stats": stats, "final": orc.params, "tau": float(orc.params["tau"]),
            "lmbda": float(orc.params["lmbda"]), "obs_std": obs_std, "act_std": act_std, "batches": batches,
            "noises": noises}


def check_coptidice_run(name, want, got):
    worst, perr = check_run(name, want, got, 2e-5, 1e-6, 2e-5)
    serr = max(abs(want["tau"] - got["tau"]), abs(want["lmbda"] - got["lmbda"]))
    assert serr < 1e-6, serr
    return worst, perr, serr


def run_coptidice_case(osrl, name, cfg, B, steps):
    """oracle.coptidice == the unmodified reference over `steps` steps at configuration `cfg` (asserted), fixture
    written to OUT/<name>.npz."""
    ref = reference_coptidice_run(osrl, cfg, B, steps)
    orc = oracle_coptidice_run(cfg, B, steps)
    worst, perr, serr = check_coptidice_run(name, ref, orc)
    print(f"[golden] {name}: oracle == reference over {steps} steps (stat rel err {worst:.2e}, "
          f"param rel err {perr:.2e}, tau/lambda abs err {serr:.1e})")
    out = {}
    for s, (b, nz) in enumerate(zip(orc["batches"], orc["noises"])):
        for k, v in b.items():
            out[f"batch{s}/{k}"] = v
        for k, v in nz.items():
            out[f"noise{s}/{k}"] = v.numpy()
    cfgd = dataclasses.asdict(cfg)
    out["meta"] = json.dumps({"algo": "coptidice", "cfg": cfgd, "B": B, "steps": steps,
                              "keys": list(orc["init"].keys()),
                              "stat_keys": sorted(ref["stats"][0].keys()), "torch": torch.__version__})
    out["stats"] = np.array([[r[k] for k in sorted(r)] for r in ref["stats"]], dtype=np.float64)
    out["observations_std"], out["actions_std"] = orc["obs_std"], orc["act_std"]
    for k, v in orc["init"].items():
        out["init/" + k] = v.numpy()
    for k, v in ref["final"].items():
        out["final/" + k] = v.numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)


if __name__ == "__main__" and "coptidice" in sys.argv[1:]:
    main_coptidice()
