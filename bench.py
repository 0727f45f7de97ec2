#!/usr/bin/env python
"""bench.py -- gradient-steps/sec of the OSRL per-step hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload = BASELINE.json configs[1]: BCQ-Lag, OfflineCarCircle-v0-shaped transitions (obs 8, act 2),
batch 256 per GPU, hidden [256,256] x2, VAE 400, 10 sampled actions, 2+2 double-Q nets, fp32.
One "step" = VAE + critic + cost-critic + actor updates + Polyak (reference: BCQLTrainer.train_one_step,
osrl/algorithms/bcql.py:283-306, fed by the loop body examples/train/train_bcql.py:142-148).

ours      : `value` -- K steps with the dataset resident in HBM (minibatch drawn on the device), timed
            with CUDA events between barriers, max over ranks.  `e2e` -- the same step through the
            public trainer API with HOST (pinned) minibatches: H2D of the 6 batch tensors and D2H of
            the step's stats inside the timed region.
reference : the reference's CPU implementation of the same step (the oracle port of the PyTorch path,
            all host threads), rank 0 only.
Data-parallel (N>1): one process per GPU (torchrun), per-GPU batch fixed at 256 (weak scaling), gradients
all-reduced with NCCL before every optimiser update; `value` = N x synchronous steps/s, i.e. batch-256
gradient-step equivalents per second over the whole job (`config.synchronous_steps_per_s` is the rate of actual
optimiser steps).  Before timing, N>1 runs a data-parallel parity check (engine under NCCL vs the single-rank oracle
on the concatenated batch, active PID multiplier) and reports it as `dp_parity`.

Extra keys of the result line: `roofline` -- step-level fraction of the measured HBM peak per SURVEY.md 8(d)
(bytes = 24 P_train + 8 P_target + batch bytes) with the per-kernel table (timed inside a replayed CUDA graph) as
`roofline.kernels`; `other_configs` -- short device-resident runs of BASELINE.json configs[2..4] (CPQ B=512,
CDT B=2048 seq 10, BEAR-Lag B=512 per GPU and the strong-scaling BEAR-Lag global B=4096) with ms/step and the same
step-level fractions; `cpu_baseline`.

--dump-outputs DIR (ours, rank 0): after the K timed steps, what the last of them left for a caller -- the step's
statistics (float32), the PID / dual scalars (float64) and every trained and target parameter tensor (float32, 6.3 MB)
-- as DIR/<name>.npy.  Model init, dataset and device sampling are seeded, so the same arguments give the same inputs
and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG = dict(state_dim=8, action_dim=2, max_action=1.0, a_hidden_sizes=[256, 256], c_hidden_sizes=[256, 256],
           vae_hidden_sizes=400, sample_action_num=10, gamma=0.99, tau=0.005, phi=0.05, lmbda=0.75, beta=0.5,
           PID=[0.1, 0.003, 0.001], num_q=2, num_qc=2, cost_limit=10, episode_len=300, actor_lr=1e-3, critic_lr=1e-3,
           vae_lr=1e-3)
BATCH = 256
DATASET_ROWS = 2_000_000          # 2e6 x 96 B packed = 192 MB per GPU  (> 126 MB L2)
REWARD_SCALE, COST_SCALE = 0.1, 1.0
# SURVEY.md section 8(d): algorithmic bytes per step = 24*P_train + 8*P_target + batch bytes (fp32)
P_TRAIN, P_TARGET = 954_452, 620_042
STEP_BYTES = 24 * P_TRAIN + 8 * P_TARGET + BATCH * (2 * 8 + 2 + 3) * 4
STEP_FLOPS = 7.285e9
WORKLOAD = "BCQ-Lag OfflineCarCircle-v0-shaped (obs 8, act 2) batch=256/GPU fp32 (BASELINE.json configs[1])"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return (float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1700.0)),
                "measured (MEASURED_PEAKS.json: hbm_gbs burst copy, bf16_tflops burst cuBLAS -- kernels are timed alone)")
    return 6650.0, 1700.0, "fallback (B200_PROFILING.md: 6.65 TB/s, ~1.7 PFLOP/s dense bf16)"


def make_dataset(rows: int, seed: int):
    from oracle import synth
    eps = rows // 300
    return synth.make_dataset(8, 2, 300, eps, seed=seed)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def calibrate_threads(step_fn, budget_s: float = 25.0):
    """The reference's small GEMMs do not scale to 100+ threads (oversubscription makes a step take seconds):
    time a few thread counts and keep the fastest, so the CPU baseline is the reference at its best."""
    cores = usable_cores()
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores})
    best, best_t = cands[0], float("inf")
    t_start = time.perf_counter()
    for c in cands:
        torch.set_num_threads(c)
        step_fn()
        t0 = time.perf_counter()
        step_fn(); step_fn()
        dt = (time.perf_counter() - t0) / 2
        if dt < best_t:
            best, best_t = c, dt
        if dt > 1.3 * best_t or time.perf_counter() - t_start > budget_s:
            break   # more threads only make the reference's small GEMMs slower from here on
    torch.set_num_threads(best)
    return best, cores


def init_params():
    """Reference arm only: the oracle port of the reference's CPU step."""
    from tests.helpers import make_oracle
    return make_oracle("bcql", CFG, 0)


def bcql_model(device: str):
    """Our arm: the public mirror class, initialised like the reference (seed_all, then construct; bcql.py:85-98)."""
    from osrl_b200.algorithms import BCQL
    from osrl_b200.common.exp_util import seed_all
    seed_all(0)
    return BCQL(8, 2, 1.0, CFG["a_hidden_sizes"], CFG["c_hidden_sizes"], CFG["vae_hidden_sizes"],
                CFG["sample_action_num"], CFG["gamma"], CFG["tau"], CFG["phi"], CFG["lmbda"], CFG["beta"], CFG["PID"],
                CFG["num_q"], CFG["num_qc"], CFG["cost_limit"], CFG["episode_len"], device=device)


# ------------------------------------------------------------------------------------------ other BASELINE configs
# SURVEY.md 8(d): algorithmic bytes = 24 P_train + 8 P_target + batch bytes; flops from the oracle's flop counter
OTHER = {
    "cpq_b512": dict(algo="cpq", batch=512, dims=(33, 8, 200), steps=200, bytes=21.47e6, flops=8.80e9,
                     workload="CPQ OfflineAntRun-v0-shaped (obs 33, act 8) batch=512 (BASELINE.json configs[2])"),
    "cdt_b2048": dict(algo="cdt", batch=2048, dims=(17, 6, 1000), steps=12, bytes=20.04e6, flops=305.8e9,
                      workload="CDT OfflineHalfCheetahVelocity-v1-shaped (obs 17, act 6) seq_len=10 batch=2048, "
                               "3 layers, E=128, dropout 0.1 (BASELINE.json configs[3])"),
    "bearl_b512": dict(algo="bearl", batch=512, dims=(8, 2, 300), steps=200, bytes=27.91e6, flops=14.6e9,
                       workload="BEAR-Lag OfflineCarCircle-v0-shaped batch=512 per GPU (BASELINE.json configs[4] shard)"),
}


def build_other(name: str, batch: int, device: str, world: int, rank: int):
    """Model + engine + resident dataset of one of the other BASELINE configs through the public mirror classes."""
    from oracle import synth
    from osrl_b200.algorithms import BEARL, CDT, CPQ, BEARLTrainer, CDTTrainer, CPQTrainer
    from osrl_b200.common.dataset import SequenceDataset
    from osrl_b200.common.exp_util import seed_all
    spec = OTHER[name]
    o, a, T = spec["dims"]
    seed_all(0)
    if spec["algo"] == "cpq":       # examples/configs/cpq_configs.py:29-51
        model = CPQ(o, a, 1.0, [256, 256], [256, 256], 400, 10, 0.99, 0.005, 0.5, 2, 2, 1.5, 10, T, device=device)
        tr = CPQTrainer(model, None, None, actor_lr=1e-4, critic_lr=1e-3, alpha_lr=1e-4, vae_lr=1e-3, reward_scale=0.1,
                        cost_scale=1.0, device=device)
    elif spec["algo"] == "bearl":   # examples/configs/bearl_configs.py:29-56
        model = BEARL(o, a, 1.0, [256, 256], [256, 256], 400, 10, 0.99, 0.005, 0.5, 0.75, 50, 0.05, 10,
                      [0.1, 0.003, 0.001], "gaussian", 2, 2, 10, T, 0, device=device)
        tr = BEARLTrainer(model, None, None, actor_lr=1e-3, critic_lr=1e-3, alpha_lr=1e-3, vae_lr=1e-3, reward_scale=0.1,
                          cost_scale=1.0, device=device)
    else:                           # examples/configs/cdt_configs.py:22-44,498-511
        model = CDT(o, a, 1.0, seq_len=10, episode_len=T, embedding_dim=128, num_layers=3, num_heads=8,
                    attention_dropout=0.1, residual_dropout=0.1, embedding_dropout=0.1, time_emb=True, use_rew=True,
                    use_cost=True, cost_transform=True, stochastic=True, init_temperature=0.1, target_entropy=-a,
                    device=device)
        tr = CDTTrainer(model, None, None, learning_rate=1e-4, weight_decay=1e-4, betas=(0.9, 0.999), clip_grad=0.25,
                        lr_warmup_steps=500, reward_scale=0.1, cost_scale=1.0, loss_cost_weight=0.02,
                        loss_state_weight=0.0, device=device)
    eng = model._bind(batch, tr._lrs, seed=4321, world_size=world, rank=rank)
    if spec["algo"] == "cdt":
        data = synth.make_dataset(o, a, T, 300, seed=200 + rank)
        SequenceDataset(data, seq_len=10, reward_scale=0.1, cost_scale=1.0, cost_sample=True,
                        cost_transform=lambda x: 200 - x).to_engine(eng)   # (synthetic episodes cost ~100)
    else:
        eng.upload_dataset(synth.make_dataset(o, a, T, max(2, 1_500_000 // T), seed=200 + rank), 0.1, 1.0)
    return model, eng


def run_other(name: str, batch: int, local: int, world: int, rank: int, barrier, peaks, comm_setup):
    """Short device-resident timing of one other config: CUDA events between barriers, max over ranks."""
    import torch.distributed as dist
    spec = OTHER[name]
    model, eng = build_other(name, batch, f"cuda:{local}", world, rank)
    if world > 1:
        comm_setup(eng)
    K = spec["steps"]
    eng.steps(5)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.steps(K)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    stats = eng.stats()
    lps = eng.launches_per_step
    eng.close()
    sps = K / ms * 1e3
    peak_gbs, peak_tf, _ = peaks
    return {"workload": spec["workload"], "per_gpu_batch": batch, "global_batch": batch * world, "steps": K,
            "ms_per_step": ms / K, "synchronous_steps_per_s": sps, "launches_per_step": lps,
            "hbm_frac": spec["bytes"] * sps / 1e9 / peak_gbs, "tflops": spec["flops"] * sps / 1e12,
            "tensor_frac_of_bf16_peak": spec["flops"] * sps / 1e12 / peak_tf,
            "tensor_frac_of_3xtf32_ceiling": spec["flops"] * sps / 1e12 / (peak_tf / 6.0),
            "finite": bool(np.isfinite(list(stats.values())).all())}


def run_preprocess(local: int, rows: int = 1_000_000, ep_len: int = 1000):
    """One-time trajectory preprocessing of a 1M-transition DSRL-shaped dataset (HalfCheetah dims): episode split +
    reward / cost to go + packed buffer.  device_ms includes the host->device copy of the raw arrays (74 MB)."""
    import time
    from oracle import cdt as ocdt
    from osrl_b200 import Engine
    from osrl_b200.common.dataset import SequenceDataset
    o, a = 17, 6
    rng = np.random.default_rng(0)
    data = {"observations": rng.standard_normal((rows, o)).astype(np.float32),
            "actions": rng.uniform(-1, 1, (rows, a)).astype(np.float32),
            "rewards": rng.standard_normal(rows).astype(np.float32),
            "costs": (rng.random(rows) < 0.1).astype(np.float32), "terminals": np.zeros(rows, bool),
            "timeouts": (np.arange(rows) % ep_len) == ep_len - 1}
    eng = Engine("cdt", batch_size=64, device=local, seed=0, state_dim=o, action_dim=a, max_action=1.0, seq_len=10,
                 episode_len=ep_len, embedding_dim=128, num_layers=3, num_heads=8, use_rew=1, use_cost=1, cost_transform=1,
                 stochastic=1, target_entropy=-float(a), learning_rate=1e-4, lr_warmup_steps=500)
    eng.preprocess_seq_dataset(data, 0.1, 1.0)          # warm-up (allocator, first touch of the host pages)
    t0 = time.perf_counter()
    info = eng.preprocess_seq_dataset(data, 0.1, 1.0)
    dev_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    ds = SequenceDataset(data, seq_len=10, reward_scale=0.1, cost_scale=1.0)
    host_ms = (time.perf_counter() - t0) * 1e3
    ds.to_engine(eng)                                     # host pack + upload of the same resident buffer
    torch.cuda.synchronize()
    host_total_ms = (time.perf_counter() - t0) * 1e3
    sample = 100_000                                      # the reference's per-transition Python loop, bounded sample
    sub = {k: v[:sample] for k, v in data.items()}
    t0 = time.perf_counter()
    trajs = ocdt.split_trajectories(sub)
    loop_ms = (time.perf_counter() - t0) * 1e3
    ok = bool(np.array_equal(info["returns"][:len(trajs)], np.array([t["returns"][0] for t in trajs], np.float32)))
    eng.close()
    return {"workload": f"process_sequence_dataset on {rows} transitions ({rows // ep_len} episodes of {ep_len}), obs 17, act 6",
            "device_ms": dev_ms, "rows_per_s_device": rows / dev_ms * 1e3, "h2d_bytes": int(rows * (o + a + 2) * 4 + 2 * rows),
            "host_numpy_mirror_ms": host_ms, "host_numpy_mirror_plus_upload_ms": host_total_ms,
            "note": "device_ms and host_numpy_mirror_plus_upload_ms both end with the packed trajectory buffer resident "
                    "in HBM and include the pageable host->device copy",
            "reference_loop_port": {"sample_rows": sample, "ms": loop_ms, "rows_per_s": sample / loop_ms * 1e3,
                                    "what": "oracle/cdt.py split_trajectories: dataset.py:137-183 restated, per-transition loop"},
            "first_returns_equal_oracle": ok, "episodes": int(eng.n_traj)}


def dump_outputs(out_dir: str, eng) -> None:
    """The engine's outputs after its last step (statistics, scalars, parameters) as out_dir/<name>.npy; '/' in a
    name becomes '.'."""
    arrays = {f"stats.{k}": np.float32(v) for k, v in eng.stats().items()}
    arrays.update({f"scalars.{k}": np.float64(v) for k, v in eng.scalars().items()})
    arrays.update({f"params.{k}": v.numpy() for k, v in eng.read_params().items()})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name.replace("/", ".") + ".npy"), a)


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import synth
    orc = init_params()
    rng = np.random.default_rng(0)
    batches = [synth.make_batch(rng, BATCH, 8, 2) for _ in range(8)]
    keys = ("observations", "next_observations", "actions", "rewards", "costs", "done")
    tb = [[torch.from_numpy(b[k]) for k in keys] for b in batches]
    torch.manual_seed(0)
    cores, avail = calibrate_threads(lambda: orc.step(*tb[0]))
    for i in range(max(1, min(args.warmup, 5))):
        orc.step(*tb[i % len(tb)])
    t0 = time.perf_counter()
    orc.step(*tb[0])
    one = time.perf_counter() - t0
    k = max(3, min(args.steps, int(120.0 / max(one, 1e-4))))   # bounded sample: <= ~2 min of CPU work
    t0 = time.perf_counter()
    for i in range(k):
        orc.step(*tb[i % len(tb)])
    dt = time.perf_counter() - t0
    v = k / dt
    sample = (f"{k} train steps (oracle port of bcql.py:283-306, torch CPU fp32) on fixed pre-collated batches; "
              f"{cores} torch threads = fastest of a sweep up to the {avail} usable cores")
    print(json.dumps({
        "impl": "reference", "metric": "gradient-steps/sec", "value": v, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": k, "warmup": args.warmup, "ms_per_step": 1e3 * dt / k, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": BATCH, "parallelism": "cpu"},
        "cpu_baseline": {"value": v, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch.distributed as dist
    from osrl_b200 import comm_unique_id
    from osrl_b200.algorithms import BCQLTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torchrun (one process per GPU)")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def comm_setup(engine):
        ids = [comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        engine.init_comm(ids[0])

    peaks = measured_peaks()
    peak_gbs, peak_tf, peak_src = peaks

    # ---- data-parallel parity, before anything is timed (N > 1): NCCL engine vs the single-rank oracle on the
    # concatenated batch -- the small config with an ACTIVE PID multiplier (tests/dp_worker.py) and one step of the
    # bench configuration itself (global batch 256 N)
    dp_parity = None
    if world > 1:
        from tests import dp_worker
        small = dp_worker.run("bcql", "nccl", steps=3, Bg=32 * world, detail=True)
        cfg_act = dict(CFG, cost_limit=0.05)
        full = dp_worker.run("bcql", "nccl", steps=1, Bg=BATCH * world, cfg=cfg_act, detail=True)
        dp_parity = {"ok": bool(small["ok"] and full["ok"]), "worst_ratio": max(small["worst_ratio"], full["worst_ratio"]),
                     "small_active_pid": small, "bench_config_one_step": full}

    # ---- device-resident path: the public model class bound to an engine, dataset shard resident in HBM
    model = bcql_model(dev)
    lrs = dict(actor_lr=CFG["actor_lr"], critic_lr=CFG["critic_lr"], vae_lr=CFG["vae_lr"])
    eng = model._bind(BATCH, lrs, seed=1234, world_size=world, rank=rank)
    if world > 1:
        comm_setup(eng)
    dp_mode = eng.dp_mode
    data = make_dataset(DATASET_ROWS, seed=100 + rank)      # each rank owns its own shard (weak scaling)
    eng.upload_dataset(data, REWARD_SCALE, COST_SCALE)

    K, W = args.steps, max(args.warmup, 3)
    eng.steps(W)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.steps(K)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launches - l0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    sync_steps_per_s = K / ms * 1e3
    value = sync_steps_per_s * world

    # ---- end-to-end through the public trainer API with host minibatches
    model2 = bcql_model(dev)

    class _Store:
        def __init__(self):
            self.last = None

        def store(self, tab=None, **kw):
            self.last = kw

    logger = _Store()
    trainer = BCQLTrainer(model2, None, logger, actor_lr=CFG["actor_lr"], critic_lr=CFG["critic_lr"],
                          vae_lr=CFG["vae_lr"], reward_scale=REWARD_SCALE, cost_scale=COST_SCALE, device=dev, seed=99)
    if world > 1:
        model2._bind(BATCH, trainer._lrs, seed=99, world_size=world, rank=rank)
        comm_setup(model2.engine)
    KE = min(K, 1000)
    rng = np.random.default_rng(7 + rank)
    n = data["observations"].shape[0]
    done = np.logical_or(data["terminals"], data["timeouts"]).astype(np.float32)
    nb = 64
    host = []
    for _ in range(nb):
        idx = rng.integers(0, n, BATCH)
        host.append([torch.from_numpy(a).pin_memory() for a in (
            data["observations"][idx], data["next_observations"][idx], data["actions"][idx],
            data["rewards"][idx] * np.float32(REWARD_SCALE), data["costs"][idx] * np.float32(COST_SCALE), done[idx])])
    h2d = sum(t.numel() * 4 for t in host[0])
    for i in range(W):
        trainer.train_one_step(*host[i % nb])
    barrier()
    e0.record()
    for i in range(KE):
        trainer.train_one_step(*host[i % nb])     # H2D of 6 tensors + step + D2H of the stats (logger.store)
    e1.record()
    barrier()
    ms_e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e = float(t.item())
    e2e_sync = KE / ms_e * 1e3 * world
    # the same loop with lagged stats (osrl_stats_lagged: the D2H read of step s-1's stats is still inside every
    # iteration, but nothing waits for step s): the host queues the next step while the GPU runs the current one
    trainer.lag_stats = True
    for i in range(W):
        trainer.train_one_step(*host[i % nb])
    barrier()
    e0.record()
    for i in range(KE):
        trainer.train_one_step(*host[i % nb])
    e1.record()
    barrier()
    ms_l = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_l], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_l = float(t.item())
    e2e_v = KE / ms_l * 1e3 * world
    d2h = 4 * len(eng.stat_names)
    assert logger.last is not None and np.isfinite(list(logger.last.values())).all()
    # the batched host call (trainer.train_batches -> osrl_steps_host): the caller hands over CHUNK loader batches at a
    # time; every step still moves its own 21.5 KB minibatch host -> device (read in place from a pinned ring by the
    # step graph) and its stat rows device -> host (one from each graph branch), all inside the timed region, and every
    # step's stats reach the logger
    trainer.lag_stats = False
    CHUNK = 100
    chunks = [[tuple(host[(c * CHUNK + i) % nb]) for i in range(CHUNK)] for c in range(max(1, KE // CHUNK))]
    for _ in range(2):
        trainer.train_batches(chunks[0])
    barrier()
    e0.record()
    for ch in chunks:
        trainer.train_batches(ch)
    e1.record()
    barrier()
    ms_b = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_b], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_b = float(t.item())
    KB = len(chunks) * CHUNK
    e2e_batched = KB / ms_b * 1e3 * world
    d2h_batched = 2 * 4 * len(eng.stat_names)
    assert logger.last is not None and np.isfinite(list(logger.last.values())).all()
    model2.engine.close()

    # ---- per-kernel timing inside a replayed graph (osrl_profile), rank 0 only, N == 1
    roof = None
    if rank == 0:
        roof = {"bound": "hbm", "achieved": STEP_BYTES * sync_steps_per_s / 1e9, "peak": peak_gbs, "unit": "GB/s",
                "frac": STEP_BYTES * sync_steps_per_s / 1e9 / peak_gbs, "traffic": None,
                "definition": "SURVEY.md 8(d): bytes per step = 24 P_train + 8 P_target + batch bytes = "
                              f"{STEP_BYTES} B; achieved = bytes x synchronous steps/s; peak = measured HBM copy bandwidth",
                "peak_source": peak_src,
                "tensor": {"flops_per_step": STEP_FLOPS, "tflops": STEP_FLOPS * sync_steps_per_s / 1e12,
                           "frac_of_bf16_peak": STEP_FLOPS * sync_steps_per_s / 1e12 / peak_tf,
                           "frac_of_3xtf32_ceiling": STEP_FLOPS * sync_steps_per_s / 1e12 / (peak_tf / 6.0),
                           "note": "fp32-accurate 3xTF32: three TF32 MMAs (half the bf16 rate) per product"}}
        tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")   # warm-cache DRAM bytes of one step (ncu)
        if os.path.exists(tp):
            tj = json.load(open(tp))
            roof["traffic"] = tj.get("dram_bytes_per_step")
            roof["traffic_source"] = tj.get("source")
    if rank == 0 and world == 1:
        prof = eng.profile(20)
        in_graph = bool(eng.lib.osrl_profile_was_in_graph(eng.h))
        agg = {}
        for name, pms, by, fl in prof:
            a = agg.setdefault(name, [0.0, 0.0, 0.0, 0])
            a[0] += pms; a[1] += by; a[2] += fl; a[3] += 1
        tot = sum(a[0] for a in agg.values())
        kern = []
        for k_, d in sorted(agg.items(), key=lambda kv: -kv[1][0]):
            tensor = k_.startswith("k_fz") or k_.startswith("k_gemm_mma") or k_.startswith("k_gemm_tc5")
            ent = {"kernel": k_, "launches_per_step": d[3], "us_per_step": 1e3 * d[0], "share_of_step_time": d[0] / tot,
                   "avg_launch_us": 1e3 * d[0] / d[3], "bound": "tensor" if tensor else "hbm",
                   "algorithmic_bytes_per_step": d[1], "algorithmic_flops_per_step": d[2],
                   "gbs": d[1] / (d[0] * 1e-3) / 1e9 if d[0] > 0 else None,
                   "tflops": d[2] / (d[0] * 1e-3) / 1e12 if d[0] > 0 else None}
            ent["frac"] = (ent["tflops"] / (peak_tf / 6.0)) if tensor else (ent["gbs"] / peak_gbs)
            ent["frac_of"] = "3xTF32 ceiling (bf16 peak / 6)" if tensor else "HBM peak (operands are L2-resident)"
            kern.append(ent)
        roof["kernels"] = kern
        roof["kernels_timing"] = ("per launch, inside a replayed CUDA graph with event-record nodes between launches "
                                  "(osrl_profile)" if in_graph else "eager launches with an event pair around each")
        roof["sequential_step_us"] = 1e3 * tot
        roof["note"] = ("the sequential step (sum of the kernels above) is longer than ms_per_step: osrl_steps overlaps the "
                        "VAE update of step s+1 with the critic / actor updates of step s on a second graph branch")

    # ---- BASELINE.json configs[2..4] (short runs) and the strong-scaling BEAR-Lag point
    others = {}
    for name, spec in OTHER.items():
        try:
            others[name] = run_other(name, spec["batch"], local, world, rank, barrier, peaks, comm_setup)
        except Exception as ex:   # a failure here must not take the headline number with it
            others[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    if 4096 % world == 0:
        try:
            r = run_other("bearl_b512", 4096 // world, local, world, rank, barrier, peaks, comm_setup)
            r["workload"] = "BEAR-Lag OfflineCarCircle-v0-shaped GLOBAL batch=4096 sharded over the GPUs (BASELINE.json configs[4], strong scaling)"
            r["hbm_frac"] = None if r.get("synchronous_steps_per_s") is None else \
                (24 * 954_454 + 8 * 620_044 + (4096 // world) * 84) * r["synchronous_steps_per_s"] / 1e9 / peak_gbs
            others["bearl_strong_b4096"] = r
        except Exception as ex:
            others["bearl_strong_b4096"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    # ---- SURVEY 8f rank 3: process_sequence_dataset on the device (rank 0, N == 1), next to the host restatements
    if rank == 0 and world == 1:
        try:
            others["seq_preprocess_1m"] = run_preprocess(local)
        except Exception as ex:
            others["seq_preprocess_1m"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- CPU baseline: the oracle port of the reference step on the host cores (bounded sample)
    cpu = None
    if world == 1:
        from oracle import synth
        orc = init_params()
        r2 = np.random.default_rng(0)
        keys = ("observations", "next_observations", "actions", "rewards", "costs", "done")
        tb = [[torch.from_numpy(b[k]) for k in keys] for b in (synth.make_batch(r2, BATCH, 8, 2) for _ in range(4))]
        cores, avail = calibrate_threads(lambda: orc.step(*tb[0]))
        t0 = time.perf_counter()
        kk = 0
        while time.perf_counter() - t0 < 12.0 and kk < 2000:
            orc.step(*tb[kk % 4])
            kk += 1
        dt = time.perf_counter() - t0
        cpu = {"value": kk / dt, "unit": "steps/s", "cores": cores, "kind": "port",
               "sample": f"{kk} BCQ-Lag train steps (batch 256) of the oracle port, pre-collated batches (no "
                         f"DataLoader); {cores} torch threads = fastest of a sweep up to the {avail} usable cores"}

    out = {
        "metric": "gradient-steps/sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": BATCH * world, "per_gpu_batch": BATCH,
                   "parallelism": f"dp{world}", "synchronous_steps_per_s": sync_steps_per_s,
                   "gradient_exchange": {"single": "none (1 GPU)", "nccl": "ncclAllReduce nodes in the step graph",
                                         "peer": "ordered sum out of NVLink peer memory inside the Adam kernel "
                                                 "(k_dp_adam), no NCCL on the step's path"}[dp_mode],
                   "value_is": "data-parallel ranks x synchronous steps/s (batch-256 step equivalents)",
                   "dataset_rows_per_gpu": DATASET_ROWS, "init": "osrl_b200.algorithms.BCQL under seed_all(0)",
                   "l2": "inputs larger than L2: the resident dataset is 192 MB per GPU and rows are drawn at "
                         "random; parameters/optimizer state (19 MB) are reused every step by construction"},
        "clocks": clk, "gpu_launches": int(launches),
        "e2e": {"value": e2e_batched, "unit": "steps/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h_batched), "steps": KB,
                "api": f"osrl_b200.algorithms.BCQLTrainer.train_batches({CHUNK} loader batches per call, pinned host "
                       "tensors) -> osrl_steps_host; per-step stats to the logger",
                "train_one_step": {"value": e2e_sync, "lagged_stats_value": e2e_v, "d2h_bytes_per_step": int(d2h),
                                   "steps": KE,
                                   "api": "BCQLTrainer.train_one_step per batch (the reference's loop unchanged): one "
                                          "synchronous sequential step graph per call; lagged = lag_stats=True"}},
        "other_configs": others,
    }
    if roof is not None:
        out["roofline"] = roof
    if cpu is not None:
        out["cpu_baseline"] = cpu
    if dp_parity is not None:
        out["dp_parity"] = dp_parity
    print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # libraries (NCCL's version banner, torchrun helpers) write to fd 1; the contract is ONE JSON line on stdout, so
    # everything but that line is sent to stderr
    global print
    real_out = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    _print = print

    def print(*a, **k):  # noqa: A001  (only the result lines go through here)
        k.setdefault("file", real_out)
        k.setdefault("flush", True)
        _print(*a, **k)

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
