"""One-time dataset preprocessing restated on flat arrays (osrl_b200/common/dataset.py) pinned against the UNMODIFIED
reference (osrl/common/dataset.py) on seeded synthetic data: process_bc_dataset (all modes incl. the Pareto frontier),
SequenceDataset with the reference's default Pareto-frontier augmentation, random augmentation, pf_only and the
sampling-probability variants.  The reference needs `oapackage` for the frontier; tests/stubs/oapackage.py restates
its two classes (brute-force non-dominated set).  What the reference computes is stored in
tests/golden/reference_dataset.npz (record_reference below, run by oracle/record_reference.py): arrays compared for
equality as sha256 digests; of SequenceDataset's relabelled targets and start probabilities, every trajectory's first
target and the whole of a fixed sample of trajectories; everything else as is."""
import random

import numpy as np
import pytest

from oracle import synth
from tests import helpers

MODES = ["all", "multi-task", "safe", "risky", "boundary", "frontier"]
GAMMAS = [1.0, 0.99]
TRAJ_SAMPLE = 64       # trajectories of each SequenceDataset case stored whole


@pytest.fixture(scope="module")
def ref_dataset():
    return helpers.load_pin("dataset")


def _data(seed=3, eps=60, T=37):
    d = synth.make_dataset(6, 2, T, eps, seed=seed)
    rng = np.random.default_rng(seed)
    d["costs"] = (rng.random(d["costs"].shape) < rng.uniform(0.02, 0.5, eps).repeat(T)).astype(np.float32)
    d["rewards"] = (d["rewards"] + rng.uniform(0, 1.5, eps).repeat(T)).astype(np.float32)
    d["timeouts"][-5:] = False
    return d


def test_pareto_front_matches_brute_force():
    from osrl_b200.common.dataset import pareto_front_2d
    rng = np.random.default_rng(1)
    for n in (1, 7, 300):
        c = rng.integers(0, 25, n).astype(float)
        r = (c * 0.7 + rng.integers(0, 12, n)).astype(float)
        brute = [i for i in range(n) if not any((c[j] <= c[i] and r[j] >= r[i]) and (c[j] < c[i] or r[j] > r[i]) for j in range(n))]
        assert brute == pareto_front_2d(c, r)


def bc_columns(process_bc_dataset, mode, gamma):
    b = {k: v.copy() for k, v in _data().items()}
    process_bc_dataset(b, 6, gamma, mode)
    return {k: (v.dtype.str, helpers.digest(v, keep_dtype=False)) for k, v in b.items()}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("gamma", GAMMAS)
def test_process_bc_dataset(ref_dataset, mode, gamma):
    from osrl_b200.common.dataset import process_bc_dataset
    a = ref_dataset["bc"][f"{mode}/{gamma}"]
    b = bc_columns(process_bc_dataset, mode, gamma)
    assert set(a) == set(b)
    for k in a:
        assert tuple(a[k]) == b[k], (mode, gamma, k)


CASES = {
    "default_augmentation": dict(augment_percent=0.2, deg=2, max_rew_decrease=100.0, max_reward=60.0, min_reward=1.0,
                                 cost_sample=True, cost_transform=lambda x: 70 - x),
    "random_aug": dict(random_aug=0.3, aug_rmin=20, aug_rmax=40, aug_cmin=2, aug_cmax=12, cgap=1, cost_sample=True,
                       cost_transform=lambda x: 70 - x),
    "pf_only": dict(pf_only=True, rmin=10, cost_bins=10, npb=2),
    "pf_sample": dict(augment_percent=0.2, deg=2, max_rew_decrease=100.0, max_reward=60.0, min_reward=1.0, pf_sample=True),
    "start_sampling": dict(start_sampling=True, prob=0.3, cost_sample=True, cost_transform=lambda x: 70 - x),
    "cost_reverse": dict(cost_reverse=True, cost_sample=True, cost_transform=lambda x: 70 - x),
}


def _sequence_dataset(cls, case):
    d = _data(seed=5, eps=900, T=16)   # enough trajectories for the 10 x 50 outlier grid (bins of <= 2 are dropped)
    np.random.seed(7); random.seed(7)
    return cls({k: v.copy() for k, v in d.items()}, seq_len=10, reward_scale=0.1, cost_scale=1.0, **CASES[case])


def _windows(ds):
    np.random.seed(11); random.seed(11)
    return [x for _, x in zip(range(5), iter(ds))]


def _sources_digest(trajs):
    """one digest of every trajectory's (observations, actions, costs), compared by value"""
    return helpers.digest(np.array([helpers.digest(x, keep_dtype=False) for t in trajs for x in t]))


def record_sequence_case(SequenceDataset, case):
    ref = _sequence_dataset(SequenceDataset, case)
    trajs = ref.dataset
    first = np.array([[t["returns"][0], t["cost_returns"][0]] for t in trajs])
    sample = np.sort(np.random.default_rng(0).choice(len(trajs), min(TRAJ_SAMPLE, len(trajs)), replace=False))
    out = {"n": len(trajs), "lengths": np.array([len(t["returns"]) for t in trajs], np.int64),
           "sources": _sources_digest([(t["observations"], t["actions"], t["costs"]) for t in trajs]),
           "first": first, "sample": sample,
           "sample_returns": [np.asarray(trajs[i]["returns"]) for i in sample],
           "sample_cost_returns": [np.asarray(trajs[i]["cost_returns"]) for i in sample],
           "sample_prob": None if ref.sample_prob is None else np.asarray(ref.sample_prob),
           "windows": [tuple(np.asarray(u) for u in x) for x in _windows(ref)]}
    if CASES[case].get("start_sampling"):
        out["n_start_idx_sample_prob"] = len(ref.start_idx_sample_prob)
        out["start_idx_sample_prob"] = [np.asarray(ref.start_idx_sample_prob[i]) for i in sample]
    return out


@pytest.mark.parametrize("case", sorted(CASES))
def test_sequence_dataset_modes(ref_dataset, case):
    """Same seeds -> same trajectories (sources, relabelled return / cost to go), same sampling probabilities, and the
    same windows from the iterator."""
    from osrl_b200.common.dataset import SequenceDataset
    ref = ref_dataset["seq"][case]
    mine = _sequence_dataset(SequenceDataset, case)
    assert ref["n"] == len(mine)
    assert np.array_equal(ref["lengths"], [hi - lo for lo, hi, _, _ in mine._traj]), case
    assert ref["sources"] == _sources_digest([(mine._obs[lo:hi], mine._act[lo:hi], mine._cost[lo:hi])
                                              for lo, hi, _, _ in mine._traj]), case
    # (relabelled targets: the frontier fit sees the same points in a different order -- 1e-6 relative)
    rtol, atol = 2e-6, 1e-5
    rtg = [np.asarray(t[2]) for t in mine._traj]
    ctg = [np.asarray(t[3]) for t in mine._traj]
    got_first = np.array([[r[0], c[0]] for r, c in zip(rtg, ctg)])
    assert np.allclose(ref["first"], got_first, rtol=rtol, atol=atol), case
    for i, w_r, w_c in zip(ref["sample"], ref["sample_returns"], ref["sample_cost_returns"]):
        assert np.allclose(w_r, rtg[i], rtol=rtol, atol=atol) and np.allclose(w_c, ctg[i], rtol=rtol, atol=atol), (case, i)
    if ref["sample_prob"] is None:
        assert mine.sample_prob is None
    else:
        assert np.allclose(ref["sample_prob"], mine.sample_prob, rtol=1e-5, atol=1e-9)
    if CASES[case].get("start_sampling"):
        assert ref["n_start_idx_sample_prob"] == len(mine.start_idx_sample_prob)
        for i, a in zip(ref["sample"], ref["start_idx_sample_prob"]):
            assert np.allclose(a, mine.start_idx_sample_prob[i], rtol=1e-6)
    for x, y in zip(ref["windows"], _windows(mine), strict=True):
        for u, v in zip(x, y):
            assert np.asarray(u).dtype == np.asarray(v).dtype and np.allclose(u, v, rtol=2e-6, atol=1e-5), case


SPLIT_KEYS = ("observations", "actions", "rewards", "costs", "returns", "cost_returns")


def _split_data():
    d = _data(seed=9, eps=40, T=23)
    rng = np.random.default_rng(2)
    d["costs"] = np.where(rng.random(d["costs"].shape) < 0.5, d["costs"], rng.random(d["costs"].shape)).astype(np.float32)
    d["terminals"][40] = True
    return d


def _split_digests(trajs):
    return [[(t[k].dtype.str, helpers.digest(t[k], keep_dtype=False)) for k in SPLIT_KEYS] for t in trajs]


@pytest.mark.parametrize("cost_reverse", [False, True])
def test_oracle_split_trajectories_is_the_reference(ref_dataset, cost_reverse):
    """oracle/cdt.py: split_trajectories -- the checker of the device preprocessing (tests/test_gpu_preproc.py) --
    against the unmodified process_sequence_dataset (dataset.py:137-183), bit for bit, with fractional costs, a
    trailing unfinished episode and both end flags."""
    from oracle import cdt as ocdt
    want = ref_dataset["split"][str(cost_reverse)]
    got = _split_digests(ocdt.split_trajectories(_split_data(), cost_reverse))
    assert len(want) == len(got)
    for w, g in zip(want, got):
        for k, wk, gk in zip(SPLIT_KEYS, w, g):
            assert tuple(wk) == gk, k


def _transition_data():
    d = _data(seed=4, eps=12, T=9)
    d["terminals"][20] = True
    return d


def _transition_record(ds, state_init):
    np.random.seed(2)
    it = iter(ds)
    out = {"columns": {k: ds.dataset[k] for k in ("done",) + (("is_init",) if state_init else ())},
           "stream": [tuple(np.asarray(x) for x in next(it)) for _ in range(25)]}
    if state_init:
        out["states"] = [np.asarray(x) for x in ds.get_dataset_states()]
    return out


@pytest.mark.parametrize("state_init", [False, True])
def test_transition_dataset_stream_is_the_reference(ref_dataset, state_init):
    """TransitionDataset (dataset.py:790-847): done / is_init columns, the float32 scaling of rewards and costs, the
    tuple layout and the index stream of __iter__ under the same numpy seed; get_dataset_states for COptiDICE."""
    from osrl_b200.common.dataset import TransitionDataset
    a = ref_dataset["transition"][str(state_init)]
    b = _transition_record(TransitionDataset(_transition_data(), 0.1, 3.0, state_init), state_init)
    for k, w in a["columns"].items():
        assert w.dtype == b["columns"][k].dtype and np.array_equal(w, b["columns"][k]), k
    for w, g in zip(a["stream"], b["stream"], strict=True):
        assert len(w) == len(g) == (7 if state_init else 6)
        for x, y in zip(w, g):
            assert x.dtype == y.dtype and np.array_equal(x, y)
    if state_init:
        for x, y in zip(a["states"], b["states"], strict=True):
            assert np.array_equal(x, y)


def record_reference(osrl):
    rd = osrl.common.dataset
    return {"bc": {f"{m}/{g}": bc_columns(rd.process_bc_dataset, m, g) for m in MODES for g in GAMMAS},
            "seq": {case: record_sequence_case(rd.SequenceDataset, case) for case in sorted(CASES)},
            "split": {str(c): _split_digests(rd.process_sequence_dataset(_split_data(), c)[0]) for c in (False, True)},
            "transition": {str(s): _transition_record(rd.TransitionDataset(_transition_data(), 0.1, 3.0, s), s)
                           for s in (False, True)}}
