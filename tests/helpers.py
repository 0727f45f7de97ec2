"""Shared helpers of the parity tests (the oracle is the checker, never the product)."""
import copy
import hashlib
import json
import os

import numpy as np
import torch

from oracle import algos

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ORACLES = {"bc": (algos.BCOracle, algos.BCConfig), "bcql": (algos.BCQLOracle, algos.BCQLConfig),
           "cpq": (algos.CPQOracle, algos.CPQConfig), "bearl": (algos.BEARLOracle, algos.BEARLConfig)}
# tolerance named by BASELINE.json north_star: losses and parameter deltas within 1e-5 relative
RTOL = 1e-5


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    return z, meta


# ---- what the unmodified reference computed, stored so that the comparisons with it run anywhere.  A pin is a nested
# structure of dicts (str keys), lists, tuples, scalars and numpy arrays; oracle/record_reference.py writes one per test
# module as tests/golden/reference_<name>.npz: the structure as JSON, the arrays' bytes back to back in one member.
def save_pin(name, obj):
    blob = []
    size = 0

    def enc(x):
        nonlocal size
        if isinstance(x, np.ndarray):
            blob.append(x.tobytes())      # (C order)
            size += x.nbytes
            return {"__array__": [x.dtype.str, list(x.shape), size - x.nbytes]}
        if isinstance(x, dict):
            assert all(isinstance(k, str) and not k.startswith("__") for k in x), list(x)
            return {k: enc(v) for k, v in x.items()}
        if isinstance(x, (list, tuple)):
            out = [enc(v) for v in x]
            return {"__tuple__": out} if isinstance(x, tuple) else out
        assert x is None or isinstance(x, (bool, int, float, str)), type(x)
        return x

    meta = json.dumps(enc(obj))
    np.savez_compressed(os.path.join(GOLDEN, f"reference_{name}.npz"), meta=meta,
                        data=np.frombuffer(b"".join(blob), np.uint8))


def load_pin(name):
    z = np.load(os.path.join(GOLDEN, f"reference_{name}.npz"), allow_pickle=False)
    data = z["data"]

    def dec(x):
        if isinstance(x, dict):
            if "__array__" in x:
                dtype, shape, off = x["__array__"]
                n = int(np.prod(shape)) * np.dtype(dtype).itemsize
                return data[off:off + n].view(dtype).reshape(shape)
            if "__tuple__" in x:
                return tuple(dec(v) for v in x["__tuple__"])
            return {k: dec(v) for k, v in x.items()}
        if isinstance(x, list):
            return [dec(v) for v in x]
        return x

    return dec(json.loads(str(z["meta"])))


def digest(a, keep_dtype=True):
    """A 64-bit sha256 prefix of an array's shape and bytes (and dtype; keep_dtype=False compares values only, as
    float64): equal digests <=> np.array_equal (and the same dtype)."""
    a = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a)
    if not keep_dtype:
        a = a.astype(np.float64)
    h = hashlib.sha256(f"{a.dtype.str if keep_dtype else ''}{a.shape}".encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def make_oracle(algo, cfg_dict, init_seed=0):
    cls, cfgcls = ORACLES[algo]
    torch.manual_seed(init_seed)
    return cls(cfgcls(**cfg_dict))


def batch_tuple(algo, b, dtype=torch.float32):
    t = {k: torch.as_tensor(np.asarray(v)).to(dtype) for k, v in b.items()}
    if algo == "bc":
        return (t["observations"], t["actions"])
    return (t["observations"], t["next_observations"], t["actions"], t["rewards"], t["costs"], t["done"])


def to_double(orc):
    """float64 twin of an oracle at its current state (conditioning probe)."""
    o = copy.deepcopy(orc)
    for k in list(o.params):
        o.params[k] = o.params[k].detach().double()
    for st in (o.opt.values() if isinstance(o.opt, dict) else [o.opt]):
        st.m = {k: v.double() for k, v in st.m.items()}
        st.v = {k: v.double() for k, v in st.v.items()}
    if hasattr(o, "pid"):
        o.pid.e_old, o.pid.e_int = o.pid.e_old.double(), o.pid.e_int.double()
    if hasattr(o, "log_alpha"):
        o.log_alpha = o.log_alpha.double()
    return o


def probe_step(orc, algo, batch, noise=None):
    """One reference step in fp32 (the reference path) and one in fp64 from the same state with the same
    noise.  Returns (stats32, stats64, grads32, grads64, params_before, params64_after).  The fp32/fp64 gap
    measures how well-conditioned each quantity is: a ReLU unit whose pre-activation rounds to +-0, or an
    Adam update with |g| ~ eps, makes the reference itself irreproducible at 1e-5."""
    o64 = to_double(orc)
    before = {k: v.detach().clone() for k, v in orc.params.items()}
    s32 = orc.step(*batch_tuple(algo, batch), noise=noise)
    nz = {k: v.double() for k, v in orc.last_noise.items()}
    with algos.precision(torch.float64):
        s64 = o64.step(*batch_tuple(algo, batch, torch.float64), noise=nz)
    g32 = {k: v.detach() for k, v in orc.last_grads.items()}
    g64 = {k: v.detach() for k, v in o64.last_grads.items()}
    return s32, s64, g32, g64, before, {k: v.detach() for k, v in o64.params.items()}


def maxrel(a, b):
    """max |a-b| / max |b|"""
    return float((a.double() - b.double()).abs().max()) / (float(b.double().abs().max()) + 1e-300)


def l2rel(a, b):
    return float((a.double() - b.double()).norm()) / (float(b.double().norm()) + 1e-300)


# ---- measured parity margins (VERDICT r1: "print and commit the measured worst error per quantity").  Every GPU
# comparison reports (test, quantity, err, tol); conftest writes the per-quantity worst err / tol of the session to
# gpurun_out/parity_margins.json, which is committed as profiles/r02_parity_margins.json.
MARGINS = {}


def record_margin(test: str, quantity: str, err: float, tol: float):
    key = f"{test}::{quantity}"
    cur = MARGINS.get(key)
    ratio = float(err) / float(tol) if tol > 0 else float("inf")
    if cur is None or ratio > cur["worst_ratio"]:
        MARGINS[key] = {"worst_ratio": ratio, "err": float(err), "tol": float(tol), "n": (cur["n"] if cur else 0) + 1}
    else:
        cur["n"] += 1
