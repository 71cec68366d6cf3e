"""Shared builders for the parity tests: the same named case on the oracle and on the device."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_run(name):
    z = np.load(os.path.join(GOLDEN, f"run_{name}.npz"), allow_pickle=False)
    cfg = json.loads(str(z["cfg"]))
    mkw = json.loads(str(z["model_kwargs"]))
    return z, cfg, mkw


def case_system(name):
    """'lorenz_N50_m11' -> (system key, kwargs)"""
    parts = name.split("_")
    key = parts[0]
    d = next((int(p[1:]) for p in parts[1:] if p[0] == "d" and p[1:].isdigit()), None)
    if key == "burgers":
        return "burgers", dict(d_x=d or 32)
    if key == "fhn":
        return "fhn_pde", dict(d_x=int(round((d / 2) ** 0.5)) if d else 4)  # d = 2 d_x^2
    return key, {}


def oracle_system(key, **kw):
    from oracle import systems as osys
    return {"lorenz": lambda: osys.Lorenz(normalization="-11"),
            "hopf": lambda: osys.Hopf(normalization="-11"),
            "burgers": lambda: osys.Burgers(normalization="-11", **kw),
            "fhn_pde": lambda: osys.FHN_PDE(**kw)}[key]()


def device_system(key, **kw):
    import nearest_neighbors_gparareal_b200 as nn
    return {"lorenz": lambda: nn.Lorenz(normalization="-11"),
            "hopf": lambda: nn.Hopf(normalization="-11"),
            "burgers": lambda: nn.Burgers(normalization="-11", **kw),
            "fhn_pde": lambda: nn.FHN_PDE(**kw)}[key]()


def make_dataset(rng, n, d):
    x = rng.uniform(-1, 1, (n, d))
    y = 1e-3 * np.sin(x @ (rng.standard_normal((d, d)) / np.sqrt(d)))
    return x, y


def scaled_err(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def samples(z):
    out = []
    for i in range(int(z["n_samples"])):
        out.append({k: z[f"s{i}_{k}"] for k in ("call", "k", "i", "n_rows", "m", "query", "starts", "preds")})
    return out
