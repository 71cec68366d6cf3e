"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz in the build container.

Runs the UNMODIFIED reference (imported from /root/reference through
oracle/ref_shim.py) and records, per case:
  * the run's known answers: K, conv_int, err, final trajectory u, dataset x / D;
  * a sample of `NNGP_p.predict` calls (query, dataset length, neighbour count,
    host-drawn Nelder-Mead starts, returned prediction) so the kernel-level
    oracle (oracle/nngp.py) can be pinned call by call;
  * RK / vector-field known answers of RK.py + systems.py.
The reference does not travel to the GPU box, the fixtures do.

usage: python -m oracle.make_golden <case> [<case> ...] | all
"""
import json
import os
import pickle
import sys
import time

import numpy as np

from .ref_shim import load_reference, REF_DIR

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _build(ns, system, N=None, d_x=None, **over):
    S = ns.systems
    if system == "lorenz":
        ode = S.Lorenz(normalization="-11", use_jax=False)
        cfg = ns.configs.Config(ode).get()
    elif system == "hopf":
        ode = S.Hopf(normalization="-11", use_jax=False)
        cfg = ns.configs.Config(ode, N=N).get()
    elif system == "brusselator":
        ode = S.Brusselator(normalization="-11", use_jax=False)
        cfg = ns.configs.Config(ode).get()
    elif system == "burgers":
        ode = S.Burgers(d_x=d_x, normalization="-11", use_jax=False)
        cfg = dict(tspan=[0, 5.9], N=N, Ng=4, Nf=2000, G="RK1", F="RK8")
    elif system == "fhn_pde":
        ode = S.FHN_PDE(d_x=d_x, use_jax=False)
        cfg = ns.configs.Config(ode, d_x=d_x).get()
    else:
        raise ValueError(system)
    cfg = dict(cfg)
    cfg.update(over)
    if N is not None and system not in ("hopf",):
        # keep the per-slice resolution of the preset, shrink the number of slices
        if system == "lorenz":
            cfg["tspan"] = [0, 18 * N / 50]
        elif system == "fhn_pde":
            cfg["tspan"] = [0, cfg["tspan"][1] * N / 512]
        cfg["N"] = N
    return ode, cfg


CASES = {
    # name: (system, build kwargs, model kwargs, epsilon, every-nth predict sampled)
    "lorenz_N50_m11": ("lorenz", {}, dict(nn=11, seed=45), 5e-7, 13),
    "lorenz_N32_m11": ("lorenz", dict(N=32), dict(nn=11, seed=45), 5e-7, 11),
    "lorenz_N50_adaptive": ("lorenz", {}, dict(nn="adaptive", seed=46), 5e-7, 17),
    "brusselator_N25_m12_R2": ("brusselator", {}, dict(nn=12, seed=45, n_restarts=2), 5e-7, 9),
    "hopf_N32_m15": ("hopf", dict(N=32), dict(nn=15, seed=45), 5e-7, 15),
    "burgers_d32_N32_m12": ("burgers", dict(N=32, d_x=32), dict(nn=12, seed=45), 5e-7, 29),
    "fhn_d32_N32_m12": ("fhn_pde", dict(N=32, d_x=4), dict(nn=12, seed=45), 5e-7, 29),
    # round 2: the BASELINE.json configurations at (or near) their stated sizes, m = 15 / 18 / 20
    "fhn_d128_N128_m20": ("fhn_pde", dict(N=128, d_x=8), dict(nn=20, seed=45), 5e-7, 41),
    # the first 64 slices of the FHN d=512 target (same d, m, G and F resolution per slice: plain Parareal needs > 30
    # iterations here, while FHN at d_x <= 12 converges in 2 whatever the model does)
    "fhn_d512_N64_m20": ("fhn_pde", dict(N=64, d_x=16), dict(nn=20, seed=45), 5e-7, 37),
    "burgers_d128_N128_m18": ("burgers", dict(N=128, d_x=128), dict(nn=18, seed=45), 5e-7, 61),
    "hopf_N64_m15_R2": ("hopf", dict(N=64), dict(nn=15, seed=45, n_restarts=2), 5e-7, 37),
    "hopf_N128_m15_R2": ("hopf", dict(N=128), dict(nn=15, seed=45, n_restarts=2), 5e-7, 97),
    "hopf_N256_m15_R2": ("hopf", dict(N=256), dict(nn=15, seed=45, n_restarts=2), 5e-7, 211),
    "hopf_N512_m15_R2": ("hopf", dict(N=512), dict(nn=15, seed=45, n_restarts=2), 5e-7, 499),
}
# no test replays predicts on the dataset of these runs, and with it their fixtures would exceed 1 MB
NO_DATASET = {"fhn_d512_N64_m20", "burgers_d128_N128_m18"}


def run_case(name):
    ns = load_reference(fast_kernel=True)
    system, bkw, mkw, eps, every = CASES[name]
    ode, cfg = _build(ns, system, **bkw)
    solver = ns.solver.SolverRK(ode.get_vector_field(), use_jax=False, **cfg)
    samples = []
    counter = [0]

    class Recording(ns.models.NNGP_p):
        # the reference's own extension idiom (Figure_2.py:304-452): subclass and wrap predict
        def get_preds(self, xm, ym, n, new_x, intrvl_i):
            state = self.rng.bit_generator.state
            out = super().get_preds(xm, ym, n, new_x, intrvl_i)
            if counter[0] % every == 0:
                probe = np.random.default_rng()
                probe.bit_generator.state = state
                n_tasks = n * 9 * self.n_restarts
                starts = np.stack([probe.integers(-8, 0, 2) for _ in range(n_tasks)])
                samples.append(dict(call=counter[0], k=self.k, i=intrvl_i, n_rows=self.x.shape[0],
                                    m=xm.shape[0], query=np.array(new_x).ravel().copy(),
                                    starts=starts.reshape(n, 9, self.n_restarts, 2).astype(np.int8),
                                    preds=np.array(out).copy()))
            counter[0] += 1
            return out

    class P(ns.parareal.Parareal):
        # reference idiom for a custom model: override _run (nnGPara_with_time.py:187-215)
        def _run(self, **kwargs):
            mdl = Recording(n=self.n, N=self.N, worker_pool=kwargs["pool"], **mkw)
            return self._parareal(mdl, **kwargs)

    p = P(ode, solver, epsilon=eps, verbose="", **cfg)
    t0 = time.time()
    # NNGP_GOLDEN_POOL=n farms the Nelder-Mead searches over n forked processes through the reference's own
    # executor seam (parareal.py:58-64); the start points are drawn in the parent, so the run is identical
    workers = int(os.environ.get("NNGP_GOLDEN_POOL", "0"))
    out = p.run(pool=workers) if workers > 0 else p.run()
    secs = time.time() - t0
    K = out["k"]
    arrays = dict(K=K, conv_int=np.array(out["conv_int"]), err=out["err"], u_final=out["u"][:, :, K - 1]
                  if out["u"].ndim == 3 else out["u"], u_last=out["u"][:, :, -1], x=out["x"], D=out["D"],
                  t=out["t"], u0=ode.get_init_cond(), n_predict_calls=counter[0], seconds=secs,
                  cfg=json.dumps({k: (v if not isinstance(v, np.ndarray) else v.tolist()) for k, v in cfg.items()}),
                  model_kwargs=json.dumps(mkw), epsilon=eps)
    if name in NO_DATASET:
        del arrays["x"], arrays["D"]
    for s_i, s in enumerate(samples):
        for key, val in s.items():
            arrays[f"s{s_i}_{key}"] = val
    arrays["n_samples"] = len(samples)
    np.savez_compressed(os.path.join(OUT, f"run_{name}.npz"), **arrays)
    print(name, "K", K, "conv_int", out["conv_int"], f"{secs:.1f}s", "samples", len(samples), flush=True)


GP_CASES = {
    # GParareal (models.py:273-473, `GPjax_p`): the full-dataset GP, needed for the three-way comparison of BASELINE configs[2]
    "burgers_d32_N32_gp": ("burgers", dict(N=32, d_x=32), {}, 5e-7),
    "lorenz_N32_gp": ("lorenz", dict(N=32), {}, 5e-7),
}


def run_gp_case(name):
    """runs the unmodified reference with model='gpjax' and records K, conv_int, err, the final iterate, the dataset
    and the hyper-parameters / jitters selected in every iteration (GPjax_p.hyp, models.py:281, 425-426)"""
    ns = load_reference(fast_kernel=True)
    system, bkw, mkw, eps = GP_CASES[name]
    ode, cfg = _build(ns, system, **bkw)
    solver = ns.solver.SolverRK(ode.get_vector_field(), use_jax=False, **cfg)
    trace = []

    class Recording(ns.models.GPjax_p):
        def fit(self, x, y, k, *a, **kw):
            super().fit(x, y, k, *a, **kw)
            trace.append((k, x.shape[0], np.array(self.thetas, dtype=float).copy(), np.array(self.jitters, dtype=float).copy()))

    class P(ns.parareal.Parareal):
        def _run(self, **kwargs):
            mdl = Recording(n=self.n, N=self.N, worker_pool=kwargs["pool"], **mkw)
            return self._parareal(mdl, **kwargs)

    p = P(ode, solver, epsilon=eps, verbose="", **cfg)
    t0 = time.time()
    workers = int(os.environ.get("NNGP_GOLDEN_POOL", "0"))
    out = p.run(pool=workers) if workers > 0 else p.run()
    secs = time.time() - t0
    K = out["k"]
    arrays = dict(K=K, conv_int=np.array(out["conv_int"]), err=out["err"], u_last=out["u"][:, :, -1], x=out["x"], D=out["D"],
                  t=out["t"], u0=ode.get_init_cond(), seconds=secs,
                  cfg=json.dumps({k: (v if not isinstance(v, np.ndarray) else v.tolist()) for k, v in cfg.items()}),
                  model_kwargs=json.dumps(mkw), epsilon=eps, n_fits=len(trace))
    for i, (k, rows, th, jit) in enumerate(trace):
        arrays[f"f{i}_k"], arrays[f"f{i}_rows"], arrays[f"f{i}_thetas"], arrays[f"f{i}_jitters"] = k, rows, th, jit
    np.savez_compressed(os.path.join(OUT, f"run_{name}.npz"), **arrays)
    print(name, "K", K, "conv_int", out["conv_int"], f"{secs:.1f}s", flush=True)


def rk_vectors():
    """Known answers of RK.py (`_RK_numpy_` via run_get_last) and systems.py vector fields."""
    ns = load_reference()
    S = ns.systems
    rng = np.random.default_rng(7)
    out = {}
    systems = {
        "lorenz": S.Lorenz(normalization="-11", use_jax=False),
        "lorenz_id": S.Lorenz(use_jax=False),
        "hopf": S.Hopf(normalization="-11", use_jax=False),
        "rossler": S.Rossler(normalization="-11", use_jax=False),
        "fhn_ode": S.FHN_ODE(normalization="-11", use_jax=False),
        "brusselator": S.Brusselator(normalization="-11", use_jax=False),
        "dblpend": S.DblPend(normalization="-11", use_jax=False),
        "thomas": S.ThomasLabyrinth(normalization="-11", use_jax=False),
        "burgers128": S.Burgers(d_x=128, normalization="-11", use_jax=False),
        "burgers32": S.Burgers(d_x=32, normalization="-11", use_jax=False),
        "fhn16": S.FHN_PDE(d_x=16, use_jax=False),
        "fhn4": S.FHN_PDE(d_x=4, use_jax=False),
        "fhn4_n": S.FHN_PDE(d_x=4, normalization="-11", use_jax=False),
    }
    for name, ode in systems.items():
        f = ode.get_vector_field()
        u0 = ode.get_init_cond()
        d = u0.shape[0]
        n_pts = 6
        U = np.stack([u0] + [u0 + 0.05 * rng.standard_normal(d) for _ in range(n_pts - 1)])
        out[f"{name}_u"] = U
        out[f"{name}_f"] = np.stack([f(0.3, u) for u in U])
        for method, steps in (("RK1", 7), ("RK2", 5), ("RK4", 6), ("RK8", 4)):
            rk = ns.RK.RK(f, method, use_jax=False)
            t0, t1 = 0.37, 0.37 + (0.36 if d < 10 else 0.05)
            out[f"{name}_{method}_t"] = np.array([t0, t1, steps])
            out[f"{name}_{method}_u1"] = np.stack([rk.run_get_last(t0, t1, steps, u) for u in U[:3]])
    np.savez_compressed(os.path.join(OUT, "rk_vectors.npz"), **out)
    print("rk_vectors", len(out), flush=True)


class _Stub:
    def __setstate__(self, state):
        self.__dict__.update(state if isinstance(state, dict) else {})


class _Unpickler(pickle.Unpickler):
    def find_class(self, module, name):
        try:
            return super().find_class(module, name)
        except Exception:
            return type(name, (_Stub,), {})


def published():
    """Known answers mined from the reference's published result pickles (SURVEY.md section 4)."""
    res = {}

    def load(path):
        with open(os.path.join(REF_DIR, path), "rb") as fh:
            return _Unpickler(fh).load()

    def summarize(obj, key_hint=None):
        runs = getattr(obj, "runs", None) or (obj.get("runs") if isinstance(obj, dict) else None)
        out = {}
        for mname, r in runs.items():
            e = np.asarray(r["err"])
            out[mname] = dict(K=int(r["k"]), conv_int=[int(v) for v in r.get("conv_int", [])],
                              err_max_per_iter=[float(np.nanmax(e[:, c])) for c in range(e.shape[1])])
        return out

    for rel in ["FHN_scal_times/FHN_scal_times_16_512_nngp", "FHN_scal_times/FHN_scal_times_16_512_para",
                "Burges_scal_final/Burges_scal_final_5.9_128_nngp"] + \
               [f"nonaut_scal_final/nonaut_scal_final_{n}_nngp" for n in (32, 64, 128, 256, 512)]:
        try:
            res[rel] = summarize(load(rel))
        except Exception as e:  # noqa
            res[rel] = {"error": repr(e)}
    try:
        rows = load("NNGP_all_but_pend")
        res["NNGP_all_but_pend"] = [[str(r[0]), int(r[1]), float(r[2]), str(r[3]), int(r[4]), float(r[5]), int(r[6])]
                                    for r in rows if isinstance(r[1], (int, np.integer)) and isinstance(r[6], (int, np.integer))]
    except Exception as e:  # noqa
        res["NNGP_all_but_pend"] = {"error": repr(e)}
    # Burgers_perf_across_m.py:98-131: rows [N, nn, seed, K, runtime, F_time, mdl_tot_t] of ~100 random seeds x nn = 11..30
    # (d = N = 128, T = 5 or 5.9 (file name), G = RK1 x 4, F = RK8 x 2000 per slice, '-11' normalisation): the published
    # distribution of K; stored as [T, nn, seed, K]
    try:
        rows = []
        bdir = os.path.join(REF_DIR, "Burges_nngp_exp_val_speed")
        for fn in sorted(os.listdir(bdir)):
            for r in load(os.path.join("Burges_nngp_exp_val_speed", fn)):
                if len(r) == 7 and int(r[3]) > 0 and int(r[0]) == 128:
                    rows.append([float(fn.split("_")[-3]), int(r[1]), int(r[2]), int(r[3])])
        res["Burgers_K_vs_m"] = sorted(rows)
    except Exception as e:  # noqa
        res["Burgers_K_vs_m"] = {"error": repr(e)}
    with open(os.path.join(OUT, "published.json"), "w") as fh:
        json.dump(res, fh, indent=0)
    print("published", {k: (v if not isinstance(v, list) else len(v)) for k, v in res.items()
                        if "error" in str(v)[:12] or isinstance(v, list)}, flush=True)


def rk_full_vectors():
    """Known answers of RK.run (`_RK_numpy_`, every step): what SolverRK.run_F_full / run_G_full return."""
    ns = load_reference()
    S = ns.systems
    rng = np.random.default_rng(11)
    out = {}
    systems = {
        "lorenz": S.Lorenz(normalization="-11", use_jax=False),
        "hopf": S.Hopf(normalization="-11", use_jax=False),
        "burgers32": S.Burgers(d_x=32, normalization="-11", use_jax=False),
        "fhn4": S.FHN_PDE(d_x=4, use_jax=False),
        "fhn6": S.FHN_PDE(d_x=6, use_jax=False),
    }
    for name, ode in systems.items():
        f = ode.get_vector_field()
        u0 = ode.get_init_cond() + 0.01 * rng.standard_normal(ode.get_dim())
        out[f"{name}_u0"] = u0
        for method, steps in (("RK1", 9), ("RK4", 7), ("RK8", 12)):
            rk = ns.RK.RK(f, method, use_jax=False)
            t0, t1 = 0.21, 0.21 + (0.4 if u0.shape[0] < 10 else 0.06)
            out[f"{name}_{method}_t"] = np.array([t0, t1, steps])
            out[f"{name}_{method}_traj"] = rk.run(t0, t1, steps, u0)
    np.savez_compressed(os.path.join(OUT, "rk_full_vectors.npz"), **out)
    print("rk_full_vectors", len(out), flush=True)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    todo = sys.argv[1:] or ["all"]
    if todo == ["all"]:
        todo = ["rk_vectors", "rk_full_vectors", "published"] + list(CASES)
    for item in todo:
        if item == "rk_vectors":
            rk_vectors()
        elif item == "rk_full_vectors":
            rk_full_vectors()
        elif item == "published":
            published()
        elif item in GP_CASES:
            run_gp_case(item)
        else:
            run_case(item)
