"""GPU: the published seed studies as per-nn ensembles against one ensemble whose members differ in nn (and T).

1. NNGP_all_but_pend, per system: one PararealEnsemble per nn value (today's only option) against one ensemble of all
   the system's runs with a per-member nn.  Runs/s of both arms, alternated, each arm warmed up once; every member's K
   must be the same in both arms.
2. A Burgers_K_vs_m sample, T in {5.0, 5.9} x nn in 11..30 x `n_seeds` published seeds: the per-(T, nn) ensembles
   against one ensemble, alternated twice; runs/s and the histogram of K_ensemble - K_published.
Writes profiles/r07/ensemble_study.json and .log with the card name and power limit read in the same process.
usage: ensemble_study.py [--burgers-seeds 8] [--out profiles/r07]"""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import nearest_neighbors_gparareal_b200 as nn

ODES = {"fhn_n": (lambda: nn.FHN_ODE(normalization='-11'), {}, 10),
        "rossler_long_n": (lambda: nn.Rossler(normalization='-11'), {}, 18),
        "non_aut32_n": (lambda: nn.Hopf(normalization='-11'), dict(N=32), 16),
        "brus_2d_n": (lambda: nn.Brusselator(normalization='-11'), {}, 24),
        "lorenz_n": (lambda: nn.Lorenz(normalization='-11'), {}, 17)}  # early_stop as in published_K_study.py


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


# the driver's own refusals of a run (PararealEnsemble and PararealDevice raise these alike); anything else is a failure
REFUSALS = ("NaN values in initial coarse solve", "RK paging")


def ks(outs, N):
    return [o['k'] if o['converged'] else N for o in outs]


def ode_study(name, runs, log):
    mk, ckw, e_stop = ODES[name]
    ode = mk()
    cfg = nn.Config(ode, **ckw).get()
    solver = nn.CudaSolverRK(ode.get_vector_field(), **cfg)
    R, tol = runs[0][4], runs[0][5]
    assert all(r[4] == R and r[5] == tol for r in runs)
    ens = nn.PararealEnsemble(ode, solver, tspan=cfg["tspan"], N=cfg["N"], verbose='')
    common = dict(model='nngp', n_restarts=R, fatol=10 ** tol, xatol=10 ** tol)
    nnv = [r[3] if r[3] == 'adaptive' else int(r[3]) for r in runs]

    def per_nn():
        out = [None] * len(runs)
        for v in dict.fromkeys(nnv):
            sel = [i for i, x in enumerate(nnv) if x == v]
            o = ens.run(seeds=[runs[i][6] for i in sel], nn=v, epsilons=[runs[i][2] for i in sel],
                        early_stops=[e_stop] * len(sel), **common)
            for i, oi in zip(sel, o):
                out[i] = oi
        return out

    def mixed():
        return ens.run(seeds=[r[6] for r in runs], nn=nnv, epsilons=[r[2] for r in runs],
                       early_stops=[e_stop] * len(runs), **common)

    try:
        ens.run(seeds=runs[0][6:7], nn=nnv[0], epsilons=[runs[0][2]], early_stops=[e_stop], **common)  # warm-up
        a, ta = timed(per_nn)
        b, tb = timed(mixed)
        a2, ta2 = timed(per_nn)
        b2, tb2 = timed(mixed)
    except Exception as exc:
        if not any(r in str(exc) for r in REFUSALS):
            raise
        log(f"{name}: not measured, the driver refused a run ({exc})")
        return None
    same_k = ks(a, cfg["N"]) == ks(b, cfg["N"]) == ks(a2, cfg["N"]) == ks(b2, cfg["N"])
    kp = np.array(ks(b, cfg["N"])) - np.array([r[1] for r in runs])
    res = dict(system=name, runs=len(runs), n_ensembles_per_nn=len(set(map(str, nnv))),
               per_nn_s=[ta, ta2], mixed_s=[tb, tb2], per_nn_runs_per_s=len(runs) / min(ta, ta2),
               mixed_runs_per_s=len(runs) / min(tb, tb2), same_K_both_arms=same_k,
               K_minus_published=dict(collections.Counter(kp.tolist())))
    log(json.dumps(res))
    return res


def burgers_study(pub, n_seeds, log):
    runs = []
    for T in (5.0, 5.9):
        for nnb in range(11, 31):
            runs += [(T, nnb, s, K) for T_, n_, s, K in pub["Burgers_K_vs_m"] if (T_, n_) == (T, nnb)][:n_seeds]
    ode = nn.Burgers(d_x=128, normalization='-11')
    solver = nn.CudaSolverRK(ode.get_vector_field(), Ng=4, Nf=2000, G='RK1', F='RK8')
    ens = nn.PararealEnsemble(ode, solver, tspan=[0, 5.0], N=128, epsilon=5e-7, verbose='')

    def per_cell():
        out = {}
        for cell in dict.fromkeys((r[0], r[1]) for r in runs):
            sel = [i for i, r in enumerate(runs) if (r[0], r[1]) == cell]
            o = ens.run(model='nngp', seeds=[runs[i][2] for i in sel], nn=cell[1], tspans=[[0, cell[0]]] * len(sel))
            out.update(zip(sel, o))
        return [out[i] for i in range(len(runs))]

    def mixed():
        return ens.run(model='nngp', seeds=[r[2] for r in runs], nn=[r[1] for r in runs],
                       tspans=[[0, r[0]] for r in runs])

    ens.run(model='nngp', seeds=[runs[0][2], runs[-1][2]], nn=[runs[0][1], runs[-1][1]],
            tspans=[[0, runs[0][0]], [0, runs[-1][0]]])  # warm-up of both arms' kernels
    ens.run(model='nngp', seeds=[runs[0][2]], nn=runs[0][1])
    a, ta = timed(per_cell)
    b, tb = timed(mixed)
    a2, ta2 = timed(per_cell)
    b2, tb2 = timed(mixed)
    v = np.array(ks(b, 128)) - np.array([r[3] for r in runs])
    res = dict(system="Burgers_K_vs_m sample", runs=len(runs), n_ensembles_per_cell=40, per_cell_s=[ta, ta2],
               mixed_s=[tb, tb2], per_cell_runs_per_s=len(runs) / min(ta, ta2), mixed_runs_per_s=len(runs) / min(tb, tb2),
               same_K_both_arms=ks(a, 128) == ks(b, 128) == ks(a2, 128) == ks(b2, 128),
               K_minus_published=dict(sorted(collections.Counter(v.tolist()).items())),
               K_minus_published_mean=float(v.mean()), within_1=float(np.mean(np.abs(v) <= 1)))
    log(json.dumps(res))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--burgers-seeds", type=int, default=8)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07"))
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    gpu = card()
    log(f"card (name, power limit): {gpu}")
    pub = json.load(open(os.path.join(ROOT, "tests", "golden", "published.json")))
    by_sys = collections.defaultdict(list)
    for r in pub["NNGP_all_but_pend"]:
        by_sys[r[0]].append(r)
    out = dict(card=gpu, all_but_pend=[], burgers=None)
    for name in ODES:
        r = ode_study(name, by_sys[name], log)
        if r:
            out["all_but_pend"].append(r)
    out["burgers"] = burgers_study(pub, args.burgers_seeds, log)
    with open(os.path.join(args.out, "ensemble_study.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(args.out, "ensemble_study.log"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
