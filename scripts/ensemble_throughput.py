"""Runs/s of many independent nnGParareal runs: sequential solo PararealDevice runs against PararealEnsemble.

For every shape the same seeds run both ways, alternated (solo set, ensemble, solo set, ensemble ...: `--reps` pairs),
and every member is checked against its solo run (K, conv_int, u bit for bit).  Then one ensemble per shape runs with the
per-kernel-class CUDA-event timing on (nngp_profile_*), so the fit / kNN / RK split is visible.  The GPU name and power
limit are printed beside the numbers.

    python scripts/ensemble_throughput.py [--quick] [--reps 1] [--out DIR]   # DIR: where the JSON result goes
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nearest_neighbors_gparareal_b200 as nn  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as exc:
        return f"unknown ({exc})"


def shapes(quick):
    burgers = dict(name="burgers_d128_N128_nn18", mk=lambda: nn.Burgers(d_x=128, normalization='-11'),
                   solver=dict(Ng=4, Nf=2000, G='RK1', F='RK8'), tspan=[0, 5.0], N=128, run=dict(nn=18))
    lorenz = dict(name="lorenz_N50_nn11", mk=lambda: nn.Lorenz(normalization='-11'),
                  solver=dict(Ng=6, Nf=450, G='RK4', F='RK4'), tspan=[0, 18], N=50, run=dict(nn=11))
    hopf = dict(name="hopf_N32_nn15_R2", mk=lambda: nn.Hopf(normalization='-11'),
                solver=dict(Ng=64, Nf=5440, G='RK1', F='RK8'), tspan=[-20, 500], N=32, run=dict(nn=15, n_restarts=2))
    if quick:
        return [(lorenz, 5), (hopf, 5), (burgers, 8)]
    return [(burgers, 1), (burgers, 8), (burgers, 32), (burgers, 96), (lorenz, 5), (lorenz, 64), (hopf, 5), (hopf, 64)]


def solver_of(ode, kw):
    return nn.CudaSolverRK(ode.get_vector_field(), **kw)


def run_solo(sh, seeds):
    import torch
    outs = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in seeds:
        ode = sh["mk"]()
        p = nn.PararealDevice(ode, solver_of(ode, sh["solver"]), tspan=sh["tspan"], N=sh["N"], epsilon=5e-7,
                              verbose='')
        outs.append(p.run(model='nngp', seed=s, **sh["run"]))
    torch.cuda.synchronize()
    return outs, time.perf_counter() - t0


def make_ensemble(sh):
    ode = sh["mk"]()
    return nn.PararealEnsemble(ode, solver_of(ode, sh["solver"]), tspan=sh["tspan"], N=sh["N"], epsilon=5e-7,
                               verbose='')


def run_ens(ens, sh, seeds):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = ens.run(model='nngp', seeds=seeds, **sh["run"])
    torch.cuda.synchronize()
    return outs, time.perf_counter() - t0


def same(a, b):
    return (a['k'] == b['k'] and a['conv_int'] == b['conv_int'] and np.array_equal(a['u'], b['u'])
            and np.array_equal(a['err'], b['err'], equal_nan=True) and a['n_rows'] == b['n_rows'])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="small shapes only (a smoke test of the script)")
    ap.add_argument("--reps", type=int, default=1, help="alternated (solo, ensemble) pairs per shape")
    ap.add_argument("--out", default=None, help="also write the results as DIR/ensemble_throughput.json")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_throughput.py measures on the GPU; no CUDA device found")
    gpu = gpu_info()
    print(f"GPU (name, power limit, max SM clock): {gpu}", flush=True)
    rows = []
    for sh, E in shapes(a.quick):
        seeds = list(range(45, 45 + E))
        ens = make_ensemble(sh)
        run_ens(ens, sh, seeds[:1])  # warm-up of both arms: module loads, workspaces, handles
        run_solo(sh, seeds[:1])
        t_solo, t_ens, ok = [], [], True
        for _ in range(a.reps):
            so, ts = run_solo(sh, seeds)
            eo, te = run_ens(ens, sh, seeds)
            t_solo.append(ts)
            t_ens.append(te)
            ok &= all(same(x, y) for x, y in zip(eo, so))
        ks = [o['k'] for o in eo]
        h = ens.handle()
        h.profile_read(reset=True)
        h.profile_enable(True)
        run_ens(ens, sh, seeds)
        prof = h.profile_read(reset=True)
        h.profile_enable(False)
        r = dict(shape=sh["name"], E=E, solo_s=min(t_solo), ensemble_s=min(t_ens),
                 solo_runs_per_s=E / min(t_solo), ensemble_runs_per_s=E / min(t_ens),
                 speedup=min(t_solo) / min(t_ens), members_equal_solo=bool(ok), K=ks,
                 profile_ms={k: round(v[0], 3) for k, v in prof.items()},
                 profile_launches={k: v[1] for k, v in prof.items()})
        rows.append(r)
        print(f"{sh['name']:24s} E={E:3d}  solo {r['solo_runs_per_s']:7.2f} runs/s  ensemble {r['ensemble_runs_per_s']:7.2f}"
              f" runs/s  x{r['speedup']:5.2f}  members==solo: {ok}  K {min(ks)}..{max(ks)}  "
              f"event ms {r['profile_ms']}", flush=True)
        if not ok:
            print("MISMATCH: a member differs from its solo run", flush=True)
    if a.out is not None:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "ensemble_throughput.json"), "w") as fh:
            json.dump(dict(gpu=gpu, reps=a.reps, results=rows), fh, indent=1)
    if not all(r["members_equal_solo"] for r in rows):
        raise SystemExit(1)


if __name__ == "__main__":
    main()
