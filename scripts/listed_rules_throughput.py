"""GPU: runs/s of the six neighbour rules of the time-aware study (models_alt.py) in the three forms a user has.

For FHN-ODE and Lorenz in the published setting (normalization '-11', Config, nn = 16, epsilon = 5e-7), the runs
rules x seeds are made
  host      by the host driver Parareal (one fit_predict launch and one read back per predict),
  device    by PararealDevice, one run after the other (the listed sweep: no host round trip inside a sweep),
  ensemble  by one PararealEnsemble of all of them.
Each arm is warmed up once (one run per rule), then the arms run in alternating order per system.  Every run's K must
be identical in the three arms.  Prints the kernel-class times of the device and ensemble arms (CUDA events) and the
card name and power limit read in the same process; writes <out>/listed_rules_throughput.json and .log.
usage: listed_rules_throughput.py [--seeds 5] [--out profiles/r08]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib
from nearest_neighbors_gparareal_b200.models_alt import NNTYPES

SYSTEMS = {"fhn": lambda: nn.FHN_ODE(normalization='-11'), "lorenz": lambda: nn.Lorenz(normalization='-11')}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def setting(system):
    ode = SYSTEMS[system]()
    cfg = nn.Config(ode).get()
    return ode, cfg, nn.CudaSolverRK(ode.get_vector_field(), **cfg)


def arm_host(system, runs):
    ks = []
    for rule, seed in runs:
        ode, cfg, solver = setting(system)
        out = nn.Parareal(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='').run(
            model='nngp', pool=nn.CudaPool(), parall='mpi', nn=16, nntype=rule, seed=seed)
        ks.append(out['k'])
    return ks


def arm_device(system, runs):
    ks = []
    for rule, seed in runs:
        ode, cfg, solver = setting(system)
        out = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='').run(
            model='nngp', nn=16, nntype=rule, seed=seed)
        ks.append(out['k'])
    return ks


def arm_ensemble(system, runs, ens_box):
    ode, cfg, solver = setting(system)
    e = nn.PararealEnsemble(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='')
    h = e.handle()
    h.profile_enable(True)
    outs = e.run(seeds=[s for _, s in runs], nn=16, nntype=[r for r, _ in runs])
    ens_box.append(h.profile_read(reset=True))
    return [o['k'] for o in outs]


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08"))
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    gpu = card()
    lines = [f"card, power limit: {gpu}"]
    res = {"card": gpu, "systems": {}}
    dh = _lib.default_handle()
    for si, system in enumerate(SYSTEMS):
        runs = [(rule, 45 + s) for rule in NNTYPES for s in range(a.seeds)]
        warm = [(rule, 45) for rule in NNTYPES]
        arms = {"host": lambda r: arm_host(system, r), "device": lambda r: arm_device(system, r),
                "ensemble": lambda r: arm_ensemble(system, r, [])}
        for name, fn in arms.items():
            fn(warm)
        order = list(arms) if si % 2 == 0 else list(arms)[::-1]
        ks, secs, classes = {}, {}, {}
        for name in order:
            box = []
            if name == "device":
                dh.profile_read(reset=True)
                dh.profile_enable(True)
            fn = (lambda r: arm_ensemble(system, r, box)) if name == "ensemble" else arms[name]
            ks[name], secs[name] = timed(lambda: fn(runs))
            if name == "device":
                classes[name] = dh.profile_read(reset=True)
                dh.profile_enable(False)
            if box:
                classes[name] = box[0]
        same = ks["host"] == ks["device"] == ks["ensemble"]
        entry = {"runs": len(runs), "order": order, "seconds": secs, "runs_per_s": {k: len(runs) / v for k, v in secs.items()},
                 "K": {f"{r}/{s}": k for (r, s), k in zip(runs, ks["host"])}, "K_identical": same,
                 "kernel_classes_ms_launches": classes}
        res["systems"][system] = entry
        lines.append(f"{system}: {len(runs)} runs ({len(NNTYPES)} rules x {a.seeds} seeds), arms in order {order}")
        for k in order:
            lines.append(f"  {k:9s} {secs[k]:8.2f} s  {len(runs) / secs[k]:7.2f} runs/s")
        lines.append(f"  K per run identical in the three arms: {same}")
        for k, c in classes.items():
            lines.append(f"  {k} kernel classes (ms, launches): " + ", ".join(f"{n} {v[0]:.1f}/{v[1]}" for n, v in c.items()))
        if not same:
            lines.append(f"  K host {ks['host']}\n  K device {ks['device']}\n  K ensemble {ks['ensemble']}")
    text = "\n".join(lines)
    print(text)
    with open(os.path.join(a.out, "listed_rules_throughput.log"), "w") as f:
        f.write(text + "\n")
    with open(os.path.join(a.out, "listed_rules_throughput.json"), "w") as f:
        json.dump(res, f, indent=1)
    sys.exit(0 if all(e["K_identical"] for e in res["systems"].values()) else 3)


if __name__ == "__main__":
    main()
