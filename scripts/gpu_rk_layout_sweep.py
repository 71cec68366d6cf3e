"""FHN fine step (d_x = 16, RK8) against the number of slices, for one build of the package, with the launch shapes the
environment variables of csrc/rk.cu force.  Prints one JSON line per (n, variant): milliseconds per fine step of
195 325 steps (scaled from --steps, median of --reps timed calls after one warm-up call with the same route), the
launches per call, and a hash of the result, so two builds can be compared for speed and for identical bits.

usage: python scripts/gpu_rk_layout_sweep.py --root <package root> --label <name> [--steps 20000] [--reps 5]
Run it once per build and alternate the builds (two builds of one package cannot share a process).
"""
import argparse
import hashlib
import json
import os
import sys

VARIANTS = {
    # name: (environment, slice counts)
    "default": ({}, (64, 148, 256, 296, 444, 512, 592)),
    "single_launch": ({"NNGP_RK_CHUNKS": "0"}, (296, 444, 512, 592)),
    "1x2_shuffle": ({"NNGP_RK_TILE": "2"}, (64, 148)),
    "1x2_shared": ({"NNGP_RK_TILE": "2", "NNGP_RK_NO_SHFL": "1"}, (64, 148)),
    "2x2_shuffle": ({"NNGP_RK_TILE": "1"}, (64, 148)),
    "2x2_shared": ({"NNGP_RK_TILE": "1", "NNGP_RK_NO_SHFL": "1"}, (64, 148)),
}
KNOBS = ("NNGP_RK_TILE", "NNGP_RK_NO_SHFL", "NNGP_RK_CHUNKS")
FINE_STEPS = 195325


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", required=True)
    ap.add_argument("--label", required=True)
    ap.add_argument("--steps", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--variants", nargs="*", default=list(VARIANTS))
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import numpy as np
    import torch
    import nearest_neighbors_gparareal_b200 as nn
    assert os.path.abspath(nn.__file__).startswith(os.path.abspath(args.root)), nn.__file__

    ode = nn.FHN_PDE(d_x=16)
    cfg = nn.Config(ode, d_x=16).get()
    solver = nn.CudaSolverRK(ode.get_vector_field(), **cfg)
    hh, sysid = solver.device()
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(0)
    st = torch.cuda.current_stream().cuda_stream
    for name in args.variants:
        env, ns = VARIANTS[name]
        for n in ns:
            rng = np.random.default_rng(n)
            u0 = torch.from_numpy(ode.get_init_cond()[None, :] + 0.01 * rng.standard_normal((n, 512))).to(dev)
            u1 = torch.empty_like(u0)
            t0 = torch.zeros(n, dtype=torch.float64, device=dev)
            t1 = t0 + 2.0
            for k in KNOBS:
                os.environ.pop(k, None)
            os.environ.update(env)
            try:
                hh.rk_batch(sysid, 8, solver.h_mode, args.steps, n, t0, t1, u0, 512, u1, 512, st)
                times = []
                for _ in range(args.reps):
                    c0 = hh.launch_count()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    hh.rk_batch(sysid, 8, solver.h_mode, args.steps, n, t0, t1, u0, 512, u1, 512, st)
                    e1.record()
                    torch.cuda.synchronize()
                    times.append(e0.elapsed_time(e1) * FINE_STEPS / args.steps)
                    launches = hh.launch_count() - c0
            finally:
                for k in KNOBS:
                    os.environ.pop(k, None)
            times.sort()
            out = u1.cpu().numpy()
            print(json.dumps({"label": args.label, "variant": name, "n": n, "ms_per_fine_step": round(times[len(times) // 2], 2),
                              "min": round(times[0], 2), "max": round(times[-1], 2), "launches": launches,
                              "steps": args.steps, "sha1": hashlib.sha1(out.tobytes()).hexdigest()[:16],
                              "finite": bool(np.isfinite(out).all()), "gpu": props.name}), flush=True)


if __name__ == "__main__":
    main()
