"""Where the one-warp search kernel's time goes on the benchmark's workload (FHN-PDE d = 512, N = 512, m = 20, R = 1,
RK8 x 195 325 fine steps per slice): objective evaluations by where they were decided (not evaluated thanks to the
look-ahead of all-inf iterations, failed at pivots 0 / 1, at pivots 2..4, or factorised further), split between
iterations that start with every vertex +inf and the others, and the warp cycles spent in each kind of iteration.

Needs a statistics build of gpfit.cu (-DNNGP_FIT_STATS: clock64 and counters inside nelder_mead), loaded through
NNGPARA_LIB.  `--build DIR` makes one from the tree's objects: gpfit.cu recompiled with the flag, the other units
taken from nearest_neighbors_gparareal_b200/build/ (run build() first).  The statistics build is slower; its cycle
shares, not its times, are the result.

usage: python scripts/fit_inf_share_probe.py --build DIR            (no GPU needed)
       NNGPARA_LIB=DIR/libnngpara.so python scripts/fit_inf_share_probe.py [--iterations 0 3]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def build_stats_lib(out_dir):
    from nearest_neighbors_gparareal_b200 import build as b
    b.build()
    os.makedirs(out_dir, exist_ok=True)
    obj = os.path.join(out_dir, "gpfit_stats.o")
    subprocess.run([b._nvcc()] + b.ARCH + b.COMMON + ["-DNNGP_FIT_STATS", "-c", os.path.join(b.CSRC, "gpfit.cu"),
                                                       "-o", obj], check=True)
    objs = [obj if src == "gpfit.cu" else os.path.join(b.OBJ_DIR, src.replace(".cu", ".o")) for src, _ in b.UNITS]
    lib = os.path.join(out_dir, "libnngpara.so")
    subprocess.run([b._nvcc()] + b.ARCH + ["-shared", "-o", lib] + objs, check=True)
    print(lib)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--build", metavar="DIR", default=None)
    ap.add_argument("--iterations", type=int, nargs="*", default=[0, 3])
    ap.add_argument("--fine-steps", type=int, default=195325)
    args = ap.parse_args()
    if args.build:
        build_stats_lib(args.build)
        return
    if "NNGPARA_LIB" not in os.environ:
        raise SystemExit("set NNGPARA_LIB to a statistics build (--build DIR)")
    import torch
    import nearest_neighbors_gparareal_b200 as nn
    from nearest_neighbors_gparareal_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("fit_inf_share_probe.py measures on the GPU; no CUDA device found")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print("gpu:", gpu[0] if gpu else "unknown", flush=True)
    N, m, dx = 512, 20, 16
    h = _lib.default_handle(0)
    ode = nn.FHN_PDE(d_x=dx)
    d = ode.get_dim()
    cfg = nn.Config(ode, d_x=dx).get()
    cfg["N"] = N
    cfg["Nf"] = args.fine_steps
    solver = nn.CudaSolverRK(ode.get_vector_field(), **cfg)
    par = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=N, epsilon=5e-7, verbose="")
    model = nn.CudaNNGP(n=d, N=N, nn=m, seed=45, handle=h)
    st = par.device_setup(model)
    for k in range(max(args.iterations) + 1):
        par.device_fine_step(st)
        if k in args.iterations:
            torch.cuda.synchronize()
            h.lib.nngp_fit_stats_dump()  # clear
            h.counters(reset=True)
            h.profile_read(reset=True)
            h.profile_enable(True)
        par.device_sweep(st, k)
        err = par.device_errors(st)
        if k in args.iterations:
            torch.cuda.synchronize()
            h.profile_enable(False)
            prof = h.profile_read(reset=True)
            runs, evals = h.counters(reset=True)
            print(f"iteration {k}: rows {h.dataset_rows()} searches {runs} evaluations {evals} "
                  f"gp_fit {prof['gp_fit'][0]:.1f} ms ({prof['gp_fit'][1]} launches, statistics build)", flush=True)
            sys.stderr.flush()
            h.lib.nngp_fit_stats_dump()
            sys.stderr.flush()
        par.device_advance(st, err)


if __name__ == "__main__":
    main()
