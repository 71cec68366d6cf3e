#!/usr/bin/env python
"""bench.py -- one nnGParareal iteration of the FHN-PDE target (BASELINE.json configs[3]) on B200.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR   # also writes what the last timed step computed, as DIR/<name>.npy

A "step" is ONE nnGParareal iteration (parareal.py:301-439) from the state after the coarse
initialisation: fine solves of all N slices (batched RK8, sharded by slice over the ranks + one
all-gather), dataset append, the serial sweep (G + kNN + d*9 Nelder-Mead GP fits + prediction per
slice) and the per-slice convergence norms.  `value` = iterations per second with every input
resident in HBM; `e2e` = the same iteration through the reference-facing Python protocols
(CudaPool.map(solver.run_F_timed) / model.fit / solver.run_G_timed / model.predict_timed) on HOST
buffers, host<->device copies inside the timed region.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Parareal iters/sec + nnGP fits/sec, FHN PDE N=512, 1-8 B200 vs CPU"
# BASELINE.md section 1: the reference's own run of this configuration (FHN-PDE d=512, N=512, m=20, published fine-step
# count) took 17 849 s for K=6 iterations on 517 CPU workers = 3.36e-4 iterations/s (derived from the result pickle
# FHN_scal_times_16_512_nngp; the reference publishes no other number for this metric)
PUBLISHED_ITERS_PER_S = 6.0 / 17849.0


def vs_baseline(args, value):
    """value / the BASELINE.md number -- only for the configuration that number was measured on"""
    same = args.dx == 16 and args.slices == 512 and args.m == 20 and args.fine_steps == 195325
    return value / PUBLISHED_ITERS_PER_S if same else None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dx", type=int, default=16, help="FHN grid side (d = 2*dx^2)")
    ap.add_argument("--slices", type=int, default=512)
    ap.add_argument("--m", type=int, default=20, help="nearest neighbours (nn)")
    ap.add_argument("--fine-steps", type=int, default=195325,
                    help="RK8 steps per slice; 195325 = the published run (FHN_PDE.py:53-54), 25 = configs.py preset")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--replicated-sweep", action="store_true",
                    help="N>1: every rank runs the whole sweep (north_star's layout) instead of sharding the fits by dimension")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="fhn", choices=["fhn", "synthetic"],
                    help="fhn: one nnGParareal iteration of BASELINE configs[3] (default, the headline); synthetic: BASELINE "
                         "configs[4], the batched nnGP kernel sweep (kNN + N x d fits), queries split over the ranks")
    ap.add_argument("--syn-n", type=int, default=16384, help="synthetic: dataset rows")
    ap.add_argument("--syn-d", type=int, default=128, help="synthetic: dimension")
    ap.add_argument("--syn-q", type=int, default=512, help="synthetic: queries (split over the ranks)")
    ap.add_argument("--iteration", type=int, default=0,
                    help="which nnGParareal iteration of the run a step is (0-based); the run is advanced there first")
    ap.add_argument("--no-full-run", action="store_true",
                    help="skip the complete solve (all K iterations through PararealDevice.run) that the default line also reports")
    ap.add_argument("--later-iteration", type=int, default=3,
                    help="with --iteration 0: also time this later iteration (2 500-row dataset, steady-state neighbours); 0 = off")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--profile-out", default=None, help="write the per-kernel-class event timings here (json)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step computed as DIR/<name>.npy (float64), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm samples timings, it does not compute the iteration")
    return args


DUMP_LIMIT = 64 * 10 ** 6  # bytes on disk, .npy headers included


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy in float64.  The arrays share their first axis; when they would take more
    than DUMP_LIMIT bytes, the same seeded sample of rows is taken from each and its row numbers go to sample_rows.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = {a.shape[0] for a in arrays.values()}
    assert len(n) == 1, "the dumped arrays must share their first axis"
    n = n.pop()
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_LIMIT - 1024 * (len(arrays) + 1)   # room for the headers
    if total > budget:
        keep = max(1, n * budget // (total + 8 * n))
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def nll_flops(m):
    """algorithmic FP64 operations of one objective evaluation (SURVEY.md section 8d):
    m^3/3 + 2 m^2 + 3 m(m+1)/2 + 4 m with exp / log / sqrt / div counted as one each"""
    return m ** 3 / 3 + 2 * m ** 2 + 3 * m * (m + 1) / 2 + 4 * m


def rk_flops(d, S, rhs_per_point=26):
    """algorithmic FP64 operations of one RK step of one slice (SURVEY.md section 8d): S stencil RHS
    (26 per grid point pair) + dense-tableau combinations as the reference evaluates them"""
    return S * rhs_per_point * (d / 2) + (S * (S - 1) / 2) * 2 * d + S * 2 * d + 2 * S * d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)"""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(args, n_dims_per_core, n_steps, warm, dims_frac=1.0):
    """oracle (NumPy/SciPy port of the reference) on all host cores; returns the list of samples"""
    import warnings
    from oracle.cpu_baseline import FhnCpuSampler
    warnings.filterwarnings("ignore")
    cores = os.cpu_count()
    T = 1100.0 * args.slices / 512 if args.dx == 16 else 1100.0
    s = FhnCpuSampler(d_x=args.dx, N=args.slices, m=args.m, T=T, cores=cores)
    d = 2 * args.dx * args.dx
    # 8 sampled predicts (SURVEY.md section 8d), each over min(d, n_dims_per_core * cores) output dimensions: at d = 512 on 16
    # cores that is 36 864 Nelder-Mead searches = ~2 minutes of CPU work, ~8 s of wall time
    n_dims = 8 * max(min(d, cores), int(dims_frac * min(d, max(cores, n_dims_per_core * cores))))
    out = []
    for it in range(warm + n_steps):
        t0 = time.perf_counter()
        r = s.sample(n_dims=n_dims, n_slices=max(8, min(args.slices, cores)), fine_steps=args.fine_steps, n_predicts=8)
        r["wall"] = time.perf_counter() - t0
        if it >= warm:
            out.append(r)
    s.close()
    return out, cores, n_dims


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port), rank 0 only"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # a quarter of the output dimensions per sampled predict: K steps of ~2 s each keep the whole run within minutes
    samples, cores, n_dims = cpu_sample(args, n_dims_per_core=1 << 20, n_steps=args.steps, warm=min(args.warmup, 1), dims_frac=0.25)
    t_iter = float(np.mean([r["t_iter"] for r in samples]))
    d = 2 * args.dx * args.dx
    sample = (f"per step: 8 predicts (queries spread over the slices) restricted to {max(1, n_dims // 8)} of {d} output dims each "
              f"({max(1, n_dims // 8) * 8 * 9} Nelder-Mead searches) "
              f"farmed over {cores} processes + {max(8, min(args.slices, cores))} fine slices of 25 RK8 steps scaled to "
              f"{args.fine_steps}; extrapolated with T_iter = ceil(N/C) t_F + (N-1)(t_G + t_predict)")
    line = {"impl": "reference", "metric": METRIC, "value": 1.0 / t_iter, "unit": "iters/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_iter, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": vs_baseline(args, 1.0 / t_iter), "dtype": "f64", "data": "synthetic",
            "config": workload_config(args), "gpu_launches": 0,
            "fits_per_s": float(np.mean([r["fits_per_s"] for r in samples])),
            "cpu_s_per_nm_run": float(np.mean([r["cpu_s_per_nm_run"] for r in samples])),
            "t_F_slice_s": float(np.mean([r["t_F_slice"] for r in samples])),
            "t_predict_s": float(np.mean([r["t_predict"] for r in samples])),
            "cpu_baseline": {"value": 1.0 / t_iter, "unit": "iters/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": 1.0 / t_iter, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args):
    d = 2 * args.dx * args.dx
    return {"workload": f"FHN-PDE {args.dx}x{args.dx} (d={d}) nnGParareal, one iteration (number --iteration of the run; "
                        f"0 = from the coarse initialisation)",
            "N_slices": args.slices, "d": d, "m": args.m, "n_restarts": 1, "jitters": 9, "G": "RK4 x25 steps/slice",
            "F": f"RK8 x{args.fine_steps} steps/slice", "seed": 45, "epsilon": 5e-7,
            "l2": "256 MiB write between timed steps (L2 flush)"}


def run_synthetic(args):
    """BASELINE.json configs[4] / SURVEY.md section 8d config 5: X ~ U(-1,1)^{n x d}, Y = 1e-3 sin(X W), W ~ N(0,1)/sqrt(d),
    Q queries = rows + 1e-3 N(0,1) (default_rng(0)), Nelder-Mead starts from default_rng(45).  The dataset is replicated,
    the queries are split over the ranks (section 8e), the [Q, d] predictions are gathered at the end (one all-gather).
    A step = kNN + the Q/W x d fits (9 searches + selection + posterior mean each) + the gather."""
    import torch
    import torch.distributed as dist
    from nearest_neighbors_gparareal_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    h = _lib.default_handle(local)
    n, d, m, Q = args.syn_n, args.syn_d, args.m, args.syn_q
    rng = np.random.default_rng(0)
    x = rng.uniform(-1, 1, (n, d))
    y = 1e-3 * np.sin(x @ (rng.standard_normal((d, d)) / np.sqrt(d)))
    q_all = x[rng.permutation(n)[:Q]] + 1e-3 * rng.standard_normal((Q, d))
    starts_all = np.random.default_rng(45).integers(-8, 0, (Q, d, 9, 1, 2)).astype(np.int8)
    h.dataset_reset()
    h.dataset_reserve(n, d)
    h.dataset_append_host(x, y)
    per = (Q + world - 1) // world
    lo, hi = min(Q, rank * per), min(Q, (rank + 1) * per)
    nq = hi - lo
    q = torch.from_numpy(q_all[lo:hi].copy()).to(dev)
    starts = torch.from_numpy(starts_all[lo:hi].copy()).to(dev)
    idx = torch.empty((max(nq, 1), m), dtype=torch.int64, device=dev)
    dst = torch.empty((max(nq, 1), m), dtype=torch.float64, device=dev)
    pred_all = torch.zeros((world * per, d), dtype=torch.float64, device=dev)
    pred = pred_all[rank * per:rank * per + max(nq, 1)]
    stream = torch.cuda.current_stream(dev).cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        if nq > 0:
            h.knn(q, nq, m, 0, idx, dst, stream)
            h.fit_predict(q, idx, dst, nq, m, 1, starts, 0.1, 0.1, pred, stream=stream)
        if world > 1:
            dist.all_gather_into_tensor(pred_all, pred_all[rank * per:(rank + 1) * per])

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
        flush.fill_(1)
    h.counters(reset=True)
    h.profile_read(reset=True)
    h.profile_enable(True)
    l0 = h.launch_count()
    sync_all()
    clocks = ClockSampler(local)
    clocks.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(args.steps):
        step()
        flush.fill_(1)
    ev[1].record()
    sync_all()
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pred": pred_all[:Q].cpu().numpy()})
    t = torch.tensor([ev[0].elapsed_time(ev[1])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    h.profile_enable(False)
    prof = h.profile_read(reset=True)
    nm_runs, nll_evals = h.counters(reset=True)
    launches = (h.launch_count() - l0) // args.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    knn_ms = prof["knn"][0] / args.steps
    knn_bytes = 8.0 * n * d + 8.0 * nq * d + 16.0 * nq * m
    fit_ms = prof["gp_fit"][0] / args.steps
    fp64_peak = h.bench_fp64(20000)
    fit_tf = (nll_evals / args.steps) * nll_flops(m) / (fit_ms * 1e-3) / 1e12 if fit_ms > 0 else 0.0
    # e2e: host queries in, host predictions out (nngp_predict_host: H2D, kNN, fits, D2H), then the gather
    e2e = None
    if not args.no_e2e:
        qh, sh = q_all[lo:hi].copy(), starts_all[lo:hi].copy()

        def e2e_step():
            ph = h.predict_host(qh, m, sh, 1, 0.1, 0.1)["pred"] if nq > 0 else np.zeros((0, d))
            if world > 1:
                buf = torch.zeros((world * per, d), dtype=torch.float64, device=dev)
                buf[rank * per:rank * per + nq] = torch.from_numpy(ph).to(dev)
                dist.all_gather_into_tensor(buf, buf[rank * per:(rank + 1) * per])
                return buf[:Q].cpu().numpy()
            return ph
        e2e_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            out = e2e_step()
        sync_all()
        secs = (time.perf_counter() - t0) / args.e2e_steps
        tt = torch.tensor([secs], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        secs = float(tt.item())
        e2e = {"value": Q * d / secs, "unit": "fits/s", "ms_per_step": 1e3 * secs, "steps": args.e2e_steps,
               "h2d_bytes_per_step": int(nq * d * 8 + nq * d * 18), "d2h_bytes_per_step": int(nq * d * 8),
               "finite": bool(np.all(np.isfinite(out))),
               "api": "nngp_predict_host (NumPy queries + starts in, NumPy predictions out) + all-gather of [Q, d]"}
    line = {"metric": METRIC, "value": Q * d / (ms_step * 1e-3), "unit": "fits/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "synthetic nnGP kernel sweep (BASELINE configs[4]): kNN + batched N x d fits, queries split over ranks",
                       "n_rows": n, "d": d, "m": m, "Q": Q, "n_restarts": 1, "jitters": 9,
                       "l2": "256 MiB write between timed steps (L2 flush)"},
            "clocks": clk, "gpu_launches": int(launches),
            "roofline": {"kernel": "sqdist_kernel<8> + select_kernel (kNN of this rank's queries)", "bound": "hbm" if nq < 16 else "fp64",
                         "achieved": knn_bytes / (knn_ms * 1e-3) / 1e9 if knn_ms > 0 else 0.0, "peak": hbm, "unit": "GB/s",
                         "frac": (knn_bytes / (knn_ms * 1e-3) / 1e9 / hbm) if knn_ms > 0 else None,
                         "traffic": None, "knn_ms": knn_ms,
                         "fp64_tflops": 3.0 * nq * n * d / (knn_ms * 1e-3) / 1e12 if knn_ms > 0 else 0.0,
                         "note": "algorithmic bytes 8nd + 8Qd + 16Qm per call against MEASURED_PEAKS.json hbm_gbs; with Q >= 16 "
                                 "queries per rank the exact (non-fused, 3 flops per coordinate) distance arithmetic is FP64-bound"},
            "roofline_second_kernel": {"kernel": "gp_fit_grouped_kernel / gp_fit_predict_kernel", "bound": "fp64",
                                       "achieved": fit_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                                       "frac": fit_tf / fp64_peak if fp64_peak else None, "fit_ms": fit_ms},
            "kernels": {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] // args.steps} for k, v in prof.items()},
            "fits_per_s": Q * d / (ms_step * 1e-3), "nm_runs_per_s_rank0": nm_runs / args.steps / (ms_step * 1e-3),
            "nll_evals_per_s_rank0": nll_evals / args.steps / (ms_step * 1e-3),
            "knn_gbs_rank0": knn_bytes / (knn_ms * 1e-3) / 1e9 if knn_ms > 0 else None}
    if e2e:
        line["e2e"] = e2e
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "synthetic":
        run_synthetic(args)
        return
    import torch
    import torch.distributed as dist
    import nearest_neighbors_gparareal_b200 as nn
    from nearest_neighbors_gparareal_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    h = _lib.default_handle(local)

    # ---- the workload: configs.py fhn_pde preset with the requested number of fine steps ----------
    N, m = args.slices, args.m
    ode = nn.FHN_PDE(d_x=args.dx)
    d = ode.get_dim()
    cfg = nn.Config(ode, d_x=args.dx).get()
    cfg["N"] = N
    cfg["tspan"] = [0, cfg["tspan"][1] * N / 512]
    cfg["Nf"] = args.fine_steps
    solver = nn.CudaSolverRK(ode.get_vector_field(), **cfg)
    par = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=N, epsilon=5e-7, verbose="",
                            shard_sweep=not args.replicated_sweep)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    fp64_peak = None

    def measure(iteration, steps, warmup, with_clocks, keep_outputs=False):
        """times `steps` repetitions of nnGParareal iteration number `iteration` (0-based) of the run: the run is
        advanced to the start of that iteration once (real iterations 0 .. iteration-1), its state is saved, and every
        timed step restores it (device copies + dataset truncation, outside the kernels but inside the timed region).
        keep_outputs: also return, on the host, the state the last timed step left (new iterate, coarse and fine
        values, per-slice errors)"""
        nonlocal fp64_peak
        model = nn.CudaNNGP(n=d, N=N, nn=m, seed=45, handle=h)
        st = par.device_setup(model)
        for k in range(iteration):
            par.device_fine_step(st)
            par.device_sweep(st, k)
            err_k = par.device_errors(st)
            par.device_advance(st, err_k)
            if st["I"] >= N:
                raise SystemExit(f"the run converged before iteration {iteration}")
        torch.cuda.synchronize(dev)
        I0, rows0 = st["I"], h.dataset_rows()
        u0_cur, uG0_cur = st["u_cur"].clone(), st["uG_cur"].clone()
        starts = torch.from_numpy(model.draw_starts(N - I0 - 1)).to(dev)
        fine_events = []

        def step():
            st["I"] = I0
            st["u_cur"].copy_(u0_cur)
            st["uG_cur"].copy_(uG0_cur)
            st["u_next"].copy_(u0_cur)
            st["uG_next"].copy_(uG0_cur)
            h.dataset_truncate(rows0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            l0 = h.launch_count()
            par.device_fine_step(st)  # the batched RK8 launches on torch's current stream (+ the all-gather for N>1)
            e1.record()
            fine_events.append((e0, e1, h.launch_count() - l0))
            par.device_sweep(st, iteration, starts=starts)
            return par.device_errors(st)  # the one device->host read of an iteration (N+1 doubles)

        for _ in range(warmup):
            err = step()
            flush.fill_(1)
        h.counters(reset=True)
        h.profile_read(reset=True)
        h.profile_enable(True)
        launches0 = h.launch_count()
        fine_events.clear()
        sync_all()
        clocks = ClockSampler(local) if with_clocks else None
        if clocks:
            clocks.start()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(steps):
            err = step()
            flush.fill_(1)
        ev[1].record()
        sync_all()
        clk = clocks.stop() if clocks else None
        outputs = None
        if keep_outputs:
            outputs = {"u_next": st["u_next"].cpu().numpy(), "uG_next": st["uG_next"].cpu().numpy(),
                       "uF": st["uF"][:N + 1].cpu().numpy(), "err": err}
        ms_total = ev[0].elapsed_time(ev[1])
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / steps
        h.profile_enable(False)
        prof = h.profile_read(reset=True)
        nm_runs, nll_evals = h.counters(reset=True)
        launches = (h.launch_count() - launches0) // steps
        if fp64_peak is None:
            fp64_peak = h.bench_fp64(20000)
        n_sweep = N - I0 - 1           # predicts of this iteration
        n_fine = N - I0                # fine solves of this iteration
        fit_ms, fit_n = prof["gp_fit"]
        fit_tf = nll_evals * nll_flops(m) / (fit_ms * 1e-3) / 1e12 if fit_ms > 0 else 0.0
        fine_ms = sum(a.elapsed_time(b) for a, b, _ in fine_events) / max(len(fine_events), 1)
        fine_launches = max(1, fine_events[-1][2]) if fine_events else 1
        f_flops = rk_flops(d, 11) * args.fine_steps * math.ceil(n_fine / world)
        rk_tf = f_flops / (fine_ms * 1e-3) / 1e12 if fine_ms > 0 else 0.0
        kernels = {k: {"ms_per_step": v[0] / steps, "launches_per_step": v[1] // steps} for k, v in prof.items()}
        return dict(ms_step=ms_step, clk=clk, launches=int(launches), kernels=kernels, err=err, fit_ms=fit_ms, fit_n=fit_n,
                    fit_tf=fit_tf, fine_ms=fine_ms, fine_launches=fine_launches, f_flops=f_flops, rk_tf=rk_tf,
                    nm_runs=nm_runs / steps, nll_evals=nll_evals / steps, n_sweep=n_sweep, n_fine=n_fine,
                    rows=int(h.dataset_rows()), I0=I0, steps=steps, outputs=outputs)

    R = measure(args.iteration, args.steps, args.warmup, with_clocks=True, keep_outputs=bool(args.dump_outputs))
    ms_step, clk, steps = R["ms_step"], R["clk"], R["steps"]
    # ---- rooflines of the two kernels that share the step (fine propagator, GP fit): FP64 pipe ------
    peak_src = ("FP64 FMA micro-benchmark run in this process (nngp_bench_fp64: 8 independent DFMA chains per thread, "
                "148 x 8 CTAs x 256 threads; profiles/r02/fp64_peak.log); MEASURED_PEAKS.json has no FP64 entry; nominal "
                "B200 FP64 is 37 TFLOP/s (the measured figure is 0.914 of it); the bound is FP64, neither HBM nor tensor "
                "cores: all state is register / shared-memory resident")
    roof_fit = {"kernel": "gp_fit_predict_kernel<20>", "bound": "fp64", "achieved": R["fit_tf"], "peak": fp64_peak,
                "unit": "TFLOP/s", "frac": R["fit_tf"] / fp64_peak if fp64_peak else None, "frac_of_nominal_37": R["fit_tf"] / 37.0,
                "traffic": 282368, "traffic_source": "profiles/r02/sweep_r2.summary.csv (dram read+write bytes per launch)",
                "peak_source": peak_src,
                "per_launch": {"launches": R["fit_n"] // steps, "avg_ms": R["fit_ms"] / max(R["fit_n"], 1),
                               "nll_evals": R["nll_evals"] * steps / max(R["fit_n"], 1), "flops_per_eval": nll_flops(m)},
                "share_of_step": R["fit_ms"] / (ms_step * steps),
                "executed_fp64_pipe_frac": 0.497, "executed_source": "profiles/r02/sweep_r2.summary.csv (sm__pipe_fp64_cycles_active, steady-state slice)",
                "note": "algorithmic flops E(m) per objective evaluation; the kernel executes ~8x that in FP64 lane-operations "
                        "(20 of 32 lanes hold rows, full-row updates, 17-FMA exponentials): FP64 pipe 50 % busy in "
                        "profiles/r02/sweep_r2.summary.csv; 45 % of the evaluations are failing factorisations that "
                        "leave early (profiles/r02/fit_failing_pivots.log)"}
    slices_rank = math.ceil(R["n_fine"] / world)
    lone = slices_rank <= 148   # at most one slice per SM: the latency shape with shuffled halo columns (csrc/rk.cu)
    quad_fit = world > 1 and (d // world) * 9 <= 3 * 148 * 3   # a rank's searches per predict <= the four-warp limit (csrc/gpfit.cu)
    if quad_fit:
        roof_fit["kernel"] = "gp_fit_spec_kernel<20> (four warps per search)"
        roof_fit["executed_fp64_pipe_frac"] = 0.37
        roof_fit["executed_source"] = ("profiles/r02/fit_quad8_r2.summary.csv (one rank's share of the 8-rank sweep: SM "
                                       "sub-partitions active 55 % of the launch, 2.0x the instructions of the one-warp "
                                       "kernel, which on the same share is active 25 % and at 20 %: fit_shard8_r2.summary.csv)")
    roof_rk = {"kernel": "rk_fhn_tile_kernel<11,1,128,SHX>" if lone else "rk_fhn_tile_kernel<11,2,64>", "bound": "fp64", "achieved": R["rk_tf"], "peak": fp64_peak,
               "unit": "TFLOP/s", "frac": R["rk_tf"] / fp64_peak if fp64_peak else None, "frac_of_nominal_37": R["rk_tf"] / 37.0,
               "traffic": 2158336, "traffic_source": "profiles/r01/rk_tile_r1.summary.csv (dram read+write bytes per launch)",
               "peak_source": peak_src,
               "per_launch": {"launches": R["fine_launches"], "avg_ms": R["fine_ms"] / R["fine_launches"],
                              "flops": R["f_flops"] / R["fine_launches"], "fine_step_ms": R["fine_ms"],
                              "slices": math.ceil(R["n_fine"] / world),
                              "steps_per_slice": args.fine_steps, "flops_per_slice_step": rk_flops(d, 11),
                              "note": "the fine step is a sequence of balanced launches over (chunk of steps, slice) "
                                      "tasks, 2 CTAs per SM (csrc/rk.cu launch_fhn_tile_s); algorithmic flops count the "
                                      "dense tableau as the reference evaluates it (SURVEY 8d), the kernel executes the 39+5 "
                                      "structural non-zeros: executed FP64 pipe utilisation 59 % (profiles/r01/rk_tile_r1.summary.csv)"},
               "executed_fp64_pipe_frac": 0.38 if lone else 0.59,
               "executed_source": "profiles/r02/rk_lone_shuffle_r2.summary.csv" if lone else "profiles/r01/rk_tile_r1.summary.csv",
               "share_of_step": R["fine_ms"] / ms_step}
    if lone:
        roof_rk["per_launch"]["note"] = ("one launch, one CTA of 128 threads per slice (at most one slice per SM): bound by "
                                         "the per-stage dependency chain, 235 cycles (DESIGN.md 4.1); algorithmic flops count "
                                         "the dense tableau as the reference evaluates it (SURVEY 8d)")
    roofline, other = (roof_rk, roof_fit) if roof_rk["share_of_step"] >= roof_fit["share_of_step"] else (roof_fit, roof_rk)
    wl = workload_config(args)
    wl["iteration"] = args.iteration
    wl["dataset_rows_after_append"] = R["rows"]
    wl["first_unconverged_slice"] = R["I0"]
    line = {"metric": METRIC, "value": 1e3 / ms_step, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": vs_baseline(args, 1e3 / ms_step), "dtype": "f64", "data": "synthetic",
            "config": wl,
            "clocks": clk, "gpu_launches": R["launches"], "roofline": roofline, "roofline_second_kernel": other,
            "kernels": R["kernels"],
            "fits_per_s": R["n_sweep"] * d / (ms_step * 1e-3), "nm_runs_per_s": R["nm_runs"] / (ms_step * 1e-3),
            "nll_evals_per_s": R["nll_evals"] / (ms_step * 1e-3),
            "nll_evals_per_nm_run": R["nll_evals"] / max(R["nm_runs"], 1),
            "fine_step_flops_per_rank": R["f_flops"], "err_max_iter": float(np.nanmax(R["err"])),
            "fp64_peak": {"measured_tflops": fp64_peak, "nominal_tflops": 37.0}}
    # ---- the same step later in the run (iteration 4 of the published K = 6: ~2 500 dataset rows, steady-state
    # neighbours, more searches that run to SciPy's evaluation limit) --------------------------------------------
    if args.iteration == 0 and args.later_iteration > 0:
        L = measure(args.later_iteration, max(1, min(2, args.steps)), 1, with_clocks=False)
        line["later_iteration"] = {"iteration": args.later_iteration, "ms_per_step": L["ms_step"], "value": 1e3 / L["ms_step"],
                                   "unit": "iters/s", "steps": L["steps"], "dataset_rows_after_append": L["rows"],
                                   "first_unconverged_slice": L["I0"], "kernels": L["kernels"],
                                   "nll_evals_per_nm_run": L["nll_evals"] / max(L["nm_runs"], 1),
                                   "fit_tflops": L["fit_tf"], "rk_tflops": L["rk_tf"], "gpu_launches": L["launches"]}

    # ---- the complete solve: every iteration until convergence through the public driver (device events around the run) --
    if args.iteration == 0 and not args.no_full_run:
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        full = par.run(model="nngp", nn=m, seed=45)
        e1.record()
        sync_all()
        secs = e0.elapsed_time(e1) * 1e-3
        tt = torch.tensor([secs], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        secs = float(tt.item())
        line["full_run"] = {"K": int(full["k"]), "converged": bool(full["converged"]), "conv_int": [int(v) for v in full["conv_int"]],
                            "seconds": secs, "iters_per_s": full["k"] / secs,
                            "seconds_without_coarse_init": secs - float(full["timings"]["G_time"]),
                            "err_max_per_iteration": [float(v) for v in np.nanmax(full["err"], axis=0)],
                            "note": "PararealDevice.run: coarse initialisation (N dependent one-slice launches) + K iterations; "
                                    "published run of the reference: K = 6 in 17 849 s on 517 CPU workers"}

    # ---- e2e: the same iteration through the reference-facing protocols on host buffers -----------
    if not args.no_e2e:
        line["e2e"] = run_e2e(args, nn, ode, solver, cfg, h, dev, world, rank, sync_all, dist)
    # ---- CPU baseline: the oracle port on this host's cores (rank 0, N=1 only) --------------------
    if world == 1 and not args.no_cpu_baseline:
        samples, cores, n_dims = cpu_sample(args, n_dims_per_core=1 << 20, n_steps=1, warm=0)
        r = samples[0]
        line["cpu_baseline"] = {
            "value": 1.0 / r["t_iter"], "unit": "iters/s", "cores": cores, "kind": "port",
            "sample": (f"8 predicts (queries spread over the slices) restricted to {max(1, n_dims // 8)} of {d} dims each "
                       f"({max(1, n_dims // 8) * 72} Nelder-Mead searches, "
                       f"{r['cpu_s_per_nm_run']*1e3:.1f} ms each) on {cores} processes + {r['n_slices']} fine slices of "
                       f"25 RK8 steps scaled to {args.fine_steps}; T_iter = ceil(N/C) t_F + (N-1)(t_G + t_predict); "
                       f"sample wall {r['wall']:.1f} s"),
            "fits_per_s": r["fits_per_s"], "t_F_slice_s": r["t_F_slice"], "t_predict_s": r["t_predict"]}
    if rank == 0:
        if args.profile_out:
            with open(args.profile_out, "w") as fh:
                json.dump(line, fh, indent=1)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, R["outputs"])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(args, nn, ode, solver, cfg, h, dev, world, rank, sync_all, dist):
    """One iteration through Parareal's protocols: pool.map(run_F_timed) -> fit -> (run_G_timed, predict_timed)*"""
    import torch
    N, d, m = args.slices, ode.get_dim(), args.m
    t = np.linspace(cfg["tspan"][0], cfg["tspan"][1], N + 1)
    pool = nn.CudaPool(sharded=(world > 1))
    # state after the coarse initialisation, on the host
    u_cur = np.empty((N + 1, d))
    u_cur[0] = ode.get_init_cond()
    for i in range(N):
        u_cur[i + 1] = solver.run_G(t[i], t[i + 1], u_cur[i])
    uG_cur = u_cur.copy()
    h2d = d2h = 0

    def iteration():
        nonlocal h2d, d2h
        model = nn.CudaNNGP(n=d, N=N, nn=m, seed=45, handle=h, shard_predict=(world > 1))
        res = list(pool.map(solver.run_F_timed, t[0:N], t[1:N + 1], [u_cur[i] for i in range(N)]))
        uF = np.empty((N + 1, d))
        uF[0] = u_cur[0]
        uF[1:] = np.array([r[0] for r in res])
        n_loc = math.ceil(N / world)
        h2d += (n_loc * d + 2 * n_loc) * 8
        d2h += n_loc * d * 8
        u_next, uG_next = u_cur.copy(), uG_cur.copy()
        u_next[1] = uF[1]
        x = u_cur[0:N]
        D = uF[1:N + 1] - uG_cur[1:N + 1]
        model.fit_timed(x, D, k=0)
        h2d += 2 * x.size * 8
        for i in range(1, N):
            uG_next[i + 1], _ = solver.run_G_timed(t[i], t[i + 1], u_next[i])
            preds = model.predict_timed(u_next[i].reshape(1, -1), uF[i + 1], uG_cur[i + 1], i=i)
            u_next[i + 1] = preds + uG_next[i + 1]
            h2d += (d + 2) * 8 + d * 8 + d * 9 * 2
            d2h += 2 * d * 8
        return np.linalg.norm(u_next - u_cur, np.inf, 1)

    iteration()  # warm-up
    h2d = d2h = 0
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        err = iteration()
    sync_all()
    secs = (time.perf_counter() - t0) / args.e2e_steps
    tt = torch.tensor([secs], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    secs = float(tt.item())
    return {"value": 1.0 / secs, "unit": "iters/s", "ms_per_step": 1e3 * secs, "steps": args.e2e_steps,
            "h2d_bytes_per_step": int(h2d // args.e2e_steps), "d2h_bytes_per_step": int(d2h // args.e2e_steps),
            "fits_per_s": (N - 1) * d / secs, "err_max_iter0": float(np.nanmax(err)),
            "api": "CudaPool.map(solver.run_F_timed) + CudaNNGP.fit_timed + per slice CudaSolverRK.run_G_timed / "
                   "CudaNNGP.predict_timed (NumPy in, NumPy out)"}


if __name__ == "__main__":
    main()
