"""Time of one device GP fit (nngp_fit_predict) per neighbour count m and search kernel, for one build of the package.

For every m and mode (warp: one warp per search, gp_fit_predict_kernel; quad: four warps per search,
gp_fit_spec_kernel) the script loads a fixed seeded dataset, finds the neighbours of nq queries once, and times
--reps fit_predict calls after --warmup untimed ones: CUDA events around each call on the caller's stream, and the
library's own per-kernel-class events for the fit launch (gp_fit class).  Rows 5-8 of the dataset copy row 4 and one
query sits on them, so the fits include searches that see +inf at every vertex and run to 400 evaluations.  Prints one
JSON line per (m, mode) with the median and minimum milliseconds and a hash of pred / nfev / thetas, so two builds can
be compared for speed and for identical bits.

usage: python scripts/gpu_fit_timing.py --root <package root> --label <name> [--ms 8 14 20] [--reps 30]
Run it once per build and alternate the builds (two builds of one package cannot share a process).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", required=True)
    ap.add_argument("--label", required=True)
    ap.add_argument("--ms", type=int, nargs="*", default=[8, 14, 16, 20, 26, 30, 32])
    ap.add_argument("--modes", nargs="*", default=["warp", "quad"])
    ap.add_argument("--n", type=int, default=2000, help="dataset rows")
    ap.add_argument("--d", type=int, default=256, help="dimension (searches per query = 9 d)")
    ap.add_argument("--nq", type=int, default=2, help="queries per fit")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import numpy as np
    import torch
    from nearest_neighbors_gparareal_b200 import _lib
    assert os.path.abspath(_lib.__file__).startswith(os.path.abspath(args.root)), _lib.__file__
    if not torch.cuda.is_available():
        raise SystemExit("gpu_fit_timing.py measures on the GPU; no CUDA device found")

    gpu = gpu_info()
    h = _lib.Handle(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    n, d, nq = args.n, args.d, args.nq
    for m in args.ms:
        rng = np.random.default_rng(1000 + m)
        x = rng.uniform(-1, 1, (n, d))
        y = 1e-3 * np.sin(x @ (rng.standard_normal((d, d)) / np.sqrt(d)))
        x[5:9] = x[4]
        y[5:9] = y[4]
        h.dataset_reset()
        h.dataset_reserve(n, d)
        h.dataset_append_host(x, y)
        q = np.concatenate([x[4:5], x[rng.permutation(n)[:nq - 1]] + 1e-3 * rng.standard_normal((nq - 1, d))])
        d_q = torch.from_numpy(q).to(dev)
        d_idx = torch.empty((nq, m), dtype=torch.int64, device=dev)
        d_dist = torch.empty((nq, m), dtype=torch.float64, device=dev)
        h.knn(d_q, nq, m, 0, d_idx, d_dist, stream.cuda_stream)
        d_starts = torch.from_numpy(rng.integers(-8, 0, (nq, d, 9, 1, 2)).astype(np.int8)).to(dev)
        d_pred = torch.empty((nq, d), dtype=torch.float64, device=dev)
        d_nfev = torch.empty((nq, d, 9, 1), dtype=torch.int32, device=dev)
        d_thetas = torch.empty((nq, d, 9, 1, 2), dtype=torch.float64, device=dev)

        def call():
            h.fit_predict(d_q, d_idx, d_dist, nq, m, 1, d_starts, 0.1, 0.1, d_pred, d_nfev=d_nfev, d_thetas=d_thetas,
                          stream=stream.cuda_stream)

        for mode in args.modes:
            h.set_fit_mode(mode)
            for _ in range(args.warmup):
                call()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
            h.profile_read(reset=True)
            h.profile_enable(True)
            for a, b in ev:
                a.record(stream)
                call()
                b.record(stream)
            torch.cuda.synchronize()
            h.profile_enable(False)
            prof = h.profile_read(reset=True)
            ms = sorted(a.elapsed_time(b) for a, b in ev)
            digest = hashlib.sha256()
            for t in (d_pred, d_nfev, d_thetas):
                digest.update(t.cpu().numpy().tobytes())
            print(json.dumps(dict(label=args.label, gpu=gpu, m=m, mode=mode, n=n, d=d, nq=nq, searches=nq * d * 9,
                                  reps=args.reps, call_ms_median=round(ms[len(ms) // 2], 4), call_ms_min=round(ms[0], 4),
                                  gp_fit_ms_per_call=round(prof["gp_fit"][0] / args.reps, 4),
                                  fit_launches_per_call=prof["gp_fit"][1] / args.reps,
                                  max_nfev=int(d_nfev.max()), hash=digest.hexdigest()[:16])), flush=True)
        h.set_fit_mode("auto")
    h.close()


if __name__ == "__main__":
    main()
