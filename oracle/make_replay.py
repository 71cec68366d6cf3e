"""TEST INFRASTRUCTURE ONLY -- builds tests/golden/run_fhn_d512_replay_k{2,3}.npz in the build container.

Input: the state dump of a DEVICE run of the full-size FHN-PDE target (d=512, N=512, m=20, RK8 x 195 325 steps per
slice -- a size the CPU reference cannot run), written by `scripts/parity_matrix.py --full --dump DIR` on the GPU box:
iterates u^k, coarse values uG^k, fine values uF^k and the first unconverged slice per iteration.
For a handful of predicts of iterations 3 and 4 (steady-state neighbours from slice ~50 on) this script rebuilds the
dataset prefix exactly as parareal.py:336-339 does, positions the PCG64 stream of models.py:114,192 where the run
had it, and calls the UNMODIFIED reference `NNGP_p.predict` (models.py:171-226) under oracle/ref_shim.py.  Stored per
predict: query, the m neighbour rows in kNN order (x, F-G), the host-drawn starts, and the reference's prediction,
per-search optimum value (fval) and the theta of the search its rule selects (models.py:212-215).  One file per
iteration keeps each under 1 MB.

usage: python -m oracle.make_replay gpurun_out/replay/fhn_full_state_id.npz [workers]
"""
import os
import sys
import time

import numpy as np

from .ref_shim import load_reference
from . import nngp as onn

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
PICKS = [(2, 4), (2, 8), (2, 14), (2, 22), (2, 40), (2, 120), (2, 400), (3, 5), (3, 6), (3, 10), (3, 18), (3, 30), (3, 80), (3, 500)]


class RecordingPool:
    """executor protocol (parareal.py:16-24) that keeps what the searches returned"""

    def __init__(self, workers):
        import concurrent.futures
        self.ex = concurrent.futures.ProcessPoolExecutor(max_workers=workers) if workers > 1 else None
        self.last = None

    def map(self, fn, *its, **kw):
        self.last = list(self.ex.map(fn, *its, chunksize=16)) if self.ex else list(map(fn, *its))
        return self.last

    def shutdown(self):
        if self.ex:
            self.ex.shutdown()


def main():
    dump = np.load(sys.argv[1])
    workers = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    u, uG, uF, I_sweep = dump["u"], dump["uG"], dump["uF"], dump["I_sweep"]
    N, d = u.shape[1] - 1, u.shape[2]
    m, n_tasks = 20, d * 9
    ns = load_reference(fast_kernel=True)
    pool = RecordingPool(workers)
    # dataset after the append of iteration k (parareal.py:336-339): x <- u^k[I-1:N], D <- uF^k[I:N+1] - uG^k[I:N+1]
    xs, ys, rows_after = [], [], []
    for k in range(uF.shape[0]):
        I = int(I_sweep[k])
        xs.append(u[k][I - 1:N])
        ys.append(uF[k][I:N + 1] - uG[k][I:N + 1])
        rows_after.append(sum(a.shape[0] for a in xs))
    meta = dict(N=N, d=d, m=m, guard=float(dump["guard"]), I_sweep=I_sweep, conv_int=dump["conv_int"],
                device_err=dump["err"])
    outs = {}
    for (k, i) in PICKS:
        if k >= uF.shape[0] or i < I_sweep[k]:
            continue
        x = np.vstack(xs[:k + 1])
        y = np.vstack(ys[:k + 1])
        rng = np.random.default_rng(45)
        skip = sum((N - int(I_sweep[kk])) * n_tasks for kk in range(k)) + (i - int(I_sweep[k])) * n_tasks
        rng.integers(-8, 0, (skip, 2))
        state = rng.bit_generator.state
        mdl = ns.models.NNGP_p(n=d, N=N, worker_pool=pool, nn=m, seed=45)
        mdl.rng.bit_generator.state = state
        mdl.fit(x, y, k)
        q = u[k + 1][i]
        t0 = time.time()
        preds = mdl.predict(q.reshape(1, -1), uF[k][i + 1], uG[k][i + 1], i=i)
        secs = time.time() - t0
        probe = np.random.default_rng()
        probe.bit_generator.state = state
        starts = probe.integers(-8, 0, (n_tasks, 2)).astype(np.int8).reshape(d, 9, 1, 2)
        res = np.array([r[:5] for r in pool.last])          # theta0, theta1, fval, jitter, j in task order
        idx, _ = onn.knn(q, x, m)
        thetas, fvals = res[:, :2].reshape(d, 9, 2), res[:, 2].reshape(d, 9)
        sel = np.array([onn.select(fvals[j]) for j in range(d)])
        out = outs.setdefault(k, dict(meta, n_predicts=0))
        p = out["n_predicts"]
        out.update({f"p{p}_k": k, f"p{p}_i": i, f"p{p}_n_rows": x.shape[0], f"p{p}_query": q,
                    f"p{p}_xm": x[idx], f"p{p}_ym": y[idx], f"p{p}_starts": starts,
                    f"p{p}_preds": np.asarray(preds), f"p{p}_theta_sel": thetas[np.arange(d), sel],
                    f"p{p}_fvals": fvals})
        out["n_predicts"] = p + 1
        dd = np.abs(u[k + 1][i + 1] - uG[k + 1][i + 1] - preds)
        print(f"predict k={k} i={i} rows={x.shape[0]} {secs:.0f}s  inf searches {np.isinf(res[:, 2]).mean():.3f}  "
              f"|device-reference| max {dd.max():.3e} median {np.median(dd):.3e}  |pred| max {np.abs(preds).max():.3e}",
              flush=True)
        np.savez_compressed(os.path.join(OUT, f"run_fhn_d512_replay_k{k}.npz"), **out)
    pool.shutdown()


if __name__ == "__main__":
    main()
