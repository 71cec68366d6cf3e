"""GPU diagnostic: where device and reference select different optima on the replayed FHN d=512 predicts, who is right
about the VALUE of the objective at the other side's optimum?  Prints, per predict, a 2x2 classification."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from nearest_neighbors_gparareal_b200 import _lib
from oracle import nngp as onn

h = _lib.default_handle(0)
dev = torch.device('cuda', 0)
zs = [np.load(os.path.join(ROOT, "tests", "golden", f"run_fhn_d512_replay_k{k}.npz")) for k in (2, 3)]
m, d = int(zs[0]["m"]), int(zs[0]["d"])
for z, p in [(z, p) for z in zs for p in range(int(z["n_predicts"]))]:
    P = {k: z[f"p{p}_{k}"] for k in ("k", "i", "query", "xm", "ym", "starts", "preds", "theta_sel", "fvals")}
    if np.abs(P["preds"]).max() < 1e-8:
        continue
    h.dataset_reset(); h.dataset_reserve(m, d); h.dataset_append_host(P["xm"], P["ym"])
    out = h.predict_host(P["query"][None], m, P["starts"][None], 1, 0.1, 0.1, details=True)
    r2 = onn.pairwise_sqdist(P["xm"], P["xm"])
    sel_r = np.array([onn.select(P["fvals"][j]) for j in range(d)])
    th_r = P["theta_sel"]
    jit_r = onn.JITTERS[sel_r]
    f_r = P["fvals"][np.arange(d), sel_r]
    th_d, jit_d, f_d = out["theta_opt"][0], out["jitter_opt"][0], out["fval_opt"][0]
    # device objective at the reference's optimum, LAPACK objective at the device's optimum
    idx = torch.arange(m, dtype=torch.int64, device=dev)[None].contiguous()
    th = torch.from_numpy(np.stack([th_r, th_d], 1)[None].copy()).to(dev)           # [1, d, 2, 2]
    j10 = torch.from_numpy((10.0 ** np.stack([jit_r, jit_d], 1))[None].copy()).to(dev)
    o = torch.empty((1, d, 2), dtype=torch.float64, device=dev)
    h.gp_nll(idx, 1, m, 2, th, j10, o)
    dv = o.cpu().numpy()[0]
    dev_at_ref, dev_at_dev = dv[:, 0], dv[:, 1]
    lap_at_dev = np.array([onn.neg_log_lik(r2, P["ym"][:, j], th_d[j], jit_d[j]) for j in range(d)])
    tol = 1e-6 * np.maximum(1.0, np.abs(f_r))
    ref_lower = f_r < f_d - tol
    dev_lower = f_d < f_r - tol
    def cls(mask, a, b, name):
        # a: value claimed by the side that found it, b: the other side's evaluation of the same point
        agree = np.abs(a[mask] - b[mask]) <= 1e-6 * np.maximum(1.0, np.abs(a[mask]))
        binf = np.isinf(b[mask])
        higher = (~agree) & (~binf) & (b[mask] > a[mask])
        lower = (~agree) & (~binf) & (b[mask] < a[mask])
        print(f"   {name}: {mask.sum()} dims; other side evaluates that optimum: same value {agree.sum()}, +inf {binf.sum()}, "
              f"higher {higher.sum()} (median gap {np.median((b[mask]-a[mask])[higher]) if higher.any() else 0:.3g}), lower {lower.sum()}")
    print(f"predict k={int(P['k'])} i={int(P['i'])}: device self-consistency max|f_dev - nll_dev(theta_dev)| "
          f"{np.nanmax(np.abs(f_d - dev_at_dev)):.2e}")
    cls(ref_lower, f_r, dev_at_ref, "reference found a lower optimum")
    cls(dev_lower, f_d, lap_at_dev, "device found a lower optimum   ")
    dp = np.abs(out["pred"][0] - P["preds"])
    big = dp > 5e-8
    print(f"   dims with |pred diff| > 5e-8: {big.sum()}; of those reference-lower {np.sum(big & ref_lower)}, device-lower {np.sum(big & dev_lower)}, same optimum value {np.sum(big & ~ref_lower & ~dev_lower)}")
    # conditioning of the selected matrices
    def cond(th, jit, j):
        K = onn.se_kernel_from_r2(r2, th) + np.eye(m) * 10 ** jit
        return np.linalg.cond(K)
    cr = np.array([cond(th_r[j], jit_r[j], j) for j in range(0, d, 8)])
    cdv = np.array([cond(th_d[j], jit_d[j], j) for j in range(0, d, 8)])
    print(f"   log10 cond of the selected kernel matrix: reference median {np.median(np.log10(cr)):.1f} max {np.log10(cr).max():.1f}; "
          f"device median {np.median(np.log10(cdv)):.1f} max {np.log10(cdv).max():.1f}")
