"""The one-warp search kernel (gp_fit_predict_kernel) screens the next 32 points of a search whose simplex is all +inf
at once, one per lane, skips the leading whole iterations whose points all fail the screen, and replays the other
screened-out points as +inf without evaluating them.  Neighbour rows that are exact copies of each other make the
kernel matrix singular, so searches start with every vertex +inf; some meet a finite value after a while and leave
the look-ahead window somewhere inside it, others run all 400 evaluations at +inf.  The searches must be the bits of
the one-by-one evaluation (NNGP_FIT_NO_HEAD_BATCH) and of the oracle's Nelder-Mead (oracle/nelder_mead.py) driven by
the device's own objective (gp_nll_kernel)."""
import os

import numpy as np
import pytest

from oracle.nelder_mead import nelder_mead

pytestmark = pytest.mark.gpu

JIT10 = [float(f"1e{a}") for a in range(-20, -11)]  # the literals of c_jit10


def _load(handle, x, y):
    handle.dataset_reset()
    handle.dataset_reserve(x.shape[0], x.shape[1])
    handle.dataset_append_host(x, y)


def _dataset(rng, n, d, m, ndup, scale):
    """rows 0..ndup-1 are copies of row 0; the other neighbours of x[0] sit at distance ~scale"""
    x = rng.uniform(-1, 1, (n, d))
    x[1:ndup] = x[0]
    x[ndup:m] = x[0] + scale * rng.standard_normal((m - ndup, d))
    y = 1e-3 * np.sin(x @ rng.standard_normal((d, d)))
    return x, y


def _allinf_points(start):
    """the points a search from `start` evaluates while every value is +inf (SciPy's order and arithmetic)"""
    s = np.array(start, dtype=float)
    sim = np.array([s, s.copy(), s.copy()])
    for k in range(2):
        sim[k + 1][k] = 1.05 * s[k] if s[k] != 0 else 0.00025
    pts = [sim[0].copy(), sim[1].copy(), sim[2].copy()]
    while len(pts) < 400:
        xb = (sim[0] + sim[1]) / 2
        pts.append(2 * xb - 1 * sim[2])
        pts.append(0.5 * xb + 0.5 * sim[2])
        sim[1] = sim[0] + 0.5 * (sim[1] - sim[0])
        pts.append(sim[1].copy())
        sim[2] = sim[0] + 0.5 * (sim[2] - sim[0])
        pts.append(sim[2].copy())
    return np.array(pts[:400])


def test_lookahead_searches_are_the_one_by_one_and_oracle_bits(handle):
    """6 912 searches on 24 neighbour sets with copied rows: all of them bit-identical to the one-by-one evaluation;
    the ones that leave an all-inf run (and five that never do) also to the oracle's search on the device objective.
    Where a search leaves the run inside the look-ahead window depends on rounding noise of the singular matrix, so
    the positions reached are printed, not required."""
    import torch
    rng = np.random.default_rng(77)
    n, d, m = 200, 32, 20
    dev = torch.device("cuda", handle.device)
    positions, never, replayed = set(), 0, 0
    handle.set_fit_mode("warp")
    try:
        for case in range(24):
            x, y = _dataset(rng, n, d, m, ndup=int(rng.integers(2, 9)), scale=10.0 ** rng.uniform(-6, -1))
            _load(handle, x, y)
            q = x[0:1] + 0.0
            starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
            got = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
            os.environ["NNGP_FIT_NO_HEAD_BATCH"] = "1"
            try:
                ref = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
            finally:
                del os.environ["NNGP_FIT_NO_HEAD_BATCH"]
            for key in ("nfev", "thetas", "fvals", "theta_opt", "fval_opt", "jitter_opt", "pred"):
                assert np.array_equal(got[key], ref[key], equal_nan=True), (case, key)

            # the device objective along every search's all-inf trajectory, in one launch
            d_idx = torch.from_numpy(np.ascontiguousarray(got["idx"][:1])).to(dev)
            pts = np.stack([[_allinf_points(starts[0, j, a, 0]) for a in range(9)] for j in range(d)])  # [d,9,400,2]
            th = torch.from_numpy(np.ascontiguousarray(pts.reshape(d, 9 * 400, 2))).to(dev)
            j10 = torch.from_numpy(np.ascontiguousarray(np.tile(np.repeat(np.array(JIT10), 400), (d, 1)))).to(dev)
            out = torch.empty((d, 9 * 400), dtype=torch.float64, device=dev)
            handle.gp_nll(d_idx, 1, m, 9 * 400, th, j10, out)
            torch.cuda.synchronize()
            pre = out.cpu().numpy().reshape(d, 9, 400)
            one_th = torch.empty((d, 1, 2), dtype=torch.float64, device=dev)
            one_j = torch.empty((d, 1), dtype=torch.float64, device=dev)
            one_out = torch.empty((d, 1), dtype=torch.float64, device=dev)
            for j in range(d):
                for a in range(9):
                    fin = np.flatnonzero(np.isfinite(pre[j, a]))
                    if fin.size == 0:
                        never += 1
                        if never > 5:
                            continue
                    elif fin[0] < 3:
                        continue  # a finite initial vertex: no all-inf run
                    else:
                        positions.add(int(fin[0] - 3) % 32)  # where the run ends inside its look-ahead window
                    calls = [0]

                    def f(theta):
                        i = calls[0]
                        calls[0] += 1
                        if i < 400 and np.array_equal(theta, pts[j, a, i]):
                            return pre[j, a, i]
                        one_th.copy_(torch.from_numpy(np.tile(theta, (d, 1, 1))))
                        one_j.fill_(JIT10[a])
                        handle.gp_nll(d_idx, 1, m, 1, one_th, one_j, one_out)
                        torch.cuda.synchronize()
                        return float(one_out[j, 0])

                    xo, fo, nfev, _, _ = nelder_mead(f, starts[0, j, a, 0].astype(float), xatol=0.1, fatol=0.1)
                    replayed += 1
                    assert nfev == got["nfev"][0, j, a, 0], (case, j, a)
                    assert np.array_equal(xo, got["thetas"][0, j, a, 0]), (case, j, a)
                    assert np.array_equal(fo, got["fvals"][0, j, a, 0]), (case, j, a)
    finally:
        handle.set_fit_mode("auto")
    print(f"look-ahead window positions where an all-inf run ended: {sorted(positions)}; searches all +inf: {never}; "
          f"searches checked against the oracle: {replayed}")
    assert never >= 5, "the case must contain searches that see +inf at all 400 evaluations"
