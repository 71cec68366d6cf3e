"""GPU: every compiled kernel a launcher can choose (a "route") against the oracle, on both sides of every threshold.

The launchers pick among compiled kernels at run time from m, n, d, the number of queries, the number of slices, d_x
and the normalisation.  Each case below asserts the route it means to take by the number of kernel launches
(`nngp_launch_count`), so a case that silently leaves its route after a threshold moves fails instead of passing on
another kernel.  Where the count cannot tell two routes apart, the case says what selects its route.

Route                                              selected when                          reached by
-------------------------------------------------  -------------------------------------  -----------------------------------
kNN (csrc/knn.cu knn_launch, scan_select_launch)
scan_select_tile_kernel                            nq <= 4, m <= 32, d <= 6144, n <= 8192  test_knn_every_route (n <= 8192),
                                                   (1 launch; < m candidate lists when      test_knn_dimensions, test_knn_ties_*,
                                                   n < 16 m)                                test_knn_inf_and_nan_rows
scan_select_kernel<16>                             same, n > 8192 (1 launch)               test_knn_every_route (n = 8193), ties,
                                                                                           inf/NaN (n = 9000)
sqdist_kernel<8>                                   nq >= 8, d <= 768                       test_knn_every_route (nq = 8, 9)
sqdist_kernel<4>                                   nq >= 4 and d <= 1536, not above        test_knn_every_route (nq = 5),
                                                                                           test_knn_dimensions (d = 1000)
sqdist_one_kernel<16>                              d <= 6144, not above (nq < 4 with       test_knn_every_route (nq = 1, 3 with
                                                   m > 32, or d > 1536)                    m = 33, 160), test_knn_dimensions
sqdist_kernel_gq                                   d > 6144                                test_knn_dimensions (d = 6145)
 + select_kernel, one level                        m <= 32, n <= 4096 (2 launches)         test_knn_every_route (n <= 4096)
 + select_kernel, two levels                       m <= 32, n > 4096 (3 launches)          test_knn_every_route (n >= 4097),
                                                                                           test_knn_ties_across_every_chunking
 + select_big_kernel                               m > 32 (2 launches)                     test_knn_every_route (m = 33, 160)
fused r2 of the tile / scan kernel                 predict_host, 1 query, m <= 32          test_fused_neighbour_matrix_*

GP (csrc/gpfit.cu DISPATCH_M, gp_fit_predict_launch; M in {6, 8, ..., 32} is the smallest size >= m, m <= 32)
gp_nll_kernel<M>, gp_mean_kernel<M>                every M (gp_prep + 1 launch)            test_objective_and_mean_every_size
gp_fit_predict_kernel<M> (warp)                    mode warp, or auto with nq < 4 or       test_search_kernels_are_one_function
                                                   m > 20 and > quad_limit searches        (mode warp), test_fused_*
gp_fit_spec_kernel<M> (quad)                       mode quad, or auto with few searches    test_search_kernels_*, test_search_vs_
                                                                                           oracle_every_size, test_fit_predict_*
gp_fit_predict_kernel<M> + gp_fit_spec_kernel<M>   mode warp, set_fit_budget(>= 3)         test_search_kernels_are_one_function
gp_fit_grouped_kernel<M> + gp_select_mean_kernel   mode grouped, or auto with nq >= 4 and  test_search_kernels_are_one_function
                                                   m <= 20 (2 launches)
gp_fit_big_kernel + gp_select_mean_big_kernel      33 <= m <= 160 (2 launches, with        test_search_vs_oracle_every_size,
                                                   gp_prep_big_kernel)                     test_fit_predict_unsorted_index_list
gp_prep_kernel / gp_order_kernel                   every predict (1 launch each)           every predict above

RK (csrc/rk.cu rk_launch, launch_fhn_tile_s / _x, launch_pde)
rk_fhn_tile_kernel<S, 2, 64 | 256, ...>            FHN even d_x, not normalised, > 1 slice test_fhn_tile_shapes_and_shuffle (d_x = 8,
                                                   per SM or NNGP_RK_TILE=1                16, 32), test_fhn_time_chunked_*
rk_fhn_tile_kernel<S, 1, 128 | 512, ...>           <= 1 slice per SM and shuffle fits, or  test_fhn_tile_shapes_and_shuffle
                                                   NNGP_RK_TILE=2
 ... SHX = true (shuffle form)                     d_x / 2 a power of two, full warps,     test_fhn_tile_shapes_and_shuffle
                                                   <= 1 slice per SM, no NNGP_RK_NO_SHFL   (d_x = 8, 16, 32 at 1 and sms slices)
 ... chunked sequence (TB = 64)                    > 2 slices per SM and steps >= 4096     test_fhn_time_chunked_fine_step_d16
 ... TRAJ = true                                   run_F_full / run_G_full                 test_full_trajectory_last_row_*
rk_pde_kernel<FhnPde, S, 256 | 1024, NORM>         FHN odd d_x or normalised; TB = 1024    test_pde_kernels_vs_oracle (d_x = 5,
                                                   when d_x^2 > 256                        17, 20 normalised)
rk_pde_kernel<BurgersPde, S, 256 | 1024, NORM>     Burgers; TB = 1024 when d > 256         test_pde_kernels_vs_oracle (d = 3, 255,
                                                                                           256, 257, 1024, both normalisations)
rk_small_kernel<SYS, S>                            the ODE systems                         test_full_trajectory_last_row_* and
                                                                                           tests/test_gpu_kernels.py

S (stages) is chosen by the RK method alone; every RK case runs RK1, RK2, RK4 and RK8.  The environment switches used
here (NNGP_RK_TILE, NNGP_RK_NO_SHFL, NNGP_RK_CHUNKS) are read on every call.
"""
import os

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from oracle import nngp as onn
from oracle import rk as ork
from oracle import systems as osys
from helpers import make_dataset, scaled_err

pytestmark = pytest.mark.gpu

EPS = 2.2e-16
# m in {1, 2, 3} and M - 1, M for every compiled size M = 6, 8, ..., 32 of the one-lane-per-row kernels
SMALL_M = sorted({1, 2, 3} | {v for M in range(6, 33, 2) for v in (M - 1, M)})
BIG_M = [33, 34, 63, 64, 159, 160]


def counted(handle, fn, *args, **kwargs):
    """(fn(...), kernel launches it made)"""
    c0 = handle.launch_count()
    out = fn(*args, **kwargs)
    return out, handle.launch_count() - c0


def load(handle, x, y):
    handle.dataset_reset()
    handle.dataset_reserve(x.shape[0], x.shape[1])
    handle.dataset_append_host(x, y)


def knn_launches(nq, m, n, d):
    """launches of knn_launch: one for the fused scan (tile kernel up to 8192 rows, scan_select_kernel beyond -- the
    count cannot tell those two apart, n does); else a distance kernel + select_big (m > 32) / one select level
    (n <= 4096) / two select levels"""
    if nq <= 4 and m <= 32 and d * 8 <= 48 * 1024:
        return 1
    if m > 32 or n <= 4096:
        return 2
    return 3


# ---------------------------------------------------------------------------------------------------------------------
# A. GP at every specialisation size
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", SMALL_M)
def test_objective_and_mean_every_size(handle, m):
    """gp_nll_kernel<M> and gp_mean_kernel<M> at every compiled M, with padding rows (m < M) and without (m = M),
    against LAPACK: objective within 1e-9 relative where cond(K) < 1e6, +inf exactly where the amplitude overflows or
    10**sx underflows; posterior mean within 1e-8 relative where cond(K) < 1e7.  M is chosen by m alone."""
    import torch
    rng = np.random.default_rng(300 + m)
    n, d, nq, nt = 200, 6, 3, 40
    x, y = make_dataset(rng, n, d)
    load(handle, x, y)
    Q = x[rng.permutation(n)[:nq]] + 1e-3 * rng.standard_normal((nq, d))
    idx, dist = handle.knn_host(Q, m)
    dev = torch.device('cuda', handle.device)
    theta = np.stack([rng.uniform(-9, 2, (nq, d, nt)), rng.uniform(-9, 0, (nq, d, nt))], axis=-1)
    theta[:, :, 0] = [-400.0, -3.0]   # 10**sx underflows -> 1/0 = inf -> NaN -> +inf
    theta[:, :, 1] = [-3.0, 400.0]    # amplitude overflows
    jit = rng.integers(-20, -11, (nq, d, nt)).astype(float)
    out = torch.empty((nq, d, nt), dtype=torch.float64, device=dev)
    _, nl = counted(handle, handle.gp_nll, torch.from_numpy(idx).to(dev), nq, m, nt, torch.from_numpy(theta).to(dev),
                    torch.from_numpy(10.0 ** jit).to(dev), out)
    assert nl == 2  # gp_prep_kernel + gp_nll_kernel<M>
    got = out.cpu().numpy()
    n_cmp = 0
    for qi in range(nq):
        r2 = onn.pairwise_sqdist(x[idx[qi]], x[idx[qi]])
        for j in range(d):
            yy = y[idx[qi], j]
            for t in range(nt):
                want = onn.neg_log_lik(r2, yy, theta[qi, j, t], jit[qi, j, t])
                g = got[qi, j, t]
                if t < 2:
                    assert np.isinf(want) and g == np.inf, (t, want, g)
                    continue
                if not np.isfinite(want):
                    continue  # a singular matrix may fail in one factorisation and squeak through in the other
                K = onn.se_kernel_from_r2(r2, theta[qi, j, t]) + np.eye(m) * 10 ** jit[qi, j, t]
                if np.linalg.cond(K) < 1e6:
                    n_cmp += 1
                    assert abs(g - want) <= 1e-9 * max(1.0, abs(want)), (theta[qi, j, t], want, g)
    assert n_cmp > nq * d * 5, n_cmp
    # posterior mean at given hyper-parameters
    th = np.stack([rng.uniform(-2.5, 0.5, (nq, d)), rng.uniform(-8, -1, (nq, d))], axis=-1)
    jt = rng.integers(-20, -11, (nq, d)).astype(float)
    pred = torch.empty((nq, d), dtype=torch.float64, device=dev)
    _, nl = counted(handle, handle.gp_mean, torch.from_numpy(Q).to(dev), torch.from_numpy(idx).to(dev),
                    torch.from_numpy(dist).to(dev), nq, m, torch.from_numpy(th).to(dev), torch.from_numpy(jt).to(dev),
                    pred)
    assert nl == 2  # gp_prep_kernel + gp_mean_kernel<M>
    gp = pred.cpu().numpy()
    n_mean = 0
    for qi in range(nq):
        r2 = onn.pairwise_sqdist(x[idx[qi]], x[idx[qi]])
        for j in range(d):
            want = onn.posterior_mean(r2, dist[qi], y[idx[qi], j], th[qi, j], jt[qi, j])
            K = onn.se_kernel_from_r2(r2, th[qi, j]) + np.eye(m) * 10 ** jt[qi, j]
            if np.linalg.cond(K) < 1e7:
                n_mean += 1
                assert abs(gp[qi, j] - want) <= 1e-8 * abs(want), (qi, j, gp[qi, j], want)
    assert n_mean >= nq * d // 2, n_mean


@pytest.mark.parametrize("m", SMALL_M)
def test_search_kernels_are_one_function(handle, m):
    """The warp, grouped and quad search kernels and the budget continuation (warp + gp_fit_spec_kernel after 3
    evaluations) at every M: the same bits for every search, selection and prediction, with R = 1 and 2.  Rows 5-8 are
    exact copies of row 4 and two queries sit on them, so kernel matrices are singular and searches see +inf at every
    vertex: the head batch and the fast-forward of the all-inf iterations run at every M.  At M = 6 a grouped search has
    3 lanes, so the head-batch ballot of gp_fit_grouped_kernel (4 bits per group) never sees 4 failing points and the
    fast-forward never fires there; results stay the same, only the speed is lost."""
    rng = np.random.default_rng(400 + m)
    n, d, nq = 300, 4, 5
    x, y = make_dataset(rng, n, d)
    x[5:9] = x[4]
    y[5:9] = y[4]
    load(handle, x, y)
    Q = np.concatenate([x[4:5] + 0.0, x[4:5] + 1e-9, x[rng.permutation(n)[:nq - 2]] + 1e-3 * rng.standard_normal((nq - 2, d))])
    # predict_host with 5 queries: sqdist + one select level, gp_prep, gp_order, then the fit launches
    fit_launches = {"warp": 1, "quad": 1, "grouped": 2, "budget": 2}  # warp and quad cannot be told apart by the count
    for R in (1, 2):
        starts = rng.integers(-8, 0, (nq, d, 9, R, 2)).astype(np.int8)
        res = {}
        try:
            for mode in ("warp", "grouped", "quad", "budget"):
                handle.set_fit_mode("warp" if mode == "budget" else mode)
                handle.set_fit_budget(3 if mode == "budget" else 0)
                res[mode], nl = counted(handle, handle.predict_host, Q, m, starts, R, 0.1, 0.1, details=True)
                assert nl == 4 + fit_launches[mode], (mode, nl)
        finally:
            handle.set_fit_budget(0)
            handle.set_fit_mode("auto")
        for mode in ("grouped", "quad", "budget"):
            for key in ("idx", "nfev", "thetas", "fvals", "theta_opt", "jitter_opt", "fval_opt", "pred"):
                assert np.array_equal(res["warp"][key], res[mode][key], equal_nan=True), (mode, key, R)
        fv = res["warp"]["fvals"]
        if m >= 2:
            assert np.isinf(fv).sum() > 0 and np.isfinite(fv).sum() > 0, "the case must contain +inf and finite searches"


def _check_against_oracle_search(out, x_rows, kq, y_rows, starts, m, label):
    """selection rule, posterior mean and objective at the device's optimum against the oracle; returns the number of
    searches on SciPy's exact trajectory and the number of searches"""
    d = y_rows.shape[1]
    r2 = onn.pairwise_sqdist(x_rows, x_rows)
    same = total = 0
    for j in range(d):
        for a in range(9):
            th, fv, ne = onn.nm_run(r2, y_rows[:, j], starts[0, j, a, 0].astype(float), onn.JITTERS[a], 0.1, 0.1)
            total += 1
            same += bool(np.array_equal(out["thetas"][0, j, a, 0], th) and out["nfev"][0, j, a, 0] == ne)
        best = onn.select(out["fvals"][0, j, :, 0])
        assert out["jitter_opt"][0, j] == -20 + best, (label, j)
        assert out["fval_opt"][0, j] == out["fvals"][0, j, best, 0], (label, j)
        assert np.array_equal(out["theta_opt"][0, j], out["thetas"][0, j, best, 0]), (label, j)
        th_o, jit_o = out["theta_opt"][0, j], out["jitter_opt"][0, j]
        cond = np.linalg.cond(onn.se_kernel_from_r2(r2, th_o) + np.eye(m) * 10 ** jit_o)
        want_f = onn.neg_log_lik(r2, y_rows[:, j], th_o, jit_o)
        want_p = onn.posterior_mean(r2, kq, y_rows[:, j], th_o, jit_o)
        assert np.isfinite(out["pred"][0, j]), (label, j)
        if cond < 1e12 and np.isfinite(want_f):
            assert abs(out["fval_opt"][0, j] - want_f) <= max(1e-8, 10 * cond * EPS) * max(1.0, abs(want_f)), (label, j, cond)
            assert abs(out["pred"][0, j] - want_p) <= max(1e-8, 4 * cond * EPS) * abs(want_p) + 1e-14, (label, j, cond)
    assert np.all(out["nfev"] >= 3) and np.all(out["nfev"] <= 400)
    return same, total


# searches on SciPy's exact trajectory, over all sizes of each test (measured on the B200: see the docstrings)
_TRAJ = {}


@pytest.mark.parametrize("m", SMALL_M + BIG_M)
def test_search_vs_oracle_every_size(handle, m):
    """One query at every M and at the big sizes, against the oracle's search (SciPy Nelder-Mead over LAPACK):
    neighbour indices and distances bit-exact, selection = the reference rule on the device's own objective values,
    prediction = the oracle's posterior mean at the device's hyper-parameters (conditioning-aware tolerance), and the
    auto mode (quad kernel for m <= 32) gives the bits of the warp kernel.  Searches leave SciPy's trajectory at the
    first comparison of two objective values that agree to the last ulp or two; the fraction that follows it to the
    end is printed and asserted per size: measured on the B200, 13/27 (m = 1) to 26/27 (m = 32) of the searches, 18/27
    at the median.  The bar, 0.45, sits just under the lowest."""
    rng = np.random.default_rng(500 + m)
    n, d = 400, 3
    x, y = make_dataset(rng, n, d)
    load(handle, x, y)
    q = x[7:8] + 1e-3 * rng.standard_normal((1, d))
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    out, nl = counted(handle, handle.predict_host, q, m, starts, 1, 0.1, 0.1, details=True)
    # fused kNN + r2, gp_order, one fit launch (quad) -- or sqdist_one + select_big, gp_prep_big, gp_order, two fits
    assert nl == (3 if m <= 32 else 6), nl
    if m <= 32:
        try:
            handle.set_fit_mode("warp")
            warp, nl = counted(handle, handle.predict_host, q, m, starts, 1, 0.1, 0.1, details=True)
        finally:
            handle.set_fit_mode("auto")
        assert nl == 3
        for key in ("nfev", "thetas", "fvals", "theta_opt", "jitter_opt", "fval_opt", "pred"):
            assert np.array_equal(out[key], warp[key], equal_nan=True), key
    oi, okq = onn.knn(q[0], x, m)
    assert np.array_equal(out["idx"][0], oi)
    same, total = _check_against_oracle_search(out, x[oi], okq, y[oi], starts, m, m)
    frac = same / total
    print(f"m={m}: {same}/{total} searches on the oracle's trajectory ({frac:.2f})")
    assert frac >= 0.45, frac


@pytest.mark.parametrize("m", list(range(1, 13)) + [40])
def test_fit_predict_unsorted_index_list(handle, m):
    """nngp_fit_predict on an explicit index list that is not in distance order (models_alt.py: the 'col_only' rule
    calls it with m = k + 1 = 1, 2, 3, ... rows of one slice): rows and distances in a shuffled order, the oracle
    composed on the same order -- selection rule, objective and posterior mean at the device's optimum, and the
    fraction of searches on SciPy's trajectory (measured on the B200: 14/27 at m = 6 to 23/27; bar 0.45)."""
    import torch
    rng = np.random.default_rng(600 + m)
    n, d = 300, 3
    x, y = make_dataset(rng, n, d)
    load(handle, x, y)
    q = x[11:12] + 1e-3 * rng.standard_normal((1, d))
    near, _ = onn.knn(q[0], x, m)
    rows = rng.permutation(near)
    if m > 2:
        assert not np.array_equal(rows, near), "the index list must not be in distance order"
    kq = onn.sqdist_rows(q[0], x[rows])
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    dev = torch.device('cuda', handle.device)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    pred = torch.empty((1, d), dtype=torch.float64, device=dev)
    th = torch.empty((1, d, 2), dtype=torch.float64, device=dev)
    jit = torch.empty((1, d), dtype=torch.float64, device=dev)
    fv = torch.empty((1, d), dtype=torch.float64, device=dev)
    nfev = torch.empty((1, d, 9, 1), dtype=torch.int32, device=dev)
    fvals = torch.empty((1, d, 9, 1), dtype=torch.float64, device=dev)
    thetas = torch.empty((1, d, 9, 1, 2), dtype=torch.float64, device=dev)
    _, nl = counted(handle, handle.fit_predict, T(q), T(rows[None].astype(np.int64)), T(kq[None]), 1, m, 1, T(starts),
                    0.1, 0.1, pred, th, jit, fv, nfev, fvals, thetas)
    handle.synchronize()
    assert nl == (3 if m <= 32 else 4), nl  # gp_prep (+_big), gp_order, quad kernel / big fit + big select
    out = dict(pred=pred.cpu().numpy(), theta_opt=th.cpu().numpy(), jitter_opt=jit.cpu().numpy(),
               fval_opt=fv.cpu().numpy(), nfev=nfev.cpu().numpy(), fvals=fvals.cpu().numpy(), thetas=thetas.cpu().numpy())
    same, total = _check_against_oracle_search(out, x[rows], kq, y[rows], starts, m, m)
    frac = same / total
    print(f"unsorted m={m}: {same}/{total} searches on the oracle's trajectory ({frac:.2f})")
    assert frac >= 0.45, frac


# ---------------------------------------------------------------------------------------------------------------------
# B. kNN on both sides of every threshold
# ---------------------------------------------------------------------------------------------------------------------
def _knn_check(handle, Q, x, m, n_rows=0):
    n = n_rows or x.shape[0]
    (idx, dist), nl = counted(handle, handle.knn_host, Q, m, n_rows=n_rows)
    assert nl == knn_launches(Q.shape[0], m, n, x.shape[1]), (Q.shape[0], m, n, nl)
    for qi in range(Q.shape[0]):
        with np.errstate(all="ignore"):
            oi, od = onn.knn(Q[qi], x[:n], m)
        assert np.array_equal(idx[qi], oi), (qi, m, n)
        assert np.array_equal(dist[qi], od, equal_nan=True), (qi, m, n)


@pytest.mark.parametrize("m", [1, 16, 17, 31, 32, 33, 160])
@pytest.mark.parametrize("n_kind", ["m", "16m-1", "16m", "4096", "4097", "8192", "8193"])
def test_knn_every_route(handle, m, n_kind):
    """Indices and squared distances bit-identical to the oracle for nq in {1, 3, 4, 5, 8, 9}: n = m (every row
    selected), n = 16 m - 1 / 16 m (the tile kernel with fewer than / exactly m candidate lists), and both sides of the
    one/two-level selection (4096) and of the tile/scan kernels (8192).  Then the same searches as a prefix (n_rows)
    of a dataset whose extra rows are the queries themselves, which a search past the prefix would return first."""
    n = {"m": m, "16m-1": 16 * m - 1, "16m": 16 * m}.get(n_kind) or int(n_kind)
    if n < m:
        pytest.skip("n < m")
    rng = np.random.default_rng(700 + n + m)
    d = 5
    x, y = make_dataset(rng, n, d)
    nqs = (1, 3, 4, 5, 8, 9)
    Qall = x[rng.integers(0, n, 9)] + 1e-3 * rng.standard_normal((9, d))
    load(handle, x, y)
    for nq in nqs:
        _knn_check(handle, Qall[:nq], x, m)
    xp = np.concatenate([x, Qall])
    load(handle, xp, np.zeros_like(xp))
    for nq in nqs:
        _knn_check(handle, Qall[:nq], xp, m, n_rows=n)


@pytest.mark.parametrize("d", [1, 255, 256, 257, 1000, 2000, 6145])
def test_knn_dimensions(handle, d):
    """Every distance kernel: the tile kernel's column tiles of 256 (d = 255 / 256 / 257), sqdist_kernel<8> and <4>
    (d <= 768 / 1536), sqdist_one_kernel<16> (d = 2000, or m > 32 with nq < 4) and sqdist_kernel_gq (d = 6145,
    where the query row no longer fits 48 KB of shared memory), with one- and two-level selection and select_big."""
    rng = np.random.default_rng(800 + d)
    for n in ((300, 4500) if d <= 2000 else (300,)):
        x = rng.uniform(-1, 1, (n, d))
        load(handle, x, np.zeros_like(x))
        Q = x[rng.integers(0, n, 9)] + 1e-3 * rng.standard_normal((9, d))
        for nq in (1, 3, 5, 9):
            for m in (20, 40):
                _knn_check(handle, Q[:nq], x, m)
        _knn_check(handle, Q[:1], x, 20, n_rows=n - 7)


def _tie_dataset(rng, n):
    """rows equal to a (nearest to the query) at indices on both sides of every chunk boundary, rows equal to b (next)
    at 60 random indices, every other row farther away: the m-th neighbour is decided by index among exact ties"""
    d = 4
    a = rng.standard_normal(d)
    b = a + 0.1
    x = a + rng.uniform(1.0, 2.0, (n, d))
    cuts = [0, 15, 16, 31, 32, 255, 256, 511, 512, 1023, 1024, 2047, 2048, 4095, 4096, 8191, 8192, n - 1]
    ia = np.array(sorted({c for c in cuts if c < n}))
    rest = np.setdiff1d(np.arange(n), ia)
    ib = rng.choice(rest, size=min(60, rest.size), replace=False)
    x[ia] = a
    x[ib] = b
    return x, a + 1e-4


@pytest.mark.parametrize("n", [600, 8192, 9000])
def test_knn_ties_across_every_chunking(handle, n):
    """Exact ties broken by ascending index across the tile kernel's 16-row lists (n <= 8192, nq <= 4), the 256-row
    CTAs of scan_select_kernel (n > 8192, nq <= 4), the 1024-row chunks of the two-level select_kernel (n > 4096,
    nq >= 5) and in select_big_kernel (m = 160)."""
    rng = np.random.default_rng(900 + n)
    x, q = _tie_dataset(rng, n)
    load(handle, x, np.zeros_like(x))
    for nq in (1, 4, 5, 9):
        Q = np.repeat(q[None], nq, axis=0)
        for m in (16, 32, 160):
            _knn_check(handle, Q, x, m)


@pytest.mark.parametrize("n", [40, 5000, 9000])
def test_knn_inf_and_nan_rows(handle, n):
    """Rows whose squared distance overflows to +inf and rows containing NaN: finite distances first, then +inf, then
    NaN, each group by index (NumPy's stable argsort), on every route."""
    rng = np.random.default_rng(1000 + n)
    d = 4
    x = rng.uniform(-1, 1, (n, d))
    if n == 40:
        kind = np.repeat([0, 1, 2], [20, 10, 10])
        rng.shuffle(kind)
    else:  # few finite and +inf rows, so the selection reaches the NaN rows
        kind = np.full(n, 2)
        pos = rng.choice(n, 30, replace=False)
        kind[pos[:10]] = 0
        kind[pos[10:]] = 1
    big = rng.choice([-1e200, 1e200], (n, d))
    x[kind == 1] = np.where(rng.random((int((kind == 1).sum()), d)) < 0.5, big[kind == 1], x[kind == 1])
    x[kind == 1, 0] = 1e200
    x[kind == 2, rng.integers(0, d)] = np.nan
    load(handle, x, np.zeros_like(x))
    Q = rng.uniform(-1, 1, (9, d))
    for nq in (1, 4, 5, 9):
        for m in (32, 160):
            if m <= n:
                _knn_check(handle, Q[:nq], x, m)


@pytest.mark.parametrize("d", [3, 300, 512])
def test_fused_neighbour_matrix_equals_gp_prep(handle, d):
    """The neighbour matrix r2 written by the fused kNN kernel (1-query predict: one launch for scan, selection and
    r2) has the bits of gp_prep_kernel's (the same query as row 0 of a 2-query call: scan_select + gp_prep, and of a
    5-query call: sqdist + select_kernel + gp_prep).  Seen through the fits (mode warp, the same kernel in all three):
    every search, selection and prediction of query 0 is identical.  d = 300 ends in a partial 256-column tile."""
    rng = np.random.default_rng(1100 + d)
    n, m = 700, 20
    x, y = make_dataset(rng, n, d)
    load(handle, x, y)
    Q = x[rng.permutation(n)[:5]] + 1e-3 * rng.standard_normal((5, d))
    starts = rng.integers(-8, 0, (5, d, 9, 1, 2)).astype(np.int8)
    res = {}
    try:
        handle.set_fit_mode("warp")
        for nq, launches in ((1, 3), (2, 4), (5, 5)):
            res[nq], nl = counted(handle, handle.predict_host, Q[:nq], m, starts[:nq], 1, 0.1, 0.1, details=True)
            assert nl == launches, (nq, nl)
    finally:
        handle.set_fit_mode("auto")
    oi, _ = onn.knn(Q[0], x, m)
    assert np.array_equal(res[1]["idx"][0], oi)
    for nq in (2, 5):
        for key in ("idx", "nfev", "thetas", "fvals", "theta_opt", "jitter_opt", "fval_opt", "pred"):
            assert np.array_equal(res[1][key][0], res[nq][key][0], equal_nan=True), (nq, key)


# ---------------------------------------------------------------------------------------------------------------------
# C. RK in every launch shape
# ---------------------------------------------------------------------------------------------------------------------
METHODS = (("RK1", 6), ("RK2", 5), ("RK4", 4), ("RK8", 3))


def _sms(handle):
    import torch
    return torch.cuda.get_device_properties(handle.device).multi_processor_count


def _rk_pair(system, size, norm):
    kw = {} if norm is None else dict(normalization=norm)
    if system == "fhn":
        return osys.FHN_PDE(d_x=size, **kw), nn.FHN_PDE(d_x=size, **kw)
    return osys.Burgers(d_x=size, **kw), nn.Burgers(d_x=size, **kw)


PDE_CASES = [("fhn", 5, None), ("fhn", 17, None), ("fhn", 20, "-11")] + \
            [("burgers", d, norm) for d in (3, 255, 256, 257, 1024) for norm in (None, "-11")]


@pytest.mark.parametrize("system,size,norm", PDE_CASES)
def test_pde_kernels_vs_oracle(handle, system, size, norm):
    """rk_pde_kernel<FhnPde | BurgersPde, S, TB, NORM> for 256 and 1024 threads (more than 256 grid points), with and
    without normalisation, every RK method, both step conventions, against the dense NumPy oracle.  The kernel is
    selected by the system, its point count and its normalisation alone (one launch whatever the instantiation).
    The step is as long as the stiffest mode allows (h times the largest eigenvalue about 1), so the stage values are
    a sizeable part of the state and a wrong last bit in one of them shows above the stencil-vs-dense rounding: measured
    on the B200, the scaled error is below 1e-15 in every case; the bar is 1e-14."""
    rng = np.random.default_rng(1200 + size)
    o, dev = _rk_pair(system, size, norm)
    n = 3
    u0 = dev.get_init_cond()[None, :] + 0.1 * rng.standard_normal((n, dev.get_dim()))
    # explicit steps at the edge of the stability region of the stencils (Burgers: diffusion nu (d - 1)^2 at the
    # highest wave number; FHN: the reaction rate 1 / tau = 10 and the v-diffusion up to 36 at d_x = 20)
    dt = 0.03 if system == "fhn" else min(0.05, 1.0 / (0.01 * (size - 1) ** 2))
    t0 = np.arange(n) * 0.5
    worst = 0.0
    for h_mode in ("linspace", "const"):
        for F, steps in METHODS:
            t1 = t0 + dt * steps
            s = nn.CudaSolverRK(dev.get_vector_field(), Ng=1, Nf=steps, F=F, G='RK1', h_mode=h_mode, handle=handle)
            got, nl = counted(handle, s.run_F_batch, t0, t1, u0)
            assert nl == 1
            want = np.stack([ork.rk_last(o.f, F, t0[i], t1[i], steps, u0[i], h_mode) for i in range(n)])
            err = scaled_err(got, want)
            worst = max(worst, err)
            assert err < 1e-14, (h_mode, F, err)
            assert not np.array_equal(got, u0)
    print(f"{system} size={size} norm={norm}: worst scaled error against the oracle {worst:.2e}")


def _fhn_variants(s, t0, t1, u0):
    """run_F_batch under every forced tile shape, with and without the shuffle form"""
    out = {}
    try:
        for tile in (None, "0", "1", "2"):
            for no_shfl in (False, True):
                if tile is None:
                    os.environ.pop("NNGP_RK_TILE", None)
                else:
                    os.environ["NNGP_RK_TILE"] = tile
                if no_shfl:
                    os.environ["NNGP_RK_NO_SHFL"] = "1"
                else:
                    os.environ.pop("NNGP_RK_NO_SHFL", None)
                out[(tile, no_shfl)] = s.run_F_batch(t0, t1, u0)
    finally:
        os.environ.pop("NNGP_RK_TILE", None)
        os.environ.pop("NNGP_RK_NO_SHFL", None)
    return out


@pytest.mark.parametrize("d_x,slices", [(8, "1"), (8, "sms"), (32, "1"), (32, "sms"), (16, "1"), (16, "sms"),
                                        (16, "sms+1")])
def test_fhn_tile_shapes_and_shuffle(handle, d_x, slices):
    """rk_fhn_tile_kernel in its 1x2 (TY = 1, 128 / 512 threads) and 2x2 (TY = 2, 64 / 256 threads) shapes, shuffle
    form (d_x / 2 a power of two, at most one slice per SM) and plain form, and the one-point-per-thread kernel
    (NNGP_RK_TILE = 0): all the same bits at 1, sms and sms + 1 slices (the shuffle form stops at sms + 1), every RK
    method, and within 1e-12 (scaled) of the NumPy oracle on a few slices."""
    rng = np.random.default_rng(1300 + d_x)
    sms = _sms(handle)
    n = {"1": 1, "sms": sms, "sms+1": sms + 1}[slices]
    o, dev = osys.FHN_PDE(d_x=d_x), nn.FHN_PDE(d_x=d_x)
    u0 = dev.get_init_cond()[None, :] + 0.01 * rng.standard_normal((n, dev.get_dim()))
    t0 = np.arange(n) * 0.01
    t1 = t0 + 0.05
    for F, steps in METHODS:
        s = nn.CudaSolverRK(dev.get_vector_field(), Ng=1, Nf=steps, F=F, G='RK1', handle=handle)
        c0 = handle.launch_count()
        out = _fhn_variants(s, t0, t1, u0)
        assert handle.launch_count() - c0 == len(out)  # one launch each: no chunking below 4096 steps
        ref = out[("0", False)]
        for key, got in out.items():
            assert np.array_equal(got, ref), (F, key)
        for i in sorted({0, n // 2, n - 1}):
            want = ork.rk_last(o.f, F, t0[i], t1[i], steps, u0[i])
            assert scaled_err(ref[i], want) < 1e-12, (F, i)


def test_fhn_time_chunked_fine_step_d16(handle):
    """The production grid (d_x = 16) with more than two slices per SM and >= 4096 steps runs as a sequence of
    balanced launches over (chunk of steps, slice) tasks: the bits of the single launch (NNGP_RK_CHUNKS = 0), both step
    conventions."""
    rng = np.random.default_rng(14)
    sms = _sms(handle)
    n = 2 * sms + 1
    dev = nn.FHN_PDE(d_x=16)
    u0 = dev.get_init_cond()[None, :] + 0.01 * rng.standard_normal((n, dev.get_dim()))
    t0 = rng.uniform(0, 1, n)
    t1 = t0 + rng.uniform(0.5, 1.5, n)
    for h_mode in ("linspace", "const"):
        s = nn.CudaSolverRK(dev.get_vector_field(), Ng=1, Nf=4100, F='RK4', G='RK1', h_mode=h_mode, handle=handle)
        got, nl = counted(handle, s.run_F_batch, t0, t1, u0)
        assert nl > 1, nl
        try:
            os.environ["NNGP_RK_CHUNKS"] = "0"
            ref, nl0 = counted(handle, s.run_F_batch, t0, t1, u0)
        finally:
            del os.environ["NNGP_RK_CHUNKS"]
        assert nl0 == 1
        assert np.all(np.isfinite(got)) and np.array_equal(got, ref), h_mode


FULL_CASES = [("lorenz", None), ("fhn", 16), ("fhn", 5), ("burgers", 257)]


@pytest.mark.parametrize("system,size", FULL_CASES)
def test_full_trajectory_last_row_equals_run_F(handle, system, size):
    """run_F_full (the TRAJ instantiations: rk_small_kernel, rk_fhn_tile_kernel, rk_pde_kernel with 256 and 1024
    threads) starts at u0, follows the oracle's trajectory, and its last row has the bits of run_F."""
    if system == "lorenz":
        o, dev = osys.Lorenz(normalization='-11'), nn.Lorenz(normalization='-11')
        tol, dt = 0.0, 0.01
    else:
        o, dev = _rk_pair(system, size, None)
        tol, dt = 1e-11, (0.02 if system == "fhn" else 2e-5)
    u0 = dev.get_init_cond()
    for F, steps in METHODS:
        s = nn.CudaSolverRK(dev.get_vector_field(), Ng=steps, Nf=steps, F=F, G=F, handle=handle)
        t1 = 0.3 + dt * steps
        traj = s.run_F_full(0.3, t1, u0)
        assert traj.shape == (steps + 1, u0.size)
        assert np.array_equal(traj[0], u0) and np.array_equal(traj[-1], s.run_F(0.3, t1, u0)), F
        want = ork.rk_full(o.f, F, 0.3, t1, steps, u0)
        if tol == 0.0:
            assert np.array_equal(traj, want), F
        else:
            assert scaled_err(traj, want) < tol, F
