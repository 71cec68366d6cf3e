"""Ensembles whose members differ in neighbour count and time span, and the per-predict-m fit behind them.

A. nngp_fit_predict_mixed: every predict equals predict_host at its own m, bit for bit, on every fit route.
B. Every member of a mixed ensemble equals its solo PararealDevice run with its own nn and tspan, bit for bit.
"""
import json
import os

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib
from helpers import device_system, make_dataset
from test_gpu_ensemble import _ensemble, _same, _setup, _solo, _solver
from test_gpu_routes import SMALL_M, counted, load

pytestmark = pytest.mark.gpu

KEYS = ("nfev", "thetas", "fvals", "theta_opt", "jitter_opt", "fval_opt", "pred")


@pytest.fixture(scope="module")
def handle():
    return _lib.Handle(0)


def _fit_launches(m, n_g, mode):
    """fit launches of one group of n_g predicts at m (gp_fit_predict_launch's route choice)"""
    if m > 32:
        return 2
    grouped = mode == "grouped" or (mode == "auto" and n_g >= 4 and m <= 20)
    return 2 if grouped else 1


@pytest.mark.parametrize("ms", [SMALL_M + [11, 11, 11, 20, 20, 20, 20], [11, 32, 33, 40, 160, 11, 40]],
                         ids=["small", "straddle"])
def test_mixed_fit_equals_predict_host_at_each_m(handle, ms):
    import torch
    rng = np.random.default_rng(7 + len(ms))
    n, d = 300, 4
    x, y = make_dataset(rng, n, d)
    x[5:9] = x[4]  # duplicated rows: singular matrices, all-inf searches and their fast-forward
    y[5:9] = y[4]
    load(handle, x, y)
    nq, ld = len(ms), max(ms)
    Q = np.stack([x[4] + (0.0 if q % 3 == 0 else 1e-9) if q % 3 < 2 else
                  x[rng.integers(n)] + 1e-3 * rng.standard_normal(d) for q in range(nq)])
    idx, dist = handle.knn_host(Q, ld)
    d_idx, d_dist = torch.from_numpy(idx).cuda(), torch.from_numpy(dist).cuda()
    groups = {m: ms.count(m) for m in set(ms)}
    for R in (1, 2):
        starts = rng.integers(-8, 0, (nq, d, 9, R, 2)).astype(np.int8)
        d_starts = torch.from_numpy(starts).cuda()
        try:
            for mode in ("warp", "grouped", "quad", "auto"):
                handle.set_fit_mode(mode)
                out = dict(pred=torch.empty((nq, d), dtype=torch.float64, device='cuda'),
                           theta_opt=torch.empty((nq, d, 2), dtype=torch.float64, device='cuda'),
                           jitter_opt=torch.empty((nq, d), dtype=torch.float64, device='cuda'),
                           fval_opt=torch.empty((nq, d), dtype=torch.float64, device='cuda'),
                           nfev=torch.empty((nq, d, 9, R), dtype=torch.int32, device='cuda'),
                           fvals=torch.empty((nq, d, 9, R), dtype=torch.float64, device='cuda'),
                           thetas=torch.empty((nq, d, 9, R, 2), dtype=torch.float64, device='cuda'))
                _, nl = counted(handle, handle.fit_predict_mixed, None, d_idx, d_dist, ms, R, d_starts, 0.1, 0.1,
                                out['pred'], out['theta_opt'], out['jitter_opt'], out['fval_opt'], out['nfev'],
                                out['fvals'], out['thetas'])
                torch.cuda.synchronize()
                # neighbour matrix at ld, the gather, per distinct m the queue order and its fit, the scatter
                assert nl == 3 + sum(1 + _fit_launches(m, g, mode) for m, g in groups.items()), (mode, nl)
                out = {k: v.cpu().numpy() for k, v in out.items()}
                for q, m in enumerate(ms):
                    ref = handle.predict_host(Q[q:q + 1], m, starts[q:q + 1], R, 0.1, 0.1, details=True)
                    assert np.array_equal(idx[q, :m], ref['idx'][0]), (mode, q, m)
                    for key in KEYS:
                        assert np.array_equal(out[key][q], ref[key][0], equal_nan=True), (mode, R, q, m, key)
        finally:
            handle.set_fit_mode("auto")


def _mixed_case(name, seeds, nns, n_restarts=None, **run_kw):
    cfg, eps, key, kw, mkw = _setup(name, n_restarts)
    mkw.pop('nn', None)
    outs = _ensemble(key, kw, cfg, eps, mkw, seeds, nn=nns, **run_kw)
    for s, v, o in zip(seeds, nns, outs):
        _same(o, _solo(key, kw, cfg, eps, dict(mkw, nn=v), s, max_rows=run_kw.get('max_rows')), (name, s, v))
    return outs


def test_members_with_their_own_nn_equal_solo_runs_lorenz():
    nns = ['adaptive', 11, 12, 13, 14, 15, 16]
    _mixed_case("lorenz_N50_m11", [45] * 7 + [46] * 7, nns + nns)


@pytest.mark.parametrize("name,seeds,nns,n_restarts", [
    ("hopf_N32_m15", [45, 46, 47], [15, 11, 'adaptive'], 2),
    ("burgers_d32_N32_m12", [45, 46, 47], [11, 18, 30], None),
    ("lorenz_N50_m11", [45, 46, 47], [11, 40, 'adaptive'], None),  # straddles m = 32
])
def test_members_with_their_own_nn_equal_solo_runs(name, seeds, nns, n_restarts):
    _mixed_case(name, seeds, nns, n_restarts)


def test_mixed_nn_with_a_growing_store():
    outs = _mixed_case("lorenz_N50_m11", [45, 46, 47], [11, 13, 'adaptive'], max_rows=51)
    assert all(o['n_rows'] > 51 for o in outs)


def test_members_with_their_own_tspan_equal_solo_runs():
    cfg, eps, key, kw, mkw = _setup("burgers_d32_N32_m12")
    mkw.pop('nn', None)
    Ts = [5.0, 5.9, 5.0, 5.9, 5.9]
    nns = [11, 11, 18, 30, 18]
    seeds = [45, 46, 47, 48, 49]
    outs = _ensemble(key, kw, cfg, eps, mkw, seeds, nn=nns, tspans=[[0, T] for T in Ts])
    for s, v, T, o in zip(seeds, nns, Ts, outs):
        assert np.array_equal(o['t'], np.linspace(0, T, cfg["N"] + 1))
        _same(o, _solo(key, kw, dict(cfg, tspan=[0, T]), eps, dict(mkw, nn=v), s), (s, v, T))
    # one time span for all, different from the ensemble's own: the uniform sweep with the members' grid
    outs = _ensemble(key, kw, cfg, eps, mkw, seeds[:2], nn=18, tspans=[[0, 5.9]] * 2)
    for s, o in zip(seeds[:2], outs):
        _same(o, _solo(key, kw, dict(cfg, tspan=[0, 5.9]), eps, dict(mkw, nn=18), s), s)


def test_burgers_published_slice_as_one_ensemble():
    """Burgers_K_vs_m: T in {5, 5.9} x nn in {11, 18, 30} x 4 published seeds in one run"""
    pub = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "published.json")))
    runs = []
    for T in (5.0, 5.9):
        for nnb in (11, 18, 30):
            runs += [(T, nnb, seed, K) for T_, n_, seed, K in pub["Burgers_K_vs_m"] if (T_, n_) == (T, nnb)][:4]
    assert len(runs) == 24
    ode = nn.Burgers(d_x=128, normalization='-11')
    solver = nn.CudaSolverRK(ode.get_vector_field(), Ng=4, Nf=2000, G='RK1', F='RK8')
    ens = nn.PararealEnsemble(ode, solver, tspan=[0, 5.0], N=128, epsilon=5e-7, verbose='')
    outs = ens.run(model='nngp', seeds=[r[2] for r in runs], nn=[r[1] for r in runs],
                   tspans=[[0, r[0]] for r in runs])
    v = np.array([(o['k'] if o['converged'] else 128) - r[3] for o, r in zip(outs, runs)])
    print(f"Burgers T x nn x 4 seeds: K_ensemble - K_published histogram {dict(zip(*np.unique(v, return_counts=True)))}")
    assert abs(v.mean()) <= 0.5 and np.mean(np.abs(v) <= 1) >= 0.85, v
    for e in (0, 9, 23):
        T, nnb, seed, _ = runs[e]
        ode1 = nn.Burgers(d_x=128, normalization='-11')
        s1 = nn.CudaSolverRK(ode1.get_vector_field(), Ng=4, Nf=2000, G='RK1', F='RK8')
        ref = nn.PararealDevice(ode1, s1, tspan=[0, T], N=128, epsilon=5e-7, verbose='').run(
            model='nngp', nn=nnb, seed=seed)
        _same(outs[e], ref, (T, nnb, seed))


def _counted(h):
    """wraps h.ensemble_sweep: the list it returns gets the launches of every call"""
    sweep, launches = h.ensemble_sweep, []

    def counted_sweep(*args):
        c0 = h.launch_count()
        try:
            sweep(*args)
        finally:
            launches.append(h.launch_count() - c0)

    h.ensemble_sweep = counted_sweep
    return launches


def test_one_nn_with_their_own_tspans_sweeps_in_place():
    """one m for all, two time spans: the in-place route reads each member's grid from the per-position table"""
    cfg, eps, key, kw, mkw = _setup("burgers_d32_N32_m12")
    mkw.pop('nn', None)
    Ts, seeds = [5.0, 5.9, 5.0, 5.9], [45, 46, 47, 48]
    ode = device_system(key, **kw)
    ens = nn.PararealEnsemble(ode, _solver(ode, cfg), tspan=cfg["tspan"], N=cfg["N"], epsilon=eps, verbose='')
    launches = _counted(ens.handle())
    outs = ens.run(model='nngp', seeds=seeds, nn=12, tspans=[[0, T] for T in Ts], **mkw)
    # the first sweep, all four members at I = 1: the time table, then per slice the queue order, the coarse step,
    # the segmented kNN and the grouped fit (searches, then selection and mean)
    assert launches[0] == 1 + 5 * (cfg["N"] - 1), launches
    for s, T, o in zip(seeds, Ts, outs):
        _same(o, _solo(key, kw, dict(cfg, tspan=[0, T]), eps, dict(mkw, nn=12), s), (s, T))


def test_row_shortfall_is_refused_by_the_library_before_any_launch():
    """nn=60 beside nn=11, and nn=60 for both, at the first iteration, where every member holds N = 50 rows"""
    cfg, eps, key, kw, mkw = _setup("lorenz_N50_m11")
    mkw.pop('nn', None)
    for nns in ([11, 60], [60, 60]):
        ode = device_system(key, **kw)
        ens = nn.PararealEnsemble(ode, _solver(ode, cfg), tspan=cfg["tspan"], N=cfg["N"], epsilon=eps, verbose='')
        launches = _counted(ens.handle())
        with pytest.raises(_lib.NNGPError, match=r"member \d+ holds 50 rows, fewer than m=60"):
            ens.run(model='nngp', seeds=[45, 46], nn=nns, **mkw)
        assert launches == [0], (nns, launches)
