"""PararealEnsemble and its kernels against the solo device path.

A. The segmented kNN (nngp_knn_segmented) equals nngp_knn run on each segment alone, after subtracting the segment's
   base, on both routes (the fused tile kernel for segments up to 8192 rows and m <= 32, asserted through the launch
   counter; the distance + selection kernels beyond), with exact ties, +inf and NaN rows; its neighbour matrix has the
   bits of the cdist arithmetic gp_prep_kernel uses.
B. Every member of an ensemble equals its solo PararealDevice run bit for bit: k, conv_int, u, err (NaN positions
   included) and n_rows.
"""
import json
import os

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib
from helpers import case_system, device_system, load_run

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def seg_handle():
    return _lib.Handle(0)


@pytest.fixture(scope="module")
def ref_handle():
    return _lib.Handle(0)


# ---------------------------------------------------------------------------------------------------------------------
# A. segmented kNN
# ---------------------------------------------------------------------------------------------------------------------
def _segment(rng, L, d, kind):
    """rows of one segment: uniform, with exact duplicates (ties by index), or with +inf / NaN rows"""
    x = rng.uniform(-1, 1, (L, d))
    if kind == 1 and L > 2:  # ties: copies of row 0 across the segment, at both ends of 16-row lists
        at = np.unique(np.concatenate([[L - 1, L // 2], rng.choice(L, min(L, 40), replace=False)]))
        x[at] = x[0]
    if kind == 2 and L > 4:
        bad = rng.choice(L, max(1, L // 3), replace=False)
        x[bad[::2], 0] = 1e200
        x[bad[1::2], rng.integers(0, d)] = np.nan
    return x


def _load_segments(h, segs, d):
    import torch
    cap = max(s.shape[0] for s in segs)
    h.seg_reset()
    h.seg_reserve(len(segs), cap, d)
    cap = h.seg_cap()  # a store that already had room keeps its layout
    for e, x in enumerate(segs):
        L = x.shape[0]
        # one iteration with I = 1 appends u_cur[0:L] as x rows (N = L)
        u = torch.zeros((L + 1, d), dtype=torch.float64, device='cuda')
        u[:L] = torch.from_numpy(x)
        y = torch.zeros_like(u)
        h.seg_append_iteration([e], [1], u, y, y, (L + 1) * d, L, d)
        assert h.seg_rows(e) == L
    return cap


def _r2_host(xs):
    """[m, m] squared distances, strict left-to-right sums (the cdist arithmetic of gp_prep_kernel)"""
    acc = np.zeros((xs.shape[0], xs.shape[0]))
    with np.errstate(over='ignore', invalid='ignore'):  # the +inf / NaN rows
        for j in range(xs.shape[1]):
            diff = xs[:, None, j] - xs[None, :, j]
            acc = acc + diff * diff
    return acc


@pytest.mark.parametrize("m", [1, 11, 32, 33, 160])
@pytest.mark.parametrize("big", [False, True])
def test_segmented_knn_equals_knn_on_each_segment(seg_handle, ref_handle, m, big):
    import torch
    d = 4
    rng = np.random.default_rng(100 * m + big)
    lengths = sorted({m, max(m, 7), 16 * m - 1, 16 * m} | ({8192, 8193} if big else {8192 if m <= 32 else 600}))
    segs = [_segment(rng, L, d, e % 3) for e, L in enumerate(lengths)]
    cap = _load_segments(seg_handle, segs, d)
    for nq in (1, 5, 64, 300):
        owner = np.arange(nq) % len(segs)
        Q = np.stack([segs[o][rng.integers(segs[o].shape[0])] + (0 if q % 2 else 1e-3 * rng.standard_normal(d))
                      for q, o in enumerate(owner)])
        ld = d + 3  # strided queries
        Qd = torch.zeros((nq, ld), dtype=torch.float64, device='cuda')
        Qd[:, :d] = torch.from_numpy(Q)
        idx = torch.empty((nq, m), dtype=torch.int64, device='cuda')
        dist = torch.empty((nq, m), dtype=torch.float64, device='cuda')
        r2 = torch.empty((nq, m, m), dtype=torch.float64, device='cuda')
        base = owner * cap
        rows = np.array([segs[o].shape[0] for o in owner])
        tile = m <= 32 and rows.max() <= 8192  # the route follows the longest segment searched
        c0 = seg_handle.launch_count()
        seg_handle.knn_segmented(Qd, ld, nq, m, base, rows, idx, dist, r2)
        nl = seg_handle.launch_count() - c0
        if tile:
            assert nl == 1, (nq, nl)
        else:
            assert nl >= 4, (nq, nl)  # distances, selection (one or two levels), base offset, neighbour matrix
        idx, dist, r2 = idx.cpu().numpy(), dist.cpu().numpy(), r2.cpu().numpy()
        for e, x in enumerate(segs):
            qs = np.nonzero(owner == e)[0]
            if qs.size == 0:
                continue
            ref_handle.dataset_reset()
            ref_handle.dataset_reserve(x.shape[0], d)
            ref_handle.dataset_append_host(x, np.zeros_like(x))
            ri, rd = ref_handle.knn_host(Q[qs], m)
            assert np.array_equal(idx[qs] - e * cap, ri), (nq, e, m)
            assert np.array_equal(dist[qs], rd, equal_nan=True), (nq, e, m)
            for q in qs[:3]:
                assert np.array_equal(r2[q], _r2_host(x[idx[q] - e * cap]), equal_nan=True), (nq, e, q)


# ---------------------------------------------------------------------------------------------------------------------
# B. members equal their solo runs
# ---------------------------------------------------------------------------------------------------------------------
def _setup(name, n_restarts=None):
    z, cfg, mkw = load_run(name)
    key, kw = case_system(name)
    mkw = dict(mkw)
    if n_restarts is not None:
        mkw['n_restarts'] = n_restarts
    mkw.pop('seed', None)
    return cfg, float(z["epsilon"]), key, kw, mkw


def _solver(ode, cfg):
    return nn.CudaSolverRK(ode.get_vector_field(), **{k: cfg[k] for k in ("Ng", "Nf", "F", "G")})


def _solo(key, kw, cfg, eps, mkw, seed, init_cond=None, early_stop=None, max_rows=None):
    ode = device_system(key, **kw)
    if init_cond is not None:
        ode.set_default_init_cond(init_cond)
    p = nn.PararealDevice(ode, _solver(ode, cfg), tspan=cfg["tspan"], N=cfg["N"], epsilon=eps, verbose='')
    return p.run(model='nngp', seed=seed, early_stop=early_stop, max_rows=max_rows, **mkw)


def _ensemble(key, kw, cfg, eps, mkw, seeds, **run_kw):
    ode = device_system(key, **kw)
    ens = nn.PararealEnsemble(ode, _solver(ode, cfg), tspan=cfg["tspan"], N=cfg["N"], epsilon=eps, verbose='')
    return ens.run(model='nngp', seeds=seeds, **mkw, **run_kw)


def _same(a, b, label=""):
    assert a['k'] == b['k'], (label, a['k'], b['k'])
    assert a['conv_int'] == b['conv_int'], (label, a['conv_int'], b['conv_int'])
    assert a['converged'] == b['converged'], label
    assert a['n_rows'] == b['n_rows'], (label, a['n_rows'], b['n_rows'])
    assert np.array_equal(a['u'], b['u']), label
    assert np.array_equal(a['err'], b['err'], equal_nan=True), label


@pytest.mark.parametrize("name,seeds,n_restarts,nn_override", [
    ("lorenz_N50_m11", list(range(45, 53)), None, None),
    ("hopf_N32_m15", [45, 46, 47, 48, 49], 2, None),
    ("fhn_d32_N32_m12", [45, 46, 47], None, None),
    ("burgers_d32_N32_m12", [45, 46, 47], None, None),
    ("lorenz_N50_m11", [45, 46], None, 40),   # m > 32: segmented distance + selection kernels, the big fit
    ("lorenz_N50_m11", [47], None, None),     # E = 1
])
def test_members_equal_solo_runs(name, seeds, n_restarts, nn_override):
    cfg, eps, key, kw, mkw = _setup(name, n_restarts)
    if nn_override is not None:
        mkw['nn'] = nn_override
    outs = _ensemble(key, kw, cfg, eps, mkw, seeds)
    assert len(outs) == len(seeds)
    for s, o in zip(seeds, outs):
        _same(o, _solo(key, kw, cfg, eps, mkw, s), (name, s))


def test_members_that_stop_at_different_iterations():
    """members differ in epsilon, early_stop and initial condition: they leave the ensemble at different iterations"""
    cfg, eps, key, kw, mkw = _setup("lorenz_N50_m11")
    seeds = [45, 46, 47, 48]
    epsilons = [eps, 1e-3, eps, 5e-6]
    stops = [None, None, 3, None]
    ics = [None, [-14.0, -15.0, 21.0], None, [-15.5, -14.0, 19.0]]
    ode = device_system(key, **kw)
    ens = nn.PararealEnsemble(ode, _solver(ode, cfg), tspan=cfg["tspan"], N=cfg["N"], epsilon=eps, verbose='')
    h = ens.handle()
    sweep, launches = h.ensemble_sweep, []

    def counted_sweep(*args):
        c0 = h.launch_count()
        sweep(*args)
        launches.append(h.launch_count() - c0)

    h.ensemble_sweep = counted_sweep
    outs = ens.run(model='nngp', seeds=seeds, epsilons=epsilons, early_stops=stops, init_conds=ics, **mkw)
    # the first sweep, all four members at I = 1: the time table, then per slice the queue order, the coarse step,
    # the segmented kNN and the grouped fit (searches, then selection and mean)
    assert launches[0] == 1 + 5 * (cfg["N"] - 1), launches
    ks = set()
    for e, s in enumerate(seeds):
        ref = _solo(key, kw, cfg, epsilons[e], mkw, s, init_cond=ics[e], early_stop=stops[e])
        _same(outs[e], ref, s)
        ks.add(outs[e]['k'])
    assert len(ks) >= 3, ks


def test_store_grows():
    """a capacity of one iteration: the segmented store is re-laid out and copied as it grows"""
    cfg, eps, key, kw, mkw = _setup("lorenz_N50_m11")
    seeds = [45, 46, 47]
    outs = _ensemble(key, kw, cfg, eps, mkw, seeds, max_rows=51)
    for s, o in zip(seeds, outs):
        assert o['n_rows'] > 51
        _same(o, _solo(key, kw, cfg, eps, mkw, s, max_rows=51), s)


def test_burgers_published_cell_as_one_ensemble():
    """Burgers_K_vs_m, T = 5, nn = 18: 16 seeds as one ensemble.  K against the published values as
    test_published_K_distribution_without_bias compares them, and three members against their solo runs bitwise."""
    pub = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "published.json")))
    cell = [(seed, K) for T, nnb, seed, K in pub["Burgers_K_vs_m"] if (T, nnb) == (5.0, 18)][:16]
    assert len(cell) == 16
    seeds = [s for s, _ in cell]
    ode = nn.Burgers(d_x=128, normalization='-11')
    solver = nn.CudaSolverRK(ode.get_vector_field(), Ng=4, Nf=2000, G='RK1', F='RK8')
    ens = nn.PararealEnsemble(ode, solver, tspan=[0, 5.0], N=128, epsilon=5e-7, verbose='')
    outs = ens.run(model='nngp', seeds=seeds, nn=18)
    v = np.array([(o['k'] if o['converged'] else 128) - K for o, (_, K) in zip(outs, cell)])
    print(f"Burgers T=5 nn=18, 16 seeds: K_ensemble - K_published histogram {dict(zip(*np.unique(v, return_counts=True)))}")
    assert abs(v.mean()) <= 0.5 and np.mean(np.abs(v) <= 1) >= 0.85, v
    for e in (0, 7, 15):
        ode1 = nn.Burgers(d_x=128, normalization='-11')
        s1 = nn.CudaSolverRK(ode1.get_vector_field(), Ng=4, Nf=2000, G='RK1', F='RK8')
        ref = nn.PararealDevice(ode1, s1, tspan=[0, 5.0], N=128, epsilon=5e-7, verbose='').run(
            model='nngp', nn=18, seed=seeds[e])
        _same(outs[e], ref, seeds[e])
