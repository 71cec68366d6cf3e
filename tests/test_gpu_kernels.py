"""GPU: kernel-level parity of the CUDA path (through the C ABI) against the CPU oracle and the
golden vectors recorded from the reference."""
import os

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib
from oracle import nngp as onn
from oracle import rk as ork
from oracle import systems as osys
from helpers import GOLDEN, load_run, make_dataset, samples, scaled_err

pytestmark = pytest.mark.gpu

BITWISE = ["lorenz", "lorenz_id", "hopf", "rossler", "fhn_ode", "brusselator"]  # closed form, no libm calls
TOLERANT = {"dblpend": 1e-14, "thomas": 1e-14, "burgers128": 1e-11, "burgers32": 1e-11, "fhn16": 1e-11,
            "fhn4": 1e-12, "fhn4_n": 1e-12}
DEV = {"lorenz": lambda: nn.Lorenz(normalization='-11'), "lorenz_id": lambda: nn.Lorenz(),
       "hopf": lambda: nn.Hopf(normalization='-11'), "rossler": lambda: nn.Rossler(normalization='-11'),
       "fhn_ode": lambda: nn.FHN_ODE(normalization='-11'), "brusselator": lambda: nn.Brusselator(normalization='-11'),
       "dblpend": lambda: nn.DblPend(normalization='-11'), "thomas": lambda: nn.ThomasLabyrinth(normalization='-11'),
       "burgers128": lambda: nn.Burgers(d_x=128, normalization='-11'),
       "burgers32": lambda: nn.Burgers(d_x=32, normalization='-11'),
       "fhn16": lambda: nn.FHN_PDE(d_x=16), "fhn4": lambda: nn.FHN_PDE(d_x=4),
       "fhn4_n": lambda: nn.FHN_PDE(d_x=4, normalization='-11')}


def relerr(a, b):
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-300)))


@pytest.fixture(scope="module")
def rkv():
    return np.load(os.path.join(GOLDEN, "rk_vectors.npz"))


@pytest.mark.parametrize("name", sorted(DEV))
def test_rk_and_vector_field_vs_reference_vectors(rkv, name):
    """device RHS + RK == reference systems.py/RK.py outputs: bit-exact for the closed-form ODEs,
    1e-11 (scaled) for the stencil form of the dense PDE operators and the libm-dependent fields"""
    ode = DEV[name]()
    f = ode.get_vector_field()
    U = rkv[f"{name}_u"]
    got = f(0.3, U)
    if name in BITWISE:
        assert np.array_equal(got, rkv[f"{name}_f"])
    else:
        assert scaled_err(got, rkv[f"{name}_f"]) < TOLERANT[name]
    assert np.array_equal(f(0.0, U[1]), got[1])  # single vector call, t ignored (autonomous)
    for method in ("RK1", "RK2", "RK4", "RK8"):
        t0, t1, steps = rkv[f"{name}_{method}_t"]
        s = nn.CudaSolverRK(f, Ng=int(steps), Nf=int(steps), F=method, G=method)
        got = s.run_F_batch([t0] * 3, [t1] * 3, U[:3])
        want = rkv[f"{name}_{method}_u1"]
        if name in BITWISE:
            assert np.array_equal(got, want), method
        else:
            assert scaled_err(got, want) < TOLERANT[name], method
        assert np.array_equal(s.run_G(t0, t1, U[2]), got[2])  # one-slice call == batched call


def test_rk_many_slices_both_step_conventions_vs_oracle():
    rng = np.random.default_rng(5)
    o = osys.Lorenz(normalization='-11')
    ode = nn.Lorenz(normalization='-11')
    n = 70  # more than two warps of slices, ragged last block
    u0 = o.u0[None, :] + 0.05 * rng.standard_normal((n, 3))
    t0 = np.linspace(0, 3, n)
    t1 = t0 + rng.uniform(0.05, 0.3, n)
    for h_mode in ("linspace", "const"):
        s = nn.CudaSolverRK(ode.get_vector_field(), Ng=3, Nf=37, F='RK8', G='RK4', h_mode=h_mode)
        got = s.run_F_batch(t0, t1, u0)
        want = np.stack([ork.rk_last(o.f, 'RK8', t0[i], t1[i], 37, u0[i], h_mode) for i in range(n)])
        assert np.array_equal(got, want), h_mode
    o2, d2 = osys.FHN_PDE(d_x=6), nn.FHN_PDE(d_x=6)
    u0 = o2.u0[None, :] + 0.01 * rng.standard_normal((9, 72))
    s = nn.CudaSolverRK(d2.get_vector_field(), Ng=5, Nf=20, F='RK8', G='RK2')
    got = s.run_F_batch(np.arange(9.0), np.arange(9.0) + 2.0, u0)
    want = np.stack([ork.rk_last(o2.f, 'RK8', float(i), i + 2.0, 20, u0[i]) for i in range(9)])
    assert scaled_err(got, want) < 1e-12
    got = s.run_G_batch(np.arange(9.0), np.arange(9.0) + 2.0, u0)
    want = np.stack([ork.rk_last(o2.f, 'RK2', float(i), i + 2.0, 5, u0[i]) for i in range(9)])
    assert scaled_err(got, want) < 1e-12
    # paging quirk of solver.py:89-96 (steps > thresh): every page runs with the total step count
    sp = nn.CudaSolverRK(ode.get_vector_field(), Ng=3, Nf=25, F='RK4', G='RK4', thresh=10)
    u = o.u0.copy()
    st = 24
    step = (0.5 - 0.0) / st
    ta = 0.0
    for page in (10, 10, 4):
        tb = ta + step * page
        u = ork.rk_last(o.f, 'RK4', ta, tb, st, u)
        ta = tb
    assert np.array_equal(sp.run_F(0.0, 0.5, o.u0), u)


@pytest.mark.parametrize("d_x", [4, 6, 16, 18])
def test_fhn_tile_kernel_equals_point_kernel_bitwise(d_x):
    """the 2x2-points-per-thread FHN kernel (csrc/rk.cu rk_fhn_tile_kernel) returns the bits of the
    one-point-per-thread kernel and of the 1x2 variant (NNGP_RK_TILE forces each), all RK methods, and all agree with
    the NumPy oracle to 1e-12 scaled"""
    import os
    rng = np.random.default_rng(d_x)
    o, ode = osys.FHN_PDE(d_x=d_x), nn.FHN_PDE(d_x=d_x)
    n = 7
    u0 = o.u0[None, :] + 0.01 * rng.standard_normal((n, 2 * d_x * d_x))
    t0 = np.arange(n) * 0.5
    t1 = t0 + 0.7
    for F, steps in (('RK8', 23), ('RK4', 11), ('RK2', 6), ('RK1', 5)):
        s = nn.CudaSolverRK(ode.get_vector_field(), Ng=3, Nf=steps, F=F, G='RK4')
        try:
            os.environ["NNGP_RK_TILE"] = "1"   # 2x2 blocks per thread
            got = s.run_F_batch(t0, t1, u0)
            os.environ["NNGP_RK_TILE"] = "2"   # 1x2 blocks per thread
            got2 = s.run_F_batch(t0, t1, u0)
            os.environ["NNGP_RK_TILE"] = "0"   # one point per thread
            ref = s.run_F_batch(t0, t1, u0)
        finally:
            del os.environ["NNGP_RK_TILE"]
        assert np.array_equal(got, ref) and np.array_equal(got2, ref), F
        want = np.stack([ork.rk_last(o.f, F, t0[i], t1[i], steps, u0[i]) for i in range(n)])
        assert scaled_err(got, want) < 1e-12, F


def test_fhn_time_chunked_fine_step_equals_single_launch_bitwise():
    """more than two slices per SM and a long step range: the fine step is executed as a sequence of balanced
    launches over (chunk of steps, slice) tasks (csrc/rk.cu launch_fhn_tile_s); NNGP_RK_CHUNKS=0 forces the single
    launch.  Same bits, both step-size conventions, slice count not a multiple of the launch size."""
    import os
    rng = np.random.default_rng(11)
    ode = nn.FHN_PDE(d_x=4)
    n = 333
    u0 = ode.get_init_cond()[None, :] + 0.01 * rng.standard_normal((n, 32))
    t0 = rng.uniform(0, 1, n)
    t1 = t0 + rng.uniform(0.5, 1.5, n)
    for h_mode in ("linspace", "const"):
        s = nn.CudaSolverRK(ode.get_vector_field(), Ng=3, Nf=4999, F='RK8', G='RK4', h_mode=h_mode)
        got = s.run_F_batch(t0, t1, u0)
        try:
            os.environ["NNGP_RK_CHUNKS"] = "0"
            ref = s.run_F_batch(t0, t1, u0)
        finally:
            del os.environ["NNGP_RK_CHUNKS"]
        assert np.all(np.isfinite(got)) and np.array_equal(got, ref), h_mode


@pytest.mark.parametrize("name", ["lorenz", "hopf", "burgers32", "fhn4", "fhn6"])
def test_rk_full_trajectory_vs_reference_vectors(name):
    """CudaSolverRK.run_F_full / run_G_full (solver.py:109-113): every step of the solve against the trajectories
    recorded from the reference's RK.run -- bit-exact for the closed-form systems, 1e-11 scaled for the PDE stencils;
    the last row is the bits of run_F"""
    z = np.load(os.path.join(GOLDEN, "rk_full_vectors.npz"))
    mk = {"lorenz": lambda: nn.Lorenz(normalization='-11'), "hopf": lambda: nn.Hopf(normalization='-11'),
          "burgers32": lambda: nn.Burgers(d_x=32, normalization='-11'), "fhn4": lambda: nn.FHN_PDE(d_x=4),
          "fhn6": lambda: nn.FHN_PDE(d_x=6)}[name]
    ode = mk()
    u0 = z[f"{name}_u0"]
    for method in ("RK1", "RK4", "RK8"):
        t0, t1, steps = z[f"{name}_{method}_t"]
        s = nn.CudaSolverRK(ode.get_vector_field(), Ng=int(steps), Nf=int(steps), F=method, G=method)
        got = s.run_F_full(t0, t1, u0)
        want = z[f"{name}_{method}_traj"]
        assert got.shape == want.shape
        if name in ("lorenz", "hopf"):
            assert np.array_equal(got, want), method
        else:
            assert scaled_err(got, want) < 1e-11, method
        assert np.array_equal(got[0], u0) and np.array_equal(got[-1], s.run_F(t0, t1, u0))
        assert np.array_equal(s.run_G_full(t0, t1, u0), got)


def test_rk_errors(handle):
    ode = nn.Burgers(d_x=2000, normalization='-11')
    s = nn.CudaSolverRK(ode.get_vector_field(), Ng=1, Nf=1, F='RK4', G='RK1')
    with pytest.raises(_lib.NNGPError, match="outside"):
        s.run_G(0.0, 1.0, ode.get_init_cond())
    ode = nn.Lorenz()
    s = nn.CudaSolverRK(ode.get_vector_field(), Ng=0, Nf=1, F='RK4', G='RK1')
    with pytest.raises(_lib.NNGPError, match="steps must be >= 1"):
        s.run_G(0.0, 1.0, ode.get_init_cond())


def test_device_exp_and_rsqrt_accuracy(handle):
    """the hand-written exp(x<=0) and 1/p inside the GP kernels: within 1 ulp of correct rounding"""
    import torch
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(0, 750, 20000), 10.0 ** rng.uniform(-300, 2.8, 20000), [0.0, 708.38, 708.4, 745.0, 1e-320]])
    dev = torch.device('cuda', handle.device)
    tx = torch.from_numpy(x).to(dev)
    te, tr = torch.empty_like(tx), torch.empty_like(tx)
    handle.selftest_math(tx, x.size, te, tr)
    ge, gr = te.cpu().numpy(), tr.cpu().numpy()
    want_e = np.exp(-x)
    big = x <= 708.39
    ulp = np.spacing(want_e[big])
    assert np.max(np.abs(ge[big] - want_e[big]) / ulp) <= 1.0
    assert np.all(ge[~big] == 0.0) and ge[x == 0.0][0] == 1.0
    pos = (x > 1e-300) & (x < 1e300)
    with np.errstate(all="ignore"):
        want_r = 1.0 / x[pos]
    assert np.max(np.abs(gr[pos] - want_r) / np.spacing(want_r)) <= 1.5
    nan = torch.tensor([float('nan')], dtype=torch.float64, device=dev)
    handle.selftest_math(nan, 1, te, tr)
    assert np.isnan(te.cpu().numpy()[0])
    # 10**x of the hyper-parameter transforms (models.py:145-148): within 2 ulp of numpy's pow on the range a
    # search can reach, library behaviour (inf / 0 / NaN) outside
    xs = np.concatenate([rng.uniform(-300, 300, 40000), rng.uniform(-12, 4, 20000), np.arange(-20.0, 3.0),
                         [-400.0, 400.0, 308.2, -323.0, np.nan]])
    tx = torch.from_numpy(xs).to(dev)
    te, tr = torch.empty_like(tx), torch.empty_like(tx)
    t10 = torch.empty(2 * xs.size, dtype=torch.float64, device=dev)  # [10**x | log|x| + 3 ln 2]
    handle.selftest_math(tx, xs.size, te, tr, t10)
    g10 = t10.cpu().numpy()[:xs.size]
    with np.errstate(all="ignore"):
        want10 = 10.0 ** xs
    fin = np.isfinite(want10) & (want10 > 1e-300)
    assert np.max(np.abs(g10[fin] - want10[fin]) / np.spacing(want10[fin])) <= 2.0
    assert g10[xs == 400.0][0] == np.inf and g10[xs == -400.0][0] == 0.0 and np.isnan(g10[-1])
    # log of the determinant accumulator: log(x) + k ln2 within 1 ulp
    xl = np.concatenate([rng.uniform(1.0, 2.0 ** 21, 20000), 10.0 ** rng.uniform(-300, 300, 20000), [1.0, 2.0, np.sqrt(2)]])
    tx = torch.from_numpy(xl).to(dev)
    te, tr = torch.empty_like(tx), torch.empty_like(tx)
    t10 = torch.empty(2 * xl.size, dtype=torch.float64, device=dev)
    handle.selftest_math(tx, xl.size, te, tr, t10)
    gl = t10.cpu().numpy()[xl.size:]
    from decimal import Decimal, getcontext
    getcontext().prec = 40
    ln2 = Decimal(2).ln()
    sub = rng.permutation(xl.size)[:3000]
    wantl = np.array([float(Decimal(float(v)).ln() + 3 * ln2) for v in xl[sub]])
    assert np.max(np.abs(gl[sub] - wantl) / np.spacing(np.abs(wantl))) <= 1.0


@pytest.mark.parametrize("n,d,m,nq", [(40, 3, 11, 1), (300, 3, 11, 5), (2000, 32, 12, 9), (3055, 512, 20, 1),
                                       (3055, 512, 20, 12), (5000, 128, 30, 33), (65, 7, 32, 3), (20, 2, 20, 2),
                                       (700, 1100, 5, 6), (20000, 8, 32, 2), (8193, 3, 20, 40), (4097, 5, 17, 1)])
def test_knn_bit_exact(handle, n, d, m, nq):
    """index sets AND squared distances bit-identical to argsort(cdist(q, x, 'sqeuclidean'))[:m]"""
    rng = np.random.default_rng(n + d)
    x, y = make_dataset(rng, n, d)
    Q = x[rng.permutation(n)[:nq]] + 1e-3 * rng.standard_normal((nq, d))
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x[:n // 2], y[:n // 2])
    handle.dataset_append_host(x[n // 2:], y[n // 2:])  # appended in two pieces like two iterations
    assert handle.dataset_rows() == n
    idx, dist = handle.knn_host(Q, m)
    for qi in range(nq):
        oi, od = onn.knn(Q[qi], x, m)
        assert np.array_equal(idx[qi], oi) and np.array_equal(dist[qi], od)
    if n > 2 * m:  # prefix search: only the first rows (what a predict at an earlier iteration sees)
        idx, dist = handle.knn_host(Q[:1], m, n_rows=n // 2)
        oi, od = onn.knn(Q[0], x[:n // 2], m)
        assert np.array_equal(idx[0], oi) and np.array_equal(dist[0], od)


def test_knn_ties_broken_by_index_and_edge_cases(handle):
    rng = np.random.default_rng(2)
    base = rng.standard_normal((30, 4))
    x = np.concatenate([base, base, base[:10]])  # exact duplicates -> exact distance ties
    y = np.zeros_like(x)
    handle.dataset_reset()
    handle.dataset_reserve(200, 4)
    handle.dataset_append_host(x, y)
    q = base[3] + 1e-4
    idx, dist = handle.knn_host(q[None], 9)
    oi, od = onn.knn(q, x, 9)
    assert np.array_equal(idx[0], oi) and np.array_equal(dist[0], od)
    assert list(idx[0][:3]) == [3, 33, 63]  # same distance, ascending index
    # exact ties across the 256-row CTAs of the one-query scan (nq = 1) and across the 1024-row chunks of the two-level
    # selection (nq = 5): still ascending index.  Only every 8th copy of row 3 is kept, so the 25 tied nearest rows
    # reach past row 4096.
    big = np.tile(base, (300, 1))  # 9000 rows, every row repeated 300 times
    big[np.arange(3, 9000, 30)[np.arange(300) % 8 != 0]] = base[0]
    handle.dataset_reset()
    handle.dataset_reserve(9000, 4)
    handle.dataset_append_host(big, np.zeros_like(big))
    oi, od = onn.knn(q, big, 25)
    for nq, launches in ((1, 1), (5, 3)):
        c0 = handle.launch_count()
        idx, dist = handle.knn_host(np.repeat(q[None], nq, axis=0), 25)
        assert handle.launch_count() - c0 == launches, nq  # scan_select_kernel / sqdist + two select_kernel levels
        for qi in range(nq):
            assert np.array_equal(idx[qi], oi) and np.array_equal(dist[qi], od)
        assert list(idx[0][:4]) == [3, 243, 483, 723] and idx[0].max() > 4096  # same distance, ascending index
    handle.dataset_reset()
    handle.dataset_reserve(200, 4)
    handle.dataset_append_host(x, y)
    # query equal to a dataset row: distance exactly 0 first
    idx, dist = handle.knn_host(base[5][None], 3)
    assert dist[0, 0] == 0.0 and idx[0, 0] == 5
    with pytest.raises(_lib.NNGPError, match="outside"):
        handle.knn_host(q[None], 161)
    with pytest.raises(_lib.NNGPError, match="fewer than m"):
        handle.knn_host(q[None], 9, n_rows=5)
    handle.dataset_reset()
    assert handle.dataset_rows() == 0
    with pytest.raises(_lib.NNGPError):
        handle.knn_host(q[None], 3)


def _gp_problem(handle, rng, n, d, m, nq, near=1e-3):
    import torch
    x, y = make_dataset(rng, n, d)
    Q = x[rng.permutation(n)[:nq]] + near * rng.standard_normal((nq, d))
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    idx, dist = handle.knn_host(Q, m)
    dev = torch.device('cuda', handle.device)
    return x, y, Q, idx, dist, dev


@pytest.mark.parametrize("n,d,m", [(300, 3, 11), (500, 6, 5), (800, 16, 20), (400, 8, 30), (900, 4, 17)])
def test_objective_parity(handle, n, d, m):
    """nll(theta) == models.py:240-252 within 1e-9 relative on well-conditioned points, and +inf exactly
    where the reference returns inf (failed factorisation / NaN)"""
    import torch
    rng = np.random.default_rng(7 + m)
    nq, nt = 3, 40
    x, y, Q, idx, dist, dev = _gp_problem(handle, rng, n, d, m, nq)
    theta = np.stack([rng.uniform(-9, 2, (nq, d, nt)), rng.uniform(-9, 0, (nq, d, nt))], axis=-1)
    theta[:, :, 0] = [-400.0, -3.0]   # 10**sx underflows -> 1/0 = inf -> NaN -> +inf
    theta[:, :, 1] = [4.0, -2.0]      # huge length scale: singular kernel matrix
    theta[:, :, 2] = [-3.0, 400.0]    # amplitude overflows
    jit = rng.integers(-20, -11, (nq, d, nt)).astype(float)
    t_idx = torch.from_numpy(idx).to(dev)
    t_th = torch.from_numpy(theta).to(dev)
    t_j10 = torch.from_numpy(10.0 ** 0 * np.array([[[10 ** j for j in row] for row in blk] for blk in jit])).to(dev)
    out = torch.empty((nq, d, nt), dtype=torch.float64, device=dev)
    handle.gp_nll(t_idx, nq, m, nt, t_th, t_j10, out)
    got = out.cpu().numpy()
    n_inf = n_cmp = 0
    for qi in range(nq):
        r2 = onn.pairwise_sqdist(x[idx[qi]], x[idx[qi]])
        for j in range(d):
            yy = y[idx[qi], j]
            for t in range(nt):
                want = onn.neg_log_lik(r2, yy, theta[qi, j, t], jit[qi, j, t])
                g = got[qi, j, t]
                if not np.isfinite(want):
                    n_inf += 1
                    # a singular matrix may fail in one factorisation and squeak through in the other
                    assert np.isinf(g) or t == 1, (theta[qi, j, t], want, g)
                    continue
                K = onn.se_kernel_from_r2(r2, theta[qi, j, t]) + np.eye(m) * 10 ** jit[qi, j, t]
                cond = np.linalg.cond(K)
                if cond < 1e6:
                    n_cmp += 1
                    assert abs(g - want) <= 1e-9 * max(1.0, abs(want)), (theta[qi, j, t], cond, want, g)
    assert n_inf >= 2 * nq * d and n_cmp > nq * d * 5


@pytest.mark.parametrize("n,d,m", [(300, 3, 11), (800, 16, 20), (400, 8, 30), (600, 5, 13)])
def test_prediction_given_identical_hyperparameters(handle, n, d, m):
    """north_star: GP predictions within 1e-8 relative given identical hyper-parameters"""
    import torch
    rng = np.random.default_rng(11 + m)
    nq = 4
    x, y, Q, idx, dist, dev = _gp_problem(handle, rng, n, d, m, nq)
    theta = np.stack([rng.uniform(-2.5, 0.5, (nq, d)), rng.uniform(-8, -1, (nq, d))], axis=-1)
    jit = rng.integers(-20, -11, (nq, d)).astype(float)
    pred = torch.empty((nq, d), dtype=torch.float64, device=dev)
    handle.gp_mean(torch.from_numpy(Q).to(dev), torch.from_numpy(idx).to(dev), torch.from_numpy(dist).to(dev),
                   nq, m, torch.from_numpy(theta).to(dev), torch.from_numpy(jit).to(dev), pred)
    got = pred.cpu().numpy()
    worst = 0.0
    for qi in range(nq):
        r2 = onn.pairwise_sqdist(x[idx[qi]], x[idx[qi]])
        for j in range(d):
            want = onn.posterior_mean(r2, dist[qi], y[idx[qi], j], theta[qi, j], jit[qi, j])
            K = onn.se_kernel_from_r2(r2, theta[qi, j]) + np.eye(m) * 10 ** jit[qi, j]
            if np.linalg.cond(K) < 1e7:
                worst = max(worst, abs(got[qi, j] - want) / abs(want))
    assert worst < 1e-8, worst


@pytest.mark.parametrize("n,d,m,R", [(300, 3, 11, 1), (600, 6, 15, 2), (800, 12, 20, 1), (300, 4, 30, 1)])
def test_fit_predict_vs_oracle(handle, n, d, m, R):
    """full predict (kNN + 9R Nelder-Mead fits per dimension + selection + mean) against the oracle on
    the same host-drawn starts.  A search leaves SciPy's trajectory at the first comparison of two objective values
    that agree to the last ulp or two (the device's LDL^T objective and LAPACK's differ there; so do two LAPACK
    builds): measured on the B200, 53-82 % of the searches follow it to the end (m = 20: 53 %, m = 11: 82 %) and the
    selected optimum agrees to 1e-6 in 83-100 % of the dimensions.  The bars below sit just under those figures; what
    is exact is asserted exactly (neighbours, the selection rule on the device's own values, the posterior mean at
    the device's hyper-parameters)."""
    rng = np.random.default_rng(100 + m)
    x, y = make_dataset(rng, n, d)
    q = x[3] + 1e-3 * rng.standard_normal(d)
    model = nn.CudaNNGP(n=d, N=4, nn=m, seed=45, n_restarts=R, handle=handle)
    model.fit(x, y, k=0)
    state = model.rng.bit_generator.state
    pred, det = model.predict(q.reshape(1, -1), None, None, i=0, return_details=True)
    orng = np.random.default_rng()
    orng.bit_generator.state = state
    starts = onn.draw_starts(orng, d, R)
    opred, odet = onn.predict(q, x, y, m, starts, return_details=True)
    assert np.array_equal(det['idx'][0], odet['idx'])
    same = 0
    for j in range(d):
        for a in range(9):
            for r in range(R):
                same += bool(np.array_equal(det['thetas'][0, j, a, r], odet['thetas'][j, a, r])
                             and det['nfev'][0, j, a, r] == odet['nfev'][j, a, r])
    frac = same / (d * 9 * R)
    assert frac > 0.5, f"only {frac:.2f} of the Nelder-Mead runs follow the SciPy trajectory exactly"
    # every run ends at (numerically) the same objective value as the reference search or better/equal basin
    finite = np.isfinite(odet['fvals']) & np.isfinite(det['fvals'][0])
    assert np.median(np.abs(det['fvals'][0][finite] - odet['fvals'][finite])) < 1e-6
    # the device's own selection is the reference rule applied to its own fvals
    for j in range(d):
        best = onn.select(det['fvals'][0, j])
        a, r = divmod(best, R)
        assert det['jitter_opt'][0, j] == -20 + a
        assert np.array_equal(det['theta_opt'][0, j], det['thetas'][0, j, a, r])
        assert det['fval_opt'][0, j] == det['fvals'][0, j, a, r]
        want = onn.posterior_mean(odet['r2'], odet['dist'], y[odet['idx'], j], det['theta_opt'][0, j], det['jitter_opt'][0, j])
        assert abs(pred[j] - want) <= 1e-8 * abs(want) + 1e-16
    assert np.all(det['nfev'] >= 3) and np.all(det['nfev'] <= 400)
    # the selected optimum is as good as the reference's in (almost) every dimension: a search that
    # diverges from the SciPy trajectory at a last-bit tie may end in another local optimum
    close = np.abs(det['fval_opt'][0] - odet['fval_opt']) <= 1e-6 * np.maximum(1.0, np.abs(odet['fval_opt']))
    print(f"fit_predict n={n} d={d} m={m} R={R}: SciPy trajectory followed exactly by {frac:.3f} of the searches, "
          f"selected optimum within 1e-6 in {close.mean():.3f} of the dimensions")
    assert close.mean() >= 0.8, (det['fval_opt'][0], odet['fval_opt'])
    assert np.all(det['fval_opt'][0] <= odet['fval_opt'] + 0.2 * np.abs(odet['fval_opt']))


def test_all_inf_searches_steady_state_neighbours(handle):
    """identical neighbour rows (the FHN target reaches a steady state): the kernel matrix is exactly singular
    for amplitudes above jitter / 4 ulp, every vertex of such a search is +inf, SciPy's fatol test sees
    |inf - inf| = NaN and the search runs all maxfev = 400 evaluations and returns its start point.  The device
    pre-decides the four points of such an iteration at once (gp_head in four lanes): results must be the bits
    of the one-by-one evaluation (NNGP_FIT_NO_HEAD_BATCH) and show the 400-evaluation pattern."""
    import os
    rng = np.random.default_rng(5)
    n, d, m = 64, 6, 20
    x = np.tile(rng.uniform(-1, 1, (1, d)), (n, 1))
    x[:8] += 1e-3 * rng.standard_normal((8, d))       # a few distinct rows far away
    y = 1e-4 * rng.standard_normal((n, d))
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    q = x[20:21] + 0.0
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    got = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
    try:
        os.environ["NNGP_FIT_NO_HEAD_BATCH"] = "1"
        ref = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
    finally:
        del os.environ["NNGP_FIT_NO_HEAD_BATCH"]
    for key in ("nfev", "thetas", "fvals", "theta_opt", "fval_opt", "jitter_opt"):
        assert np.array_equal(got[key], ref[key], equal_nan=True), key
    assert np.array_equal(got["pred"], ref["pred"], equal_nan=True)
    inf_runs = np.isinf(got["fvals"][0])
    assert inf_runs.sum() >= 5, "the case must contain searches that see +inf everywhere"
    assert np.all(got["nfev"][0][inf_runs] == 400)
    assert np.array_equal(got["thetas"][0][inf_runs], starts[0][inf_runs].astype(float))
    assert np.all(got["nfev"][0][~inf_runs] < 400)


def test_predict_is_repeatable_after_other_workspace_users(handle):
    """the fit kernel leaves its completion counters zero for the next launch; anything else that uses the
    handle's workspace in between (micro-benchmarks, a large kNN) must not leave them dirty"""
    rng = np.random.default_rng(3)
    n, d, m = 900, 64, 20
    x, y = make_dataset(rng, n, d)
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    q = x[5:6] + 1e-3
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    first = handle.predict_host(q, m, starts, 1, 0.1, 0.1)["pred"]
    handle.bench_fp64(200)
    handle.knn_host(x[:64] + 1e-3, m)
    again = handle.predict_host(q, m, starts, 1, 0.1, 0.1)["pred"]
    assert np.all(np.isfinite(first)) and np.array_equal(first, again)


@pytest.mark.parametrize("name", ["lorenz_N50_m11", "hopf_N32_m15", "burgers_d32_N32_m12", "fhn_d32_N32_m12"])
def test_predict_on_reference_run_samples(handle, name):
    """device predict on (query, dataset prefix, starts) recorded inside a run of the unmodified
    reference.  The neighbour sets are the reference's.  The reference's selection among its 9R
    searches is decided by the last bits of fval whenever several searches end in the same flat valley
    of the likelihood (DESIGN.md, "ties"), so the check is: the device finds an optimum as good as the
    reference's, and its prediction is the reference's posterior mean at the device's hyper-parameters."""
    z, cfg, mkw = load_run(name)
    x, D = z["x"], z["D"]
    d = x.shape[1]
    handle.dataset_reset()
    handle.dataset_reserve(x.shape[0], d)
    handle.dataset_append_host(x, D)
    as_good = total = same_pred = 0
    for s in samples(z)[:4 if d > 8 else 8]:
        n = int(s["n_rows"])
        m = int(s["m"])
        R = s["starts"].shape[2]
        out = handle.predict_host(s["query"][None], m, s["starts"][None], R, 0.1, 0.1, n_rows=n, details=True)
        oi, okq = onn.knn(s["query"], x[:n], m)
        assert np.array_equal(out["idx"][0], oi)
        r2 = onn.pairwise_sqdist(x[oi], x[oi])
        dims = range(d) if d <= 8 else range(0, d, 5)
        for j in dims:
            yj = D[oi, j]
            ref_f = min(onn.nm_run(r2, yj, s["starts"][j, a, r].astype(float), onn.JITTERS[a], 0.1, 0.1)[1]
                        for a in range(9) for r in range(R))
            g_f = out["fval_opt"][0, j]
            total += 1
            as_good += bool(g_f <= ref_f + 1e-8 * max(1.0, abs(ref_f)))
            want = onn.posterior_mean(r2, okq, yj, out["theta_opt"][0, j], out["jitter_opt"][0, j])
            K = onn.se_kernel_from_r2(r2, out["theta_opt"][0, j]) + np.eye(m) * 10 ** out["jitter_opt"][0, j]
            cond = np.linalg.cond(K)
            tol = max(1e-8, 4 * cond * 2.2e-16)  # forward error bound of any backward-stable solve
            assert abs(out["pred"][0, j] - want) <= tol * abs(want) + 1e-14, (j, out["pred"][0, j], want, cond)
            same_pred += bool(abs(out["pred"][0, j] - s["preds"][j]) <= 1e-8 * abs(s["preds"][j]) + 1e-13)
    assert as_good >= 0.9 * total, (as_good, total)
    # measured on the B200 (profiles/r02): 24/24 Lorenz, 19/24 Hopf, 27/28 Burgers, 20/21 FHN recorded predictions
    # reproduced to 1e-8 relative; the rest are selections among equally good searches (previous assert)
    assert same_pred >= 0.75 * total, (same_pred, total)
    print(f"{name}: optimum as good as the reference's in {as_good}/{total}, identical prediction in {same_pred}/{total}")


def test_empty_and_extreme_inputs(handle):
    """edge cases through the C ABI: zero slices / rows / queries are no-ops, m = 1 and m = 32 (the lane limit)
    work, a dataset shorter than m is an error (the reference would silently use fewer neighbours only in
    'adaptive' mode, which the host mirror clamps before calling), d = 1"""
    rng = np.random.default_rng(9)
    ode = nn.Lorenz(normalization='-11')
    s = nn.CudaSolverRK(ode.get_vector_field(), Ng=3, Nf=5, F='RK4', G='RK1')
    assert s.run_F_batch(np.zeros(0), np.zeros(0), np.zeros((0, 3))).shape == (0, 3)
    n, d = 50, 1
    x = rng.uniform(-1, 1, (n, d))
    y = 1e-3 * np.sin(3 * x)
    handle.dataset_reset()
    handle.dataset_reserve(64, d)
    handle.dataset_append_host(x[:0], y[:0])          # zero rows
    assert handle.dataset_rows() == 0
    handle.dataset_append_host(x, y)
    idx, dist = handle.knn_host(np.zeros((0, d)), 5)  # zero queries
    assert idx.shape == (0, 5)
    q = np.array([[0.123]])
    for m in (1, 2, 32):
        starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
        out = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
        oi, okq = onn.knn(q[0], x, m)
        assert np.array_equal(out["idx"][0], oi)
        r2 = onn.pairwise_sqdist(x[oi], x[oi])
        want = onn.posterior_mean(r2, okq, y[oi, 0], out["theta_opt"][0, 0], out["jitter_opt"][0, 0])
        K = onn.se_kernel_from_r2(r2, out["theta_opt"][0, 0]) + np.eye(m) * 10 ** out["jitter_opt"][0, 0]
        cond = np.linalg.cond(K)
        assert np.isfinite(out["pred"][0, 0]), m
        if np.isfinite(want) and cond < 1e12:  # beyond, LAPACK and the device may disagree on whether K factorises
            assert abs(out["pred"][0, 0] - want) <= max(1e-8, 4 * cond * 2.2e-16) * abs(want) + 1e-14, (m, cond)
        assert np.all(out["nfev"] >= 3) and np.all(out["nfev"] <= 400)
    with pytest.raises(_lib.NNGPError, match="fewer than m"):
        handle.knn_host(q, 32, n_rows=20)
    with pytest.raises(_lib.NNGPError, match="outside"):
        handle.predict_host(q, 161, rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8), 1, 0.1, 0.1)


def test_predict_dimension_blocks_equal_full_predict(handle):
    """nngp_predict_host_block: the fits of a predict split by output dimension (a rank's share) give, block by
    block, the bits of the full predict -- predictions and per-search details"""
    rng = np.random.default_rng(21)
    n, d, m = 700, 24, 14
    x, y = make_dataset(rng, n, d)
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    q = x[11:12] + 1e-3
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    full = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
    for world in (2, 3, 8):
        dl = d // world
        for rank in range(world):
            j0 = rank * dl
            part = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True, block=(j0, dl))
            assert np.array_equal(part["idx"], full["idx"])
            for key in ("pred", "theta_opt", "jitter_opt", "fval_opt", "nfev", "fvals", "thetas"):
                assert np.array_equal(part[key][0, j0:j0 + dl], full[key][0, j0:j0 + dl]), (key, world, rank)
    with pytest.raises(_lib.NNGPError, match="outside"):
        handle.predict_host(q, m, starts, 1, 0.1, 0.1, block=(20, 8))
    with pytest.raises(_lib.NNGPError, match="single query"):
        handle.predict_host(np.concatenate([q, q]), m, np.concatenate([starts, starts]), 1, 0.1, 0.1, block=(0, 8))


def _steady_neighbour_sets():
    """neighbour sets of the steady state of an FHN-PDE run (tests/golden/steady_fhn_d32.npz: rows identical to
    ~1e-15), plus variants whose first ndup rows are EXACT duplicates -- the regime of the FHN d=512 target from
    slice ~50 on, where the kernel matrix is singular whenever the jitter is below one ulp of the amplitude"""
    z = np.load(os.path.join(GOLDEN, "steady_fhn_d32.npz"))
    x, y, u = z["x"], z["y"], z["u"]
    m = 20
    sets = []
    for qi, ndup in ((40, 1), (60, 1), (80, 1), (50, 2), (50, 3), (70, 5), (70, 10), (90, 20)):
        idx, _ = onn.knn(u[qi], x, m)
        xm, ym = x[idx].copy(), y[idx].copy()
        for t in range(1, ndup):
            xm[t], ym[t] = xm[0], ym[0]
        sets.append((xm, ym, ndup))
    return sets, m


def test_failure_set_matches_lapack_in_both_directions(handle):
    """The objective is +inf where the factorisation fails (models.py:86-92, 250-251).  On nearly singular
    matrices whether LAPACK's potrf fails is decided by its rounding: a literal potf2 restatement disagrees
    with the installed LAPACK on 1-4 % of such evaluations (oracle/experiments/pivot_rule_study.py), so the set
    cannot be reproduced exactly.  The bar: device-inf-where-reference-finite AND reference-inf-where-device-
    finite are each <= 2 % of the evaluations, neither direction dominates, and outside a band of condition
    numbers around 1/ulp the two sets are identical."""
    import torch
    rng = np.random.default_rng(2)
    sets, m = _steady_neighbour_sets()
    dev = torch.device('cuda', handle.device)
    nt = 120
    tot = dev_only = ref_only = both_inf = 0
    for xm, ym, ndup in sets:
        d = xm.shape[1]
        handle.dataset_reset()
        handle.dataset_reserve(m, d)
        handle.dataset_append_host(xm, ym)
        idx, dist = handle.knn_host(xm[:1], m)
        dims = [0, 5, 17]
        theta = rng.uniform(-8.5, 0.5, (1, d, nt, 2))
        jit = rng.integers(-20, -11, (1, d, nt)).astype(float)
        out = torch.empty((1, d, nt), dtype=torch.float64, device=dev)
        handle.gp_nll(torch.from_numpy(idx).to(dev), 1, m, nt, torch.from_numpy(theta).to(dev),
                      torch.from_numpy(10.0 ** jit).to(dev), out)
        got = out.cpu().numpy()[0]
        r2 = onn.pairwise_sqdist(xm[idx[0]], xm[idx[0]])
        for j in dims:
            for t in range(nt):
                want = onn.neg_log_lik(r2, ym[idx[0], j], theta[0, j, t], jit[0, j, t])
                g = got[j, t]
                tot += 1
                gi, wi = np.isinf(g), np.isinf(want)
                both_inf += bool(gi and wi)
                if gi != wi:
                    dev_only += bool(gi)
                    ref_only += bool(wi)
                    # the disagreements sit where the jitter is within a few ulp of the amplitude
                    amp, jv = 10.0 ** theta[0, j, t, 1], 10.0 ** jit[0, j, t]
                    assert jv < 64 * 2.2e-16 * amp * m, (theta[0, j, t], jit[0, j, t], g, want)
    print(f"failure sets: {tot} evaluations, both +inf {both_inf}, device only {dev_only}, reference only {ref_only}")
    assert both_inf > 0.1 * tot
    assert dev_only <= 0.02 * tot and ref_only <= 0.02 * tot, (dev_only, ref_only, tot)
    assert abs(dev_only - ref_only) <= 0.012 * tot, (dev_only, ref_only, tot)


def test_nelder_mead_vs_oracle_on_steady_state_neighbours(handle):
    """the regime that dominates the FHN target (57 % of its evaluations): searches over steady-state neighbour
    sets, against the ORACLE's Nelder-Mead (SciPy restatement over LAPACK) on the same starts.  Searches that
    see +inf at every vertex must run the full 400 evaluations in both and return their start point; where the
    optimiser trajectories agree they agree bit for bit; the selected optimum is as good as the oracle's and the
    prediction is the oracle's posterior mean at the device's hyper-parameters."""
    rng = np.random.default_rng(8)
    sets, m = _steady_neighbour_sets()
    n_all_inf = n_all_inf_same = n_runs = n_same = n_sel = n_sel_good = 0
    for xm, ym, ndup in sets[::2] + sets[-1:]:
        d = xm.shape[1]
        handle.dataset_reset()
        handle.dataset_reserve(m, d)
        handle.dataset_append_host(xm, ym)
        q = xm[:1] + 0.0
        starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
        out = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
        idx = out["idx"][0]
        r2 = onn.pairwise_sqdist(xm[idx], xm[idx])
        kq = onn.sqdist_rows(q[0], xm[idx])
        for j in (0, 7, 19, 31):
            ofv = np.empty(9)
            for a in range(9):
                th, fv, ne = onn.nm_run(r2, ym[idx, j], starts[0, j, a, 0].astype(float), onn.JITTERS[a], 0.1, 0.1)
                ofv[a] = fv
                n_runs += 1
                g_th, g_fv, g_ne = out["thetas"][0, j, a, 0], out["fvals"][0, j, a, 0], out["nfev"][0, j, a, 0]
                if np.isinf(fv) and ne == 400:
                    n_all_inf += 1
                    n_all_inf_same += bool(np.isinf(g_fv) and g_ne == 400 and np.array_equal(g_th, th))
                n_same += bool(np.array_equal(g_th, th) and g_ne == ne)
            n_sel += 1
            g_f = out["fval_opt"][0, j]
            o_f = ofv[onn.select(ofv)]
            n_sel_good += bool(g_f <= o_f + 0.05 * max(1.0, abs(o_f)))
            want = onn.posterior_mean(r2, kq, ym[idx, j], out["theta_opt"][0, j], out["jitter_opt"][0, j])
            if np.isfinite(want):
                # all rows (nearly) identical: the mean is y * m amp / (m amp + jitter) whatever wins the selection
                assert abs(out["pred"][0, j] - want) <= 1e-6 * abs(want) + 1e-13, (ndup, j, out["pred"][0, j], want)
            assert np.isfinite(out["pred"][0, j])
    print(f"steady state: {n_runs} searches, identical trajectory {n_same}, all-inf (400 evaluations) in the oracle "
          f"{n_all_inf}, of which identical on the device {n_all_inf_same}; selected optimum as good {n_sel_good}/{n_sel}")
    assert n_all_inf >= 5
    assert n_all_inf_same >= 0.9 * n_all_inf
    assert n_same >= 0.5 * n_runs
    assert n_sel_good >= 0.9 * n_sel


def _replay_predicts():
    """(metadata, predicts) of the replay fixtures, one file per iteration (iterations 3 and 4 of the run)"""
    preds = []
    for k in (2, 3):
        z = np.load(os.path.join(GOLDEN, f"run_fhn_d512_replay_k{k}.npz"))
        preds += [{key: z[f"p{p}_{key}"] for key in ("k", "i", "n_rows", "query", "xm", "ym", "starts", "preds",
                                                      "theta_sel", "fvals")} for p in range(int(z["n_predicts"]))]
    return z, preds


def test_replayed_fhn_d512_predicts_against_the_reference(handle):
    """Predicts of iterations 3-4 of the FULL-SIZE FHN target (d=512, N=512, m=20; state dumped from a device
    run) replayed through the unmodified reference `NNGP_p.predict` under the shim (oracle/make_replay.py ->
    tests/golden/run_fhn_d512_replay_k*.npz): same neighbour rows, same host-drawn starts.  From slice ~20 on the
    trajectory sits at its steady state and the predicted correction is < 1e-9 -- nothing there can move K; the
    slices that decide K are the first ~15, where the correction is 1e-7 .. 4e-6 against epsilon = 5e-7.
    Asserted per predict, in BOTH directions:
      * searches that end at +inf (they ran 400 evaluations) in the reference but not on the device, and on the
        device but not in the reference: each <= 4 % of the 4608 searches (a literal potf2 restatement disagrees with the
        installed LAPACK on 1-4 % of such evaluations; observed here: <= 2.7 %, only on steady-state predicts whose
        correction is ~1e-15);
      * where one side selects a lower objective value than the other, the OTHER side's evaluation of that very point
        (device objective at the reference's optimum, LAPACK objective at the device's optimum) is not lower in
        >= 90 % of the cases: the selected kernel matrices have condition numbers ~1e17 (asserted), the value
        of the objective there is rounding noise of whoever evaluates it, and each side's "better" optimum is the
        minimum over its own noise -- not an optimum the other side failed to find;
      * |prediction - reference prediction| <= epsilon everywhere, <= epsilon / 10 in >= 85 % of the 512
        dimensions, median <= 2e-9.
    The reference's own optimiser trajectories are not reproducible below 1 ulp of the objective (LAPACK rounding,
    DESIGN.md section 2): ~25 % of the searches end in a different optimum, which is what bounds the agreement."""
    import torch
    z, preds = _replay_predicts()
    m, d = int(z["m"]), int(z["d"])
    dev = torch.device('cuda', handle.device)
    eps = 5e-7
    worst = 0.0
    for P in preds:
        handle.dataset_reset()
        handle.dataset_reserve(m, d)
        handle.dataset_append_host(P["xm"], P["ym"])
        out = handle.predict_host(P["query"][None], m, P["starts"][None], 1, 0.1, 0.1, details=True)
        assert np.array_equal(out["idx"][0], np.arange(m)), "neighbour order (rows are stored in kNN order)"
        g_f, r_f = out["fvals"][0, :, :, 0], P["fvals"]
        gi, ri = np.isinf(g_f), np.isinf(r_f)
        n_s = g_f.size
        dev_only, ref_only = int(np.sum(gi & ~ri)), int(np.sum(ri & ~gi))
        fin = ~gi & ~ri
        close = np.abs(g_f[fin] - r_f[fin]) <= 1e-6 * np.maximum(1.0, np.abs(r_f[fin]))
        # selected optimum per dimension (models.py:212-215 applied to each side's own searches)
        r_sel = np.array([r_f[j][onn.select(r_f[j])] for j in range(d)])
        g_sel = out["fval_opt"][0]
        tol = 1e-6 * np.maximum(1.0, np.abs(r_sel))
        dev_lower, ref_lower = g_sel < r_sel - tol, r_sel < g_sel - tol
        r_arg = np.array([onn.select(r_f[j]) for j in range(d)])
        th_r, jit_r = P["theta_sel"], onn.JITTERS[r_arg]
        th_d, jit_d = out["theta_opt"][0], out["jitter_opt"][0]
        r2 = onn.pairwise_sqdist(P["xm"], P["xm"])
        o = torch.empty((1, d, 1), dtype=torch.float64, device=dev)
        handle.gp_nll(torch.arange(m, dtype=torch.int64, device=dev)[None].contiguous(), 1, m, 1,
                      torch.from_numpy(th_r[None, :, None, :].copy()).to(dev),
                      torch.from_numpy((10.0 ** jit_r)[None, :, None].copy()).to(dev), o)
        dev_at_ref = o.cpu().numpy()[0, :, 0]
        lap_at_dev = np.array([onn.neg_log_lik(r2, P["ym"][:, j], th_d[j], jit_d[j]) if dev_lower[j] else np.nan
                               for j in range(d)])
        confirmed_r = int(np.sum(dev_at_ref[ref_lower] < r_sel[ref_lower] - tol[ref_lower]))   # device agrees it is lower
        confirmed_d = int(np.sum(lap_at_dev[dev_lower] < g_sel[dev_lower] - tol[dev_lower]))
        conds = [np.linalg.cond(onn.se_kernel_from_r2(r2, th_r[j]) + np.eye(m) * 10 ** jit_r[j]) for j in range(0, d, 16)]
        dp = np.abs(out["pred"][0] - P["preds"])
        worst = max(worst, dp.max())
        print(f"replay k={int(P['k'])} i={int(P['i'])}: +inf searches device-only {dev_only} reference-only {ref_only} "
              f"(both {int(np.sum(gi & ri))}/{n_s}); search optima equal {close.mean():.3f}; selected optimum lower on "
              f"device {int(dev_lower.sum())} (LAPACK evaluates it even lower in {confirmed_d}) / reference "
              f"{int(ref_lower.sum())} (device evaluates it even lower in {confirmed_r}) of {d}, log10 cond of the selected "
              f"matrices median {np.median(np.log10(conds)):.1f}; |pred - ref| max {dp.max():.2e} median "
              f"{np.median(dp):.2e}, > eps/10 in {int(np.sum(dp > eps / 10))} dims; |ref pred| max {np.abs(P['preds']).max():.2e}")
        assert dev_only <= 0.04 * n_s and ref_only <= 0.04 * n_s, (dev_only, ref_only)
        assert confirmed_r <= 0.1 * max(10, ref_lower.sum()) and confirmed_d <= 0.25 * max(10, dev_lower.sum()), \
            (confirmed_r, confirmed_d)
        if np.abs(P["preds"]).max() > 1e-7 and int(P["i"]) < 12:
            assert np.median(np.log10(conds)) > 14, "the early-slice optima sit at numerically singular matrices"
        assert np.all(np.isfinite(out["pred"][0]))
        assert dp.max() <= eps and np.mean(dp <= eps / 10) >= 0.85 and np.median(dp) <= 2e-9, \
            (dp.max(), np.mean(dp <= eps / 10), np.median(dp))
    assert worst > 1e-8, "the fixture must contain predicts from the slices that decide K"


@pytest.mark.parametrize("n,d,m,R", [(600, 8, 20, 1), (500, 6, 10, 2), (400, 5, 13, 1), (300, 4, 32, 1), (300, 3, 5, 1)])
def test_grouped_search_kernel_equals_one_search_per_warp_bitwise(handle, n, d, m, R):
    """gp_fit_grouped_kernel (several Nelder-Mead searches per warp, two matrix rows per lane) performs, per matrix
    entry, the operations of the one-search-per-warp kernel in the same order: every search ends at the same bits
    (theta, objective, evaluation count) and so do selection and prediction -- also with failing factorisations
    (duplicated rows) and padded rows (m odd)."""
    rng = np.random.default_rng(40 + m)
    x, y = make_dataset(rng, n, d)
    x[5:9] = x[4]                      # exact duplicates: singular kernel matrices, +inf objectives
    y[5:9] = y[4]
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    nq = 7
    Q = np.concatenate([x[4:5] + 0.0, x[rng.permutation(n)[:nq - 1]] + 1e-3 * rng.standard_normal((nq - 1, d))])
    starts = rng.integers(-8, 0, (nq, d, 9, R, 2)).astype(np.int8)
    res = {}
    try:
        for mode in ("warp", "grouped"):
            handle.set_fit_mode(mode)
            res[mode] = handle.predict_host(Q, m, starts, R, 0.1, 0.1, details=True)
    finally:
        handle.set_fit_mode("auto")
    for key in ("idx", "nfev", "thetas", "fvals", "theta_opt", "fval_opt", "jitter_opt", "pred"):
        assert np.array_equal(res["warp"][key], res["grouped"][key], equal_nan=True), key
    assert np.isinf(res["warp"]["fvals"]).sum() > 0 and np.isfinite(res["warp"]["fvals"]).sum() > 0


@pytest.mark.parametrize("n,d,m", [(300, 3, 33), (400, 3, 48), (500, 2, 64), (700, 3, 100), (400, 4, 160)])
def test_more_than_32_neighbours(handle, n, d, m):
    """nn='adaptive' gives m = max(10, k+2) (models.py:172-175): past iteration 30 the neighbour set exceeds one lane
    per row.  The large-m path (one CTA per search, matrix in shared memory) against the oracle: neighbour indices
    bit-exact, searches mostly on SciPy's trajectory, objective and posterior mean at the device's optimum equal to
    the oracle's (LAPACK) where the matrix is well conditioned."""
    rng = np.random.default_rng(60 + m)
    x, y = make_dataset(rng, n, d)
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    q = x[7:8] + 1e-3 * rng.standard_normal((1, d))
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    out = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
    oi, okq = onn.knn(q[0], x, m)
    assert np.array_equal(out["idx"][0], oi)
    r2 = onn.pairwise_sqdist(x[oi], x[oi])
    same = total = checked = 0
    for j in range(d):
        for a in range(9):
            th, fv, ne = onn.nm_run(r2, y[oi, j], starts[0, j, a, 0].astype(float), onn.JITTERS[a], 0.1, 0.1)
            total += 1
            same += bool(np.array_equal(out["thetas"][0, j, a, 0], th) and out["nfev"][0, j, a, 0] == ne)
        best = onn.select(out["fvals"][0, j, :, 0])
        assert out["jitter_opt"][0, j] == -20 + best and out["fval_opt"][0, j] == out["fvals"][0, j, best, 0]
        th_o, jit_o = out["theta_opt"][0, j], out["jitter_opt"][0, j]
        K = onn.se_kernel_from_r2(r2, th_o) + np.eye(m) * 10 ** jit_o
        cond = np.linalg.cond(K)
        want_f = onn.neg_log_lik(r2, y[oi, j], th_o, jit_o)
        want_p = onn.posterior_mean(r2, okq, y[oi, j], th_o, jit_o)
        assert np.isfinite(out["pred"][0, j])
        if cond < 1e12 and np.isfinite(want_f):
            checked += 1
            assert abs(out["fval_opt"][0, j] - want_f) <= max(1e-8, 10 * cond * 2.2e-16) * max(1.0, abs(want_f)), (j, cond)
            assert abs(out["pred"][0, j] - want_p) <= max(1e-8, 4 * cond * 2.2e-16) * abs(want_p) + 1e-14, (j, cond)
    assert np.all(out["nfev"] >= 3) and np.all(out["nfev"] <= 400)
    print(f"m={m}: {same}/{total} searches on the oracle's trajectory, {checked}/{d} optima well conditioned")
    assert same >= 0.4 * total


@pytest.mark.parametrize("n,d,m", [(64, 6, 20), (500, 8, 20), (300, 5, 11), (300, 4, 31)])
def test_continuation_kernel_equals_sequential_search_bitwise(handle, n, d, m):
    """gp_fit_spec_kernel (the four warps of a CTA evaluate reflection / expansion / both contractions -- or, when
    every vertex is +inf, reflection / inside contraction / both shrunk vertices -- side by side, the state machine
    consumes them in SciPy's order) continues searches parked after `budget` evaluations: thetas, objective values,
    evaluation counts, selection and prediction must be the bits of the purely sequential search, whatever the
    budget (3 = every search is continued from its initial simplex)."""
    rng = np.random.default_rng(70 + m)
    if n == 64:   # steady-state-like: identical rows, searches that run to 400 evaluations on +inf
        x = np.tile(rng.uniform(-1, 1, (1, d)), (n, 1))
        x[:8] += 1e-3 * rng.standard_normal((8, d))
        y = 1e-4 * rng.standard_normal((n, d))
        q = x[20:21] + 0.0
    else:
        x, y = make_dataset(rng, n, d)
        x[5:8] = x[4]
        y[5:8] = y[4]
        q = x[4:5] + 1e-4 * rng.standard_normal((1, d))
    handle.dataset_reset()
    handle.dataset_reserve(n, d)
    handle.dataset_append_host(x, y)
    starts = rng.integers(-8, 0, (1, d, 9, 1, 2)).astype(np.int8)
    res = {}
    try:
        handle.set_fit_mode("warp")
        for budget in (0, 100, 30, 3):
            handle.set_fit_budget(budget)
            res[budget] = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
        handle.set_fit_budget(0)
        handle.set_fit_mode("quad")   # whole searches on four warps, from the initial simplex
        res["quad"] = handle.predict_host(q, m, starts, 1, 0.1, 0.1, details=True)
    finally:
        handle.set_fit_budget(0)
        handle.set_fit_mode("auto")
    for budget in (100, 30, 3, "quad"):
        for key in ("nfev", "thetas", "fvals", "theta_opt", "fval_opt", "jitter_opt", "pred"):
            assert np.array_equal(res[0][key], res[budget][key], equal_nan=True), (key, budget)
    assert res[0]["nfev"].max() > 100, "the case must contain searches longer than the default budget"
