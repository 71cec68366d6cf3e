"""CPU: host-side logic and the C-ABI boundary (no compute calls: there is no GPU here)."""
import os
import pickle
import re
import subprocess
import sys

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib, parareal as ppara
from oracle import systems as osys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "nngpara.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nngp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol_at_abi_version_2():
    if not os.path.exists(_lib.LIB_PATH):
        from nearest_neighbors_gparareal_b200.build import build
        build()
    lib = _lib.load_library()
    syms = header_symbols()
    assert len(syms) >= 25
    for name in syms:
        assert hasattr(lib, name), name
    assert sorted(_lib.SIGNATURES) == syms
    assert lib.nngp_abi_version() == 2


def test_tableau_equals_reference_tableau():
    """the Butcher tableaus compiled into the library == RK.py:30-48 (oracle restatement), bit for bit"""
    import ctypes
    from oracle import rk as ork
    lib = _lib.load_library()
    for name, code in _lib.METHODS.items():
        S = ctypes.c_int(0)
        a, b, c = np.zeros(121), np.zeros(11), np.zeros(11)
        assert lib.nngp_get_tableau(code, ctypes.byref(S), a.ctypes.data, b.ctypes.data, c.ctypes.data) == 0
        s = S.value
        oa, ob, oc = ork.tableau(name)
        assert np.array_equal(a[:s * s].reshape(s, s), oa) and np.array_equal(b[:s], ob) and np.array_equal(c[:s], oc)
    assert lib.nngp_get_tableau(3, ctypes.byref(S), a.ctypes.data, b.ctypes.data, c.ctypes.data) != 0


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.NNGPError, match="no CPU fallback|no CUDA device"):
        _lib.Handle(0)


def test_start_points_stream_is_the_reference_stream():
    """models.py:192 draws rng.integers(-8,0,2) once per task; the vectorised draw is identical"""
    m = nn.CudaNNGP(n=5, N=8, nn=11, seed=45, n_restarts=2)
    ref = np.random.default_rng(45)
    want = np.stack([ref.integers(-8, 0, 2) for _ in range(3 * 5 * 9 * 2)]).reshape(3, 5, 9, 2, 2)
    got = np.concatenate([m.draw_starts(1), m.draw_starts(2)])
    assert got.dtype == np.int8 and np.array_equal(got, want)
    assert got.min() >= -8 and got.max() <= -1
    assert m.neighbours(0) == 11
    assert nn.CudaNNGP(n=5, N=8).neighbours(0) == 10 and nn.CudaNNGP(n=5, N=8).neighbours(20) == 22


def test_systems_mirror_reference_initial_conditions_and_presets():
    pairs = [(nn.Lorenz(normalization='-11'), osys.Lorenz(normalization='-11')),
             (nn.Hopf(normalization='-11'), osys.Hopf(normalization='-11')),
             (nn.Burgers(d_x=128, normalization='-11'), osys.Burgers(d_x=128, normalization='-11')),
             (nn.FHN_PDE(d_x=16), osys.FHN_PDE(d_x=16)), (nn.Rossler(), osys.Rossler())]
    for dev, ora in pairs:
        assert np.array_equal(dev.get_init_cond(), ora.u0), dev.name
        assert dev.name == ora.name and dev.get_dim() == ora.dim()
    for dev, ora, N in [(nn.Lorenz(normalization='-11'), osys.Lorenz(normalization='-11'), None),
                        (nn.Hopf(normalization='-11'), osys.Hopf(normalization='-11'), 64),
                        (nn.FHN_PDE(d_x=16), osys.FHN_PDE(d_x=16), None), (nn.Brusselator(), osys.Brusselator(), None)]:
        got = nn.Config(dev, N=N, d_x=getattr(dev, 'd_x', None)).get()
        want = osys.preset(ora, N=N)
        assert {k: got[k] for k in want} == want
    assert nn.Hopf(normalization='-11').name == 'Hopf'
    h = nn.Hopf(normalization='-11')
    nn.Config(h, N=32)
    assert h.name == 'Hopf_32'  # configs.py:149
    # FHN stencil coefficients == entries of the reference's dense a*(DXX+DYY), b*(DXX+DYY)
    o = osys.FHN_PDE(d_x=16)
    A = 2.8e-4 * (o.DXX + o.DYY)
    B = 5e-3 * (o.DXX + o.DYY)
    p = nn.FHN_PDE(d_x=16).device_params()
    assert p[0] == 16 and p[1] == A[0, 0] and p[2] == A[0, 1] == A[0, 16] == A[0, 15] and p[3] == B[5, 5] and p[4] == B[5, 6]
    assert np.count_nonzero(A[7]) == 5
    ob = osys.Burgers(d_x=32, normalization='-11')
    pb = nn.Burgers(d_x=32, normalization='-11').device_params()
    assert pb[0] == ob.Dxx[3, 4] == ob.Dxx[0, 31] and pb[1] == ob.Dxx[3, 3] and pb[2] == ob.Dx[3, 4] == -ob.Dx[3, 2] == -ob.Dx[0, 31]


def test_protocol_errors_match_reference():
    ode = nn.Lorenz(normalization='-11')
    with pytest.raises(Exception, match='ode must be an instance of the ODE class'):
        nn.Parareal(object(), None, [0, 1], 4)
    with pytest.raises(Exception, match='solver must be an instance of the SolverAbstr class'):
        nn.Parareal(ode, object(), [0, 1], 4)
    with pytest.raises(NotImplementedError, match='Only RK1, RK2, RK4 and RK8'):
        nn.CudaSolverRK(ode.get_vector_field(), 4, 8, 'RK3', 'RK1')
    with pytest.raises(NotImplementedError, match='Only identity and -11'):
        nn.Lorenz(normalization='01')
    with pytest.raises(Exception, match='no CPU fallback'):
        nn.CudaSolverRK(lambda t, u: u, 4, 8, 'RK4', 'RK1')
    s = nn.CudaSolverRK(ode.get_vector_field(), Ng=4, Nf=8, F='RK4', G='RK1', extra_key_is_swallowed=1)
    p = nn.Parareal(ode, s, tspan=[0, 1], N=4, Ng=4, Nf=8, F='RK4', G='RK1')
    with pytest.raises(Exception, match='Not implemented'):
        p._make_model('elm', pool=None)            # parareal.py:94-97: unknown / out-of-scope model names
    gp = p._make_model('gpjax', pool=None)         # GParareal's full GP (models.py:273-473) is available
    assert gp.name == 'GP' and gp.fatol == 1e-4 and len(gp.thetas) == 3
    s2 = pickle.loads(pickle.dumps(s))
    assert s2.Nf == 8 and s2.ode.name == 'Lorenz'


def test_cuda_pool_batches_solver_calls():
    from nearest_neighbors_gparareal_b200.solver import SolverAbstr

    class Fake(SolverAbstr):  # run_F_timed is the inherited, decorator-wrapped method (its __name__ is lost)
        def __init__(self):
            self.calls = 0

        def run_F_batch(self, t0, t1, u0):
            self.calls += 1
            return u0 + (t1 - t0)[:, None]

        def run_F(self, t0, t1, u0):
            raise AssertionError("must be batched")

    f = Fake()
    pool = nn.CudaPool()
    u0 = [np.zeros(3), np.ones(3), 2 * np.ones(3)]
    out = list(pool.map(f.run_F_timed, [0, 1, 2], [1, 3, 5], u0))
    assert f.calls == 1 and len(out) == 3
    assert np.array_equal(out[2][0], 2 * np.ones(3) + 3) and out[0][1] >= 0
    assert list(pool.map(lambda a, b: a + b, [1, 2], [3, 4])) == [4, 6]
    assert list(nn.MyPool.map(lambda a: a * 2, [1, 2], chunksize=4)) == [2, 4]


def test_slice_block_partition_covers_all_slices():
    for N in (5, 32, 512):
        for I in (0, 1, 7, N - 1):
            if I >= N:
                continue
            for world in (1, 2, 3, 8):
                owned = []
                for r in range(world):
                    chunk, lo, cnt = ppara.slice_block(I, N, r, world)
                    assert lo == min(I + r * chunk, N)
                    owned += list(range(lo, lo + cnt))
                assert owned == list(range(I, N))


_WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
from nearest_neighbors_gparareal_b200.parareal import slice_block, gather_fine_rows
rank, world = int(sys.argv[2]), int(sys.argv[3])
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=sys.argv[4])
dist.init_process_group("gloo", rank=rank, world_size=world)
N, d = 13, 5
ok = True
for I in (0, 1, 4, 12):
    uF = torch.full((N + 1 + N + world, d), -1.0, dtype=torch.float64)
    keep = torch.arange(d, dtype=torch.float64) + 100.0
    uF[:I + 1] = keep
    chunk, lo, cnt = slice_block(I, N, rank, world)
    for s in range(lo, lo + cnt):                      # stand-in for the RK launch of this rank's block
        uF[s + 1] = torch.arange(d, dtype=torch.float64) * 0.5 + s
    gather_fine_rows(uF, I, chunk, rank, world)
    want = torch.stack([torch.arange(d, dtype=torch.float64) * 0.5 + s for s in range(I, N)])
    ok &= bool(torch.equal(uF[I + 1:N + 1], want)) and bool(torch.equal(uF[:I + 1], keep.expand(I + 1, d)))
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 3)
'''


def test_time_slice_sharding_all_gather_gloo_world2(tmp_path):
    """N>1 path on CPU: two ranks each fill their block of fine-solve rows, one all-gather, all rows everywhere"""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(r), "2", port]) for r in range(2)]
    codes = [p.wait(timeout=180) for p in procs]
    assert codes == [0, 0]


_WORKER_DIM = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np, torch, torch.distributed as dist
from nearest_neighbors_gparareal_b200.models import CudaNNGP
from nearest_neighbors_gparareal_b200.utils import dim_block
rank, world = int(sys.argv[2]), int(sys.argv[3])
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=sys.argv[4])
dist.init_process_group("gloo", rank=rank, world_size=world)
ok = True
for d in (8, 6):
    model = CudaNNGP(n=d, N=4, nn=5, shard_predict=True)   # no device call is made in this test
    blk = model._block()
    ok &= blk == dim_block(d, rank, world)
    j0, dl = blk
    pred = np.full((1, d), np.nan)
    pred[0, j0:j0 + dl] = np.arange(j0, j0 + dl) * 1.5 + 7      # this rank's share of the fits
    full = model._gather(pred, blk)
    ok &= bool(np.array_equal(full, (np.arange(d) * 1.5 + 7)[None, :]))
    ok &= model._device_gather_buffer() is None               # gloo: the gather goes through host tensors
model = CudaNNGP(n=7, N=4, nn=5, shard_predict=True)     # 7 % 2 != 0: not sharded
ok &= model._block() is None
ok &= CudaNNGP(n=8, N=4, nn=5)._block() is None           # sharding is opt-in
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 3)
'''


def test_dimension_sharded_predict_all_gather_gloo_world2(tmp_path):
    """N>1 host path on CPU: each rank holds the predictions of its block of output dimensions, one all-gather of
    d/W doubles, the full prediction everywhere (CudaNNGP._block / _gather)"""
    script = tmp_path / "worker_dim.py"
    script.write_text(_WORKER_DIM)
    port = str(31500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(r), "2", port]) for r in range(2)]
    codes = [p.wait(timeout=180) for p in procs]
    assert codes == [0, 0]


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the reference's CPU path = the oracle port on the host cores) prints ONE JSON
    line with the contract keys; small workload so that it runs in seconds on CPU.  Under torchrun only rank 0
    prints (checked through the RANK environment variable)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--dx", "4", "--slices", "16", "--fine-steps", "50"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env={**os.environ, "RANK": "0"})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "iters/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["gpu_launches"] == 0 and line["dtype"] == "f64"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["N_slices"] == 16 and line["config"]["d"] == 32
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env={**os.environ, "RANK": "1"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_intermediate_checkpoint_and_resume_host_driver(tmp_path):
    """parareal.py:114-209, 420-431 in the host mirror: `store_int=True` dumps the loop state after every iteration,
    `load_int_dump` resumes it; the resumed run ends exactly like the uninterrupted one.  CPU: a NumPy solver
    (oracle RK on the Lorenz field) behind the SolverAbstr protocol, the plain Parareal model."""
    import pickle
    from oracle import rk as ork, systems as osys
    from nearest_neighbors_gparareal_b200.solver import SolverAbstr
    o = osys.Lorenz(normalization='-11')

    class NpSolver(SolverAbstr):
        def run_F(self, t0, t1, u0):
            return ork.rk_last(o.f, 'RK4', t0, t1, 60, np.asarray(u0, dtype=float))

        def run_G(self, t0, t1, u0):
            return ork.rk_last(o.f, 'RK1', t0, t1, 6, np.asarray(u0, dtype=float))

    def driver():
        return nn.Parareal(nn.Lorenz(normalization='-11'), NpSolver(), tspan=[0, 1.0], N=10, epsilon=1e-10, verbose='')

    full = driver().run(model='parareal', pool=nn.MyPool())
    assert full['converged'] and full['k'] > 4
    part = driver().run(model='parareal', pool=nn.MyPool(), early_stop=3, store_int=True, int_dir=str(tmp_path),
                        int_name='ck')
    assert part['k'] == 3 and not part['converged']
    with open(tmp_path / 'ck' / 'ck_2', 'rb') as fh:
        dump = pickle.load(fh)
    assert dump.ode is None and dump.solver is None and dump.objs['k'] == 2 and dump.objs['kwargs']['pool'] is None
    p3 = driver()
    res = p3.load_int_dump(dump, pool=nn.MyPool())
    assert res['k'] == full['k'] and res['conv_int'] == full['conv_int'] and res['converged']
    assert np.array_equal(res['u_last'], full['u_last'])
    assert np.array_equal(res['err'], full['err'], equal_nan=True)
    assert np.array_equal(res['u'], full['u'])            # the history of iterates is restored too
    # build_cont_traj (parareal.py:487-508) needs run_F_full of the solver protocol
    class NpSolverFull(NpSolver):
        def run_F_full(self, t0, t1, u0):
            return ork.rk_full(o.f, 'RK4', t0, t1, 60, np.asarray(u0, dtype=float))
    p4 = nn.Parareal(nn.Lorenz(normalization='-11'), NpSolverFull(), tspan=[0, 1.0], N=10, epsilon=1e-10, verbose='')
    out4 = p4.run(model='parareal', pool=nn.MyPool())
    traj = p4.build_cont_traj()
    assert traj.shape == (10 * 61, 3) and np.array_equal(traj[60], out4['u_last'][1] * 0 + traj[60])
    assert np.allclose(traj[60::61][:, :], np.stack([ork.rk_last(o.f, 'RK4', out4['t'][i], out4['t'][i + 1], 60,
                                                                out4['u_last'][i]) for i in range(10)]), rtol=0, atol=0)
    with pytest.raises(Exception, match='do not match'):
        nn.Parareal(nn.Rossler(), NpSolver(), tspan=[0, 1.0], N=10, verbose='').load_int_dump(dump, pool=nn.MyPool())


def test_reference_side_binding_derives_from_reference_classes():
    """integration/cuda_backend.py: the plug-ins are subclasses of the reference's own classes (skipped where the
    reference is not on the machine); construction needs no GPU"""
    from integration.ref_env import find_reference
    if find_reference() is None:
        pytest.skip("reference modules not on this machine")
    from integration.cuda_backend import bind
    B = bind()
    ref = B.ref
    ode = B.FHN_PDE(d_x=4)
    cfg = B.Config(ode, d_x=4).get()
    solver = B.CudaSolverRK(ode.get_vector_field(), **cfg)
    model = B.CudaNNGP(n=ode.get_dim(), N=cfg["N"], worker_pool=None, nn=12, seed=45)
    par = B.CudaParareal(ode, solver, **cfg)     # parareal.py:37-41 type checks pass
    assert isinstance(ode, ref.systems.FHN_PDE) and isinstance(solver, ref.solver.SolverRK)
    assert isinstance(model, ref.models.NNGP_p) and isinstance(par, ref.parareal.Parareal)
    assert type(par)._parareal is ref.parareal.Parareal._parareal
    assert model.fatol == 0.1 and model.nn == 12 and model.name == 'NNGP'
    assert np.array_equal(ode.get_init_cond(), nn.FHN_PDE(d_x=4).get_init_cond())
    with pytest.raises(Exception, match="instance of the ODE class"):
        ref.parareal.Parareal(object(), solver, **cfg)


def test_lockstep_nelder_mead_equals_scipy_bit_for_bit():
    """gp_full._NM (the step-function Nelder-Mead that drives the batched GParareal fits) against the installed
    scipy.optimize.minimize on objectives with flat valleys, +inf regions and evaluation-limit runs"""
    from scipy.optimize import minimize
    from nearest_neighbors_gparareal_b200.gp_full import _NM
    rng = np.random.default_rng(3)

    def rosen(x):
        return (1 - x[0]) ** 2 + 100 * (x[1] - x[0] ** 2) ** 2

    def walled(x):
        return np.inf if x[0] < 0.3 else (x[0] - 1) ** 2 + abs(x[1]) ** 1.5

    def all_inf(x):
        return np.inf

    def noisy(x):
        return np.sin(5 * x[0]) * np.cos(3 * x[1]) + 0.1 * x[0] ** 2 + 0.1 * x[1] ** 2

    for f in (rosen, walled, all_inf, noisy):
        for _ in range(6):
            x0 = rng.uniform(-2, 2, 2) if f is not walled else np.array([rng.uniform(0.31, 2), rng.uniform(-1, 1)])
            for tol in (1e-4, 1e-1):
                nm = _NM(x0, tol, tol)
                while not nm.done:
                    nm.step(float(f(nm.pt)))
                x, fv = nm.result()
                with np.errstate(all="ignore"):
                    ref = minimize(f, x0, method='Nelder-Mead', options={'fatol': tol, 'xatol': tol})
                assert nm.fcalls == ref.nfev, (f.__name__, x0, nm.fcalls, ref.nfev)
                assert np.array_equal(x, ref.x) and (fv == ref.fun or (np.isinf(fv) and np.isinf(ref.fun)))


def test_position_based_neighbour_rules_pick_the_documented_rows():
    """models_alt.CudaNNGPAlt.neighbour_rows against a direct transcription of the generators of
    nnGPara_with_time.py:98-171 on a synthetic observation cube (no device call)"""
    from nearest_neighbors_gparareal_b200.models_alt import CudaNNGPAlt
    rng = np.random.default_rng(0)
    N, n, k = 12, 2, 3
    first = [0, 1, 3, 4]                      # first unconverged slice per iteration
    data_x = np.full((N, n, N), np.nan)
    rows = []
    for j in range(k + 1):
        for s in range(first[j], N):
            data_x[s, :, j] = rng.standard_normal(n)
            rows.append(data_x[s, :, j].copy())
    x = np.array(rows)

    def ref_cycle(mtx, it, sl, by_row):
        def cyc(a, b):
            done_a = False
            while True:
                try:
                    yield next(a)
                except StopIteration:
                    done_a = True
                try:
                    yield next(b)
                except StopIteration:
                    if done_a:
                        break
        if by_row:   # 'row': iterations outermost
            for row in range(it, -1, -1):
                for col in cyc(iter(range(sl, -1, -1)), iter(range(sl + 1, mtx.shape[0]))):
                    if not np.any(np.isnan(mtx[col, :, row])):
                        yield mtx[col, :, row]
        else:        # 'col_full': slices outermost
            for col in cyc(iter(range(sl, -1, -1)), iter(range(sl + 1, mtx.shape[0]))):
                for row in range(it, -1, -1):
                    if not np.any(np.isnan(mtx[col, :, row])):
                        yield mtx[col, :, row]

    for nntype, by_row in (('row', True), ('col_full', False)):
        m = CudaNNGPAlt.__new__(CudaNNGPAlt)
        m.nntype, m.nn, m.k, m.x, m.data_x = nntype, 7, k, x, data_x
        present = ~np.isnan(data_x[:, 0, :k + 1])
        m._present = present
        m._first = np.array(first)
        m._offset = np.concatenate([[0], np.cumsum(N - m._first)])[:k + 1]
        for i in (4, 7, 11):
            gen = ref_cycle(data_x[:, :, :k + 1], k, i, by_row)
            want = np.array([next(gen) for _ in range(7)])
            assert np.array_equal(x[m.neighbour_rows(i)], want), (nntype, i)
    m.nntype = 'col_only'
    assert np.array_equal(x[m.neighbour_rows(6)], data_x[6, :, :k + 1].T)
