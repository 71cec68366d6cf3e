"""The position-based neighbour rules of the time-aware study (models_alt.py) on the device drivers.

A. nngp_listed_prep: distances and neighbour matrix of host-chosen lists, bit for bit the strict left-to-right sums.
B. PararealDevice with each rule equals the host driver Parareal with the same nntype, bit for bit (published setting).
C. Every member of an ensemble of rules x seeds (and nearest-neighbour members) equals its solo PararealDevice run.
D. The listed sweep called one slice and one dimension block at a time equals the whole listed sweep.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib
from nearest_neighbors_gparareal_b200.models_alt import NNTYPES
from nearest_neighbors_gparareal_b200.utils import dim_block
from helpers import make_dataset
from test_gpu_routes import load

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYSTEMS = {"fhn": lambda: nn.FHN_ODE(normalization='-11'), "lorenz": lambda: nn.Lorenz(normalization='-11')}


@pytest.fixture(scope="module")
def handle():
    return _lib.Handle(0)


def _strict(a, b):
    """sum_j (a_j - b_j)^2 left to right, one rounding per operation (NumPy never contracts to FMA)"""
    s = np.zeros(np.broadcast_shapes(a.shape, b.shape)[:-1])
    for j in range(a.shape[-1]):
        diff = a[..., j] - b[..., j]
        s = s + diff * diff
    return s


@pytest.mark.parametrize("d", [2, 3, 128, 512])
def test_listed_prep_is_the_strict_sum(handle, d):
    import torch
    rng = np.random.default_rng(d)
    n = 400
    x, y = make_dataset(rng, n, d)
    load(handle, x, y)
    for m in list(range(1, 34)) + [40, 160]:
        nq, ld = 3, m + (m % 3)
        rows = rng.integers(0, n, (nq, ld))  # unsorted
        rows[1, :m // 2] = rows[1, 0]        # repeated rows: zero distances, singular matrices
        q = np.stack([x[rows[0, 0]] + 1e-3 * rng.standard_normal(d), rng.uniform(-1, 1, d), x[rows[2, -1]]])
        dq = torch.zeros((nq, d + 1), dtype=torch.float64, device='cuda')  # row stride d + 1
        dq[:, :d] = torch.from_numpy(q)
        dist = torch.full((nq, ld), -1.0, dtype=torch.float64, device='cuda')
        r2 = torch.full((nq, ld, ld), -1.0, dtype=torch.float64, device='cuda')
        handle.listed_prep(dq, d + 1, nq, m, torch.from_numpy(rows).cuda(), ld, dist, r2)
        torch.cuda.synchronize()
        dist, r2 = dist.cpu().numpy(), r2.cpu().numpy()
        for k in range(nq):
            xr = x[rows[k, :m]]
            assert np.array_equal(dist[k, :m], _strict(xr, q[k][None, :])), (d, m, k)
            assert np.array_equal(r2[k, :m, :m], _strict(xr[:, None, :], xr[None, :, :])), (d, m, k)
            assert np.all(dist[k, m:] == -1.0) and np.all(r2[k, m:, :] == -1.0) and np.all(r2[k, :, m:] == -1.0)


@pytest.mark.parametrize("m", [7, 16, 33])
def test_fit_from_the_listed_prep_equals_fit_predict(handle, m):
    """same pred, theta_opt and nfev as nngp_fit_predict given the host-computed distances"""
    import torch
    rng = np.random.default_rng(m)
    n, d, R = 300, 4, 1
    x, y = make_dataset(rng, n, d)
    load(handle, x, y)
    rows = rng.permutation(n)[:m][None, :]
    q = x[rows[0, 0]] + 1e-3 * rng.standard_normal(d)
    starts = torch.from_numpy(rng.integers(-8, 0, (1, d, 9, R, 2)).astype(np.int8)).cuda()
    d_rows, d_q = torch.from_numpy(rows).cuda(), torch.from_numpy(q[None, :]).cuda()
    dist = torch.empty((1, m), dtype=torch.float64, device='cuda')
    r2 = torch.empty((1, m, m), dtype=torch.float64, device='cuda')
    handle.listed_prep(d_q, d, 1, m, d_rows, m, dist, r2)
    outs = []
    for dd in (dist, torch.from_numpy(_strict(x[rows[0]], q[None, :])[None, :]).cuda()):
        o = dict(pred=torch.empty((1, d), dtype=torch.float64, device='cuda'),
                 theta=torch.empty((1, d, 2), dtype=torch.float64, device='cuda'),
                 nfev=torch.empty((1, d, 9, R), dtype=torch.int32, device='cuda'))
        handle.fit_predict(d_q, d_rows, dd, 1, m, R, starts, 0.1, 0.1, o['pred'], d_theta=o['theta'], d_nfev=o['nfev'])
        outs.append({k: v.cpu().numpy() for k, v in o.items()})
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k], equal_nan=True), k


def _published(system):
    ode = SYSTEMS[system]()
    cfg = nn.Config(ode).get()
    return ode, cfg, nn.CudaSolverRK(ode.get_vector_field(), **cfg)


@pytest.mark.parametrize("system", ["fhn", "lorenz"])
def test_device_driver_equals_the_host_driver_for_every_rule(system):
    """the published nngptime_diff_subsets2 setting: nn = 16, seed 45, epsilon 5e-7"""
    for nntype in NNTYPES:
        ode, cfg, solver = _published(system)
        host = nn.Parareal(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='').run(
            model='nngp', pool=nn.CudaPool(), parall='mpi', nn=16, nntype=nntype, seed=45)
        ode, cfg, solver = _published(system)
        dev = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='').run(
            model='nngp', nn=16, nntype=nntype, seed=45)
        assert dev['k'] == host['k'], (nntype, dev['k'], host['k'])
        assert dev['conv_int'] == host['conv_int'], nntype
        assert dev['n_rows'] == host['x'].shape[0], nntype
        assert np.array_equal(dev['u'], host['u_last']), nntype
        assert np.array_equal(dev['err'], host['err'], equal_nan=True), nntype


def test_device_driver_refuses_checkpoints_of_a_position_rule():
    ode, cfg, solver = _published("lorenz")
    p = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='')
    with pytest.raises(Exception, match="store_int"):
        p.run(model='nngp', nn=16, nntype='row', seed=45, store_int=True)


def _same(a, b, label):
    assert a['k'] == b['k'], (label, a['k'], b['k'])
    assert a['conv_int'] == b['conv_int'], label
    assert a['converged'] == b['converged'], label
    assert a['n_rows'] == b['n_rows'], (label, a['n_rows'], b['n_rows'])
    assert np.array_equal(a['u'], b['u']), label
    assert np.array_equal(a['err'], b['err'], equal_nan=True), label


def _solo(system, seed, nn_, nntype, eps=5e-7, early_stop=None):
    ode, cfg, solver = _published(system)
    return nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=eps, verbose='').run(
        model='nngp', nn=nn_, nntype=nntype, seed=seed, early_stop=early_stop)


def test_ensemble_of_rules_and_seeds_equals_solo_runs():
    rules = [r for r in NNTYPES for _ in (45, 46)] + ['nn', 'nn']
    seeds = [45, 46] * len(NNTYPES) + [47, 48]
    nns = [16] * (2 * len(NNTYPES)) + [11, 'adaptive']
    ode, cfg, solver = _published("lorenz")
    outs = nn.PararealEnsemble(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='').run(
        seeds=seeds, nn=nns, nntype=rules)
    for e, out in enumerate(outs):
        _same(out, _solo("lorenz", seeds[e], nns[e], rules[e]), (e, rules[e], seeds[e]))


def test_ensemble_members_leave_at_different_iterations_and_cross_into_the_big_kernels():
    """a col_only member with a tiny epsilon runs to early_stop = 36: m = k + 1 passes 32"""
    members = [('col_only', 45, 16, 1e-13, 36), ('row', 46, 16, 5e-7, 3), ('nn', 47, 16, 5e-7, None),
               ('col+rnd', 45, 'adaptive', 1e-6, None), ('row_col', 46, 12, 5e-7, 6), ('col_full', 45, 16, 1e-9, 20)]
    ode, cfg, solver = _published("lorenz")
    outs = nn.PararealEnsemble(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='').run(
        seeds=[m[1] for m in members], nn=[m[2] for m in members], nntype=[m[0] for m in members],
        epsilons=[m[3] for m in members], early_stops=[m[4] for m in members])
    assert outs[0]['k'] == 36
    for e, (rule, seed, nn_, eps, stop) in enumerate(members):
        _same(outs[e], _solo("lorenz", seed, nn_, rule, eps=eps, early_stop=stop), (e, rule))


@pytest.mark.parametrize("system,nntype", [("lorenz", "row"), ("lorenz", "col+rnd"), ("fhn", "col_full")])
def test_listed_sweep_by_dimension_block_equals_the_whole_sweep(system, nntype):
    """one slice and one output-dimension block per call (the dimension-sharded sweep of W ranks, with the all-gather
    of row i+1 done by the W calls writing their blocks of it) equals one call over all slices"""
    import torch
    ode, cfg, solver = _published(system)
    p = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=5e-7, verbose='')
    model = p._make_model('nngp', pool=nn.CudaPool(), nn=16, nntype=nntype, seed=45)
    st = p.device_setup(model)
    h, n, N = st['h'], p.n, p.N
    p.device_fine_step(st)
    I = st['I']
    h.append_iteration(st['u_cur'], st['uF'], st['uG_cur'], N, I, n, st['stream'])
    rows = model.neighbour_table([I - 1], I)
    starts = torch.from_numpy(model.draw_starts(N - I)).to(st['dev'])
    args = (st['sys'], st['mG'], solver.h_mode, solver.Ng, st['t'], N, I)
    u_w, g_w = st['u_next'].clone(), st['uG_next'].clone()
    u_b, g_b = st['u_next'].clone(), st['uG_next'].clone()
    h.sweep_listed_shard(*args, I, N - I, rows, model.n_restarts, starts, model.fatol, model.xatol, u_w, g_w, n, 0, n,
                         st['stream'])
    W = n
    for i in range(I, N):
        for r in range(W):
            j0, dl = dim_block(n, r, W)
            h.sweep_listed_shard(*args, i, 1, rows, model.n_restarts, starts, model.fatol, model.xatol, u_b, g_b, n, j0,
                                 dl, st['stream'])
    torch.cuda.synchronize()
    assert torch.equal(u_w, u_b) and torch.equal(g_w, g_b)
    assert not torch.equal(u_w, st['u_next'])


_WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
rank, world, port = int(sys.argv[2]), int(sys.argv[3]), sys.argv[4]
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=port, RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
import numpy as np, torch, torch.distributed as dist
import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import _lib
torch.cuda.set_device(rank)
dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
solo = [dist.new_group([r]) for r in range(world)][rank]
ok = True
for nntype in ("row", "col+rnd"):
    outs = {}
    for label, group, shard in (("single", solo, False), ("sharded", None, True)):
        ode = nn.FHN_PDE(d_x=4)
        solver = nn.CudaSolverRK(ode.get_vector_field(), handle=_lib.default_handle(rank), Ng=5, Nf=40, F='RK8', G='RK4')
        p = nn.PararealDevice(ode, solver, tspan=[0, 8], N=16, epsilon=1e-6, verbose='', group=group, shard_sweep=shard)
        outs[label] = p.run(model='nngp', nn=8, nntype=nntype, seed=45)
    same = (outs["sharded"]['k'] == outs["single"]['k'] and np.array_equal(outs["sharded"]['u'], outs["single"]['u'])
            and np.array_equal(outs["sharded"]['err'], outs["single"]['err'], equal_nan=True))
    print(f"rank {rank} {nntype}: K={outs['sharded']['k']} bitwise equal to the single-GPU run: {same}", flush=True)
    ok &= same
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 3)
'''


def test_two_rank_listed_sweep_equals_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker_listed.py"
    script.write_text(_WORKER)
    port = str(35500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(r), "2", port], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
