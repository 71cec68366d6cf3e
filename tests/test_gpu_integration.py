"""GPU: the reference's UNMODIFIED driver (`parareal.Parareal._parareal`, parareal.py:212-471) running on
libnngpara.so through integration/cuda_backend.py -- classes that derive from the reference's own SolverRK / NNGP_p /
ODE / Parareal, so its isinstance checks (parareal.py:37-41) and executor protocol are the real ones.

The tests that execute the reference's code need its modules (NNGP_REFERENCE_DIR, or the git-ignored copy baseline/_ref
made by scripts/stage_reference.sh) and skip without them.  What the reference driver computed on this backend is also
stored (tests/golden/reference_driver_on_cuda_backend.json), and the package's own drivers are checked against it on
every run."""
import json
import os

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from helpers import GOLDEN, load_run, case_system, device_system
from integration.ref_env import find_reference

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(find_reference() is None, reason="reference modules not on this machine")


def _ref_ode(B, key, kw):
    return {"lorenz": lambda: B.Lorenz(normalization="-11"), "hopf": lambda: B.Hopf(normalization="-11"),
            "burgers": lambda: B.Burgers(normalization="-11", **kw), "fhn_pde": lambda: B.FHN_PDE(**kw)}[key]()


@pytest.mark.parametrize("name", ["lorenz_N32_m11", "fhn_d32_N32_m12", "hopf_N32_m15"])
def test_package_drivers_reproduce_the_reference_driver_run(name):
    """the host-protocol driver and the device-resident driver end with the K / conv_int that the reference's unmodified
    driver reached on this backend (stored), agree bit for bit with each other, and meet the reference's own NumPy run"""
    with open(os.path.join(GOLDEN, "reference_driver_on_cuda_backend.json")) as fh:
        want = json.load(fh)[name]
    z, cfg, mkw = load_run(name)
    key, kw = case_system(name)
    ode = device_system(key, **kw)
    solver = nn.CudaSolverRK(ode.get_vector_field(), **{k: cfg[k] for k in ("Ng", "Nf", "F", "G")})
    host = nn.Parareal(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=float(z["epsilon"]), verbose='') \
        .run(model='nngp', pool=nn.CudaPool(), parall='mpi', **mkw)
    dev = nn.PararealDevice(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=float(z["epsilon"]), verbose='') \
        .run(model='nngp', **mkw)
    K = host['k']
    assert host['converged'] and K == want["K"] and host['conv_int'] == want["conv_int"]
    assert dev['k'] == K and dev['conv_int'] == host['conv_int']
    assert np.array_equal(dev['u'], host['u_last']) and np.array_equal(dev['err'], host['err'], equal_nan=True)
    assert host['u'].shape == (cfg["N"] + 1, ode.get_dim(), K) and host['err'].shape == (cfg["N"] + 1, K)
    if name != "hopf_N32_m15":
        assert K == int(z["K"])
    else:
        assert abs(K - int(z["K"])) <= 1


@needs_reference
@pytest.mark.parametrize("name", ["lorenz_N32_m11", "fhn_d32_N32_m12", "hopf_N32_m15"])
def test_unmodified_reference_driver_on_cuda_backend(name):
    from integration.cuda_backend import bind
    B = bind()
    ref = B.ref
    z, cfg, mkw = load_run(name)
    key, kw = case_system(name)
    ode = _ref_ode(B, key, kw)
    solver = B.CudaSolverRK(ode.get_vector_field(), **{k: cfg[k] for k in ("Ng", "Nf", "F", "G")})
    # the reference's own type checks accept the plug-ins
    assert isinstance(ode, ref.systems.ODE) and isinstance(solver, ref.solver.SolverAbstr)
    p = B.CudaParareal(ode, solver, tspan=cfg["tspan"], N=cfg["N"], epsilon=float(z["epsilon"]), verbose='')
    assert type(p)._parareal is ref.parareal.Parareal._parareal      # the loop that runs is the reference's
    out = p.run(model='nngp', pool=B.CudaPool(), parall='mpi', **mkw)
    K = out['k']
    print(f"{name}: unmodified reference driver on the CUDA backend: K={K} conv_int={out['conv_int']} "
          f"(reference run: K={int(z['K'])} conv_int={[int(v) for v in z['conv_int']]}) "
          f"runtime {out['timings']['runtime']:.2f}s  F {out['timings']['F_time']:.2f}s  "
          f"model {out['timings']['mdl_tot_t']:.2f}s")
    assert out['converged']
    # the reference's result layout (parareal.py:469-471)
    N, n = cfg["N"], ode.get_dim()
    assert out['u'].shape == (N + 1, n, K) and out['err'].shape == (N + 1, K)
    for k_ in ('t', 'u', 'err', 'x', 'D', 'k', 'data_x', 'data_D', 'timings', 'debug_dict', 'converged', 'conv_int'):
        assert k_ in out, k_
    # bit-identical to the package's own host-protocol driver and to the device-resident driver
    ode2 = device_system(key, **kw)
    solver2 = nn.CudaSolverRK(ode2.get_vector_field(), **{k: cfg[k] for k in ("Ng", "Nf", "F", "G")})
    host = nn.Parareal(ode2, solver2, tspan=cfg["tspan"], N=N, epsilon=float(z["epsilon"]), verbose='') \
        .run(model='nngp', pool=nn.CudaPool(), parall='mpi', **mkw)
    assert K == host['k'] and out['conv_int'] == host['conv_int']
    assert np.array_equal(out['u'][:, :, K - 1], host['u'][:, :, K - 1])
    assert np.array_equal(out['err'], host['err'], equal_nan=True)
    dev = nn.PararealDevice(ode2, solver2, tspan=cfg["tspan"], N=N, epsilon=float(z["epsilon"]), verbose='') \
        .run(model='nngp', **mkw)
    assert K == dev['k'] and out['conv_int'] == dev['conv_int']
    # against the recorded run of the reference on its own NumPy path: same K where the run is not borderline
    if name != "hopf_N32_m15":
        assert K == int(z["K"])
    else:
        assert abs(K - int(z["K"])) <= 1


@needs_reference
def test_reference_plain_parareal_on_cuda_solver():
    """model='parareal' (BareParareal of the reference, models.py:74-83) with the CUDA solver and pool: the published
    Lorenz K = 15 (Table 2 of the reference)"""
    from integration.cuda_backend import bind
    B = bind()
    ode = B.Lorenz(normalization='-11')
    cfg = B.Config(ode).get()
    solver = B.CudaSolverRK(ode.get_vector_field(), **cfg)
    out = B.CudaParareal(ode, solver, verbose='', **cfg).run(model='parareal', pool=B.CudaPool(), parall='mpi')
    assert out['k'] == 15 and out['conv_int'] == [1, 2, 3, 5, 8, 14, 17, 20, 26, 30, 33, 37, 40, 43, 50]


@needs_reference
def test_checkpoints_cross_the_boundary_in_both_directions(tmp_path):
    """intermediate dumps (parareal.py:114-209, 420-431): (a) written by the REFERENCE driver running on the CUDA
    backend and resumed by the reference's own load_int_dump; (b) the same dump resumed by this package's driver;
    (c) a dump written by this package's driver resumed by the reference's load_int_dump.  All three end exactly
    like the uninterrupted run."""
    import pickle
    from integration.cuda_backend import bind
    from nearest_neighbors_gparareal_b200.checkpoint import load_dump
    B = bind()
    z, cfg, mkw = load_run("lorenz_N32_m11")
    rk = {k: cfg[k] for k in ("Ng", "Nf", "F", "G")}

    def ref_driver():
        ode = B.Lorenz(normalization="-11")
        return B.CudaParareal(ode, B.CudaSolverRK(ode.get_vector_field(), **rk), tspan=cfg["tspan"], N=cfg["N"],
                              epsilon=float(z["epsilon"]), verbose='')

    def pkg_driver():
        ode = nn.Lorenz(normalization="-11")
        return nn.Parareal(ode, nn.CudaSolverRK(ode.get_vector_field(), **rk), tspan=cfg["tspan"], N=cfg["N"],
                           epsilon=float(z["epsilon"]), verbose='')

    full = ref_driver().run(model='nngp', pool=B.CudaPool(), parall='mpi', **mkw)
    K = full['k']
    # (a) reference writes, reference resumes
    part = ref_driver().run(model='nngp', pool=B.CudaPool(), parall='mpi', early_stop=3, store_int=True,
                            int_dir=str(tmp_path), int_name='rf', **mkw)
    assert part['k'] == 3
    with open(tmp_path / 'rf' / 'rf_2', 'rb') as fh:
        dump = pickle.load(fh)
    assert isinstance(dump, B.ref.parareal.Parareal) and isinstance(dump.mdl, B.ref.models.NNGP_p)
    pa = ref_driver()
    ra = pa.load_int_dump(dump, ode=pa.ode, solver=pa.solver, pool=B.CudaPool(), early_stop=None, store_int=False)
    assert ra['k'] == K and ra['conv_int'] == full['conv_int']
    assert np.array_equal(ra['u'][:, :, K - 1], full['u'][:, :, K - 1])
    # (b) reference writes, this package resumes
    rb = pkg_driver().load_int_dump(load_dump(tmp_path / 'rf' / 'rf_2'), early_stop=None, store_int=False)
    assert rb['k'] == K and rb['conv_int'] == full['conv_int']
    assert np.array_equal(rb['u'][:, :, K - 1], full['u'][:, :, K - 1])   # the reference returns u^0 .. u^{K-1}
    # (c) this package writes, the reference resumes
    pkg_driver().run(model='nngp', pool=nn.CudaPool(), parall='mpi', early_stop=3, store_int=True,
                     int_dir=str(tmp_path), int_name='pk', **mkw)
    with open(tmp_path / 'pk' / 'pk_2', 'rb') as fh:
        dump_c = pickle.load(fh)
    pc = ref_driver()
    rc = pc.load_int_dump(dump_c, ode=pc.ode, solver=pc.solver, pool=B.CudaPool(), early_stop=None, store_int=False)
    assert rc['k'] == K and rc['conv_int'] == full['conv_int']
    assert np.array_equal(rc['u'][:, :, K - 1], full['u'][:, :, K - 1])
