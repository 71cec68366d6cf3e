"""Host-side logic of PararealEnsemble (no GPU): packing of the Nelder-Mead starts, member bookkeeping, validation."""
import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import ensemble as ens
from nearest_neighbors_gparareal_b200.models import CudaNNGP


def test_pack_starts_keeps_each_members_solo_draw_order():
    """slice-major packing; member p's blocks are its solo draw_starts(N - I_p) in order, one per slice it sweeps"""
    N, d, R = 9, 3, 2
    I_pos = [2, 2, 5, 8]
    models = [CudaNNGP(n=d, N=N, seed=s, nn=11, n_restarts=R) for s in (45, 46, 47, 48)]
    blocks = [mdl.draw_starts(N - I) for mdl, I in zip(models, I_pos)]
    packed = ens.pack_starts(blocks, I_pos, N)
    assert packed.shape == (sum(N - I for I in I_pos), d, 9, R, 2) and packed.dtype == np.int8
    at = 0
    for i in range(min(I_pos), N):
        for p, I in enumerate(I_pos):
            if I <= i:
                assert np.array_equal(packed[at], blocks[p][i - I])
                at += 1
    # the solo run draws the same blocks from the same seed
    for p, (s, I) in enumerate(zip((45, 46, 47, 48), I_pos)):
        solo = CudaNNGP(n=d, N=N, seed=s, nn=11, n_restarts=R).draw_starts(N - I)
        assert np.array_equal(solo, blocks[p])


def test_member_order_running_first_by_I():
    I = np.array([4, 1, 7, 1, 9, 3])
    done = np.array([False, False, True, False, False, True])
    order = ens.member_order(I, done)
    assert list(order) == [1, 3, 0, 4, 5, 2]  # running by (I, position), then the finished ones
    assert list(ens.member_order(np.array([2, 2, 2]), np.zeros(3, bool))) == [0, 1, 2]


def test_fine_rows_cover_each_running_members_unconverged_slices():
    N = 6
    rows, sl = ens.fine_rows([0, 3, 6], N)
    assert list(sl) == [0, 1, 2, 3, 4, 5, 3, 4, 5]
    assert list(rows) == [0, 1, 2, 3, 4, 5, 7 + 3, 7 + 4, 7 + 5]
    assert ens.fine_rows([], N)[0].size == 0


def test_advance_matches_the_solo_rule():
    eps = 1e-6
    err = np.array([0.0, 5.0, 1e-7, 1e-8, 2e-6, 1e-9])
    e = err.copy()
    assert ens.advance(e, 1, eps) == 3 and e[1] == 0.0  # slices 2, 3 below eps, 4 is not
    e = np.array([0.0, 0.0, 9.0, 1e-9])
    assert ens.advance(e, 2, eps) == 3  # I = N - 1 -> N: converged
    e = np.array([0.0, 1.0, np.nan, 0.0])
    assert ens.advance(e, 0, eps) == 0  # NaN never converges


@pytest.mark.parametrize("kw,msg", [
    (dict(seeds=[]), "non-empty"),
    (dict(seeds=None), "non-empty"),
    (dict(seeds=[1, 2], epsilons=[1e-6]), "one per member"),
    (dict(seeds=[1, 2], early_stops=[1, 2, 3]), "one per member"),
    (dict(seeds=[1, 2], init_conds=[None]), "one per member"),
    (dict(seeds=[1], store_int=True), "store_int"),
    (dict(seeds=[1], model='parareal'), "'nngp' model only"),
    (dict(seeds=[1], model='gpjax'), "'nngp' model only"),
    (dict(seeds=[1], nn=161), "160"),
])
def test_run_rejects_what_cannot_run_as_one_launch_per_slice(kw, msg):
    ode = nn.Lorenz(normalization='-11')
    solver = nn.CudaSolverRK(ode.get_vector_field(), Ng=6, Nf=450, G='RK4', F='RK4')
    e = nn.PararealEnsemble(ode, solver, tspan=[0, 18], N=50, verbose='')
    with pytest.raises(ValueError, match=msg):
        e.run(**kw)


def test_run_rejects_an_unknown_argument():
    """e.g. the solo run's early_stop: the ensemble takes early_stops, one per member"""
    ode = nn.Lorenz(normalization='-11')
    solver = nn.CudaSolverRK(ode.get_vector_field(), Ng=6, Nf=450, G='RK4', F='RK4')
    with pytest.raises(TypeError):
        nn.PararealEnsemble(ode, solver, tspan=[0, 18], N=50, verbose='').run(seeds=[1], early_stop=3)


def test_constructor_needs_the_device_solver():
    ode = nn.Lorenz(normalization='-11')
    with pytest.raises(Exception, match="CudaSolverRK"):
        nn.PararealEnsemble(ode, object(), tspan=[0, 18], N=50)
