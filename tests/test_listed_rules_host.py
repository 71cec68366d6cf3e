"""Host side of the position-based neighbour rules on the device drivers (no GPU): the neighbour lists the drivers
build from their per-iteration first rows equal the host driver's choice, and what cannot run is refused up front."""
import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from nearest_neighbors_gparareal_b200 import ensemble as ens
from nearest_neighbors_gparareal_b200.models import CudaNNGP
from nearest_neighbors_gparareal_b200.models_alt import NNTYPES, CudaNNGPAlt

RULES = [r for r in NNTYPES if r != 'nn']


def _host_fit(self, x, y, k, *args, **kwargs):
    """CudaNNGP.fit without the device upload (models.py:157-159 keeps x, y, k)"""
    self.k, self.x, self.y = k, x, y


def _cube(first, N, d, rng):
    """the host driver's data_x after iterations 0 .. len(first)-1: column j holds slices first[j] .. N-1"""
    data_x = np.full((N, d, N), np.nan)
    for j, f in enumerate(first):
        data_x[f:, :, j] = rng.standard_normal((N - f, d))
    return data_x


@pytest.mark.parametrize("rule", RULES)
@pytest.mark.parametrize("first", [[0, 1, 1, 4, 6], [0, 3, 3, 3, 9, 10]])
def test_device_tables_equal_the_host_drivers_rows(monkeypatch, rule, first):
    """converged prefixes that move between iterations; the table of every iteration (built from the first rows only)
    equals neighbour_rows(i) slice by slice after fit(data_x=...), and col+rnd's rng2 carries over iterations"""
    monkeypatch.setattr(CudaNNGP, 'fit', _host_fit)
    N, d, nn_ = 14, 3, 6
    host = CudaNNGPAlt(n=d, N=N, nn=nn_, nntype=rule, seed=45)
    dev = CudaNNGPAlt(n=d, N=N, nn=nn_, nntype=rule, seed=45)
    rng = np.random.default_rng(0)
    for k in range(len(first)):
        I = first[k] + 1  # the sweep of iteration k starts after the slice its fine step made exact
        data_x = _cube(first[:k + 1], N, d, rng)
        n_rows = sum(N - f for f in first[:k + 1])
        host.fit(np.zeros((n_rows, d)), np.zeros((n_rows, d)), k, data_x=data_x)
        want = np.array([host.neighbour_rows(i) for i in range(I, N)], dtype=np.int64)
        got = dev.neighbour_table(first[:k + 1], I)
        assert got.dtype == np.int64 and got.shape == (N - I, k + 1 if rule == 'col_only' else nn_)
        assert np.array_equal(got, want), (rule, k)
        assert got.min() >= 0 and got.max() < n_rows
    assert host.rng2.bit_generator.state == dev.rng2.bit_generator.state


def test_listed_rows_are_global_and_a_shortage_names_the_member():
    mdl = CudaNNGPAlt(n=2, N=8, nn=5, nntype='row', seed=46)
    tab = ens.listed_rows(mdl, 3, [0], 1, 3 * 100)
    ref = CudaNNGPAlt(n=2, N=8, nn=5, nntype='row', seed=46).neighbour_table([0], 1)
    assert np.array_equal(tab, ref + 300)
    # iteration 0 of N = 4 holds 4 observations, fewer than nn = 16
    short = CudaNNGPAlt(n=2, N=4, nn=16, nntype='col_full', seed=45)
    with pytest.raises(ValueError, match=r"member 2: .*only 4 observations for nn=16"):
        ens.listed_rows(short, 2, [0], 1, 0)


@pytest.mark.parametrize("kw,msg", [
    (dict(seeds=[1, 2], nn=16, nntype='rows'), "member 0: unknown nntype 'rows'"),
    (dict(seeds=[1, 2], nn=16, nntype=['row', 'colonly']), "member 1: unknown nntype"),
    (dict(seeds=[1, 2], nn=16, nntype=['row']), "nntype has 1 entries"),
    (dict(seeds=[1, 2], nn=16, nntype=['row', 'nn', 'col_only']), "nntype has 3 entries"),
    (dict(seeds=[1, 2], nntype=['nn', 'row_col']), "member 1: .*integer nn"),
])
def test_ensemble_rules_are_validated_before_any_device_call(kw, msg):
    """PararealEnsemble.run refuses before it creates a handle (this machine may have no GPU at all)"""
    ode = nn.Lorenz(normalization='-11')
    solver = nn.CudaSolverRK(ode.get_vector_field(), Ng=6, Nf=450, G='RK4', F='RK4')
    e = nn.PararealEnsemble(ode, solver, tspan=[0, 18], N=50, verbose='')
    with pytest.raises(ValueError, match=msg):
        e.run(**kw)
    assert e._h is None


def test_valid_rules():
    assert ens.check_run_args(dict(seeds=[1, 2, 3]), nn=[16, 'adaptive', 16],
                              nntype=['row', 'col+rnd', 'nn']) == 3
    assert ens.check_run_args(dict(seeds=[1, 2]), nn=16, nntype='col_full') == 2
