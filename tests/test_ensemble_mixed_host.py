"""Host-side logic of ensembles whose members differ in neighbour count and time span (no GPU)."""
import os
import re

import numpy as np
import pytest

from nearest_neighbors_gparareal_b200 import _lib
from nearest_neighbors_gparareal_b200 import ensemble as ens
from nearest_neighbors_gparareal_b200.models import CudaNNGP
from nearest_neighbors_gparareal_b200.models_alt import CudaNNGPAlt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("kw,msg", [
    (dict(seeds=[1, 2], nn=[11]), "one per member"),
    (dict(seeds=[1, 2], nn=[11, 12, 13]), "one per member"),
    (dict(seeds=[1, 2], nn=[11, 0]), "160"),
    (dict(seeds=[1, 2], nn=['adaptive', 161]), "160"),
    (dict(seeds=[1, 2], nn=[11, 'fixed']), "adaptive"),
    (dict(seeds=[1, 2], nn=[11, 12.5]), "160"),
    (dict(seeds=[1, 2], tspans=[[0, 5]]), "one per member"),
    (dict(seeds=[1, 2], tspans=[[0, 5], [0, 0]]), "t1 > t0"),
    (dict(seeds=[1, 2], tspans=[None, [5.9, 5.0]]), "t1 > t0"),
])
def test_per_member_arguments_are_validated(kw, msg):
    nn = kw.pop('nn', 'adaptive')
    with pytest.raises(ValueError, match=msg):
        ens.check_run_args(kw, nn=nn)


def test_valid_per_member_arguments():
    assert ens.check_run_args(dict(seeds=[1, 2, 3], tspans=[None, [0, 5.0], [0, 5.9]]),
                              nn=['adaptive', 11, 160]) == 3
    assert ens.check_run_args(dict(seeds=[1, 2]), nn=np.array([11, 30])) == 2


def test_sweep_m_follows_the_member_order():
    m_members = [11, 12, 18, 30]
    I = np.array([3, 1, 2, 1])
    done = np.array([False, False, False, True])
    order = ens.member_order(I, done)
    sw = order[:3]  # running members in state order
    m_pos = ens.sweep_tables(m_members, sw)
    assert list(sw) == [1, 2, 0]
    assert list(m_pos) == [12, 18, 11] and m_pos.dtype == np.int32


class _StubHandle:
    """records what PararealEnsemble passes to the sweep"""

    def __init__(self):
        self.calls = []

    def ensemble_sweep(self, *args):
        self.calls.append(args)


def _sweep(models, t_members, sw, k=0, I_sw=None, listed_sw=None, lists=None):
    """launch_sweep over the members sw (state order) -> the arguments of the one Handle.ensemble_sweep call:
    [4] the grids, [8] the per-position m, [16] the listed flags, [17] the neighbour lists"""
    import torch
    h = _StubHandle()
    sw = np.asarray(sw)
    m_pos = ens.sweep_tables([mdl.neighbours(k) for mdl in models], sw)
    I_sw = np.zeros(sw.size, np.int64) if I_sw is None else I_sw
    listed_sw = np.zeros(sw.size, bool) if listed_sw is None else listed_sw
    lists = [None] * sw.size if lists is None else lists
    ens.launch_sweep(h, torch.from_numpy(t_members), 8, 4, 0, 1, 4, sw, I_sw, m_pos, listed_sw, lists, models[0], None,
                     None, None, 3, None)
    assert len(h.calls) == 1
    return h.calls[0]


def test_uniform_lists_reach_the_one_sweep():
    E = 4
    models = [CudaNNGP(n=3, N=4, seed=s, nn=v) for s, v in zip(range(E), [18] * E)]
    t = np.tile(np.linspace(0, 5.0, 5), (E, 1))
    sw = [2, 0, 3, 1]
    args = _sweep(models, t, sw)
    assert list(args[8]) == [18] * E and args[8].dtype == np.int32
    assert np.array_equal(args[4].numpy(), t[sw])
    assert args[16] is None and args[17] is None
    # 'adaptive' members at an iteration where they all use the same m
    models = [CudaNNGP(n=3, N=4, seed=s, nn='adaptive') for s in range(3)]
    args = _sweep(models, t[:3], [1, 2, 0], k=5)
    assert list(args[8]) == [models[0].neighbours(5)] * 3
    assert args[16] is None


def test_mixed_lists_reach_the_one_sweep():
    models = [CudaNNGP(n=3, N=4, seed=s, nn=v) for s, v in zip(range(3), ['adaptive', 11, 40])]
    t = np.stack([np.linspace(0, T, 5) for T in (5.0, 5.9, 5.0)])
    args = _sweep(models, t, [1, 2, 0], k=3)
    assert list(args[8]) == [11, 40, 10]
    assert np.array_equal(args[4].numpy(), t[[1, 2, 0]])
    assert args[16] is None
    # same nn, different time spans
    models = [CudaNNGP(n=3, N=4, seed=s, nn=11) for s in range(2)]
    t = np.stack([np.linspace(0, 5.0, 5), np.linspace(0, 5.9, 5)])
    args = _sweep(models, t, [1, 0])
    assert list(args[8]) == [11, 11]
    assert np.array_equal(args[4].numpy(), t[[1, 0]])


def test_listed_positions_pass_their_flags_and_lists():
    """state order [member 2 (rule 'row', I = 1), member 0 (kNN, I = 2), member 1 (rule 'row_col', I = 3)]"""
    N, cap = 8, 100
    models = [CudaNNGP(n=2, N=N, seed=45, nn=5), CudaNNGPAlt(n=2, N=N, seed=46, nn=4, nntype='row_col'),
              CudaNNGPAlt(n=2, N=N, seed=47, nn=6, nntype='row')]
    t = np.tile(np.linspace(0, 5.0, N + 1), (3, 1))
    sw, I_sw = np.array([2, 0, 1]), np.array([1, 2, 3])
    first = {0: [1], 1: [0, 2], 2: [0]}  # first unconverged slice of each iteration (the I of its sweep is one more)
    lists = [ens.listed_rows(models[e], e, first[e], I, e * cap) if e > 0 else None for e, I in zip(sw, I_sw)]
    args = _sweep(models, t, sw, I_sw=I_sw, listed_sw=np.array([True, False, True]), lists=lists)
    assert list(args[16]) == [True, False, True]
    assert list(args[8]) == [6, 5, 4]
    assert args[17][1] is None
    for p, e in ((0, 2), (2, 1)):
        block = args[17][p]
        assert block.shape == (N - I_sw[p], args[8][p]), (p, block.shape)
        assert block.min() >= e * cap and block.max() < (e + 1) * cap


def test_one_ensemble_sweep_entry_point_is_declared_and_bound():
    with open(os.path.join(ROOT, 'include', 'nngpara.h')) as f:
        header = f.read()
    for name in ('nngp_ensemble_sweep', 'nngp_fit_predict_mixed'):
        assert re.search(r'\bint\s+' + name + r'\(', header), name
        assert name in _lib.SIGNATURES
    for name in ('nngp_ensemble_sweep' + suffix for suffix in ('_mixed', '_listed')):  # the entry points it replaced
        assert name not in _lib.SIGNATURES
        for sub in ('include', os.path.join('nearest_neighbors_gparareal_b200', 'csrc')):
            for fn in os.listdir(os.path.join(ROOT, sub)):
                with open(os.path.join(ROOT, sub, fn)) as f:
                    assert name not in f.read(), (name, fn)
