"""Host-side logic of ensembles whose members differ in neighbour count and time span (no GPU)."""
import os
import re

import numpy as np
import pytest

from nearest_neighbors_gparareal_b200 import _lib
from nearest_neighbors_gparareal_b200 import ensemble as ens
from nearest_neighbors_gparareal_b200.models import CudaNNGP

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


def test_sweep_tables_follow_the_member_order():
    m_members = [11, 12, 18, 30]
    t_members = np.stack([np.linspace(0, T, 5) for T in (5.0, 5.9, 5.0, 5.9)])
    I = np.array([3, 1, 2, 1])
    done = np.array([False, False, False, True])
    order = ens.member_order(I, done)
    sw = order[:3]  # running members in state order
    m_pos, t_pos = ens.sweep_tables(m_members, t_members, sw)
    assert list(sw) == [1, 2, 0]
    assert list(m_pos) == [12, 18, 11] and m_pos.dtype == np.int32
    assert np.array_equal(t_pos, t_members[[1, 2, 0]]) and t_pos.flags['C_CONTIGUOUS']


class _StubHandle:
    """records which sweep entry point PararealEnsemble calls"""

    def __init__(self):
        self.calls = []

    def ensemble_sweep(self, *args):
        self.calls.append(('ensemble_sweep', args))

    def ensemble_sweep_mixed(self, *args):
        self.calls.append(('ensemble_sweep_mixed', args))


def _sweep(models, t_members, k=0):
    import torch
    h = _StubHandle()
    sw = np.arange(len(models))
    m_pos, t_pos = ens.sweep_tables([mdl.neighbours(k) for mdl in models], t_members, sw)
    ens.launch_sweep(h, torch.from_numpy(t_members), 8, 4, 0, 1, 4, sw, np.zeros(len(models), np.int64), m_pos, t_pos, models[0], None,
                     None, None, 3, None)
    assert len(h.calls) == 1
    return h.calls[0]


def test_uniform_lists_take_the_unchanged_sweep():
    E = 4
    models = [CudaNNGP(n=3, N=4, seed=s, nn=v) for s, v in zip(range(E), [18] * E)]
    t = np.tile(np.linspace(0, 5.0, 5), (E, 1))
    name, args = _sweep(models, t)
    assert name == 'ensemble_sweep'
    assert args[8] == 18  # the scalar m of nngp_ensemble_sweep
    assert np.array_equal(args[4].numpy(), t[0])
    # 'adaptive' members at an iteration where they all use the same m
    name, _ = _sweep([CudaNNGP(n=3, N=4, seed=s, nn='adaptive') for s in range(3)], t[:3], k=5)
    assert name == 'ensemble_sweep'


def test_mixed_lists_take_the_mixed_sweep():
    models = [CudaNNGP(n=3, N=4, seed=s, nn=v) for s, v in zip(range(3), ['adaptive', 11, 40])]
    t = np.tile(np.linspace(0, 5.0, 5), (3, 1))
    name, args = _sweep(models, t, k=3)
    assert name == 'ensemble_sweep_mixed'
    assert list(args[8]) == [10, 11, 40]
    # same nn, different time spans
    models = [CudaNNGP(n=3, N=4, seed=s, nn=11) for s in range(2)]
    t = np.stack([np.linspace(0, 5.0, 5), np.linspace(0, 5.9, 5)])
    name, args = _sweep(models, t)
    assert name == 'ensemble_sweep_mixed'
    assert np.array_equal(args[4].numpy(), t)


def test_new_entry_points_are_declared_and_bound():
    with open(os.path.join(ROOT, 'include', 'nngpara.h')) as f:
        header = f.read()
    for name in ('nngp_ensemble_sweep_mixed', 'nngp_fit_predict_mixed'):
        assert re.search(r'\bint\s+' + name + r'\(', header), name
        assert name in _lib.SIGNATURES
