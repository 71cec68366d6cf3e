"""rk_fhn_tile_kernel's alternating left / right column-load order (csrc/rk.cu), in the shapes no other test reaches:
grids whose half width d_x / 2 is not a power of two, so that warps cover partial block rows and a block row starts at
any lane, and the production fine step of 512 slices as its chunked launch sequence."""
import os

import numpy as np
import pytest

import nearest_neighbors_gparareal_b200 as nn
from oracle import rk as ork
from oracle import systems as osys
from helpers import scaled_err

pytestmark = pytest.mark.gpu

METHODS = (("RK1", 6), ("RK2", 5), ("RK4", 4), ("RK8", 3))


def _sms(handle):
    import torch
    return torch.cuda.get_device_properties(handle.device).multi_processor_count


def _run(handle, s, t0, t1, u0, **env):
    """run_F_batch under the given csrc/rk.cu environment switches: (result, kernel launches)"""
    keys = ("NNGP_RK_TILE", "NNGP_RK_NO_SHFL", "NNGP_RK_CHUNKS")
    try:
        for k in keys:
            os.environ.pop(k, None)
        os.environ.update(env)
        c0 = handle.launch_count()
        out = s.run_F_batch(t0, t1, u0)
        return out, handle.launch_count() - c0
    finally:
        for k in keys:
            os.environ.pop(k, None)


@pytest.mark.parametrize("d_x", [12, 20])
def test_fhn_partial_row_warps_equal_point_kernel(handle, d_x):
    """d_x = 12 and 20 (block rows of 6 and 10 lanes): the 2x2 (TY = 2) and 1x2 (TY = 1) blocks, which here always use
    shared-memory column loads, give the bits of the one-point-per-thread kernel (NNGP_RK_TILE = 0) for every RK method,
    at 1 and sms + 1 slices, and stay within 1e-12 (scaled) of the NumPy oracle."""
    rng = np.random.default_rng(400 + d_x)
    o, dev = osys.FHN_PDE(d_x=d_x), nn.FHN_PDE(d_x=d_x)
    for n in (1, _sms(handle) + 1):
        u0 = dev.get_init_cond()[None, :] + 0.01 * rng.standard_normal((n, dev.get_dim()))
        t0 = np.arange(n) * 0.01
        t1 = t0 + 0.05
        for F, steps in METHODS:
            s = nn.CudaSolverRK(dev.get_vector_field(), Ng=1, Nf=steps, F=F, G='RK1', handle=handle)
            ref, _ = _run(handle, s, t0, t1, u0, NNGP_RK_TILE="0")
            for tile in ("1", "2"):
                got, nl = _run(handle, s, t0, t1, u0, NNGP_RK_TILE=tile)
                assert nl == 1
                assert np.array_equal(got, ref), (n, F, tile)
            for i in sorted({0, n - 1}):
                assert scaled_err(ref[i], ork.rk_last(o.f, F, t0[i], t1[i], steps, u0[i])) < 1e-12, (n, F, i)


def _chunked_launches(n, sms):
    """launches of launch_fhn_tile_x's chunked sequence: 2 CTAs per SM, the smallest chunk count >= 24 that fills the
    last launch, else 32"""
    per_launch = 2 * sms
    chunks = next((c for c in range(24, 65) if (n * c) % per_launch == 0), 32)
    return -(-n * chunks // per_launch)


def test_fhn_production_fine_step_chunked_equals_single_launch(handle):
    """The fine step of the benchmarked target, 512 slices at d_x = 16 with >= 4096 steps, runs as the chunked launch
    sequence (64 launches on 148 SMs) and returns the bits of the single launch (NNGP_RK_CHUNKS = 0), both step
    conventions."""
    sms = _sms(handle)
    n = 512
    if n <= 2 * sms:
        pytest.skip(f"{sms} SMs hold 512 slices in one balanced launch")
    rng = np.random.default_rng(512)
    dev = nn.FHN_PDE(d_x=16)
    u0 = dev.get_init_cond()[None, :] + 0.01 * rng.standard_normal((n, dev.get_dim()))
    t0 = rng.uniform(0, 1, n)
    t1 = t0 + rng.uniform(0.5, 1.5, n)
    for h_mode in ("linspace", "const"):
        s = nn.CudaSolverRK(dev.get_vector_field(), Ng=1, Nf=4100, F='RK8', G='RK1', h_mode=h_mode, handle=handle)
        got, nl = _run(handle, s, t0, t1, u0)
        assert nl == _chunked_launches(n, sms), nl
        ref, nl0 = _run(handle, s, t0, t1, u0, NNGP_RK_CHUNKS="0")
        assert nl0 == 1
        assert np.all(np.isfinite(got)) and np.array_equal(got, ref), h_mode
