"""nearest_neighbors_gparareal_b200 -- B200 (sm_100a) implementation of the nnGParareal hot path.

Host-side mirror of the reference's Python surface (parareal.py / models.py / solver.py /
systems.py / configs.py / utils.py) over the C ABI of libnngpara.so (include/nngpara.h):
hand-written CUDA kernels for the batched explicit RK propagators, the exact FP64 kNN and the
per-slice / per-dimension GP fit + predict.  There is NO CPU fallback: importing the device
classes without the built library, or creating a handle without a Blackwell GPU, raises.
"""
from .utils import Normalize
from .systems import (ODE, FHN_ODE, Rossler, Hopf, DblPend, Brusselator, Lorenz, ThomasLabyrinth,
                      FHN_PDE, Burgers)
from .configs import Config
from .solver import SolverAbstr, CudaSolverRK, SolverRK
from .models import ModelAbstr, BareParareal, CudaNNGP, NNGP_p
from .gp_full import CudaGP, GPjax_p
from .pool import MyPool, CudaPool
from .parareal import Parareal, PararealLight, PararealDevice
from .ensemble import PararealEnsemble

__all__ = ["Normalize", "ODE", "FHN_ODE", "Rossler", "Hopf", "DblPend", "Brusselator", "Lorenz",
           "ThomasLabyrinth", "FHN_PDE", "Burgers", "Config", "SolverAbstr", "CudaSolverRK",
           "SolverRK", "ModelAbstr", "BareParareal", "CudaNNGP", "NNGP_p", "CudaGP", "GPjax_p", "MyPool", "CudaPool",
           "Parareal", "PararealLight", "PararealDevice", "PararealEnsemble"]
