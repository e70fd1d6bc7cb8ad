"""HJ value functions for the safety filter, computed on the GPU (liblsm_b200_hj.so, include/lsm_b200_hj.h).

The reference loads value functions that `hj_reachability` (JAX) computed offline. This module computes the same kind
of grid - the backward reachable tube of the filter's relative dynamics, WENO5 / global Lax-Friedrichs / TVD-RK3 in
float64, the declared scheme of DESIGN.md "HJ value functions" - with the project's own CUDA kernel, and wraps it as an
`HjGrid` that `B200GraphVecEnv(args, value_grid=...)` and `SafetyFilter(dynamics, value_grid=...)` accept.

    grid = reachability.value_grid('double_integrator')          # default lattice, 4 s horizon
    env = B200GraphVecEnv(args, value_grid=grid)
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._build import parse_dynamics
from .config import AirTaxiConfig, DoubleIntegratorConfig
from .hj_grid import (AIRTAXI_GRID_HI, AIRTAXI_GRID_LO, AIRTAXI_GRID_SHAPE, DI_GRID_HI, DI_GRID_LO, DI_GRID_SHAPE,
                      HjGrid, make_hj_handle)

NDIM = {0: 4, 1: 5}
PERIODIC = {0: (False,) * 4, 1: (False, False, True, False, False)}
# horizons after which the default lattices have converged (DESIGN.md "HJ value functions": max|V(H) - V(H/2)|)
DEFAULT_HORIZON = {0: 4.0, 1: 60.0}


def _problem(dyn: int, shape: Sequence[int], lo, hi, cfl: float) -> _lib.LsmHjProblem:
    nd = NDIM[dyn]
    shape, lo, hi = tuple(int(s) for s in shape), [float(x) for x in lo], [float(x) for x in hi]
    if len(shape) != nd or len(lo) != nd or len(hi) != nd:
        raise ValueError(f"dynamics {dyn} has {nd} dims: shape, lo and hi need {nd} entries each")
    pr = _lib.LsmHjProblem()
    pr.dynamics = dyn
    for d in range(nd):
        pr.shape[d], pr.lo[d], pr.hi[d] = shape[d], lo[d], hi[d]
    pr.cfl = float(cfl)
    return pr


def dissipation(dynamics, shape, lo, hi, cfl: float = 0.75):
    """The global Lax-Friedrichs coefficients (ndim float64) and the CFL time step of a lattice."""
    dyn = parse_dynamics(dynamics)
    pr = _problem(dyn, shape, lo, hi, cfl)
    lib = _lib.load_hj()
    alpha = (C.c_double * 5)()
    dt = C.c_double()
    _lib.check(lib.lsm_hj_dissipation(C.byref(pr), alpha, C.byref(dt)), 'lsm_hj_dissipation', lib)
    return np.array(alpha[:NDIM[dyn]], dtype=np.float64), float(dt.value)


def solve(dynamics, initial_values: torch.Tensor, lo, hi, horizons, cfl: float = 0.75) -> torch.Tensor:
    """V(tau) for each tau in `horizons` (non-decreasing, >= 0) of the backward reachable tube from V(0) =
    `initial_values` (a CUDA float64 tensor of the lattice's shape): float64 `(K, *shape)` on the same device. Runs on
    torch's current stream and does not synchronise."""
    dyn = parse_dynamics(dynamics)
    if not (isinstance(initial_values, torch.Tensor) and initial_values.is_cuda and initial_values.dtype == torch.float64):
        raise TypeError("initial_values must be a CUDA float64 tensor")
    pr = _problem(dyn, initial_values.shape, lo, hi, cfl)
    h = np.ascontiguousarray(np.atleast_1d(np.asarray(horizons, dtype=np.float64)))
    if h.ndim != 1 or h.size == 0:
        raise ValueError("horizons must be a non-empty 1-D sequence")
    lib = _lib.load_hj()
    dev = initial_values.device
    with torch.cuda.device(dev):
        init = initial_values.contiguous()
        nbytes = lib.lsm_hj_work_bytes(C.byref(pr))
        if nbytes <= 0:
            _lib.check(2, 'lsm_hj_work_bytes', lib)
        work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty((h.size,) + tuple(init.shape), dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.lsm_hj_solve(C.byref(pr), C.c_void_p(init.data_ptr()), h.ctypes.data_as(C.POINTER(C.c_double)),
                              int(h.size), C.c_void_p(out.data_ptr()), C.c_void_p(work.data_ptr()), C.c_void_p(stream))
        _lib.check(rc, 'lsm_hj_solve', lib)
    return out


def target(dynamics, shape, lo, hi, separation_distance: float) -> np.ndarray:
    """l(x) = sqrt(x0^2 + x1^2) - separation_distance on the lattice (float64; positive = safe)."""
    dyn = parse_dynamics(dynamics)
    g = HjGrid(lo=np.asarray(lo, np.float64), hi=np.asarray(hi, np.float64), shape=tuple(int(s) for s in shape),
               periodic=PERIODIC[dyn], values=None)
    x0, x1 = g.coordinate_vectors()[:2]
    x0 = x0.reshape((-1,) + (1,) * (g.ndim - 1))
    x1 = x1.reshape((1, -1) + (1,) * (g.ndim - 2))
    return np.broadcast_to(np.sqrt(x0 * x0 + x1 * x1) - float(separation_distance), g.shape).copy()


def value_grid(dynamics, separation_distance: Optional[float] = None, shape=None, lo=None, hi=None,
               horizon: Optional[float] = None, target_separation_distance: Optional[float] = None) -> HjGrid:
    """A computed value function as the `HjGrid` the environment and `SafetyFilter` consume. Solves the tube of
    l(x) = |x[:2]| - separation_distance to `horizon` on the lattice (defaults: the dynamics' separation distance, the
    DI_GRID_* / AIRTAXI_GRID_* lattice, 4 s / 60 s) and stores it the way the reference's value-function files do
    (stored = -V, hj_grid.make_hj_handle), so the filter sees it at `target_separation_distance` (default: the
    separation distance it was solved for). Solves on the current CUDA device."""
    dyn = parse_dynamics(dynamics)
    if separation_distance is None:
        separation_distance = (DoubleIntegratorConfig if dyn == 0 else AirTaxiConfig).SEPARATION_DISTANCE
    shape = tuple(shape if shape is not None else (DI_GRID_SHAPE if dyn == 0 else AIRTAXI_GRID_SHAPE))
    lo = lo if lo is not None else (DI_GRID_LO if dyn == 0 else AIRTAXI_GRID_LO)
    hi = hi if hi is not None else (DI_GRID_HI if dyn == 0 else AIRTAXI_GRID_HI)
    horizon = DEFAULT_HORIZON[dyn] if horizon is None else float(horizon)
    if target_separation_distance is None:
        target_separation_distance = separation_distance
    dev = torch.device('cuda', torch.cuda.current_device())
    l = torch.as_tensor(target(dyn, shape, lo, hi, separation_distance), device=dev)
    v = solve(dyn, l, lo, hi, [horizon])[0].cpu().numpy()
    return make_hj_handle(-v, lo, hi, PERIODIC[dyn], separation_distance, target_separation_distance)
