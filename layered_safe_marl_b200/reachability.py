"""HJ value functions for the safety filter, computed on the GPU (liblsm_b200_hj.so, include/lsm_b200_hj.h).

The reference loads value functions that `hj_reachability` (JAX) computed offline. This module computes the same kind
of grid - the backward reachable tube of the filter's relative dynamics, WENO5 / global Lax-Friedrichs / TVD-RK3 in
float64, the declared scheme of DESIGN.md "HJ value functions" - with the project's own CUDA kernel, and wraps it as an
`HjGrid` that `B200GraphVecEnv(args, value_grid=...)` and `SafetyFilter(dynamics, value_grid=...)` accept.

    grid = reachability.value_grid('double_integrator')          # default lattice, 4 s horizon
    env = B200GraphVecEnv(args, value_grid=grid)

`game` chooses what the other agent of the pair does (DESIGN.md "HJ value functions"): 'cooperative' (the default,
the reference's game: it plays its part of the avoidance manoeuvre), 'adversarial' (it does its worst: the value the
ego alone can guarantee) or 'constant' (it holds its controls at 0: traffic that runs no filter).

    grid = reachability.value_grid('airtaxi', game='adversarial')

It also computes the airtaxi time-to-reach grid the reward looks up (DESIGN.md "Time-to-reach grid"): the same scheme
on a reach problem to the goal, with first-arrival times taken during the solve.

    env = B200GraphVecEnv(args, ttr_grid=reachability.ttr_grid())
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._build import parse_dynamics
from .config import AirTaxiConfig, DoubleIntegratorConfig
from .hj_grid import (AIRTAXI_GRID_HI, AIRTAXI_GRID_LO, AIRTAXI_GRID_SHAPE, DI_GRID_HI, DI_GRID_LO, DI_GRID_SHAPE,
                      TTR_GRID_HI, TTR_GRID_LO, TTR_GRID_SHAPE, HjGrid, make_hj_handle)

NDIM = {0: 4, 1: 5}
PERIODIC = {0: (False,) * 4, 1: (False, False, True, False, False)}
# horizons after which the default lattices have converged (DESIGN.md "HJ value functions": max|V(H) - V(H/2)|)
DEFAULT_HORIZON = {0: 4.0, 1: 60.0}
# the games of lsm_hj_game_solve (include/lsm_b200_hj.h)
GAMES = {'cooperative': 0, 'adversarial': 1, 'constant': 2}
TTR_PERIODIC = (False, False, True, False)
# horizon of the default TTR lattice: every cell more than 2 km inside the x/y boundary is reached by then
# (DESIGN.md "Time-to-reach grid")
DEFAULT_TTR_HORIZON = 300.0


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


@contextlib.contextmanager
def _on_device(lib, work_bytes: str, pr, values: torch.Tensor):
    """On `values`' device: (`values` made contiguous, the work buffer `work_bytes` sizes for `pr`, the handle of
    torch's current stream) for one solve."""
    dev = values.device
    with torch.cuda.device(dev):
        nbytes = getattr(lib, work_bytes)(C.byref(pr))
        if nbytes <= 0:
            _lib.check(2, work_bytes, lib)
        yield (values.contiguous(), torch.empty(nbytes, dtype=torch.uint8, device=dev),
               torch.cuda.current_stream(dev).cuda_stream)


def parse_game(game) -> int:
    """'cooperative' / 'adversarial' / 'constant' or its code 0 / 1 / 2 -> the code."""
    if isinstance(game, str):
        if game not in GAMES:
            raise ValueError(f"unknown game {game!r}: one of {sorted(GAMES)}")
        return GAMES[game]
    if isinstance(game, (int, np.integer)) and not isinstance(game, bool) and int(game) in GAMES.values():
        return int(game)
    raise ValueError(f"unknown game {game!r}: one of {sorted(GAMES)} or its code 0, 1, 2")


def dissipation(dynamics, shape, lo, hi, cfl: float = 0.75, game='cooperative'):
    """The global Lax-Friedrichs coefficients (ndim float64) and the CFL time step of a lattice for a game."""
    dyn = parse_dynamics(dynamics)
    g = parse_game(game)
    pr = _problem(dyn, shape, lo, hi, cfl)
    lib = _lib.load_hj()
    alpha = (C.c_double * 5)()
    dt = C.c_double()
    _lib.check(lib.lsm_hj_game_dissipation(C.byref(pr), g, alpha, C.byref(dt)), 'lsm_hj_game_dissipation', lib)
    return np.array(alpha[:NDIM[dyn]], dtype=np.float64), float(dt.value)


def solve(dynamics, initial_values: torch.Tensor, lo, hi, horizons, cfl: float = 0.75,
          game='cooperative') -> torch.Tensor:
    """V(tau) for each tau in `horizons` (non-decreasing, >= 0) of the backward reachable tube from V(0) =
    `initial_values` (a CUDA float64 tensor of the lattice's shape) in `game` (GAMES): float64 `(K, *shape)` on the
    same device. Runs on torch's current stream and does not synchronise."""
    dyn = parse_dynamics(dynamics)
    g = parse_game(game)
    if not (isinstance(initial_values, torch.Tensor) and initial_values.is_cuda and initial_values.dtype == torch.float64):
        raise TypeError("initial_values must be a CUDA float64 tensor")
    pr = _problem(dyn, initial_values.shape, lo, hi, cfl)
    h = np.ascontiguousarray(np.atleast_1d(np.asarray(horizons, dtype=np.float64)))
    if h.ndim != 1 or h.size == 0:
        raise ValueError("horizons must be a non-empty 1-D sequence")
    lib = _lib.load_hj()
    with _on_device(lib, 'lsm_hj_work_bytes', pr, initial_values) as (init, work, stream):
        out = torch.empty((h.size,) + tuple(init.shape), dtype=torch.float64, device=init.device)
        rc = lib.lsm_hj_game_solve(C.byref(pr), g, C.c_void_p(init.data_ptr()), h.ctypes.data_as(C.POINTER(C.c_double)),
                                   int(h.size), C.c_void_p(out.data_ptr()), C.c_void_p(work.data_ptr()),
                                   C.c_void_p(stream))
        _lib.check(rc, 'lsm_hj_game_solve', lib)
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
               horizon: Optional[float] = None, target_separation_distance: Optional[float] = None,
               game='cooperative') -> HjGrid:
    """A computed value function as the `HjGrid` the environment and `SafetyFilter` consume. Solves the tube of
    l(x) = |x[:2]| - separation_distance in `game` (GAMES) to `horizon` on the lattice (defaults: the dynamics'
    separation distance, the DI_GRID_* / AIRTAXI_GRID_* lattice, 4 s / 60 s for every game) and stores it the way the
    reference's value-function files do (stored = -V, hj_grid.make_hj_handle), so the filter sees it at
    `target_separation_distance` (default: the separation distance it was solved for). Solves on the current CUDA
    device."""
    dyn = parse_dynamics(dynamics)
    g = parse_game(game)
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
    v = solve(dyn, l, lo, hi, [horizon], game=g)[0].cpu().numpy()
    return make_hj_handle(-v, lo, hi, PERIODIC[dyn], separation_distance, target_separation_distance)


def _ttr_problem(shape: Sequence[int], lo, hi, cfl: float) -> _lib.LsmHjTtrProblem:
    shape, lo, hi = tuple(int(s) for s in shape), [float(x) for x in lo], [float(x) for x in hi]
    if len(shape) != 4 or len(lo) != 4 or len(hi) != 4:
        raise ValueError("the time-to-reach lattice has 4 dims [x, y, theta, v]: shape, lo and hi need 4 entries each")
    pr = _lib.LsmHjTtrProblem()
    for d in range(4):
        pr.shape[d], pr.lo[d], pr.hi[d] = shape[d], lo[d], hi[d]
    pr.cfl = float(cfl)
    return pr


def ttr_dissipation(shape, lo, hi, cfl: float = 0.75):
    """The time-to-reach solve's Lax-Friedrichs coefficients (4 float64) and CFL time step on a lattice."""
    pr = _ttr_problem(shape, lo, hi, cfl)
    lib = _lib.load_hj()
    alpha = (C.c_double * 4)()
    dt = C.c_double()
    _lib.check(lib.lsm_hj_ttr_dissipation(C.byref(pr), alpha, C.byref(dt)), 'lsm_hj_ttr_dissipation', lib)
    return np.array(alpha[:], dtype=np.float64), float(dt.value)


def solve_ttr(target: torch.Tensor, lo, hi, horizon: float, cfl: float = 0.75):
    """Time-to-reach of the target set {target <= 0} (a CUDA float64 tensor on the [x, y, theta, v] lattice) up to
    `horizon`: `(ttr, V(horizon))`, float64 tensors of the lattice's shape on the same device; ttr is +inf where the
    target is not reached by the horizon. Runs on torch's current stream and does not synchronise."""
    if not (isinstance(target, torch.Tensor) and target.is_cuda and target.dtype == torch.float64):
        raise TypeError("target must be a CUDA float64 tensor")
    pr = _ttr_problem(target.shape, lo, hi, cfl)
    lib = _lib.load_hj()
    with _on_device(lib, 'lsm_hj_ttr_work_bytes', pr, target) as (l, work, stream):
        ttr = torch.empty_like(l)
        V = torch.empty_like(l)
        rc = lib.lsm_hj_ttr_solve(C.byref(pr), C.c_void_p(l.data_ptr()), float(horizon), C.c_void_p(ttr.data_ptr()),
                                  C.c_void_p(V.data_ptr()), C.c_void_p(work.data_ptr()), C.c_void_p(stream))
        _lib.check(rc, 'lsm_hj_ttr_solve', lib)
    return ttr, V


def ttr_target(shape, lo, hi, goal_radius: float = AirTaxiConfig.DISTANCE_TO_GOAL_THRESHOLD,
               heading_threshold: Optional[float] = AirTaxiConfig.GOAL_HEADING_THRESHOLD) -> np.ndarray:
    """The goal set as l(x) <= 0 on the [x, y, theta, v] lattice (float64): max(sqrt(x^2 + y^2) - r,
    (r / h) ((0.5 - 0.5 cos theta) - h)) with h = 0.5 - 0.5 cos(heading_threshold), the position and heading tests of
    the airtaxi goal check. `heading_threshold=None` gives the position-only target sqrt(x^2 + y^2) - r. The goal-speed
    test has no axis on this lattice."""
    g = HjGrid(lo=np.asarray(lo, np.float64), hi=np.asarray(hi, np.float64), shape=tuple(int(s) for s in shape),
               periodic=TTR_PERIODIC, values=None)
    if g.ndim != 4:
        raise ValueError("the time-to-reach lattice has 4 dims [x, y, theta, v]")
    x, y, th, _ = g.coordinate_vectors()
    r = float(goal_radius)
    l = np.sqrt(x[:, None, None, None] ** 2 + y[None, :, None, None] ** 2) - r
    if heading_threshold is not None:
        h = 0.5 - 0.5 * math.cos(float(heading_threshold))
        l = np.maximum(l, (r / h) * ((0.5 - 0.5 * np.cos(th[None, None, :, None])) - h))
    return np.broadcast_to(l, g.shape).copy()


def ttr_grid(shape=TTR_GRID_SHAPE, lo=TTR_GRID_LO, hi=TTR_GRID_HI, horizon: float = DEFAULT_TTR_HORIZON,
             ttr_max: Optional[float] = None, goal_radius: float = AirTaxiConfig.DISTANCE_TO_GOAL_THRESHOLD,
             heading_threshold: Optional[float] = AirTaxiConfig.GOAL_HEADING_THRESHOLD, cfl: float = 0.75) -> HjGrid:
    """A computed airtaxi time-to-reach grid as the `HjGrid` `B200GraphVecEnv(args, ttr_grid=...)` takes, laid out like
    `hj_grid.load_reference_ttr_pickle`'s (float32 values, no gradients, theta periodic). Solves the reach problem of
    `ttr_target(...)` to `horizon` on the current CUDA device; cells not reached by then hold `ttr_max` (default: the
    horizon), which is also the reward's value for states off the lattice."""
    ttr_max = float(horizon) if ttr_max is None else float(ttr_max)
    dev = torch.device('cuda', torch.cuda.current_device())
    l = torch.as_tensor(ttr_target(shape, lo, hi, goal_radius, heading_threshold), device=dev)
    t = solve_ttr(l, lo, hi, horizon, cfl)[0].cpu().numpy()
    values = np.where(np.isinf(t), ttr_max, t).astype(np.float32)
    return HjGrid(lo=np.asarray(lo, np.float64), hi=np.asarray(hi, np.float64), shape=tuple(values.shape),
                  periodic=TTR_PERIODIC, values=values, grads=None, separation_distance=0.0, ttr_max=ttr_max)
