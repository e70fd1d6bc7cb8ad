"""Regular-grid value functions for the HJ safety filter and the airtaxi TTR reward.

Host-side mirror of `HjDataHandle` (reference `multiagent/safety_filter.py:154-174`) and of
the TTR loading in `make_world` (reference `navigation_graph_safe.py:128-138`).

The reference unpickles Drive-hosted grids (`data/*.pkl`, reference README.md:80-81) that are
not available offline, so this module also provides **deterministic synthetic grids** of the
reference's dimensionality (4-D double integrator `[x, y, dvx, dvy]`, 5-D airtaxi
`[x_r, y_r, theta_rel (periodic), v_a, v_b]`, 4-D TTR `[x, y, theta (periodic), v]`).
Their SHAPE is assumed (the Drive files' shape is not recoverable offline) and every report
says "synthetic grid".

Gradients follow the declared semantics of the oracle (`oracle/ref_stubs/hj_reachability`):
central differences inside, first-order one-sided at non-periodic ends, wrap on periodic dims.
"""
from __future__ import annotations

import math
import pickle
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import numpy as np

from .config import AirTaxiConfig, DoubleIntegratorConfig


@dataclass
class HjGrid:
    """values: float32 array of `shape`; grads: float32 `shape + (ndim,)` or None."""
    lo: np.ndarray
    hi: np.ndarray
    shape: Tuple[int, ...]
    periodic: Tuple[bool, ...]
    values: np.ndarray
    grads: Optional[np.ndarray] = None
    # separation distance the VALUES currently encode (HjDataHandle.separation_distance)
    separation_distance: float = 0.0
    ttr_max: float = 0.0

    @property
    def ndim(self) -> int:
        return len(self.shape)

    @property
    def spacings(self) -> np.ndarray:
        n = np.asarray(self.shape, dtype=np.float64)
        per = np.asarray(self.periodic, dtype=bool)
        return np.where(per, (self.hi - self.lo) / n, (self.hi - self.lo) / (n - 1.0))

    def coordinate_vectors(self):
        sp = self.spacings
        return [self.lo[d] + sp[d] * np.arange(self.shape[d], dtype=np.float64) for d in range(self.ndim)]


def grad_values(values: np.ndarray, spacings: Sequence[float], periodic: Sequence[bool]) -> np.ndarray:
    """Central / one-sided / wrapped finite differences; returns float32 `shape + (ndim,)`."""
    v = np.asarray(values, dtype=np.float64)
    out = np.empty(v.shape + (v.ndim,), dtype=np.float32)
    for d in range(v.ndim):
        h = float(spacings[d])
        vm = np.moveaxis(v, d, 0)
        g = np.empty_like(vm)
        if periodic[d]:
            g[:] = (np.roll(vm, -1, axis=0) - np.roll(vm, 1, axis=0)) / (2.0 * h)
        else:
            g[1:-1] = (vm[2:] - vm[:-2]) / (2.0 * h)
            g[0] = (vm[1] - vm[0]) / h
            g[-1] = (vm[-1] - vm[-2]) / h
        out[..., d] = np.moveaxis(g, 0, d)
    return out


def make_hj_handle(stored_values: np.ndarray, lo, hi, periodic, data_separation_distance: float,
                   target_separation_distance: float) -> HjGrid:
    """`HjDataHandle.__init__`: values_hj = -stored - (target - data_sep); grads of that."""
    lo = np.asarray(lo, dtype=np.float64)
    hi = np.asarray(hi, dtype=np.float64)
    shift = float(target_separation_distance) - float(data_separation_distance)
    # float32 storage (JAX default dtype) - the arithmetic order mirrors the reference expression
    values_hj = (-np.asarray(stored_values, dtype=np.float32) - np.float32(shift)).astype(np.float32)
    grid = HjGrid(lo=lo, hi=hi, shape=tuple(values_hj.shape), periodic=tuple(bool(p) for p in periodic),
                  values=values_hj, separation_distance=float(target_separation_distance))
    grid.grads = grad_values(values_hj, grid.spacings, grid.periodic)
    return grid


# --------------------------------------------------------------------------------------------
# deterministic synthetic grids (seed-free analytic functions sampled on the lattice)
# --------------------------------------------------------------------------------------------
DI_GRID_SHAPE = (41, 41, 21, 21)
DI_GRID_LO = (-4.5, -4.5, -1.0, -1.0)
DI_GRID_HI = (4.5, 4.5, 1.0, 1.0)
AIRTAXI_GRID_SHAPE = (41, 41, 24, 9, 9)
AIRTAXI_GRID_LO = (-5.5, -5.5, -math.pi, AirTaxiConfig.V_MIN, AirTaxiConfig.V_MIN)
AIRTAXI_GRID_HI = (5.5, 5.5, math.pi, AirTaxiConfig.V_MAX, AirTaxiConfig.V_MAX)
TTR_GRID_SHAPE = (41, 41, 24, 9)
TTR_GRID_LO = (-8.0, -8.0, -math.pi, AirTaxiConfig.V_MIN)
TTR_GRID_HI = (8.0, 8.0, math.pi, AirTaxiConfig.V_MAX)
TTR_MAX = 200.0


def _lattice(lo, hi, shape, periodic):
    n = np.asarray(shape, dtype=np.float64)
    lo = np.asarray(lo, dtype=np.float64)
    hi = np.asarray(hi, dtype=np.float64)
    per = np.asarray(periodic, dtype=bool)
    sp = np.where(per, (hi - lo) / n, (hi - lo) / (n - 1.0))
    vecs = [lo[d] + sp[d] * np.arange(shape[d], dtype=np.float64) for d in range(len(shape))]
    return np.meshgrid(*vecs, indexing='ij')


def synthetic_di_stored_values(shape=DI_GRID_SHAPE, lo=DI_GRID_LO, hi=DI_GRID_HI,
                               data_separation_distance=DoubleIntegratorConfig.SEPARATION_DISTANCE):
    """Stored convention of the Drive file: NEGATIVE inside the safe set (safety_filter.py:164-166).

    safe value  V = r - sep - c^2 / (2 a),  c = closing speed along the line of sight,
    a = 1.0 m/s^2 (two vehicles braking at 0.5 each). stored = -V.
    """
    x, y, dvx, dvy = _lattice(lo, hi, shape, (False,) * 4)
    r = np.sqrt(x * x + y * y)
    rdot = (x * dvx + y * dvy) / np.maximum(r, 1e-9)
    c = np.maximum(0.0, -rdot)
    v_safe = r - data_separation_distance - c * c / (2.0 * 1.0)
    return (-v_safe).astype(np.float32)


def synthetic_di_grid(target_separation_distance=DoubleIntegratorConfig.SEPARATION_DISTANCE,
                      data_separation_distance=DoubleIntegratorConfig.SEPARATION_DISTANCE,
                      shape=DI_GRID_SHAPE) -> HjGrid:
    stored = synthetic_di_stored_values(shape=shape, data_separation_distance=data_separation_distance)
    return make_hj_handle(stored, DI_GRID_LO, DI_GRID_HI, (False,) * 4, data_separation_distance,
                          target_separation_distance)


def synthetic_airtaxi_stored_values(shape=AIRTAXI_GRID_SHAPE, lo=AIRTAXI_GRID_LO, hi=AIRTAXI_GRID_HI,
                                    data_separation_distance=AirTaxiConfig.SEPARATION_DISTANCE):
    """5-D relative state in the ego frame; closing speed from the relative velocity
    (v_b cos(th) - v_a, v_b sin(th)); braking term with a = 0.002 km/s^2 and a 5 s turn lag."""
    x, y, th, va, vb = _lattice(lo, hi, shape, (False, False, True, False, False))
    r = np.sqrt(x * x + y * y)
    rvx = vb * np.cos(th) - va
    rvy = vb * np.sin(th)
    rdot = (x * rvx + y * rvy) / np.maximum(r, 1e-9)
    c = np.maximum(0.0, -rdot)
    v_safe = r - data_separation_distance - 5.0 * c - c * c / (2.0 * 0.002)
    return (-v_safe).astype(np.float32)


def synthetic_airtaxi_grid(target_separation_distance=AirTaxiConfig.SEPARATION_DISTANCE,
                           data_separation_distance=AirTaxiConfig.SEPARATION_DISTANCE,
                           shape=AIRTAXI_GRID_SHAPE) -> HjGrid:
    stored = synthetic_airtaxi_stored_values(shape=shape, data_separation_distance=data_separation_distance)
    return make_hj_handle(stored, AIRTAXI_GRID_LO, AIRTAXI_GRID_HI, (False, False, True, False, False),
                          data_separation_distance, target_separation_distance)


def synthetic_ttr_grid(shape=TTR_GRID_SHAPE, lo=TTR_GRID_LO, hi=TTR_GRID_HI) -> HjGrid:
    """4-D time-to-reach in the goal frame: distance at nominal speed + a heading-error turn time."""
    lo = np.asarray(lo, dtype=np.float64)
    hi = np.asarray(hi, dtype=np.float64)
    x, y, th, v = _lattice(lo, hi, shape, (False, False, True, False))
    d = np.sqrt(x * x + y * y)
    ttr = d / AirTaxiConfig.V_NOMINAL + 0.5 * np.abs(th) / AirTaxiConfig.ANGULAR_RATE_MAX \
        + 20.0 * np.abs(v - AirTaxiConfig.V_NOMINAL) / (AirTaxiConfig.V_MAX - AirTaxiConfig.V_MIN)
    ttr = np.minimum(ttr, TTR_MAX).astype(np.float32)
    return HjGrid(lo=lo, hi=hi, shape=tuple(shape), periodic=(False, False, True, False), values=ttr,
                  ttr_max=TTR_MAX)


def load_reference_pickle(file_name: str, target_separation_distance: float) -> HjGrid:
    """Load a Drive-format VALUE-FUNCTION pickle (`data/*_value_function.pkl`; needs `hj_reachability_utils` importable
    for unpickling, exactly like the reference). Field names: safety_filter.py:158-166. The time-to-reach file
    (`data/airtaxi_ttr_function.pkl`) has a different convention - use `load_reference_ttr_pickle` for it."""
    with open(file_name, 'rb') as f:
        data = pickle.load(f)
    meta = data.grid_meta_data
    shape = tuple(int(s) for s in meta.shape)
    periodic_dims = tuple(getattr(meta, 'periodic_dims', ()) or ())
    periodic = tuple(d in periodic_dims for d in range(len(shape)))
    return make_hj_handle(np.asarray(data.values), meta.domain_lo, meta.domain_hi, periodic,
                          data.info['separation_distance'], target_separation_distance)


def _periodic_mask(meta, ndim: int):
    periodic_dims = tuple(getattr(meta, 'periodic_dims', ()) or ())
    return tuple(d in periodic_dims for d in range(ndim))


def load_reference_ttr_pickle(file_name: str) -> HjGrid:
    """Load a Drive-format time-to-reach pickle the way `make_world` does (reference
    navigation_graph_safe.py:128-138): the values are used RAW (no negation, no separation shift, no gradients),
    `ttr_max` comes from `data.ttr_max` (the reward's fallback for out-of-range states, :751-755), periodic dims
    from the grid meta data. Needs `hj_reachability_utils` importable for unpickling, exactly like the reference."""
    with open(file_name, 'rb') as f:
        data = pickle.load(f)
    meta = data.grid_meta_data
    values = np.ascontiguousarray(np.asarray(data.values), dtype=np.float32)
    return HjGrid(lo=np.asarray(meta.domain_lo, dtype=np.float64), hi=np.asarray(meta.domain_hi, dtype=np.float64),
                  shape=tuple(int(s) for s in values.shape), periodic=_periodic_mask(meta, values.ndim), values=values,
                  grads=None, separation_distance=0.0, ttr_max=float(data.ttr_max))
