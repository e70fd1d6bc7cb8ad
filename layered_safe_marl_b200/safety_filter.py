"""SafetyFilter - the HJ safety filter as a standalone batched operator on the GPU.

The reference applies its safety layer through per-agent Python handles (multiagent/safety_filter.py:
`DoubleIntegratorSafetyHandle` / `KinematicVehicleSafetyHandle.apply_safety_filter`, `get_value_of_relative_state`) and
`World.apply_safety_filter` (core.py:648-677). This module exposes the same computation for states this simulator does
not own - another simulator, hardware, logged trajectories, hand-built conflicts - through the sm_100a kernels behind
`lsm_safety_filter` / `lsm_hj_lookup` (include/lsm_b200.h). The arithmetic is the environment's own: a filter over the
env's state returns exactly the env's safe action, filtered flag and deconflicting agent.

    sf = SafetyFilter('double_integrator')             # own handle, synthetic grid unless one is given
    sf = SafetyFilter.of(env)                          # the env's handle, library, grid and interpolation mode
    safe, filtered, index, value = sf.apply(ego, others, ego_action, other_actions)
    safe, filtered, deconflict = sf.apply_world(states, actions, done)
    value, grad = sf.values(ego=ego, other=other, gradients=True)

Every call launches on torch's current stream of the filter's device, returns device tensors and never synchronises.
"""
from __future__ import annotations

import argparse
import ctypes as C
import warnings
from typing import Optional

import torch

from . import _lib
from .config import DYN_DOUBLE_INTEGRATOR, scenario_params_from_args
from .hj_grid import HjGrid, synthetic_airtaxi_grid, synthetic_di_grid

_F64 = torch.float64


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class SafetyFilter:
    def __init__(self, dynamics: str = 'double_integrator', value_grid: Optional[HjGrid] = None,
                 interp_float32: bool = False, device='cuda:0'):
        """A filter with a handle of its own. `dynamics`: 'double_integrator' or 'airtaxi'. `value_grid`: an HjGrid
        (hj_grid.load_reference_pickle for the reference's value-function files); None uses the synthetic grid the
        environment uses without one. `interp_float32`: the float32 grid interpolation (LSM_FLAG_INTERP_FLOAT32)."""
        if dynamics not in ('double_integrator', 'airtaxi'):
            raise ValueError(f"dynamics must be 'double_integrator' or 'airtaxi', not {dynamics!r}")
        if not torch.cuda.is_available():
            raise RuntimeError("SafetyFilter needs a CUDA device; there is no CPU fallback")
        from .vec_env import _DeviceGrid, make_config_struct
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        # a minimal valid scenario of the filter's dynamics: only dt, cbf_rate, coordination_range and the interpolation
        # flag reach the operator. The shape is one the product library specialises, so the handle builds the
        # corner-packed value table and the padded gradient rows of the env's fast path.
        args = argparse.Namespace(dynamics_type=dynamics, num_agents=8 if dynamics == 'double_integrator' else 10,
                                  num_landmarks=2, episode_length=25, num_env_steps=25, n_rollout_threads=1,
                                  world_size=4, use_safety_filter=True, num_internal_step=1,
                                  interp_float32=bool(interp_float32))
        self.params = scenario_params_from_args(args)
        if value_grid is None:
            warnings.warn("SafetyFilter: no value grid given - using the synthetic grid (hj_grid.synthetic_*_grid); "
                          "load the reference's value function with hj_grid.load_reference_pickle", stacklevel=2)
            value_grid = synthetic_di_grid() if self.params.dynamics == DYN_DOUBLE_INTEGRATOR else synthetic_airtaxi_grid()
        self._owned = True
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            cfg = make_config_struct(self.params)
            self._check(self.lib.lsm_create(C.byref(cfg), C.byref(self._h)), 'lsm_create')
            self.value_grid = _DeviceGrid(value_grid, self.device)
            self._check(self.lib.lsm_set_value_grid(self._h, C.byref(self.value_grid.desc)), 'lsm_set_value_grid')
        self._env = None
        self.dynamics = self.params.dynamics
        self.ndim = 4 if self.dynamics == DYN_DOUBLE_INTEGRATOR else 5
        self.grid_separation_distance = float(value_grid.separation_distance)

    @classmethod
    def of(cls, env) -> 'SafetyFilter':
        """A filter over the handle of a B200GraphVecEnv: same library (a per-shape library included), grid, constants
        and interpolation mode. The env must have a value grid (use_safety_filter or the HJ-value reward)."""
        if env.value_grid is None:
            raise ValueError("SafetyFilter.of: the environment has no value grid (use_safety_filter or HJ_VALUE)")
        self = cls.__new__(cls)
        self.lib = env.lib
        self.device = env.device
        self.params = env.params
        self._h = env._h
        self._owned = False
        self._env = env          # keeps the handle and the grid alive
        self.value_grid = env.value_grid
        self.dynamics = env.params.dynamics
        self.ndim = 4 if self.dynamics == DYN_DOUBLE_INTEGRATOR else 5
        self.grid_separation_distance = float(env.value_grid.desc.separation_distance)
        return self

    def close(self):
        if getattr(self, '_owned', False) and self._h:
            self.lib.lsm_destroy(self._h)
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        _lib.check(rc, what, self.lib)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f64(self, t, shape, name):
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name} must be a torch tensor on {self.device}")
        if t.device != self.device:
            raise ValueError(f"{name} is on {t.device}, the filter on {self.device}")
        if not t.is_floating_point():
            raise TypeError(f"{name} must be a floating-point tensor")
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")
        return t.to(_F64).contiguous()

    def _sep(self, separation_distance, n):
        if separation_distance is None:
            return None
        if isinstance(separation_distance, torch.Tensor):
            return self._f64(separation_distance, (n,), 'separation_distance')
        return torch.full((n,), float(separation_distance), dtype=_F64, device=self.device)

    # ------------------------------------------------------------------------------------------
    def apply(self, ego, others, ego_action, other_actions, active=None, separation_distance=None):
        """The safety handle's apply_safety_filter for B independent egos, each against M candidate others.
        ego (B, 4), others (B, M, 4), ego_action (B, 2), other_actions (B, M, 2) decoded controls; active (B, M) bool
        (None = all slots); separation_distance float or (B,) (None = the grid's own: no value shift).
        Returns safe_action (B, 2) float64, filtered (B,) bool, index (B,) int32 (deconflicting slot, -1 without an
        active slot), value (B,) float64 (its HJ value, +inf when none is active or the state is NaN)."""
        B = int(ego.shape[0]) if isinstance(ego, torch.Tensor) and ego.dim() == 2 else -1
        M = int(others.shape[1]) if isinstance(others, torch.Tensor) and others.dim() == 3 else -1
        if B < 0 or M < 0:
            raise ValueError("ego must be (B, 4) and others (B, M, 4)")
        ego = self._f64(ego, (B, 4), 'ego')
        others = self._f64(others, (B, M, 4), 'others')
        ego_action = self._f64(ego_action, (B, 2), 'ego_action')
        other_actions = self._f64(other_actions, (B, M, 2), 'other_actions')
        act = None
        if active is not None:
            if not isinstance(active, torch.Tensor) or active.device != self.device or tuple(active.shape) != (B, M):
                raise ValueError(f"active must be a ({B}, {M}) tensor on {self.device}")
            act = active.to(torch.bool).contiguous()
        sep = self._sep(separation_distance, B)
        safe = torch.empty((B, 2), dtype=_F64, device=self.device)
        filtered = torch.empty((B,), dtype=torch.bool, device=self.device)
        index = torch.empty((B,), dtype=torch.int32, device=self.device)
        value = torch.empty((B,), dtype=_F64, device=self.device)
        io = _lib.LsmFilterIo()
        io.num_rows = B; io.num_slots = M
        io.ego = ego.data_ptr(); io.ego_action = ego_action.data_ptr()
        io.others = others.data_ptr() if M > 0 else None
        io.other_actions = other_actions.data_ptr() if M > 0 else None
        io.active = act.data_ptr() if act is not None and M > 0 else None
        io.separation_distance = sep.data_ptr() if sep is not None else None
        io.safe_action = safe.data_ptr(); io.filtered = filtered.data_ptr(); io.index = index.data_ptr()
        io.value = value.data_ptr()
        self._check(self.lib.lsm_safety_filter(self._h, C.byref(io), self._stream()), 'lsm_safety_filter')
        return safe, filtered, index, value

    def apply_world(self, states, actions, done, separation_distance=None):
        """World.apply_safety_filter (core.py:648-677) over n worlds of N agents: the others of agent i are the agents
        j != i that are not done, in ascending j. states (n, N, 4), actions (n, N, 2) decoded controls, done (n, N) bool;
        separation_distance float or (n,). Returns safe_action (n, N, 2), filtered (n, N) bool and deconflict (n, N) int32,
        the global agent index (-1 for done agents and agents without another live agent). Done agents keep their raw
        action, unfiltered."""
        n, N = int(states.shape[0]), int(states.shape[1])
        states = self._f64(states, (n, N, 4), 'states')
        actions = self._f64(actions, (n, N, 2), 'actions')
        if not isinstance(done, torch.Tensor) or done.device != self.device or tuple(done.shape) != (n, N):
            raise ValueError(f"done must be a ({n}, {N}) tensor on {self.device}")
        done = done.to(torch.bool)
        # slot k of agent i is agent j = k + (k >= i): every other agent in ascending order
        i = torch.arange(N, device=self.device).view(N, 1)
        k = torch.arange(max(N - 1, 0), device=self.device).view(1, -1)
        j = k + (k >= i).to(k.dtype)                                     # (N, N-1)
        others = states[:, j]                                            # (n, N, N-1, 4)
        other_actions = actions[:, j]
        active = ~done[:, j] & ~done.view(n, N, 1)                       # a done ego has no active slot
        sep = separation_distance
        if isinstance(sep, torch.Tensor):
            sep = self._f64(sep, (n,), 'separation_distance').view(n, 1).expand(n, N).reshape(n * N)
        safe, filtered, index, _ = self.apply(states.reshape(n * N, 4), others.reshape(n * N, N - 1, 4),
                                              actions.reshape(n * N, 2), other_actions.reshape(n * N, N - 1, 2),
                                              active.reshape(n * N, N - 1), sep)
        index = index.view(n, N)
        deconflict = torch.where(index >= 0, index + (index >= i.view(1, N)).to(index.dtype), index).to(torch.int32)
        return safe.view(n, N, 2), filtered.view(n, N), deconflict

    def values(self, rel=None, ego=None, other=None, gradients: bool = False, separation_distance=None):
        """get_value_of_relative_state (safety_filter.py:192-201, 345-354) of K relative states rel (K, d), or of the
        (ego, other) state pairs (K, 4) each, whose relative state the kernel forms itself. d = 4 (double integrator) or
        5 (airtaxi). Returns value (K,) float64 (+inf for a NaN state; shifted by -(sep - grid separation)) and, with
        gradients=True, the gradient (K, d), else None."""
        if rel is not None:
            K = int(rel.shape[0])
            rel = self._f64(rel, (K, self.ndim), 'rel')
        else:
            if ego is None or other is None:
                raise ValueError("give rel, or ego and other")
            K = int(ego.shape[0])
            ego = self._f64(ego, (K, 4), 'ego')
            other = self._f64(other, (K, 4), 'other')
        sep = self._sep(separation_distance, K)
        value = torch.empty((K,), dtype=_F64, device=self.device)
        grad = torch.empty((K, self.ndim), dtype=_F64, device=self.device) if gradients else None
        io = _lib.LsmLookupIo()
        io.num_points = K
        io.rel = _ptr(rel).value if rel is not None else None
        io.ego = ego.data_ptr() if rel is None else None
        io.other = other.data_ptr() if rel is None else None
        io.separation_distance = sep.data_ptr() if sep is not None else None
        io.value = value.data_ptr()
        io.grad = grad.data_ptr() if grad is not None else None
        io.rel_out = None
        self._check(self.lib.lsm_hj_lookup(self._h, C.byref(io), self._stream()), 'lsm_hj_lookup')
        return value, grad
