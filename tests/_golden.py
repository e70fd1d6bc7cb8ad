"""Helpers shared by the parity tests: load tests/golden/*.npz, build params, compare."""
from __future__ import annotations

import argparse
import glob
import json
import os

import numpy as np

from layered_safe_marl_b200 import config as cfg
from layered_safe_marl_b200 import hj_grid

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
# a checkout of the original project (DINaMo-MIT/Layered-Safe-MARL), which the fixture generators under oracle/ drive; only
# the tests that regenerate fixtures need it and they skip without it
REFERENCE = os.environ.get('LSM_REFERENCE_PATH', '')
REFERENCE_SKIP = "needs a checkout of the original project: set LSM_REFERENCE_PATH"


def have_reference(subdir):
    return bool(REFERENCE) and os.path.isdir(os.path.join(REFERENCE, subdir))


STATE_KEYS = ('agent_values', 'p_dist', 'state_time', 'done', 'safety_filtered', 'deconflicting_agent_index',
              'min_relative_distance', 'goal_min_time', 'action_diff', 'reached_goal', 'landmark_pos',
              'landmark_heading', 'landmark_speed', 'times_required', 'dists_to_goal', 'dist_left_to_goal',
              'num_agent_collisions', 'current_step', 'curriculum_ratio', 'ep_travel_length',
              'ep_travel_distance', 'ep_done', 'ep_conflict', 'ep_multi_engagement', 'ep_min_distance')

# relative tolerance of the north star for continuous values; fixtures store outputs as float32. The absolute term only
# covers values that are zero up to roundoff (a difference of two nearly equal angles / positions): 1e-9, i.e. it adds
# nothing to the relative bar for any value above 1e-4 (round 1 used 2e-6; every CPU and GPU parity test passes at 1e-9)
RTOL = 1e-5
ATOL = 1e-9


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, '*.npz')))


class BinaryFlags:
    def __init__(self, flags):
        for k in ('SAFETY_VIOLATION', 'HJ_VALUE', 'POTENTIAL_CONFLICT', 'SEPARATION_DISTANCE_CURRICULUM',
                  'INITIAL_PHASE_USE_SAFETY_FILTER', 'DIFF_FROM_FILTERED_ACTION'):
            setattr(self, k, bool(flags.get(k, False)))


def default_args(**kw):
    d = dict(scenario_name='navigation_graph_safe', dynamics_type='double_integrator', num_agents=3,
             num_scripted_agents=0, num_obstacles=0, collaborative=False, use_dones=False,
             episode_length=25, num_env_steps=5_000_000, n_rollout_threads=32, world_size=4,
             num_landmarks=2, use_safety_filter=False, num_internal_step=1, graph_feat_type='relative',
             use_masking=True, num_walls=0, zeroshift=3, discrete_action=True, algorithm_name='rmappo')
    d.update(kw)
    return argparse.Namespace(**d)


def load_case(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + '.npz'))
    meta = json.loads(str(z['meta']))
    args = default_args(**meta['args'])
    flags = BinaryFlags(meta['flags'])
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    assert params.num_total_episode == meta['num_total_episode']
    return z, meta, args, flags, params


_GRID_CACHE = {}


def grids_for(params):
    """Synthetic value / TTR grids the fixtures were generated with."""
    key = params.dynamics
    if key not in _GRID_CACHE:
        if params.dynamics == cfg.DYN_DOUBLE_INTEGRATOR:
            need = bool(params.flags & (cfg.FLAG_USE_SAFETY_FILTER | cfg.FLAG_HJ_VALUE))
            _GRID_CACHE[key] = (hj_grid.synthetic_di_grid(), None)
        else:
            _GRID_CACHE[key] = (hj_grid.synthetic_airtaxi_grid(), hj_grid.synthetic_ttr_grid())
    return _GRID_CACHE[key]


def value_grid_for(params):
    """HjDataHandle is constructed with the scenario's INITIAL separation distance
    (navigation_graph_safe.py:186-196): 0 when SEPARATION_DISTANCE_CURRICULUM else the target."""
    vg, tg = grids_for(params)
    return vg, tg


OBSTACLE_KEYS = ('obstacle_pos', 'num_obstacle_collisions')      # fixtures of the declared obstacle extension only


def _state_keys(z, prefix):
    return STATE_KEYS + tuple(k for k in OBSTACLE_KEYS if prefix + k in z.files)


def state0(z, batch=True):
    s = {k: np.array(z['s0_' + k]) for k in _state_keys(z, 's0_')}
    if batch:
        s = {k: v[None] for k, v in s.items()}
    return s


def state_at(z, t, batch=True):
    s = {k: np.array(z['st_' + k][t]) for k in _state_keys(z, 'st_')}
    if batch:
        s = {k: v[None] for k, v in s.items()}
    return s


def assert_close(got, want, what, rtol=RTOL, atol=ATOL):
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    both_inf = np.isinf(got) & np.isinf(want) & (np.sign(got) == np.sign(want))
    err = np.abs(got - want)
    tol = atol + rtol * np.maximum(np.abs(want), np.abs(got))
    bad = ~(both_inf | (err <= tol))
    if bad.any():
        idx = np.argwhere(bad)[:5]
        msg = "; ".join(f"{tuple(i)}: got {got[tuple(i)]!r} want {want[tuple(i)]!r}" for i in idx)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} elements differ beyond rtol={rtol}: {msg}")


def assert_same_mask(got, want, what):
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    if not np.array_equal(got, want):
        idx = np.argwhere(got != want)[:5]
        raise AssertionError(f"{what}: {int((got != want).sum())} mismatching entries, first at {idx.tolist()}")
