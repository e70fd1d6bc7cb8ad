"""The HJ pair values V(x_i - x_j) the specialised pipeline leaves behind for the next step's safety filter
(safety_filter.py:192-201, 345-354), compared bit for bit between every way the library can produce them:

  * behind the emit kernel (pair placement 0), from the emit records or - behind a masked reset - the state tensors,
    in one range and in three chunked ranges with a ragged last one;
  * between the agent and the emit kernel (placement 3), from the same inputs;
  * in front of the next agent kernel (placement 2), always from the state tensors;
  * at the tail of the agent kernel (placement 4), from the records in shared memory;
  * behind the emit kernel with the scattered stencil instead of the corner-packed table (packed_grid 0).

Only the entries the next agent kernel reads are compared: envs whose curriculum has the filter on, i != j, neither
agent done. The scratch is read with lsm_debug_pair_values."""
import numpy as np
import pytest
import torch

import _golden as G

pytestmark = pytest.mark.gpu

SHAPES = {
    # world_size 12 > the grid's +-4.5 box: many relative states lie outside it (declared clamp)
    'di8': dict(num_agents=8, world_size=12),
    'di32': dict(num_agents=32, world_size=4),
    'di8_obst4': dict(num_agents=8, world_size=2, num_obstacles=4, obstacle_extension=True),
    'air10': dict(dynamics_type='airtaxi', num_agents=10, world_size=6),
    'air10_obst4': dict(dynamics_type='airtaxi', num_agents=10, world_size=6, num_obstacles=4, obstacle_extension=True),
}
VARIANTS = [dict(pair_placement=0), dict(pair_placement=0, chunks=3), dict(pair_placement=3), dict(pair_placement=2),
            dict(pair_placement=4), dict(pair_placement=0, packed_grid=0)]
EPISODE_LENGTH = 6


def _episode(ratio):
    """num_current_episode whose curriculum ratio is `ratio` (config.py: num_total_episode)."""
    total = 5_000_000 // EPISODE_LENGTH // 32
    return int(round(ratio * total))


def _pair_values(env):
    from layered_safe_marl_b200 import _lib
    out = torch.empty((env.n, env.N, env.N), dtype=torch.float64, device=env.device)
    _lib.check(env.lib.lsm_debug_pair_values(env._h, out.data_ptr(), env._stream()), 'lsm_debug_pair_values')
    torch.cuda.synchronize(env.device)
    return out.cpu().numpy().view(np.int64).copy()


def _read_mask(state):
    """entries the next step's agent kernel reads: filter on (ratio_sloped(ratio, 0.25, 0.75) > 0), i != j, both
    agents not done"""
    on = state['curriculum_ratio'] > 0.25
    live = ~state['done']
    N = live.shape[1]
    return on[:, None, None] & live[:, :, None] & live[:, None, :] & ~np.eye(N, dtype=bool)[None]


def _grid_node_state(env, state):
    """agent 0 of every env at the origin (airtaxi: heading 0), agent 1 placed so that the relative state of the pair
    (0, 1) is a node of the value grid's lattice (hj_grid.HjGrid.coordinate_vectors)"""
    from layered_safe_marl_b200 import config as cfg, hj_grid
    di = env.params.dynamics == cfg.DYN_DOUBLE_INTEGRATOR
    grid = hj_grid.synthetic_di_grid() if di else hj_grid.synthetic_airtaxi_grid()   # the env's default grid
    s = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in state.items()}
    av = s['agent_values']
    rng = np.random.default_rng(3)
    node = [vec[rng.integers(0, len(vec), av.shape[0])] for vec in grid.coordinate_vectors()]
    zero = np.zeros(av.shape[0])
    if di:
        # rel = (ex - ox, ey - oy, evx - ovx, evy - ovy) with the other at the origin at rest
        av[:, 0] = np.stack(node[:4], axis=-1)
        av[:, 1] = 0.0
    else:
        # ego at the origin heading 0: rel = (ox, oy, o_theta - 0, e_speed, o_speed)
        av[:, 0] = np.stack([zero, zero, zero, node[3]], axis=-1)
        av[:, 1] = np.stack([node[0], node[1], node[2], node[4]], axis=-1)
    s['agent_values'] = av
    return s


def _run(args, n, tuning):
    """Snapshots (pair values, read mask, comparable envs, launch) of the state after every launch of a fixed script.
    Placement 2 computes the values of a state in front of the step that starts from it: its values of state k are
    the ones left after launch k + 1 when that launch is a step from the unedited state k."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    env = B200GraphVecEnv(args, num_envs=n, seed=11, tuning=dict(tuning))
    assert env.launch_info()['pair_placement'] == tuning['pair_placement']
    if 'chunks' in tuning:
        assert env.launch_info()['chunks'] == tuning['chunks']
    N = args.num_agents
    rng = np.random.default_rng(7)
    every = np.ones(n, dtype=bool)
    mask3 = torch.as_tensor((np.arange(n) % 3 == 1).astype(np.uint8), device=env.device)
    snaps = []

    def snap(launch, fresh=every):
        # fresh: envs whose values this launch produced in every placement (placement 4 refreshes only the envs of a
        # masked reset; after a state edit the others are recomputed in front of the next step)
        snaps.append((_pair_values(env), _read_mask(env.get_state()), fresh, launch))

    def step(ep):
        env.step(torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=env.device), ep)
        snap('step')

    def masked_reset(ep):
        from layered_safe_marl_b200 import _lib
        _lib.check(env.lib.lsm_reset(env._h, mask3.data_ptr(), ep, env.seed, 1, env._stream()), 'lsm_reset')

    mid, low = _episode(0.5), _episode(0.1)
    env.reset(mid); snap('reset')                # every env: filter on
    for _ in range(8):                           # auto-resets at curriculum ratio 0.1: those envs have the filter off
        step(low)
    masked_reset(mid); snap('masked reset')      # masked reset after steps
    step(low)
    step(low)
    env.set_state(_grid_node_state(env, env.get_state()))
    masked_reset(mid); snap('edit', mask3.cpu().numpy().astype(bool))   # first launch after set_state: masked reset
    step(low)
    env.set_state(_grid_node_state(env, env.get_state()))
    env.observe(); snap('edit')                  # observe on grid nodes
    step(low)
    env.reset_from_state(mid); snap('reset')     # unmasked reset without sampling
    step(low)
    step(low)
    env.close()
    return snaps


@pytest.mark.parametrize('shape', list(SHAPES))
def test_pair_values_bit_identical_across_placements(shape):
    args = G.default_args(use_safety_filter=True, episode_length=EPISODE_LENGTH, **SHAPES[shape])
    n = 64 if shape == 'di32' else 333
    runs = [_run(args, n, v) for v in VARIANTS]
    ref = runs[0]
    # coverage: values were read, some envs had the filter off, some agents were done
    masks = np.stack([m for _, m, _, _ in ref])
    assert masks.any(axis=(2, 3)).any() and not masks.any(axis=(2, 3)).all(), "no mix of filter-on / filter-off envs"
    for v, run in zip(VARIANTS[1:], runs[1:]):
        front = v['pair_placement'] == 2
        for k, (vals, mask, fresh, _) in enumerate(ref):
            if front:
                if k + 1 >= len(run) or run[k + 1][3] != 'step':
                    continue
                got = run[k + 1][0]
            else:
                got = run[k][0]
            m = mask & fresh[:, None, None] if v['pair_placement'] == 4 else mask
            bad = np.argwhere(m & (got != vals))
            assert bad.size == 0, (f"{shape} {v}: state {k}: {len(bad)} pair values differ, first (env, i, j) = "
                                   f"{tuple(bad[0])}: {vals[tuple(bad[0])].view(np.float64)} vs {got[tuple(bad[0])].view(np.float64)}")
