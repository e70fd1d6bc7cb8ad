"""The float32 interpolation mode (args.interp_float32, LSM_FLAG_INTERP_FLOAT32: what hj_reachability's
Grid.interpolate computes without jax_enable_x64, which the reference never enables) on the specialised pipeline.

  * routing: every shape LSM_SPEC_LIST names runs the three-kernel pipeline in this mode, with its usual launches;
  * CUDA == C oracle with zero tolerance for discrete outputs and the float64 state, on seeded batches with auto-resets;
  * the pair values the next step's filter reads: bit-identical across placements, and equal to the oracle's float32
    lookup of the relative state computed on the host;
  * the capabilities of the specialised pipeline in this mode: fused edge list, compact host adjacency, graph replay,
    chunked launches, emit_only."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

import _golden as G

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle'))

from test_cuda_parity import _compare_with_oracle      # noqa: E402
from test_pair_values import VARIANTS, _run, _episode, _grid_node_state, _pair_values, _read_mask, EPISODE_LENGTH  # noqa: E402

pytestmark = pytest.mark.gpu

# LSM_SPEC_LIST (lsm_kernels.cu): (dynamics, N, obstacles), two landmarks each
SPEC_SHAPES = [('double_integrator', 8, 0), ('double_integrator', 3, 0), ('double_integrator', 32, 0),
               ('double_integrator', 4, 0), ('double_integrator', 16, 0), ('airtaxi', 10, 0), ('airtaxi', 4, 0),
               ('airtaxi', 8, 0), ('airtaxi', 16, 0), ('airtaxi', 10, 4), ('double_integrator', 8, 4)]


def _args(dyn, N, O=0, **kw):
    air = dyn == 'airtaxi'
    d = dict(dynamics_type=dyn, num_agents=N, use_safety_filter=True, world_size=6 if air else 3, episode_length=12,
             interp_float32=True)
    if O:
        d.update(num_obstacles=O, obstacle_extension=True)
    d.update(kw)
    return G.default_args(**d)


@pytest.mark.parametrize('dyn,N,O', SPEC_SHAPES)
def test_listed_shapes_run_the_specialised_pipeline(dyn, N, O):
    from layered_safe_marl_b200 import B200GraphVecEnv
    infos = []
    for f32 in (False, True):
        env = B200GraphVecEnv(_args(dyn, N, O, interp_float32=f32), num_envs=16, seed=0)
        infos.append(env.launch_info())
        env.close()
    f64, f32 = infos
    assert f32['specialised'] == 1
    assert f32['launches_per_step'] == f64['launches_per_step'] and f32['pair_placement'] == f64['pair_placement']
    assert f32['blocks_per_sm'] == f64['blocks_per_sm']


def test_other_shapes_keep_the_generic_kernel():
    from layered_safe_marl_b200 import B200GraphVecEnv
    env = B200GraphVecEnv(_args('airtaxi', 6), num_envs=16, seed=0)
    assert env.launch_info()['specialised'] == 0
    env.close()


ORACLE_CASES = {
    # name: (args, RewardBinaryConfig switches, envs, steps)
    'cfg2': (dict(dyn='double_integrator', N=8, world_size=4), {}, 512, 25),
    'cfg3': (dict(dyn='airtaxi', N=10), dict(POTENTIAL_CONFLICT=True), 128, 20),
    'air10_obst4': (dict(dyn='airtaxi', N=10, O=4), dict(POTENTIAL_CONFLICT=True), 96, 16),
    'di8_obst4': (dict(dyn='double_integrator', N=8, O=4, world_size=1), {}, 193, 20),
    'di32': (dict(dyn='double_integrator', N=32, world_size=4), {}, 24, 20),
    'di8_hj_value': (dict(dyn='double_integrator', N=8), dict(HJ_VALUE=True), 160, 16),
    'air10_hj_value': (dict(dyn='airtaxi', N=10), dict(HJ_VALUE=True, POTENTIAL_CONFLICT=True), 96, 16),
    'di8_internal2': (dict(dyn='double_integrator', N=8, num_internal_step=2), {}, 160, 16),
    'air10_internal2': (dict(dyn='airtaxi', N=10, num_internal_step=2), {}, 96, 16),
    'di8_global': (dict(dyn='double_integrator', N=8, graph_feat_type='global'), {}, 160, 16),
    'air4_global': (dict(dyn='airtaxi', N=4, graph_feat_type='global'), {}, 160, 16),
}


@pytest.mark.parametrize('case', list(ORACLE_CASES))
def test_float32_mode_matches_the_oracle_bit_for_bit(case):
    kw, flags, n, T = ORACLE_CASES[case]
    kw = dict(kw)
    args = _args(kw.pop('dyn'), kw.pop('N'), kw.pop('O', 0), **kw)
    ora, cu = _compare_with_oracle(args, G.BinaryFlags(flags), n=n, T=T, episode=6249, seed=43, auto_reset=True)
    assert cu.env.launch_info()['specialised'] == 1
    st = cu.env.get_state()
    assert (st['safety_filtered'] != 0).any(), f"{case}: the filter never acted"


def test_airtaxi_rewards_match_the_oracle_bit_for_bit():
    """The airtaxi TTR term (-0.04 * TTR(goal-relative state)) reaches only the float32 reward, which the oracle
    comparison checks within a tolerance. Without POTENTIAL_CONFLICT every reward term is the same float64 arithmetic
    on both sides, so the rewards must agree bit for bit; float64 TTR lookups move some of them by an ulp."""
    import oracle_env as O
    from layered_safe_marl_b200 import B200GraphVecEnv, config as cfg
    args = _args('airtaxi', 10)
    flags = G.BinaryFlags({})
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = G.value_grid_for(params)
    n, episode = 256, 6249
    ora = O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=19, nthreads=8)
    env = B200GraphVecEnv(args, num_envs=n, seed=19, binary_cfg=flags, auto_reset=True)
    assert env.launch_info()['specialised'] == 1
    prev = O.set_relative_state_form(1)
    try:
        ora.reset(episode=episode, sample=True)
        env.reset(episode)
        rng = np.random.default_rng(4)
        for t in range(12):
            a = rng.integers(0, 25, (n, 10)).astype(np.int32)
            ora.step(a, episode=episode, auto_reset=True)
            env.step(torch.as_tensor(a, device=env.device), episode)
            got = env.reward.cpu().numpy()
            assert np.array_equal(env.get_state()['agent_values'], ora.get_state()['agent_values']), f"t={t}: states differ"
            bad = np.argwhere(got.view(np.int32) != np.asarray(ora.reward, dtype=np.float32).view(np.int32))
            assert bad.size == 0, f"t={t}: {len(bad)} rewards differ, first {tuple(bad[0])}: {got[tuple(bad[0])]!r} vs {ora.reward[tuple(bad[0])]!r}"
    finally:
        O.set_relative_state_form(prev)


PAIR_SHAPES = {
    'di8': dict(num_agents=8, world_size=12),
    'di8_obst4': dict(num_agents=8, world_size=2, num_obstacles=4, obstacle_extension=True),
    'air10': dict(dynamics_type='airtaxi', num_agents=10, world_size=6),
}


def _oracle_values(env, state, mask):
    """Raw float32-mode HJ value of every read (env, i, j) of `mask` through the oracle's lsmo_interpolate, from the
    relative state computed on the host: plain differences (double integrator), the rotation into the ego frame with
    lsm_sincos of the ego heading (airtaxi). numpy float64 arithmetic has no FMA, like the kernels."""
    import oracle_env as O
    from layered_safe_marl_b200 import config as cfg, hj_grid
    di = env.params.dynamics == cfg.DYN_DOUBLE_INTEGRATOR
    grid = hj_grid.synthetic_di_grid() if di else hj_grid.synthetic_airtaxi_grid()     # the env's default value grid
    s, keep = O.make_grid(grid)
    av = state['agent_values']
    e, i, j = np.nonzero(mask)
    ego, oth = av[e, i], av[e, j]
    if di:
        rel = ego - oth
    else:
        se = env.math_eval(3, ego[:, 2]); ce = env.math_eval(4, ego[:, 2])
        ddx, ddy = oth[:, 0] - ego[:, 0], oth[:, 1] - ego[:, 1]
        rel = np.stack([ddx * ce + ddy * se, ddy * ce - ddx * se, oth[:, 2] - ego[:, 2], ego[:, 3], oth[:, 3]], axis=-1)
    nd = rel.shape[1]
    lib = O.lib()
    want = np.empty(len(e))
    for f32 in (1, 0):
        lib.lsmo_set_interp_float32(f32)
        try:
            out = np.empty(len(e))
            for k in range(len(e)):
                out[k] = lib.lsmo_interpolate(ctypes.byref(s), (ctypes.c_double * nd)(*rel[k]), ctypes.c_int(-1))
        finally:
            lib.lsmo_set_interp_float32(0)
        out[np.isnan(out)] = np.inf
        if f32:
            want = out
        else:
            f64 = out
    return (e, i, j), want, f64


@pytest.mark.parametrize('shape', list(PAIR_SHAPES))
def test_pair_values_across_placements_and_against_the_oracle(shape):
    args = G.default_args(use_safety_filter=True, episode_length=EPISODE_LENGTH, interp_float32=True, **PAIR_SHAPES[shape])
    n = 333
    runs = [_run(args, n, v) for v in VARIANTS]
    ref = runs[0]
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


@pytest.mark.parametrize('shape', list(PAIR_SHAPES))
def test_pair_values_equal_the_oracle_float32_lookup(shape):
    """Every entry the next step reads, after steps with auto-resets, a masked reset, set_state onto grid nodes +
    observe and reset_from_state, against the oracle's float32 lookup of the host-computed relative state."""
    from layered_safe_marl_b200 import B200GraphVecEnv, _lib
    args = G.default_args(use_safety_filter=True, episode_length=EPISODE_LENGTH, interp_float32=True, **PAIR_SHAPES[shape])
    n, N = 200, args.num_agents
    env = B200GraphVecEnv(args, num_envs=n, seed=11)
    assert env.launch_info()['specialised'] == 1
    rng = np.random.default_rng(5)
    mask3 = torch.as_tensor((np.arange(n) % 3 == 1).astype(np.uint8), device=env.device)
    checked = differ_f64 = outside = 0

    def check(tag):
        nonlocal checked, differ_f64, outside
        st = env.get_state()
        mask = _read_mask(st)
        got = _pair_values(env).view(np.float64)
        idx, want, f64 = _oracle_values(env, st, mask)
        g = got[idx]
        bad = np.nonzero(g.view(np.int64) != want.view(np.int64))[0]
        assert bad.size == 0, (f"{shape} {tag}: {bad.size} of {g.size} pair values differ from the oracle's float32 lookup; "
                               f"first (env, i, j) = {tuple(int(a[bad[0]]) for a in idx)}: {g[bad[0]]!r} vs {want[bad[0]]!r}")
        checked += g.size
        differ_f64 += int((want != f64).sum())
        outside += int(np.isinf(want).sum())

    mid, low = _episode(0.5), _episode(0.1)
    env.reset(mid); check('reset')
    for t in range(6):
        env.step(torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=env.device), low)
        check(f'step {t}')
    _lib.check(env.lib.lsm_reset(env._h, mask3.data_ptr(), mid, env.seed, 1, env._stream()), 'lsm_reset')
    env.step(torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=env.device), low)
    check('step after a masked reset')
    env.set_state(_grid_node_state(env, env.get_state()))
    env.observe(); check('observe on grid nodes')
    env.reset_from_state(mid); check('reset_from_state')
    env.close()
    assert checked > 1000
    assert differ_f64 > checked // 4, "the float32 and float64 lookups agree almost everywhere: float32 mode is not in effect"


def _bits(a):
    a = a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint8)


@pytest.mark.parametrize('shape', ['di8', 'air10'])
def test_edge_list_in_float32_mode(shape):
    """Fused COO edge output == process_adj of the dense adjacency, through steps with auto-resets and a masked reset."""
    from test_edge_output import _check, _masked_reset, _step_both, EPISODE
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(dyn='double_integrator', N=8, world_size=2), air10=dict(dyn='airtaxi', N=10))[shape]
    args = _args(kw.pop('dyn'), kw.pop('N'), **kw)
    n = 300
    twin = B200GraphVecEnv(args, num_envs=n, seed=5)
    env = B200GraphVecEnv(args, num_envs=n, seed=5)
    assert env.launch_info()['specialised'] == 1
    env.enable_edge_output()
    gen = torch.Generator(); gen.manual_seed(3)
    twin.reset(EPISODE); env.reset(EPISODE)
    _check(env, twin, f"{shape} reset")
    _step_both(env, twin, gen, shape, k=6)
    mask = torch.zeros(n, dtype=torch.uint8, device=env.device); mask[::3] = 1
    _masked_reset(twin, mask); _masked_reset(env, mask)
    _check(env, twin, f"{shape} masked reset")
    _step_both(env, twin, gen, f"{shape} after the masked reset", k=3)


@pytest.mark.parametrize('shape', ['di8', 'air10'])
def test_host_outputs_in_float32_mode_are_byte_identical(shape):
    """numpy_outputs=True takes the compact-adjacency host path in this mode; every returned array equals the
    device-resident env's dense outputs byte for byte."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(dyn='double_integrator', N=8, world_size=2), air10=dict(dyn='airtaxi', N=10))[shape]
    args = _args(kw.pop('dyn'), kw.pop('N'), **kw)
    n, T, episode = 300, 16, 6249
    dev_env = B200GraphVecEnv(args, num_envs=n, seed=3)
    host_env = B200GraphVecEnv(args, num_envs=n, seed=3, numpy_outputs=True, host_chunks=5, host_threads=3)
    assert host_env._compact is not None
    o1, o2 = dev_env.reset(episode), host_env.reset(episode)
    for a, b in zip(o1[:4], o2[:4]):
        assert np.array_equal(_bits(a), _bits(b))
    rng = np.random.default_rng(1)
    for t in range(T):
        idx = rng.integers(0, 25, (n, args.num_agents)).astype(np.int32)
        o1 = dev_env.step(torch.as_tensor(idx, device=dev_env.device), episode)
        o2 = host_env.step(idx, episode)
        for k, (a, b) in enumerate(zip(o1[:6], o2[:6])):
            assert np.array_equal(_bits(a), _bits(b)), f"step {t} output {k}"


def _snapshot(env):
    st = env.get_state()
    return [_bits(env.obs), _bits(env.node_obs), _bits(env.adj), _bits(env.reward), _bits(env.done)] + \
        [np.ascontiguousarray(st[k]).view(np.uint8) for k in ('agent_values', 'safety_filtered', 'deconflicting_agent_index')]


@pytest.mark.parametrize('shape', ['di8', 'air10'])
def test_graph_replay_and_chunks_are_bit_identical(shape):
    """use_graph = 1 (replayed launches) and chunks = 4 (four env ranges on library streams) against plain single-range
    launches, step by step, through auto-resets; then emit_only rewrites the same node_obs / adj."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(dyn='double_integrator', N=8, world_size=2), air10=dict(dyn='airtaxi', N=10))[shape]
    args = _args(kw.pop('dyn'), kw.pop('N'), episode_length=9, **kw)
    n, T, episode = 1024, 24, 6249
    tunings = [dict(chunks=1), dict(chunks=1, use_graph=1), dict(chunks=4)]
    envs = [B200GraphVecEnv(args, num_envs=n, seed=5, tuning=t) for t in tunings]
    assert [e.launch_info()['chunks'] for e in envs] == [1, 1, 4]
    acts = [torch.empty((n, args.num_agents), dtype=torch.int32, device=e.device) for e in envs]   # fixed pointers: replay
    for e in envs:
        e.reset(episode)
    gen = torch.Generator(); gen.manual_seed(9)
    for t in range(T):
        a = torch.randint(0, 25, (n, args.num_agents), generator=gen, dtype=torch.int32)
        for e, buf in zip(envs, acts):
            buf.copy_(a)
            e.step(buf, episode)
        torch.cuda.synchronize()
        ref = _snapshot(envs[0])
        for tu, e in zip(tunings[1:], envs[1:]):
            for k, (x, y) in enumerate(zip(ref, _snapshot(e))):
                assert np.array_equal(x, y), f"{shape} {tu}: step {t}: output {k} differs from plain launches"
    assert envs[1].launch_info()['graph_replays'] > 0
    for e in envs:
        before = (_bits(e.node_obs), _bits(e.adj))
        e.emit_only(); e.emit_only()
        torch.cuda.synchronize()
        assert np.array_equal(before[0], _bits(e.node_obs)) and np.array_equal(before[1], _bits(e.adj)), "emit_only is not idempotent"
