"""The HJ safety filter as a standalone operator (SafetyFilter / lsm_safety_filter / lsm_hj_lookup).

CPU: the C oracle's filter over independent rows (tests/filter_rows_oracle.c: oracle/lsm_oracle.c's apply_safety_filter, one
world per row) reproduces every filter decision of the reference's golden rollouts, and the ctypes mirrors of the two new structs match the C header.
GPU: the CUDA operator against the same golden decisions, against the oracle bit for bit (rotation form of the relative
state), and against the environment's own step bit for bit.
"""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))
sys.path.insert(0, os.path.join(REPO, 'tests'))

import _golden as G  # noqa: E402
import oracle_env as O  # noqa: E402
from layered_safe_marl_b200 import config as cfg, hj_grid  # noqa: E402

FILTER_FIXTURES = ('di8_filter', 'di8_filter_f32', 'di8_filter_allflags', 'di16_dense', 'di2_landmarks4',
                   'di4_obst3_filter_global', 'di1_single_filter', 'at10_filter_pc', 'at10_filter_pc_f32',
                   'at10_obst4_filter_pc', 'at6_allflags', 'at3_landmarks3')


# ------------------------------------------------------------------------------------------------------------------
# the oracle over rows (tests/filter_rows_oracle.c), compiled once per session with the oracle's flags
# ------------------------------------------------------------------------------------------------------------------
_ROWS_LIB = None


def _rows_lib():
    global _ROWS_LIB
    if _ROWS_LIB is None:
        tmp = tempfile.mkdtemp(prefix='lsm_filter_rows_')
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, 'libfilter_rows_oracle.so')
        subprocess.check_call(['gcc', '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math', '-shared', '-o', out,
                               os.path.join(REPO, 'tests', 'filter_rows_oracle.c'), '-lm', '-lpthread'])
        lib = ctypes.CDLL(out)
        lib.lsmt_safety_filter_rows.restype = ctypes.c_int
        lib.lsmt_safety_filter_rows.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                ctypes.c_int32] + [ctypes.c_void_p] * 10
        lib.lsmt_hj_lookup.restype = ctypes.c_int
        lib.lsmt_hj_lookup.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 6
        _ROWS_LIB = lib
    return _ROWS_LIB


def _p(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def oracle_rows(params: dict, value_grid, ego, others, ego_action, other_actions, active=None, sep=None, rel_form=0):
    """The oracle's safety filter for B egos against M slots each: (safe [B, 2], filtered [B], index [B], value [B])."""
    p = O.make_params(params)
    g, keep = O.make_grid(value_grid)
    ego = np.ascontiguousarray(ego, dtype=np.float64)
    B = ego.shape[0]
    others = np.ascontiguousarray(others, dtype=np.float64)
    M = others.shape[1]
    others = others.reshape(B, M, 4)
    ua = np.ascontiguousarray(ego_action, dtype=np.float64).reshape(B, 2)
    uo = np.ascontiguousarray(other_actions, dtype=np.float64).reshape(B, M, 2)
    act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8).reshape(B, M)
    sp = None if sep is None else np.ascontiguousarray(np.broadcast_to(np.asarray(sep, dtype=np.float64), (B,)))
    safe = np.zeros((B, 2)); filt = np.zeros(B, np.uint8); idx = np.zeros(B, np.int32); val = np.zeros(B)
    rc = _rows_lib().lsmt_safety_filter_rows(ctypes.byref(p), ctypes.byref(g), rel_form, B, M, _p(ego), _p(others), _p(ua),
                                             _p(uo), _p(act), _p(sp), _p(safe), _p(filt), _p(idx), _p(val))
    assert rc == 0
    return safe, filt.astype(bool), idx, val


def oracle_lookup(params: dict, value_grid, rel=None, ego=None, other=None, sep=None, rel_form=0):
    """The oracle's shifted value (+inf for NaN) and gradient of relative states or (ego, other) pairs."""
    p = O.make_params(params)
    g, keep = O.make_grid(value_grid)
    nd = 4 if int(params['dynamics']) == 0 else 5
    if rel is not None:
        rel = np.ascontiguousarray(rel, dtype=np.float64).reshape(-1, nd)
        K = rel.shape[0]
    else:
        ego = np.ascontiguousarray(ego, dtype=np.float64).reshape(-1, 4)
        other = np.ascontiguousarray(other, dtype=np.float64).reshape(-1, 4)
        K = ego.shape[0]
    sp = None if sep is None else np.ascontiguousarray(np.broadcast_to(np.asarray(sep, dtype=np.float64), (K,)))
    val = np.zeros(K); grad = np.zeros((K, nd))
    rc = _rows_lib().lsmt_hj_lookup(ctypes.byref(p), ctypes.byref(g), rel_form, K, _p(rel), _p(ego), _p(other), _p(sp),
                                    _p(val), _p(grad))
    assert rc == 0
    return val, grad


def _golden_rows(name):
    """Every filtered step of a fixture as operator rows: (params, list of (states, raw, done, sep, t), z)."""
    z, meta, args, flags, params = G.load_case(name)
    assert params.num_internal_step == 1
    t0, t1 = O.action_tables(params.dynamics)
    steps = []
    for t in range(z['actions'].shape[0]):
        if not bool(z['st_world_use_safety_filter'][t]):
            continue
        pre = z['s0_agent_values'] if t == 0 else z['st_agent_values'][t - 1]
        done = z['s0_done'] if t == 0 else z['st_done'][t - 1]
        a = np.asarray(z['actions'][t], dtype=np.int64)
        raw = np.stack([t0[a // 5], t1[a % 5]], axis=-1)
        steps.append((np.asarray(pre, np.float64), raw, np.asarray(done, bool), float(z['st_separation_distance'][t]), t))
    return params, steps, z


def _world_rows(states, raw, done):
    """World.apply_safety_filter's rows: agent i against every j != i, inactive when i or j is done."""
    N = states.shape[0]
    js = np.array([[j for j in range(N) if j != i] for i in range(N)], dtype=np.int64).reshape(N, N - 1)
    others = states[js]
    u_o = raw[js]
    active = ~done[js] & ~done[:, None]
    return js, others, u_o, active


def _check_golden(z, t, N, js, safe, filt, idx, raw, name):
    dec = np.where(idx >= 0, idx + (idx >= np.arange(N)), -1)     # slot k of agent i is agent k + (k >= i)
    G.assert_same_mask(filt, z['st_safety_filtered'][t].astype(bool), f'{name} t={t} safety_filtered')
    G.assert_same_mask(dec, z['st_deconflicting_agent_index'][t], f'{name} t={t} deconflicting index')
    G.assert_close(np.linalg.norm(raw - safe, axis=-1), z['st_action_diff'][t], f'{name} t={t} action_diff')


@pytest.mark.parametrize('name', FILTER_FIXTURES)
def test_oracle_rows_reproduce_the_reference_filter(name):
    params, steps, z = _golden_rows(name)
    vg, _ = G.value_grid_for(params)
    assert steps, f"{name}: no filtered step"
    decisions = 0
    for states, raw, done, sep, t in steps:
        N = states.shape[0]
        js, others, u_o, active = _world_rows(states, raw, done)
        safe, filt, idx, _ = oracle_rows(params.asdict(), vg, states, others, raw, u_o, active, sep)
        _check_golden(z, t, N, js, safe, filt, idx, raw, name)
        decisions += int((~done).sum())
    assert decisions > 0


def test_filter_io_structs_match_the_c_header(tmp_path):
    from layered_safe_marl_b200 import _lib
    structs = [('lsm_filter_io', _lib.LsmFilterIo), ('lsm_lookup_io', _lib.LsmLookupIo)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lsm_b200.h"', 'int main(void) {']
    for cname, cls in structs:
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / 'io.c'
    exe = tmp_path / 'io.exe'
    src.write_text('\n'.join(lines))
    subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), '-o', str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    for cname, cls in structs:
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f'{cname}.{fname}']) == getattr(cls, fname).offset, f"offsetof({cname}, {fname})"


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _params(dyn, f32):
    args = G.default_args(dynamics_type='double_integrator' if dyn == 0 else 'airtaxi', num_agents=8 if dyn == 0 else 10,
                          use_safety_filter=True, interp_float32=f32)
    return cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags({}))


def _grid(dyn):
    return hj_grid.synthetic_di_grid() if dyn == 0 else hj_grid.synthetic_airtaxi_grid()


def _random_rows(dyn, B, M, rng, spread=1.0):
    if dyn == 0:
        ego = np.concatenate([rng.uniform(-spread, spread, (B, 2)), rng.uniform(-0.5, 0.5, (B, 2))], axis=-1)
        oth = np.concatenate([rng.uniform(-spread, spread, (B, M, 2)), rng.uniform(-0.5, 0.5, (B, M, 2))], axis=-1)
        ua, uo = rng.choice(np.linspace(-0.5, 0.5, 5), (B, 2)), rng.choice(np.linspace(-0.5, 0.5, 5), (B, M, 2))
    else:
        vmin, vmax = cfg.AirTaxiConfig.V_MIN, cfg.AirTaxiConfig.V_MAX
        ego = np.concatenate([rng.uniform(-3 * spread, 3 * spread, (B, 2)), rng.uniform(-4, 4, (B, 1)),
                              rng.uniform(vmin, vmax, (B, 1))], axis=-1)
        oth = np.concatenate([rng.uniform(-3 * spread, 3 * spread, (B, M, 2)), rng.uniform(-4, 4, (B, M, 1)),
                              rng.uniform(vmin, vmax, (B, M, 1))], axis=-1)
        ua = np.stack([rng.choice(np.linspace(-0.1, 0.1, 5), B), rng.choice(np.linspace(-0.001, 0.002, 5), B)], -1)
        uo = np.stack([rng.choice(np.linspace(-0.1, 0.1, 5), (B, M)), rng.choice(np.linspace(-0.001, 0.002, 5), (B, M))], -1)
    return ego, oth, ua, uo


def _edge_case_rows(dyn, rng, M=5):
    """Masked slots, all slots masked, out-of-grid and NaN states, rows beyond coordination range, exact value ties
    (an other duplicated into two slots) and all-inf values."""
    ego, oth, ua, uo = _random_rows(dyn, 64, M, rng, spread=0.5)
    act = np.ones((64, M), bool)
    act[0:8, ::2] = False                          # masked slots
    act[8:12] = False                              # every slot masked
    oth[12:16, :, 0] += 40.0                       # others far outside the grid box and the coordination range
    ego[16:20, 1] -= 7.0                           # ego outside the grid box in y, others still in range
    ego[20:22, 2] = np.nan                         # NaN ego: every value +inf
    oth[22:26, 1, 3] = np.nan                      # one NaN other
    oth[26:28, 0, 0] = np.nan                      # NaN distance in the first slot
    oth[28:36, 1] = oth[28:36, 0]                  # exact value ties: the first slot wins
    uo[28:36, 1] = uo[28:36, 0]
    oth[36:40, 2:] = oth[36:40, 1:2]               # three-way tie
    oth[40:44] = np.nan                            # all-inf values (NaN others)
    return ego, oth, ua, uo, act


def _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, act, sep, what):
    import torch
    d = sf.device
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=d)
    sep_t = None if sep is None else (t(sep) if np.ndim(sep) else float(sep))
    safe, filt, idx, val = sf.apply(t(ego), t(oth), t(ua), t(uo), None if act is None else t(act), sep_t)
    torch.cuda.synchronize()
    o_safe, o_filt, o_idx, o_val = oracle_rows(params.asdict(), vg, ego, oth, ua, uo, act, sep, rel_form=1)
    safe, filt, idx, val = safe.cpu().numpy(), filt.cpu().numpy(), idx.cpu().numpy(), val.cpu().numpy()
    assert np.array_equal(idx, o_idx), f"{what}: index differs at rows {np.argwhere(idx != o_idx)[:5].ravel()}"
    assert np.array_equal(filt, o_filt), f"{what}: filtered differs at rows {np.argwhere(filt != o_filt)[:5].ravel()}"
    assert np.array_equal(safe, o_safe), f"{what}: safe_action differs at rows {np.argwhere((safe != o_safe).any(-1))[:5].ravel()}"
    assert np.array_equal(val, o_val), f"{what}: value differs at rows {np.argwhere(val != o_val)[:5].ravel()}"
    return filt


@pytest.mark.gpu
@pytest.mark.parametrize('dyn', [0, 1])
@pytest.mark.parametrize('f32', [False, True])
def test_operator_matches_the_oracle_bit_for_bit(dyn, f32):
    from layered_safe_marl_b200 import SafetyFilter
    params, vg = _params(dyn, f32), _grid(dyn)
    sf = SafetyFilter('double_integrator' if dyn == 0 else 'airtaxi', value_grid=vg, interp_float32=f32)
    rng = np.random.default_rng(100 + 2 * dyn + f32)
    M = 7 if dyn == 0 else 9
    ego, oth, ua, uo = _random_rows(dyn, 4096, M, rng)
    filt = _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, None, None, 'random')
    assert 0 < filt.sum() < filt.size
    sep = rng.uniform(0.0, 1.0, 4096) * params.separation_distance_target
    _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, rng.random((4096, M)) < 0.7, sep, 'random, masked, per-row sep')
    _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, None, 0.25 * params.separation_distance_target, 'scalar sep')
    ego, oth, ua, uo, act = _edge_case_rows(dyn, rng)
    _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, act, None, 'edge cases')
    for M in (0, 1):
        ego, oth, ua, uo = _random_rows(dyn, 333, M, rng)
        _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, None, None, f'M={M}')
    ego, oth, ua, uo = _random_rows(dyn, 0, 3, rng)
    _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, None, None, 'B=0')


@pytest.mark.gpu
def test_operator_large_batch_matches_the_oracle():
    from layered_safe_marl_b200 import SafetyFilter
    params, vg = _params(0, False), _grid(0)
    sf = SafetyFilter('double_integrator', value_grid=vg)
    rng = np.random.default_rng(7)
    B = (1 << 21) + 77
    ego, oth, ua, uo = _random_rows(0, B, 2, rng)
    _compare_to_oracle(sf, params, vg, ego, oth, ua, uo, None, None, 'B > 2^21')


@pytest.mark.gpu
@pytest.mark.parametrize('name', FILTER_FIXTURES)
def test_operator_reproduces_the_reference_filter(name):
    import torch
    from layered_safe_marl_b200 import SafetyFilter
    params, steps, z = _golden_rows(name)
    vg, _ = G.value_grid_for(params)
    sf = SafetyFilter('double_integrator' if params.dynamics == 0 else 'airtaxi', value_grid=vg,
                      interp_float32=bool(params.flags & cfg.FLAG_INTERP_FLOAT32))
    for states, raw, done, sep, t in steps:
        N = states.shape[0]
        d = sf.device
        safe, filt, dec = sf.apply_world(torch.as_tensor(states[None], device=d), torch.as_tensor(raw[None], device=d),
                                         torch.as_tensor(done[None], device=d), sep)
        safe, filt, dec = safe[0].cpu().numpy(), filt[0].cpu().numpy(), dec[0].cpu().numpy()
        G.assert_same_mask(filt, z['st_safety_filtered'][t].astype(bool), f'{name} t={t} safety_filtered')
        G.assert_same_mask(dec, z['st_deconflicting_agent_index'][t], f'{name} t={t} deconflicting index')
        G.assert_close(np.linalg.norm(raw - safe, axis=-1), z['st_action_diff'][t], f'{name} t={t} action_diff')


def _lookup_points(dyn, rng):
    lo = np.array(hj_grid.DI_GRID_LO if dyn == 0 else hj_grid.AIRTAXI_GRID_LO)
    hi = np.array(hj_grid.DI_GRID_HI if dyn == 0 else hj_grid.AIRTAXI_GRID_HI)
    nd = lo.size
    inner = lo + (hi - lo) * rng.random((2000, nd))
    boundary = np.concatenate([np.tile(lo, (nd, 1)), np.tile(hi, (nd, 1)), lo + (hi - lo) * rng.integers(0, 2, (64, nd))])
    outside = lo + (hi - lo) * rng.uniform(-1.0, 2.0, (256, nd))
    nan = inner[:16].copy()
    nan[np.arange(16), np.arange(16) % nd] = np.nan
    pts = [inner, boundary, outside, nan]
    if dyn == 1:
        wrap = inner[:256].copy()
        wrap[:, 2] += rng.choice([-4 * np.pi, -2 * np.pi, 2 * np.pi, 6 * np.pi], 256)
        pts.append(wrap)
    return np.concatenate(pts)


@pytest.mark.gpu
@pytest.mark.parametrize('dyn', [0, 1])
@pytest.mark.parametrize('f32', [False, True])
def test_values_and_gradients_match_the_oracle(dyn, f32):
    import torch
    from layered_safe_marl_b200 import SafetyFilter
    params, vg = _params(dyn, f32), _grid(dyn)
    sf = SafetyFilter('double_integrator' if dyn == 0 else 'airtaxi', value_grid=vg, interp_float32=f32)
    rng = np.random.default_rng(11 + dyn)
    rel = _lookup_points(dyn, rng)
    sep = rng.uniform(0, 1, rel.shape[0]) * params.separation_distance_target
    v, g = sf.values(rel=torch.as_tensor(rel, device=sf.device), gradients=True, separation_distance=torch.as_tensor(sep, device=sf.device))
    ov, og = oracle_lookup(params.asdict(), vg, rel=rel, sep=sep)
    assert np.array_equal(v.cpu().numpy(), ov)
    assert np.array_equal(g.cpu().numpy(), og, equal_nan=True)
    assert np.isinf(ov[-16 - (256 if dyn else 0):][:16]).all()
    ego, oth, _, _ = _random_rows(dyn, 3000, 1, rng)
    oth = oth[:, 0]
    v, g = sf.values(ego=torch.as_tensor(ego, device=sf.device), other=torch.as_tensor(oth, device=sf.device), gradients=True)
    ov, og = oracle_lookup(params.asdict(), vg, ego=ego, other=oth, rel_form=1)
    assert np.array_equal(v.cpu().numpy(), ov)
    assert np.array_equal(g.cpu().numpy(), og, equal_nan=True)


# ------------------------------------------------------------------------------------------------------------------
# against the environment's own step
# ------------------------------------------------------------------------------------------------------------------
ENV_CASES = [
    ('cfg2', dict(dynamics_type='double_integrator', num_agents=8), 4096, True),
    ('cfg3', dict(dynamics_type='airtaxi', num_agents=10), 16384, True),
    ('cfg3_obst4', dict(dynamics_type='airtaxi', num_agents=10, num_obstacles=4, obstacle_extension=True), 16384, True),
    ('generic_di5', dict(dynamics_type='double_integrator', num_agents=5), 1024, False),
    ('generic_at6', dict(dynamics_type='airtaxi', num_agents=6), 1024, False),
]


def _curriculum_sep(params, ratios):
    lib = O.lib()
    lib.lsmo_curriculum.argtypes = [ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p]
    lib.lsmo_curriculum.restype = None
    p = O.make_params(params.asdict())
    out = np.zeros(12)
    seps, filt = np.zeros(len(ratios)), np.zeros(len(ratios), bool)
    cache = {}
    for k, r in enumerate(ratios):
        if r not in cache:
            lib.lsmo_curriculum(ctypes.byref(p), float(r), out.ctypes.data_as(ctypes.c_void_p))
            cache[r] = (out[9], out[11] != 0.0)
        seps[k], filt[k] = cache[r]
    return seps, filt


@pytest.mark.gpu
@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('case', [c[0] for c in ENV_CASES])
def test_apply_world_matches_the_env_step(case, f32):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, SafetyFilter, layout as LY
    _, kw, n, spec = next(c for c in ENV_CASES if c[0] == case)
    args = G.default_args(use_safety_filter=True, episode_length=40, interp_float32=f32, **kw)
    env = B200GraphVecEnv(args, num_envs=n, seed=5)
    assert env.launch_info()['specialised'] == int(spec)
    sf = SafetyFilter.of(env)
    episode = env.params.num_total_episode - 1
    env.reset(episode)
    N = env.N
    t0, t1 = O.action_tables(env.params.dynamics)
    t0, t1 = torch.as_tensor(t0, device=env.device), torch.as_tensor(t1, device=env.device)
    gen = torch.Generator(device=env.device).manual_seed(3)
    checked = 0
    for step in range(20):
        states = torch.stack([env.agent_f64[k] for k in (LY.AF_X, LY.AF_Y, LY.AF_S2, LY.AF_S3)], dim=-1).clone()
        done = env.agent_i32[LY.AI_DONE].clone().bool()
        ratios = env.env_f64[LY.EF_CURRICULUM_RATIO].cpu().numpy()
        sep, world_filter = _curriculum_sep(env.params, ratios)
        assert world_filter.all()
        if spec and step % 5 == 0:
            # values(ego, other) of every ordered pair == the pipeline's pair values of the same state (raw: grid's sep)
            pv = torch.full((n, N, N), float('nan'), dtype=torch.float64, device=env.device)
            env._check(env.lib.lsm_debug_pair_values(env._h, ctypes.c_void_p(pv.data_ptr()), env._stream()), 'pair values')
            e = states.view(n, N, 1, 4).expand(n, N, N, 4).reshape(-1, 4)
            o = states.view(n, 1, N, 4).expand(n, N, N, 4).reshape(-1, 4)
            v, _ = sf.values(ego=e, other=o)
            live = (~done.view(n, N, 1) & ~done.view(n, 1, N) & ~torch.eye(N, dtype=torch.bool, device=env.device)).reshape(-1)
            if step > 0:
                assert torch.equal(v[live], pv.reshape(-1)[live])
        a = torch.randint(0, 25, (n, N), device=env.device, dtype=torch.int32, generator=gen)
        raw = torch.stack([t0[(a // 5).long()], t1[(a % 5).long()]], dim=-1)
        safe, filt, dec = sf.apply_world(states, raw, done, torch.as_tensor(sep, device=env.device))
        env.step(a, episode)
        # an env that auto-reset in this step holds its new episode's state and bookkeeping
        live = ~done & ~env.env_i32[LY.EI_JUST_RESET].bool().view(n, 1)
        done = done & ~env.env_i32[LY.EI_JUST_RESET].bool().view(n, 1)
        env_safe = env.safe_action
        env_filt = env.agent_i32[LY.AI_SAFETY_FILTERED].bool()
        env_dec = env.agent_i32[LY.AI_DECONFLICT_IDX]
        assert torch.equal(filt[live], env_filt[live]), f"step {step}: filtered"
        assert torch.equal(dec[live], env_dec[live]), f"step {step}: deconflict"
        assert bool((dec[done] == -1).all()) and bool((env_dec[done] == -1).all())
        if spec or env.params.dynamics == 0:
            assert torch.equal(safe[live], env_safe[live]), f"step {step}: safe action"
        else:   # generic airtaxi kernel: literal relative-state form
            assert float((safe[live] - env_safe[live]).abs().max()) <= 1e-12
        checked += int(env_filt[live].sum())
    assert checked > 0


@pytest.mark.gpu
def test_of_env_on_a_shape_library_and_a_side_stream():
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, SafetyFilter, layout as LY
    args = G.default_args(dynamics_type='airtaxi', num_agents=6, use_safety_filter=True, episode_length=40,
                          specialise_shape=True)
    env = B200GraphVecEnv(args, num_envs=256, seed=2)
    assert env.launch_info()['specialised'] == 1
    sf = SafetyFilter.of(env)
    env.reset(env.params.num_total_episode - 1)
    states = torch.stack([env.agent_f64[k] for k in (LY.AF_X, LY.AF_Y, LY.AF_S2, LY.AF_S3)], dim=-1).clone()
    done = env.agent_i32[LY.AI_DONE].bool()
    raw = torch.zeros((256, 6, 2), dtype=torch.float64, device=env.device)
    ref = sf.apply_world(states, raw, done)
    side = torch.cuda.Stream(device=env.device)
    side.wait_stream(torch.cuda.current_stream(env.device))
    with torch.cuda.stream(side):
        big = states.repeat(64, 1, 1)            # produced on the side stream, consumed there
        out = sf.apply_world(big, raw.repeat(64, 1, 1), done.repeat(64, 1))
    torch.cuda.current_stream(env.device).wait_stream(side)
    for r, o in zip(ref, out):
        assert torch.equal(o[:256], r) and torch.equal(o[-256:], r)


@pytest.mark.gpu
def test_errors_are_reported():
    import torch
    from layered_safe_marl_b200 import SafetyFilter, _lib
    sf = SafetyFilter('double_integrator', value_grid=hj_grid.synthetic_di_grid())
    with pytest.raises(ValueError):
        sf.apply(torch.zeros((4, 4), dtype=torch.float64), torch.zeros((4, 2, 4), dtype=torch.float64),
                 torch.zeros((4, 2)), torch.zeros((4, 2, 2)))
    # a handle without a value grid
    lib = _lib.load()
    from layered_safe_marl_b200.vec_env import make_config_struct
    h = ctypes.c_void_p()
    _lib.check(lib.lsm_create(ctypes.byref(make_config_struct(_params(0, False))), ctypes.byref(h)), 'lsm_create')
    try:
        io = _lib.LsmFilterIo()
        io.num_rows = 1
        assert lib.lsm_safety_filter(h, ctypes.byref(io), None) != 0
        assert b'value grid' in lib.lsm_last_error()
        lio = _lib.LsmLookupIo()
        lio.num_points = 1
        assert lib.lsm_hj_lookup(h, ctypes.byref(lio), None) != 0
    finally:
        lib.lsm_destroy(h)
