"""The HJ grid lookups on grid geometries users bind, not only the synthetic lattices.

Every lookup has branches that depend on the bound grid: the pair kernel's compile-time periodic mask and its run-time
twin (pair_rt), the out-of-line wrap of relative headings outside [lo, hi), the exact division by the spacing
(div_exact), the corner-packed table (n slots on periodic dims, n + 1 elsewhere) and the 2 GiB rule that skips it, the
padded 5-D gradient rows. GEOMETRIES is a family of grids that reaches each of them:

  * the default grids, as controls;
  * small odd and even shapes, 2-node dims of every kind (2-node periodic heading included);
  * asymmetric domains whose spacing is not a short binary fraction;
  * periodic masks other than the pair kernel's (double integrator with dim 2 periodic, airtaxi with none): pair_rt;
  * headings on [0, 2pi): about half of the in-grid relative headings take the slow wrap;
  * a double-integrator grid whose packed table would exceed 2 GiB: the scattered lookup;
  * TTR grids of another shape, with headings on [0, 2pi) and with a 2-node speed dim.

CPU: the oracle's interpolation equals the reference stub's on every geometry, in both arithmetics, and div_exact equals
the division on every spacing. GPU: SafetyFilter lookups and the filter, the env pipeline and its pair values against
the oracle bit for bit; re-binding a live handle; refused grids leave the bound one in place.
"""
from __future__ import annotations

import ctypes
import functools
import math
import os
import sys

import numpy as np
import pytest

import _golden as G
from test_host_logic import check_div_exact

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))

import oracle_env as O  # noqa: E402
from layered_safe_marl_b200 import config as cfg, hj_grid  # noqa: E402

PI = math.pi
VMIN, VMAX = cfg.AirTaxiConfig.V_MIN, cfg.AirTaxiConfig.V_MAX
DI_LO, DI_HI = hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI
AT_LO, AT_HI = hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI
TTR_LO, TTR_HI = hj_grid.TTR_GRID_LO, hj_grid.TTR_GRID_HI
DI_NOPER = (False,) * 4
DI_PER2 = (False, False, True, False)
AT_PER = (False, False, True, False, False)
TTR_PER = (False, False, True, False)

# name: (kind, shape, lo, hi, periodic); kind 'di' / 'at' value grids, 'ttr' time-to-reach grids
GEOMETRIES = {
    'di_default': ('di', hj_grid.DI_GRID_SHAPE, DI_LO, DI_HI, DI_NOPER),
    'di_odd': ('di', (7, 9, 5, 3), DI_LO, DI_HI, DI_NOPER),
    'di_even': ('di', (8, 6, 4, 10), DI_LO, DI_HI, DI_NOPER),
    'di_2node': ('di', (2, 5, 2, 2), DI_LO, DI_HI, DI_NOPER),
    'di_asym': ('di', (37, 29, 13, 11), (-3.7, -4.1, -1.3, -0.9), (5.3, 3.9, 1.1, 1.2), DI_NOPER),
    'di_per2': ('di', (9, 9, 12, 7), DI_LO, DI_HI, DI_PER2),                 # pair_rt
    'di_per2_2node': ('di', (9, 7, 2, 5), DI_LO, DI_HI, DI_PER2),            # pair_rt, 2-node periodic dim
    # 54 M cells: 218 MB of values, 870 MB of gradients; the packed table (3.7 GB) is not built
    'di_huge': ('di', (121, 121, 61, 61), DI_LO, DI_HI, DI_NOPER),
    'at_default': ('at', hj_grid.AIRTAXI_GRID_SHAPE, AT_LO, AT_HI, AT_PER),
    'at_odd_even': ('at', (9, 11, 6, 3, 4), AT_LO, AT_HI, AT_PER),
    'at_2node': ('at', (2, 7, 2, 2, 3), AT_LO, AT_HI, AT_PER),               # 2-node x, heading (periodic), speed
    'at_asym': ('at', (37, 23, 17, 5, 7), (-3.7, -6.2, -PI, VMIN, VMIN), (5.3, 4.9, PI, VMAX, VMAX), AT_PER),
    'at_noper': ('at', (11, 11, 9, 3, 3), AT_LO, AT_HI, (False,) * 5),      # pair_rt
    'at_theta_2pi': ('at', (13, 13, 12, 4, 4), (-5.5, -5.5, 0.0, VMIN, VMIN), (5.5, 5.5, 2 * PI, VMAX, VMAX), AT_PER),
    'ttr_default': ('ttr', hj_grid.TTR_GRID_SHAPE, TTR_LO, TTR_HI, TTR_PER),
    'ttr_shape': ('ttr', (29, 35, 16, 7), TTR_LO, TTR_HI, TTR_PER),
    'ttr_theta_2pi': ('ttr', (33, 33, 20, 9), (-8.0, -8.0, 0.0, VMIN), (8.0, 8.0, 2 * PI, VMAX), TTR_PER),
    'ttr_2node_speed': ('ttr', (41, 41, 24, 2), TTR_LO, TTR_HI, TTR_PER),
}
VALUE_GRIDS = [k for k, v in GEOMETRIES.items() if v[0] != 'ttr']
SMALL_GRIDS = [k for k in GEOMETRIES if k != 'di_huge']


@functools.lru_cache(maxsize=None)
def grid(name) -> hj_grid.HjGrid:
    """The analytic synthetic values sampled on the geometry's lattice (values vary along every dim; on a geometry
    whose mask differs from the dynamics' own they are data on another lattice, which is all a lookup test needs)."""
    kind, shape, lo, hi, per = GEOMETRIES[name]
    if kind == 'ttr':
        g = hj_grid.synthetic_ttr_grid(shape=shape, lo=lo, hi=hi)
        assert g.periodic == per
        return g
    if kind == 'di':
        sep = cfg.DoubleIntegratorConfig.SEPARATION_DISTANCE
        stored = hj_grid.synthetic_di_stored_values(shape=shape, lo=lo, hi=hi)
    else:
        sep = cfg.AirTaxiConfig.SEPARATION_DISTANCE
        stored = hj_grid.synthetic_airtaxi_stored_values(shape=shape, lo=lo, hi=hi)
    return hj_grid.make_hj_handle(stored, lo, hi, per, sep, sep)


def probe_points(g, rng, nodes, inner):
    """Positions (K, ndim) where lookups go wrong: lattice nodes and +-1..8 ulps along one dim (node 0 and the last
    node of every dim included), the upper face (hi and hi - 1 ulp), random inner points, points outside the box and
    past the +-1e9-spacing clamp, NaN in each dim, and periodic dims shifted by whole periods (2 pi for a heading)."""
    lo, hi, sp = np.asarray(g.lo, float), np.asarray(g.hi, float), g.spacings
    nd, shape = g.ndim, np.asarray(g.shape)
    coords = g.coordinate_vectors()

    def box(k):
        return lo + (hi - lo) * rng.random((k, nd))

    pts = [box(inner)]
    for d in range(nd):
        idx = rng.integers(0, shape, (nodes, nd))
        idx[0] = 0
        idx[1] = shape - 1
        base = np.stack([coords[k][idx[:, k]] for k in range(nd)], axis=-1)
        pts.append(base)
        up, dn = base.copy(), base.copy()
        for _ in range(8):
            up, dn = up.copy(), dn.copy()
            up[:, d] = np.nextafter(up[:, d], np.inf)
            dn[:, d] = np.nextafter(dn[:, d], -np.inf)
            pts += [up, dn]
        face = box(4)
        face[:2, d] = hi[d]
        face[2:, d] = np.nextafter(hi[d], -np.inf)
        far = box(4)
        far[:, d] = [lo[d] - 3e9 * sp[d], hi[d] + 3e9 * sp[d], -1e300, 1e300]
        nan = box(1)
        nan[0, d] = np.nan
        pts += [face, far, nan]
        if g.periodic[d]:
            w = box(16)
            w[:, d] += (hi[d] - lo[d]) * rng.choice([-3.0, -1.0, 1.0, 2.0, 5.0], 16)
            pts.append(w)
    pts.append(lo + (hi - lo) * rng.uniform(-1.0, 2.0, (max(inner // 2, 8), nd)))
    return np.concatenate(pts)


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def _same(a, b):
    return a == b or (math.isnan(a) and math.isnan(b))


@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('name', SMALL_GRIDS)
def test_oracle_interpolation_matches_the_stub(name, f32):
    """lsmo_interpolate == the reference stub's Grid.interpolate, value and every gradient component, bit for bit."""
    sys.path.insert(0, os.path.join(REPO, 'oracle', 'ref_stubs'))
    import hj_reachability as hj
    g = grid(name)
    stub = hj.Grid(g.lo, g.hi, g.shape, tuple(d for d in range(g.ndim) if g.periodic[d]))
    s, keep = O.make_grid(g)
    pts = probe_points(g, np.random.default_rng(sum(map(ord, name)) + f32), nodes=3, inner=48)
    lib = O.lib()
    lib.lsmo_set_interp_float32(int(f32))
    hj.FLOAT32_INTERPOLATION = f32
    try:
        with np.errstate(over='ignore'):      # the float32 stub casts +-1e300 to +-inf, as jax does
            for x in pts:
                xc = (ctypes.c_double * g.ndim)(*x)
                want = float(stub.interpolate(g.values, x))
                got = lib.lsmo_interpolate(ctypes.byref(s), xc, ctypes.c_int(-1))
                assert _same(got, want), f"{name} f32={f32} x={x.tolist()}: value {got!r} vs stub {want!r}"
                if g.grads is None:
                    continue
                want_g = stub.interpolate(g.grads, x)
                for d in range(g.ndim):
                    got = lib.lsmo_interpolate(ctypes.byref(s), xc, ctypes.c_int(d))
                    assert _same(got, float(want_g[d])), f"{name} f32={f32} x={x.tolist()}: grad[{d}] {got!r} vs {want_g[d]!r}"
    finally:
        lib.lsmo_set_interp_float32(0)
        hj.FLOAT32_INTERPOLATION = False


@pytest.mark.parametrize('name', list(GEOMETRIES))
def test_div_exact_equals_division_on_every_spacing(name):
    _, shape, lo, hi, per = GEOMETRIES[name]
    check_div_exact(lo, hi, shape, per, name, np.random.default_rng(5))


def test_geometry_family_reaches_every_branch():
    """The family holds what the docstring promises; the pair kernels' masks are kPairPeriodic (lsm_kernel_spec.cuh)."""
    pair_mask = {'di': 0, 'at': 1 << 2}
    masks = {n: sum(1 << d for d, p in enumerate(v[4]) if p) for n, v in GEOMETRIES.items()}
    assert {n for n in VALUE_GRIDS if masks[n] != pair_mask[GEOMETRIES[n][0]]} == {'di_per2', 'di_per2_2node', 'at_noper'}
    for kind in ('di', 'at', 'ttr'):
        assert any(2 in v[1] for v in GEOMETRIES.values() if v[0] == kind), kind
    assert any(v[1][d] == 2 and v[4][d] for v in GEOMETRIES.values() for d in range(len(v[1])))   # 2-node periodic
    _, shape, _, _, per = GEOMETRIES['di_huge']
    packed = math.prod(n if p else n + 1 for n, p in zip(shape, per)) * 16 * 4
    assert packed > 2 << 30 and math.prod(shape) < 2 ** 31


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _dynamics(name):
    return 'double_integrator' if GEOMETRIES[name][0] == 'di' else 'airtaxi'


def _tensor(a, device):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a), device=device)


def _lookups(sf, g, rng):
    """Outputs of one handle on seeded inputs: values + gradients of relative states (per-point separation), of
    (ego, other) pairs, and the filter over random and edge-case rows. Same rng state -> same inputs."""
    from test_safety_filter_op import _edge_case_rows, _random_rows
    import torch
    dyn = 0 if sf.ndim == 4 else 1
    rel = probe_points(g, rng, nodes=16, inner=2000)
    sep = rng.uniform(0, 1, rel.shape[0]) * sf.params.separation_distance_target
    v, gr = sf.values(rel=_tensor(rel, sf.device), gradients=True, separation_distance=_tensor(sep, sf.device))
    # positions spread over twice the box: relative states inside and outside it
    spread = float(np.max(np.abs([g.lo[0], g.hi[0], g.lo[1], g.hi[1]])))
    ego, oth, ua, uo = _random_rows(dyn, 3000, 1, rng, spread=spread if dyn == 0 else spread / 3.0)
    pv, pg = sf.values(ego=_tensor(ego, sf.device), other=_tensor(oth[:, 0], sf.device), gradients=True)
    ego2, oth2, ua2, uo2 = _random_rows(dyn, 2048, 5, rng, spread=spread / 2 if dyn == 0 else spread / 6.0)
    act = rng.random((2048, 5)) < 0.8
    rows = [(ego2, oth2, ua2, uo2, act, None), _edge_case_rows(dyn, rng) + (None,)]
    out = dict(rel=rel, sep=sep, v=v, g=gr, ego=ego, oth=oth[:, 0], pv=pv, pg=pg, rows=rows)
    out['filter'] = [sf.apply(*[_tensor(a, sf.device) for a in r[:5]], r[5]) for r in rows]
    torch.cuda.synchronize(sf.device)
    return out


def _check_against_oracle(sf, g, rng, what):
    from test_safety_filter_op import _compare_to_oracle, oracle_lookup
    out = _lookups(sf, g, rng)
    p = sf.params.asdict()
    ov, og = oracle_lookup(p, g, rel=out['rel'], sep=out['sep'])
    bad = np.argwhere(out['v'].cpu().numpy() != ov).ravel()
    assert bad.size == 0, f"{what}: rel value differs at {bad.size} points, first x={out['rel'][bad[0]].tolist()}"
    assert np.array_equal(out['g'].cpu().numpy(), og, equal_nan=True), f"{what}: rel gradient"
    ov, og = oracle_lookup(p, g, ego=out['ego'], other=out['oth'], rel_form=1)
    assert np.array_equal(out['pv'].cpu().numpy(), ov), f"{what}: (ego, other) value"
    assert np.array_equal(out['pg'].cpu().numpy(), og, equal_nan=True), f"{what}: (ego, other) gradient"
    for k, (ego, oth, ua, uo, act, sep) in enumerate(out['rows']):
        _compare_to_oracle(sf, sf.params, g, ego, oth, ua, uo, act, sep, f'{what}: filter rows {k}')


def _env(name, f32, N=None, tuning=None, ttr=None, n=4):
    from layered_safe_marl_b200 import B200GraphVecEnv
    dyn = _dynamics(name)
    N = N or (8 if dyn == 'double_integrator' else 10)
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=True, interp_float32=f32)
    return B200GraphVecEnv(args, num_envs=n, seed=1, value_grid=grid(name), ttr_grid=None if ttr is None else grid(ttr),
                           tuning=tuning)


@pytest.mark.gpu
@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('name', VALUE_GRIDS)
def test_filter_lookups_match_the_oracle(name, f32):
    """SafetyFilter.values (relative and (ego, other) form, gradients) and .apply on three handles: a specialised one
    with the packed table (none for di_huge: over 2 GiB), a specialised env's with packed_grid=0, and a generic-shape
    env's (no packed table, no padded gradient rows)."""
    from layered_safe_marl_b200 import SafetyFilter
    g = grid(name)
    seed = sum(map(ord, name)) + f32
    sf = SafetyFilter(_dynamics(name), value_grid=g, interp_float32=f32)
    _check_against_oracle(sf, g, np.random.default_rng(seed), f'{name} packed')
    sf.close()
    for label, N, tuning in (('packed_grid=0', None, dict(packed_grid=0)), ('generic', 5 if g.ndim == 4 else 6, None)):
        env = _env(name, f32, N=N, tuning=tuning)
        assert env.launch_info()['specialised'] == int(label != 'generic')
        _check_against_oracle(SafetyFilter.of(env), g, np.random.default_rng(seed), f'{name} {label}')
        env.close()


# env pipeline: (dynamics, agents, world_size, value grid, TTR grid); cfg2 / cfg3 run the specialised pipeline
ENV_CASES = {
    'cfg2_di_per2': ('double_integrator', 8, 4, 'di_per2', None),              # pair_rt
    'cfg2_di_per2_2node': ('double_integrator', 8, 4, 'di_per2_2node', None),  # pair_rt, 2-node periodic dim
    'cfg2_di_2node': ('double_integrator', 8, 4, 'di_2node', None),
    'cfg2_di_asym': ('double_integrator', 8, 4, 'di_asym', None),
    'cfg2_di_huge': ('double_integrator', 8, 4, 'di_huge', None),              # no packed table (> 2 GiB)
    'cfg3_at_noper': ('airtaxi', 10, 6, 'at_noper', 'ttr_shape'),              # pair_rt
    'cfg3_at_theta_2pi': ('airtaxi', 10, 6, 'at_theta_2pi', 'ttr_theta_2pi'),  # slow wrap
    'cfg3_at_2node': ('airtaxi', 10, 6, 'at_2node', 'ttr_2node_speed'),
    'generic_di5_per2': ('double_integrator', 5, 4, 'di_per2', None),
    'generic_di5_per2_2node': ('double_integrator', 5, 4, 'di_per2_2node', None),
    'generic_at6_theta_2pi': ('airtaxi', 6, 6, 'at_theta_2pi', 'ttr_theta_2pi'),
    'generic_at6_2node': ('airtaxi', 6, 6, 'at_2node', 'ttr_2node_speed'),
}


def _pair_value_check(env, sf, what):
    """lsm_debug_pair_values == SafetyFilter.values(ego, other) of the current state on every live pair; returns the
    live mask (n, N, N)."""
    import torch
    from layered_safe_marl_b200 import layout as LY
    n, N = env.n, env.N
    pv = torch.full((n, N, N), float('nan'), dtype=torch.float64, device=env.device)
    env._check(env.lib.lsm_debug_pair_values(env._h, ctypes.c_void_p(pv.data_ptr()), env._stream()), 'pair values')
    states = torch.stack([env.agent_f64[k] for k in (LY.AF_X, LY.AF_Y, LY.AF_S2, LY.AF_S3)], dim=-1)
    done = env.agent_i32[LY.AI_DONE].bool()
    e = states.view(n, N, 1, 4).expand(n, N, N, 4).reshape(-1, 4)
    o = states.view(n, 1, N, 4).expand(n, N, N, 4).reshape(-1, 4)
    v, _ = sf.values(ego=e, other=o)
    live = (~done.view(n, N, 1) & ~done.view(n, 1, N) & ~torch.eye(N, dtype=torch.bool, device=env.device))
    flat = live.reshape(-1)
    bad = (v[flat] != pv.reshape(-1)[flat]).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.numel()} pair values differ from SafetyFilter.values"
    return live.cpu().numpy()


def _node_state(env, g, state, rng):
    """Pair (0, 1) of every env on a lattice node of the bound grid: agent 0 at the origin (airtaxi: heading 0), agent 1
    placed so that their relative state is the node. Every third env takes the last node of every dim, the next one
    node 0 of every dim, the rest random nodes."""
    s = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in state.items()}
    av = s['agent_values']
    n = av.shape[0]
    shape = np.asarray(g.shape)
    idx = rng.integers(0, shape, (n, g.ndim))
    idx[0::3] = shape - 1
    idx[1::3] = 0
    node = [vec[idx[:, d]] for d, vec in enumerate(g.coordinate_vectors())]
    zero = np.zeros(n)
    if g.ndim == 4:
        av[:, 0] = np.stack(node, axis=-1)      # rel = ego - other, other at the origin at rest
        av[:, 1] = 0.0
    else:
        av[:, 0] = np.stack([zero, zero, zero, node[3]], axis=-1)
        av[:, 1] = np.stack([node[0], node[1], node[2], node[4]], axis=-1)
    s['agent_values'] = av
    return s


def _refused_grids(g, device):
    """Descriptors of g's dimensionality the library must refuse: a 1-node dim, exactly 2^31 cells, and a cell count
    whose product overflows 64 bits. They point at a small valid device buffer, so a refusal that came after a read
    would still not fault."""
    import torch
    from layered_safe_marl_b200 import _lib
    buf = torch.zeros(64, dtype=torch.float32, device=device)
    one = list(g.shape)
    one[1] = 1
    big = [1024, 1024, 1024, 2] if g.ndim == 4 else [1024, 1024, 512, 2, 2]
    huge = [2 ** 31 - 1] * g.ndim
    descs = []
    for shape in (one, big, huge):
        d = _lib.LsmGridDesc()
        d.ndim = g.ndim
        for k in range(g.ndim):
            d.shape[k] = shape[k]
            d.periodic[k] = int(bool(g.periodic[k]))
            d.lo[k] = float(g.lo[k])
            d.hi[k] = float(g.hi[k])
        d.separation_distance = float(g.separation_distance)
        d.ttr_max = float(g.ttr_max)
        d.values = buf.data_ptr()
        d.grads = buf.data_ptr()
        descs.append((shape, d))
    return buf, descs


def _refuse(lib, h, setter, g, device):
    keep, descs = _refused_grids(g, device)
    for shape, d in descs:
        rc = getattr(lib, setter)(h, ctypes.byref(d))
        msg = lib.lsm_last_error()
        assert rc == 2, f"{setter} shape {shape}: returned {rc}, expected 2 ({msg})"
        if shape[1] != 1:
            assert b'cells' in msg, msg
    del keep


@pytest.mark.gpu
@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('case', list(ENV_CASES))
def test_env_pipeline_matches_the_oracle(case, f32):
    """Seeded batches with the filter on at a late curriculum episode through the CUDA env and the C oracle, both bound to
    the case's grids (test_cuda_parity's bar); then, on the specialised pipeline, its pair values against SafetyFilter
    after steps and after pair (0, 1) was put on lattice nodes. cfg3_at_theta_2pi first has both grids re-bound with
    refused descriptors: the bound ones stay in use."""
    import torch
    from test_cuda_parity import _compare_with_oracle
    from layered_safe_marl_b200 import SafetyFilter
    dyn, N, world, vname, tname = ENV_CASES[case]
    args = G.default_args(dynamics_type=dyn, num_agents=N, world_size=world, use_safety_filter=True, episode_length=40,
                          interp_float32=f32)
    flags = G.BinaryFlags(dict(POTENTIAL_CONFLICT=True) if dyn == 'airtaxi' else {})
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = grid(vname), (grid(tname) if tname else None)

    def refuse(env):
        _refuse(env.lib, env._h, 'lsm_set_value_grid', vg, env.device)
        _refuse(env.lib, env._h, 'lsm_set_ttr_grid', tg, env.device)

    ora, cu = _compare_with_oracle(args, flags, n=128, T=10, episode=params.num_total_episode - 1, seed=21,
                                   auto_reset=True, grids=(vg, tg), prepare=refuse if case == 'cfg3_at_theta_2pi' else None)
    env = cu.env
    spec = env.launch_info()['specialised'] == 1
    assert spec == case.startswith('cfg')
    if not spec:
        return
    sf = SafetyFilter.of(env)
    rng = np.random.default_rng(4)
    for step in range(3):
        env.step(torch.as_tensor(rng.integers(0, 25, (env.n, N)).astype(np.int32), device=env.device),
                 params.num_total_episode - 1)
        _pair_value_check(env, sf, f'{case} step {step}')
    env.set_state(_node_state(env, vg, env.get_state(), rng))
    env.observe()
    live = _pair_value_check(env, sf, f'{case} on lattice nodes')
    assert live[0::3, 0, 1].sum() > 0 and live[1::3, 0, 1].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('packed', [True, False])
@pytest.mark.parametrize('dyn', ['double_integrator', 'airtaxi'])
def test_rebinding_a_live_handle(dyn, packed, f32):
    """lsm_set_value_grid on a handle already in use, with a second geometry and then a third (other mask, shape and
    spacing): every lookup equals a fresh handle bound to that grid, bit for bit, and the oracle."""
    from layered_safe_marl_b200 import SafetyFilter, _lib
    from layered_safe_marl_b200.vec_env import _DeviceGrid
    seq = ['di_default', 'di_per2', 'di_odd'] if dyn == 'double_integrator' else ['at_default', 'at_theta_2pi', 'at_2node']

    def handle(name):
        if packed:
            return SafetyFilter(dyn, value_grid=grid(name), interp_float32=f32), None
        env = _env(name, f32, tuning=dict(packed_grid=0))
        return SafetyFilter.of(env), env

    sf, env = handle(seq[0])
    _lookups(sf, grid(seq[0]), np.random.default_rng(0))
    bound = []
    for k, name in enumerate(seq[1:]):
        dg = _DeviceGrid(grid(name), sf.device)
        bound.append(dg)
        _lib.check(sf.lib.lsm_set_value_grid(sf._h, ctypes.byref(dg.desc)), 'lsm_set_value_grid')
        fresh, fresh_env = handle(name)
        got, want = _lookups(sf, grid(name), np.random.default_rng(k)), _lookups(fresh, grid(name), np.random.default_rng(k))
        for key in ('v', 'g', 'pv', 'pg'):
            a, b = got[key].cpu().numpy(), want[key].cpu().numpy()
            assert np.array_equal(a, b, equal_nan=True), f"{dyn} re-bound to {name}: {key}"
        for r, (a, b) in enumerate(zip(got['filter'], want['filter'])):
            for x, y in zip(a, b):
                assert np.array_equal(x.cpu().numpy(), y.cpu().numpy()), f"{dyn} re-bound to {name}: filter rows {r}"
        _check_against_oracle(sf, grid(name), np.random.default_rng(k + 10), f'{dyn} re-bound to {name}')
        fresh.close()
        if fresh_env is not None:
            fresh_env.close()
    sf.close()
    if env is not None:
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('packed', [True, False])
@pytest.mark.parametrize('name', ['di_asym', 'at_theta_2pi'])
def test_refused_grid_leaves_the_bound_one(name, packed):
    """lsm_set_value_grid with a 1-node dim or 2^31 cells or more returns 2 before it reads the arrays, and the handle
    keeps giving the oracle's values of the grid bound before."""
    from layered_safe_marl_b200 import SafetyFilter
    g = grid(name)
    env = None
    if packed:
        sf = SafetyFilter(_dynamics(name), value_grid=g)
    else:
        env = _env(name, False, tuning=dict(packed_grid=0))
        sf = SafetyFilter.of(env)
    _check_against_oracle(sf, g, np.random.default_rng(1), f'{name} before')
    _refuse(sf.lib, sf._h, 'lsm_set_value_grid', g, sf.device)
    _check_against_oracle(sf, g, np.random.default_rng(2), f'{name} after the refusals')
    sf.close()
    if env is not None:
        env.close()
