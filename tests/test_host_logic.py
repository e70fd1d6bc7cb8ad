"""CPU: host-side logic - config mirror, layout agreement with the oracle header, C-ABI exports,
lazy infos against the golden info dicts, synthetic grids, sharding over gloo (world_size 2)."""
import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest

import _golden as G

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))

from layered_safe_marl_b200 import config as cfg  # noqa: E402
from layered_safe_marl_b200 import hj_grid, infos, layout as LY, sharding  # noqa: E402


def test_config_mirrors_reference_constants():
    # multiagent/config.py:3-83
    assert cfg.AirTaxiConfig.V_MIN == 60 * 0.514444 * 0.001
    assert cfg.AirTaxiConfig.COORDINATION_RANGE == 3 * 1.60934
    assert cfg.DoubleIntegratorConfig.COORDINATION_RANGE == 4
    assert cfg.RewardWeightConfig.GOAL_REACH == 50 and cfg.RewardWeightConfig.MIN_REWARD == -40
    p = cfg.scenario_params_from_args(G.default_args(num_agents=8, use_safety_filter=True, episode_length=250))
    assert p.num_entities == 24 and p.obs_dim == 7 and p.node_feat_dim == 10
    assert p.num_total_episode == 5_000_000 // 250 // 32
    assert p.flags & cfg.FLAG_USE_SAFETY_FILTER and p.flags & cfg.FLAG_USE_MASKING


def test_invalid_configs_fail_like_the_reference():
    with pytest.raises(ValueError, match="obstacle 0 not supported"):
        cfg.scenario_params_from_args(G.default_args(num_obstacles=2))
    # the declared extension is opt-in and changes the entity count only
    p = cfg.scenario_params_from_args(G.default_args(num_obstacles=2, obstacle_extension=True))
    assert p.num_obstacles == 2 and p.num_entities == 3 * 3 + 2
    with pytest.raises(ValueError, match="num_obstacles"):
        cfg.scenario_params_from_args(G.default_args(num_obstacles=33, obstacle_extension=True))
    with pytest.raises(AssertionError):
        cfg.scenario_params_from_args(G.default_args(num_landmarks=1))
    with pytest.raises(NotImplementedError):
        cfg.scenario_params_from_args(G.default_args(use_masking=False))


def _enum_values(header, prefix):
    txt = open(header).read()
    out = {}
    for block in re.findall(r'enum\s*\{([^}]*)\}', txt, flags=re.S):
        block = re.sub(r'/\*.*?\*/', '', block, flags=re.S)
        val = -1
        for item in block.split(','):
            item = item.strip()
            if not item:
                continue
            if '=' in item:
                name, v = [x.strip() for x in item.split('=')]
                try:
                    val = int(eval(v, {}, {}))
                except Exception:
                    continue
            else:
                name = item
                val += 1
            if name.startswith(prefix):
                out[name[len(prefix):]] = val
    return out


def test_layout_matches_public_and_oracle_headers():
    pub = os.path.join(REPO, 'include', 'lsm_b200.h')
    ora = os.path.join(REPO, 'oracle', 'lsm_oracle.h')
    for pre_pub, pre_ora in (('LSM_AF_', 'LSMO_AF_'), ('LSM_AI_', 'LSMO_AI_'), ('LSM_LF_', 'LSMO_LF_'),
                             ('LSM_EI_', 'LSMO_EI_'), ('LSM_EP_', 'LSMO_EP_'), ('LSM_FLAG_', 'LSMO_FLAG_')):
        a, b = _enum_values(pub, pre_pub), _enum_values(ora, pre_ora)
        assert a and a == b, (pre_pub, a, b)
    af = _enum_values(pub, 'LSM_AF_')
    for k, v in af.items():
        if k != 'COUNT':
            assert getattr(LY, 'AF_' + k) == v
    assert af['COUNT'] == LY.AF_COUNT
    ai = _enum_values(pub, 'LSM_AI_')
    for k, v in ai.items():
        if k != 'COUNT':
            assert getattr(LY, 'AI_' + k) == v
    for pre in ('TF_', 'TI_'):
        for k, v in _enum_values(pub, 'LSM_' + pre).items():
            assert getattr(LY, pre + k) == v
    import oracle_env as O
    assert O.AF_COUNT == LY.AF_COUNT and O.AI_COUNT == LY.AI_COUNT and O.AF['DIST_LEFT'] == LY.AF_DIST_LEFT


def test_c_abi_library_exports_every_declared_symbol():
    """Loads liblsm_b200.so without calling any compute entry point (no GPU here)."""
    from layered_safe_marl_b200 import _build, _lib
    path = _build.build()
    lib = ctypes.CDLL(path)
    declared = set(re.findall(r'\b(lsm_[a-z_]+)\s*\(', open(os.path.join(REPO, 'include', 'lsm_b200.h')).read()))
    declared = {d for d in declared if not d.startswith('lsm_b200')}
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    for sym in declared:
        assert getattr(lib, sym) is not None
    lib.lsm_abi_version.restype = ctypes.c_int
    assert lib.lsm_abi_version() == 5
    # struct sizes must agree with the header (checked via the oracle's identical layout of lsm_config)
    import oracle_env as O
    assert ctypes.sizeof(_lib.LsmConfig) == ctypes.sizeof(O.Params)
    assert ctypes.sizeof(_lib.LsmGridDesc) == ctypes.sizeof(O.Grid)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(REPO, 'layered_safe_marl_b200')
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                txt = open(os.path.join(root, f)).read()
                assert 'oracle_env' not in txt and 'lsm_oracle' not in txt and 'liblsm_oracle' not in txt, f


def test_grad_values_matches_declared_semantics():
    g = hj_grid.synthetic_di_grid(shape=(9, 9, 5, 5))
    sys.path.insert(0, os.path.join(REPO, 'oracle', 'ref_stubs'))
    import hj_reachability as hj
    grid = hj.Grid(g.lo, g.hi, g.shape, ())
    want = grid.grad_values(g.values)
    np.testing.assert_array_equal(g.grads, want)
    a = hj_grid.synthetic_airtaxi_grid(shape=(7, 7, 8, 3, 3))
    grid = hj.Grid(a.lo, a.hi, a.shape, (2,))
    np.testing.assert_array_equal(a.grads, grid.grad_values(a.values))


def _fma(a, b, c):
    """fma(a, b, c) in float64: exact product and sum, one rounding (float(Fraction) is correctly rounded)."""
    from fractions import Fraction
    return float(Fraction(a) * Fraction(b) + Fraction(c))


@pytest.mark.parametrize('which', ['di', 'airtaxi', 'ttr'])
def test_div_exact_equals_division_on_the_synthetic_grids(which):
    """lsm_grid.cuh div_exact: the HJ stencil divides by the grid spacing b through y = RN(1/b) as
    q0 = a*y; r = fma(-b, q0, a); q = fma(r, y, q0). Markstein's proof that q = RN(a/b) assumes y is within one ulp of
    1/b in a sense RN(1/b) does not always meet, so check every dimension of the three synthetic grids: dividends
    a = x - lo for the grid nodes +-8 ulps, the box faces and random positions within two box widths outside."""
    g = dict(di=hj_grid.synthetic_di_grid, airtaxi=hj_grid.synthetic_airtaxi_grid, ttr=hj_grid.synthetic_ttr_grid)[which]()
    check_div_exact(g.lo, g.hi, g.shape, g.periodic, which, np.random.default_rng(11))


def check_div_exact(lo_, hi_, shape, periodic, what, rng):
    """div_exact(x - lo, spacing) == (x - lo) / spacing on every dimension of a grid geometry (see the test above)."""
    for d in range(len(shape)):
        lo, hi, n = float(lo_[d]), float(hi_[d]), int(shape[d])
        b = (hi - lo) / n if periodic[d] else (hi - lo) / (n - 1.0)      # lsm_capi.cu fill_grid
        y = 1.0 / b
        xs = [lo, hi]
        for k in range(n):
            x = lo + b * k
            xs.append(x)
            up = dn = x
            for _ in range(8):
                up, dn = math.nextafter(up, math.inf), math.nextafter(dn, -math.inf)
                xs += [up, dn]
        w = hi - lo
        xs += [float(v) for v in rng.uniform(lo - 2.0 * w, hi + 2.0 * w, 2000)]
        for x in xs:
            a = x - lo
            q0 = a * y
            r = _fma(-b, q0, a)
            q = _fma(r, y, q0)
            assert q == a / b, f"{what} dim {d}: x={x!r} a={a!r} b={b!r}: div_exact {q!r} vs {a / b!r}"


def test_oracle_interpolation_matches_stub():
    import oracle_env as O
    sys.path.insert(0, os.path.join(REPO, 'oracle', 'ref_stubs'))
    import hj_reachability as hj
    a = hj_grid.synthetic_airtaxi_grid(shape=(7, 7, 8, 3, 3))
    grid = hj.Grid(a.lo, a.hi, a.shape, (2,))
    s, keep = O.make_grid(a)
    rng = np.random.default_rng(0)
    # the float64 arithmetic: an earlier oracle step / reset / observe in the float32 mode leaves the oracle's switch set
    O.lib().lsmo_set_interp_float32(0)
    for _ in range(200):
        x = rng.uniform(a.lo - 1.0, a.hi + 1.0)
        x[2] = rng.uniform(-10, 10)
        xc = (ctypes.c_double * 5)(*x)
        got = O.lib().lsm_interpolate if False else O.lib().lsmo_interpolate(ctypes.byref(s), xc, ctypes.c_int(-1))
        want = float(grid.interpolate(a.values, x))
        assert got == want
        for d in range(5):
            gd = O.lib().lsmo_interpolate(ctypes.byref(s), xc, ctypes.c_int(d))
            assert gd == float(grid.interpolate(a.grads, x)[d])


def test_oracle_float32_interpolation_matches_stub_bit_for_bit():
    """The second declared arithmetic of Grid.interpolate (LSM_FLAG_INTERP_FLOAT32: position, weights, products and the
    corner sum in float32, as jax computes without x64): C oracle == numpy stub exactly, and it is NOT the float64 mode."""
    import oracle_env as O
    sys.path.insert(0, os.path.join(REPO, 'oracle', 'ref_stubs'))
    import hj_reachability as hj
    a = hj_grid.synthetic_airtaxi_grid(shape=(7, 7, 8, 3, 3))
    grid = hj.Grid(a.lo, a.hi, a.shape, (2,))
    s, keep = O.make_grid(a)
    rng = np.random.default_rng(1)
    differ = 0
    O.lib().lsmo_set_interp_float32(1)
    hj.FLOAT32_INTERPOLATION = True
    try:
        for _ in range(200):
            x = rng.uniform(a.lo - 1.0, a.hi + 1.0)
            x[2] = rng.uniform(-10, 10)
            xc = (ctypes.c_double * 5)(*x)
            got = O.lib().lsmo_interpolate(ctypes.byref(s), xc, ctypes.c_int(-1))
            want = grid.interpolate(a.values, x)
            assert isinstance(want, np.float32) and got == float(want)
            for d in range(5):
                assert O.lib().lsmo_interpolate(ctypes.byref(s), xc, ctypes.c_int(d)) == float(grid.interpolate(a.grads, x)[d])
            hj.FLOAT32_INTERPOLATION = False
            differ += float(grid.interpolate(a.values, x)) != got
            hj.FLOAT32_INTERPOLATION = True
    finally:
        O.lib().lsmo_set_interp_float32(0)
        hj.FLOAT32_INTERPOLATION = False
    assert differ > 150          # the float64 mode gives a different number almost everywhere


@pytest.mark.parametrize('name', ['di3_nofilter_goals', 'di8_filter_allflags', 'at10_filter_pc', 'di4_collab_conflict'])
def test_lazy_infos_reproduce_reference_info_dicts(name):
    """infos.compute_agent_infos from (previous, current) golden state == the reference's info dicts."""
    z, meta, args, flags, params = G.load_case(name)
    N = params.num_agents
    for t in range(1, meta['T']):
        af = np.zeros((LY.AF_COUNT, 1, N)); ai = np.zeros((LY.AI_COUNT, 1, N), dtype=np.int32)
        ei = np.zeros((LY.EI_COUNT, 1), dtype=np.int32)
        ei[LY.EI_PARITY] = 1                                     # slot B = newest, slot A = previous step
        cur = G.state_at(z, t, batch=False); prev = G.state_at(z, t - 1, batch=False)
        af[LY.AF_X, 0] = cur['agent_values'][:, 0]; af[LY.AF_Y, 0] = cur['agent_values'][:, 1]
        af[LY.AF_MIN_REL_DIST, 0] = cur['min_relative_distance']; af[LY.AF_GOAL_MIN_TIME, 0] = cur['goal_min_time']
        af[LY.AF_TIMES_REQ_B, 0] = cur['times_required']; af[LY.AF_TIMES_REQ_A, 0] = prev['times_required']
        af[LY.AF_DISTS_GOAL_B, 0] = cur['dists_to_goal']; af[LY.AF_DISTS_GOAL_A, 0] = prev['dists_to_goal']
        af[LY.AF_DIST_LEFT, 0] = cur['dist_left_to_goal']
        ai[LY.AI_NUM_COLLISIONS, 0] = cur['num_agent_collisions']; ai[LY.AI_SAFETY_FILTERED, 0] = cur['safety_filtered']
        sep = infos.separation_distance_of(params, np.array([float(cur['curriculum_ratio'])]))
        out = infos.compute_agent_infos(af, ai, ei, z['info_individual_reward'][t][None], sep)
        for k in ('individual_reward', 'min_relative_distance', 'Dist_to_goal', 'Time_req_to_goal', 'Num_agent_collisions',
                  'Num_obst_collisions', 'Distance_mean', 'Distance_variance', 'Mean_by_variance', 'Dists_traveled',
                  'Time_taken', 'Time_mean', 'Time_stddev', 'Time_mean_by_stddev', 'Min_time_to_goal', 'position'):
            G.assert_close(out[k][0], z['info_' + k][t], f'{name} t={t} info[{k}]', rtol=1e-9, atol=1e-12)
        for k in ('Departed', 'Safety filtered', 'Safety violated'):
            G.assert_same_mask(out[k][0].astype(bool), z['info_' + k][t].astype(bool), f'{name} t={t} info[{k}]')


def test_shard_range_is_a_partition():
    for total, world in ((4096, 8), (65536, 8), (10, 4), (7, 8)):
        covered = []
        for r in range(world):
            first, n = sharding.shard_range(total, world, r)
            covered += list(range(first, first + n))
        assert covered == list(range(total))


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    first, n = sharding.shard_range(10, world, rank)
    ep = torch.arange(first, first + n, dtype=torch.float64).view(n, 1).repeat(1, LY.EP_COUNT)
    stats = sharding.allreduce_episode_stats(ep)
    q.put((rank, first, n, stats['travel_time_mean']))
    dist.destroy_process_group()


def test_episode_stats_allreduce_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [r[1:3] for r in res] == [(0, 5), (5, 5)]
    for r in res:
        assert abs(r[3] - 4.5) < 1e-12    # mean of 0..9 over both shards


class _FakeMeta:          # stand-ins for hj_reachability_utils' pickled containers (field names: safety_filter.py:158-166,
    pass                  # navigation_graph_safe.py:132-138)


class _FakeData:
    pass


def test_reference_pickle_loaders(tmp_path):
    """Value-function pickles go through HjDataHandle's negate + shift + gradients; the TTR pickle is used raw with
    ttr_max from the file (navigation_graph_safe.py:128-138, 751-755)."""
    import pickle
    from layered_safe_marl_b200 import hj_grid as H
    rng = np.random.default_rng(0)
    meta = _FakeMeta(); meta.domain_lo = [-1.0, -2.0, -np.pi, 0.03]; meta.domain_hi = [1.0, 2.0, np.pi, 0.09]
    meta.shape = (5, 6, 8, 3); meta.periodic_dims = (2,)
    ttr = _FakeData(); ttr.grid_meta_data = meta; ttr.values = rng.uniform(0, 50, meta.shape); ttr.ttr_max = 123.5
    p = tmp_path / 'ttr.pkl'
    with open(p, 'wb') as f:
        pickle.dump(ttr, f)
    g = H.load_reference_ttr_pickle(str(p))
    assert g.ttr_max == 123.5 and g.grads is None and g.periodic == (False, False, True, False)
    assert g.values.dtype == np.float32 and np.array_equal(g.values, ttr.values.astype(np.float32))   # raw: no sign flip, no shift
    assert np.array_equal(g.lo, np.asarray(meta.domain_lo)) and g.shape == meta.shape
    val = _FakeData(); val.grid_meta_data = meta; val.values = rng.normal(size=meta.shape); val.info = {'separation_distance': 0.5}
    p2 = tmp_path / 'val.pkl'
    with open(p2, 'wb') as f:
        pickle.dump(val, f)
    h = H.load_reference_pickle(str(p2), 0.8)
    want = (-val.values.astype(np.float32) - np.float32(0.8 - 0.5)).astype(np.float32)
    assert np.array_equal(h.values, want) and h.separation_distance == 0.8 and h.grads.shape == meta.shape + (4,)


@pytest.mark.parametrize('N,L', [(8, 2), (3, 2), (10, 2), (32, 2)])
def test_expand_adjacency_host_matches_numpy(N, L):
    """lsm_expand_adjacency_host (a HOST function of the product library: the e2e path ships one thresholded E x E matrix
    per env + per-observer keep masks over PCIe and rebuilds the reference's (n, N, E, E) array on the host) against
    the definition adj[e, i, a, b] = keep_i[a] & keep_i[b] ? base[e, a, b] : 0, byte for byte, for row widths that take
    the vector path (E % 4 == 0) and the scalar one."""
    from layered_safe_marl_b200 import _lib
    lib = _lib.load()
    E = N * (1 + L); W = (E + 31) // 32
    rng = np.random.default_rng(N)
    n = 37
    base = rng.uniform(0, 4, (n, E, E)).astype(np.float32)
    base[rng.uniform(size=base.shape) < 0.3] = 0.0
    keep_bits = rng.uniform(size=(n, N, E)) < 0.8
    keep_bits[0] = True
    keep = np.zeros((n, N, W), dtype=np.uint32)
    for e in range(E):
        keep[..., e >> 5] |= (keep_bits[..., e].astype(np.uint32) << np.uint32(e & 31))
    want = np.where(keep_bits[:, :, :, None] & keep_bits[:, :, None, :], base[:, None], np.float32(0.0)).astype(np.float32)
    for threads, cached in ((1, 0), (3, 0), (0, 0), (4, 1)):
        out = np.full((n, N, E, E), np.nan, dtype=np.float32)
        _lib.check(lib.lsm_expand_adjacency_host(base.ctypes.data_as(ctypes.c_void_p), keep.ctypes.data_as(ctypes.c_void_p),
                                                 out.ctypes.data_as(ctypes.c_void_p), n, N, E, threads, cached), 'expand')
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), f"threads={threads} cached={cached}"


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors of include/lsm_b200.h (layered_safe_marl_b200/_lib.py) and of oracle/lsm_oracle.h (oracle/oracle_env.py)
    have the C compiler's sizes and field offsets - a struct edited on one side only would otherwise corrupt memory silently."""
    import subprocess
    import oracle_env as O
    from layered_safe_marl_b200 import _lib
    checks = [('lsm_b200.h', os.path.join(REPO, 'include'), [('lsm_config', _lib.LsmConfig), ('lsm_grid_desc', _lib.LsmGridDesc),
                                                            ('lsm_buffers', _lib.LsmBuffers), ('lsm_tuning', _lib.LsmTuning),
                                                            ('lsm_launch_info', _lib.LsmLaunchInfo), ('lsm_host_io', _lib.LsmHostIo)]),
              ('lsm_oracle.h', os.path.join(REPO, 'oracle'), [('lsmo_params', O.Params), ('lsmo_grid', O.Grid), ('lsmo_buffers', O.Buffers)])]
    for header, inc, structs in checks:
        lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{header}"', 'int main(void) {']
        for cname, cls in structs:
            lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
            for fname, _ in cls._fields_:
                cfield = 'reserved' if fname == '_reserved' else fname
                lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {cfield}));')
        lines += ['  return 0;', '}']
        src = tmp_path / (header + '.c'); exe = tmp_path / (header + '.exe')
        src.write_text('\n'.join(lines))
        subprocess.check_call(['gcc', '-I', inc, '-o', str(exe), str(src)])
        got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
        for cname, cls in structs:
            assert int(got[cname]) == ctypes.sizeof(cls), f"sizeof({cname}): C {got[cname]} vs ctypes {ctypes.sizeof(cls)}"
            for fname, _ in cls._fields_:
                assert int(got[f'{cname}.{fname}']) == getattr(cls, fname).offset, f"offsetof({cname}, {fname})"


def test_edited_dynamics_limits_are_refused(monkeypatch):
    """The acceleration / speed / turn-rate limits are compile-time constants of the kernels; a config class edited
    without a rebuild must fail loudly instead of simulating something else than it says."""
    args = G.default_args(num_agents=3)
    cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags({}))
    monkeypatch.setattr(cfg.DoubleIntegratorConfig, 'ACCELX_MAX', 0.75)
    with pytest.raises(ValueError, match='compiled into the kernels'):
        cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags({}))
