"""Shapes outside the product library's LSM_SPEC_LIST on the specialised pipeline: args.specialise_shape selects a
library built for exactly that shape (_build.build_shape, -DLSM_SHAPE).

CPU: the per-shape build (ABI, no rebuild when current, concurrent builders, the domain it refuses).
GPU: routing; the reference-pinned golden rollouts of every fixture the product library does not specialise; the C oracle
with zero tolerance for discrete outputs and the float64 state at the extreme and flag-heavy shapes; and the
capabilities the generic kernel lacks (fused edge list with chunked launches, compact host adjacency, graph replay, pair
values across placements), now at unlisted shapes. The GPU tests build their 14 libraries once, in parallel."""
import ctypes
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import _golden as G

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))

from layered_safe_marl_b200 import _build, _lib      # noqa: E402

gpu = pytest.mark.gpu
DI, AT = 'double_integrator', 'airtaxi'
ALLFLAGS = dict(SAFETY_VIOLATION=True, HJ_VALUE=True, POTENTIAL_CONFLICT=True, SEPARATION_DISTANCE_CURRICULUM=True,
                INITIAL_PHASE_USE_SAFETY_FILTER=True, DIFF_FROM_FILTERED_ACTION=True)
# the six golden fixtures whose shapes the product library runs on the generic kernel
GOLDEN_UNLISTED = {'at3_landmarks3', 'at6_allflags', 'di1_single_filter', 'di2_landmarks4', 'di3_obst2', 'di4_obst3_filter_global'}


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the build
# ----------------------------------------------------------------------------------------------------------------------
def _build_in(dirname, shape, extra_env=None):
    """build_shape into `dirname` in a process of its own -> CompletedProcess (stdout: the library path)."""
    code = (f"import sys; sys.path.insert(0, {REPO!r}); from layered_safe_marl_b200 import _build; "
            f"_build.SHAPES_DIR = {str(dirname)!r}; print(_build.build_shape(*{shape!r}))")
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.Popen([sys.executable, '-c', code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)


@pytest.fixture(scope='module')
def built_di1(tmp_path_factory):
    d = tmp_path_factory.mktemp('shapes')
    p = _build_in(d, (DI, 1, 2, 0))
    out, err = p.communicate()
    assert p.returncode == 0, err[-3000:]
    return d, out.strip()


def test_build_shape_exports_the_abi(built_di1):
    d, path = built_di1
    assert os.path.basename(path) == 'liblsm_b200_di1_l2_o0.so' and os.path.dirname(path) == str(d)
    lib = ctypes.CDLL(path)
    for sym in _lib.EXPORTED_SYMBOLS:
        getattr(lib, sym)
    lib.lsm_abi_version.restype = ctypes.c_int
    assert lib.lsm_abi_version() == 5


def test_second_build_does_not_rebuild(built_di1):
    d, path = built_di1
    before = os.stat(path).st_mtime_ns
    # an nvcc that cannot run: the call must not need it
    p = _build_in(d, (DI, 1, 2, 0), extra_env={'NVCC': os.path.join(str(d), 'no-such-nvcc')})
    out, err = p.communicate()
    assert p.returncode == 0, err[-3000:]
    assert out.strip() == path and os.stat(path).st_mtime_ns == before


def test_concurrent_builders_leave_one_loadable_library(tmp_path):
    procs = [_build_in(tmp_path, (AT, 5, 2, 0)) for _ in range(2)]
    outs = [p.communicate() for p in procs]
    for p, (out, err) in zip(procs, outs):
        assert p.returncode == 0, err[-3000:]
    paths = {out.strip() for out, _ in outs}
    assert len(paths) == 1
    names = sorted(f for f in os.listdir(tmp_path) if not f.endswith('.lock'))
    assert names == ['liblsm_b200_at5_l2_o0.so'], names          # no temporaries left behind
    lib = ctypes.CDLL(paths.pop())
    lib.lsm_abi_version.restype = ctypes.c_int
    assert lib.lsm_abi_version() == 5


@pytest.mark.parametrize('shape', [(DI, 33, 2, 0), (DI, 0, 2, 0), (AT, 4, 1, 0), (AT, 32, 5, 0), (DI, 8, 2, 33),
                                   (DI, 8, 2, -1), ('unicycle', 4, 2, 0)])
def test_shapes_outside_the_domain_are_refused(shape):
    with pytest.raises(ValueError):
        _build.build_shape(*shape)
    r = subprocess.run([sys.executable, '-m', 'layered_safe_marl_b200._build', '--shape', ','.join(map(str, shape))],
                       cwd=REPO, capture_output=True, text=True)
    assert r.returncode != 0 and 'ValueError' in r.stderr


def test_the_templates_refuse_an_out_of_domain_shape_at_compile_time(tmp_path):
    """The kernels' static_asserts, past the Python check: 33 agents."""
    with pytest.raises(RuntimeError, match='static assertion|static_assert'):
        _build._nvcc(['-DLSM_SHAPE=330200'], str(tmp_path / 'bad.so'))


def test_nvcc_failure_is_an_error(tmp_path, monkeypatch):
    monkeypatch.setenv('NVCC', os.path.join(str(tmp_path), 'no-such-nvcc'))
    monkeypatch.setattr(_build, 'SHAPES_DIR', str(tmp_path))
    with pytest.raises(RuntimeError, match='nvcc'):
        _build.build_shape(DI, 7, 2, 0)
    assert not [f for f in os.listdir(tmp_path) if f.endswith('.so')]


@pytest.mark.parametrize('N,E', [(32, 192), (32, 191), (16, 165)])
def test_host_adjacency_expansion_at_the_largest_entity_counts(N, E):
    """The host expansion of the compact adjacency (numpy_outputs=True) at the entity counts only shape libraries reach
    (E up to N + N * L + O = 192): byte for byte against its definition, on the vector path with disconnected entities
    (E % 4 == 0: per-observer column mask) and on the scalar row path."""
    lib = _lib.load()
    W = (E + 31) // 32
    rng = np.random.default_rng(E)
    n = 6
    base = rng.uniform(0, 4, (n, E, E)).astype(np.float32)
    base[rng.uniform(size=base.shape) < 0.3] = 0.0
    keep_bits = rng.uniform(size=(n, N, E)) < 0.8
    keep_bits[0, 0] = True
    keep = np.zeros((n, N, W), dtype=np.uint32)
    for e in range(E):
        keep[..., e >> 5] |= (keep_bits[..., e].astype(np.uint32) << np.uint32(e & 31))
    want = np.where(keep_bits[:, :, :, None] & keep_bits[:, :, None, :], base[:, None], np.float32(0.0)).astype(np.float32)
    for threads, cached in ((1, 0), (3, 1)):
        out = np.full((n, N, E, E), np.nan, dtype=np.float32)
        _lib.check(lib.lsm_expand_adjacency_host(base.ctypes.data_as(ctypes.c_void_p), keep.ctypes.data_as(ctypes.c_void_p),
                                                 out.ctypes.data_as(ctypes.c_void_p), n, N, E, threads, cached), 'expand', lib)
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), f"threads={threads} cached={cached}"


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
# every unlisted shape the GPU tests below run: (dynamics, N, L, O)
SHAPES = [(AT, 3, 3, 0), (AT, 6, 2, 0), (DI, 1, 2, 0), (DI, 2, 4, 0), (DI, 3, 2, 2), (DI, 4, 2, 3), (DI, 5, 2, 0),
          (DI, 6, 3, 0), (DI, 32, 4, 0), (DI, 32, 2, 32), (AT, 2, 5, 0), (AT, 6, 2, 9), (AT, 12, 2, 0),
          (AT, 32, 4, 32)]     # the largest environment lsm_create accepts: E = 192, 6 mask words


@pytest.fixture(scope='module')
def variants():
    """Build every shape's library once, nvcc processes in parallel."""
    with ThreadPoolExecutor(max_workers=max(1, min(len(SHAPES), os.cpu_count() or 1))) as ex:
        return dict(zip(SHAPES, ex.map(lambda s: _build.build_shape(*s), SHAPES)))


def _args(dyn, N, L=2, O=0, **kw):
    d = dict(dynamics_type=dyn, num_agents=N, num_landmarks=L, use_safety_filter=True, world_size=6 if dyn == AT else 3,
             episode_length=12, specialise_shape=True)
    if O:
        d.update(num_obstacles=O, obstacle_extension=True)
    d.update(kw)
    return G.default_args(**d)


def _product_specialises(args):
    import argparse
    from layered_safe_marl_b200 import B200GraphVecEnv
    plain = argparse.Namespace(**{k: v for k, v in vars(args).items() if k != 'specialise_shape'})
    env = B200GraphVecEnv(plain, num_envs=1, seed=0)
    spec = env.launch_info()['specialised']
    env.close()
    return spec == 1


@gpu
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: f'{s[0][:2]}{s[1]}_l{s[2]}_o{s[3]}')
def test_unlisted_shapes_run_the_specialised_pipeline(variants, shape):
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = _args(*shape)
    env = B200GraphVecEnv(args, num_envs=16, seed=0)
    li = env.launch_info()
    assert li['specialised'] == 1 and li['launches_per_step'] == 3, li
    assert env.lib is _lib.load(variants[shape]) and env.lib is not _lib.load()
    env.close()
    args.specialise_shape = False
    env = B200GraphVecEnv(args, num_envs=16, seed=0)
    assert env.launch_info()['specialised'] == 0 and env.lib is _lib.load()
    env.close()


@gpu
def test_listed_shapes_keep_the_product_library():
    from layered_safe_marl_b200 import B200GraphVecEnv
    for shape in ((DI, 8, 2, 0), (AT, 10, 2, 4)):
        env = B200GraphVecEnv(_args(*shape), num_envs=16, seed=0)
        assert env.launch_info()['specialised'] == 1 and env.lib is _lib.load()
        env.close()


@gpu
def test_envs_of_different_libraries_in_one_process(variants):
    """Two shape libraries and the product library side by side, launches interleaved: each env's outputs and state
    equal those of the same env run alone."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    cfgs = [_args(DI, 5, world_size=2), _args(AT, 6), _args(DI, 8, world_size=2)]
    n, T = 200, 8

    def snap(e):
        return [e.obs.cpu().numpy().tobytes(), e.adj.cpu().numpy().tobytes(), e.node_obs.cpu().numpy().tobytes(),
                np.ascontiguousarray(e.get_state()['agent_values']).tobytes()]

    def run(envs, streams):
        gens = [np.random.default_rng(k) for k in streams]
        for e in envs:
            e.reset(6249)
        out = [[] for _ in envs]
        for t in range(T):
            for e, g in zip(envs, gens):
                e.step(torch.as_tensor(g.integers(0, 25, (n, e.N)).astype(np.int32), device=e.device), 6249)
            torch.cuda.synchronize()
            for k, e in enumerate(envs):
                out[k].append(snap(e))
        return out

    together = [B200GraphVecEnv(a, num_envs=n, seed=3) for a in cfgs]
    assert len({id(e.lib) for e in together}) == 3 and together[2].lib is _lib.load()
    assert all(e.launch_info()['specialised'] == 1 for e in together)
    got = run(together, range(len(cfgs)))
    for e in together:
        e.close()
    for k, a in enumerate(cfgs):
        alone = B200GraphVecEnv(a, num_envs=n, seed=3)
        want = run([alone], [k])[0]
        alone.close()
        for t in range(T):
            assert got[k][t] == want[t], f"env {k} step {t}: the interleaved run differs from the same env run alone"


@gpu
def test_the_product_library_leaves_exactly_the_six_golden_shapes_unspecialised():
    unlisted = set()
    for name in G.golden_names():
        _, _, args, _, _ = G.load_case(name)
        if not _product_specialises(args):
            unlisted.add(name)
    assert unlisted == GOLDEN_UNLISTED


@gpu
@pytest.mark.parametrize('name', G.golden_names())
def test_golden_rollout_with_the_shape_library(variants, name):
    from test_cuda_parity import CudaAdapter
    from test_oracle_golden import rollout_with_tie_policy
    z, meta, args, flags, params = G.load_case(name)
    if _product_specialises(args):
        pytest.skip("the product library specialises this shape")
    args.specialise_shape = True
    probe = CudaAdapter(args, flags)
    assert probe.env.launch_info()['specialised'] == 1
    probe.env.close()
    env, ties = rollout_with_tie_policy(lambda: CudaAdapter(args, flags), z, meta, name,
                                        lambda e, a: e.step(a, episode=meta['episode']))
    assert env.env.launch_info()['specialised'] == 1
    if ties:
        print(f"{name}: roundoff ties at {ties}")
    else:
        env.reset_from_state(meta['episode'])
        G.assert_close(env.ep_info[0], z['ep_info'], f'{name} ep_info')


ORACLE_CASES = {
    # name: (shape, args, RewardBinaryConfig switches, envs, steps)
    'di1': ((DI, 1, 2, 0), dict(episode_length=5, world_size=1), dict(SAFETY_VIOLATION=True, POTENTIAL_CONFLICT=True, HJ_VALUE=True), 130, 14),
    'di5_allflags': ((DI, 5, 2, 0), dict(episode_length=10, world_size=2, collaborative=True), ALLFLAGS, 300, 25),
    'di6_l3': ((DI, 6, 3, 0), dict(episode_length=9, world_size=2), {}, 256, 20),
    'di32_l4': ((DI, 32, 4, 0), dict(episode_length=250, world_size=4), dict(SAFETY_VIOLATION=True, POTENTIAL_CONFLICT=True, HJ_VALUE=True), 12, 6),
    'di32_o32': ((DI, 32, 2, 32), dict(episode_length=250, world_size=2), dict(SAFETY_VIOLATION=True, POTENTIAL_CONFLICT=True, HJ_VALUE=True), 12, 6),
    'at2_l5': ((AT, 2, 5, 0), dict(episode_length=6, world_size=6), dict(SAFETY_VIOLATION=True, POTENTIAL_CONFLICT=True, HJ_VALUE=True), 130, 14),
    'at6_o9': ((AT, 6, 2, 9), dict(episode_length=5, world_size=1), dict(POTENTIAL_CONFLICT=True), 96, 12),
    'at32_l4_o32': ((AT, 32, 4, 32), dict(episode_length=250, world_size=6), dict(SAFETY_VIOLATION=True, POTENTIAL_CONFLICT=True, HJ_VALUE=True), 8, 5),
    'at12_pc': ((AT, 12, 2, 0), dict(episode_length=350, world_size=6), dict(POTENTIAL_CONFLICT=True), 128, 16),
    'di4_o3_global': ((DI, 4, 2, 3), dict(episode_length=8, world_size=1, graph_feat_type='global'), {}, 193, 16),
    'di5_internal2': ((DI, 5, 2, 0), dict(episode_length=10, world_size=2, num_internal_step=2), {}, 160, 16),
    'di6_l3_f32': ((DI, 6, 3, 0), dict(episode_length=9, world_size=2, interp_float32=True), {}, 256, 16),
    'at6_f32': ((AT, 6, 2, 0), dict(episode_length=12, world_size=6, interp_float32=True), dict(POTENTIAL_CONFLICT=True), 128, 16),
}


@gpu
@pytest.mark.parametrize('case', list(ORACLE_CASES))
def test_shape_library_matches_the_oracle_bit_for_bit(variants, case):
    from test_cuda_parity import _compare_with_oracle
    shape, kw, flags, n, T = ORACLE_CASES[case]
    args = _args(*shape, **kw)
    ora, cu = _compare_with_oracle(args, G.BinaryFlags(flags), n=n, T=T, episode=6249, seed=43, auto_reset=True)
    assert cu.env.launch_info()['specialised'] == 1


def _bits(a):
    import torch
    a = a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint8)


EDGE_SHAPES = {'di6_l3': ((DI, 6, 3, 0), dict(world_size=2), 600), 'di32_l4': ((DI, 32, 4, 0), dict(world_size=3), 200),
               'at6_o9': ((AT, 6, 2, 9), dict(world_size=2), 600), 'di1': ((DI, 1, 2, 0), dict(world_size=1), 2000)}   # 32 envs per warp: 2000 envs to split into 3 ranges


@gpu
@pytest.mark.parametrize('shape', list(EDGE_SHAPES))
def test_edge_list_with_chunked_launches(variants, shape):
    """Fused COO edge output == process_adj of the dense adjacency (test_edge_output._check) on three env ranges, through
    steps with auto-resets and a masked reset."""
    import torch
    from test_edge_output import _check, _masked_reset, _step_both, EPISODE
    from layered_safe_marl_b200 import B200GraphVecEnv
    sh, kw, n = EDGE_SHAPES[shape]
    args = _args(*sh, episode_length=7, **kw)
    twin = B200GraphVecEnv(args, num_envs=n, seed=5, tuning=dict(chunks=3))
    env = B200GraphVecEnv(args, num_envs=n, seed=5, tuning=dict(chunks=3))
    li = env.launch_info()
    assert li['specialised'] == 1 and li['chunks'] == 3, li
    env.enable_edge_output()
    gen = torch.Generator(); gen.manual_seed(3)
    twin.reset(EPISODE); env.reset(EPISODE)
    _check(env, twin, f"{shape} reset")
    _step_both(env, twin, gen, shape, k=9)
    mask = torch.zeros(n, dtype=torch.uint8, device=env.device); mask[::3] = 1
    _masked_reset(twin, mask); _masked_reset(env, mask)
    _check(env, twin, f"{shape} masked reset")
    _step_both(env, twin, gen, f"{shape} after the masked reset", k=3)
    assert int(env.edge_offsets[-1]) > 0


@gpu
@pytest.mark.parametrize('shape', [(DI, 5, 2, 0), (AT, 6, 2, 9), (DI, 1, 2, 0), (AT, 32, 4, 32)],
                         ids=['di5', 'at6_o9', 'di1', 'at32_l4_o32'])
def test_host_outputs_are_byte_identical(variants, shape):
    """numpy_outputs=True takes the compact-adjacency host path at an unlisted shape; every returned array equals the
    device-resident env's outputs byte for byte."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = _args(*shape, world_size=2)
    n, T, episode = (300 if shape[1] < 32 else 24), 16, 6249     # E = 192: 4.7 MB of adjacency per environment
    dev_env = B200GraphVecEnv(args, num_envs=n, seed=3)
    host_env = B200GraphVecEnv(args, num_envs=n, seed=3, numpy_outputs=True, host_chunks=5, host_threads=3)
    assert host_env._compact is not None and host_env.launch_info()['specialised'] == 1
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


@gpu
@pytest.mark.parametrize('shape', [(DI, 6, 3, 0), (AT, 12, 2, 0)], ids=['di6_l3', 'at12'])
def test_graph_replay_and_chunks_are_bit_identical(variants, shape):
    """use_graph = 1 (replayed launches) and chunks = 4 against plain single-range launches, step by step, through
    auto-resets; then emit_only rewrites the same node_obs / adj."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = _args(*shape, episode_length=9, world_size=2 if shape[0] == DI else 6)
    n, T, episode = 1024, 20, 6249
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


PAIR_SHAPES = {'di5': dict(num_agents=5, world_size=12), 'di6_l3': dict(num_agents=6, num_landmarks=3, world_size=3),
               'at6_o9': dict(dynamics_type=AT, num_agents=6, world_size=4, num_obstacles=9, obstacle_extension=True),
               'at12': dict(dynamics_type=AT, num_agents=12, world_size=6)}


@gpu
@pytest.mark.parametrize('shape', list(PAIR_SHAPES))
def test_pair_values_bit_identical_across_placements(variants, shape):
    """test_pair_values' script (steps with auto-resets at curriculum ratio 0.1, masked reset, set_state onto grid nodes,
    observe, reset_from_state) in every placement: the values the next step reads agree bit for bit."""
    from test_pair_values import VARIANTS, _run, EPISODE_LENGTH
    args = G.default_args(use_safety_filter=True, episode_length=EPISODE_LENGTH, specialise_shape=True, **PAIR_SHAPES[shape])
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
