"""N2 (SURVEY.md section 8f), fused COO edge output (lsm_set_edge_output) where random rollouts never take it: masked
resets (also the first launch after enabling, and after new buffers), count blocks over several scan rounds, a capacity
shorter than the list, graph replay / pair placement 4 / output re-binding / state edits, and distances within a few
ulps of the radius or of zero.

The reference is the reference's own process_adj (gnn.py:376-407, `_process_adj` of test_rollout_and_eval) on the dense
adjacency of a twin env that runs without edge output and gets the same calls. Every comparison is bit for bit."""
import math
import os
import sys

import numpy as np
import pytest
import torch

import _golden as G
from test_rollout_and_eval import _process_adj

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle'))

pytestmark = pytest.mark.gpu

EPISODE = 6249
SHAPES = {
    'di8': dict(num_agents=8, world_size=2),
    'air10': dict(dynamics_type='airtaxi', num_agents=10, world_size=6),
    'di8_obst4': dict(num_agents=8, world_size=2, num_obstacles=4, obstacle_extension=True),
}
SENTINEL_ADJ = -7.0


def _envs(args, n, seed=5, tuning=None):
    """(env, twin): the same seeded batch; only `env` gets the edge output."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    twin = B200GraphVecEnv(args, num_envs=n, seed=seed, tuning=dict(tuning or {}))
    env = B200GraphVecEnv(args, num_envs=n, seed=seed, tuning=dict(tuning or {}))
    return env, twin


def _enable(env, dense, capacity=None):
    env.enable_edge_output(capacity=capacity, dense_adj=dense)
    if not dense:
        env.adj.fill_(SENTINEL_ADJ)


def _masked_reset(env, mask, episode=EPISODE):
    from layered_safe_marl_b200 import _lib
    _lib.check(env.lib.lsm_reset(env._h, mask.data_ptr(), episode, env.seed, 1, env._stream()), 'lsm_reset')


def _first_bad_graph(got, want):
    bad = torch.nonzero(got != want)
    return int(bad[0, 0]) if bad.numel() else None


def _bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int64)


def _check(env, twin, tag, dense=True):
    """env's fused list against process_adj of twin's dense adjacency (and env's dense output against twin's)."""
    E, N = twin.E, twin.N
    ref = twin.adj.reshape(-1, E, E)
    ri, ra = _process_adj(ref)
    cnt = (ref.reshape(ref.shape[0], -1) != 0).sum(dim=1).to(torch.int32)
    off = torch.cumsum(cnt.long(), 0) - cnt.long()
    g = _first_bad_graph(env.edge_counts, cnt)
    assert g is None, (f"{tag}: edge_counts of graph {g} (env {g // N}, observer {g % N}) = {int(env.edge_counts[g])}, "
                       f"process_adj has {int(cnt[g])}")
    g = _first_bad_graph(env.edge_offsets[:-1], off)
    assert g is None, (f"{tag}: edge_offsets of graph {g} (env {g // N}, observer {g % N}) = {int(env.edge_offsets[g])}, "
                       f"exclusive cumsum is {int(off[g])}")
    nnz = int(env.edge_offsets[-1])
    assert nnz == ri.shape[1], f"{tag}: nnz {nnz} vs {ri.shape[1]}"
    assert nnz <= env.edge_capacity
    assert torch.equal(env.edge_index[:, :nnz], ri), f"{tag}: edge_index"
    assert torch.equal(_bits(env.edge_attr[:nnz]), _bits(ra[:, 0])), f"{tag}: edge_attr"
    ei, ea = env.edges()
    assert ei.shape == ri.shape and ea.shape == ra.shape
    if dense:
        assert torch.equal(_bits(env.adj), _bits(twin.adj)), f"{tag}: dense adjacency differs from the twin's"
    else:
        assert bool((env.adj == SENTINEL_ADJ).all()), f"{tag}: dense_adj=False must not touch the dense tensor"
    assert torch.equal(_bits(env.node_obs), _bits(twin.node_obs)), f"{tag}: node_obs"


def _step_both(env, twin, gen, tag, dense=True, k=1, actions=None):
    """k steps of both envs with the same random actions (written into `actions` when given: graph replay keys on the
    action pointer)."""
    for j in range(k):
        a = torch.randint(0, 25, (twin.n, twin.N), generator=gen, dtype=torch.int32).to(twin.device)
        if actions is not None:
            a = actions.copy_(a)
        twin.step(a, EPISODE)
        env.step(a, EPISODE)
        _check(env, twin, f"{tag} step {j}", dense)


def _masks(n, device):
    out = {}
    for name in ('every_third', 'env0', 'last', 'zeros', 'ones'):
        m = torch.zeros(n, dtype=torch.uint8, device=device)
        if name == 'every_third':
            m[::3] = 1
        elif name == 'env0':
            m[0] = 1
        elif name == 'last':
            m[-1] = 1
        elif name == 'ones':
            m[:] = 1
        out[name] = m
    return out


@pytest.mark.parametrize('when', ['right_after_enable', 'mid_rollout', 're_enabled'])
@pytest.mark.parametrize('dense', [True, False])
@pytest.mark.parametrize('chunks', [1, 3])
@pytest.mark.parametrize('shape', list(SHAPES))
def test_masked_reset_keeps_the_edge_list_exact(shape, chunks, dense, when):
    """A masked lsm_reset re-emits EVERY env into the list (the offsets of all later graphs move), so the counts of the
    envs outside the mask must describe their current record: checked as the first launch after enable_edge_output,
    in the middle of a rollout, and after a second enable (new zero-filled buffers) and after disable + enable; masks
    of every third env, env 0 only, the last env only, none and all. Then 3 more steps, which start from the counts the
    reset left behind."""
    args = G.default_args(use_safety_filter=True, episode_length=7, **SHAPES[shape])
    n = 512
    gen = torch.Generator(device='cpu'); gen.manual_seed(7)
    pair = None
    for k, (mname, mask) in enumerate(_masks(n, torch.device('cuda', 0)).items()):
        tag = f"{shape} chunks={chunks} dense={dense} {when} mask={mname}"
        if when == 'right_after_enable' or pair is None:
            env, twin = pair = _envs(args, n, tuning=dict(chunks=chunks))
            assert env.launch_info()['chunks'] == chunks
            twin.reset(EPISODE); env.reset(EPISODE)
            if when == 'mid_rollout':
                _enable(env, dense)
            elif when == 're_enabled':
                _enable(env, dense)
                _step_both(env, twin, gen, f"{tag} warm-up", dense, k=3)
        if when == 'right_after_enable':
            _enable(env, dense)
        elif when == 'mid_rollout':
            _step_both(env, twin, gen, f"{tag} before", dense, k=4)
        else:
            if k % 2:
                env.disable_edge_output()
                a = torch.randint(0, 25, (n, twin.N), generator=gen, dtype=torch.int32).to(twin.device)
                twin.step(a, EPISODE); env.step(a, EPISODE)
                assert torch.equal(_bits(env.adj), _bits(twin.adj))
            _enable(env, dense)
        _masked_reset(twin, mask)
        _masked_reset(env, mask)
        _check(env, twin, f"{tag} after the masked reset", dense)
        _step_both(env, twin, gen, f"{tag} after", dense, k=3)


@pytest.mark.parametrize('n,chunks', [(4096, 1), (4097, 1), (20000, 1), (70001, 1), (20000, 4)])
def test_count_scan_over_many_blocks(n, chunks):
    """The last count block scans the block totals in rounds of 1024 (8 per thread): n = 4096 is one round (1024 blocks of
    4 envs), 4097 adds a second round of one block, 20000 has 2000 blocks of 10 envs, 70001 hits the cap of 32 envs per
    block with a ragged last block; chunks=4 gives every range its own slice of the block arrays. 6 steps with an
    auto-reset among them: the ticket counter must be re-armed by every launch."""
    args = G.default_args(num_agents=3, use_safety_filter=False, episode_length=4, world_size=20)
    env, twin = _envs(args, n, seed=11, tuning=dict(chunks=chunks))
    assert env.launch_info()['chunks'] == chunks
    _enable(env, True)
    twin.reset(EPISODE); env.reset(EPISODE)
    _check(env, twin, f"n={n} reset")
    gen = torch.Generator(device='cpu'); gen.manual_seed(3)
    _step_both(env, twin, gen, f"n={n}", k=6)
    assert int(env.edge_offsets[-1]) > 0


def _sentinel_buffers(cap, nnz, graphs, weight_dtype=torch.float32):
    dev = torch.device('cuda', 0)
    ei = torch.full((2 * cap + nnz,), -1234567, dtype=torch.int64, device=dev)
    ea = torch.full((cap + nnz,), -7.0, dtype=weight_dtype, device=dev)
    cnt = torch.full((graphs,), -1, dtype=torch.int32, device=dev)
    off = torch.full((graphs + 1,), -1, dtype=torch.int64, device=dev)
    return ei, ea, cnt, off


def _check_truncated(tag, cap, bufs, ri, ra, cnt, off):
    ei, ea, c, o = bufs
    nnz = ri.shape[1]
    assert torch.equal(c, cnt), f"{tag}: counts"
    assert torch.equal(o[:-1], off) and int(o[-1]) == nnz, f"{tag}: offsets / nnz"
    assert torch.equal(ei[:cap], ri[0, :cap]) and torch.equal(ei[cap:2 * cap], ri[1, :cap]), f"{tag}: kept prefix"
    assert bool((ei[2 * cap:] == -1234567).all()), f"{tag}: edge_index written past capacity"
    assert torch.equal(ea[:cap], ra[:cap]), f"{tag}: kept attributes"
    assert bool((ea[cap:] == -7.0).all()), f"{tag}: edge_attr written past capacity"


@pytest.mark.parametrize('path', ['fused_chunks1', 'fused_chunks3', 'edge_list', 'world_graph'])
def test_capacity_shorter_than_the_list(path):
    """lsm_b200.h: entries past `capacity` are dropped, counts / offsets / nnz stay exact. The buffers are LARGER than
    the capacity passed and filled with a sentinel, so a write past `capacity` lands inside the allocation and shows."""
    from layered_safe_marl_b200 import _lib
    import ctypes as C
    args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=9, world_size=4)
    n = 512
    chunks = 3 if path == 'fused_chunks3' else 1
    env, twin = _envs(args, n, tuning=dict(chunks=chunks))
    assert env.launch_info()['chunks'] == chunks
    twin.reset(EPISODE); env.reset(EPISODE)
    gen = torch.Generator(device='cpu'); gen.manual_seed(9)
    for _ in range(4):
        a = torch.randint(0, 25, (n, 8), generator=gen, dtype=torch.int32).to(twin.device)
        twin.step(a, EPISODE); env.step(a, EPISODE)
    twin.observe()
    E, graphs = twin.E, n * twin.N
    p = lambda t: C.c_void_p(t.data_ptr())
    if path == 'world_graph':
        wi, ww, woff = twin.world_graph()
        wcnt = (woff[1:] - woff[:-1]).to(torch.int32)
        nnz = wi.shape[1]
        for cap in (nnz - 1, nnz // 2):
            bufs = _sentinel_buffers(cap, nnz, n, torch.float64)
            _lib.check(env.lib.lsm_world_graph(env._h, *(p(b) for b in bufs), cap, env._stream()), 'lsm_world_graph')
            _check_truncated(f"world_graph cap={cap}", cap, bufs, wi, ww, wcnt, woff[:-1])
        return
    ref = twin.adj.reshape(-1, E, E)
    ri, ra = _process_adj(ref)
    ra = ra[:, 0]
    cnt = (ref.reshape(graphs, -1) != 0).sum(dim=1).to(torch.int32)
    off = torch.cumsum(cnt.long(), 0) - cnt.long()
    nnz = ri.shape[1]
    assert nnz > 100
    for cap in (nnz - 1, nnz // 2):
        bufs = _sentinel_buffers(cap, nnz, graphs)
        if path == 'edge_list':
            _lib.check(env.lib.lsm_edge_list(env._h, p(twin.adj), *(p(b) for b in bufs), cap, env._stream()), 'lsm_edge_list')
        else:
            _lib.check(env.lib.lsm_set_edge_output(env._h, *(p(b) for b in bufs), cap, 1), 'lsm_set_edge_output')
            env.observe()
        _check_truncated(f"{path} cap={cap}", cap, bufs, ri, ra, cnt, off)
        if path != 'edge_list':
            _enable(env, True, capacity=cap)
            env.observe()
            with pytest.raises(RuntimeError, match='capacity'):
                env.edges()
        else:
            with pytest.raises(RuntimeError, match='capacity'):
                env.edge_list(twin.adj, capacity=cap)


@pytest.mark.parametrize('shape', ['di8_graph', 'air10_graph', 'di8_tail'])
def test_edge_output_through_replay_placements_and_rebinding(shape):
    """Edge output with graph replay (use_graph=1), with the pair values left behind by the agent kernel
    (pair_placement=4), across set_output_buffers re-pointing node_obs / adj, set_state(get_state()) + observe() and
    reset_from_state(): after every call the list equals process_adj of the twin."""
    kw, tuning = dict(di8_graph=(SHAPES['di8'], dict(use_graph=1)), air10_graph=(SHAPES['air10'], dict(use_graph=1)),
                      di8_tail=(SHAPES['di8'], dict(pair_placement=4)))[shape]
    args = G.default_args(use_safety_filter=True, episode_length=7, **kw)
    n = 160
    env, twin = _envs(args, n, seed=13, tuning=tuning)
    _enable(env, True)
    twin.reset(EPISODE); env.reset(EPISODE)
    _check(env, twin, 'reset')
    gen = torch.Generator(device='cpu'); gen.manual_seed(4)
    actions = torch.zeros((n, twin.N), dtype=torch.int32, device=twin.device)
    for t in range(14):
        if t == 4:
            env.set_output_buffers(node_obs=torch.full_like(env.node_obs, 3.0), adj=torch.full_like(env.adj, 3.0))
        if t == 7:
            for e in (twin, env):
                e.set_state(e.get_state()); e.observe()
            _check(env, twin, f't={t} set_state + observe')
        if t == 10:
            twin.reset_from_state(EPISODE); env.reset_from_state(EPISODE)
            _check(env, twin, f't={t} reset_from_state')
        _step_both(env, twin, gen, f't={t}', actions=actions)
    li = env.launch_info()
    if 'graph' in shape:
        assert li['graph_replays'] >= 3, li
    else:
        assert li['pair_placement'] == 4 and li['launches_per_step'] == 2, li


def _lt(T):
    """lsm_capi.cu: min{t : sqrt_rn(t) >= T}."""
    t = T * T
    while t > 0.0 and math.sqrt(t) >= T:
        t = math.nextafter(t, 0.0)
    while math.sqrt(t) < T:
        t = math.nextafter(t, math.inf)
    return t


def _with_sum(dx, target):
    """dy such that RN(RN(dx*dx) + RN(dy*dy)) == target exactly (the kernels' float64 d2)."""
    dx2 = dx * dx
    dy0 = math.sqrt(target - dx2)
    for direction in (math.inf, 0.0):
        dy = dy0
        for _ in range(400):
            if dx2 + dy * dy == target:
                return dy
            dy = math.nextafter(dy, direction)
    raise AssertionError(f"no dy for d2 = {target!r}")


@pytest.mark.parametrize('dyn', ['double_integrator', 'airtaxi'])
def test_radius_ties_in_count_and_emit_kernels(dyn):
    """The count kernel and the emit kernel decide the radius twice; both must match the reference's strict
    `dist < max_edge_dist` and its float32 adjacency (no edge where float32(dist) is 0). States built on the host: an
    agent at the origin and its first goal landmark at a distance whose float64 square takes every double in
    [r2_lt - 4 ulp, r2_lt + 4 ulp], then coincident and near-coincident pairs (d2 = 0, d2 subnormal, d around 2^-150).
    Checked: the dense pattern and values, the count kernel's counts, the fused list, the oracle's pattern, and the
    world graph (inclusive radius, float64 weights, an edge for every d2 > 0)."""
    import oracle_env as O
    from layered_safe_marl_b200 import B200GraphVecEnv, config as cfg
    N = 4                                  # a specialised shape of both dynamics
    R = float((cfg.DoubleIntegratorConfig if dyn == 'double_integrator' else cfg.AirTaxiConfig).COORDINATION_RANGE)
    r2 = _lt(R)
    targets = [r2]
    for _ in range(4):
        targets = [math.nextafter(targets[0], 0.0)] + targets + [math.nextafter(targets[-1], math.inf)]
    dx = math.nextafter(R - 1e-4, 0.0)
    goal = [(dx, _with_sum(dx, t)) for t in targets]
    tiny = [0.0, 1e-160, 1e-150, 2.0 ** -150, math.nextafter(2.0 ** -150, 1.0), 2.0 ** -149, 1e-40, 1e-20, 1e-14]
    goal += [(d, 0.0) for d in tiny]
    n = len(goal)
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=False, episode_length=50, world_size=4)
    params = cfg.scenario_params_from_args(args)
    env = B200GraphVecEnv(args, num_envs=n, seed=3)
    E, M = env.E, env.M
    env.reset(EPISODE)
    s = env.get_state()
    # every other entity far from everything else (>= 20 apart)
    far = np.array([[40.0 + 20.0 * k, -40.0] for k in range(E)])
    av = np.array(s['agent_values'])
    av[:, :, :2] = far[None, :N]
    av[:, :, 2:] = 0.0
    av[:, 0, :2] = 0.0
    lp = np.broadcast_to(far[None, N:N + M], (n, M, 2)).copy()
    lp[:, 0] = np.array(goal)
    s['agent_values'], s['landmark_pos'] = av, lp
    s['done'] = np.zeros_like(s['done']); s['reached_goal'] = np.zeros_like(s['reached_goal'])
    env.set_state(s)
    _enable(env, True)
    env.observe()
    # the plain reference: the kernels' float64 d2 (exact differences), correctly rounded sqrt
    pos = np.concatenate([av[:, :, :2], lp], axis=1)
    d = pos[:, :, None, :] - pos[:, None, :, :]
    d2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]
    assert [float(v) for v in d2[:len(targets), 0, N]] == targets
    dist = np.sqrt(d2)
    want = np.where(dist < R, dist, 0.0).astype(np.float32)          # float32(0 < d < R), 0 where it rounds to 0
    on = want != 0
    assert on[:len(targets), 0, N].tolist() == [t < r2 for t in targets]
    got = env.adj.cpu().numpy()
    for i in range(N):
        G.assert_same_mask(got[:, i] != 0, on, f"{dyn}: dense pattern, observer {i}")
    big = on & (d2 >= 1e-30)      # the kernel's value is sqrt(max(d2, 1e-30)) through rsqrt: 4e-7 relative
    G.assert_close(got[:, 0][big], want[big], f"{dyn}: dense values", rtol=4e-7, atol=0.0)
    ref = torch.from_numpy(np.repeat(want[:, None], N, axis=1).reshape(-1, E, E)).to(env.device)
    cnt = (ref.reshape(n * N, -1) != 0).sum(dim=1).to(torch.int32)
    assert torch.equal(env.edge_counts, cnt), f"{dyn}: count kernel"
    ri, _ = _process_adj(ref)
    ei, ea = env.edges()
    assert torch.equal(ei, ri), f"{dyn}: fused edge_index"
    _, ra = _process_adj(env.adj.reshape(-1, E, E))
    assert torch.equal(_bits(ea), _bits(ra)), f"{dyn}: fused edge_attr"
    vg, tg = G.value_grid_for(params)
    ora = O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=3, nthreads=4)
    ora.set_state(s)
    ora.observe()
    for i in range(N):
        G.assert_same_mask(ora.adj[:, i] != 0, on, f"{dyn}: oracle pattern, observer {i}")
    # world graph: 0 < d <= R (float64 weights, so every positive d2 is an edge)
    wi, ww, woff = env.world_graph()
    wi, ww, woff = wi.cpu().numpy(), ww.cpu().numpy(), woff.cpu().numpy()
    won = (dist <= R) & (d2 > 0.0)
    for e in range(n):
        rows, cols = np.nonzero(won[e])
        sl = slice(woff[e], woff[e + 1])
        assert np.array_equal(wi[0, sl], rows) and np.array_equal(wi[1, sl], cols), f"{dyn}: world graph env {e}"
        assert np.array_equal(ww[sl], dist[e][rows, cols]), f"{dyn}: world graph weights env {e}"


def test_cfg2_full_size_edges():
    """The benchmark's cfg2 shape (4096 envs x 8 agents, one range, 1024 count blocks) with the dense adjacency on: 3
    steps, the fused list against process_adj of the same env's dense output."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(num_agents=8, use_safety_filter=True, world_size=4, episode_length=250)
    n = 4096
    env = B200GraphVecEnv(args, num_envs=n, seed=1234)
    assert env.launch_info()['chunks'] == 1
    _enable(env, True)
    env.reset(EPISODE)
    gen = torch.Generator(device='cpu'); gen.manual_seed(1)
    for t in range(3):
        a = torch.randint(0, 25, (n, 8), generator=gen, dtype=torch.int32).to(env.device)
        env.step(a, EPISODE)
        _check(env, env, f"cfg2 t={t}")
