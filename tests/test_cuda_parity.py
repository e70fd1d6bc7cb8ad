"""GPU: the CUDA environment (through the C ABI) against (1) the golden rollouts of the unmodified
reference and (2) the C oracle on batches of seeded environments.

Bar: adjacency pattern, done flags, goal counters, filter masks, deconflicting indices, collision and
episode counters bit-exact in EVERY environment (no tolerated fraction); against the oracle the float64 state is
bit-identical too (shared float64 sin / cos / atan2, include/lsm_math.h); float32 observations and the golden
rollouts of the reference within 1e-5 relative (tests/_golden.RTOL)."""
import os
import sys

import numpy as np
import pytest

import _golden as G

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle'))

pytestmark = pytest.mark.gpu

CASES = G.golden_names()


class CudaAdapter:
    """Gives the CUDA env the attribute surface the shared check_step helper expects."""

    def __init__(self, args, flags, n=1, seed=0, auto_reset=False, value_grid=None, ttr_grid=None):
        import torch
        from layered_safe_marl_b200 import B200GraphVecEnv
        self.torch = torch
        self.env = B200GraphVecEnv(args, num_envs=n, seed=seed, binary_cfg=flags, auto_reset=auto_reset,
                                   value_grid=value_grid, ttr_grid=ttr_grid)

    def set_state(self, s):
        self.env.set_state(s)

    def get_state(self):
        return self.env.get_state()

    def step(self, actions, episode=0):
        self.env.step(self.torch.as_tensor(np.asarray(actions), dtype=self.torch.int32, device=self.env.device), episode)
        self.torch.cuda.synchronize()

    def observe(self):
        self.env.observe()
        self.torch.cuda.synchronize()

    def reset_from_state(self, episode):
        self.env.reset_from_state(episode)
        self.torch.cuda.synchronize()

    @property
    def obs(self): return self.env.obs.cpu().numpy()
    @property
    def node_obs(self): return self.env.node_obs.cpu().numpy()
    @property
    def adj(self): return self.env.adj.cpu().numpy()
    @property
    def reward(self): return self.env.reward.cpu().numpy()
    @property
    def done(self): return self.env.done.cpu().numpy()
    @property
    def ep_info(self): return self.env.ep_info.cpu().numpy()


@pytest.mark.parametrize('name', CASES)
def test_golden_reset_observation(name):
    z, meta, args, flags, params = G.load_case(name)
    env = CudaAdapter(args, flags)
    env.set_state(G.state0(z))
    env.observe()
    G.assert_close(env.obs[0], z['obs0'], 'obs0')
    G.assert_close(env.node_obs[0], z['node_obs0'], 'node_obs0')
    G.assert_same_mask(env.adj[0] != 0, z['adj0'] != 0, 'adj0 pattern')
    G.assert_close(env.adj[0], z['adj0'], 'adj0')


@pytest.mark.parametrize('name', CASES)
def test_golden_rollout(name):
    from test_oracle_golden import rollout_with_tie_policy
    z, meta, args, flags, params = G.load_case(name)
    env, ties = rollout_with_tie_policy(lambda: CudaAdapter(args, flags), z, meta, name,
                                        lambda e, a: e.step(a, episode=meta['episode']))
    if ties:
        print(f"{name}: roundoff ties at {ties}")
    else:
        env.reset_from_state(meta['episode'])
        G.assert_close(env.ep_info[0], z['ep_info'], f'{name} ep_info')


DISCRETE_KEYS = ('reached_goal', 'done', 'safety_filtered', 'deconflicting_agent_index', 'num_agent_collisions',
                 'ep_travel_length', 'ep_conflict', 'ep_multi_engagement', 'ep_done', 'current_step')
# float64 state: the CUDA kernels and the oracle execute the same IEEE operations (no FMA contraction, shared
# sin / cos / atan2 of include/lsm_math.h), so these are compared BIT FOR BIT
EXACT_STATE_KEYS = ('agent_values', 'p_dist', 'min_relative_distance', 'times_required', 'dists_to_goal',
                    'dist_left_to_goal', 'ep_travel_distance', 'ep_min_distance', 'action_diff',
                    'landmark_pos', 'landmark_heading', 'landmark_speed', 'curriculum_ratio')


def _report_divergence(tag, so, sc, ora, cu, prev_state_equal, n):
    """Print, per divergent env, the first differing quantity and whether the two sides entered the step from
    bit-identical states (if they did, the divergence was created inside this step)."""
    lines = []
    bad = np.zeros(n, dtype=bool)
    for k in DISCRETE_KEYS:
        a, b = np.asarray(so[k]).reshape(n, -1), np.asarray(sc[k]).reshape(n, -1)
        for e in np.nonzero((a != b).any(axis=1))[0]:
            if not bad[e]:
                j = int(np.nonzero(a[e] != b[e])[0][0])
                lines.append(f"  env {e}: {k}[{j}] oracle={a[e, j]} cuda={b[e, j]}; states equal before the step: {bool(prev_state_equal[e])}")
            bad[e] = True
    pa, pb = (ora.adj != 0).reshape(n, -1), (cu.adj != 0).reshape(n, -1)
    for e in np.nonzero((pa != pb).any(axis=1))[0]:
        if not bad[e]:
            j = int(np.nonzero(pa[e] != pb[e])[0][0])
            lines.append(f"  env {e}: adjacency pattern entry {j} oracle={ora.adj.reshape(n, -1)[e, j]!r} cuda={cu.adj.reshape(n, -1)[e, j]!r}; "
                         f"states equal before the step: {bool(prev_state_equal[e])}")
        bad[e] = True
    d = (ora.done != cu.done).reshape(n, -1).any(axis=1)
    for e in np.nonzero(d & ~bad)[0]:
        lines.append(f"  env {e}: done flags oracle={ora.done[e]} cuda={cu.done[e]}")
    bad |= d
    if lines:
        print(f"{tag}: {int(bad.sum())} of {n} envs diverge in a discrete output")
        print("\n".join(lines[:12]))
    return bad


def _compare_with_oracle(args, flags, n, T, episode, seed, auto_reset, grids=None, prepare=None):
    """Same Philox-seeded resets and the same actions through the CUDA env and the C oracle. ZERO tolerance for
    discrete outputs and for the float64 state; float32 observations within tests/_golden.RTOL (the emission uses
    rsqrt / angle-difference identities, <= 4e-7 relative). `grids`: the (value, TTR) grids both sides bind (default:
    the synthetic grids); `prepare(env)` runs on the CUDA env before the first reset."""
    import torch
    import oracle_env as O
    from layered_safe_marl_b200 import config as cfg
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = G.value_grid_for(params) if grids is None else grids
    ora = O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=seed, nthreads=8)
    cu = CudaAdapter(args, flags, n=n, seed=seed, auto_reset=auto_reset, value_grid=vg, ttr_grid=tg)
    if prepare is not None:
        prepare(cu.env)
    # the specialised pipeline evaluates the airtaxi relative position in its rotation form (lsm_step_common.cuh
    # relative_state_rot); the oracle restates both forms (oracle/lsm_oracle.c at_relative_state)
    spec = cu.env.launch_info()['specialised'] == 1
    prev_form = O.set_relative_state_form(1 if (spec and params.dynamics != 0) else 0)
    try:
        ora.reset(episode=episode, sample=True)
        cu.env.reset(episode)
        torch.cuda.synchronize()
        rng = np.random.default_rng(seed + 7)
        state_equal = np.ones(n, dtype=bool)

        def compare(tag):
            nonlocal state_equal
            so, sc = ora.get_state(), cu.get_state()
            bad = _report_divergence(tag, so, sc, ora, cu, state_equal, n)
            if params.num_obstacles > 0:      # declared obstacle extension: positions bit for bit, collision counters exact
                assert np.array_equal(so['obstacle_pos'], sc['obstacle_pos']), f"{tag}: obstacle positions differ"
                assert np.array_equal(so['num_obstacle_collisions'], sc['num_obstacle_collisions']), f"{tag}: obstacle collision counters differ"
            assert not bad.any(), f"{tag}: {int(bad.sum())} of {n} envs diverged in a discrete output (see the report above)"
            eq = np.ones(n, dtype=bool)
            for k in EXACT_STATE_KEYS:
                a, b = np.asarray(so[k]).reshape(n, -1), np.asarray(sc[k]).reshape(n, -1)
                same = ((a == b) | (np.isnan(a) & np.isnan(b))).all(axis=1)
                if not same.all():
                    e = int(np.nonzero(~same)[0][0]); j = int(np.nonzero(~((a[e] == b[e]) | (np.isnan(a[e]) & np.isnan(b[e]))))[0][0])
                    raise AssertionError(f"{tag}: float64 state '{k}' not bit-identical in {int((~same).sum())} envs; first: env {e} "
                                         f"[{j}] oracle={a[e, j]!r} cuda={b[e, j]!r}")
                eq &= same
            state_equal = eq
            G.assert_close(cu.obs, ora.obs, f'{tag} obs')
            G.assert_close(cu.node_obs, ora.node_obs, f'{tag} node_obs')
            G.assert_close(cu.adj, ora.adj, f'{tag} adj')
            G.assert_close(cu.reward, ora.reward, f'{tag} reward')

        compare('reset')
        for t in range(T):
            a = rng.integers(0, 25, (n, params.num_agents)).astype(np.int32)
            ora.step(a, episode=episode, auto_reset=auto_reset)
            cu.step(a, episode=episode)
            compare(f't={t}')
            G.assert_close(cu.ep_info, ora.ep_info, f't={t} ep_info')
    finally:
        O.set_relative_state_form(prev_form)
    return ora, cu


def test_oracle_batch_di_filter():
    """BASELINE config 2 shape (DI, 8 agents, filter on) on 512 seeded envs, 25 steps."""
    args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=250, world_size=4)
    _compare_with_oracle(args, G.BinaryFlags({}), n=512, T=25, episode=6249, seed=11, auto_reset=True)


def test_oracle_batch_di_nofilter_autoreset():
    """Config 1 shape with short episodes so that device-side auto-reset (Philox sampler) is exercised."""
    args = G.default_args(num_agents=3, use_safety_filter=False, episode_length=6, world_size=4)
    _compare_with_oracle(args, G.BinaryFlags({}), n=257, T=20, episode=0, seed=5, auto_reset=True)


def test_oracle_batch_di_allflags():
    args = G.default_args(num_agents=5, use_safety_filter=True, episode_length=10, world_size=2, collaborative=True)
    flags = G.BinaryFlags(dict(SAFETY_VIOLATION=True, HJ_VALUE=True, POTENTIAL_CONFLICT=True,
                               SEPARATION_DISTANCE_CURRICULUM=True, INITIAL_PHASE_USE_SAFETY_FILTER=True,
                               DIFF_FROM_FILTERED_ACTION=True))
    _compare_with_oracle(args, flags, n=300, T=25, episode=3500, seed=3, auto_reset=True)


def test_oracle_batch_airtaxi_filter_pc():
    """BASELINE config 3 shape (airtaxi, 10 agents, POTENTIAL_CONFLICT, filter on), obstacle-free."""
    args = G.default_args(dynamics_type='airtaxi', num_agents=10, use_safety_filter=True, episode_length=350, world_size=6)
    _compare_with_oracle(args, G.BinaryFlags(dict(POTENTIAL_CONFLICT=True)), n=256, T=25, episode=6249, seed=2,
                         auto_reset=True)


@pytest.mark.parametrize('shape', ['di', 'di_global', 'airtaxi_cfg3', 'di8_spec', 'airtaxi_generic'])
def test_oracle_batch_obstacle_extension(shape):
    """The DECLARED obstacle extension (BASELINE config 3 '+ obstacles'; the reference raises, see config.scenario_params_from_args):
    CUDA == C oracle on seeded batches (the specialised pipeline for the two obstacle shapes LSM_SPEC_LIST names - BASELINE
    config 3's 10 airtaxi agents + 4 obstacles and the 8-agent double integrator + 4 obstacles - the generic kernel otherwise) - Philox obstacle placement, agent positions redrawn while they collide
    with an obstacle, obstacle nodes / edges, Num_obst_collisions, auto-reset. The oracle itself is pinned by the fixtures
    di3_obst2 / di4_obst3_filter_global / at10_obst4_filter_pc (reference code + the two completed statements). Many
    obstacles in a small world so that rejections and collisions are frequent."""
    kw = dict(di=dict(num_agents=5, num_obstacles=12, world_size=1, episode_length=8, use_safety_filter=True),
              di_global=dict(num_agents=3, num_obstacles=32, world_size=1, episode_length=6, graph_feat_type='global'),
              airtaxi_cfg3=dict(dynamics_type='airtaxi', num_agents=10, num_obstacles=4, world_size=6, episode_length=350,
                                use_safety_filter=True),
              di8_spec=dict(num_agents=8, num_obstacles=4, world_size=1, episode_length=7, use_safety_filter=True),
              airtaxi_generic=dict(dynamics_type='airtaxi', num_agents=6, num_obstacles=9, world_size=1, episode_length=5,
                                   use_safety_filter=True))[shape]
    args = G.default_args(obstacle_extension=True, **kw)
    flags = G.BinaryFlags(dict(POTENTIAL_CONFLICT=True) if shape.startswith('airtaxi') else {})
    n, T = (96, 12) if shape.startswith('airtaxi') else (193, 20)
    ora, cu = _compare_with_oracle(args, flags, n=n, T=T, episode=6249 if shape != 'di_global' else 0, seed=17, auto_reset=True)
    assert cu.env.launch_info()['specialised'] == (1 if shape in ('airtaxi_cfg3', 'di8_spec') else 0)
    s = cu.get_state()
    if shape != 'airtaxi_cfg3':
        assert s['num_obstacle_collisions'].sum() > 0, "the scenario was meant to produce obstacle collisions"
    # COO edge list over E = N(1+L) + O entities in process_adj order (gnn.py:376-407): numpy nonzero of the dense tensor
    adj = cu.adj.reshape(n * args.num_agents, cu.env.E, cu.env.E)
    g, r, c = np.nonzero(adj)
    ei, ea = cu.env.edge_list()
    assert np.array_equal(ei.cpu().numpy(), np.stack([g * cu.env.E + r, g * cu.env.E + c]))
    assert np.array_equal(ea.cpu().numpy()[:, 0], adj[g, r, c])
    # the info dicts carry the counter (navigation_graph_safe.py:433)
    infos = cu.env.step(cu.torch.zeros((n, args.num_agents), dtype=cu.torch.int32, device=cu.env.device), 0)[6]
    st = cu.get_state()
    just_reset = cu.env.env_i32[3].cpu().numpy() != 0
    for e in range(0, n, 37):
        if not just_reset[e]:
            assert [infos[e][i]['Num_obst_collisions'] for i in range(args.num_agents)] == list(st['num_obstacle_collisions'][e])


def test_oracle_batch_dense32():
    """BASELINE config 4 shape (32 agents, E=96) on a few envs."""
    args = G.default_args(num_agents=32, use_safety_filter=True, episode_length=250, world_size=4)
    _compare_with_oracle(args, G.BinaryFlags({}), n=24, T=6, episode=6249, seed=9, auto_reset=True)


@pytest.mark.parametrize('shape', ['n32_l4', 'n32_l2_o32', 'n1', 'n2_l5_airtaxi'])
def test_oracle_batch_extreme_shapes(shape):
    """Maximum and minimum sizes on the generic kernel: 32 agents x 4 landmarks (128 landmarks = LSM_MAX_LANDMARKS, the np.int8
    index limit Q8; E = 160), 32 agents + 32 obstacles (E = 128), a single agent (empty "others" lists everywhere), and
    5 landmarks per airtaxi agent - against the C oracle, whose behaviour at 1 agent and at 3 / 4 landmarks is pinned by the
    fixtures di1_single_filter / at3_landmarks3 / di2_landmarks4."""
    kw = dict(n32_l4=dict(num_agents=32, num_landmarks=4, use_safety_filter=True, episode_length=250, world_size=4),
              n32_l2_o32=dict(num_agents=32, num_obstacles=32, obstacle_extension=True, use_safety_filter=True, episode_length=250,
                              world_size=2),
              n1=dict(num_agents=1, use_safety_filter=True, episode_length=5, world_size=1),
              n2_l5_airtaxi=dict(dynamics_type='airtaxi', num_agents=2, num_landmarks=5, use_safety_filter=True, episode_length=6,
                                 world_size=6))[shape]
    args = G.default_args(**kw)
    flags = G.BinaryFlags(dict(SAFETY_VIOLATION=True, POTENTIAL_CONFLICT=True, HJ_VALUE=True))
    n, T = (7, 4) if shape.startswith('n32') else (130, 14)
    ora, cu = _compare_with_oracle(args, flags, n=n, T=T, episode=6249, seed=23, auto_reset=True)
    assert cu.env.launch_info()['specialised'] == 0


def test_episode_stats_entry_point():
    """lsm_episode_stats (column sums of the episode summaries + env count in one launch) against numpy on the same buffer."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(num_agents=3, use_safety_filter=False, episode_length=4)
    env = B200GraphVecEnv(args, num_envs=1037, seed=4)
    env.reset(0)
    rng = np.random.default_rng(0)
    for _ in range(9):          # two auto-resets: the summaries are populated
        env.step(torch.as_tensor(rng.integers(0, 25, (1037, 3)).astype(np.int32), device=env.device), 0)
    want = env.ep_info.cpu().numpy().mean(axis=0)
    got = env.episode_stats()
    from layered_safe_marl_b200 import layout as LY
    assert np.allclose([got[k] for k in LY.EP_INFO_KEYS], want, rtol=1e-12, atol=0) and want[0] > 0


def test_onehot_actions_and_numpy_outputs():
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(num_agents=4, use_safety_filter=False, episode_length=25)
    e1 = B200GraphVecEnv(args, num_envs=33, seed=1)
    e2 = B200GraphVecEnv(args, num_envs=33, seed=1, numpy_outputs=True)
    e1.reset(0); e2.reset(0)
    rng = np.random.default_rng(0)
    for _ in range(5):
        idx = rng.integers(0, 25, (33, 4))
        onehot = np.eye(25)[idx]            # what GMPERunner.collect builds (graph_mpe_runner.py:431-433)
        o1 = e1.step(torch.as_tensor(idx, device=e1.device))
        o2 = e2.step(onehot)
        assert isinstance(o2[0], np.ndarray) and o2[0].dtype == np.float32
        for a, b in zip(o1[:6], o2[:6]):
            np.testing.assert_array_equal(a.cpu().numpy(), b)
    infos = o2[6]
    assert len(infos) == 33 and len(infos[0]) >= 4 and 'Safety filtered' in infos[0][0]


@pytest.mark.parametrize('shape', ['di8', 'air10', 'di32'])
def test_pair_value_variants_agree(shape):
    """The next step's HJ pair values may be produced at four places of the pipeline (behind the emit kernel, in front
    of the agent kernel, between the two, at the tail of the agent kernel itself; lsm_tuning.pair_placement) and from two layouts of the value grid (corner-packed
    table, scattered gathers; lsm_tuning.packed_grid). All of them must drive the filter identically: same deconflicting
    agent, same activation mask and bit-identical states."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(num_agents=8, world_size=4), air10=dict(dynamics_type='airtaxi', num_agents=10, world_size=6),
              di32=dict(num_agents=32, world_size=4))[shape]
    args = G.default_args(use_safety_filter=True, episode_length=250, **kw)
    n, T, episode = (64, 12, 6249) if shape != 'di32' else (16, 6, 6249)
    variants = [dict(pair_placement=0), dict(pair_placement=2), dict(pair_placement=3), dict(pair_placement=4),
                dict(pair_placement=0, packed_grid=0)]
    results = []
    rng = np.random.default_rng(4)
    acts = rng.integers(0, 25, (T, n, args.num_agents)).astype(np.int32)
    for tuning in variants:
        env = B200GraphVecEnv(args, num_envs=n, seed=21, tuning=tuning)
        assert env.launch_info()['pair_placement'] == tuning['pair_placement']
        env.reset(episode)
        filt = []
        for t in range(T):
            env.step(torch.as_tensor(acts[t], device=env.device), episode)
            s = env.get_state()
            filt.append((s['safety_filtered'].copy(), s['deconflicting_agent_index'].copy()))
        results.append((env.get_state(), filt, env.safe_action.cpu().numpy()))
        env.close()
    ref_state, ref_filt, ref_safe = results[0]
    assert sum(int(f[0].sum()) for f in ref_filt) > 0, "no filter activation in this rollout: the test would be vacuous"
    for (state, filt, safe), v in zip(results[1:], variants[1:]):
        for t in range(T):
            assert np.array_equal(filt[t][0], ref_filt[t][0]), f"{v}: filter mask differs at step {t}"
            assert np.array_equal(filt[t][1], ref_filt[t][1]), f"{v}: deconflicting agent differs at step {t}"
        assert np.array_equal(state['agent_values'], ref_state['agent_values']), f"{v}: states differ"
        assert np.array_equal(safe, ref_safe), f"{v}: applied controls differ"


@pytest.mark.parametrize('shape', ['di8', 'air10'])
def test_chunked_launches_identical(shape):
    """Big batches are split into env ranges on library-owned streams (fork / join by events; lsm_tuning.chunks). The
    split must not change a single bit of any output or state, including ragged last ranges and auto-resets."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(num_agents=8, world_size=4), air10=dict(dynamics_type='airtaxi', num_agents=10, world_size=6))[shape]
    args = G.default_args(use_safety_filter=True, episode_length=7, **kw)
    n, T, episode = 333, 10, 6249
    rng = np.random.default_rng(8)
    acts = rng.integers(0, 25, (T, n, args.num_agents)).astype(np.int32)
    outs = []
    for chunks in (1, 3, 4):
        env = B200GraphVecEnv(args, num_envs=n, seed=5, tuning=dict(chunks=chunks))
        assert env.launch_info()['chunks'] == chunks
        env.reset(episode)
        trace = []
        for t in range(T):
            o = env.step(torch.as_tensor(acts[t], device=env.device), episode)
            trace.append([x.cpu().numpy().copy() for x in o[:6]])
        outs.append((trace, env.get_state(), env.ep_info.cpu().numpy()))
        env.close()
    for trace, state, ep in outs[1:]:
        for t in range(T):
            for a, b in zip(trace[t], outs[0][0][t]):
                assert np.array_equal(a, b, equal_nan=True), f"step {t}: chunked output differs"
        for k in state:
            assert np.array_equal(np.asarray(state[k]), np.asarray(outs[0][1][k]), equal_nan=True), f"state {k} differs"
        assert np.array_equal(ep, outs[0][2], equal_nan=True)


@pytest.mark.parametrize('shape', ['di8', 'air10', 'di3', 'air10_obst4'])
def test_host_outputs_compact_adjacency_is_byte_identical(shape):
    """Host-facing path (numpy_outputs=True, what the unmodified runner consumes): the adjacency crosses PCIe as one
    thresholded E x E matrix per env + per-observer keep masks and is expanded on the host. Every returned array must be
    byte-identical to the device-resident env's dense outputs - with goals reached (disconnected landmarks), agents done
    and auto-resets in the rollout, and with the D2H copy chunked (n >= 256)."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(num_agents=8, world_size=2, use_safety_filter=True),
              air10=dict(dynamics_type='airtaxi', num_agents=10, world_size=6, use_safety_filter=True),
              di3=dict(num_agents=3, world_size=2, use_safety_filter=False),
              air10_obst4=dict(dynamics_type='airtaxi', num_agents=10, world_size=6, use_safety_filter=True, num_obstacles=4,
                               obstacle_extension=True))[shape]
    args = G.default_args(episode_length=12, **kw)
    n, T, episode = 300, 30, 6249
    dev_env = B200GraphVecEnv(args, num_envs=n, seed=3)
    # uneven env ranges and thread shares on purpose (300 envs in 7 ranges, 3 host threads)
    # (ordinary stores for one shape, streaming stores for the others: both expansion paths)
    host_env = B200GraphVecEnv(args, num_envs=n, seed=3, numpy_outputs=True, host_chunks=7, host_threads=3,
                               host_cached_stores=(shape == 'air10'))
    assert host_env._compact is not None
    o1, o2 = dev_env.reset(episode), host_env.reset(episode)
    for a, b in zip(o1[:4], o2[:4]):
        assert np.array_equal(a.cpu().numpy().view(np.uint8), np.ascontiguousarray(b).view(np.uint8))
    rng = np.random.default_rng(1)
    saw_disconnected = False
    for t in range(T):
        idx = rng.integers(0, 25, (n, args.num_agents)).astype(np.int32)
        o1 = dev_env.step(torch.as_tensor(idx, device=dev_env.device), episode)
        # the one-call host step (lsm_step_host) takes indices or one-hot rows, pageable or page-locked
        if t % 3 == 0:
            o2 = host_env.step(idx, episode)
        elif t % 3 == 1:
            o2 = host_env.step(np.eye(25, dtype=np.float32)[idx], episode)
        else:
            pinned = torch.from_numpy(np.eye(25, dtype=np.float32)[idx]).pin_memory()
            o2 = host_env.step(pinned.numpy(), episode)
        for k, (a, b) in enumerate(zip(o1[:6], o2[:6])):
            assert np.array_equal(a.cpu().numpy().view(np.uint8), np.ascontiguousarray(b).view(np.uint8)), f"step {t} output {k}"
        st = dev_env.get_state()
        saw_disconnected |= bool((st['reached_goal'] > 0).any())
    assert saw_disconnected or shape.startswith('air10'), "no goal was reached: the keep masks were never exercised"


def test_infos_on_an_auto_reset_step_are_the_terminal_steps():
    """graphworker returns the TERMINAL step's per-agent info dicts and appends the episode summary
    (onpolicy/envs/env_wrappers.py:861-874); the device state of such an env already belongs to the new episode. The
    kernels snapshot the info fields before the reset; LazyInfos must return them. Checked against the oracle stepped
    WITHOUT auto-reset from the same pre-step state."""
    import torch
    import oracle_env as O
    from layered_safe_marl_b200 import B200GraphVecEnv, config as cfg, infos as I, layout as LY
    args = G.default_args(num_agents=4, use_safety_filter=True, episode_length=5, world_size=2)
    flags = G.BinaryFlags({})
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = G.value_grid_for(params)
    n, episode = 64, 6249
    env = B200GraphVecEnv(args, num_envs=n, seed=17, binary_cfg=flags)
    env.reset(episode)
    rng = np.random.default_rng(5)
    checked = 0
    for t in range(12):
        pre = env.get_state()
        idx = rng.integers(0, 25, (n, 4)).astype(np.int32)
        out = env.step(torch.as_tensor(idx, device=env.device), episode)
        infos = out[6]
        jr = infos.just_reset()
        if not jr.any():
            continue
        ora = O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=17, nthreads=4)
        ora.set_state(pre)
        ora.step(idx, episode=episode, auto_reset=False)
        want = I.compute_agent_infos(ora.agent_f64, ora.agent_i32, ora.env_i32, ora.reward,
                                     I.separation_distance_of(params, ora.env_f64[LY.EF_CURRICULUM_RATIO]))
        for e in np.nonzero(jr)[0]:
            got = infos[int(e)]
            assert len(got) == 5 and 'done_percentage' in got[4]          # N agent dicts + the episode summary
            for i in range(4):
                for k in I.AGENT_INFO_KEYS:
                    if k == 'individual_reward':
                        G.assert_close(got[i][k], want[k][e, i], f'{k}')
                    else:
                        assert np.array_equal(np.asarray(got[i][k]), np.asarray(want[k][e, i]), equal_nan=True), \
                            f"t={t} env {e} agent {i} info['{k}']: got {got[i][k]!r} want {want[k][e, i]!r}"
            checked += 1
    assert checked >= 10, "episode_length=5 must produce auto-resets in 12 steps"


def test_pinned_host_actions_are_used_in_place():
    """Host-facing path (lsm_step_host): a page-locked one-hot array is DMA'd straight from the caller's memory, a pageable
    one goes through the library's staging buffer; both give the same step."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=25, world_size=4)
    rng = np.random.default_rng(2)
    idx = rng.integers(0, 25, (4, 40, 8))
    onehot = np.eye(25, dtype=np.float32)[idx]
    pinned = torch.from_numpy(onehot.copy()).pin_memory()
    outs = []
    for use_pinned in (False, True):
        env = B200GraphVecEnv(args, num_envs=40, seed=9, numpy_outputs=True)
        env.reset(6249)
        trace = []
        for t in range(4):
            a = pinned[t].numpy() if use_pinned else onehot[t]
            o = env.step(a, 6249)
            trace.append([np.array(x) for x in o[:6]])
        outs.append(trace)
        env.close()
    for ta, tb in zip(*outs):
        for x, y in zip(ta, tb):
            assert np.array_equal(x, y, equal_nan=True)


@pytest.mark.parametrize('dyn,N', [('double_integrator', 4), ('double_integrator', 16), ('airtaxi', 4), ('airtaxi', 8), ('airtaxi', 16)])
def test_oracle_batch_reference_script_shapes(dyn, N):
    """The shapes the reference's own scripts ship with (train.sh: 4 agents; eval_airtaxi.sh: 8 / 16; eval_double_integrator.sh: 4)
    run the specialised pipeline; same bar as the benchmark shapes."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    air = dyn == 'airtaxi'
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=True, episode_length=350 if air else 250,
                          world_size=6 if air else 4)
    probe = B200GraphVecEnv(args, num_envs=4, seed=0)
    assert probe.launch_info()['specialised'] == 1
    probe.close()
    _compare_with_oracle(args, G.BinaryFlags(dict(POTENTIAL_CONFLICT=air)), n=96, T=12, episode=6249, seed=13 + N,
                         auto_reset=True)


@pytest.mark.parametrize('dyn,N', [('double_integrator', 8), ('airtaxi', 4)])
def test_oracle_batch_global_features_run_the_specialised_pipeline(dyn, N):
    """graph_feat_type='global' (navigation_graph_safe.py:1017-1036: 7-wide observer-independent node rows) on the
    specialised three-kernel pipeline, against the oracle on a seeded batch with goals reached and auto-resets."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    air = dyn == 'airtaxi'
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=True, episode_length=9, world_size=6 if air else 3,
                          graph_feat_type='global')
    probe = B200GraphVecEnv(args, num_envs=4, seed=0)
    assert probe.launch_info()['specialised'] == 1 and probe.F == 7
    probe.close()
    _compare_with_oracle(args, G.BinaryFlags({}), n=200, T=14, episode=6249, seed=31, auto_reset=True)


@pytest.mark.parametrize('dyn,N', [('double_integrator', 8), ('airtaxi', 10), ('airtaxi', 6)])
def test_oracle_batch_float32_interpolation(dyn, N):
    """LSM_FLAG_INTERP_FLOAT32 (args.interp_float32): the float32 arithmetic of Grid.interpolate (a parity mode; it runs on
    the generic fused kernel for every shape) - same zero-tolerance bar against the oracle."""
    air = dyn == 'airtaxi'
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=True, episode_length=12, world_size=6 if air else 3,
                          interp_float32=True)
    _compare_with_oracle(args, G.BinaryFlags(dict(POTENTIAL_CONFLICT=air, HJ_VALUE=(N == 6))), n=160, T=16, episode=6249, seed=41,
                         auto_reset=True)


@pytest.mark.parametrize('shape', ['di8', 'air10'])
def test_graph_replay_is_bit_identical(shape):
    """lsm_tuning.use_graph: once the same parameter block repeats, a step's launches are replayed from a CUDA graph. The
    replayed steps must be bit-identical to plain launches - across an episode-number change (in-place graph update),
    re-pointed output buffers, a state edit (pair kernel in front of the next step) and auto-resets."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(num_agents=8, world_size=2, use_safety_filter=True),
              air10=dict(dynamics_type='airtaxi', num_agents=10, world_size=6, use_safety_filter=True))[shape]
    args = G.default_args(episode_length=9, **kw)
    n, T = 192, 40
    envs = [B200GraphVecEnv(args, num_envs=n, seed=5, tuning=dict(use_graph=g)) for g in (0, 1)]
    rng = np.random.default_rng(8)
    acts = [torch.zeros((n, args.num_agents), dtype=torch.int32, device=e.device) for e in envs]
    alt = [(torch.empty_like(e.node_obs), torch.empty_like(e.adj)) for e in envs]
    for e in envs:
        e.reset(6249)
    for t in range(T):
        idx = torch.as_tensor(rng.integers(0, 25, (n, args.num_agents)).astype(np.int32))
        episode = 6249 if t < 25 else 3000
        outs = []
        for e, a, (nb, ab) in zip(envs, acts, alt):
            a.copy_(idx)
            if t == 15:
                e.set_output_buffers(node_obs=nb, adj=ab)
            if t == 30:
                st = e.get_state(); e.set_state(st)          # marks the pair values stale: pair kernel in front once
            o = e.step(a, episode)
            outs.append([x.cpu().numpy().copy() for x in o[:6]])
        for k, (x, y) in enumerate(zip(*outs)):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"step {t} output {k}"
    sa, sb = envs[0].get_state(), envs[1].get_state()
    for k in sa:
        assert np.array_equal(np.asarray(sa[k]), np.asarray(sb[k]), equal_nan=True), f"state {k}"
    li0, li1 = envs[0].launch_info(), envs[1].launch_info()
    assert li0['graph_replays'] == 0 and li0['graph_captures'] == 0
    assert li1['graph_replays'] >= T - 12 and 1 <= li1['graph_captures'] <= 8, li1
    for e in envs:
        e.close()


@pytest.mark.parametrize('shape', ['di8', 'air10', 'di4'])
def test_pair_tail_placement_through_resets(shape):
    """pair_placement=4 (the agent kernel leaves the next step's pair values behind itself) against the pair kernel behind
    the emit kernel: bit-identical outputs and states through auto-resets, a curriculum episode where the filter is off
    for part of the envs' life, a state edit (stale values -> pair kernel in front once) and a masked reset."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    kw = dict(di8=dict(num_agents=8, world_size=2), air10=dict(dynamics_type='airtaxi', num_agents=10, world_size=6),
              di4=dict(num_agents=4, world_size=2))[shape]
    args = G.default_args(use_safety_filter=True, episode_length=7, **kw)
    n, T = 160, 36
    envs = [B200GraphVecEnv(args, num_envs=n, seed=13, tuning=dict(pair_placement=p)) for p in (0, 4)]
    assert [e.launch_info()['launches_per_step'] for e in envs] == [3, 2]
    rng = np.random.default_rng(3)
    for e in envs:
        e.reset(6249)
    for t in range(T):
        idx = rng.integers(0, 25, (n, args.num_agents)).astype(np.int32)
        episode = 6249 if t < 20 else 3500
        outs = []
        for e in envs:
            if t == 12:
                st = e.get_state(); e.set_state(st)
            if t == 24:
                mask = torch.zeros(n, dtype=torch.uint8, device=e.device); mask[::3] = 1
                from layered_safe_marl_b200 import _lib
                _lib.check(e.lib.lsm_reset(e._h, mask.data_ptr(), 3500, e.seed, 1, e._stream()), 'lsm_reset')
            o = e.step(torch.as_tensor(idx, device=e.device), episode)
            outs.append([x.cpu().numpy().copy() for x in o[:6]] + [e.safe_action.cpu().numpy().copy()])
        for k, (x, y) in enumerate(zip(*outs)):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"step {t} output {k}"
    sa, sb = envs[0].get_state(), envs[1].get_state()
    assert int(sa['safety_filtered'].sum()) >= 0
    for k in sa:
        assert np.array_equal(np.asarray(sa[k]), np.asarray(sb[k]), equal_nan=True), f"state {k}"
    for e in envs:
        e.close()
