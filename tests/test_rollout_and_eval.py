"""N1 / N4 rows (SURVEY.md section 8f): device rollout storage, GraphDummyVecEnv surface, deterministic eval scenarios.

CPU tests check the host logic against numpy restatements of the reference lines they mirror and run the
eval scenarios through the C oracle; GPU tests check the CUDA path (zero-copy slot binding, parity with the oracle)."""
import os
import sys
import types

import numpy as np
import pytest
import torch

import _golden as G

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle'))

from layered_safe_marl_b200 import config as cfg, eval_scenarios as ES
from layered_safe_marl_b200.rollout import DeviceGraphRolloutBuffer
from layered_safe_marl_b200.spaces import Discrete


def _fake_env(n, N, L, D, F, device='cpu'):
    e = types.SimpleNamespace()
    e.num_envs, e.N, e.E, e.D, e.F, e.device = n, N, N * (1 + L), D, F, torch.device(device)
    e.action_space = [Discrete(25) for _ in range(N)]
    e.agent_id = torch.arange(N, dtype=torch.int32).view(1, N, 1).expand(n, N, 1).contiguous()
    return e


ROLLOUT_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'aux', 'rollout_buffer.npz')


def _drive(rb, z, n, N, T, p):
    """One pass of T inserts with the fixture's inputs, then compute_returns - what GMPERunner.run does per episode."""
    for t in range(T):
        k = p * T + t
        g = lambda name: torch.from_numpy(z['in_' + name][k])
        rb.insert((g('obs'), torch.from_numpy(z['in_agent_id']), g('node_obs'), g('adj'), g('rewards')[..., 0], g('dones'), None),
                  values=g('values'), actions=g('actions'), action_log_probs=g('action_log_probs'),
                  rnn_states=g('rnn_states'), rnn_states_critic=g('rnn_states_critic'))
    rb.compute_returns(torch.from_numpy(z['in_next_values'][p]))


@pytest.mark.parametrize('use_gae', [True, False])
@pytest.mark.parametrize('proper', [False, True])
@pytest.mark.parametrize('centralized', [True, False])
def test_rollout_buffer_matches_the_reference_buffer(use_gae, proper, centralized):
    """DeviceGraphRolloutBuffer against the UNMODIFIED reference: GMPERunner.insert (graph_mpe_runner.py:444-487) +
    GraphReplayBuffer.insert / compute_returns / after_update (graph_buffer.py:168-373) run on seeded inputs by
    oracle/gen_rollout_golden.py (fixture tests/golden/aux/rollout_buffer.npz): two passes over the buffer, whole envs
    done, GAE and discounted returns, with and without use_proper_time_limits, centralised and decentralised critic
    inputs. Every stored array must be identical; the returns (a float32 recursion) to 1e-6."""
    z = np.load(ROLLOUT_GOLDEN)
    n, N, L, D, F, T = (int(v) for v in z['meta'])
    env = _fake_env(n, N, L, D, F)
    rb = DeviceGraphRolloutBuffer(env, episode_length=T, gamma=0.97, gae_lambda=0.9, use_gae=use_gae,
                                  use_proper_time_limits=proper, use_centralized_V=centralized, hidden_size=8)
    tag = f"gae{int(use_gae)}_ptl{int(proper)}_cv{int(centralized)}"
    obs0 = torch.from_numpy(z['in_obs0'])
    rb.warmup(reset_out=(obs0, torch.from_numpy(z['in_agent_id']), torch.zeros_like(rb.node_obs[0]), torch.zeros_like(rb.adj[0])))
    rb.bad_masks.copy_(torch.from_numpy(z['in_bad_masks']))
    for p in range(2):
        _drive(rb, z, n, N, T, p)
        assert rb.step == 0                      # wrapped around after T inserts
        for key in z.files:
            pre = f"{tag}_pass{p}_"
            if not key.startswith(pre) or '_after_' in key:
                continue
            name = key[len(pre):]
            got, want = getattr(rb, name).numpy(), z[key]
            if name in ('returns', 'value_preds'):
                np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6, err_msg=key)
            else:
                np.testing.assert_array_equal(got, want, err_msg=key)
        rb.after_update()
        for name in ('share_obs', 'obs', 'masks', 'active_masks', 'rnn_states'):
            np.testing.assert_array_equal(getattr(rb, name)[0].numpy(), z[f"{tag}_pass{p}_after_{name}0"], err_msg=name)
    oh = DeviceGraphRolloutBuffer.one_hot_actions(torch.from_numpy(z['in_actions'][0].astype(np.int64)))
    assert oh.shape == (n, N, 25) and float(oh.sum()) == n * N
    assert np.array_equal(oh.numpy(), np.squeeze(np.eye(25)[z['in_actions'][0].astype(np.int64)], 2).astype(np.float32))   # graph_mpe_runner.py:431-433


@pytest.mark.skipif(not G.have_reference('onpolicy'), reason=G.REFERENCE_SKIP)
def test_rollout_golden_fixture_is_reproducible_from_the_reference(tmp_path):
    """Regenerate the fixture from the original project and compare with the committed one."""
    import subprocess
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(repo, 'oracle', 'gen_rollout_golden.py')).read().replace(
        "os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'aux', 'rollout_buffer.npz')", repr(str(tmp_path / 'r.npz'))).replace(
        "os.makedirs(os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'aux'), exist_ok=True)", "pass").replace(
        "HERE = os.path.dirname(os.path.abspath(__file__))", f"HERE = {os.path.join(repo, 'oracle')!r}")
    script = tmp_path / 'gen.py'
    script.write_text(src)
    subprocess.check_call([sys.executable, str(script)], stdout=subprocess.DEVNULL)
    a, b = np.load(ROLLOUT_GOLDEN), np.load(tmp_path / 'r.npz')
    assert sorted(a.files) == sorted(b.files)
    for k in a.files:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_runner_view_feeds_an_unmodified_collect():
    """GMPERunner.collect (graph_mpe_runner.py:398-415) reads `np.concatenate(self.buffer.<field>[step])`. The view
    returned by DeviceGraphRolloutBuffer.runner_view() answers that call with the (n*N, ...) reshape of the DEVICE tensor
    (NumPy's __array_function__ protocol): no host concatenation, no copy - and the same values numpy would produce."""
    n, N, L, D, F, T = 4, 3, 2, 7, 10, 3
    env = _fake_env(n, N, L, D, F)
    rb = DeviceGraphRolloutBuffer(env, episode_length=T)
    g = torch.Generator().manual_seed(0)
    for name in ('share_obs', 'obs', 'node_obs', 'adj', 'rnn_states', 'rnn_states_critic', 'masks'):
        getattr(rb, name).copy_(torch.rand(getattr(rb, name).shape, generator=g))
    view = rb.runner_view()
    for step in (0, 2):
        for name in ('share_obs', 'obs', 'node_obs', 'adj', 'agent_id', 'share_agent_id', 'rnn_states', 'rnn_states_critic', 'masks'):
            got = np.concatenate(getattr(view, name)[step])          # exactly the expression the runner evaluates
            assert torch.is_tensor(got) and got.data_ptr() == getattr(rb, name)[step].data_ptr()     # a view, not a copy
            want = np.concatenate(getattr(rb, name)[step].numpy())
            assert tuple(got.shape) == want.shape and np.array_equal(got.numpy(), want)


@pytest.mark.parametrize('name,N', [('circular', 6), ('two_vehicle_conflict', 2), ('three_vehicle_conflict', 3)])
def test_eval_scenarios_run_through_the_oracle(name, N):
    import oracle_env as O
    dyn = 'double_integrator' if name == 'circular' else 'airtaxi'
    kw = dict(num_agents=N, dynamics_type=dyn) if name == 'circular' else {}
    s = ES.build(name, **kw)
    assert s['agent_values'].shape == (1, N, 4) and s['landmark_pos'].shape == (1, 2 * N, 2)
    mind = {}
    for use_filter in (False, True):
        args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=use_filter, episode_length=400,
                              world_size=4 if dyn == 'double_integrator' else 6)
        params = cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags({}))
        vg, tg = G.value_grid_for(params)
        ora = O.OracleEnv(params.asdict(), 1, value_grid=vg, ttr_grid=tg, seed=0, nthreads=1)
        ora.set_state({k: v for k, v in s.items() if k != 'note'})
        ora.reset(episode=params.num_total_episode - 1, sample=False)
        m = np.inf
        act = np.full((1, N), 12, dtype=np.int32)          # zero acceleration / zero turn-rate primitive
        for t in range(60 if dyn == 'airtaxi' else 80):
            ora.step(act, episode=params.num_total_episode - 1, auto_reset=False)
            st = ora.get_state()
            mr = np.asarray(st['min_relative_distance'])
            m = min(m, float(mr[np.isfinite(mr)].min())) if np.isfinite(mr).any() else m
        mind[use_filter] = m
    # the conflict examples are head-on without the filter; the HJ filter (synthetic grid) must not make them closer
    if name != 'circular':
        assert mind[True] >= mind[False] - 1e-9, mind


@pytest.mark.gpu
def test_dummy_vec_env_has_no_auto_reset_and_returns_reset_count():
    from layered_safe_marl_b200 import B200GraphDummyVecEnv
    args = G.default_args(num_agents=3, episode_length=4)
    env = B200GraphDummyVecEnv(args, num_envs=7, seed=3)
    env.reset(0)
    a = torch.zeros((7, 3), dtype=torch.int32, device=env.device)
    for t in range(6):
        out = env.step(a, 0)
        assert len(out) == 8 and out[7] == 0
    st = env.get_state()
    assert (st['current_step'] == 6).all()             # past episode_length: no reset happened
    assert out[5].all()                                # every agent reports done (time limit)


@pytest.mark.gpu
def test_zero_copy_rollout_equals_copying_rollout():
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=250, world_size=4)
    T = 5
    envs = [B200GraphVecEnv(args, num_envs=64, seed=9) for _ in range(2)]
    bufs = [DeviceGraphRolloutBuffer(envs[0], T, zero_copy=False), DeviceGraphRolloutBuffer(envs[1], T, zero_copy=True)]
    for b in bufs:
        b.warmup(num_current_episode=6249)
    gen = torch.Generator(device='cpu'); gen.manual_seed(1)
    for t in range(T):
        a = torch.randint(0, 25, (64, 8), generator=gen, dtype=torch.int32).to(envs[0].device)
        for env, b in zip(envs, bufs):
            b.insert(env.step(a, 6249), actions=a.unsqueeze(-1).float())
    torch.cuda.synchronize()
    for k in ('obs', 'share_obs', 'node_obs', 'adj', 'rewards', 'masks', 'active_masks', 'actions'):
        assert torch.equal(getattr(bufs[0], k), getattr(bufs[1], k)), k
    assert float(bufs[1].adj.abs().sum()) > 0 and float(bufs[1].node_obs.abs().sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize('name,N', [('circular', 8), ('three_vehicle_conflict', 3)])
def test_eval_scenarios_cuda_matches_oracle(name, N):
    import oracle_env as O
    from layered_safe_marl_b200 import B200GraphDummyVecEnv
    dyn = 'double_integrator' if name == 'circular' else 'airtaxi'
    kw = dict(num_agents=N, dynamics_type=dyn) if name == 'circular' else {}
    s = {k: v for k, v in ES.build(name, **kw).items() if k != 'note'}
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=True, episode_length=400,
                          world_size=4 if dyn == 'double_integrator' else 6)
    params = cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags({}))
    vg, tg = G.value_grid_for(params)
    ep = params.num_total_episode - 1
    ora = O.OracleEnv(params.asdict(), 1, value_grid=vg, ttr_grid=tg, seed=0, nthreads=1)
    env = B200GraphDummyVecEnv(args, num_envs=1, seed=0)
    ora.set_state(s); ora.reset(episode=ep, sample=False)
    env.set_state(s); env.reset_from_state(ep)
    rng = np.random.default_rng(4)
    for t in range(40):
        a = rng.integers(0, 25, (1, N)).astype(np.int32)
        ora.step(a, episode=ep, auto_reset=False)
        out = env.step(torch.as_tensor(a, device=env.device), ep)
        so, sc = ora.get_state(), env.get_state()
        for k in ('reached_goal', 'done', 'safety_filtered', 'deconflicting_agent_index'):
            np.testing.assert_array_equal(np.asarray(so[k]), np.asarray(sc[k]), err_msg=f't={t} {k}')
        np.testing.assert_array_equal(ora.adj != 0, out[3].cpu().numpy() != 0)
        G.assert_close(out[2].cpu().numpy(), ora.node_obs, f't={t} node_obs')
        G.assert_close(out[4].cpu().numpy(), ora.reward, f't={t} reward')


def _process_adj(adj):
    """TransformerConvNet.process_adj, reference onpolicy/algorithms/utils/gnn.py:376-407 (3-D case), verbatim semantics."""
    batch_size, num_nodes, _ = adj.shape
    edge_index = adj.nonzero(as_tuple=False)
    edge_attr = adj[edge_index[:, 0], edge_index[:, 1], edge_index[:, 2]]
    batch = edge_index[:, 0] * num_nodes
    edge_index = torch.stack([batch + edge_index[:, 1], batch + edge_index[:, 2]], dim=0)
    return edge_index, edge_attr.unsqueeze(1)


@pytest.mark.gpu
@pytest.mark.parametrize('N,dyn,world,chunks', [(8, 'double_integrator', 4, 1), (8, 'double_integrator', 10, 3), (3, 'double_integrator', 6, 1),
                                                 (10, 'airtaxi', 6, 1), (10, 'airtaxi', 14, 4), (32, 'double_integrator', 4, 1),
                                                 (32, 'double_integrator', 16, 2), (-8, 'double_integrator', 3, 2), (-10, 'airtaxi', 6, 1)])
def test_fused_edge_output_matches_process_adj(N, dyn, world, chunks):
    """N2, fused: the emission kernel writes (edge_index, edge_attr) itself (lsm_set_edge_output). Bit-exact against the
    reference's process_adj (gnn.py:376-407) applied to the dense adjacency of a twin env, at the cfg2 / cfg3 / cfg4
    shapes, dense and sparse worlds, chunked launches (per-range prefixes joined by events), goals reached and
    auto-resets; then with dense_adj=False (no dense tensor written at all) against the same twin."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    obst = 4 if N < 0 else 0          # negative N: the same shape with 4 obstacles (declared extension, specialised pipeline)
    N = abs(N)
    n = 61 if N == 32 else 203
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=(N != 3), episode_length=9, world_size=world,
                          num_obstacles=obst, obstacle_extension=obst > 0)
    twin = B200GraphVecEnv(args, num_envs=n, seed=5)
    env = B200GraphVecEnv(args, num_envs=n, seed=5, tuning=dict(chunks=chunks))
    assert env.launch_info()['chunks'] == chunks
    env.enable_edge_output(dense_adj=True)
    sparse = B200GraphVecEnv(args, num_envs=n, seed=5, tuning=dict(chunks=chunks))
    sparse.enable_edge_output(dense_adj=False)
    sparse.adj.fill_(-7.0)
    episode = 6249
    o0, o1, o2 = twin.reset(episode), env.reset(episode), sparse.reset(episode)

    def check(tag):
        ri, ra = _process_adj(twin.adj.reshape(-1, twin.E, twin.E))
        for e, name in ((env, 'dense+edges'), (sparse, 'edges only')):
            ei, ea = e.edges()
            assert ei.dtype == torch.int64 and ea.dtype == torch.float32
            assert ei.shape == ri.shape, f"{tag} {name}: nnz {ei.shape[1]} vs {ri.shape[1]}"
            assert torch.equal(ei, ri) and torch.equal(ea, ra), f"{tag} {name}"
            cnt = (twin.adj.reshape(-1, twin.E * twin.E) != 0).sum(dim=1).to(torch.int32)
            assert torch.equal(e.edge_counts, cnt), f"{tag} {name}: per-graph counts"
            assert torch.equal(e.edge_offsets[:-1], torch.cumsum(cnt.long(), 0) - cnt.long()), f"{tag} {name}: offsets"
        assert torch.equal(env.adj, twin.adj) and torch.equal(env.node_obs, twin.node_obs), f"{tag}: dense outputs changed"
        assert torch.equal(sparse.node_obs, twin.node_obs)
        assert bool((sparse.adj == -7.0).all()), f"{tag}: dense_adj=False must not touch the dense tensor"

    check('reset')
    gen = torch.Generator(device='cpu'); gen.manual_seed(2)
    for t in range(12):                                   # crosses an auto-reset
        a = torch.randint(0, 25, (n, N), generator=gen, dtype=torch.int32).to(env.device)
        twin.step(a, episode); env.step(a, episode)
        out = sparse.step(a, episode)
        assert out[3] is None
        check(f't={t}')


@pytest.mark.gpu
@pytest.mark.parametrize('N,dyn', [(8, 'double_integrator'), (3, 'double_integrator'), (10, 'airtaxi')])
def test_edge_list_matches_process_adj(N, dyn):
    """N2: the device COO builder against the reference's own torch code on the adjacency of real steps
    (bit-exact integer indices, bit-exact float32 attributes, ragged graphs incl. empty ones)."""
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=False, episode_length=12,
                          world_size=8 if dyn == 'double_integrator' else 12)     # sparse: many pairs beyond the radius
    env = B200GraphVecEnv(args, num_envs=97, seed=5)
    env.reset(0)
    gen = torch.Generator(device='cpu'); gen.manual_seed(2)
    for t in range(14):                                   # crosses an auto-reset
        a = torch.randint(0, 25, (97, N), generator=gen, dtype=torch.int32).to(env.device)
        out = env.step(a, 0)
        adj = out[3]
        ei, ea = env.edge_list()
        ri, ra = _process_adj(adj.reshape(-1, env.E, env.E))
        assert ei.dtype == torch.int64 and ea.dtype == torch.float32 and ea.shape == ra.shape
        assert torch.equal(ei, ri), f't={t}'
        assert torch.equal(ea, ra), f't={t}'
    # an all-zero adjacency (no edges at all) and a user-supplied tensor
    z = torch.zeros_like(env.adj)
    ei, ea = env.edge_list(z)
    assert ei.shape == (2, 0) and ea.shape == (0, 1)


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['di4', 'at4', 'boundary', 'di4_obst3'])
def test_world_graph_matches_reference_update_graph(tag):
    """Row a16: lsm_world_graph against world.edge_list / world.edge_weight recorded from the unmodified reference's
    update_graph (navigation_graph_safe.py:996-1015; fixture + generator oracle/gen_world_graph_golden.py): every
    recorded step of a rollout is loaded as one environment of a batch. Integer indices and float64 weights bit-exact;
    the inclusive radius (an entity exactly 4.0 away IS connected, one ulp farther is not) is part of the fixture.
    'di4_obst3': the declared obstacle extension (obstacle nodes in the world graph; update_graph is reference code)."""
    import json
    from layered_safe_marl_b200 import B200GraphVecEnv
    obst = tag.endswith('obst3')
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'aux', 'world_graph_obstacles.npz' if obst else 'world_graph.npz'))
    meta = json.loads(str(z['meta']))[tag]
    steps = meta['steps']
    args = G.default_args(num_landmarks=2, use_safety_filter=False, obstacle_extension=obst, **meta['args'])
    env = B200GraphVecEnv(args, num_envs=steps, seed=0)
    env.reset(0)
    s = env.get_state()
    for k in ('agent_values', 'done', 'reached_goal', 'landmark_pos', 'landmark_heading', 'landmark_speed') + \
            (('obstacle_pos', 'num_obstacle_collisions') if obst else ()):
        s[k] = z[f'{tag}__{k}']
    env.set_state(s)
    ei, ew, off = env.world_graph()
    ei, ew, off = ei.cpu().numpy(), ew.cpu().numpy(), off.cpu().numpy()
    lens = z[f'{tag}__edge_list_len']
    assert np.array_equal(np.diff(off), lens), "edges per environment"
    assert np.array_equal(ei, z[f'{tag}__edge_list'])
    assert np.array_equal(ew, z[f'{tag}__edge_weight'])
    if tag == 'boundary':
        pairs = set(map(tuple, ei.T.tolist()))
        assert (0, 1) in pairs and (1, 0) in pairs and (0, 2) not in pairs
    else:
        assert lens.min() < lens.max()          # disconnected entities changed the graph along the rollout


@pytest.mark.parametrize('tag,name,kw', [('circular', 'circular', dict(num_agents=6, dynamics_type='double_integrator', world_size=4.0)),
                                         ('circular_at', 'circular', dict(num_agents=5, dynamics_type='airtaxi', world_size=6.0)),
                                         ('two_vehicle_conflict', 'two_vehicle_conflict', {}),
                                         ('three_vehicle_conflict', 'three_vehicle_conflict', {})])
def test_eval_scenarios_match_the_reference_scenario_class(tag, name, kw):
    """N4: the injectable initial states of eval_scenarios.py against what the reference's own scenario class builds
    (fixture recorded by oracle/gen_eval_scenarios_golden.py from navigation_graph_safe_eval.py through the import stubs):
    agent states and the first goal of every agent - position, heading, speed."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'aux', 'eval_scenarios.npz'))
    s = ES.build(name, **kw)
    N = z[f'{tag}__agent_values'].shape[0]
    np.testing.assert_allclose(s['agent_values'][0], z[f'{tag}__agent_values'], rtol=0, atol=1e-12)
    np.testing.assert_allclose(s['landmark_pos'][0, :N], z[f'{tag}__goal0_pos'], rtol=0, atol=1e-12)
    np.testing.assert_allclose(s['landmark_heading'][0, :N], z[f'{tag}__goal0_heading'], rtol=0, atol=1e-12)
    np.testing.assert_allclose(s['landmark_speed'][0, :N], z[f'{tag}__goal0_speed'], rtol=0, atol=1e-12)
