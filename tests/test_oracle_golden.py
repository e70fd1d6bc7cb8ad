"""CPU: the C oracle (oracle/lsm_oracle.c) against golden rollouts of the UNMODIFIED reference.

Bar: adjacency pattern, done flags, goal counters, filter masks and deconflicting indices bit-exact;
continuous values within 1e-5 relative (tests/_golden.RTOL) at every step of the rollout.
"""
import os
import sys

import numpy as np
import pytest

import _golden as G

sys.path.insert(0, os.path.join(G.os.path.dirname(G.GOLDEN_DIR), '..', 'oracle'))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle'))
import oracle_env as O  # noqa: E402

CASES = G.golden_names()


def make_oracle(params, n=1, seed=0):
    vg, tg = G.value_grid_for(params)
    return O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=seed)


def test_fixtures_present():
    assert len(CASES) >= 10


@pytest.mark.parametrize('name', CASES)
def test_reset_observation(name):
    z, meta, args, flags, params = G.load_case(name)
    env = make_oracle(params)
    env.set_state(G.state0(z))
    env.observe()
    G.assert_close(env.obs[0], z['obs0'], 'obs0')
    G.assert_close(env.node_obs[0], z['node_obs0'], 'node_obs0')
    G.assert_same_mask(env.adj[0] != 0, z['adj0'] != 0, 'adj0 pattern')
    G.assert_close(env.adj[0], z['adj0'], 'adj0')


def check_step(env, z, t, name):
    """Compare env (after stepping to time t) with the golden record; raises AssertionError."""
    tag = f"{name} t={t}"
    G.assert_same_mask(env.adj[0] != 0, z['adj'][t] != 0, f'{tag} adj pattern')
    G.assert_same_mask(env.done[0].astype(bool), z['done'][t], f'{tag} done')
    s = env.get_state()
    G.assert_same_mask(s['reached_goal'][0], z['st_reached_goal'][t], f'{tag} reached_goal')
    G.assert_same_mask(s['done'][0], z['st_done'][t], f'{tag} agent.done')
    G.assert_same_mask(s['safety_filtered'][0], z['st_safety_filtered'][t], f'{tag} safety_filtered')
    G.assert_same_mask(s['deconflicting_agent_index'][0], z['st_deconflicting_agent_index'][t], f'{tag} deconflict idx')
    G.assert_same_mask(s['num_agent_collisions'][0], z['st_num_agent_collisions'][t], f'{tag} collisions')
    if 'st_num_obstacle_collisions' in z.files:      # declared obstacle extension
        G.assert_same_mask(s['num_obstacle_collisions'][0], z['st_num_obstacle_collisions'][t], f'{tag} obstacle collisions')
    for k in ('ep_travel_length', 'ep_conflict', 'ep_multi_engagement', 'ep_done'):
        G.assert_same_mask(s[k][0], z['st_' + k][t], f'{tag} {k}')
    G.assert_close(s['agent_values'][0], z['st_agent_values'][t], f'{tag} state')
    for k in ('p_dist', 'state_time', 'min_relative_distance', 'action_diff', 'times_required', 'dists_to_goal',
              'dist_left_to_goal', 'ep_travel_distance', 'ep_min_distance'):
        G.assert_close(s[k][0], z['st_' + k][t], f'{tag} {k}')
    G.assert_close(env.obs[0], z['obs'][t], f'{tag} obs')
    G.assert_close(env.node_obs[0], z['node_obs'][t], f'{tag} node_obs')
    G.assert_close(env.adj[0], z['adj'][t], f'{tag} adj')
    G.assert_close(env.reward[0], z['reward'][t], f'{tag} reward')


def rollout_with_tie_policy(make_env, z, meta, name, step_fn, max_ties=3):
    """Free-running rollout from the golden initial state.

    Threshold TIES: the action set is discrete, so double-integrator velocities live on a 0.05 lattice
    and e.g. the filter's `rel_v < 0.45` test (safety_filter.py:333-338) or `speed > 0.5` can sit exactly
    on a threshold, where the outcome is decided by the last-bit roundoff of scipy's RK45 in the reference.
    Policy (stated, counted, bounded): when a step mismatches, redo it (a) from the reference's own
    pre-step state, then (b) from that state with 1e-13 perturbations; if one of those reproduces the
    golden step the mismatch is a roundoff tie -> re-synchronise on the golden state and continue.
    Anything else is a real failure."""
    env = make_env()
    env.set_state(G.state0(z))
    ties = []
    rng = np.random.default_rng(0)
    for t in range(meta['T']):
        step_fn(env, z['actions'][t][None])
        try:
            check_step(env, z, t, name)
            continue
        except AssertionError as first:
            prev = G.state0(z) if t == 0 else G.state_at(z, t - 1)
            ok = False
            for k in range(17):
                pert = {kk: np.array(v) for kk, v in prev.items()}
                if k > 0:
                    pert['agent_values'] = pert['agent_values'] + rng.uniform(-1e-13, 1e-13, pert['agent_values'].shape)
                env.set_state(pert)
                step_fn(env, z['actions'][t][None])
                try:
                    check_step(env, z, t, name)
                    ok = True
                    break
                except AssertionError:
                    pass
            if not ok:
                raise first
            ties.append((t, str(first)[:120]))
            env.set_state(G.state_at(z, t))   # re-synchronise on the reference state
    assert len(ties) <= max_ties, f"{name}: too many roundoff ties {ties}"
    return env, ties


@pytest.mark.parametrize('name', CASES)
def test_rollout(name):
    z, meta, args, flags, params = G.load_case(name)
    env, ties = rollout_with_tie_policy(lambda: make_oracle(params), z, meta, name,
                                        lambda e, a: e.step(a, episode=meta['episode'], auto_reset=False))
    if ties:
        print(f"{name}: roundoff ties at {ties}")
    else:
        # episode summary reported by the next reset (environment.py:1046-1074)
        env.reset(episode=meta['episode'], sample=False)
        G.assert_close(env.ep_info[0], z['ep_info'], f'{name} ep_info')


@pytest.mark.parametrize('name', [c for c in CASES if c.startswith('at')])
def test_rollout_rotation_form(name):
    """The airtaxi relative position in its ROTATION form (what the specialised CUDA pipeline evaluates, selected in the
    oracle with set_relative_state_form(1)) reproduces the reference's golden rollouts under the same bar as the literal
    form of safety_filter.py:277-284 - discrete outputs included."""
    z, meta, args, flags, params = G.load_case(name)
    prev = O.set_relative_state_form(1)
    try:
        env, ties = rollout_with_tie_policy(lambda: make_oracle(params), z, meta, name,
                                            lambda e, a: e.step(a, episode=meta['episode'], auto_reset=False))
    finally:
        O.set_relative_state_form(prev)
    if ties:
        print(f"{name} (rotation form): roundoff ties at {ties}")


@pytest.mark.skipif(not G.have_reference('multiagent'), reason=G.REFERENCE_SKIP)
def test_golden_fixtures_are_reproducible_from_the_reference(tmp_path):
    """Regenerate a few fixtures from the original project with the committed generator (pure reference code, filter on, the declared
    obstacle extension, 3 landmarks per agent) and compare every array with the committed .npz, bit for bit."""
    import subprocess
    names = ['di3_nofilter_ep0', 'di8_filter', 'di3_obst2', 'at3_landmarks3']
    env = dict(os.environ, LSM_GOLDEN_OUT=str(tmp_path))
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call([sys.executable, os.path.join(repo, 'oracle', 'gen_golden.py')] + names, env=env, cwd=str(tmp_path),
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    for name in names:
        new = np.load(os.path.join(str(tmp_path), name + '.npz'))
        old = np.load(os.path.join(G.GOLDEN_DIR, name + '.npz'))
        assert sorted(new.files) == sorted(old.files), name
        for k in old.files:
            if k == 'meta':
                assert str(new[k]) == str(old[k]), f"{name} meta"
            else:
                assert np.array_equal(new[k], old[k], equal_nan=True), f"{name}: array '{k}' differs from the committed fixture"


def test_relative_state_forms_agree_on_a_batch():
    """Literal vs rotation form on 256 seeded airtaxi environments x 25 steps (BASELINE config 3 shape): every
    divergence in a discrete output is counted and printed; the continuous states agree to 1e-9."""
    args = G.default_args(dynamics_type='airtaxi', num_agents=10, use_safety_filter=True, episode_length=350, world_size=6)
    from layered_safe_marl_b200 import config as cfg
    flags = G.BinaryFlags(dict(POTENTIAL_CONFLICT=True))
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = G.value_grid_for(params)
    n, T, episode = 256, 25, 6249
    envs = [O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=2, nthreads=8) for _ in range(2)]
    rng = np.random.default_rng(9)
    acts = rng.integers(0, 25, (T, n, params.num_agents)).astype(np.int32)
    for form, env in enumerate(envs):
        prev = O.set_relative_state_form(form)
        try:
            env.reset(episode=episode, sample=True)
            for t in range(T):
                env.step(acts[t], episode=episode, auto_reset=True)
        finally:
            O.set_relative_state_form(prev)
    a, b = envs[0].get_state(), envs[1].get_state()
    diverged = np.zeros(n, dtype=bool)
    for k in ('reached_goal', 'done', 'safety_filtered', 'deconflicting_agent_index', 'num_agent_collisions'):
        diverged |= (np.asarray(a[k]) != np.asarray(b[k])).reshape(n, -1).any(axis=1)
    print(f"literal vs rotation form: {int(diverged.sum())} of {n} envs differ in a discrete output after {T} steps")
    assert diverged.sum() <= 2, "the two forms differ by ~1e-16: a divergence needs a state within roundoff of a threshold"
    ok = ~diverged
    G.assert_close(np.asarray(b['agent_values'])[ok], np.asarray(a['agent_values'])[ok], 'states', rtol=1e-9, atol=1e-12)
