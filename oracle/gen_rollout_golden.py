#!/usr/bin/env python
"""Golden fixture for SURVEY 8f row N1: runs the UNMODIFIED reference rollout path

    GMPERunner.insert        /root/reference/onpolicy/runner/shared/graph_mpe_runner.py:444-487
    GraphReplayBuffer        /root/reference/onpolicy/utils/graph_buffer.py:45-373 (insert, after_update, compute_returns)

on seeded inputs and records inputs + the buffer's resulting arrays in tests/golden/aux/rollout_buffer.npz. The reference
is imported from the checkout LSM_REFERENCE_PATH names (only here); gym comes from oracle/ref_stubs, the logging
packages the runner module imports at the top (tensorboardX, wandb, imageio) are empty stand-ins.

usage: LSM_REFERENCE_PATH=<checkout of the original project> python oracle/gen_rollout_golden.py
"""
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get('LSM_REFERENCE_PATH', '')
if not REF or not os.path.isdir(os.path.join(REF, 'onpolicy')):
    sys.exit("set LSM_REFERENCE_PATH to a checkout of the original project")
sys.path.insert(0, os.path.join(HERE, 'ref_stubs'))
sys.path.insert(0, REF)
for _name in ('tensorboardX', 'wandb', 'imageio'):
    _m = types.ModuleType(_name); _m.SummaryWriter = object; sys.modules.setdefault(_name, _m)

from onpolicy.utils.graph_buffer import GraphReplayBuffer          # noqa: E402
from onpolicy.runner.shared.graph_mpe_runner import GMPERunner     # noqa: E402


class Box:            # only .shape and the class name are read (get_shape_from_obs_space)
    def __init__(self, shape): self.shape = tuple(shape)


class Discrete:
    def __init__(self, n): self.n = n


def make(n, N, L, D, F, T, use_gae, proper, centralized, gamma=0.97, lam=0.9, hidden=8, recurrent_N=1):
    E = N * (1 + L)
    args = types.SimpleNamespace(episode_length=T, n_rollout_threads=n, hidden_size=hidden, recurrent_N=recurrent_N, gamma=gamma,
                                 gae_lambda=lam, use_gae=use_gae, use_popart=False, use_valuenorm=False,
                                 use_proper_time_limits=proper, use_centralized_V=centralized)
    buf = GraphReplayBuffer(args, N, Box((D,)), Box((D * N,)) if centralized else Box((D,)), Box((E, F)), Box((1,)), Box((N,)),
                            Box((E, E)), Discrete(25))
    runner = types.SimpleNamespace(recurrent_N=recurrent_N, hidden_size=hidden, n_rollout_threads=n, num_agents=N,
                                   use_centralized_V=centralized, buffer=buf)
    return args, buf, runner


def main():
    out = {}
    n, N, L, D, F, T = 5, 3, 2, 7, 10, 6
    E = N * (1 + L)
    rng = np.random.default_rng(2024)
    agent_id = np.tile(np.arange(N, dtype=np.int32).reshape(1, N, 1), (n, 1, 1))
    # one input stream (two passes over the buffer: after_update in between), shared by every variant
    steps = []
    for t in range(2 * T):
        dones = rng.random((n, N)) < 0.3
        if t in (2, 9):
            dones[1] = True                       # a whole env done: active_masks back to one
        steps.append(dict(obs=rng.normal(size=(n, N, D)).astype(np.float32), node_obs=rng.normal(size=(n, N, E, F)).astype(np.float32),
                          adj=rng.random(size=(n, N, E, E)).astype(np.float32), rewards=rng.normal(size=(n, N, 1)).astype(np.float32),
                          dones=dones, values=rng.normal(size=(n, N, 1)).astype(np.float32),
                          actions=rng.integers(0, 25, (n, N, 1)).astype(np.float32),
                          action_log_probs=rng.normal(size=(n, N, 1)).astype(np.float32),
                          rnn_states=rng.normal(size=(n, N, 1, 8)).astype(np.float32),
                          rnn_states_critic=rng.normal(size=(n, N, 1, 8)).astype(np.float32)))
    next_values = rng.normal(size=(2, n, N, 1)).astype(np.float32)
    bad_masks = (rng.random((T + 1, n, N, 1)) > 0.2).astype(np.float32)      # only the proper-time-limit variants read them
    obs0 = rng.normal(size=(n, N, D)).astype(np.float32)
    for k in steps[0]:
        out['in_' + k] = np.stack([s[k] for s in steps])
    out['in_next_values'] = next_values; out['in_bad_masks'] = bad_masks; out['in_obs0'] = obs0; out['in_agent_id'] = agent_id
    out['meta'] = np.array([n, N, L, D, F, T])
    for use_gae in (True, False):
        for proper in (False, True):
            for centralized in (True, False):
                tag = f"gae{int(use_gae)}_ptl{int(proper)}_cv{int(centralized)}"
                args, buf, runner = make(n, N, L, D, F, T, use_gae, proper, centralized)
                # warmup (graph_mpe_runner.py:253-300): slot 0
                share0 = np.expand_dims(obs0.reshape(n, -1), 1).repeat(N, axis=1) if centralized else obs0
                buf.share_obs[0] = share0.copy(); buf.obs[0] = obs0.copy(); buf.agent_id[0] = agent_id.copy()
                buf.share_agent_id[0] = (np.expand_dims(agent_id.reshape(n, -1), 1).repeat(N, axis=1) if centralized else agent_id).copy()
                buf.bad_masks[:] = bad_masks
                for p in range(2):
                    for t in range(T):
                        s = steps[p * T + t]
                        data = (s['obs'], agent_id, s['node_obs'], s['adj'], agent_id, s['rewards'], s['dones'], None, s['values'],
                                s['actions'], s['action_log_probs'], s['rnn_states'].copy(), s['rnn_states_critic'].copy())
                        GMPERunner.insert(runner, data)           # the reference's own method, unmodified
                    buf.compute_returns(next_values[p])
                    first = tag == 'gae1_ptl0_cv1'        # the env-produced arrays do not depend on the variant: kept once
                    names = ('share_obs', 'share_agent_id', 'value_preds', 'returns', 'masks', 'active_masks')
                    if first:
                        names += ('obs', 'node_obs', 'adj', 'agent_id', 'rnn_states', 'rnn_states_critic', 'actions',
                                  'action_log_probs', 'rewards')
                    for name in names:
                        out[f"{tag}_pass{p}_{name}"] = getattr(buf, name).copy()
                    buf.after_update()
                    for name in ('share_obs', 'obs', 'masks', 'active_masks', 'rnn_states'):
                        out[f"{tag}_pass{p}_after_{name}0"] = getattr(buf, name)[0].copy()
    os.makedirs(os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'aux'), exist_ok=True)
    path = os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'aux', 'rollout_buffer.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
