"""Device-resident rollout storage for the step path (SURVEY.md section 8f, row N1).

Mirrors the environment-facing half of the reference's host-side loop

    GMPERunner.warmup / insert      onpolicy/runner/shared/graph_mpe_runner.py:253-300, 444-487
    GraphReplayBuffer.__init__      onpolicy/utils/graph_buffer.py:45-166   (field names, shapes, dtypes)
    GraphReplayBuffer.insert        onpolicy/utils/graph_buffer.py:168-251
    GraphReplayBuffer.after_update  onpolicy/utils/graph_buffer.py:253-283
    GraphReplayBuffer.compute_returns (GAE / discounted sum, no value normaliser)   graph_buffer.py:285-373

but keeps every array in HBM, so one rollout step never crosses PCIe: the reference builds `masks`,
`active_masks`, `share_obs` and the one-hot actions with numpy on the host and copies every observation
array twice (np.stack in the vec-env, `.copy()` in the buffer).

With `zero_copy=True` the simulator's kernels write obs / node_obs / adj / rewards straight into the
buffer's slot for the next step (lsm_set_output_buffers re-binds the output pointers, no copy at all).

torch is used for storage and for the few elementwise mask operations; the learner (policy, GAE
consumers, minibatch generators) is out of scope.
"""
from __future__ import annotations

import torch


class DeviceGraphRolloutBuffer:
    def __init__(self, env, episode_length: int, use_centralized_V: bool = True, gamma: float = 0.99,
                 gae_lambda: float = 0.95, use_gae: bool = True, use_proper_time_limits: bool = False,
                 recurrent_N: int = 1, hidden_size: int = 64, zero_copy: bool = False):
        self.env = env
        self.episode_length = T = int(episode_length)
        self.n_rollout_threads = n = env.num_envs
        self.num_agents = N = env.N
        self.use_centralized_V = bool(use_centralized_V)
        self.gamma, self.gae_lambda = float(gamma), float(gae_lambda)
        self._use_gae, self._use_proper_time_limits = bool(use_gae), bool(use_proper_time_limits)
        self.recurrent_N, self.hidden_size = int(recurrent_N), int(hidden_size)
        self.zero_copy = bool(zero_copy)
        dev, f32 = env.device, torch.float32
        E, D, F = env.E, env.D, env.F
        so = D * N if self.use_centralized_V else D
        sa = N if self.use_centralized_V else 1
        self.share_obs = torch.zeros((T + 1, n, N, so), dtype=f32, device=dev)
        self.obs = torch.zeros((T + 1, n, N, D), dtype=f32, device=dev)
        self.node_obs = torch.zeros((T + 1, n, N, E, F), dtype=f32, device=dev)
        self.adj = torch.zeros((T + 1, n, N, E, E), dtype=f32, device=dev)
        self.agent_id = torch.zeros((T + 1, n, N, 1), dtype=torch.int32, device=dev)
        self.share_agent_id = torch.zeros((T + 1, n, N, sa), dtype=torch.int32, device=dev)
        self.rnn_states = torch.zeros((T + 1, n, N, self.recurrent_N, self.hidden_size), dtype=f32, device=dev)
        self.rnn_states_critic = torch.zeros_like(self.rnn_states)
        self.value_preds = torch.zeros((T + 1, n, N, 1), dtype=f32, device=dev)
        self.returns = torch.zeros_like(self.value_preds)
        self.available_actions = torch.ones((T + 1, n, N, env.action_space[0].n), dtype=f32, device=dev)
        self.actions = torch.zeros((T, n, N, 1), dtype=f32, device=dev)
        self.action_log_probs = torch.zeros((T, n, N, 1), dtype=f32, device=dev)
        self.rewards = torch.zeros((T, n, N, 1), dtype=f32, device=dev)
        self.masks = torch.ones((T + 1, n, N, 1), dtype=f32, device=dev)
        self.bad_masks = torch.ones_like(self.masks)
        self.active_masks = torch.ones_like(self.masks)
        self.step = 0
        # agent ids never change (scenario.get_id == agent index): every slot is filled once instead of on every insert
        self.agent_id.copy_(env.agent_id.view(1, n, N, 1).expand(T + 1, n, N, 1))
        if self.use_centralized_V:
            self.share_agent_id.copy_(env.agent_id.view(1, n, 1, N).expand(T + 1, n, N, N))
        else:
            self.share_agent_id.copy_(self.agent_id)
        # zero-copy: per-step reward / done landing zones the kernels write into
        self._done_u8 = torch.zeros((n, N), dtype=torch.uint8, device=dev)
        self._bound_slot = None

    # ------------------------------------------------------------------------------------------
    def _share(self, obs, agent_id):
        """(n, N, d) -> (n, N, N*d): every agent sees the concatenation (graph_mpe_runner.py:470-483)."""
        n, N = self.n_rollout_threads, self.num_agents
        if not self.use_centralized_V:
            return obs, agent_id
        so = obs.reshape(n, 1, -1).expand(n, N, obs.shape[-1] * N)
        sa = agent_id.reshape(n, 1, -1).expand(n, N, agent_id.shape[-1] * N)
        return so, sa

    def bind_next_slot(self):
        """zero-copy: point the simulator's outputs at slot step+1 (observations) / slot step (rewards)."""
        if not self.zero_copy:
            return
        s = self.step
        self.env.set_output_buffers(obs=self.obs[s + 1], node_obs=self.node_obs[s + 1], adj=self.adj[s + 1],
                                    reward=self.rewards[s].view(self.n_rollout_threads, self.num_agents),
                                    done=self._done_u8)
        self._bound_slot = s

    def warmup(self, reset_out=None, num_current_episode: int = 0):
        """GMPERunner.warmup (graph_mpe_runner.py:253-300): reset the envs, fill slot 0."""
        if self.zero_copy:
            self.env.set_output_buffers(obs=self.obs[0], node_obs=self.node_obs[0], adj=self.adj[0])
            reset_out = self.env.reset(num_current_episode)
        elif reset_out is None:
            reset_out = self.env.reset(num_current_episode)
        obs, agent_id, node_obs, adj = reset_out[:4]
        if not self.zero_copy:
            self.obs[0].copy_(obs); self.node_obs[0].copy_(node_obs); self.adj[0].copy_(adj)
        so, _ = self._share(self.obs[0], agent_id)
        self.share_obs[0].copy_(so)
        self.step = 0
        self.bind_next_slot()
        return reset_out

    def insert(self, step_out, values=None, actions=None, action_log_probs=None, rnn_states=None,
               rnn_states_critic=None):
        """GMPERunner.insert + GraphReplayBuffer.insert for one env.step result
        (obs, agent_id, node_obs, adj, rewards, dones, infos)."""
        obs, agent_id, node_obs, adj, rewards, dones = step_out[:6]
        s = self.step
        dones = dones.to(torch.bool)
        if rnn_states is not None:
            rnn_states = torch.where(dones[..., None, None], torch.zeros_like(rnn_states), rnn_states)
            self.rnn_states[s + 1].copy_(rnn_states)
        if rnn_states_critic is not None:
            rnn_states_critic = torch.where(dones[..., None, None], torch.zeros_like(rnn_states_critic), rnn_states_critic)
            self.rnn_states_critic[s + 1].copy_(rnn_states_critic)
        if self.zero_copy and self._bound_slot == s:
            # the step kernels already wrote obs / node_obs / adj / rewards / done in place: masks, active masks and the
            # centralised share_obs of slot s+1 in ONE launch (lsm_rollout_insert)
            import ctypes as C
            from . import _lib
            env = self.env
            so_ptr = C.c_void_p(self.share_obs[s + 1].data_ptr()) if self.use_centralized_V else None
            _lib.check(env.lib.lsm_rollout_insert(env._h, C.c_void_p(self.obs[s + 1].data_ptr()), C.c_void_p(self._done_u8.data_ptr()),
                                                  so_ptr, C.c_void_p(self.masks[s + 1].data_ptr()),
                                                  C.c_void_p(self.active_masks[s + 1].data_ptr()), env._stream()), 'lsm_rollout_insert', env.lib)
            if not self.use_centralized_V:
                self.share_obs[s + 1].copy_(self.obs[s + 1])
        else:
            dones_env = dones.all(dim=1)                                   # np.all(dones, axis=1)
            masks = (~dones).to(torch.float32).unsqueeze(-1)               # masks[dones] = 0
            active = masks.clone()
            active[dones_env] = 1.0                                        # active_masks[dones_env] = 1
            self.obs[s + 1].copy_(obs); self.node_obs[s + 1].copy_(node_obs); self.adj[s + 1].copy_(adj)
            self.rewards[s].copy_(rewards.reshape(self.n_rollout_threads, self.num_agents, 1))
            so, _ = self._share(self.obs[s + 1], agent_id)
            self.share_obs[s + 1].copy_(so)
            self.masks[s + 1].copy_(masks)
            self.active_masks[s + 1].copy_(active)
        if actions is not None:
            self.actions[s].copy_(actions.reshape(self.actions[s].shape))
        if action_log_probs is not None:
            self.action_log_probs[s].copy_(action_log_probs.reshape(self.action_log_probs[s].shape))
        if values is not None:
            self.value_preds[s].copy_(values.reshape(self.value_preds[s].shape))
        self.step = (s + 1) % self.episode_length
        self.bind_next_slot()

    def after_update(self):
        """Copy the last time step to index 0 (graph_buffer.py:253-283)."""
        for name in ('share_obs', 'obs', 'node_obs', 'adj', 'agent_id', 'share_agent_id', 'rnn_states',
                     'rnn_states_critic', 'masks', 'bad_masks', 'active_masks', 'available_actions'):
            t = getattr(self, name)
            t[0].copy_(t[-1])
        self.bind_next_slot()

    def compute_returns(self, next_value):
        """graph_buffer.py:285-373 without a value normaliser (popart / valuenorm belong to the learner)."""
        T = self.rewards.shape[0]
        if self._use_gae:
            self.value_preds[-1].copy_(next_value.reshape(self.value_preds[-1].shape))
            gae = torch.zeros_like(self.value_preds[0])
            for step in reversed(range(T)):
                delta = self.rewards[step] + self.gamma * self.value_preds[step + 1] * self.masks[step + 1] \
                    - self.value_preds[step]
                gae = delta + self.gamma * self.gae_lambda * self.masks[step + 1] * gae
                if self._use_proper_time_limits:
                    gae = gae * self.bad_masks[step + 1]
                self.returns[step] = gae + self.value_preds[step]
        else:
            self.returns[-1].copy_(next_value.reshape(self.returns[-1].shape))
            for step in reversed(range(T)):
                r = self.returns[step + 1] * self.gamma * self.masks[step + 1] + self.rewards[step]
                if self._use_proper_time_limits:
                    r = r * self.bad_masks[step + 1] + (1 - self.bad_masks[step + 1]) * self.value_preds[step]
                self.returns[step] = r

    def runner_view(self):
        """Adapter for an UNMODIFIED `GMPERunner.collect` (graph_mpe_runner.py:398-415), which evaluates
        `np.concatenate(self.buffer.<field>[step])` for nine fields to flatten (n, N, ...) into (n*N, ...). On the
        returned view that expression yields the reshaped DEVICE tensor (a view of the buffer, no host round trip);
        the reference policy passes tensors through `check()` unchanged (onpolicy/algorithms/utils/util.py:15-17)."""
        return _RunnerView(self)

    @staticmethod
    def one_hot_actions(actions, n_actions: int = 25):
        """np.eye(n)[actions] of GMPERunner.collect (graph_mpe_runner.py:431-433), on device. The simulator also
        accepts the integer indices directly, which skips this tensor altogether."""
        return torch.nn.functional.one_hot(actions.reshape(actions.shape[0], actions.shape[1]).long(), n_actions).to(torch.float32)


class _ConcatSlot:
    """`buffer.<field>[step]` of a runner view: np.concatenate(slot) -> tensor.reshape(n*N, ...) via NEP 18."""

    def __init__(self, tensor):
        self._t = tensor

    # np.concatenate's dispatcher iterates its first argument looking for objects that implement
    # __array_function__; one sentinel is enough and keeps the call O(1) in the number of environments
    def __len__(self):
        return 1

    def __iter__(self):
        yield self

    def __getitem__(self, k):
        if k == 0:
            return self
        raise IndexError(k)

    def __array_function__(self, func, types, args, kwargs):
        import numpy as np
        if func is np.concatenate and len(args) >= 1 and args[0] is self and not kwargs.get('axis'):
            t = self._t
            return t.reshape((t.shape[0] * t.shape[1],) + tuple(t.shape[2:]))
        return NotImplemented

    @property
    def tensor(self):
        return self._t


class _FieldView:
    def __init__(self, tensor):
        self._t = tensor

    def __getitem__(self, step):
        return _ConcatSlot(self._t[step])


class _RunnerView:
    _FIELDS = ('share_obs', 'obs', 'node_obs', 'adj', 'agent_id', 'share_agent_id', 'rnn_states', 'rnn_states_critic', 'masks',
               'available_actions', 'active_masks')

    def __init__(self, buf):
        self._buf = buf

    def __getattr__(self, name):
        if name in _RunnerView._FIELDS:
            return _FieldView(getattr(self._buf, name))
        return getattr(self._buf, name)
