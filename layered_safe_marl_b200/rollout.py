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

With `graph_storage='records'` (requires `zero_copy=True` and the specialised pipeline) the buffer keeps the graph
observation of every slot as the per-env emit records the step left behind (`records`, 1-7 % of the dense node_obs +
adj bytes) instead of node_obs / adj: the env writes its dense outputs into ONE scratch pair the acting forward reads,
and `graph_rows` / `graph_batch` re-emit any (step, env, agent) row on the GPU, bit for bit what the dense buffer holds
(lsm_copy_records / lsm_emit_from_records). The other fields, share_obs included, are stored as in the dense mode.

torch is used for storage and for the few elementwise mask operations; the learner (policy, GAE
consumers, minibatch generators) is out of scope.
"""
from __future__ import annotations

import numpy as np
import torch


class DeviceGraphRolloutBuffer:
    def __init__(self, env, episode_length: int, use_centralized_V: bool = True, gamma: float = 0.99,
                 gae_lambda: float = 0.95, use_gae: bool = True, use_proper_time_limits: bool = False,
                 recurrent_N: int = 1, hidden_size: int = 64, zero_copy: bool = False, graph_storage: str = 'dense'):
        self.env = env
        self.episode_length = T = int(episode_length)
        self.n_rollout_threads = n = env.num_envs
        self.num_agents = N = env.N
        self.use_centralized_V = bool(use_centralized_V)
        self.gamma, self.gae_lambda = float(gamma), float(gae_lambda)
        self._use_gae, self._use_proper_time_limits = bool(use_gae), bool(use_proper_time_limits)
        self.recurrent_N, self.hidden_size = int(recurrent_N), int(hidden_size)
        self.zero_copy = bool(zero_copy)
        if graph_storage not in ('dense', 'records'):
            raise ValueError(f"graph_storage must be 'dense' or 'records', got {graph_storage!r}")
        self.graph_storage = graph_storage
        dev, f32 = env.device, torch.float32
        E, D, F = env.E, env.D, env.F
        so = D * N if self.use_centralized_V else D
        sa = N if self.use_centralized_V else 1
        self.share_obs = torch.zeros((T + 1, n, N, so), dtype=f32, device=dev)
        self.obs = torch.zeros((T + 1, n, N, D), dtype=f32, device=dev)
        if graph_storage == 'records':
            if not self.zero_copy:
                raise ValueError("graph_storage='records' needs zero_copy=True: the records are those of the env's own step")
            R = env.record_bytes()
            if R == 0:
                raise ValueError("graph_storage='records' needs the specialised pipeline, and this shape runs the generic "
                                 "kernel (set args.specialise_shape to build a library for it)")
            self.records = torch.zeros((T + 1, n, R), dtype=torch.uint8, device=dev)
            self.node_obs = self.adj = None
            # the dense outputs of the current step only (what the acting forward reads)
            self._graph_scratch = (torch.zeros((n, N, E, F), dtype=f32, device=dev), torch.zeros((n, N, E, E), dtype=f32, device=dev))
        else:
            self.records = None
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
        node_obs, adj = self._graph_scratch if self.records is not None else (self.node_obs[s + 1], self.adj[s + 1])
        self.env.set_output_buffers(obs=self.obs[s + 1], node_obs=node_obs, adj=adj,
                                    reward=self.rewards[s].view(self.n_rollout_threads, self.num_agents),
                                    done=self._done_u8)
        self._bound_slot = s

    def warmup(self, reset_out=None, num_current_episode: int = 0):
        """GMPERunner.warmup (graph_mpe_runner.py:253-300): reset the envs, fill slot 0."""
        if self.zero_copy:
            node_obs, adj = self._graph_scratch if self.records is not None else (self.node_obs[0], self.adj[0])
            self.env.set_output_buffers(obs=self.obs[0], node_obs=node_obs, adj=adj)
            reset_out = self.env.reset(num_current_episode)
            if self.records is not None:
                self.env.copy_records(self.records[0])
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
            if self.records is not None:
                env.copy_records(self.records[s + 1])
        elif self.records is not None:
            raise RuntimeError("graph_storage='records' stores the env's own step: insert the output of the step that "
                               "followed warmup / the previous insert")
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
        for name in ('share_obs', 'obs', 'node_obs', 'adj', 'records', 'agent_id', 'share_agent_id', 'rnn_states',
                     'rnn_states_critic', 'masks', 'bad_masks', 'active_masks', 'available_actions'):
            t = getattr(self, name)
            if t is not None:
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

    def graph_rows(self, t, env, agent, node_obs=None, adj=None, edges: bool = False):
        """Graph observation rows (node_obs[t, env, agent], adj[t, env, agent]) for B index triples, t in [0, T]:
        -> ((B, E, F), (B, E, E)). Dense storage gathers them; records storage re-emits them on the GPU. Host (CPU tensor
        or numpy) indices out of range raise IndexError; out-of-range CUDA indices give zero rows in records storage.
        With edges=True the matrices come as the edge list the GNN builds from them instead:
        -> (node_obs (B, E, F), edge_index (2, nnz) int64, edge_attr (nnz, 1) float32), equal to process_adj(adj) of
        the rows; records storage computes it from the records without any dense matrix (one host sync to read nnz)."""
        if edges and adj is not None:
            raise ValueError("adj is not written with edges=True")
        T1, n = self.episode_length + 1, self.n_rollout_threads
        dev = self.env.device
        on_dev = all(torch.is_tensor(x) and x.is_cuda for x in (t, env, agent))
        if not on_dev:
            t, env, agent = (torch.as_tensor(np.asarray(x)).reshape(-1).to(torch.int64) for x in (t, env, agent))
            for x, bound, name in ((t, T1, 't'), (env, n, 'env'), (agent, self.num_agents, 'agent')):
                if x.numel() and (int(x.min()) < 0 or int(x.max()) >= bound):
                    raise IndexError(f"{name} out of range [0, {bound})")
            t, env, agent = t.to(dev), env.to(dev), agent.to(dev)
        t, env, agent = (x.reshape(-1).to(torch.int64) for x in (t, env, agent))
        if self.records is None:
            no, ad = self.node_obs[t, env, agent], self.adj[t, env, agent]
            if node_obs is not None:
                node_obs.copy_(no); no = node_obs
            if edges:
                return (no,) + process_adj(ad)
            if adj is not None:
                adj.copy_(ad); ad = adj
            return no, ad
        # an env index out of range must not alias another env's record: it becomes an invalid record
        ok = (t >= 0) & (t < T1) & (env >= 0) & (env < n)
        record = torch.where(ok, t * n + env, torch.full_like(t, -1))
        return self._emit(self.records, record, agent, node_obs, adj, edges)

    def graph_batch(self, rows, node_obs=None, adj=None, edges: bool = False):
        """Rows of the (T, n, N) flattening a minibatch generator indexes: equal to
        (node_obs[:-1].reshape(-1, E, F)[rows], adj[:-1].reshape(-1, E, E)[rows]) of the dense storage.
        With edges=True: (node_obs rows, *process_adj(adj rows)) - item b of the edge list is position b of `rows` -
        which records storage computes from the records without any dense matrix (one host sync to read nnz)."""
        if edges and adj is not None:
            raise ValueError("adj is not written with edges=True")
        T, n, N = self.episode_length, self.n_rollout_threads, self.num_agents
        if not (torch.is_tensor(rows) and rows.is_cuda):
            rows = torch.as_tensor(np.asarray(rows)).reshape(-1).to(torch.int64)
            if rows.numel() and (int(rows.min()) < 0 or int(rows.max()) >= T * n * N):
                raise IndexError(f"row out of range [0, {T * n * N})")
            rows = rows.to(self.env.device)
        rows = rows.reshape(-1).to(torch.int64)
        if self.records is None:
            E = self.env.E
            no = self.node_obs[:-1].reshape(-1, E, self.node_obs.shape[-1])[rows]
            ad = self.adj[:-1].reshape(-1, E, E)[rows]
            if node_obs is not None:
                node_obs.copy_(no); no = node_obs
            if edges:
                return (no,) + process_adj(ad)
            if adj is not None:
                adj.copy_(ad); ad = adj
            return no, ad
        # row r is record r // N of the first T slots (an out-of-range row: a record index outside them), observer r % N
        return self._emit(self.records[:-1], torch.div(rows, N, rounding_mode='floor'), rows % N, node_obs, adj, edges)

    def _emit(self, records, record, observer, node_obs, adj, edges):
        """Records storage: the rows' node_obs and adj, or node_obs and the edge list (lsm_emit_from_records without
        the matrices, then lsm_edges_from_records)."""
        if not edges:
            return self.env.emit_from_records(records, record, observer, node_obs, adj)
        no, _ = self.env.emit_from_records(records, record, observer, node_obs, dense_adj=False)
        return (no,) + self.env.edges_from_records(records, record, observer)

    def graph_nbytes(self) -> int:
        """Bytes of graph-observation storage: node_obs + adj (dense), or the records plus the one-step dense scratch
        pair (records). Every other field (share_obs, the largest of them) is the same in both modes."""
        if self.records is None:
            return self.node_obs.nbytes + self.adj.nbytes
        return self.records.nbytes + sum(x.nbytes for x in self._graph_scratch)

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


def process_adj(adj):
    """The reference's TransformerConvNet.process_adj (onpolicy/algorithms/utils/gnn.py:376-407) on a (B, E, E) batch:
    -> (edge_index (2, nnz) int64 = [b * E + row, b * E + col] of the non-zeros in row-major order, edge_attr (nnz, 1))."""
    nz = adj.nonzero()
    base = nz[:, 0] * adj.shape[1]
    return torch.stack([base + nz[:, 1], base + nz[:, 2]], dim=0), adj[nz[:, 0], nz[:, 1], nz[:, 2]].unsqueeze(1)


class _FieldView:
    def __init__(self, tensor):
        self._t = tensor

    def __getitem__(self, step):
        return _ConcatSlot(self._t[step])


class _ScratchFieldView:
    """node_obs / adj of a records-storage buffer: only the current step is held densely."""

    def __init__(self, buf, k):
        self._buf, self._k = buf, k

    def __getitem__(self, step):
        if step != self._buf.step:
            raise IndexError(f"graph_storage='records' holds node_obs / adj densely for the current step ({self._buf.step}) "
                             f"only, not step {step}: use graph_rows / graph_batch")
        return _ConcatSlot(self._buf._graph_scratch[self._k])


class _RunnerView:
    _FIELDS = ('share_obs', 'obs', 'node_obs', 'adj', 'agent_id', 'share_agent_id', 'rnn_states', 'rnn_states_critic', 'masks',
               'available_actions', 'active_masks')

    def __init__(self, buf):
        self._buf = buf

    def __getattr__(self, name):
        if name in ('node_obs', 'adj') and self._buf.records is not None:
            return _ScratchFieldView(self._buf, 0 if name == 'node_obs' else 1)
        if name in _RunnerView._FIELDS:
            return _FieldView(getattr(self._buf, name))
        return getattr(self._buf, name)
