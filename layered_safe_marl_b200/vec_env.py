"""B200GraphVecEnv - device-resident drop-in for the reference's vectorised graph environment.

Mirrors `GraphSubprocVecEnv` (reference onpolicy/envs/env_wrappers.py:951-1028) over
`GraphMPEEnv(args)` (multiagent/MPE_env.py:56-84): same constructor inputs (the argparse Namespace
`make_world` reads), same attributes (spaces), same `reset` / `step` / `step_async` / `step_wait`
signatures and return tuples

    reset(num_current_episode) -> (obs, agent_id, node_obs, adj, infos)
    step(actions, num_current_episode) -> (obs, agent_id, node_obs, adj, rewards, dones, infos)

for `num_envs` environments that live on one GPU. All arithmetic happens in the hand-written
sm_100a kernel behind the C ABI of include/lsm_b200.h; torch only provides device memory and the
CUDA stream. There is no CPU fallback.

Returned arrays are float32 CUDA tensors that alias the environment's output buffers: they stay
valid until the next `step`/`reset` (pass `copy=True` to get private clones, or `numpy_outputs=True`
to get host numpy arrays like the reference returns).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np
import torch

from . import _build, _lib
from . import layout as LY
from .config import (DYN_DOUBLE_INTEGRATOR, FLAG_SHARED_REWARD, FLAG_USE_SAFETY_FILTER, FLAG_HJ_VALUE,
                     RewardBinaryConfig, RewardWeightConfig, ScenarioParams, scenario_params_from_args)
from .hj_grid import HjGrid, synthetic_airtaxi_grid, synthetic_di_grid, synthetic_ttr_grid
from .infos import LazyInfos
from .spaces import Box, Discrete


def action_tables(dynamics: int):
    """np.linspace tables of MultiAgentBaseEnv._set_action (reference multiagent/environment.py:387-410)."""
    if dynamics == DYN_DOUBLE_INTEGRATOR:
        return np.linspace(-0.5, 0.5, 5), np.linspace(-0.5, 0.5, 5)
    return np.linspace(-0.1, 0.1, 5), np.linspace(-0.001, 0.002, 5)


def make_config_struct(p: ScenarioParams) -> _lib.LsmConfig:
    c = _lib.LsmConfig()
    for name, _ in _lib.LsmConfig._fields_:
        if name in ('_pad', 'act_tab0', 'act_tab1'):
            continue
        setattr(c, name, getattr(p, name))
    t0, t1 = action_tables(p.dynamics)
    c.act_tab0 = (C.c_double * 5)(*[float(v) for v in t0])
    c.act_tab1 = (C.c_double * 5)(*[float(v) for v in t1])
    return c


def _bind_to_gpu_numa_node(device) -> Optional[int]:
    """Pin this process (and the host worker threads it creates later) to the CPUs of the NUMA node the GPU hangs off, so
    that pinned staging buffers are allocated node-local (first touch) and the adjacency expander writes local memory.
    A no-op on single-node hosts / when sysfs has no answer. Returns the node or None."""
    try:
        bus = torch.cuda.get_device_properties(device).pci_bus_id if hasattr(torch.cuda.get_device_properties(device), 'pci_bus_id') else None
        if bus is None:
            import subprocess
            bus = subprocess.check_output(['nvidia-smi', '--query-gpu=pci.bus_id', '--format=csv,noheader', '-i',
                                           str(device.index)], text=True).strip()
        bus = bus.lower()
        if len(bus.split(':')[0]) == 8:
            bus = bus[4:]
        node = int(open(f'/sys/bus/pci/devices/{bus}/numa_node').read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            a, _, b = part.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


class _DeviceGrid:
    """An HjGrid uploaded to the GPU + its C descriptor."""

    def __init__(self, grid: HjGrid, device):
        self.values = torch.from_numpy(np.ascontiguousarray(grid.values, dtype=np.float32)).to(device)
        self.grads = None
        if grid.grads is not None:
            self.grads = torch.from_numpy(np.ascontiguousarray(grid.grads, dtype=np.float32)).to(device)
        d = _lib.LsmGridDesc()
        d.ndim = grid.ndim
        for k in range(grid.ndim):
            d.shape[k] = int(grid.shape[k])
            d.periodic[k] = int(bool(grid.periodic[k]))
            d.lo[k] = float(grid.lo[k])
            d.hi[k] = float(grid.hi[k])
        d.separation_distance = float(grid.separation_distance)
        d.ttr_max = float(grid.ttr_max)
        d.values = self.values.data_ptr()
        d.grads = self.grads.data_ptr() if self.grads is not None else None
        self.desc = d


class B200GraphVecEnv:
    def __init__(self, args, num_envs: Optional[int] = None, device='cuda:0', seed: int = 0,
                 value_grid: Optional[HjGrid] = None, ttr_grid: Optional[HjGrid] = None,
                 binary_cfg=RewardBinaryConfig, weight_cfg=RewardWeightConfig, env_id_base: int = 0,
                 numpy_outputs: bool = False, auto_reset: bool = True, tuning: Optional[dict] = None,
                 host_threads: Optional[int] = None, numa_bind: bool = False, host_chunks: Optional[int] = None,
                 host_cached_stores: Optional[bool] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("B200GraphVecEnv needs a CUDA device; there is no CPU fallback")
        self.lib = _lib.load()   # raises if the sm_100a library is missing
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        if numa_bind:
            _bind_to_gpu_numa_node(self.device)
        self._dev_ctx = torch.cuda.device(self.device)
        self._dev_ctx.__enter__()      # lsm_create adopts the current device; restored at the end of __init__
        try:
            self._init(args, num_envs, seed, value_grid, ttr_grid, binary_cfg, weight_cfg, env_id_base, numpy_outputs,
                       auto_reset, tuning, host_threads, host_chunks, host_cached_stores)
        finally:
            self._dev_ctx.__exit__(None, None, None)

    def _init(self, args, num_envs, seed, value_grid, ttr_grid, binary_cfg, weight_cfg, env_id_base, numpy_outputs,
              auto_reset, tuning, host_threads, host_chunks=None, host_cached_stores=None):
        self.params = scenario_params_from_args(args, binary_cfg=binary_cfg, weight_cfg=weight_cfg)
        p = self.params
        self.num_envs = int(num_envs if num_envs is not None else args.n_rollout_threads)
        self.n = self.num_envs
        self.num_agents = self.N = p.num_agents
        self.L = p.num_landmarks
        self.M = self.N * self.L
        self.O = p.num_obstacles          # declared extension (config.scenario_params_from_args); 0 in every shipped script
        self.E = self.N + self.M + self.O
        self.D = p.obs_dim
        self.F = p.node_feat_dim
        self.seed = int(seed)
        self.env_id_base = int(env_id_base)
        self.numpy_outputs = bool(numpy_outputs)
        self.auto_reset = bool(auto_reset)
        self._step_id = 0

        # --- spaces (environment.py:85-204, 928-960); only .shape / .n / class name are read by callers
        N, E = self.N, self.E
        self.action_space = [Discrete(LY.NUM_ACTIONS) for _ in range(N)]
        self.observation_space = [Box(-np.inf, np.inf, (self.D,)) for _ in range(N)]
        self.share_observation_space = [Box(-np.inf, np.inf, (self.D * N,)) for _ in range(N)]
        self.node_observation_space = [Box(-np.inf, np.inf, (E, self.F)) for _ in range(N)]
        self.adj_observation_space = [Box(-np.inf, np.inf, (E, E)) for _ in range(N)]
        self.edge_observation_space = [Box(-np.inf, np.inf, (1,)) for _ in range(N)]
        self.agent_id_observation_space = [Box(-np.inf, np.inf, (1,)) for _ in range(N)]
        self.share_agent_id_observation_space = [Box(-np.inf, np.inf, (N,)) for _ in range(N)]

        # --- handle
        cfg = make_config_struct(p)
        self._cfg = cfg
        self._h = C.c_void_p()
        self._check(self.lib.lsm_create(C.byref(cfg), C.byref(self._h)), 'lsm_create')
        if bool(getattr(args, 'specialise_shape', False)) and not os.environ.get('LSM_LIB') and \
                self.launch_info()['specialised'] == 0:
            # a shape the product library runs on the generic kernel: the library of exactly this shape (built by nvcc
            # on first use, _build.build_shape), which runs the specialised pipeline
            self.lib.lsm_destroy(self._h)
            self._h = C.c_void_p()
            self.lib = _lib.load(_build.build_shape(p.dynamics, N, self.L, self.O))
            self._check(self.lib.lsm_create(C.byref(cfg), C.byref(self._h)), 'lsm_create')
        if tuning:
            # launch-shape overrides (include/lsm_b200.h lsm_tuning): chunks, pair_placement, packed_grid, use_graph
            unknown = set(tuning) - {'chunks', 'pair_placement', 'packed_grid', 'use_graph'}
            if unknown:
                raise ValueError(f"unknown tuning keys {sorted(unknown)}")
            t = _lib.LsmTuning(int(tuning.get('chunks', 0)), int(tuning.get('pair_placement', -1)),
                               int(tuning.get('packed_grid', -1)), int(tuning.get('use_graph', -1)))
            self._check(self.lib.lsm_set_tuning(self._h, C.byref(t)), 'lsm_set_tuning')

        # --- grids (HjDataHandle / TTR loading); synthetic when none is given
        needs_vg = bool(p.flags & (FLAG_USE_SAFETY_FILTER | FLAG_HJ_VALUE))
        self.value_grid = None
        self.ttr_grid = None
        if needs_vg:
            if value_grid is None:
                value_grid = synthetic_di_grid() if p.dynamics == DYN_DOUBLE_INTEGRATOR else synthetic_airtaxi_grid()
            self.value_grid = _DeviceGrid(value_grid, self.device)
            self._check(self.lib.lsm_set_value_grid(self._h, C.byref(self.value_grid.desc)), 'lsm_set_value_grid')
        if p.dynamics != DYN_DOUBLE_INTEGRATOR:
            if ttr_grid is None:
                ttr_grid = synthetic_ttr_grid()
            self.ttr_grid = _DeviceGrid(ttr_grid, self.device)
            self._check(self.lib.lsm_set_ttr_grid(self._h, C.byref(self.ttr_grid.desc)), 'lsm_set_ttr_grid')

        # --- state + output buffers in HBM
        n, M = self.n, self.M
        dev = self.device
        f64, i32, f32 = torch.float64, torch.int32, torch.float32
        self.agent_f64 = torch.zeros((LY.AF_COUNT, n, N), dtype=f64, device=dev)
        for k in (LY.AF_EP_MIN_DIST, LY.AF_MIN_REL_DIST, LY.AF_GOAL_MIN_TIME):
            self.agent_f64[k].fill_(float('inf'))
        for k in (LY.AF_TIMES_REQ_A, LY.AF_TIMES_REQ_B, LY.AF_DISTS_GOAL_A, LY.AF_DISTS_GOAL_B, LY.AF_DIST_LEFT):
            self.agent_f64[k].fill_(-1.0)
        self.agent_i32 = torch.zeros((LY.AI_COUNT, n, N), dtype=i32, device=dev)
        self.agent_i32[LY.AI_DECONFLICT_IDX].fill_(-1)
        self.landmarks = torch.zeros((LY.LF_COUNT, n, M), dtype=f64, device=dev)
        self.obstacles = torch.zeros((2, n, self.O), dtype=f64, device=dev)
        self.env_f64 = torch.zeros((LY.EF_COUNT, n), dtype=f64, device=dev)
        self.env_i32 = torch.zeros((LY.EI_COUNT, n), dtype=i32, device=dev)
        self.obs = torch.zeros((n, N, self.D), dtype=f32, device=dev)
        self.node_obs = torch.zeros((n, N, E, self.F), dtype=f32, device=dev)
        self.adj = torch.zeros((n, N, E, E), dtype=f32, device=dev)
        self.reward = torch.zeros((n, N), dtype=f32, device=dev)
        self.done = torch.zeros((n, N), dtype=torch.uint8, device=dev)
        self.safe_action = torch.zeros((n, N, 2), dtype=f64, device=dev)
        self.ep_info = torch.zeros((n, LY.EP_COUNT), dtype=f64, device=dev)
        self.reward_individual = None
        if p.flags & FLAG_SHARED_REWARD:
            self.reward_individual = torch.zeros((n, N), dtype=f32, device=dev)
        # terminal-step snapshot of the info fields of auto-resetting envs (written only on a reset, read by LazyInfos)
        self.term_f64 = torch.zeros((LY.TF_COUNT, n, N), dtype=f64, device=dev)
        self.term_i32 = torch.zeros((LY.TI_COUNT, n, N), dtype=i32, device=dev)
        self.term_env_f64 = torch.zeros((n,), dtype=f64, device=dev)
        # agent ids are constant (scenario.get_id -> global_id == agent index)
        self.agent_id = torch.arange(N, dtype=torch.int32, device=dev).view(1, N, 1).expand(n, N, 1).contiguous()
        self._agent_id_np = None
        b = _lib.LsmBuffers()
        b.num_envs = n
        b.env_id_base = self.env_id_base
        for name in ('agent_f64', 'agent_i32', 'landmarks', 'env_f64', 'env_i32', 'obs', 'node_obs', 'adj',
                     'reward', 'done', 'safe_action', 'ep_info', 'term_f64', 'term_i32', 'term_env_f64'):
            setattr(b, name, getattr(self, name).data_ptr())
        b.reward_individual = self.reward_individual.data_ptr() if self.reward_individual is not None else None
        b.obstacles = self.obstacles.data_ptr() if self.O > 0 else None
        self._buffers = b
        self._check(self.lib.lsm_bind_buffers(self._h, C.byref(b)), 'lsm_bind_buffers')
        # pinned staging for host-side callers (the unmodified runner hands numpy one-hot actions)
        self._act_pinned = None
        self._act_dev = None
        self._pending_actions = None
        self._pending_episode = None
        self._host_out = None
        self.closed = False
        # host-facing path (numpy_outputs): the adjacency crosses PCIe as ONE thresholded E x E matrix per env + the
        # per-observer keep masks and is expanded on the host (lsm_set_compact_adjacency / lsm_expand_adjacency_host)
        self._compact = None
        # streaming (non-temporal) stores by default for the host-side adjacency expansion; ordinary stores were within the
        # run-to-run noise of the hosts measured (profiles/experiments/r02_e2e_probe_threads_chunks.txt)
        self.host_cached_stores = bool(host_cached_stores) if host_cached_stores is not None else False
        self.host_profile = None      # set to {} to accumulate wall-clock seconds of the host-side phases of _outputs
        if host_threads is None:
            local_world = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))
            try:
                cores = len(os.sched_getaffinity(0))
            except AttributeError:
                cores = os.cpu_count() or 1
            host_threads = max(1, min(16, cores // local_world))
        self.host_threads = int(host_threads)
        self.host_chunks = int(host_chunks) if host_chunks else 0
        if self.numpy_outputs and self.launch_info()['specialised'] == 1:
            Wm = (E + 31) // 32
            cpt = {'base': torch.zeros((n, E, E), dtype=f32, device=dev),
                   'keep': torch.zeros((n, N, Wm), dtype=i32, device=dev)}
            cpt['base_h'] = torch.empty((n, E, E), dtype=f32).pin_memory()
            cpt['keep_h'] = torch.empty((n, N, Wm), dtype=i32).pin_memory()
            cpt['adj_h'] = torch.zeros((n, N, E, E), dtype=f32)     # zero-fill = first touch of every page
            Fr = self.F
            cpt['obs_h'] = torch.zeros((n, N, self.D), dtype=f32).pin_memory()
            cpt['node_h'] = torch.zeros((n, N, E, Fr), dtype=f32).pin_memory()
            cpt['reward_h'] = torch.zeros((n, N), dtype=f32).pin_memory()
            cpt['done_h'] = torch.zeros((n, N), dtype=torch.uint8).pin_memory()
            self._check(self.lib.lsm_set_compact_adjacency(self._h, C.c_void_p(cpt['base'].data_ptr()),
                                                          C.c_void_p(cpt['keep'].data_ptr())), 'lsm_set_compact_adjacency')
            self._compact = cpt

    def _host_io(self, with_step: bool):
        cpt = self._compact
        io = _lib.LsmHostIo()
        io.obs = cpt['obs_h'].data_ptr(); io.node_obs = cpt['node_h'].data_ptr(); io.adj = cpt['adj_h'].data_ptr()
        io.reward = cpt['reward_h'].data_ptr() if with_step else None
        io.done = cpt['done_h'].data_ptr() if with_step else None
        io.adj_base_staging = cpt['base_h'].data_ptr(); io.adj_keep_staging = cpt['keep_h'].data_ptr()
        io.threads = self.host_threads; io.chunks = self.host_chunks; io.cached_stores = int(self.host_cached_stores)
        return io

    def _host_results(self, with_step: bool):
        cpt = self._compact
        if self._agent_id_np is None:
            self._agent_id_np = self.agent_id.cpu().numpy()
        node = cpt['node_h'].numpy()
        if node.shape != tuple(self.node_obs.shape):
            node = node.reshape(tuple(self.node_obs.shape))
        res = [cpt['obs_h'].numpy(), self._agent_id_np, node, cpt['adj_h'].numpy()]
        if with_step:
            res += [cpt['reward_h'].numpy(), cpt['done_h'].numpy().view(np.bool_)]
        return res

    def _check(self, rc: int, what: str):
        _lib.check(rc, what, self.lib)

    # ------------------------------------------------------------------------------------------
    def launch_info(self) -> dict:
        li = _lib.LsmLaunchInfo()
        self._check(self.lib.lsm_get_launch_info(self._h, C.byref(li)), 'lsm_get_launch_info')
        return {k: int(getattr(li, k)) for k, _ in _lib.LsmLaunchInfo._fields_}

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _stage_actions(self, actions):
        """-> (idx_ptr, onehot_ptr). Accepts (n,N) integer indices or (n,N,25) one-hot, torch or numpy."""
        n, N = self.n, self.N
        if isinstance(actions, np.ndarray) or not torch.is_tensor(actions):
            a = np.asarray(actions)
            if a.ndim == 3:
                a = np.ascontiguousarray(a, dtype=np.float32)
            else:
                a = np.ascontiguousarray(a, dtype=np.int32)
            tdt = torch.float32 if a.ndim == 3 else torch.int32
            if self._act_dev is None or tuple(self._act_dev.shape) != a.shape or self._act_dev.dtype != tdt:
                self._act_dev = torch.empty(a.shape, dtype=tdt, device=self.device)
                self._act_pinned = None
            src = torch.from_numpy(a) if (a.flags.writeable and self.numpy_outputs) else None
            if src is not None and src.is_pinned():
                # the caller's array already lives in page-locked memory: DMA straight from it. With numpy_outputs the
                # stream is synchronised before `step` returns, so the caller cannot overwrite it too early.
                self._act_dev.copy_(src, non_blocking=True)
                self._act_src_keepalive = src
            else:
                if self._act_pinned is None:
                    self._act_pinned = torch.empty(a.shape, dtype=self._act_dev.dtype).pin_memory()
                    self._act_evt = torch.cuda.Event()
                else:
                    self._act_evt.synchronize()      # the previous step's H2D copy has left the staging buffer
                self._act_pinned.numpy()[...] = a
                self._act_dev.copy_(self._act_pinned, non_blocking=True)
                self._act_evt.record(torch.cuda.current_stream(self.device))
            t = self._act_dev
        else:
            t = actions
            if t.device != self.device:
                t = t.to(self.device, non_blocking=True)
            if t.dim() == 3:
                if t.dtype != torch.float32:
                    t = t.to(torch.float32)
            elif t.dtype != torch.int32:
                t = t.to(torch.int32)
            t = t.contiguous()
        self._act_keepalive = t
        if t.dim() == 3:
            assert tuple(t.shape) == (n, N, LY.NUM_ACTIONS), f"one-hot actions must be {(n, N, LY.NUM_ACTIONS)}"
            return None, C.c_void_p(t.data_ptr())
        assert tuple(t.shape) == (n, N), f"action indices must be {(n, N)}"
        return C.c_void_p(t.data_ptr()), None

    def _outputs(self, with_step: bool, copy: bool):
        outs = [self.obs, self.agent_id, self.node_obs, self.adj]
        if not getattr(self, '_edge_dense', True) and not self.numpy_outputs:
            # edge output without the dense adjacency: nothing was written there
            res = [self.obs, self.agent_id, self.node_obs, None]
            if with_step:
                res += [self.reward, self.done.view(torch.bool)]
            return [t.clone() if (copy and t is not None) else t for t in res]
        if with_step:
            outs += [self.reward, self.done.view(torch.bool)]
        if self.numpy_outputs:
            # host arrays like the reference returns (float64 there; float32 here - every consumer casts).
            # Staged through pinned buffers that are reused every step: valid until the next step/reset.
            cpt = self._compact
            stream = torch.cuda.current_stream(self.device)
            if cpt is not None:
                # compact adjacency over PCIe, expanded by the library's host threads while the later ranges and node_obs
                # are still in flight (lsm_fetch_host); returns when every host array is complete
                io = self._host_io(with_step)
                self._check(self.lib.lsm_fetch_host(self._h, C.byref(io), self._stream()), 'lsm_fetch_host')
                return self._host_results(with_step)
            # generic-kernel configurations: dense adjacency straight into pinned buffers
            if self._host_out is None:
                self._host_out = {}
            res = []
            for t in outs:
                key = t.data_ptr()
                if t is self.agent_id:
                    if self._agent_id_np is None:
                        self._agent_id_np = t.cpu().numpy()
                    res.append(self._agent_id_np)
                    continue
                hb = self._host_out.get(key)
                if hb is None:
                    hb = torch.empty(t.shape, dtype=t.dtype, device='cpu').pin_memory()
                    self._host_out[key] = hb
                hb.copy_(t, non_blocking=True)
                res.append(hb)
            stream.synchronize()
            return [r if isinstance(r, np.ndarray) else r.numpy() for r in res]
        if copy:
            return [t.clone() for t in outs]
        return outs

    # ------------------------------------------------------------------------------------------
    def reset(self, num_current_episode: int = 0, copy: bool = False):
        """GraphSubprocVecEnv.reset (env_wrappers.py:998-1005): every env draws a new scenario."""
        self._step_id += 1
        self._check(self.lib.lsm_reset(self._h, None, int(num_current_episode), self.seed, 1, self._stream()),
                   'lsm_reset')
        obs, agent_id, node_obs, adj = self._outputs(False, copy)
        infos = LazyInfos(self, self._step_id, reset_only=True)
        return obs, agent_id, node_obs, adj, infos

    def reset_from_state(self, num_current_episode: int = 0):
        """reset bookkeeping + observation for the currently injected agents / landmarks (no sampling)."""
        self._step_id += 1
        self._check(self.lib.lsm_reset(self._h, None, int(num_current_episode), self.seed, 0, self._stream()),
                   'lsm_reset')
        return self._outputs(False, False)

    def observe(self):
        """Re-emit obs / node_obs / adj from the current state (after set_state)."""
        self._check(self.lib.lsm_observe(self._h, self._stream()), 'lsm_observe')
        return self._outputs(False, False)

    def emit_only(self):
        """Relaunch the graph-emission kernel alone (measurement hook; rewrites node_obs / adj with the same values)."""
        self._check(self.lib.lsm_emit_only(self._h, self._stream()), 'lsm_emit_only')

    def record_bytes(self) -> int:
        """emit_record_bytes of the handle (0 on the generic kernel); asked once, it is fixed per handle."""
        if getattr(self, '_rec_bytes', None) is None:
            self._rec_bytes = self.launch_info()['emit_record_bytes']
        return self._rec_bytes

    def copy_records(self, dst):
        """Copy the emit records of the last step / reset / observe into `dst`, a contiguous uint8 CUDA tensor of
        num_envs * emit_record_bytes bytes (lsm_copy_records; specialised pipeline only)."""
        assert dst.is_cuda and dst.dtype == torch.uint8 and dst.is_contiguous() and dst.numel() == self.n * self.record_bytes(), \
            "dst: contiguous uint8 CUDA tensor of the records' size"
        self._check(self.lib.lsm_copy_records(self._h, C.c_void_p(dst.data_ptr()), self._stream()), 'lsm_copy_records')

    def emit_from_records(self, records, record, observer, node_obs=None, adj=None, dense_adj: bool = True):
        """Re-emit graph observations from stored records (lsm_emit_from_records) on torch's current stream.

        records: uint8 CUDA tensor whose last dimension is emit_record_bytes (copy_records output, any leading shape);
        record / observer: B indices into the flattened records and the observing agent. CPU tensors or numpy arrays
        are range-checked here (IndexError); CUDA tensors go to the kernel unchecked, which zero-fills invalid items.
        -> (node_obs (B, E, F), adj (B, E, E)), written into the given tensors or into new ones. With dense_adj=False
        the matrices are not written and adj is None (edges_from_records gives their edge list)."""
        num_records, record, observer = self._record_items(records, record, observer, 'emit_from_records')
        B, E = record.numel(), self.E
        if node_obs is None:
            node_obs = torch.empty((B, E, self.F), dtype=torch.float32, device=self.device)
        if adj is None and dense_adj:
            adj = torch.empty((B, E, E), dtype=torch.float32, device=self.device)
        elif not dense_adj and adj is not None:
            raise ValueError("adj given with dense_adj=False")
        for t, shape, name in ((node_obs, (B, E, self.F), 'node_obs'), (adj, (B, E, E), 'adj')):
            assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and tuple(t.shape) == shape), \
                f"{name}: need a contiguous float32 CUDA tensor of shape {shape}"
        io = _lib.LsmRecordEmitIo(B, num_records, records.data_ptr(), record.data_ptr(), observer.data_ptr(),
                                  node_obs.data_ptr(), adj.data_ptr() if adj is not None else None)
        self._check(self.lib.lsm_emit_from_records(self._h, C.byref(io), self._stream()), 'lsm_emit_from_records')
        return node_obs, adj

    def edges_from_records(self, records, record, observer):
        """COO edge list of the matrices emit_from_records would write for the same items (lsm_edges_from_records),
        computed from the records without any dense matrix: -> (edge_index (2, nnz) int64, edge_attr (nnz, 1) float32),
        what the reference's TransformerConvNet.process_adj (gnn.py:376-407) returns for that (B, E, E) batch. Indices
        are handled as by emit_from_records; an invalid CUDA item has no edges. A counting pass, one host sync to read
        nnz, allocations of exactly nnz edges, then the fill pass."""
        num_records, record, observer = self._record_items(records, record, observer, 'edges_from_records')
        B = record.numel()
        counts = torch.empty((B,), dtype=torch.int32, device=self.device)
        offsets = torch.empty((B + 1,), dtype=torch.int64, device=self.device)
        io = _lib.LsmRecordEdgesIo(B, num_records, records.data_ptr(), record.data_ptr(), observer.data_ptr(),
                                   counts.data_ptr(), offsets.data_ptr(), None, None, 0)
        self._check(self.lib.lsm_edges_from_records(self._h, C.byref(io), self._stream()), 'lsm_edges_from_records')
        nnz = int(offsets[B].item())
        edge_index = torch.empty((2, nnz), dtype=torch.int64, device=self.device)
        edge_attr = torch.empty((nnz, 1), dtype=torch.float32, device=self.device)
        if nnz > 0:
            io.edge_index, io.edge_attr, io.capacity = edge_index.data_ptr(), edge_attr.data_ptr(), nnz
            self._check(self.lib.lsm_edges_from_records(self._h, C.byref(io), self._stream()), 'lsm_edges_from_records')
        return edge_index, edge_attr

    def _record_items(self, records, record, observer, what: str):
        """-> (num_records, record int64, observer int32) of a record store and its items, checked as documented in
        emit_from_records."""
        R = self.record_bytes()
        if R == 0:
            raise RuntimeError(f"{what} needs the specialised pipeline (this handle runs the generic kernel)")
        assert records.is_cuda and records.dtype == torch.uint8 and records.is_contiguous() and records.shape[-1] == R, \
            f"records: contiguous uint8 CUDA tensor with a last dimension of {R} bytes"
        num_records = records.numel() // R
        record, observer = self._item_index(record, num_records, torch.int64), self._item_index(observer, self.N, torch.int32)
        if record.shape != observer.shape:
            raise ValueError(f"record and observer must have the same shape, got {tuple(record.shape)} and {tuple(observer.shape)}")
        return num_records, record, observer

    def _item_index(self, idx, bound: int, dtype):
        """Index tensor for the kernel: host indices are checked against [0, bound); device indices are not."""
        if torch.is_tensor(idx) and idx.is_cuda:
            return idx.reshape(-1).to(dtype).contiguous()
        idx = torch.as_tensor(np.asarray(idx)).reshape(-1).to(torch.int64)
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= bound):
            raise IndexError(f"index out of range [0, {bound})")
        return idx.to(device=self.device, dtype=dtype)

    def debug_timeline(self, arm: bool = True):
        """Diagnostics: read the per-kernel %globaltimer timeline of the launches since the last arm (dict of ns relative
        to the first kernel's start, or None when nothing was armed), then re-arm / disarm."""
        out = (C.c_uint64 * 7)()
        had = getattr(self, '_tl_armed', False)
        self._check(self.lib.lsm_debug_timeline(self._h, int(bool(arm)), out if had else None), 'lsm_debug_timeline')
        self._tl_armed = bool(arm)
        if not had:
            return None
        names = ('pair_start', 'pair_body_end', 'agent_start', 'agent_end', 'emit_start', 'emit_end', 'pair_end')
        v = {k: int(out[j]) for j, k in enumerate(names)}
        starts = [v[k] for k in ('pair_start', 'agent_start', 'emit_start') if v[k] != 2 ** 64 - 1]
        t0 = min(starts) if starts else 0
        return {k: (None if x in (0, 2 ** 64 - 1) else (x - t0)) for k, x in v.items()}

    def step_async(self, actions, num_current_episode=None):
        self._pending_actions = actions
        self._pending_episode = num_current_episode

    def step_wait(self, copy: bool = False):
        actions, episode = self._pending_actions, self._pending_episode
        self._pending_actions = None
        ep = 0 if episode is None else int(episode)
        if self._compact is not None and not torch.is_tensor(actions):
            # host actions in, host arrays out: the whole step is ONE C-ABI call (lsm_step_host)
            a = np.asarray(actions)
            a = np.ascontiguousarray(a, dtype=np.float32 if a.ndim == 3 else np.int32)
            want = (self.n, self.N, LY.NUM_ACTIONS) if a.ndim == 3 else (self.n, self.N)
            assert a.shape == want, f"actions must be {(self.n, self.N)} indices or {(self.n, self.N, LY.NUM_ACTIONS)} one-hot"
            self._step_id += 1
            io = self._host_io(True)
            ptr = C.c_void_p(a.ctypes.data)
            self._check(self.lib.lsm_step_host(self._h, None if a.ndim == 3 else ptr, ptr if a.ndim == 3 else None, ep,
                                              self.seed, int(self.auto_reset), C.byref(io), self._stream()), 'lsm_step_host')
            obs, agent_id, node_obs, adj, rewards, dones = self._host_results(True)
            infos = LazyInfos(self, self._step_id, reset_only=False)
            return obs, agent_id, node_obs, adj, rewards, dones, infos
        idx_ptr, onehot_ptr = self._stage_actions(actions)
        self._step_id += 1
        self._check(self.lib.lsm_step(self._h, idx_ptr, onehot_ptr, ep, self.seed, int(self.auto_reset),
                                     self._stream()), 'lsm_step')
        obs, agent_id, node_obs, adj, rewards, dones = self._outputs(True, copy)
        infos = LazyInfos(self, self._step_id, reset_only=False)
        return obs, agent_id, node_obs, adj, rewards, dones, infos

    def step(self, actions, num_current_episode=None, copy: bool = False):
        """ShareVecEnv.step (env_wrappers.py:103-110)."""
        self.step_async(actions, num_current_episode)
        return self.step_wait(copy=copy)

    def close(self):
        if not self.closed and self._h:
            self.lib.lsm_destroy(self._h)
            self._h = C.c_void_p()
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------
    # named-state interchange (checkpoint / parity injection); leading axis = env
    def set_output_buffers(self, obs=None, node_obs=None, adj=None, reward=None, done=None):
        """Re-point the per-step outputs at caller-owned CUDA tensors (e.g. a rollout-buffer slot). The env keeps
        references so the memory stays alive; `step`/`reset` then return these tensors."""
        def chk(t, like, name):
            if t is None:
                return None
            assert t.is_cuda and t.is_contiguous() and t.dtype == like.dtype and tuple(t.shape) == tuple(like.shape), \
                f"{name}: need a contiguous {like.dtype} CUDA tensor of shape {tuple(like.shape)}"
            return t
        obs, node_obs, adj = chk(obs, self.obs, 'obs'), chk(node_obs, self.node_obs, 'node_obs'), chk(adj, self.adj, 'adj')
        reward, done = chk(reward, self.reward, 'reward'), chk(done, self.done, 'done')
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self.lib.lsm_set_output_buffers(self._h, ptr(obs), ptr(node_obs), ptr(adj), ptr(reward), ptr(done)),
                   'lsm_set_output_buffers')
        for name, t in (('obs', obs), ('node_obs', node_obs), ('adj', adj), ('reward', reward), ('done', done)):
            if t is not None:
                setattr(self, name, t)

    def edge_list(self, adj=None, capacity=None):
        """(edge_index (2, nnz) int64, edge_attr (nnz, 1) float32) of `adj` (default: the last step's adjacency) in
        the order of the reference's TransformerConvNet.process_adj (gnn.py:376-407) for the (num_envs*N, E, E)
        batch the runner feeds the policy - without materialising adj.nonzero(). One host sync (reads nnz)."""
        if adj is None and self._compact is not None:
            raise RuntimeError("numpy_outputs=True keeps the adjacency compact on the device; pass adj= explicitly")
        a = self.adj if adj is None else adj
        assert a.is_cuda and a.dtype == torch.float32 and a.is_contiguous() and a.numel() == self.n * self.N * self.E * self.E
        graphs = self.n * self.N
        cap = int(capacity) if capacity is not None else graphs * self.E * (self.E - 1)
        if getattr(self, '_edge_cap', 0) < cap:
            self._edge_index = torch.empty((2, cap), dtype=torch.int64, device=self.device)
            self._edge_attr = torch.empty((cap,), dtype=torch.float32, device=self.device)
            self._edge_counts = torch.empty((graphs,), dtype=torch.int32, device=self.device)
            self._edge_offsets = torch.empty((graphs + 1,), dtype=torch.int64, device=self.device)
            self._edge_cap = cap
        self._check(self.lib.lsm_edge_list(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(self._edge_index.data_ptr()),
                                          C.c_void_p(self._edge_attr.data_ptr()), C.c_void_p(self._edge_counts.data_ptr()),
                                          C.c_void_p(self._edge_offsets.data_ptr()), self._edge_cap, self._stream()),
                   'lsm_edge_list')
        nnz = int(self._edge_offsets[graphs].item())
        if nnz > self._edge_cap:
            raise RuntimeError(f"edge list needs {nnz} entries, capacity is {self._edge_cap}")
        return self._edge_index[:, :nnz], self._edge_attr[:nnz].unsqueeze(1)

    def enable_edge_output(self, capacity: Optional[int] = None, dense_adj: bool = True):
        """From now on every step / reset / observe also writes the COO edge list of its adjacency - the
        `(edge_index, edge_attr)` the reference's GNN derives with `process_adj` on every forward (gnn.py:376-407, 545-564)
        - straight from the emission kernel: no post-pass over the dense tensor, and with `dense_adj=False` the dense
        adjacency is not written at all (`step` then returns None in its place). No host synchronisation: read the result
        with `edges()` (syncs once to size the views) or use `edge_index` / `edge_attr` / `edge_offsets` directly
        (`edge_offsets[-1]` = nnz on the device). `capacity` defaults to the worst case N * E * (E - 1) per env."""
        graphs = self.n * self.N
        cap = int(capacity) if capacity is not None else graphs * self.E * (self.E - 1)
        self.edge_index = torch.zeros((2, cap), dtype=torch.int64, device=self.device)
        self.edge_attr = torch.zeros((cap,), dtype=torch.float32, device=self.device)
        self.edge_counts = torch.zeros((graphs,), dtype=torch.int32, device=self.device)
        self.edge_offsets = torch.zeros((graphs + 1,), dtype=torch.int64, device=self.device)
        self.edge_capacity = cap
        self._edge_dense = bool(dense_adj)
        with torch.cuda.device(self.device):
            self._check(self.lib.lsm_set_edge_output(self._h, C.c_void_p(self.edge_index.data_ptr()), C.c_void_p(self.edge_attr.data_ptr()),
                                                    C.c_void_p(self.edge_counts.data_ptr()), C.c_void_p(self.edge_offsets.data_ptr()),
                                                    cap, int(bool(dense_adj))), 'lsm_set_edge_output')

    def disable_edge_output(self):
        self._check(self.lib.lsm_set_edge_output(self._h, None, None, None, None, 0, 1), 'lsm_set_edge_output')
        self.edge_index = self.edge_attr = self.edge_counts = self.edge_offsets = None
        self._edge_dense = True

    def edges(self):
        """(edge_index (2, nnz) int64, edge_attr (nnz, 1) float32) of the last step, as `process_adj` would return them
        for the (num_envs * N, E, E) batch. One host sync (reads nnz to size the views)."""
        if getattr(self, 'edge_index', None) is None:
            raise RuntimeError("call enable_edge_output() first")
        nnz = int(self.edge_offsets[-1].item())
        if nnz > self.edge_capacity:
            raise RuntimeError(f"edge list needs {nnz} entries, capacity is {self.edge_capacity}")
        return self.edge_index[:, :nnz], self.edge_attr[:nnz].unsqueeze(1)

    def world_graph(self):
        """The renderer's per-environment graph (`world.edge_list`, `world.edge_weight` of SafeAamScenario.update_graph,
        navigation_graph_safe.py:996-1015; inclusive radius, disconnected entities removed) for the current state.
        -> (edge_list (2, nnz) int64 with entity indices, edge_weight (nnz,) float64, offsets (num_envs + 1,) int64):
        env e owns the columns offsets[e] : offsets[e + 1]. One host sync."""
        n, E = self.n, self.E
        cap = n * E * (E - 1)
        ei = torch.empty((2, cap), dtype=torch.int64, device=self.device)
        ew = torch.empty((cap,), dtype=torch.float64, device=self.device)
        cnt = torch.empty((n,), dtype=torch.int32, device=self.device)
        off = torch.empty((n + 1,), dtype=torch.int64, device=self.device)
        self._check(self.lib.lsm_world_graph(self._h, C.c_void_p(ei.data_ptr()), C.c_void_p(ew.data_ptr()), C.c_void_p(cnt.data_ptr()),
                                            C.c_void_p(off.data_ptr()), cap, self._stream()), 'lsm_world_graph')
        nnz = int(off[-1].item())
        return ei[:, :nnz], ew[:nnz], off

    def invalidate(self):
        """Call after writing the state tensors (agent_f64, agent_i32, env_f64, landmarks) directly."""
        self._check(self.lib.lsm_invalidate(self._h), 'lsm_invalidate')

    def set_state(self, s: dict):
        dev = self.device
        self.invalidate()

        def t(v, dtype):
            return torch.as_tensor(np.asarray(v), dtype=dtype, device=dev)

        f, i = self.agent_f64, self.agent_i32
        v = t(s['agent_values'], torch.float64)
        f[LY.AF_X].copy_(v[..., 0]); f[LY.AF_Y].copy_(v[..., 1]); f[LY.AF_S2].copy_(v[..., 2]); f[LY.AF_S3].copy_(v[..., 3])
        f[LY.AF_P_DIST].copy_(t(s['p_dist'], torch.float64)); f[LY.AF_STATE_TIME].copy_(t(s['state_time'], torch.float64))
        f[LY.AF_MIN_REL_DIST].copy_(t(s['min_relative_distance'], torch.float64))
        f[LY.AF_GOAL_MIN_TIME].copy_(t(s['goal_min_time'], torch.float64))
        tr = t(s['times_required'], torch.float64); dg = t(s['dists_to_goal'], torch.float64)
        f[LY.AF_TIMES_REQ_A].copy_(tr); f[LY.AF_TIMES_REQ_B].copy_(tr)
        f[LY.AF_DISTS_GOAL_A].copy_(dg); f[LY.AF_DISTS_GOAL_B].copy_(dg)
        f[LY.AF_DIST_LEFT].copy_(t(s['dist_left_to_goal'], torch.float64))
        f[LY.AF_EP_TRAVEL_DIST].copy_(t(s['ep_travel_distance'], torch.float64))
        f[LY.AF_EP_MIN_DIST].copy_(t(s['ep_min_distance'], torch.float64))
        f[LY.AF_ACTION_DIFF].copy_(t(s['action_diff'], torch.float64))
        i[LY.AI_REACHED].copy_(t(s['reached_goal'], torch.int32)); i[LY.AI_DONE].copy_(t(s['done'], torch.int32))
        i[LY.AI_SAFETY_FILTERED].copy_(t(s['safety_filtered'], torch.int32))
        i[LY.AI_DECONFLICT_IDX].copy_(t(s['deconflicting_agent_index'], torch.int32))
        i[LY.AI_NUM_COLLISIONS].copy_(t(s['num_agent_collisions'], torch.int32))
        i[LY.AI_EP_TRAVEL_LEN].copy_(t(s['ep_travel_length'], torch.int32))
        i[LY.AI_EP_CONFLICT].copy_(t(s['ep_conflict'], torch.int32))
        i[LY.AI_EP_MULTI].copy_(t(s['ep_multi_engagement'], torch.int32))
        i[LY.AI_EP_DONE].copy_(t(s['ep_done'], torch.int32))
        lp = t(s['landmark_pos'], torch.float64); lh = t(s['landmark_heading'], torch.float64)
        lm = self.landmarks
        lm[LY.LF_X].copy_(lp[..., 0]); lm[LY.LF_Y].copy_(lp[..., 1]); lm[LY.LF_HEADING].copy_(lh)
        lm[LY.LF_SPEED].copy_(t(s['landmark_speed'], torch.float64))
        # sin / cos of the landmark headings: the same float64 implementation (include/lsm_math.h) the on-device reset
        # sampler uses, evaluated on the host, so an injected state is bit-identical to a sampled one
        lh_np = np.ascontiguousarray(s['landmark_heading'], dtype=np.float64)
        lm[LY.LF_SIN].copy_(t(self.math_eval(0, lh_np), torch.float64)); lm[LY.LF_COS].copy_(t(self.math_eval(1, lh_np), torch.float64))
        self.env_f64[LY.EF_CURRICULUM_RATIO].copy_(t(s['curriculum_ratio'], torch.float64))
        self.env_i32[LY.EI_CURRENT_STEP].copy_(t(s['current_step'], torch.int32))
        if self.O > 0 and 'obstacle_pos' in s:      # a state without obstacle keys (e.g. eval_scenarios.build) keeps the current obstacles
            op = t(s['obstacle_pos'], torch.float64)
            self.obstacles[0].copy_(op[..., 0]); self.obstacles[1].copy_(op[..., 1])
            if 'num_obstacle_collisions' in s:
                i[LY.AI_NUM_OBST_COLLISIONS].copy_(t(s['num_obstacle_collisions'], torch.int32))

    def math_eval(self, op: int, a, b=None):
        """include/lsm_math.h on the host (op 0 sin, 1 cos, 2 atan2(a, b)): the kernels' own float64 trigonometry."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        out = np.empty_like(a)
        bp = None
        if b is not None:
            b = np.ascontiguousarray(b, dtype=np.float64)
            bp = b.ctypes.data_as(C.c_void_p)
        self._check(self.lib.lsm_math_eval(int(op), a.ctypes.data_as(C.c_void_p), bp, out.ctypes.data_as(C.c_void_p), a.size),
                   'lsm_math_eval')
        return out

    def get_state(self) -> dict:
        f = self.agent_f64.cpu().numpy(); i = self.agent_i32.cpu().numpy()
        lm = self.landmarks.cpu().numpy()
        ei = self.env_i32.cpu().numpy(); ef = self.env_f64.cpu().numpy()
        par = ei[LY.EI_PARITY][:, None].astype(bool)
        s = {}
        s['agent_values'] = np.stack([f[LY.AF_X], f[LY.AF_Y], f[LY.AF_S2], f[LY.AF_S3]], axis=-1)
        s['p_dist'] = f[LY.AF_P_DIST]; s['state_time'] = f[LY.AF_STATE_TIME]
        s['min_relative_distance'] = f[LY.AF_MIN_REL_DIST]; s['goal_min_time'] = f[LY.AF_GOAL_MIN_TIME]
        s['times_required'] = np.where(par, f[LY.AF_TIMES_REQ_B], f[LY.AF_TIMES_REQ_A])
        s['dists_to_goal'] = np.where(par, f[LY.AF_DISTS_GOAL_B], f[LY.AF_DISTS_GOAL_A])
        s['dist_left_to_goal'] = f[LY.AF_DIST_LEFT]
        s['ep_travel_distance'] = f[LY.AF_EP_TRAVEL_DIST]; s['ep_min_distance'] = f[LY.AF_EP_MIN_DIST]
        s['action_diff'] = f[LY.AF_ACTION_DIFF]
        s['reached_goal'] = i[LY.AI_REACHED]; s['done'] = i[LY.AI_DONE].astype(bool)
        s['safety_filtered'] = i[LY.AI_SAFETY_FILTERED].astype(bool)
        s['deconflicting_agent_index'] = i[LY.AI_DECONFLICT_IDX]
        s['num_agent_collisions'] = i[LY.AI_NUM_COLLISIONS].astype(np.float64)
        s['ep_travel_length'] = i[LY.AI_EP_TRAVEL_LEN].astype(np.float64)
        s['ep_conflict'] = i[LY.AI_EP_CONFLICT].astype(np.float64)
        s['ep_multi_engagement'] = i[LY.AI_EP_MULTI].astype(np.float64)
        s['ep_done'] = i[LY.AI_EP_DONE].astype(np.float64)
        s['landmark_pos'] = np.stack([lm[LY.LF_X], lm[LY.LF_Y]], axis=-1)
        s['landmark_heading'] = lm[LY.LF_HEADING]; s['landmark_speed'] = lm[LY.LF_SPEED]
        s['curriculum_ratio'] = ef[LY.EF_CURRICULUM_RATIO]; s['current_step'] = ei[LY.EI_CURRENT_STEP]
        if self.O > 0:
            ob = self.obstacles.cpu().numpy()
            s['obstacle_pos'] = np.stack([ob[0], ob[1]], axis=-1)
            s['num_obstacle_collisions'] = i[LY.AI_NUM_OBST_COLLISIONS].astype(np.float64)
        return s

    # ------------------------------------------------------------------------------------------
    def episode_stats(self, reduce_group=None) -> dict:
        """Mean of the last reported episode summaries over the envs of this shard; with
        `reduce_group` (True = default group, or a torch.distributed group) the mean over all shards
        (one NCCL all_reduce of 9 doubles - the only collective of this path)."""
        from .sharding import allreduce_episode_stats
        # column sums + env count in one launch of the library (lsm_episode_stats), then at most one all-reduce of 9 doubles
        sums = torch.empty((LY.EP_COUNT + 1,), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.lsm_episode_stats(self._h, C.c_void_p(sums.data_ptr()), self._stream()), 'lsm_episode_stats')
        if reduce_group is None:
            vals = (sums[:-1] / sums[-1]).cpu().numpy()
            return {k: float(vals[j]) for j, k in enumerate(LY.EP_INFO_KEYS)}
        return allreduce_episode_stats(self.ep_info, None if reduce_group is True else reduce_group, sums=sums)


class B200GraphDummyVecEnv(B200GraphVecEnv):
    """`GraphDummyVecEnv` surface (reference onpolicy/envs/env_wrappers.py:904-948): the in-process vec-env the
    reference uses for rendering / CSV evaluation (graph_mpe_runner.py:649-940). Differences from the
    subprocess variant, reproduced here: `step` returns an 8-tuple ending in `reset_count` (always 0) and
    environments are NOT auto-reset when all their agents are done."""

    def __init__(self, args, num_envs=None, **kw):
        kw['auto_reset'] = False
        super().__init__(args, num_envs=num_envs, **kw)

    def step_wait(self, copy: bool = False):
        out = super().step_wait(copy=copy)
        return (*out, 0)
