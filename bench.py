#!/usr/bin/env python
"""bench.py - throughput of the fused step kernel on BASELINE.json's headline configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg3|cfg4|cfg1]

A "step" is one `env.step` of every environment of the shard (BASELINE configs[1]: double
integrator, 8 agents, 2 landmarks per agent, HJ safety filter on with the synthetic value grid,
4096 environments per GPU). Prints ONE JSON line (rank 0).

  value     agent-steps/s, whole job, actions already resident in HBM, CUDA-event timed per step with
            an L2 flush between timed steps; max over ranks.
  e2e       the same metric through the public API the reference's runner calls
            (B200GraphVecEnv.step with HOST one-hot actions in pinned memory, every returned array
            copied back to pinned host memory) - host<->device copies inside the timed region.
  roofline  WHOLE STEP: algorithmic bytes of one env.step of the batch (SURVEY.md 8d) / mean event-timed step vs the
            measured HBM copy peak; `dominant_kernel` = lsm_emit_kernel timed alone on its 8d OUTPUT bytes.
  workloads the other BASELINE configs (cfg3, cfg4, cfg5) measured the same way, shorter (value, ms, whole-step frac).
  cpu_baseline   the C oracle (a port of the reference's Python path) on this box's host cores, bounded sample.
  timeline_us    diagnostics: device-side (%globaltimer) window of each kernel of one flushed step, us after the first
            block of the step (measured in a separate loop after the timed regions).

`--impl reference` times the CPU oracle port alone (the reference itself is Python and does not exist
on the GPU box); rank 0 only.

`--steps K` is the number of timed steps of the headline measurement (of every arm). `--dump-outputs DIR` writes, after
the timed steps, what the last timed step returned to its caller as DIR/<name>.npy (see dump_outputs); the inputs are
seeded, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from as it found it
REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))

import numpy as np  # noqa: E402

METRIC = "agent-steps/sec (graph obs + HJ filter on)"
UNIT = "agent-steps/s"

WORKLOADS = {
    # name: (args overrides, RewardBinaryConfig switches, envs per GPU, episode index)
    'cfg2': (dict(dynamics_type='double_integrator', num_agents=8, num_landmarks=2, use_safety_filter=True,
                  world_size=4, episode_length=250), {}, 4096, 6249),
    'cfg3': (dict(dynamics_type='airtaxi', num_agents=10, num_landmarks=2, use_safety_filter=True,
                  world_size=6, episode_length=350), dict(POTENTIAL_CONFLICT=True), 16384, 6249),
    'cfg4': (dict(dynamics_type='double_integrator', num_agents=32, num_landmarks=2, use_safety_filter=True,
                  world_size=4, episode_length=250), {}, 8192, 6249),
    'cfg1': (dict(dynamics_type='double_integrator', num_agents=3, num_landmarks=2, use_safety_filter=False,
                  world_size=4, episode_length=25), {}, 4096, 0),
    # BASELINE configs[2] WITH its obstacles: the declared obstacle extension (the reference raises for obstacles)
    'cfg3_obst4': (dict(dynamics_type='airtaxi', num_agents=10, num_landmarks=2, use_safety_filter=True, world_size=6,
                        episode_length=350, num_obstacles=4, obstacle_extension=True), dict(POTENTIAL_CONFLICT=True), 16384, 6249),
}
WORKLOAD_DESC = {
    'cfg2': "BASELINE configs[1]: double integrator (crazyflie) 8 agents, HJ safety filter on (synthetic value grid "
            "41x41x21x21), 4096 parallel envs per B200",
    'cfg3': "BASELINE configs[2] (obstacle-free): airtaxi 10 agents, POTENTIAL_CONFLICT reward, filter on, 16384 envs per B200",
    'cfg4': "BASELINE configs[3]: dense 32 agents, 8192 envs per B200",
    'cfg1': "BASELINE configs[0] shape: double integrator 3 agents, filter off, 4096 envs per B200",
    'cfg3_obst4': "BASELINE configs[2] with 4 obstacles (declared extension, not reference-pinned: the reference raises for "
                  "obstacles): airtaxi 10 agents + 4 obstacles, POTENTIAL_CONFLICT, filter on, 16384 envs per B200",
}


def algorithmic_bytes_per_env_step(N, L, D, F, O=0):
    """SURVEY.md 8(d): fp32 outputs + fp64 state read/write + flags + action index (O obstacles: extension only)."""
    E = N * (1 + L) + O
    return 4 * N * (E * F + E * E + D + 2) + 77 * N


def measured_peak():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


DUMP_BYTES = 64 * 1000 * 1000     # upper bound of the files --dump-outputs writes, headers included


def dump_outputs(out_dir, arrays, seed=0):
    """`--dump-outputs`: save {name: array with the environments on axis 0} (torch or numpy) as <out_dir>/<name>.npy,
    float64 arrays as float64 and everything else (float32 observations, int agent ids, bool / uint8 dones) as float32.
    When the whole batch would exceed DUMP_BYTES, every array keeps the same fixed sample of environments: the sorted
    indices of a default_rng(seed) draw without replacement, as many as fit."""
    import torch
    arrays = {k: (v if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()}
    wide = {k: v.dtype in (torch.float64, np.float64) for k, v in arrays.items()}
    n = int(next(iter(arrays.values())).shape[0])
    per_env = sum(int(np.prod(v.shape[1:])) * (8 if wide[k] else 4) for k, v in arrays.items())
    keep = min(n, (DUMP_BYTES - 1024 * len(arrays)) // per_env)
    idx = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False)) if keep < n else None
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        if idx is not None:       # sample before the copy: a whole cfg4 adjacency is 9.7 GB
            v = v[torch.as_tensor(idx, device=v.device)] if torch.is_tensor(v) else v[idx]
        a = v.detach().cpu().numpy() if torch.is_tensor(v) else v
        np.save(os.path.join(out_dir, k + '.npy'), np.ascontiguousarray(a, dtype=np.float64 if wide[k] else np.float32))
    return {"dir": out_dir, "envs": int(keep), "of_envs": n, "arrays": sorted(arrays)}


class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                                          '-lms', '20', '-i', str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ''
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in out.strip().splitlines():
            parts = [x.strip() for x in line.split(',')]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_args(workload):
    import _golden as G
    kw, flags, n_envs, episode = WORKLOADS[workload]
    return G.default_args(**kw), G.BinaryFlags(flags), n_envs, episode


def oracle_throughput(workload, n_envs, steps, warmup, nthreads, seed=0):
    """Time the C oracle port (reference algorithm on CPU) on a bounded sample."""
    import _golden as G
    sys.path.insert(0, os.path.join(REPO, 'oracle'))
    import oracle_env as O
    from layered_safe_marl_b200 import config as cfg
    args, flags, _, episode = build_args(workload)
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = G.value_grid_for(params)
    env = O.OracleEnv(params.asdict(), n_envs, value_grid=vg, ttr_grid=tg, seed=seed, nthreads=nthreads)
    env.reset(episode=episode, sample=True)
    rng = np.random.default_rng(1234)
    acts = rng.integers(0, 25, (warmup + steps, n_envs, params.num_agents)).astype(np.int32)
    for t in range(warmup):
        env.step(acts[t], episode=episode, auto_reset=True)
    t0 = time.perf_counter()
    for t in range(warmup, warmup + steps):
        env.step(acts[t], episode=episode, auto_reset=True)
    dt = time.perf_counter() - t0
    return n_envs * params.num_agents * steps / dt, dt, params, env


def run_reference(a):
    """`--impl reference`: the CPU oracle port with every host thread; rank 0 only. The timed loop runs --steps steps
    (a 0.05 s sample moves by +-20 %: ask for a few seconds' worth)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_sample = 1024
    steps_run = a.steps
    val, dt, params, ora = oracle_throughput(a.workload, n_sample, steps_run, a.warmup, cores)
    if a.dump_outputs:
        info = dump_outputs(a.dump_outputs, dict(obs=ora.obs, node_obs=ora.node_obs, adj=ora.adj, rewards=ora.reward,
                                                 dones=ora.done))
        print(f"outputs of the last timed step: {info}", file=sys.stderr, flush=True)
    sample = (f"{n_sample} envs x {steps_run} steps ({dt:.1f} s) of {a.workload} on {cores} host threads "
              f"(C oracle port of the reference's Python path)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "steps_run": steps_run, "warmup": a.warmup, "ms_per_step": 1000.0 * dt / steps_run, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD_DESC[a.workload], "sample_envs": n_sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def measure_brief(workload, device, rank, world, steps, warmup, flush):
    """One of the other BASELINE configs, measured like the headline one (flushed CUDA-event timing per step, max over
    ranks) but shorter: -> {value, ms_per_step, ms_per_step_back_to_back, whole_step_frac, ...}."""
    import torch
    import torch.distributed as dist
    from layered_safe_marl_b200 import B200GraphVecEnv
    args, flags, n_envs, episode = build_args(workload)
    env = B200GraphVecEnv(args, num_envs=n_envs, device=device, seed=1234, binary_cfg=flags, env_id_base=rank * n_envs)
    N = env.N
    gen = torch.Generator(device=device); gen.manual_seed(77 + rank)
    actions = torch.randint(0, 25, (warmup + steps, n_envs, N), generator=gen, device=device, dtype=torch.int32)
    env.reset(episode)
    for t in range(warmup):
        env.step(actions[t], episode)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for t in range(steps):
        flush.fill_(0.0)
        starts[t].record(); env.step(actions[warmup + t], episode); stops[t].record()
    torch.cuda.synchronize()
    total_ms = float(sum(s.elapsed_time(e) for s, e in zip(starts, stops)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps):
        env.step(actions[warmup + t], episode)
    e1.record(); torch.cuda.synchronize()
    b2b_ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([total_ms, b2b_ms], dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms, b2b_ms = float(tt[0]), float(tt[1])
    peak, _ = measured_peak()
    bytes_per_step = algorithmic_bytes_per_env_step(N, env.L, env.D, env.F, env.O) * n_envs
    li = env.launch_info()
    out = {"workload": WORKLOAD_DESC[workload], "envs_per_gpu": n_envs, "num_agents": N, "steps": steps,
           "value": n_envs * world * N * steps / (total_ms / 1000.0), "unit": UNIT, "ms_per_step": total_ms / steps,
           "ms_per_step_back_to_back": b2b_ms / steps, "algorithmic_bytes_per_step": bytes_per_step,
           "whole_step_frac": bytes_per_step / (total_ms / steps / 1000.0) / 1e9 / peak,
           "launches_per_step": li.get('launches_per_step', 1), "chunks": li.get('chunks', 1)}
    env.close()
    del env, actions
    torch.cuda.empty_cache()
    return out


def run_ours(a):
    import torch
    import torch.distributed as dist
    from layered_safe_marl_b200 import B200GraphVecEnv

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local_rank}'))
    device = torch.device(f'cuda:{local_rank}')
    torch.cuda.set_device(device)

    args, flags, n_envs, episode = build_args(a.workload)
    if a.envs:
        n_envs = a.envs
    env = B200GraphVecEnv(args, num_envs=n_envs, device=device, seed=1234, binary_cfg=flags,
                          env_id_base=rank * n_envs, tuning=dict(use_graph=a.use_graph))
    N, L, D, F = env.N, env.L, env.D, env.F
    K, W = a.steps, a.warmup
    gen = torch.Generator(device=device); gen.manual_seed(1234 + rank)
    actions = torch.randint(0, 25, (W + K, n_envs, N), generator=gen, device=device, dtype=torch.int32)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)   # 256 MiB > 126 MB L2
    # --use-graph 1 only: the step reads its actions from ONE device buffer (as a policy loop with a static output tensor
    # would leave them) - with unchanged pointers the library replays the step's launches from a CUDA graph
    act = torch.empty((n_envs, N), dtype=torch.int32, device=device) if a.use_graph == 1 else None

    def step_actions(t):
        if act is None:
            return actions[t]
        act.copy_(actions[t])
        return act

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()      # sampled every 20 ms over warm-up + timed loops + e2e (the GPU is busy throughout)
    env.reset(episode)
    for t in range(W):
        env.step(step_actions(t), episode)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    torch.cuda.synchronize()
    # Every timed step is bracketed by its own pair of events, so a host hiccup between "start recorded" and "kernels
    # enqueued" would be billed to the device. Keep the host out of the measurement: no garbage collection inside the
    # loop, and an untimed lead-in (a few more L2 flushes, ~1 ms of GPU work) so that the launches of the first timed
    # steps are already queued when the GPU reaches them - as they are for every later step, the host being ~2.5 x
    # faster per iteration than the GPU.
    gc.collect(); gc.disable()
    for _ in range(12):
        flush.fill_(0.0)
    t_wall0 = time.perf_counter()
    for t in range(K):
        x = step_actions(W + t)               # this step's actions (not timed: resident in HBM when the step starts)
        flush.fill_(0.0)                      # L2 flush between timed iterations (not timed)
        starts[t].record()
        last = env.step(x, episode)           # agent -> emit -> pair kernels (launch_info.launches_per_step)
        stops[t].record()
    torch.cuda.synchronize()
    gc.enable()
    t_wall = time.perf_counter() - t_wall0
    if a.dump_outputs and rank == 0:
        # the returned tensors alias the env's output buffers: save them before any later step overwrites them
        obs, agent_id, node_obs, adj, rewards, dones, _ = last
        info = dump_outputs(a.dump_outputs, dict(obs=obs, agent_id=agent_id, node_obs=node_obs, adj=adj, rewards=rewards,
                                                 dones=dones))
        print(f"outputs of the last timed step: {info}", file=sys.stderr, flush=True)
    step_ms = np.array([s.elapsed_time(e) for s, e in zip(starts, stops)])
    total_ms = float(step_ms.sum())
    if os.environ.get('LSM_BENCH_DUMP'):
        print(f"[rank {rank}] per-step us: " + ' '.join(f"{v * 1e3:.1f}" for v in step_ms), file=sys.stderr, flush=True)
    # back-to-back (no flush) timing for reference
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(K):
        env.step(step_actions(W + t), episode)
    e1.record()
    torch.cuda.synchronize()
    noflush_ms = e0.elapsed_time(e1)
    # no flush, but the big outputs rotate over slots whose total size exceeds L2 (what a rollout buffer does: every step
    # writes node_obs / adj into the next slot), so they are never L2 resident while the few-MB state stays warm
    slot_bytes = (env.node_obs.numel() + env.adj.numel()) * 4
    n_slots = max(2, int(np.ceil(2.5 * 126e6 / slot_bytes)))
    rot_ms = None
    if slot_bytes * n_slots < 40e9:
        slots = [(torch.empty_like(env.node_obs), torch.empty_like(env.adj)) for _ in range(n_slots)]
        for t in range(min(W, 5)):
            env.set_output_buffers(node_obs=slots[t % n_slots][0], adj=slots[t % n_slots][1])
            env.step(actions[t], episode)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for t in range(K):
            env.set_output_buffers(node_obs=slots[t % n_slots][0], adj=slots[t % n_slots][1])
            env.step(actions[W + t], episode)
        r1.record()
        torch.cuda.synchronize()
        rot_ms = r0.elapsed_time(r1)
        del slots
    # the dominant kernel alone (graph emission: >= 96 % of the algorithmic bytes), same flush between launches
    li0 = env.launch_info()
    emit_ms = None
    if li0.get('specialised', 0):
        es = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        ee = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        for t in range(K):
            flush.fill_(0.0)
            es[t].record()
            env.emit_only()
            ee[t].record()
        torch.cuda.synchronize()
        emit_ms = float(np.mean([s.elapsed_time(e) for s, e in zip(es, ee)]))
    # device-side timeline of one step (diagnostics, outside every timed region): %globaltimer first-block-in /
    # last-block-out of each kernel, median over a few flushed steps
    timeline = None
    if li0.get('specialised', 0) and rank == 0:
        rows = []
        env.debug_timeline(True)
        for t in range(min(K, 15)):
            flush.fill_(0.0)
            env.step(actions[W + t], episode)
            rows.append(env.debug_timeline(True))
        env.debug_timeline(False)
        timeline = {k: (round(float(np.median([r[k] for r in rows if r[k] is not None])) / 1000.0, 2)
                        if any(r[k] is not None for r in rows) else None) for k in rows[0]}
    if world > 1:
        tt = torch.tensor([total_ms, noflush_ms], dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms, noflush_ms = float(tt[0]), float(tt[1])
        stats = env.episode_stats(reduce_group=True)   # the only collective of this path: episode statistics
    else:
        stats = env.episode_stats()
    total_envs = n_envs * world
    value = total_envs * N * K / (total_ms / 1000.0)

    # ---- e2e: host one-hot actions in, every returned array back to pinned host memory --------------
    Ke = max(3, a.e2e_steps)        # its own step count (reported as e2e.steps): 20 steps moved by +-15 % from run to run
    We = 5
    env_h = B200GraphVecEnv(args, num_envs=n_envs, device=device, seed=4321, binary_cfg=flags,
                            env_id_base=rank * n_envs, numpy_outputs=True, numa_bind=a.numa_bind)
    env_h.reset(episode)
    rng = np.random.default_rng(99 + rank)
    onehot_host = torch.from_numpy(np.eye(25, dtype=np.float32)[rng.integers(0, 25, (min(Ke + We, 16), n_envs, N))]).pin_memory()   # a pool of distinct action sets, cycled
    pool = onehot_host.shape[0]
    for t in range(We):
        env_h.step(onehot_host[t % pool].numpy(), episode)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    chk = 0.0
    for t in range(Ke):
        out = env_h.step(onehot_host[(We + t) % pool].numpy(), episode)
        chk += float(out[4][0, 0])            # touch the host result
    s1.record()
    torch.cuda.synchronize()
    e2e_ms = s0.elapsed_time(s1)
    if world > 1:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt[0])
    e2e_value = total_envs * N * Ke / (e2e_ms / 1000.0)
    clocks = sampler.stop() if rank == 0 else None
    h2d = n_envs * N * 25 * 4
    dense_adj_bytes = n_envs * N * env.E * env.E * 4
    small = n_envs * (N * D * 4 + N * env.E * F * 4 + N * 4 + N)          # obs, node_obs, rewards, dones
    compact = env_h._compact is not None
    if compact:
        # the adjacency crosses PCIe as one thresholded E x E matrix per env + per-observer keep masks
        d2h = small + n_envs * (env.E * env.E * 4 + N * ((env.E + 31) // 32) * 4)
    else:
        d2h = small + dense_adj_bytes
    e2e_host = {"adjacency": ("compact over PCIe (1 E x E matrix + N keep masks per env) in env ranges, each range expanded to the dense "
                              f"(n,N,E,E) float32 array by {env_h.host_threads} host threads as it lands, while "
                              "the DMA engine moves the later ranges and node_obs; the whole step is one C-ABI call (lsm_step_host)")
                             if compact else "dense over PCIe",
                "host_bytes_written_per_step": d2h + (dense_adj_bytes if compact else 0),
                "host_threads": env_h.host_threads,
                "host_stores": "ordinary" if env_h.host_cached_stores else "streaming"}
    env_h.close()
    del env_h

    # ---- the other BASELINE configs, same method, shorter (every rank takes part: max over ranks inside) -------------
    extra = None
    if a.workload == 'cfg2' and not a.no_extra_workloads:
        extra = {}
        env.close()
        torch.cuda.empty_cache()
        for w, ks in (('cfg3', 40), ('cfg3_obst4', 40), ('cfg4', 20)):
            extra[w] = measure_brief(w, device, rank, world, ks, 5, flush)
        extra['cfg5'] = measure_rollout(device, rank, world, 8192, 50, 25)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline: the WHOLE STEP on SURVEY 8d's algorithmic bytes; the dominant kernel as a sub-key ----------------
    li_spec = li0.get('specialised', 1)
    peak, peak_src = measured_peak()
    bytes_per_step = algorithmic_bytes_per_env_step(N, L, D, F, int(getattr(args, 'num_obstacles', 0))) * n_envs
    step_s = float(step_ms.mean()) / 1000.0
    achieved = bytes_per_step / step_s / 1e9
    traffic = None
    tp = os.path.join(REPO, 'profiles', 'traffic_r02.json')
    if not os.path.exists(tp):
        tp = os.path.join(REPO, 'profiles', 'traffic_r01.json')
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get(a.workload)
        except Exception:
            traffic = None
    step_traffic = None          # ncu dram bytes of all kernels of one step (profiles/traffic_r02.json "<workload>_step"), or null
    try:
        with open(tp) as f:
            step_traffic = json.load(f).get(a.workload + '_step')
    except Exception:
        step_traffic = None
    dominant = None
    if emit_ms is not None:
        # lsm_emit_kernel alone on ITS 8d bytes: node_obs + adj written (the per-env record it reads is an implementation
        # intermediate and is not counted)
        out_bytes = n_envs * (4 * N * env.E * (F + env.E))
        dominant = {"kernel": "lsm_emit_kernel<dyn,N,L> (graph emission), timed alone with the same L2 flush",
                    "algorithmic_bytes_per_launch": out_bytes, "mean_launch_ms": emit_ms,
                    "achieved": out_bytes / (emit_ms / 1000.0) / 1e9, "frac": out_bytes / (emit_ms / 1000.0) / 1e9 / peak,
                    "traffic": traffic,
                    "note": "traffic = ncu dram bytes of this kernel per launch (profiles/traffic_r0*.json). When the step's "
                            "output fits the 126 MB L2 (cfg2: 107 MB) about half of it is still dirty in L2 when the kernel "
                            "ends, so traffic / algorithmic ~ 0.5 there; at cfg3 / cfg4 (outputs >> L2) it is ~1.0"}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": step_traffic, "peak_source": peak_src,
                "kernel": ("whole step = lsm_agent_kernel + lsm_emit_kernel + lsm_pair_kernel" if li_spec else "lsm_generic_kernel<dyn>"),
                "algorithmic_bytes_per_launch": bytes_per_step, "mean_launch_ms": step_s * 1000.0,
                "median_ms": float(np.median(step_ms)), "launches": li0.get('launches_per_step', 1),
                "dominant_kernel": dominant}

    # ---- CPU baseline (bounded sample) ----------------------------------------------------------
    cpu = None
    if not a.no_cpu_baseline:
        cores = os.cpu_count() or 1
        n_s = 1024
        probe, dtp, _, _ = oracle_throughput(a.workload, n_s, 3, 1, cores)
        steps_s = int(max(5, min(20000, 12.0 / max(dtp / 3, 1e-6))))      # ~12 s of CPU work on every host thread
        val, dts, _, _ = oracle_throughput(a.workload, n_s, steps_s, 2, cores)
        cpu = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n_s} envs x {steps_s} steps of {a.workload} ({dts:.1f} s) with the C oracle port of the "
                         f"reference's Python path on {cores} host threads; the Python reference itself measured "
                         f"1.0e3 agent-steps/s on 8 cores (BASELINE.md)"}

    li = li0
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD_DESC[a.workload], "envs_per_gpu": n_envs, "num_agents": N,
                       "landmarks_per_agent": L, "entities": env.E, "value_grid": "synthetic (shape assumed)",
                       "l2": "256 MiB flush between timed steps", "parallelism": f"env-shard x{world}",
                       "launch": li},
            "ms_per_step_back_to_back": noflush_ms / K,
            "value_back_to_back": total_envs * N * K / (noflush_ms / 1000.0),
            "rotating_outputs": None if rot_ms is None else {
                "ms_per_step": rot_ms / K, "value": n_envs * N * K / (rot_ms / 1000.0), "slots": n_slots,
                "note": "this rank, no L2 flush: node_obs / adj of consecutive steps go to different slots (total > 2.5 x L2), "
                        "like a rollout buffer; the few-MB state stays L2-warm as in a real run"},
            "wall_s_timed_loop": t_wall,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": Ke, "ms_per_step": e2e_ms / Ke,
                    "api": "B200GraphVecEnv.step(host one-hot float32 actions) -> host numpy obs/agent_id/node_obs/adj/rewards/dones",
                    "host_side": e2e_host},
            "gpu_launches": K * li.get('launches_per_step', 1),
            "timeline_us": timeline,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "workloads": extra,
            "episode_stats": stats}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_rollout(device, rank, world, n_envs, K, W, dump_dir=None):
    """BASELINE configs[4] shape - rollout collection of the onpolicy GraphMPE runner (8 agents, 8192 envs per GPU) with
    the device-resident rollout buffer: env.step writes observations / graphs / rewards straight into the buffer slot
    (zero copy), insert() builds masks / share_obs on the device. The policy forward is NOT part of this repo: actions
    are drawn on the device (stated in `config`). Each step lands in a different 221 MB slot of the 5.7 GB buffer, i.e.
    the outputs are larger than L2 without a flush."""
    import torch
    import torch.distributed as dist
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    args, flags, _, episode = build_args('cfg2')
    T = 25
    env = B200GraphVecEnv(args, num_envs=n_envs, device=device, seed=1234, binary_cfg=flags, env_id_base=rank * n_envs)
    buf = DeviceGraphRolloutBuffer(env, T, use_centralized_V=True, zero_copy=True)
    N = env.N
    gen = torch.Generator(device=device); gen.manual_seed(7 + rank)
    buf.warmup(num_current_episode=episode)

    def collect(steps):
        out = None
        for _ in range(steps):
            actions = torch.randint(0, 25, (n_envs, N), generator=gen, device=device, dtype=torch.int32)
            out = env.step(actions, episode)
            buf.insert(out, actions=actions)
            if buf.step == 0:
                buf.after_update()
        return out
    collect(W)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); last = collect(K); e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dump_dir and rank == 0:
        # zero copy: the returned tensors are views of the buffer slot the last step wrote; no step runs before the dump
        obs, agent_id, node_obs, adj, rewards, dones, _ = last
        info = dump_outputs(dump_dir, dict(obs=obs, agent_id=agent_id, node_obs=node_obs, adj=adj, rewards=rewards,
                                           dones=dones))
        print(f"outputs of the last timed step: {info}", file=sys.stderr, flush=True)
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=device); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ms = float(tt[0])
    peak, peak_src = measured_peak()
    bytes_per_step = algorithmic_bytes_per_env_step(N, env.L, env.D, env.F, env.O) * n_envs
    li = env.launch_info()
    out = {"workload": "BASELINE configs[4] shape: rollout collection (env.step + rollout-buffer insert, zero copy) "
                       "8 agents x 8192 envs per B200, HJ filter on; policy forward excluded (actions drawn on device)",
           "envs_per_gpu": n_envs, "num_agents": N, "buffer_steps": T, "steps": K,
           "value": n_envs * world * N * K / (ms / 1000.0), "unit": UNIT, "ms_per_step": ms / K,
           "algorithmic_bytes_per_step": bytes_per_step, "whole_step_frac": bytes_per_step / (ms / K / 1000.0) / 1e9 / peak,
           "peak_source": peak_src, "launch": li,
           "l2": "every step lands in a different 221 MB buffer slot (outputs > L2), no flush"}
    env.close()
    del buf, env
    torch.cuda.empty_cache()
    return out


def run_rollout(a):
    """`--workload cfg5` as the headline line (see measure_rollout)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1')); rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local_rank}'))
    device = torch.device(f'cuda:{local_rank}'); torch.cuda.set_device(device)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    r = measure_rollout(device, rank, world, a.envs or 8192, a.steps, a.warmup, dump_dir=a.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peak, _ = measured_peak()
        li = r['launch']
        line = {"metric": METRIC, "value": r['value'], "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": r['ms_per_step'], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": r['workload'], "envs_per_gpu": r['envs_per_gpu'], "num_agents": r['num_agents'],
                           "buffer_steps": r['buffer_steps'], "l2": r['l2'], "launch": li},
                "clocks": clocks, "e2e": None, "gpu_launches": a.steps * (li.get('launches_per_step', 1) + 1),
                "roofline": {"bound": "hbm", "achieved": r['whole_step_frac'] * peak, "peak": peak, "unit": "GB/s",
                             "frac": r['whole_step_frac'], "traffic": None, "peak_source": r['peak_source'],
                             "kernel": "whole collection step (3 kernels + lsm_rollout_insert)",
                             "algorithmic_bytes_per_launch": r['algorithmic_bytes_per_step']},
                "cpu_baseline": None}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS) + ['cfg5'])
    ap.add_argument('--envs', type=int, default=0, help='envs per GPU (default: the workload’s)')
    ap.add_argument('--e2e-steps', type=int, default=60)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--numa-bind', action='store_true', help='e2e: pin the process to the CPUs of the NUMA node of its GPU')
    ap.add_argument('--use-graph', type=int, default=-1, choices=[-1, 0, 1],
                    help='lsm_tuning.use_graph of the device-timed env: -1 automatic (= plain launches), 0 plain launches, 1 graph replay from a static action buffer')
    ap.add_argument('--no-extra-workloads', action='store_true', help='skip the cfg3 / cfg4 / cfg5 sub-blocks of the default line')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, save what the last one returned as DIR/<name>.npy (float32 / float64, '
                         'at most 64 MB: a fixed sample of the environments when the batch is larger; rank 0)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.warmup < 3:
        a.warmup = 3
    if a.impl == 'reference':
        if a.workload == 'cfg5':
            a.workload = 'cfg2'       # the same environment; the reference arm times env.step only
        run_reference(a)
    elif a.workload == 'cfg5':
        run_rollout(a)
    else:
        run_ours(a)


if __name__ == '__main__':
    main()
