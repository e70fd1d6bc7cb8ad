"""Step time of shapes outside the product library's shape list: the generic fused kernel (product library) against the
library built for exactly that shape (args.specialise_shape, _build.build_shape; specialised three-kernel pipeline).
bench.py's flushed method: a 256 MiB L2 flush before every timed step, one CUDA event pair per step, an untimed lead-in
of flushes so that the first timed launches are queued.

    python tools/shape_bench.py --runs 3 [--workloads di6,di12,...] [--steps 60] [--out FILE]

Arms, alternated run by run, each in a process of its own (the library is chosen when it is loaded):
    generic   product library (the shape is not in LSM_SPEC_LIST: lsm_generic_kernel)
    variant   the shape's own library (LSM_LIB=<its path>): what args.specialise_shape selects
The workload `*_host` is the numpy_outputs=True step with host actions (one C-ABI call; the variant takes the compact
adjacency over PCIe, the generic kernel dense pinned copies), timed with the host clock around the returning step.
Every result line carries the card name, power limit and SM clocks read in the same process."""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_DI = dict(dynamics_type='double_integrator', use_safety_filter=True, world_size=4, episode_length=250)
_AT = dict(dynamics_type='airtaxi', use_safety_filter=True, world_size=6, episode_length=350)
# name: (args overrides, RewardBinaryConfig switches, envs) - sizes a user runs: the BASELINE workloads' env counts
WORKLOADS = {
    'di6': (dict(_DI, num_agents=6, num_landmarks=2), {}, 4096),
    'di12': (dict(_DI, num_agents=12, num_landmarks=2), {}, 4096),
    'di8_l3': (dict(_DI, num_agents=8, num_landmarks=3), {}, 4096),
    'di32_l4': (dict(_DI, num_agents=32, num_landmarks=4), {}, 1024),            # E = 160: one emit block per SM
    'at6': (dict(_AT, num_agents=6, num_landmarks=2), dict(POTENTIAL_CONFLICT=True), 16384),
    'at10_o2': (dict(_AT, num_agents=10, num_landmarks=2, num_obstacles=2, obstacle_extension=True),
                dict(POTENTIAL_CONFLICT=True), 16384),
    'di12_host': (dict(_DI, num_agents=12, num_landmarks=2), {}, 4096),
}
ARMS = ('generic', 'variant')
EPISODE = 6249


def gpu_facts():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(','), [s.strip() for s in out.split(',')]))
    except Exception as e:       # the timings stand without it; say so in the line
        return {'error': repr(e)}


def build_args(workload):
    import _golden as G
    kw, flags, n_envs = WORKLOADS[workload]
    return G.default_args(**kw), G.BinaryFlags(flags), n_envs


def shape_of(workload):
    kw = WORKLOADS[workload][0]
    return (kw['dynamics_type'], kw['num_agents'], kw['num_landmarks'], kw.get('num_obstacles', 0))


def measure(arm, workload, steps, warmup):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args, flags, n_envs = build_args(workload)
    host = workload.endswith('_host')
    device = torch.device('cuda:0')
    env = B200GraphVecEnv(args, num_envs=n_envs, device=device, seed=1234, binary_cfg=flags, numpy_outputs=host)
    li = env.launch_info()
    want = 1 if arm == 'variant' else 0
    if li['specialised'] != want:
        raise SystemExit(f"{arm} {workload}: launch_info specialised = {li['specialised']}, expected {want}")
    gen = torch.Generator(device=device); gen.manual_seed(1234)
    actions = torch.randint(0, 25, (warmup + steps, n_envs, env.N), generator=gen, device=device, dtype=torch.int32)
    host_actions = actions.cpu().numpy() if host else None
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)   # 256 MiB > 126 MB L2
    env.reset(EPISODE)
    for t in range(warmup):
        env.step(host_actions[t] if host else actions[t], EPISODE)
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ms = []
    gc.collect(); gc.disable()
    for _ in range(12):
        flush.fill_(0.0)
    for t in range(steps):
        flush.fill_(0.0)
        if host:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            env.step(host_actions[warmup + t], EPISODE)      # returns complete host arrays
            ms.append((time.perf_counter() - t0) * 1e3)
        else:
            starts[t].record()
            env.step(actions[warmup + t], EPISODE)
            stops[t].record()
    torch.cuda.synchronize()
    gc.enable()
    if not host:
        ms = [s.elapsed_time(e) for s, e in zip(starts, stops)]
    env.close()
    dyn, N, L, O = shape_of(workload)
    return {'arm': arm, 'workload': workload, 'dynamics': dyn, 'N': N, 'L': L, 'O': O, 'E': N + N * L + O, 'envs': n_envs,
            'steps': steps, 'ms_per_step': sum(ms) / steps, 'ms_median': sorted(ms)[steps // 2],
            'timer': 'host clock, numpy_outputs' if host else 'cuda events, flushed',
            'specialised': li['specialised'], 'launches_per_step': li['launches_per_step'],
            'emit_blocks_per_sm': li['emit_blocks_per_sm'], 'emit_block_threads': li['emit_block_threads']}


def child(a):
    sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, 'tests'))
    facts = gpu_facts()
    r = measure(a.arm, a.workloads, a.steps, a.warmup)
    r['gpu'] = facts
    print(json.dumps(r), flush=True)


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--runs', type=int, default=3)
    p.add_argument('--workloads', default=','.join(WORKLOADS))
    p.add_argument('--steps', type=int, default=60)
    p.add_argument('--warmup', type=int, default=10)
    p.add_argument('--out', default=None, help='also append the result lines to this file')
    p.add_argument('--arm', default=None, help=argparse.SUPPRESS)      # child process
    a = p.parse_args()
    if a.arm:
        return child(a)
    sys.path.insert(0, REPO)
    from concurrent.futures import ThreadPoolExecutor
    from layered_safe_marl_b200 import _build
    workloads = a.workloads.split(',')
    shapes = sorted({shape_of(w) for w in workloads})
    with ThreadPoolExecutor(max_workers=len(shapes)) as ex:          # before any timing: nvcc runs in parallel
        paths = dict(zip(shapes, ex.map(lambda s: _build.build_shape(*s), shapes)))
    lines = []
    for run in range(a.runs):
        for w in workloads:
            for arm in ARMS:
                env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
                env.pop('LSM_LIB', None)
                if arm == 'variant':
                    env['LSM_LIB'] = paths[shape_of(w)]
                out = subprocess.run([sys.executable, os.path.abspath(__file__), '--arm', arm, '--workloads', w,
                                      '--steps', str(a.steps), '--warmup', str(a.warmup)], env=env, capture_output=True, text=True)
                if out.returncode != 0:
                    raise SystemExit(f"{arm} {w} failed:\n{out.stderr[-3000:]}{out.stdout[-2000:]}")
                for line in out.stdout.splitlines():
                    if line.startswith('{'):
                        r = json.loads(line); r['run'] = run
                        lines.append(r)
                        print(json.dumps(r), flush=True)
    print("\nms per step (min .. max over runs); generic / variant")
    for w in workloads:
        v = {arm: [r['ms_per_step'] for r in lines if r['workload'] == w and r['arm'] == arm] for arm in ARMS}
        print(f"  {w:9s} generic {min(v['generic']):.4f}..{max(v['generic']):.4f}   variant {min(v['variant']):.4f}.."
              f"{max(v['variant']):.4f}   ratio {min(v['generic']) / min(v['variant']):.2f}x")
    if a.out:
        with open(a.out, 'a') as f:
            for r in lines:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
