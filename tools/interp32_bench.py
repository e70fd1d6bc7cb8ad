"""Step time of the float32 interpolation mode (args.interp_float32) on the specialised pipeline beside the float64
product, at the BASELINE shapes. bench.py's flushed method: a 256 MiB L2 flush before
every timed step, one CUDA event pair per step, an untimed lead-in of flushes so that the first timed launches are queued.

    python tools/interp32_bench.py --runs 3 [--workloads cfg2,cfg3,cfg3_obst4,cfg4] [--steps 60] [--out FILE]

Arms, alternated run by run, each in a process of its own:
    f32_spec     product library, interp_float32=True   (specialised pipeline, float32 agent / pair kernels)
    f64_spec     product library, float64 (the default)
Every result line carries the card name, power limit and SM clocks read in the same process."""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = ('cfg2', 'cfg3', 'cfg3_obst4', 'cfg4')
ARMS = ('f32_spec', 'f64_spec')


def gpu_facts():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(','), [s.strip() for s in out.split(',')]))
    except Exception as e:       # the timings stand without it; say so in the line
        return {'error': repr(e)}


def measure(arm, workload, steps, warmup):
    import torch
    sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, 'tests'))
    import bench
    from layered_safe_marl_b200 import B200GraphVecEnv
    args, flags, n_envs, episode = bench.build_args(workload)
    args.interp_float32 = arm.startswith('f32')
    device = torch.device('cuda:0')
    env = B200GraphVecEnv(args, num_envs=n_envs, device=device, seed=1234, binary_cfg=flags)
    li = env.launch_info()
    gen = torch.Generator(device=device); gen.manual_seed(1234)
    actions = torch.randint(0, 25, (warmup + steps, n_envs, env.N), generator=gen, device=device, dtype=torch.int32)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)   # 256 MiB > 126 MB L2
    env.reset(episode)
    for t in range(warmup):
        env.step(actions[t], episode)
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    gc.collect(); gc.disable()
    for _ in range(12):
        flush.fill_(0.0)
    for t in range(steps):
        x = actions[warmup + t]
        flush.fill_(0.0)
        starts[t].record()
        env.step(x, episode)
        stops[t].record()
    torch.cuda.synchronize()
    gc.enable()
    ms = [s.elapsed_time(e) for s, e in zip(starts, stops)]
    env.close()
    return {'arm': arm, 'workload': workload, 'envs': n_envs, 'steps': steps, 'ms_per_step': sum(ms) / steps,
            'ms_median': sorted(ms)[steps // 2], 'specialised': li['specialised'], 'launches_per_step': li['launches_per_step']}


def child(a):
    facts = gpu_facts()
    for w in a.workloads.split(','):
        r = measure(a.arm, w, a.steps, a.warmup)
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
    lines = []
    for run in range(a.runs):
        for arm in ARMS:
            env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
            out = subprocess.run([sys.executable, os.path.abspath(__file__), '--arm', arm, '--workloads', a.workloads,
                                  '--steps', str(a.steps), '--warmup', str(a.warmup)], env=env, capture_output=True, text=True)
            if out.returncode != 0:
                raise SystemExit(f"{arm} failed:\n{out.stderr[-3000:]}")
            for line in out.stdout.splitlines():
                if line.startswith('{'):
                    r = json.loads(line); r['run'] = run
                    lines.append(r)
                    print(json.dumps(r), flush=True)
    print("\nms per flushed step (min .. max over runs)")
    for w in a.workloads.split(','):
        row = []
        for arm in ARMS:
            v = [r['ms_per_step'] for r in lines if r['workload'] == w and r['arm'] == arm]
            row.append(f"{arm} {min(v):.4f}..{max(v):.4f}")
        print(f"  {w:11s} " + '   '.join(row))
    if a.out:
        with open(a.out, 'a') as f:
            for r in lines:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
