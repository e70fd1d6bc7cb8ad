"""Rollout storage by emit record against the dense rollout buffer, on one GPU (needs a CUDA device; no fallback).

    python tools/record_buffer_bench.py [--out FILE] [--rows 32768] [--calls 30]

1. collected-step time (bench.py cfg5's method: env.step + buffer insert, zero copy, actions drawn on the device) of the
   dense buffer and the records buffer at cfg2 (4096 envs) and cfg5 (8192 envs), alternated in the same process;
   the difference is the cost of lsm_copy_records
2. minibatch re-emission (graph_batch of random rows) at the cfg2 / cfg3 / cfg4 shapes against index_select of the same
   rows from a dense buffer: CUDA events, L2 overwritten (256 MB write) before every call, median over --calls calls;
   bytes = records read + rows written, as a fraction of the 6531.6 GB/s copy peak measured for this repository
3. graph-storage bytes per env-slot of both modes, from the shapes
The card's name, power limit and SM clocks are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

COPY_PEAK_GBS = 6531.6
T_BUF = 25
# name -> (bench.py workload whose arguments are used, envs)
SHAPES = {'cfg2': ('cfg2', 4096), 'cfg3': ('cfg3', 16384), 'cfg4': ('cfg4', 8192)}


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], stdout=subprocess.PIPE,
                             text=True, check=True).stdout.strip().splitlines()[0]
        return dict(zip(q.split(','), [x.strip() for x in out.split(',')]))
    except Exception as exc:    # the numbers are still reported; the card is then unnamed
        return {'error': str(exc)}


def collected_step_ms(bench, n_envs, K=50, W=25, reps=3):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    args, flags, _, episode = bench.build_args('cfg2')
    runs = {}
    for mode in ('dense', 'records'):
        env = B200GraphVecEnv(args, num_envs=n_envs, seed=1234, binary_cfg=flags)
        buf = DeviceGraphRolloutBuffer(env, T_BUF, zero_copy=True, graph_storage=mode)
        buf.warmup(num_current_episode=episode)
        gen = torch.Generator(device=env.device); gen.manual_seed(7)
        runs[mode] = (env, buf, gen)

    def collect(mode, steps):
        env, buf, gen = runs[mode]
        for _ in range(steps):
            a = torch.randint(0, 25, (n_envs, env.N), generator=gen, device=env.device, dtype=torch.int32)
            buf.insert(env.step(a, episode), actions=a)
            if buf.step == 0:
                buf.after_update()
    res = {m: [] for m in runs}
    for _ in range(reps):
        for mode in runs:
            collect(mode, W)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); collect(mode, K); e1.record()
            torch.cuda.synchronize()
            res[mode].append(e0.elapsed_time(e1) / K)
    out = {'envs': n_envs, 'steps': K, 'reps': reps}
    for m, v in res.items():
        out[f'{m}_ms_per_step'] = sorted(v)[len(v) // 2]
        out[f'{m}_ms_all'] = v
        out[f'{m}_graph_bytes'] = runs[m][1].graph_nbytes()
    out['copy_records_us_per_step'] = (out['records_ms_per_step'] - out['dense_ms_per_step']) * 1000.0
    for env, buf, _ in runs.values():
        env.close()
    return out


def median_call_us(fn, calls, flush):
    import torch
    ts = []
    for _ in range(calls):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1000.0)
    return sorted(ts)[len(ts) // 2]


def reemission(bench, name, rows, calls, flush):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    wl, n = SHAPES[name]
    args, flags, _, episode = bench.build_args(wl)
    env = B200GraphVecEnv(args, num_envs=n, seed=1, binary_cfg=flags)
    N, E, F = env.N, env.E, env.F
    R = env.launch_info()['emit_record_bytes']
    store = torch.empty((T_BUF, n, R), dtype=torch.uint8, device=env.device)
    env.reset(episode)
    gen = torch.Generator(device=env.device); gen.manual_seed(3)
    for t in range(T_BUF):
        env.step(torch.randint(0, 25, (n, N), generator=gen, device=env.device, dtype=torch.int32), episode)
        env.copy_records(store[t])
    idx = torch.randint(0, T_BUF * n * N, (rows,), generator=gen, device=env.device)
    rec, obs_i = torch.div(idx, N, rounding_mode='floor'), (idx % N).to(torch.int32)
    no = torch.empty((rows, E, F), device=env.device); ad = torch.empty((rows, E, E), device=env.device)
    env.emit_from_records(store, rec, obs_i, no, ad)       # warm-up
    torch.cuda.synchronize()
    us = median_call_us(lambda: env.emit_from_records(store, rec, obs_i, no, ad), calls, flush)
    out_bytes = rows * E * (F + E) * 4
    nbytes = rows * R + out_bytes
    res = {'shape': name, 'envs': n, 'N': N, 'E': E, 'F': F, 'record_bytes': R, 'rows': rows, 'calls': calls,
           'reemit_us': us, 'reemit_rows_per_s': rows / (us * 1e-6), 'reemit_bytes': nbytes,
           'reemit_GBps': nbytes / (us * 1e-6) / 1e9, 'reemit_frac_of_copy_peak': nbytes / (us * 1e-6) / 1e9 / COPY_PEAK_GBS,
           'dense_bytes_per_env_slot': N * E * (F + E) * 4, 'record_bytes_per_env_slot': R}
    env.close()
    del store
    # dense gather of the same number of rows from a dense buffer of the same shape (fewer slots where T = 25 does not fit)
    free = torch.cuda.mem_get_info()[0]
    slots = T_BUF
    while slots > 1 and slots * n * N * E * (F + E) * 4 > 0.6 * free:
        slots //= 2
    dense_bytes = slots * n * N * E * (F + E) * 4
    if dense_bytes <= 0.6 * free:
        dn = torch.empty((slots * n * N, E, F), device='cuda'); da = torch.empty((slots * n * N, E, E), device='cuda')
        gi = torch.randint(0, slots * n * N, (rows,), generator=gen, device='cuda')

        def gather():
            torch.index_select(dn, 0, gi, out=no); torch.index_select(da, 0, gi, out=ad)
        gather()
        torch.cuda.synchronize()
        g = median_call_us(gather, calls, flush)
        res.update(dense_gather_slots=slots, dense_gather_buffer_bytes=dense_bytes, dense_gather_us=g,
                   dense_gather_GBps=2 * out_bytes / (g * 1e-6) / 1e9, reemit_over_gather=us / g)
        del dn, da
    else:
        res.update(dense_gather_us='not measured: no dense buffer of this shape fits')
    torch.cuda.empty_cache()
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--out', default=None, help='also write the JSON lines to this file')
    ap.add_argument('--rows', type=int, default=32768)
    ap.add_argument('--calls', type=int, default=30)
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("record_buffer_bench needs a CUDA device")
    import bench
    lines = [{'gpu': gpu_info(), 'copy_peak_GBps': COPY_PEAK_GBS}]
    for n in (4096, 8192):
        lines.append({'collected_step': collected_step_ms(bench, n)})
        print(json.dumps(lines[-1]), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for name in SHAPES:
        lines.append({'reemission': reemission(bench, name, a.rows, a.calls, flush)})
        print(json.dumps(lines[-1]), flush=True)
    lines.append({'gpu_after': gpu_info()})
    print(json.dumps(lines[0])); print(json.dumps(lines[-1]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            for l in lines:
                f.write(json.dumps(l) + '\n')


if __name__ == '__main__':
    main()
