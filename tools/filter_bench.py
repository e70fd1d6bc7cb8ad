"""Time the standalone safety filter (SafetyFilter.apply / lsm_safety_filter) with CUDA events, beside the env's cfg2 step.

    python tools/filter_bench.py [--calls 50] [--out path.json]

Sizes: double integrator 32 768 rows x 7 others (cfg2's egos), airtaxi 163 840 x 9 (cfg3's egos), double integrator
1 048 576 x 7, each in both interpolation modes. The L2 is overwritten (a 256 MB memset) before every timed call, so
every call reads its inputs and the grid from HBM; the memset is outside the timed window. Prints one JSON object with
the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))

SIZES = [('di', 32768, 7), ('airtaxi', 163840, 9), ('di', 1048576, 7)]


def card():
    try:
        q = subprocess.check_output(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader',
                                     '-i', str(torch.cuda.current_device())], text=True).strip()
        return q
    except Exception as exc:  # pragma: no cover
        return f'unknown ({exc})'


def timed(fn, calls, flush):
    start = [torch.cuda.Event(enable_timing=True) for _ in range(calls)]
    end = [torch.cuda.Event(enable_timing=True) for _ in range(calls)]
    for k in range(calls):
        flush.zero_()
        start[k].record()
        fn()
        end[k].record()
    torch.cuda.synchronize()
    ts = sorted(s.elapsed_time(e) * 1e3 for s, e in zip(start, end))
    return ts[len(ts) // 2], sum(ts) / len(ts)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args(argv)
    import _golden as G
    from layered_safe_marl_b200 import B200GraphVecEnv, SafetyFilter, hj_grid
    dev = torch.device('cuda:0')
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    res = {'card': card(), 'calls': a.calls, 'l2': 'overwritten (256 MB memset) before every timed call', 'operator': []}
    for dyn, B, M in SIZES:
        for f32 in (False, True):
            grid = hj_grid.synthetic_di_grid() if dyn == 'di' else hj_grid.synthetic_airtaxi_grid()
            sf = SafetyFilter('double_integrator' if dyn == 'di' else 'airtaxi', value_grid=grid, interp_float32=f32,
                              device=dev)
            span = torch.tensor([1.0, 1.0, 0.5, 0.5] if dyn == 'di' else [3.0, 3.0, 3.14, 0.02], dtype=torch.float64, device=dev)
            base = torch.tensor([0.0, 0.0, 0.0, 0.0] if dyn == 'di' else [0.0, 0.0, 0.0, 0.066], dtype=torch.float64, device=dev)
            ego = base + span * (2 * torch.rand((B, 4), generator=gen, device=dev, dtype=torch.float64) - 1)
            oth = base + span * (2 * torch.rand((B, M, 4), generator=gen, device=dev, dtype=torch.float64) - 1)
            us = 0.5 if dyn == 'di' else 0.001
            ua = us * (2 * torch.rand((B, 2), generator=gen, device=dev, dtype=torch.float64) - 1)
            uo = us * (2 * torch.rand((B, M, 2), generator=gen, device=dev, dtype=torch.float64) - 1)
            active = torch.rand((B, M), generator=gen, device=dev) < 0.9
            for _ in range(a.warmup):
                out = sf.apply(ego, oth, ua, uo, active)
            med, mean = timed(lambda: sf.apply(ego, oth, ua, uo, active), a.calls, flush)
            in_bytes = B * (4 + 2) * 8 + B * M * ((4 + 2) * 8 + 1)
            res['operator'].append(dict(dynamics=dyn, rows=B, slots=M, interp_float32=f32, us_per_call_median=round(med, 2),
                                        us_per_call_mean=round(mean, 2), rows_per_s=B / (med * 1e-6),
                                        lookups_per_s=B * M / (med * 1e-6), input_bytes_per_s=in_bytes / (med * 1e-6),
                                        filtered_fraction=float(out[1].float().mean())))
            print(json.dumps(res['operator'][-1]), flush=True)
            del sf
    # the env's cfg2 step (8 double-integrator agents x 4096 envs, filter on) in the same run
    for f32 in (False, True):
        args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=250, world_size=4, interp_float32=f32)
        env = B200GraphVecEnv(args, num_envs=4096, seed=1, binary_cfg=G.BinaryFlags({}))
        ep = env.params.num_total_episode - 1
        env.reset(ep)
        acts = torch.randint(0, 25, (a.calls + a.warmup, 4096, 8), device=dev, dtype=torch.int32, generator=gen)
        for k in range(a.warmup):
            env.step(acts[k], ep)
        it = iter(range(a.warmup, a.warmup + a.calls))
        med, mean = timed(lambda: env.step(acts[next(it)], ep), a.calls, flush)
        res.setdefault('env_cfg2_step', []).append(dict(interp_float32=f32, us_per_step_median=round(med, 2),
                                                        us_per_step_mean=round(mean, 2)))
        print(json.dumps(res['env_cfg2_step'][-1]), flush=True)
        env.close()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
