"""PPO inputs on the device, on one GPU (needs a CUDA device; no fallback).

    python tools/ppo_inputs_bench.py [--out FILE] [--calls 11]

1. returns: compute_returns' torch loop (returns_loop, GAE with and without use_proper_time_limits) against the kernel
   (returns_kernel, lsm_compute_returns) at the step counts and column counts of cfg2 (T = 250, C = 4096 * 8),
   cfg3 (T = 350, C = 16384 * 10) and cfg4 (T = 250, C = 8192 * 32), on seeded synthetic tensors
2. advantages: compute_advantages' work, the loop's returns followed by the trainer's expression in torch on the device
   (returns[:-1] - value_preds[:-1], masked float64 nanmean / nanstd, normalisation) against one kernel pass with
   advantages and moments plus the normalisation (three launches)
3. minibatches: one epoch of feed_forward_batches (4 minibatches) and recurrent_batches (L = 10, 4 minibatches) over a
   25-slot records buffer at cfg2, edges=False and True: us per minibatch, and the share of the graph rows (graph_rows
   on the same indices timed alone) against the other fields' gathers
CUDA events around whole calls ended by a device synchronise, the L2 overwritten (256 MB write) before every timed call,
the two paths alternated, medians. Both paths' outputs are compared once (returns bit for bit). Bytes come from the shapes
(float32 arrays of T or T + 1 rows of C columns; the kernel reads each input once and writes each output once) and are
reported as a share of the 6531.6 GB/s copy peak measured for this repository; the bound is bytes / peak.
The card's name, power limit and SM clocks are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from record_buffer_bench import COPY_PEAK_GBS, gpu_info      # noqa: E402

# name -> (T, columns)
SHAPES = {'cfg2': (250, 4096 * 8), 'cfg3': (350, 16384 * 10), 'cfg4': (250, 8192 * 32)}
OUT = os.path.join(REPO, 'profiles', 'experiments', 'r09_ppo_inputs_bench.jsonl')


def timed(paths, calls, flush):
    """-> {key: [us]}: each path once per round, alternated, the L2 overwritten before every call."""
    import torch
    ts = {k: [] for k in paths}
    for _ in range(calls):
        for k, fn in paths.items():
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1) * 1000.0)
    return ts


def med(v):
    return sorted(v)[len(v) // 2]


def inputs(T, C, seed):
    import torch
    g = torch.Generator(device='cuda').manual_seed(seed)
    r = lambda rows: torch.randn((rows, C), generator=g, device='cuda')
    u = lambda rows: (torch.rand((rows, C), generator=g, device='cuda') < 0.97).float()
    return dict(rewards=r(T), value_preds=r(T + 1), returns=torch.zeros((T + 1, C), device='cuda'), masks=u(T + 1),
                bad_masks=u(T + 1), active_masks=u(T + 1), next_value=r(1)[0])


def returns_run(name, calls, flush):
    import torch
    from layered_safe_marl_b200.rollout import returns_kernel, returns_loop
    T, C = SHAPES[name]
    x = inputs(T, C, 1)
    out = []
    for ptl in (False, True):
        args = lambda ret: (x['rewards'], x['value_preds'], ret, x['masks'], x['bad_masks'], x['next_value'], 0.99, 0.95,
                            True, ptl)
        ret_l, ret_k = x['returns'].clone(), x['returns'].clone()
        paths = {'loop': lambda: returns_loop(*args(ret_l)), 'kernel': lambda: returns_kernel(*args(ret_k))}
        for fn in paths.values():
            fn()
        torch.cuda.synchronize()
        equal = torch.equal(ret_l.view(torch.int32), ret_k.view(torch.int32))
        ts = timed(paths, calls, flush)
        nbytes = 4 * C * ((4 if ptl else 3) * T + 1 + T + 1)      # r, v, m (, b) read; returns written; next value
        k = med(ts['kernel'])
        out.append({'what': 'compute_returns', 'shape': name, 'T': T, 'columns': C, 'use_gae': True,
                    'use_proper_time_limits': ptl, 'returns_equal_bitwise': equal, 'loop_us': med(ts['loop']),
                    'kernel_us': k, 'speedup': med(ts['loop']) / k, 'bytes': nbytes,
                    'bound_us_at_copy_peak': nbytes / (COPY_PEAK_GBS * 1e3), 'share_of_copy_peak': nbytes / (k * 1e3) / COPY_PEAK_GBS,
                    'loop_us_all': ts['loop'], 'kernel_us_all': ts['kernel']})
        print(json.dumps(out[-1]), flush=True)
    return out, x


def advantages_run(name, x, calls, flush):
    import torch
    from layered_safe_marl_b200.rollout import returns_kernel, returns_loop
    T, C = SHAPES[name]
    ret_l, ret_k = x['returns'].clone(), x['returns'].clone()
    adv_k = torch.empty_like(x['rewards'])
    stats = torch.empty(2, device='cuda')
    args = lambda ret: (x['rewards'], x['value_preds'], ret, x['masks'], x['bad_masks'], x['next_value'], 0.99, 0.95,
                        True, False)
    inactive = x['active_masks'][:-1] == 0

    def torch_path():
        returns_loop(*args(ret_l))
        adv = ret_l[:-1] - x['value_preds'][:-1]
        a = adv.double().masked_fill(inactive, float('nan'))
        mean = torch.nanmean(a)
        std = torch.nanmean((a - mean) ** 2).sqrt()
        mean, std = mean.float(), std.float()
        return (adv - mean) / (std + 1e-5), mean, std

    def kernel_path():
        returns_kernel(*args(ret_k), advantages=adv_k, active_masks=x['active_masks'], stats=stats)
        return (adv_k - stats[0]) / (stats[1] + 1e-5), stats[0], stats[1]

    a, b = torch_path(), kernel_path()
    torch.cuda.synchronize()
    equal_returns = torch.equal(ret_l.view(torch.int32), ret_k.view(torch.int32))
    mean_rel = abs(float(a[1]) - float(b[1])) / max(abs(float(a[1])), 1e-30)
    ts = timed({'torch': torch_path, 'kernel': kernel_path}, calls, flush)
    nbytes = 4 * C * (6 * T + 2)              # r, v, m, active read; returns, advantages written; next value, value_preds[T]
    k = med(ts['kernel'])
    res = {'what': 'compute_advantages', 'shape': name, 'T': T, 'columns': C, 'returns_equal_bitwise': equal_returns,
           'mean_rel_diff_torch_vs_kernel': mean_rel, 'torch_us': med(ts['torch']), 'kernel_us': k,
           'speedup': med(ts['torch']) / k, 'bytes_kernel_pass': nbytes,
           'bound_us_at_copy_peak': nbytes / (COPY_PEAK_GBS * 1e3),
           'share_of_copy_peak_incl_normalisation': nbytes / (k * 1e3) / COPY_PEAK_GBS,
           'torch_us_all': ts['torch'], 'kernel_us_all': ts['kernel']}
    print(json.dumps(res), flush=True)
    return res


def minibatch_run(calls, flush, T_BUF=25):
    import bench
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    args, flags, _, episode = bench.build_args('cfg2')
    n = 4096
    env = B200GraphVecEnv(args, num_envs=n, seed=1, binary_cfg=flags)
    N = env.N
    buf = DeviceGraphRolloutBuffer(env, T_BUF, zero_copy=True, graph_storage='records')
    buf.warmup(num_current_episode=episode)
    gen = torch.Generator(device=env.device); gen.manual_seed(3)
    for _ in range(T_BUF):
        a = torch.randint(0, 25, (n, N), generator=gen, device=env.device, dtype=torch.int32)
        buf.insert(env.step(a, episode), actions=a)
    buf.compute_returns(torch.randn((n, N, 1), device='cuda'))
    adv = buf.compute_advantages()[0]
    nmb, L = 4, 10
    out = []
    for kind in ('feed_forward', 'recurrent'):
        count = T_BUF * n * N if kind == 'feed_forward' else T_BUF * n * N // L
        perm = torch.randperm(count, device='cuda', generator=gen)
        for edges in (False, True):
            if kind == 'feed_forward':
                epoch = lambda: [b for b in buf.feed_forward_batches(adv, nmb, edges=edges, perm=perm)]
            else:
                epoch = lambda: [b for b in buf.recurrent_batches(adv, nmb, L, edges=edges, perm=perm)]
            batches = epoch()
            rows = batches[0]['obs'].shape[0]
            # the graph rows of the same minibatches, alone
            idx = []
            for i in range(nmb):
                if kind == 'feed_forward':             # rows of the (T, n, N) flattening
                    r = perm[i * rows:(i + 1) * rows]
                    idx.append((torch.div(r, n * N, rounding_mode='floor'), torch.div(r, N, rounding_mode='floor') % n, r % N))
                else:                                  # rows of the (n, N, T) flattening
                    mbs = rows // L
                    first = perm[i * mbs:(i + 1) * mbs] * L
                    r = (first.view(1, -1) + torch.arange(L, device='cuda').view(-1, 1)).reshape(-1)
                    col = torch.div(r, T_BUF, rounding_mode='floor')
                    idx.append((r % T_BUF, torch.div(col, N, rounding_mode='floor'), col % N))
            graph = lambda: [buf.graph_rows(*i, edges=edges) for i in idx]
            del batches
            graph()
            torch.cuda.synchronize()
            ts = timed({'epoch': epoch, 'graph': graph}, calls, flush)
            e, g = med(ts['epoch']), med(ts['graph'])
            out.append({'what': 'minibatches', 'generator': kind, 'edges': edges, 'shape': 'cfg2', 'envs': n, 'slots': T_BUF,
                        'num_mini_batch': nmb, 'data_chunk_length': L if kind == 'recurrent' else None,
                        'rows_per_minibatch': rows, 'epoch_us': e, 'us_per_minibatch': e / nmb,
                        'graph_rows_us_per_minibatch': g / nmb, 'other_fields_us_per_minibatch': (e - g) / nmb,
                        'graph_share': g / e, 'epoch_us_all': ts['epoch'], 'graph_us_all': ts['graph']})
            print(json.dumps(out[-1]), flush=True)
    env.close()
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--out', default=OUT, help='write the JSON lines to this file')
    ap.add_argument('--calls', type=int, default=11)
    ap.add_argument('--shapes', default=','.join(SHAPES))
    ap.add_argument('--skip-minibatches', action='store_true')
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ppo_inputs_bench needs a CUDA device")
    lines = [{'gpu': gpu_info()}]
    print(json.dumps(lines[0]), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for name in a.shapes.split(','):
        res, x = returns_run(name, a.calls, flush)
        lines += res
        lines.append(advantages_run(name, x, a.calls, flush))
        del x
        torch.cuda.empty_cache()
    if not a.skip_minibatches:
        lines += minibatch_run(a.calls, flush)
    lines.append({'gpu_after': gpu_info()})
    print(json.dumps(lines[-1]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        for l in lines:
            f.write(json.dumps(l) + '\n')


if __name__ == '__main__':
    main()
