"""Learner minibatch edge lists from a records rollout buffer, on one GPU (needs a CUDA device; no fallback).

    python tools/record_edges_bench.py [--out FILE] [--rows 32768] [--calls 30]

At the cfg2 / cfg3 / cfg4 shapes, --rows random rows of a 25-slot DeviceGraphRolloutBuffer(graph_storage='records'):
  (a) today's learner path: graph_batch(rows) -> dense (B, E, E) adjacency, then process_adj's torch expression
      (adj.nonzero(), [b*E+i, b*E+j], the gather of the values)
  (b) graph_batch(rows, edges=True): node rows re-emitted without the matrices, edge list straight from the records
CUDA events around whole calls (both contain one host sync: nonzero / reading nnz), the L2 overwritten by a 256 MB write
before every call, (a) and (b) alternated, medians over --calls calls. Both paths' outputs are compared once (they must
be equal). Bytes written per row come from the shapes and the mean edge count of the rows:
  (a) node rows 4EF + dense matrix 4E^2 + per edge: nonzero's (nnz, 3) int64 24, edge_index 16, edge_attr 4
  (b) node rows 4EF + count 4 + offset 8 + per edge: edge_index 16, edge_attr 4
The card's name, power limit and SM clocks are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from record_buffer_bench import SHAPES, T_BUF, gpu_info      # noqa: E402


def shape_run(bench, name, rows, calls, flush):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    from layered_safe_marl_b200.rollout import process_adj
    wl, n = SHAPES[name]
    args, flags, _, episode = bench.build_args(wl)
    env = B200GraphVecEnv(args, num_envs=n, seed=1, binary_cfg=flags)
    N, E, F = env.N, env.E, env.F
    buf = DeviceGraphRolloutBuffer(env, T_BUF, zero_copy=True, graph_storage='records')
    buf.warmup(num_current_episode=episode)
    gen = torch.Generator(device=env.device); gen.manual_seed(3)
    for _ in range(T_BUF):
        a = torch.randint(0, 25, (n, N), generator=gen, device=env.device, dtype=torch.int32)
        buf.insert(env.step(a, episode), actions=a)
    idx = torch.randint(0, T_BUF * n * N, (rows,), generator=gen, device=env.device)

    def dense_path():
        no, ad = buf.graph_batch(idx)
        return (no,) + process_adj(ad)

    def edge_path():
        return buf.graph_batch(idx, edges=True)

    ra, rb = dense_path(), edge_path()       # warm-up, and the equality check
    torch.cuda.synchronize()
    equal = all(torch.equal(x.contiguous().view(torch.int32) if x.dtype == torch.float32 else x,
                            y.contiguous().view(torch.int32) if y.dtype == torch.float32 else y) for x, y in zip(ra, rb))
    nnz = int(rb[1].shape[1])
    del ra, rb
    ts = {'a': [], 'b': []}
    for _ in range(calls):
        for key, fn in (('a', dense_path), ('b', edge_path)):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); out = fn(); e1.record()
            torch.cuda.synchronize()
            ts[key].append(e0.elapsed_time(e1) * 1000.0)
            del out
    med = {k: sorted(v)[len(v) // 2] for k, v in ts.items()}
    deg = nnz / rows
    bytes_a = 4 * E * F + 4 * E * E + deg * (24 + 16 + 4)
    bytes_b = 4 * E * F + 4 + 8 + deg * (16 + 4)
    res = {'shape': name, 'envs': n, 'N': N, 'E': E, 'F': F, 'slots': T_BUF, 'rows': rows, 'calls': calls,
           'nnz': nnz, 'edges_per_row': deg, 'outputs_equal': equal,
           'a_dense_then_process_adj_us': med['a'], 'b_edges_from_records_us': med['b'], 'b_over_a': med['b'] / med['a'],
           'a_us_all': ts['a'], 'b_us_all': ts['b'],
           'a_bytes_written_per_row': bytes_a, 'b_bytes_written_per_row': bytes_b}
    env.close()
    del buf
    torch.cuda.empty_cache()
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--out', default=None, help='also write the JSON lines to this file')
    ap.add_argument('--rows', type=int, default=32768)
    ap.add_argument('--calls', type=int, default=30)
    ap.add_argument('--shapes', default=','.join(SHAPES))
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("record_edges_bench needs a CUDA device")
    import bench
    lines = [{'gpu': gpu_info()}]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for name in a.shapes.split(','):
        lines.append({'minibatch_edges': shape_run(bench, name, a.rows, a.calls, flush)})
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
