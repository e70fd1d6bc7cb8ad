#!/usr/bin/env python
"""Per-kernel timeline of one step (diagnostics): %globaltimer first-block-in / last-block-out of the agent, emit and
pair kernels, medians over K flushed (or back-to-back) steps.  usage: tools/timeline.py <workload> [--b2b = warm L2, no flush] [--steps K]"""
import argparse, os, sys
import numpy as np
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, 'tests'))
import torch
import bench as B
from layered_safe_marl_b200 import B200GraphVecEnv

ap = argparse.ArgumentParser(); ap.add_argument('workload'); ap.add_argument('--b2b', action='store_true'); ap.add_argument('--steps', type=int, default=30)
a = ap.parse_args()
args, flags, n_envs, episode = B.build_args(a.workload)
env = B200GraphVecEnv(args, num_envs=n_envs, seed=1234, binary_cfg=flags)
K = a.steps
acts = torch.randint(0, 25, (K + 10, n_envs, env.N), device=env.device, dtype=torch.int32)
flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=env.device)
env.reset(episode)
for t in range(10):
    env.step(acts[t], episode)
rows = []
env.debug_timeline(True)
for t in range(K):
    if not a.b2b:
        flush.fill_(0.0)                # cold L2, like bench.py's timed steps
    env.step(acts[10 + t], episode)     # --b2b: warm L2 (no flush), but still one recorded step at a time
    rows.append(env.debug_timeline(True))
keys = list(rows[0].keys())
print(a.workload, 'b2b' if a.b2b else 'flushed')
for k in keys:
    vals = [r[k] for r in rows if r[k] is not None]
    if vals:
        print(f"  {k:14s} median {np.median(vals) / 1000.0:9.2f} us   min {min(vals) / 1000.0:9.2f}   max {max(vals) / 1000.0:9.2f}")
