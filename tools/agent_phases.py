#!/usr/bin/env python
"""Where the specialised agent kernel's time goes, phase by phase (lab build only).

Every env group (one warp) of lsm_agent_kernel stamps (%globaltimer, clock64) at its phase boundaries
(lsm_device.cuh PH_*); the product library has no stamps. Durations are taken from clock64 (per SM, cycle resolution)
and converted to ns with the ratio of the globaltimer and clock64 spans over all groups. Prints, per phase, the median
over groups and the breakdown of the group that finishes last (the kernel's critical chain), each the median over
K steps, flushed (256 MiB L2 overwrite before every step, like bench.py's timed steps) or back-to-back (--b2b).

A load is issued in the phase that names it but waited for where its value is first used, so DRAM latency lands in
the phase of the first use.

usage: LSM_LIB=layered_safe_marl_b200/liblsm_b200_exp.so tools/agent_phases.py [cfg2] [--b2b] [--steps K]
(`python -c "from layered_safe_marl_b200 import _build; _build.build_experiments()"` builds the lab library)"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, 'tests'))
import torch  # noqa: E402
import bench as B  # noqa: E402
from layered_safe_marl_b200 import B200GraphVecEnv  # noqa: E402
from layered_safe_marl_b200 import _lib  # noqa: E402

PHASES = ('loads', 'landmarks+curriculum', 'decode+filter+integrate', 'goal+reward+done', 'others+bookkeeping',
          'summary+auto-reset', 'state write-back', 'emit records')
SLOTS = len(PHASES) + 1

ap = argparse.ArgumentParser()
ap.add_argument('workload', nargs='?', default='cfg2')
ap.add_argument('--b2b', action='store_true', help='no L2 flush between the stamped steps')
ap.add_argument('--steps', type=int, default=10)
a = ap.parse_args()
if not os.environ.get('LSM_LIB'):
    sys.exit("set LSM_LIB to the lab build (liblsm_b200_exp.so): the product library has no phase stamps")

args, flags, n_envs, episode = B.build_args(a.workload)
env = B200GraphVecEnv(args, num_envs=n_envs, seed=1234, binary_cfg=flags)
lib = env.lib
lib.lsm_debug_phase_stamps.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.POINTER(C.c_longlong)]
lib.lsm_debug_phase_stamps.restype = C.c_int
K = a.steps
gen = torch.Generator(device=env.device); gen.manual_seed(1234)
acts = torch.randint(0, 25, (K + 20, n_envs, env.N), generator=gen, device=env.device, dtype=torch.int32)
flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=env.device)
env.reset(episode)
for t in range(20):
    env.step(acts[t], episode)
torch.cuda.synchronize()

cap = (n_envs + 31) * SLOTS * 2
buf = (C.c_uint64 * cap)()
nw = C.c_longlong(0)
steps = []
_lib.check(lib.lsm_debug_phase_stamps(env._h, 1, None, 0, None), 'lsm_debug_phase_stamps')
env.debug_timeline(True)
windows = []
for t in range(K):
    if not a.b2b:
        flush.fill_(0.0)
    env.step(acts[20 + t], episode)
    _lib.check(lib.lsm_debug_phase_stamps(env._h, 1, buf, cap, C.byref(nw)), 'lsm_debug_phase_stamps')
    tl = env.debug_timeline(True)
    windows.append((tl['agent_end'] - tl['agent_start']) / 1000.0)
    st = np.frombuffer(buf, dtype=np.uint64, count=nw.value).reshape(-1, SLOTS, 2).astype(np.int64)
    steps.append(st[st[:, 0, 0] != 0])          # groups the step ran (all of them for a full batch)
env.debug_timeline(False)
_lib.check(lib.lsm_debug_phase_stamps(env._h, 0, None, 0, None), 'lsm_debug_phase_stamps')

li = env.launch_info()
print(f"{a.workload} {'back-to-back' if a.b2b else 'flushed'}: {n_envs} envs, {steps[0].shape[0]} env groups, "
      f"{K} steps, torch {torch.__version__}, {torch.cuda.get_device_name()}")
print(f"launch: {li}")
med_rows, crit_rows, spans, dispatch, ns_per_clk = [], [], [], [], []
for st in steps:
    gt, clk = st[:, :, 0], st[:, :, 1]
    r = (gt[:, -1] - gt[:, 0]).sum() / max(1, (clk[:, -1] - clk[:, 0]).sum())
    ns_per_clk.append(r)
    dur = np.diff(clk, axis=1) * r                      # [groups][phase] ns
    med_rows.append(np.median(dur, axis=0))
    t0 = gt[:, 0].min()
    last = int(np.argmax(gt[:, -1]))
    crit_rows.append(np.concatenate([[gt[last, 0] - t0], dur[last]]))
    spans.append((gt[:, -1].max() - t0, np.median(gt[:, -1] - gt[:, 0]), np.max(gt[:, -1] - gt[:, 0])))
    dispatch.append(np.percentile(gt[:, 0] - t0, [50, 100]))
med = np.median(np.array(med_rows), axis=0) / 1000.0
crit = np.median(np.array(crit_rows), axis=0) / 1000.0
sp = np.median(np.array(spans), axis=0) / 1000.0
dp = np.median(np.array(dispatch), axis=0) / 1000.0
print(f"SM clock from the stamps: {1.0 / np.median(ns_per_clk):.3f} GHz")
print(f"agent kernel window (product timeline, first block in -> last block out): median {np.median(windows):.2f} us "
      f"(min {min(windows):.2f}, max {max(windows):.2f})")
print(f"first group start -> last group end {sp[0]:.2f} us; one group start -> end: median {sp[1]:.2f} us, max {sp[2]:.2f} us")
print(f"group start after the first one: median {dp[0]:.2f} us, last {dp[1]:.2f} us")
print(f"{'phase':26s} {'median group us':>16s} {'last-ending group us':>21s}")
print(f"{'(start offset)':26s} {'':>16s} {crit[0]:21.2f}")
for k, name in enumerate(PHASES):
    print(f"{name:26s} {med[k]:16.2f} {crit[k + 1]:21.2f}")
print(f"{'sum':26s} {med.sum():16.2f} {crit[1:].sum():21.2f}")
