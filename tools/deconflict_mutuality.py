"""How often the safety filter's deconfliction is not mutual: agent i deconflicts against j (its first-minimum
neighbour, AI_DECONFLICT_IDX; SafetyFilter.apply_world's `deconflict`) while j deconflicts against some k != i. The
cooperative value function assumes j plays its part against i; this counts how often it cannot.

    python tools/deconflict_mutuality.py [--envs 1024] [--steps 200] [--out FILE.jsonl]

Random discrete actions on cfg2-shaped (8 double-integrator agents) and cfg3-shaped (10 airtaxi agents) worlds, with
the computed cooperative value grid (reachability.value_grid). Per step and live agent with a partner: whether the
partner's partner is the agent. Prints one JSON line per config: the non-mutual share over all such agent-steps and
over those whose filter fired."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))

import _golden as G  # noqa: E402
from layered_safe_marl_b200 import B200GraphVecEnv, reachability as R  # noqa: E402


def measure(case, n, steps, seed=0):
    if case == 'cfg2':
        args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=250, world_size=4)
        flags, dyn = G.BinaryFlags({}), 0
    else:
        args = G.default_args(dynamics_type='airtaxi', num_agents=10, use_safety_filter=True, episode_length=350,
                              world_size=6)
        flags, dyn = G.BinaryFlags(dict(POTENTIAL_CONFLICT=True)), 1
    env = B200GraphVecEnv(args, num_envs=n, seed=seed, binary_cfg=flags, value_grid=R.value_grid(dyn))
    episode = 6249                  # late in the curriculum, where the filter is on (the parity tests' episode)
    env.reset(episode)
    rng = np.random.default_rng(seed)
    N = args.num_agents
    tot = dict(partnered=0, non_mutual=0, filtered=0, filtered_non_mutual=0)
    for t in range(steps):
        a = torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=env.device)
        env.step(a, episode)
        s = env.get_state()
        d = np.asarray(s['deconflicting_agent_index']).astype(np.int64)
        live = ~np.asarray(s['done']) & (d >= 0)
        back = np.take_along_axis(d, np.clip(d, 0, N - 1), axis=1)
        non_mutual = live & (back != np.arange(N)[None, :])
        filt = live & np.asarray(s['safety_filtered'])
        tot['partnered'] += int(live.sum())
        tot['non_mutual'] += int(non_mutual.sum())
        tot['filtered'] += int(filt.sum())
        tot['filtered_non_mutual'] += int((non_mutual & filt).sum())
    return dict(what='deconflict_mutuality', case=case, envs=n, steps=steps, agents=N, **tot,
                non_mutual_share=tot['non_mutual'] / max(tot['partnered'], 1),
                filtered_non_mutual_share=tot['filtered_non_mutual'] / max(tot['filtered'], 1))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--envs', type=int, default=1024)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    for case in ('cfg2', 'cfg3'):
        rec = json.dumps(measure(case, a.envs, a.steps))
        print(rec, flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(rec + '\n')


if __name__ == '__main__':
    main()
