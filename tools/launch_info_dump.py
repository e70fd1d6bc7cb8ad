#!/usr/bin/env python
"""launch_info() of a fixed set of handles, one JSON line each, for comparing the launch geometry of two library builds
(select a build with LSM_LIB=<path>; diff the outputs).

    python tools/launch_info_dump.py                      the listed shapes x float32 / float64 x filter on / off, pair
                                                          placements 0 / 2 / 3 / 4 x chunks 1 / 3, one generic-kernel shape
    python tools/launch_info_dump.py --shape airtaxi,6,2,0
                                                          one shape x float32 / float64 x filter on / off; with LSM_LIB
                                                          the library it names, else the shape's own (_build.build_shape)"""
import argparse
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, 'tests'))
import _golden as G
from layered_safe_marl_b200 import B200GraphVecEnv

# the shapes lsm_kernels.cu's LSM_SPEC_LIST specialises: (dynamics, agents, obstacles)
LISTED = [('double_integrator', 8, 0), ('double_integrator', 3, 0), ('double_integrator', 32, 0), ('double_integrator', 4, 0),
          ('double_integrator', 16, 0), ('airtaxi', 10, 0), ('airtaxi', 4, 0), ('airtaxi', 8, 0), ('airtaxi', 16, 0),
          ('airtaxi', 10, 4), ('double_integrator', 8, 4)]
N_ENVS = 512        # enough env groups for 3 chunks at every listed shape


def dump(case, dynamics, N, O, f32=False, filt=True, tuning=None, L=2, specialise=False):
    args = G.default_args(dynamics_type=dynamics, num_agents=N, num_landmarks=L, num_obstacles=O, obstacle_extension=O > 0,
                          use_safety_filter=filt, interp_float32=f32, specialise_shape=specialise)
    env = B200GraphVecEnv(args, num_envs=N_ENVS, seed=1, tuning=tuning)
    print(json.dumps({'case': case, 'launch_info': env.launch_info()}, sort_keys=True), flush=True)
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--shape', default=None, metavar='DYNAMICS,N,L,O')
    a = ap.parse_args()
    if a.shape:
        dyn, N, L, O = a.shape.split(',')
        for f32 in (False, True):
            for filt in (True, False):
                dump(f'{a.shape} f32={f32} filter={filt}', dyn, int(N), int(O), f32, filt, L=int(L), specialise=True)
        return
    for dyn, N, O in LISTED:
        for f32 in (False, True):
            for filt in (True, False):
                dump(f'{dyn} N={N} O={O} f32={f32} filter={filt}', dyn, N, O, f32, filt)
    for dyn, N in (('double_integrator', 8), ('airtaxi', 10)):
        for placement in (0, 2, 3, 4):
            for chunks in (1, 3):
                dump(f'{dyn} N={N} placement={placement} chunks={chunks}', dyn, N, 0,
                     tuning=dict(pair_placement=placement, chunks=chunks))
    dump('double_integrator N=6 O=0 (generic kernel)', 'double_integrator', 6, 0)


if __name__ == '__main__':
    main()
