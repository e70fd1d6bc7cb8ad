"""Time the HJ reachability solver (liblsm_b200_hj.so) on one GPU and print one JSON line per measurement.

    python tools/hj_solve_bench.py [--out FILE.jsonl] [--steps 20] [--eager-max-cells 30000000]
    python tools/hj_solve_bench.py --ttr [--out FILE.jsonl] [--steps 20]


Per lattice (the two default lattices and refined ones of 10^7-10^8 cells):
- stage_us: per-stage kernel time from CUDA events, (solve to 2S steps - solve to S steps) / (3 S), so the initial
  copy, the upload and the snapshot drop out;
- solve_ms: the whole solve to the default horizon (default lattices) or to S steps (refined), events around the call;
- eager: the same scheme as torch eager ops (tests/hj_solve_oracle.py written against torch), the baseline a user would
  otherwise write, per RK3 step;
- cell_updates_per_s, fp64_ops_per_cell_stage and min_bytes_per_cell_stage (counted from the kernel source: a division
  counts as one op), the achieved FP64 op rate and the share of the measured HBM copy bandwidth (a 4 GiB
  device-to-device copy in the same run);
- convergence: max|V(H) - V(H/2)| of each default lattice at its default horizon.
With --ttr, the airtaxi time-to-reach solve (reachability.solve_ttr) on the default TTR lattice and a refined one,
with the same stage_us / solve_ms / rate / bound fields (no eager baseline) and, per lattice, the fraction of cells
still unreached at the default horizon and at twice it.
The card's name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))

from layered_safe_marl_b200 import hj_grid, reachability as R  # noqa: E402
import hj_solve_oracle as HO  # noqa: E402

# counted from csrc/lsm_hj.cu: weno5 = 64 ops + 4 divisions; per dim 12 (differences) + 2 weno5 + 2 (average) + 4
# (dissipation); Hamiltonian 11 (double integrator) / 19 (airtaxi); 6 for min(0, .) and the RK combination
WENO_OPS = 68
PER_DIM = 12 + 2 * WENO_OPS + 2 + 4
OPS = {0: 4 * PER_DIM + 11 + 6, 1: 5 * PER_DIM + 19 + 6}
# compulsory traffic per cell and stage: the stencil input read once, u0 read (stages 2 and 3), the output written
BYTES = (8 + 8 * 2 / 3 + 8)
# TTR: 4 dims; Hamiltonian 9 (v cos, v sin, two products and a sum, two control terms); 6 as above. Stage 3's arrival
# test reads the ttr slot only where V <= 0 and writes it once per cell, so it is left out of the per-stage bound.
TTR_OPS = 4 * PER_DIM + 9 + 6
TTR_CASES = [('ttr_default', hj_grid.TTR_GRID_SHAPE), ('ttr_refined', (81, 81, 48, 17))]

CASES = [('di_default', 0, hj_grid.DI_GRID_SHAPE, hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI),
         ('at_default', 1, hj_grid.AIRTAXI_GRID_SHAPE, hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI),
         ('di_refined', 0, (81, 81, 41, 41), hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI),
         ('at_refined', 1, (81, 81, 48, 17, 17), hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI)]
SEP = {0: 0.5, 1: 1500 * 0.0003048}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else 'unknown'


def timed(fn, reps=1):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_peak_gbs():
    n = 1 << 29                                  # 4 GiB of float64
    src = torch.empty(n, dtype=torch.float64, device='cuda')
    dst = torch.empty_like(src)
    ms = timed(lambda: dst.copy_(src), reps=10)
    return 2 * 8 * n / (ms * 1e-3) / 1e9


class Eager:
    """The declared scheme as torch eager ops on the GPU (one RK3 step per call)."""

    def __init__(self, lat, alpha, dev='cuda'):
        self.lat, self.alpha = lat, [float(a) for a in alpha]
        nd = len(lat.shape)
        bc = lambda v, d: torch.as_tensor(v, device=dev).view((1,) * d + (-1,) + (1,) * (nd - d - 1))
        self.c = [bc(lat.coords[d], d) for d in range(nd)]
        if lat.dyn == 1:
            self.cth, self.sth = bc(lat.cth, 2), bc(lat.sth, 2)
            va, vb = self.c[3], self.c[4]
            lo2 = torch.full(np.broadcast_shapes(va.shape, vb.shape), HO.AT_AMIN, dtype=torch.float64, device=dev)
            hi2, lo3, hi3 = lo2.clone().fill_(HO.AT_AMAX), lo2.clone(), lo2.clone().fill_(HO.AT_AMAX)
            for cond, which in ((va <= HO.AT_VMIN, 0), (va >= HO.AT_VMAX, 1), (vb <= HO.AT_VMIN, 2), (vb >= HO.AT_VMAX, 3)):
                cond = cond.expand(lo2.shape)
                for arr, val in ((lo2, HO.AT_AMIN), (hi2, HO.AT_AMAX), (lo3, HO.AT_AMIN), (hi3, HO.AT_AMAX)):
                    arr[cond] = val
                (lo2, hi2, lo3, hi3)[which][cond] = 0.0
            self.boxes = (lo2, hi2, lo3, hi3)

    def pad(self, v, axis):
        m = torch.movedim(v, axis, 0)
        n = m.shape[0]
        if self.lat.periodic[axis]:
            idx = torch.as_tensor(np.arange(-3, n + 3) % n, device=v.device)
            return torch.movedim(m[idx], 0, axis)
        sg = lambda x: torch.where(x > 0, 1.0, torch.where(x < 0, -1.0, 0.0)).to(x.dtype)
        g0 = sg(m[0]) * torch.abs(m[1] - m[0])
        gn = sg(m[n - 1]) * torch.abs(m[n - 1] - m[n - 2])
        lo = [m[0] + g0 * float(j) for j in (3, 2, 1)]
        hi = [m[n - 1] + gn * float(j) for j in (1, 2, 3)]
        return torch.movedim(torch.cat([torch.stack(lo), m, torch.stack(hi)]), 0, axis)

    def derivs(self, v, axis):
        p = torch.movedim(self.pad(v, axis), axis, 0)
        n = v.shape[axis]
        D = [(p[j + 1:j + 1 + n] - p[j:j + n]) * self.lat.inv_dx[axis] for j in range(6)]
        return (torch.movedim(HO.weno5(D[0], D[1], D[2], D[3], D[4]), 0, axis),
                torch.movedim(HO.weno5(D[5], D[4], D[3], D[2], D[1]), 0, axis))

    def rate(self, u):
        nd = u.dim()
        pl, pr = zip(*[self.derivs(u, d) for d in range(nd)])
        q = [(pl[d] + pr[d]) * 0.5 for d in range(nd)]
        if self.lat.dyn == 0:
            H = q[0] * self.c[2] + q[1] * self.c[3]
            for a in (q[2], q[3], -q[2], -q[3]):
                H = H + a * torch.where(a < 0, -HO.DI_U, HO.DI_U)
        else:
            x, y = self.c[0], self.c[1]
            f0 = -self.c[3] + self.c[4] * self.cth
            H = q[0] * f0 + q[1] * (self.c[4] * self.sth)
            a = [(q[0] * y + q[1] * (-x)) + q[2] * (-1.0), q[2], q[3], q[4]]
            lo2, hi2, lo3, hi3 = self.boxes
            lo = [-HO.AT_W, -HO.AT_W, lo2, lo3]
            hi = [HO.AT_W, HO.AT_W, hi2, hi3]
            for k in range(4):
                lk = lo[k] if torch.is_tensor(lo[k]) else torch.tensor(lo[k], dtype=torch.float64, device=u.device)
                hk = hi[k] if torch.is_tensor(hi[k]) else torch.tensor(hi[k], dtype=torch.float64, device=u.device)
                H = H + a[k] * torch.where(a[k] < 0, lk, hk)
        diss = self.alpha[0] * ((pr[0] - pl[0]) * 0.5)
        for d in range(1, nd):
            diss = diss + self.alpha[d] * ((pr[d] - pl[d]) * 0.5)
        hh = H + diss
        return torch.clamp(hh, max=0.0)

    def step(self, u, h):
        u1 = u + h * self.rate(u)
        u2 = 0.75 * u + 0.25 * (u1 + h * self.rate(u1))
        return HO.C13 * u + HO.C23 * (u2 + h * self.rate(u2))


def run_ttr(steps, peak):
    lo, hi = hj_grid.TTR_GRID_LO, hj_grid.TTR_GRID_HI
    H = R.DEFAULT_TTR_HORIZON
    out = []
    for name, shape in TTR_CASES:
        cells = int(np.prod(shape))
        alpha, dt = R.ttr_dissipation(shape, lo, hi)
        l = torch.as_tensor(R.ttr_target(shape, lo, hi), device='cuda')
        S = steps
        t1 = timed(lambda: R.solve_ttr(l, lo, hi, S * dt), reps=3)
        t2 = timed(lambda: R.solve_ttr(l, lo, hi, 2 * S * dt), reps=3)
        stage_us = (t2 - t1) * 1e3 / (3 * S)
        rec = dict(what='ttr_solve', case=name, shape=list(shape), cells=cells, dt=dt, alpha=list(alpha),
                   stage_us=round(stage_us, 2), cell_updates_per_s=cells / (3 * stage_us * 1e-6),
                   fp64_ops_per_cell_stage=TTR_OPS, min_bytes_per_cell_stage=round(BYTES, 2),
                   fp64_ops_per_s=TTR_OPS * cells / (stage_us * 1e-6),
                   hbm_share_of_copy_peak=round(BYTES * cells / (stage_us * 1e-6) / (peak * 1e9), 4),
                   horizon=H, steps=math.ceil(H / dt))
        rec['solve_ms'] = round(timed(lambda: R.solve_ttr(l, lo, hi, H), reps=3), 3)
        for k, h in (('unreached_at_H', H), ('unreached_at_2H', 2 * H)):
            ttr = R.solve_ttr(l, lo, hi, h)[0]
            rec[k] = float(torch.isinf(ttr).double().mean())
            if k == 'unreached_at_H':
                rec['ttr_max_finite'] = float(ttr[torch.isfinite(ttr)].max())
        out.append(rec)
        del l
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--out', default=None, help='append the JSON lines to this file as well')
    ap.add_argument('--steps', type=int, default=20, help='RK3 steps S of the per-stage difference')
    ap.add_argument('--eager-max-cells', type=int, default=30_000_000, help='skip the eager baseline above this size')
    ap.add_argument('--ttr', action='store_true', help='time the airtaxi time-to-reach solve instead')
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    info = gpu_info()
    peak = copy_peak_gbs()
    lines = [dict(what='setup', gpu=info, hbm_copy_peak_gbs=round(peak, 1))]
    if a.ttr:
        lines += run_ttr(a.steps, peak)
    for name, dyn, shape, lo, hi in ([] if a.ttr else CASES):
        cells = int(np.prod(shape))
        alpha, dt = R.dissipation(dyn, shape, lo, hi)
        l = torch.as_tensor(R.target(dyn, shape, lo, hi, SEP[dyn]), device='cuda')
        S = a.steps
        t1 = timed(lambda: R.solve(dyn, l, lo, hi, [S * dt]), reps=3)
        t2 = timed(lambda: R.solve(dyn, l, lo, hi, [2 * S * dt]), reps=3)
        stage_us = (t2 - t1) * 1e3 / (3 * S)
        rec = dict(what='solve', case=name, dynamics=dyn, shape=list(shape), cells=cells, dt=dt, alpha=list(alpha),
                   stage_us=round(stage_us, 2), cell_updates_per_s=cells / (3 * stage_us * 1e-6),
                   fp64_ops_per_cell_stage=OPS[dyn], min_bytes_per_cell_stage=round(BYTES, 2),
                   fp64_ops_per_s=OPS[dyn] * cells / (stage_us * 1e-6),
                   hbm_share_of_copy_peak=round(BYTES * cells / (stage_us * 1e-6) / (peak * 1e9), 4))
        if name.endswith('default'):
            H = R.DEFAULT_HORIZON[dyn]
            rec['horizon'] = H
            rec['steps'] = math.ceil(H / dt)
            rec['solve_ms'] = round(timed(lambda: R.solve(dyn, l, lo, hi, [H]), reps=1), 3)
            V = R.solve(dyn, l, lo, hi, [H / 2, H])
            rec['convergence_max_abs_V(H)-V(H/2)'] = float((V[1] - V[0]).abs().max())
            rec['V_range'] = [float(V[1].min()), float(V[1].max())]
        else:
            rec['steps'] = S
            rec['solve_ms'] = round(t1, 3)
        if cells <= a.eager_max_cells:
            eg = Eager(HO.Lattice(dyn, shape, lo, hi), alpha)
            ms = timed(lambda: eg.step(l, dt), reps=3)
            rec['eager_step_ms'] = round(ms, 3)
            rec['kernel_step_ms'] = round(3 * stage_us * 1e-3, 4)
            rec['speedup_vs_eager'] = round(ms / (3 * stage_us * 1e-3), 1)
            ref = R.solve(dyn, l, lo, hi, [dt])[0]
            rec['eager_max_abs_diff'] = float((eg.step(l, dt) - ref).abs().max())
        lines.append(rec)
        del l
        torch.cuda.empty_cache()
    for rec in lines:
        s = json.dumps(rec)
        print(s, flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(s + '\n')


if __name__ == '__main__':
    main()
