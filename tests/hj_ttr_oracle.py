"""The declared airtaxi time-to-reach scheme in numpy, op for op (test infrastructure: the reference the TTR solve of
liblsm_b200_hj.so is checked against; DESIGN.md "Time-to-reach grid", include/lsm_b200_hj.h).

The WENO5 derivatives, ghosts, the cos / sin of the theta nodes and the TVD-RK3 combinations are those of
tests/hj_solve_oracle.py, imported from it. What differs:

- State [x, y, theta (periodic), v]: one airtaxi relative to its goal, in the goal's frame.
- H(x, p) = p0 (v cos th) + p1 (v sin th) + sum_k a_k (a_k < 0 ? hi_k : lo_k) with a = (p2, p3): the controls
  minimise (a reach problem). Boxes w in +-AT_W, a in [AT_AMIN, AT_AMAX] (float32-rounded); v <= AT_VMIN gives a >= 0,
  v >= AT_VMAX gives a <= 0, each test restarting from the unsaturated box.
- dV/dtau = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i) / 2), the avoid solve's sign.
- alpha = [max |v cos th|, max |v sin th|, AT_W, max(|AT_AMIN|, |AT_AMAX|)] over the nodes; dt = cfl / sum(alpha / dx).
- First arrival: ttr = 0 where l <= 0, +inf elsewhere; after each RK3 step (tau0, h, start V0, end V1) a cell still at
  +inf with V1 <= 0 takes tau0 + h * (V0 / (V0 - V1)).
"""
from __future__ import annotations

import numpy as np

from hj_solve_oracle import AT_AMAX, AT_AMIN, AT_VMAX, AT_VMIN, AT_W, C13, C23, derivs, trig

PERIODIC = (False, False, True, False)


class Lattice:
    def __init__(self, shape, lo, hi):
        self.shape = tuple(int(s) for s in shape)
        self.periodic = PERIODIC
        lo, hi = [float(x) for x in lo], [float(x) for x in hi]
        n = self.shape
        self.spacing = [(hi[d] - lo[d]) / float(n[d]) if PERIODIC[d] else (hi[d] - lo[d]) / float(n[d] - 1)
                        for d in range(4)]
        self.coords = [lo[d] + self.spacing[d] * np.arange(n[d], dtype=np.float64) for d in range(4)]
        self.inv_dx = [1.0 / s for s in self.spacing]
        self.cth, self.sth = trig(self.coords[2])

    def sub(self, starts, stops):
        """The lattice of a sub-block [starts, stops) with this lattice's spacings (for per-cell evaluations)."""
        s = Lattice.__new__(Lattice)
        s.periodic, s.spacing, s.inv_dx = self.periodic, self.spacing, self.inv_dx
        s.shape = tuple(b - a for a, b in zip(starts, stops))
        s.coords = [c[a:b] for c, a, b in zip(self.coords, starts, stops)]
        s.cth, s.sth = self.cth[starts[2]:stops[2]], self.sth[starts[2]:stops[2]]
        return s


def dissipation(lat: Lattice, cfl: float = 0.75):
    v = lat.coords[3][None, :]
    alpha = [float(np.max(np.abs(v * lat.cth[:, None]))), float(np.max(np.abs(v * lat.sth[:, None]))), AT_W,
             max(abs(AT_AMIN), abs(AT_AMAX))]
    s = alpha[0] / lat.spacing[0]
    for d in range(1, 4):
        s = s + alpha[d] / lat.spacing[d]
    return np.array(alpha), cfl / s


def _bcast(vec, d):
    return vec.reshape((1,) * d + (-1,) + (1,) * (3 - d))


def hamiltonian(lat: Lattice, q):
    """H(x, q) on the lattice, q = [q0 .. q3] arrays of its shape."""
    c, s = _bcast(lat.cth, 2), _bcast(lat.sth, 2)
    v = _bcast(lat.coords[3], 3)
    f0 = v * c
    f1 = v * s
    H = q[0] * f0 + q[1] * f1
    lo3 = np.full(v.shape, AT_AMIN); hi3 = np.full(v.shape, AT_AMAX)
    for cond, which in ((v <= AT_VMIN, 'lo3'), (v >= AT_VMAX, 'hi3')):
        lo3[cond] = AT_AMIN; hi3[cond] = AT_AMAX
        {'lo3': lo3, 'hi3': hi3}[which][cond] = 0.0
    a = [q[2], q[3]]
    lo = [-AT_W, lo3]
    hi = [AT_W, hi3]
    for k in range(2):
        H = H + a[k] * np.where(a[k] < 0.0, hi[k], lo[k])
    return H


def rate(lat: Lattice, u, alpha):
    """L(u) = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i)/2)."""
    pl, pr = zip(*[derivs(u, d, lat.inv_dx[d], lat.periodic[d]) for d in range(4)])
    q = [(pl[d] + pr[d]) * 0.5 for d in range(4)]
    H = hamiltonian(lat, q)
    diss = alpha[0] * ((pr[0] - pl[0]) * 0.5)
    for d in range(1, 4):
        diss = diss + alpha[d] * ((pr[d] - pl[d]) * 0.5)
    hh = H + diss
    return np.where(hh < 0.0, hh, 0.0)


def rk3_step(lat: Lattice, u, alpha, h):
    u1 = u + h * rate(lat, u, alpha)
    u2 = 0.75 * u + 0.25 * (u1 + h * rate(lat, u1, alpha))
    return C13 * u + C23 * (u2 + h * rate(lat, u2, alpha))


def arrive(ttr, u0, u3, tau0, h):
    """The write-once first-arrival update after one step from u0 to u3 (in place on ttr)."""
    hit = (u3 <= 0.0) & (ttr == np.inf)
    with np.errstate(divide='ignore', invalid='ignore'):
        t = tau0 + h * (u0 / (u0 - u3))
    ttr[hit] = t[hit]


def solve(target, lo, hi, horizon, cfl=0.75):
    """(ttr, V(horizon)), float64 arrays of the target's shape."""
    lat = Lattice(np.shape(target), lo, hi)
    alpha, dt = dissipation(lat, cfl)
    u = np.array(target, dtype=np.float64)
    ttr = np.where(u <= 0.0, 0.0, np.inf)
    tau, horizon = 0.0, float(horizon)
    while tau < horizon:
        tau0 = tau
        if horizon - tau <= dt:
            h, tau = horizon - tau, horizon
        else:
            h, tau = dt, tau + dt
        u3 = rk3_step(lat, u, alpha, h)
        arrive(ttr, u, u3, tau0, h)
        u = u3
    return ttr, u


def step_at(lat: Lattice, u_block, starts, alpha, h):
    """One RK3 step evaluated at the centre of a block cut from the full lattice (exact when the block reaches 9 nodes
    past the centre in every dim or ends at the lattice's own boundary)."""
    stops = [a + s for a, s in zip(starts, u_block.shape)]
    return rk3_step(lat.sub(starts, stops), u_block, alpha, h)
