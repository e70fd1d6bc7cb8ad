"""The declared HJ reachability scheme in numpy, op for op (test infrastructure: the reference liblsm_b200_hj.so is
checked against; DESIGN.md "HJ value functions").

It restates `hj_reachability`'s default "very_high" method (WENO5 upwind derivatives, global Lax-Friedrichs, TVD-RK3,
`backwards_reachable_tube`) for the filter's relative dynamics (oracle/lsm_oracle.c apply_safety_filter), in float64:

- Lattice: node k of dim d at lo + k * spacing, spacing (hi-lo)/n on periodic dims and (hi-lo)/(n-1) otherwise; C order.
  Double integrator [px, py, vx, vy] (no periodic dim); airtaxi [x_r, y_r, theta_rel (periodic), v_a, v_b].
- WENO5 (Jiang-Peng, Osher-Fedkiw 3.4): D_j = (v[j+1] - v[j]) * (1 / spacing) over the window v[k-3 .. k+3]; the left
  derivative takes (D_0 .. D_4), the right one (D_5 .. D_1); smoothness indicators in the 13/12 and 1/4 forms,
  alpha_j = d_j / (S_j + 1e-6)^2 with d = 0.1 / 0.6 / 0.3 and the result sum(alpha phi) / sum(alpha). Ghost nodes wrap
  on periodic dims; otherwise v[-j] = v[0] + sign(v[0]) |v[1] - v[0]| j and v[n-1+j] = v[n-1] + sign(v[n-1])
  |v[n-1] - v[n-2]| j.
- H(x, p) = p . f(x) + sum_k a_k u*_k with a = p^T G and u*_k = a_k < 0 ? lo_k : hi_k, both agents' controls maximising
  (float32-rounded boxes; the airtaxi speed saturation as written, each test restarting from the unsaturated boxes).
- dV/dtau = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i) / 2). This is hj_reachability's backward solve:
  its Euler step with time_direction = -1 applies the Lax-Friedrichs flux to -H, which makes the dissipation enter
  with a plus sign in tau = -t (upwind: for dV/dtau = c V_x, c > 0 it gives c p+).
- alpha_i = max over nodes |f_i| + sum_k max over nodes |G_ik| max(|lo_k|, |hi_k|) (unsaturated boxes);
  dt = cfl / sum_i(alpha_i / spacing_i); h = min(dt, horizon - tau), tau set to the horizon when it is reached.
- TVD-RK3: u1 = u + h L(u); u2 = 3/4 u + 1/4 (u1 + h L(u1)); u3 = 1/3 u + 2/3 (u2 + h L(u2)).
"""
from __future__ import annotations

import numpy as np

C13, C16, C56, C76, C116 = 1.0 / 3.0, 1.0 / 6.0, 5.0 / 6.0, 7.0 / 6.0, 11.0 / 6.0
C1312, C23, EPS = 13.0 / 12.0, 2.0 / 3.0, 1e-6
DI_U = 0.5
AT_W = float(np.float32(0.1))
AT_AMIN, AT_AMAX = float(np.float32(-0.001)), float(np.float32(0.002))
AT_VMIN, AT_VMAX = 60 * 0.514444 * 0.001, 175 * 0.514444 * 0.001
PERIODIC = {0: (False,) * 4, 1: (False, False, True, False, False)}


def trig(theta):
    """cos and sin of the theta nodes with include/lsm_math.h (the solver's own host evaluation)."""
    import ctypes
    from layered_safe_marl_b200 import _lib
    lib = _lib.load()
    a = np.ascontiguousarray(theta, dtype=np.float64)
    out = []
    for op in (1, 0):
        o = np.empty_like(a)
        _lib.check(lib.lsm_math_eval(op, a.ctypes.data_as(ctypes.c_void_p), None, o.ctypes.data_as(ctypes.c_void_p), a.size),
                   'lsm_math_eval')
        out.append(o)
    return out[0], out[1]


class Lattice:
    def __init__(self, dyn, shape, lo, hi):
        self.dyn, self.shape = int(dyn), tuple(int(s) for s in shape)
        self.periodic = PERIODIC[self.dyn]
        lo, hi = [float(x) for x in lo], [float(x) for x in hi]
        n = self.shape
        self.spacing = [(hi[d] - lo[d]) / float(n[d]) if self.periodic[d] else (hi[d] - lo[d]) / float(n[d] - 1)
                        for d in range(len(n))]
        self.coords = [lo[d] + self.spacing[d] * np.arange(n[d], dtype=np.float64) for d in range(len(n))]
        self.inv_dx = [1.0 / s for s in self.spacing]
        self.cth = self.sth = None
        if self.dyn == 1:
            self.cth, self.sth = trig(self.coords[2])

    def sub(self, starts, stops):
        """The lattice of a sub-block [starts, stops) with this lattice's spacings (for per-cell evaluations)."""
        s = Lattice.__new__(Lattice)
        s.dyn, s.periodic, s.spacing, s.inv_dx = self.dyn, self.periodic, self.spacing, self.inv_dx
        s.shape = tuple(b - a for a, b in zip(starts, stops))
        s.coords = [c[a:b] for c, a, b in zip(self.coords, starts, stops)]
        s.cth = None if self.cth is None else self.cth[starts[2]:stops[2]]
        s.sth = None if self.sth is None else self.sth[starts[2]:stops[2]]
        return s


def dissipation(lat: Lattice, cfl: float = 0.75):
    c = lat.coords
    if lat.dyn == 0:
        alpha = [np.max(np.abs(c[2])), np.max(np.abs(c[3])), DI_U + DI_U, DI_U + DI_U]
    else:
        va = c[3][None, :, None]
        vb = c[4][None, None, :]
        f0 = np.max(np.abs(-va + vb * lat.cth[:, None, None]))
        f1 = np.max(np.abs(vb * lat.sth[:, None, None]))
        a3 = max(abs(AT_AMIN), abs(AT_AMAX))
        alpha = [f0 + AT_W * np.max(np.abs(c[1])), f1 + AT_W * np.max(np.abs(c[0])), AT_W + AT_W, a3, a3]
    alpha = [float(a) for a in alpha]
    s = alpha[0] / lat.spacing[0]
    for d in range(1, len(alpha)):
        s = s + alpha[d] / lat.spacing[d]
    return np.array(alpha), cfl / s


def sign(x):
    return np.where(x > 0.0, 1.0, np.where(x < 0.0, -1.0, 0.0))


def pad(v, axis, periodic):
    """v with 3 ghost nodes on each side of `axis`."""
    m = np.moveaxis(v, axis, 0)
    n = m.shape[0]
    if periodic:
        idx = np.arange(-3, n + 3) % n
        return np.moveaxis(m[idx], 0, axis)
    g0 = sign(m[0]) * np.abs(m[1] - m[0])
    gn = sign(m[n - 1]) * np.abs(m[n - 1] - m[n - 2])
    lo = [m[0] + g0 * float(j) for j in (3, 2, 1)]
    hi = [m[n - 1] + gn * float(j) for j in (1, 2, 3)]
    return np.moveaxis(np.concatenate([np.stack(lo), m, np.stack(hi)]), 0, axis)


def weno5(v1, v2, v3, v4, v5):
    phi1 = (v1 * C13 - v2 * C76) + v3 * C116
    phi2 = (v2 * -C16 + v3 * C56) + v4 * C13
    phi3 = (v3 * C13 + v4 * C56) - v5 * C16
    a = (v1 - 2.0 * v2) + v3; b = (v1 - 4.0 * v2) + 3.0 * v3
    s1 = C1312 * (a * a) + 0.25 * (b * b)
    a = (v2 - 2.0 * v3) + v4; b = v2 - v4
    s2 = C1312 * (a * a) + 0.25 * (b * b)
    a = (v3 - 2.0 * v4) + v5; b = (3.0 * v3 - 4.0 * v4) + v5
    s3 = C1312 * (a * a) + 0.25 * (b * b)
    t1, t2, t3 = s1 + EPS, s2 + EPS, s3 + EPS
    a1, a2, a3 = 0.1 / (t1 * t1), 0.6 / (t2 * t2), 0.3 / (t3 * t3)
    return ((a1 * phi1 + a2 * phi2) + a3 * phi3) / ((a1 + a2) + a3)


def derivs(v, axis, inv_dx, periodic):
    """WENO5 (left, right) derivatives of v along `axis`."""
    p = np.moveaxis(pad(v, axis, periodic), axis, 0)
    n = v.shape[axis]
    D = [(p[j + 1:j + 1 + n] - p[j:j + n]) * inv_dx for j in range(6)]
    left = weno5(D[0], D[1], D[2], D[3], D[4])
    right = weno5(D[5], D[4], D[3], D[2], D[1])
    return np.moveaxis(left, 0, axis), np.moveaxis(right, 0, axis)


def _bcast(vec, d, nd):
    return vec.reshape((1,) * d + (-1,) + (1,) * (nd - d - 1))


def rate(lat: Lattice, u, alpha):
    """L(u) = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i)/2)."""
    nd = u.ndim
    pl, pr = zip(*[derivs(u, d, lat.inv_dx[d], lat.periodic[d]) for d in range(nd)])
    q = [(pl[d] + pr[d]) * 0.5 for d in range(nd)]
    if lat.dyn == 0:
        vx, vy = _bcast(lat.coords[2], 2, nd), _bcast(lat.coords[3], 3, nd)
        H = q[0] * vx + q[1] * vy
        for a in (q[2], q[3], -q[2], -q[3]):
            H = H + a * np.where(a < 0.0, -DI_U, DI_U)
    else:
        x, y = _bcast(lat.coords[0], 0, nd), _bcast(lat.coords[1], 1, nd)
        c, s = _bcast(lat.cth, 2, nd), _bcast(lat.sth, 2, nd)
        va, vb = _bcast(lat.coords[3], 3, nd), _bcast(lat.coords[4], 4, nd)
        f0 = -va + vb * c
        f1 = vb * s
        H = q[0] * f0 + q[1] * f1
        a = [(q[0] * y + q[1] * (-x)) + q[2] * (-1.0), q[2], q[3], q[4]]
        shp = (1, 1, 1, lat.shape[3], lat.shape[4])
        va_b, vb_b = np.broadcast_to(va, shp), np.broadcast_to(vb, shp)
        lo2 = np.full(shp, AT_AMIN); hi2 = np.full(shp, AT_AMAX); lo3 = np.full(shp, AT_AMIN); hi3 = np.full(shp, AT_AMAX)
        for cond, which in ((va_b <= AT_VMIN, 'lo2'), (va_b >= AT_VMAX, 'hi2'), (vb_b <= AT_VMIN, 'lo3'), (vb_b >= AT_VMAX, 'hi3')):
            for arr, val in ((lo2, AT_AMIN), (hi2, AT_AMAX), (lo3, AT_AMIN), (hi3, AT_AMAX)):
                arr[cond] = val
            {'lo2': lo2, 'hi2': hi2, 'lo3': lo3, 'hi3': hi3}[which][cond] = 0.0
        lo = [-AT_W, -AT_W, lo2, lo3]
        hi = [AT_W, AT_W, hi2, hi3]
        for k in range(4):
            H = H + a[k] * np.where(a[k] < 0.0, lo[k], hi[k])
    diss = alpha[0] * ((pr[0] - pl[0]) * 0.5)
    for d in range(1, nd):
        diss = diss + alpha[d] * ((pr[d] - pl[d]) * 0.5)
    hh = H + diss
    return np.where(hh < 0.0, hh, 0.0)


def rk3_step(lat: Lattice, u, alpha, h):
    u1 = u + h * rate(lat, u, alpha)
    u2 = 0.75 * u + 0.25 * (u1 + h * rate(lat, u1, alpha))
    return C13 * u + C23 * (u2 + h * rate(lat, u2, alpha))


def solve(dyn, initial, lo, hi, horizons, cfl=0.75):
    """V(tau) for each tau of `horizons`: float64 (K, *shape)."""
    lat = Lattice(dyn, np.shape(initial), lo, hi)
    alpha, dt = dissipation(lat, cfl)
    u = np.array(initial, dtype=np.float64)
    tau, out = 0.0, []
    for target in horizons:
        target = float(target)
        while tau < target:
            if target - tau <= dt:
                h, tau = target - tau, target
            else:
                h, tau = dt, tau + dt
            u = rk3_step(lat, u, alpha, h)
        out.append(u.copy())
    return np.stack(out)


def step_at(lat: Lattice, u_block, starts, alpha, h):
    """One RK3 step evaluated at the centre of a block cut from the full lattice: exact when the block reaches 9 nodes
    past the centre in every dim or ends at the lattice's own boundary (three stages of a 3-node stencil)."""
    stops = [a + s for a, s in zip(starts, u_block.shape)]
    return rk3_step(lat.sub(starts, stops), u_block, alpha, h)
