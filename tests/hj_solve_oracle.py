"""The declared HJ reachability scheme in numpy, op for op (test infrastructure: the reference every solve of
liblsm_b200_hj.so is checked against; DESIGN.md "HJ value functions" and "Time-to-reach grid", include/lsm_b200_hj.h).

It restates `hj_reachability`'s default "very_high" method (WENO5 upwind derivatives, global Lax-Friedrichs, TVD-RK3,
`backwards_reachable_tube`) for the filter's relative dynamics (oracle/lsm_oracle.c apply_safety_filter), in float64:

- Lattice: node k of dim d at lo + k * spacing, spacing (hi-lo)/n on periodic dims and (hi-lo)/(n-1) otherwise; C order.
  Double integrator [px, py, vx, vy] (no periodic dim); airtaxi [x_r, y_r, theta_rel (periodic), v_a, v_b].
- WENO5 (Jiang-Peng, Osher-Fedkiw 3.4): D_j = (v[j+1] - v[j]) * (1 / spacing) over the window v[k-3 .. k+3]; the left
  derivative takes (D_0 .. D_4), the right one (D_5 .. D_1); smoothness indicators in the 13/12 and 1/4 forms,
  alpha_j = d_j / (S_j + 1e-6)^2 with d = 0.1 / 0.6 / 0.3 and the result sum(alpha phi) / sum(alpha). Ghost nodes wrap
  on periodic dims; otherwise v[-j] = v[0] + sign(v[0]) |v[1] - v[0]| j and v[n-1+j] = v[n-1] + sign(v[n-1])
  |v[n-1] - v[n-2]| j.
- H(x, p) = p . f(x) + sum_k a_k u*_k with a = p^T G (float32-rounded boxes; the airtaxi speed saturation as written,
  each test restarting from the unsaturated boxes). The controls split into the ego's and the other agent's: double
  integrator [ax_e, ay_e | ax_o, ay_o] (k = 0, 1 | 2, 3); airtaxi [w_a, w_b, a_a, a_b] with k = 0, 2 the ego's and
  k = 1, 3 the other's. The ego's controls maximise, u*_k = a_k < 0 ? lo_k : hi_k; the other agent's depend on the game
  of lsm_hj_game_solve: 0 cooperative, maximise as well; 1 adversarial, minimise, u*_k = a_k < 0 ? hi_k : lo_k;
  2 constant, held at 0, their terms dropped from H.
- dV/dtau = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i) / 2). This is hj_reachability's backward solve:
  its Euler step with time_direction = -1 applies the Lax-Friedrichs flux to -H, which makes the dissipation enter
  with a plus sign in tau = -t (upwind: for dV/dtau = c V_x, c > 0 it gives c p+).
- alpha_i = max over nodes |f_i| + sum_k max over nodes |G_ik| max(|lo_k|, |hi_k|) over the controls in play
  (unsaturated boxes): all four in games 0 and 1, the ego's two in game 2; dt = cfl / sum_i(alpha_i / spacing_i);
  h = min(dt, horizon - tau), tau set to the horizon when it is reached.
- TVD-RK3: u1 = u + h L(u); u2 = 3/4 u + 1/4 (u1 + h L(u1)); u3 = 1/3 u + 2/3 (u2 + h L(u2)).

The airtaxi time-to-reach solve (Lattice kind TTR) is the same scheme on a reach problem:
- State [x, y, theta (periodic), v]: one airtaxi relative to its goal, in the goal's frame.
- H(x, p) = p0 (v cos th) + p1 (v sin th) + sum_k a_k (a_k < 0 ? hi_k : lo_k) with a = (p2, p3): the controls
  minimise. Boxes w in +-AT_W, a in [AT_AMIN, AT_AMAX]; v <= AT_VMIN gives a >= 0, v >= AT_VMAX gives a <= 0, each test
  restarting from the unsaturated box.
- alpha = [max |v cos th|, max |v sin th|, AT_W, max(|AT_AMIN|, |AT_AMAX|)] over the nodes.
- First arrival: ttr = 0 where l <= 0, +inf elsewhere; after each RK3 step (tau0, h, start V0, end V1) a cell still at
  +inf with V1 <= 0 takes tau0 + h * (V0 / (V0 - V1)).
"""
from __future__ import annotations

import numpy as np

C13, C16, C56, C76, C116 = 1.0 / 3.0, 1.0 / 6.0, 5.0 / 6.0, 7.0 / 6.0, 11.0 / 6.0
C1312, C23, EPS = 13.0 / 12.0, 2.0 / 3.0, 1e-6
DI_U = 0.5
AT_W = float(np.float32(0.1))
AT_AMIN, AT_AMAX = float(np.float32(-0.001)), float(np.float32(0.002))
AT_VMIN, AT_VMAX = 60 * 0.514444 * 0.001, 175 * 0.514444 * 0.001
TTR = 2                 # the Lattice kind of the time-to-reach solve, next to dynamics 0 and 1
PERIODIC = {0: (False,) * 4, 1: (False, False, True, False, False), TTR: (False, False, True, False)}
COOPERATIVE, ADVERSARIAL, CONSTANT = 0, 1, 2
GAMES = (COOPERATIVE, ADVERSARIAL, CONSTANT)


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
    """The lattice of dynamics 0 (double integrator), 1 (airtaxi) or TTR."""

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
        if self.dyn != 0:
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


def dissipation(lat: Lattice, cfl: float = 0.75, game: int = COOPERATIVE):
    c = lat.coords
    if lat.dyn == 0:
        u = DI_U if game == CONSTANT else DI_U + DI_U
        alpha = [np.max(np.abs(c[2])), np.max(np.abs(c[3])), u, u]
    elif lat.dyn == 1:
        va = c[3][None, :, None]
        vb = c[4][None, None, :]
        f0 = np.max(np.abs(-va + vb * lat.cth[:, None, None]))
        f1 = np.max(np.abs(vb * lat.sth[:, None, None]))
        a3 = max(abs(AT_AMIN), abs(AT_AMAX))
        alpha = [f0 + AT_W * np.max(np.abs(c[1])), f1 + AT_W * np.max(np.abs(c[0])),
                 AT_W if game == CONSTANT else AT_W + AT_W, a3, 0.0 if game == CONSTANT else a3]
    else:
        v = c[3][None, :]
        alpha = [np.max(np.abs(v * lat.cth[:, None])), np.max(np.abs(v * lat.sth[:, None])), AT_W,
                 max(abs(AT_AMIN), abs(AT_AMAX))]
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


def is_other(dyn, k):
    """Whether control k of the avoid Hamiltonian is the other agent's."""
    return k >= 2 if dyn == 0 else k % 2 == 1


def _term(H, dyn, k, a, lo, hi, game):
    if game == COOPERATIVE or not is_other(dyn, k):
        return H + a * np.where(a < 0.0, lo, hi)
    if game == ADVERSARIAL:
        return H + a * np.where(a < 0.0, hi, lo)
    return H


def avoid_hamiltonian(lat: Lattice, q, game: int = COOPERATIVE):
    """H_game(x, q) of dynamics 0 or 1 on the lattice, q = [q0 ..] arrays of its shape."""
    nd = len(q)
    if lat.dyn == 0:
        vx, vy = _bcast(lat.coords[2], 2, nd), _bcast(lat.coords[3], 3, nd)
        H = q[0] * vx + q[1] * vy
        for k, a in enumerate((q[2], q[3], -q[2], -q[3])):
            H = _term(H, 0, k, a, -DI_U, DI_U, game)
        return H
    x, y = _bcast(lat.coords[0], 0, nd), _bcast(lat.coords[1], 1, nd)
    c, s = _bcast(lat.cth, 2, nd), _bcast(lat.sth, 2, nd)
    va, vb = _bcast(lat.coords[3], 3, nd), _bcast(lat.coords[4], 4, nd)
    f0 = -va + vb * c
    f1 = vb * s
    H = q[0] * f0 + q[1] * f1
    a = [(q[0] * y + q[1] * (-x)) + q[2] * (-1.0), q[2], q[3], q[4]]
    # the speed saturation: each test restarts from the unsaturated boxes, so only the last one that holds applies
    shp = (1, 1, 1, lat.shape[3], lat.shape[4])
    va_b, vb_b = np.broadcast_to(va, shp), np.broadcast_to(vb, shp)
    last = np.full(shp, -1)
    for j, cond in enumerate((va_b <= AT_VMIN, va_b >= AT_VMAX, vb_b <= AT_VMIN, vb_b >= AT_VMAX)):
        last = np.where(cond, j, last)
    lo = [-AT_W, -AT_W, np.where(last == 0, 0.0, AT_AMIN), np.where(last == 2, 0.0, AT_AMIN)]
    hi = [AT_W, AT_W, np.where(last == 1, 0.0, AT_AMAX), np.where(last == 3, 0.0, AT_AMAX)]
    for k in range(4):
        H = _term(H, 1, k, a[k], lo[k], hi[k], game)
    return H


def ttr_hamiltonian(lat: Lattice, q):
    """H(x, q) of the time-to-reach solve on the lattice, q = [q0 .. q3] arrays of its shape."""
    c, s = _bcast(lat.cth, 2, 4), _bcast(lat.sth, 2, 4)
    v = _bcast(lat.coords[3], 3, 4)
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


def rate(lat: Lattice, u, alpha, game: int = COOPERATIVE):
    """L(u) = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i)/2), H the TTR Hamiltonian or the avoid one of
    `game`."""
    nd = u.ndim
    pl, pr = zip(*[derivs(u, d, lat.inv_dx[d], lat.periodic[d]) for d in range(nd)])
    q = [(pl[d] + pr[d]) * 0.5 for d in range(nd)]
    H = ttr_hamiltonian(lat, q) if lat.dyn == TTR else avoid_hamiltonian(lat, q, game)
    diss = alpha[0] * ((pr[0] - pl[0]) * 0.5)
    for d in range(1, nd):
        diss = diss + alpha[d] * ((pr[d] - pl[d]) * 0.5)
    hh = H + diss
    return np.where(hh < 0.0, hh, 0.0)


def rk3_step(lat: Lattice, u, alpha, h, game: int = COOPERATIVE):
    u1 = u + h * rate(lat, u, alpha, game)
    u2 = 0.75 * u + 0.25 * (u1 + h * rate(lat, u1, alpha, game))
    return C13 * u + C23 * (u2 + h * rate(lat, u2, alpha, game))


def arrive(ttr, u0, u3, tau0, h):
    """The write-once first-arrival update after one step from u0 to u3 (in place on ttr)."""
    hit = (u3 <= 0.0) & (ttr == np.inf)
    with np.errstate(divide='ignore', invalid='ignore'):
        t = tau0 + h * (u0 / (u0 - u3))
    ttr[hit] = t[hit]


def _solve(lat: Lattice, initial, horizons, cfl, game, ttr=None):
    """V(tau) for each tau of `horizons`: float64 (K, *shape). With `ttr`, the arrival update after every step."""
    alpha, dt = dissipation(lat, cfl, game)
    u = np.array(initial, dtype=np.float64)
    tau, out = 0.0, []
    for horizon in horizons:
        horizon = float(horizon)
        while tau < horizon:
            tau0 = tau
            if horizon - tau <= dt:
                h, tau = horizon - tau, horizon
            else:
                h, tau = dt, tau + dt
            u3 = rk3_step(lat, u, alpha, h, game)
            if ttr is not None:
                arrive(ttr, u, u3, tau0, h)
            u = u3
        out.append(u.copy())
    return np.stack(out)


def solve(dyn, initial, lo, hi, horizons, cfl=0.75, game: int = COOPERATIVE):
    """V(tau) of `game` for each tau of `horizons`: float64 (K, *shape)."""
    return _solve(Lattice(dyn, np.shape(initial), lo, hi), initial, horizons, cfl, game)


def solve_ttr(target, lo, hi, horizon, cfl=0.75):
    """The time-to-reach solve: (ttr, V(horizon)), float64 arrays of the target's shape."""
    ttr = np.where(np.asarray(target) <= 0.0, 0.0, np.inf)
    V = _solve(Lattice(TTR, np.shape(target), lo, hi), target, [horizon], cfl, COOPERATIVE, ttr)[0]
    return ttr, V


def step_at(lat: Lattice, u_block, starts, alpha, h, game: int = COOPERATIVE):
    """One RK3 step evaluated at the centre of a block cut from the full lattice: exact when the block reaches 9 nodes
    past the centre in every dim or ends at the lattice's own boundary (three stages of a 3-node stencil)."""
    stops = [a + s for a, s in zip(starts, u_block.shape)]
    return rk3_step(lat.sub(starts, stops), u_block, alpha, h, game)
