"""The HJ games of lsm_hj_game_solve in numpy, op for op (test infrastructure; include/lsm_b200_hj.h, DESIGN.md "HJ
value functions").

The scheme is tests/hj_solve_oracle.py's - its Lattice, ghost padding, WENO5 and derivatives are used as they are -
with one Hamiltonian per game. The controls split into the ego's and the other agent's: double integrator
[ax_e, ay_e | ax_o, ay_o] (k = 0, 1 | 2, 3); airtaxi [w_a, w_b, a_a, a_b] with k = 0, 2 the ego's and k = 1, 3 the
other's. The ego's controls maximise (u*_k = a_k < 0 ? lo_k : hi_k). The other agent's:

- 0 cooperative: maximise as well (hj_solve_oracle.rate);
- 1 adversarial: minimise, u*_k = a_k < 0 ? hi_k : lo_k;
- 2 constant: held at 0, their terms dropped from H.

The boxes, including the airtaxi speed saturation of v_b, are the cooperative game's. Lax-Friedrichs alpha sums over
the controls in play: the cooperative alpha for games 0 and 1; for game 2 [max|vx|, max|vy|, 0.5, 0.5] (double
integrator) and [f0 + W max|y|, f1 + W max|x|, W, max(|a_min|, |a_max|), 0] (airtaxi).
"""
from __future__ import annotations

import numpy as np

import hj_solve_oracle as HO
from hj_solve_oracle import AT_AMAX, AT_AMIN, AT_VMAX, AT_VMIN, AT_W, C13, C23, DI_U, Lattice, _bcast, derivs  # noqa: F401

COOPERATIVE, ADVERSARIAL, CONSTANT = 0, 1, 2
GAMES = (COOPERATIVE, ADVERSARIAL, CONSTANT)


def is_other(dyn, k):
    """Whether control k of the Hamiltonian is the other agent's."""
    return k >= 2 if dyn == 0 else k % 2 == 1


def dissipation(lat: Lattice, cfl: float = 0.75, game: int = COOPERATIVE):
    alpha, _ = HO.dissipation(lat, cfl)
    alpha = [float(a) for a in alpha]
    if game == CONSTANT:
        if lat.dyn == 0:
            alpha[2], alpha[3] = DI_U, DI_U
        else:
            alpha[2], alpha[4] = AT_W, 0.0
    s = alpha[0] / lat.spacing[0]
    for d in range(1, len(alpha)):
        s = s + alpha[d] / lat.spacing[d]
    return np.array(alpha), cfl / s


def _term(H, dyn, k, a, lo, hi, game):
    if game == COOPERATIVE or not is_other(dyn, k):
        return H + a * np.where(a < 0.0, lo, hi)
    if game == ADVERSARIAL:
        return H + a * np.where(a < 0.0, hi, lo)
    return H


def rate(lat: Lattice, u, alpha, game: int = COOPERATIVE):
    """L(u) = min(0, H_game(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i)/2)."""
    nd = u.ndim
    pl, pr = zip(*[derivs(u, d, lat.inv_dx[d], lat.periodic[d]) for d in range(nd)])
    q = [(pl[d] + pr[d]) * 0.5 for d in range(nd)]
    if lat.dyn == 0:
        vx, vy = _bcast(lat.coords[2], 2, nd), _bcast(lat.coords[3], 3, nd)
        H = q[0] * vx + q[1] * vy
        for k, a in enumerate((q[2], q[3], -q[2], -q[3])):
            H = _term(H, 0, k, a, -DI_U, DI_U, game)
    else:
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
    diss = alpha[0] * ((pr[0] - pl[0]) * 0.5)
    for d in range(1, nd):
        diss = diss + alpha[d] * ((pr[d] - pl[d]) * 0.5)
    hh = H + diss
    return np.where(hh < 0.0, hh, 0.0)


def rk3_step(lat: Lattice, u, alpha, h, game: int = COOPERATIVE):
    u1 = u + h * rate(lat, u, alpha, game)
    u2 = 0.75 * u + 0.25 * (u1 + h * rate(lat, u1, alpha, game))
    return C13 * u + C23 * (u2 + h * rate(lat, u2, alpha, game))


def solve(dyn, initial, lo, hi, horizons, cfl=0.75, game: int = COOPERATIVE):
    """V(tau) of `game` for each tau of `horizons`: float64 (K, *shape)."""
    lat = Lattice(dyn, np.shape(initial), lo, hi)
    alpha, dt = dissipation(lat, cfl, game)
    u = np.array(initial, dtype=np.float64)
    tau, out = 0.0, []
    for target in horizons:
        target = float(target)
        while tau < target:
            if target - tau <= dt:
                h, tau = target - tau, target
            else:
                h, tau = dt, tau + dt
            u = rk3_step(lat, u, alpha, h, game)
        out.append(u.copy())
    return np.stack(out)
