"""The HJ reachability solver (liblsm_b200_hj.so, layered_safe_marl_b200.reachability) against the differential game it
solves. Every reference here is written independently of the solver and of its numpy restatement
(tests/hj_solve_oracle.py), so a misreading the two share - a sign of the airtaxi rotation term or of f1, the speed
saturation rule - fails here although the bit-identity tests pass.

1. The Hamiltonian, cell by cell. The relative dynamics are derived from absolute-frame agents (point masses; unicycles
   x' = v cos th, y' = v sin th, th' = w, v' = a) composed with the filter's relative-state map and differentiated by
   central differences; H_ref(x, c) is the maximum of c . r' over the 16 corners of the joint control box. For affine
   initial values u = c . x + b, one step of h = 1e-7 gives (V(h) - u) / h = min(0, H_ref) at every cell 3 nodes away
   from the non-periodic edges and the theta seam: WENO5 returns the slope exactly there and the Lax-Friedrichs
   dissipation vanishes. CPU on the oracle, GPU on the kernel. The dissipation coefficients bound |r'_i|.
2. Closed-form tubes of rotated slabs |n . p| - r, which exercise all four double-integrator dims.
3. Computed grids read through SafetyFilter.values against simulated trajectories: no admissible control ends with a
   smaller distance margin than V promises (V is a supremum), and choosing the corner that maximises V attains it.
"""
import math
import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'tests'))

import hj_solve_oracle as HO  # noqa: E402
from layered_safe_marl_b200 import hj_grid  # noqa: E402
from layered_safe_marl_b200 import reachability as R  # noqa: E402
from layered_safe_marl_b200.config import AirTaxiConfig as ATC, DoubleIntegratorConfig as DIC  # noqa: E402

gpu = pytest.mark.gpu
DI_LAT = (hj_grid.DI_GRID_SHAPE, hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI)
AT_LAT = (hj_grid.AIRTAXI_GRID_SHAPE, hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI)
PERIODIC = {0: (False,) * 4, 1: (False, False, True, False, False)}

# ----------------------------------------------------------------------------------------------------------------------
# Reference dynamics
# ----------------------------------------------------------------------------------------------------------------------
# control boxes of apply_safety_filter (oracle/lsm_oracle.c): float32-rounded bounds
F32 = lambda x: float(np.float32(x))  # noqa: E731
DI_A = F32(DIC.ACCELX_MAX)
AT_W, AT_AMIN, AT_AMAX = F32(ATC.ANGULAR_RATE_MAX), F32(ATC.ACCEL_MIN), F32(ATC.ACCEL_MAX)
V_MIN, V_MAX = ATC.V_MIN, ATC.V_MAX
CD_STEP = 1e-4          # central-difference step of the relative-state derivative (s)


def _rel(dyn, ego, oth):
    """The filter's relative state of absolute (..., 4) states: ego - other (double integrator); the rotation form of
    at_relative_state (oracle/lsm_oracle.c) - the other's position in the ego's frame, the relative heading, both
    speeds (airtaxi)."""
    if dyn == 0:
        return ego - oth
    ddx, ddy = oth[..., 0] - ego[..., 0], oth[..., 1] - ego[..., 1]
    ce, se = np.cos(ego[..., 2]), np.sin(ego[..., 2])
    return np.stack([ddx * ce + ddy * se, ddy * ce - ddx * se, oth[..., 2] - ego[..., 2], ego[..., 3], oth[..., 3]], -1)


def _abs_rate(dyn, s, c0, c1):
    """Time derivative of an absolute state: point mass (x, y, vx, vy) under (ax, ay) = (c0, c1); unicycle
    (x, y, theta, v) under (w, a) = (c0, c1)."""
    if dyn == 0:
        return np.stack([s[..., 2], s[..., 3], c0, c1], -1)
    return np.stack([s[..., 3] * np.cos(s[..., 2]), s[..., 3] * np.sin(s[..., 2]), c0, c1], -1)


def _split(dyn, u):
    """The joint control (..., 4) in the filter's column order -> ((ego c0, c1), (other c0, c1)). Double integrator
    [ax_e, ay_e, ax_o, ay_o]; airtaxi [w_a, w_b, a_a, a_b] (a = ego, b = other)."""
    if dyn == 0:
        return (u[..., 0], u[..., 1]), (u[..., 2], u[..., 3])
    return (u[..., 0], u[..., 2]), (u[..., 1], u[..., 3])


def _rel_rate(dyn, ego, oth, u):
    """dr/dt of the relative state under joint control u, by central difference of the absolute motion."""
    (e0, e1), (o0, o1) = _split(dyn, u)
    de, do = _abs_rate(dyn, ego, e0, e1), _abs_rate(dyn, oth, o0, o1)
    plus = _rel(dyn, ego + CD_STEP * de, oth + CD_STEP * do)
    minus = _rel(dyn, ego - CD_STEP * de, oth - CD_STEP * do)
    return (plus - minus) / (2.0 * CD_STEP)


def _abs_pair(dyn, r, rng):
    """Absolute (ego, other) states whose relative state is r (..., nd): a seeded other (double integrator) or a seeded
    ego position and heading (airtaxi)."""
    shp = r.shape[:-1]
    if dyn == 0:
        oth = np.stack([rng.uniform(-3, 3, shp), rng.uniform(-3, 3, shp), rng.uniform(-0.5, 0.5, shp),
                        rng.uniform(-0.5, 0.5, shp)], -1)
        return oth + r, oth
    th = rng.uniform(-math.pi, math.pi, shp)
    ce, se = np.cos(th), np.sin(th)
    ex, ey = rng.uniform(-3, 3, shp), rng.uniform(-3, 3, shp)
    ego = np.stack([ex, ey, th, r[..., 3]], -1)
    oth = np.stack([ex + r[..., 0] * ce - r[..., 1] * se, ey + r[..., 0] * se + r[..., 1] * ce, th + r[..., 2],
                    r[..., 4]], -1)
    return ego, oth


def _boxes(dyn, r):
    """(lo, hi) of the joint control box at relative states r (..., nd), each (..., 4). Airtaxi: the speed saturation
    of apply_safety_filter (oracle/lsm_oracle.c) - an ego at or below V_MIN may not decelerate, at or above V_MAX may
    not accelerate, likewise the other. That reference restarts every test from the unsaturated box, so only the LAST
    condition that holds (in the order ego <= V_MIN, ego >= V_MAX, other <= V_MIN, other >= V_MAX) saturates; with both
    speeds saturated the ego's bound is NOT applied. This is a quirk of the reference, reproduced here on purpose: the
    solver's Hamiltonian is the reference's."""
    shp = r.shape[:-1]
    if dyn == 0:
        return np.full(shp + (4,), -DI_A), np.full(shp + (4,), DI_A)
    last = np.full(shp, -1)
    for k, cond in enumerate((r[..., 3] <= V_MIN, r[..., 3] >= V_MAX, r[..., 4] <= V_MIN, r[..., 4] >= V_MAX)):
        last = np.where(cond, k, last)
    lo = np.stack([np.full(shp, -AT_W), np.full(shp, -AT_W), np.where(last == 0, 0.0, AT_AMIN),
                   np.where(last == 2, 0.0, AT_AMIN)], -1)
    hi = np.stack([np.full(shp, AT_W), np.full(shp, AT_W), np.where(last == 1, 0.0, AT_AMAX),
                   np.where(last == 3, 0.0, AT_AMAX)], -1)
    return lo, hi


def _corner_rates(dyn, r, rng, saturate=True):
    """r' at the 16 corners of the control box: (16, ..., nd)."""
    ego, oth = _abs_pair(dyn, r, rng)
    lo, hi = _boxes(dyn, r) if saturate else _boxes(dyn, np.full_like(r, 0.5 * (V_MIN + V_MAX)))
    out = []
    for k in range(16):
        bits = np.array([(k >> j) & 1 for j in range(4)], bool)
        out.append(_rel_rate(dyn, ego, oth, np.where(bits, hi, lo)))
    return np.stack(out)


# ----------------------------------------------------------------------------------------------------------------------
# 1. The Hamiltonian, cell by cell
# ----------------------------------------------------------------------------------------------------------------------
PROBE_H = 1e-7
EDGE = 3                # nodes kept away from non-periodic edges and the theta seam


def _speed_axis():
    """13 speed nodes, 3 past V_MIN and V_MAX on each side, with node 3 bit-equal to V_MIN and node 9 bit-equal to
    V_MAX (the lattice's own lo + k (hi - lo) / (n - 1)): the saturated speeds are probed cells, and the <= / >= tests
    see their boundary value."""
    lo, hi, n = 0.0012861100000000002, 0.11960823, 13
    return lo, hi, n


def _probe_lattices():
    slo, shi, sn = _speed_axis()
    return {
        0: [((11, 11, 15, 15), DI_LAT[1], DI_LAT[2])],
        # positions within +-0.2 km: the drift dominates the turn terms, so H < 0 at about half the cells
        1: [((11, 11, 12, sn, sn), (-0.2, -0.2, -math.pi, slo, slo), (0.2, 0.2, math.pi, shi, shi))],
    }


ODD_LATTICES = {
    0: ((13, 10, 17, 11), (-3.0, -4.0, -1.1, -1.3), (0.9, 2.5, 1.0, 1.1)),
    1: ((10, 13, 11, 13, 13), (-0.15, -0.25, -math.pi, _speed_axis()[0], _speed_axis()[0]),
        (0.25, 0.15, math.pi, _speed_axis()[1], _speed_axis()[1])),
}


# Probe gradients c: mixed signs, some components zero. The control terms of H are >= 0 (|.| of the switching functions
# times the box), so the drift components are the large ones: H < 0 at 28-59 % of the probed cells of each. Airtaxi:
# small theta components (each agent's turn term is W |c2|), speed components large enough that the accelerations
# (~2e-3 km/s^2) weigh far above the 1e-6 tolerance.
PROBE_C = {
    0: [(0.8, -0.5, 0.1, -0.05), (-0.6, 0.0, 0.12, 0.0), (0.0, 1.1, 0.0, -0.2), (-0.4, 0.9, -0.15, 0.1)],
    1: [(1.0, -0.6, 0.02, 8.0, -6.0), (0.0, 1.2, 0.0, -7.0, 5.0), (0.9, 0.7, -0.02, -5.0, 0.0),
        (0.7, -1.1, 0.0, 10.0, -10.0)],
}


def _probe_c(dyn, k):
    return np.array(PROBE_C[dyn][k], dtype=np.float64)


def _coords(dyn, shape, lo, hi):
    g = hj_grid.HjGrid(lo=np.asarray(lo, np.float64), hi=np.asarray(hi, np.float64), shape=tuple(shape),
                       periodic=PERIODIC[dyn], values=None)
    return g.coordinate_vectors()


def _probe(dyn, shape, lo, hi, c, solve):
    """Solve one step of PROBE_H from u = c . x + b; compare on the interior cells. Returns (rate, H_ref, r, u, V) over
    the interior cells (rate = (V - u) / h)."""
    vecs = _coords(dyn, shape, lo, hi)
    X = np.stack(np.meshgrid(*vecs, indexing='ij'), -1)
    b = 0.3
    u = X @ c + b
    V = solve(u)
    inner = tuple(slice(EDGE, n - EDGE) for n in shape)
    r, ui, Vi = X[inner].reshape(-1, len(shape)), u[inner].ravel(), V[inner].ravel()
    rates = _corner_rates(dyn, r, np.random.default_rng(5))
    H = np.max(rates @ c, axis=0)
    return (Vi - ui) / PROBE_H, H, r, ui, Vi


def _check_probe(dyn, shape, lo, hi, c, solve):
    rate, H, r, u, V = _probe(dyn, shape, lo, hi, c, solve)
    scale = np.abs(H).max()
    tol = 64 * np.finfo(np.float64).eps * np.abs(u).max() / PROBE_H + 1e-6 * scale
    err = np.abs(rate - np.minimum(H, 0.0))
    neg = H < 0
    print(f"dyn {dyn} {shape} c={np.round(c, 3)}: {r.shape[0]} cells, H < 0 at {neg.mean():.0%}, |H| <= {scale:.3e}, "
          f"max |(V - u)/h - min(0, H_ref)| = {err.max():.3e} (tol {tol:.3e})")
    assert 0.2 < neg.mean() < 0.9, "the probe needs cells on both sides of H = 0"
    i = int(np.argmax(err))
    assert err.max() <= tol, f"cell {r[i]}: (V - u)/h = {rate[i]!r}, min(0, H_ref) = {min(H[i], 0.0)!r}"
    # where the game leaves the cell alone, V(h) is u up to the RK3 combinations' rounding
    still = H > 1e-6 * scale
    assert (np.abs(V - u)[still] <= 4 * np.spacing(np.abs(u[still]))).all()
    return H, r


def _assert_saturation_cases(H, r):
    """Every saturation case of _boxes occurs among the cells the game moves (H_ref < 0)."""
    neg = H < 0
    va, vb = r[neg, 3], r[neg, 4]
    assert (va == V_MIN).any() and (va == V_MAX).any() and (vb == V_MIN).any() and (vb == V_MAX).any()
    free = lambda v: (v > V_MIN) & (v < V_MAX)  # noqa: E731
    for what, m in (('ego <= V_MIN', (va <= V_MIN) & free(vb)), ('ego >= V_MAX', (va >= V_MAX) & free(vb)),
                    ('other <= V_MIN', free(va) & (vb <= V_MIN)), ('other >= V_MAX', free(va) & (vb >= V_MAX)),
                    ('both saturated', ((va <= V_MIN) | (va >= V_MAX)) & ((vb <= V_MIN) | (vb >= V_MAX)))):
        assert m.any(), what


def test_probe_lattice_hits_the_speed_bounds_bit_for_bit():
    for lat in (_probe_lattices()[1][0], ODD_LATTICES[1]):
        shape, lo, hi = lat
        for d in (3, 4):
            v = _coords(1, shape, lo, hi)[d]
            assert v[EDGE] == V_MIN and v[-1 - EDGE] == V_MAX, (d, v[EDGE], v[-1 - EDGE])
            assert (v[:EDGE] < V_MIN).all() and (v[-EDGE:] > V_MAX).all()
    for d in (3, 4):    # the same lattice must also agree with the oracle's and the solver's node formula
        o = HO.Lattice(1, _probe_lattices()[1][0][0], *_probe_lattices()[1][0][1:]).coords[d]
        assert o[EDGE] == V_MIN and o[-1 - EDGE] == V_MAX


def test_reference_rates_match_the_written_relative_dynamics():
    """The central-difference rates are the relative dynamics of DESIGN.md "HJ value functions": double integrator
    r' = (vx, vy, ax_e - ax_o, ay_e - ay_o); airtaxi r' = (-v_a + v_b cos th + w_a y, v_b sin th - w_a x, w_b - w_a,
    a_a, a_b)."""
    rng = np.random.default_rng(11)
    for dyn in (0, 1):
        nd = 4 if dyn == 0 else 5
        r = rng.uniform(-1, 1, (500, nd))
        if dyn == 1:
            r[:, 2] *= math.pi
            r[:, 3:] = rng.uniform(V_MIN, V_MAX, (500, 2))
        u = rng.uniform(-1, 1, (500, 4)) * (DI_A if dyn == 0 else np.array([AT_W, AT_W, AT_AMAX, AT_AMAX]))
        ego, oth = _abs_pair(dyn, r, rng)
        got = _rel_rate(dyn, ego, oth, u)
        if dyn == 0:
            want = np.stack([r[:, 2], r[:, 3], u[:, 0] - u[:, 2], u[:, 1] - u[:, 3]], -1)
        else:
            x, y, th, va, vb = r.T
            want = np.stack([-va + vb * np.cos(th) + u[:, 0] * y, vb * np.sin(th) - u[:, 0] * x, u[:, 1] - u[:, 0],
                             u[:, 2], u[:, 3]], -1)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-9)


@pytest.mark.parametrize('seed', [0, 1, 2, 3])
@pytest.mark.parametrize('dyn', [0, 1])
def test_oracle_hamiltonian_cell_by_cell(dyn, seed):
    c = _probe_c(dyn, seed)
    for shape, lo, hi in _probe_lattices()[dyn]:
        H, r = _check_probe(dyn, shape, lo, hi, c, lambda u: HO.solve(dyn, u, lo, hi, [PROBE_H])[0])
        if dyn == 1:
            _assert_saturation_cases(H, r)


@pytest.mark.parametrize('dyn', [0, 1])
def test_dissipation_bounds_every_rate(dyn):
    """Global Lax-Friedrichs is monotone only if alpha_i >= max |r'_i| over the lattice and the control box (the
    unsaturated box, which contains every saturated one). The double integrator's bound is attained exactly: the
    coefficients are the maxima themselves. So are the airtaxi's when the lattice has the nodes theta = -pi, +-pi/2
    where the drift and the turn term peak together (the default lattice)."""
    if dyn == 0:
        lats = [DI_LAT, ((9, 11, 7, 5), (-2.0, -3.0, -0.4, -1.3), (1.0, 3.0, 0.9, 0.2))]
    else:
        lats = [((9, 9) + AT_LAT[0][2:], AT_LAT[1], AT_LAT[2]), _probe_lattices()[1][0], ODD_LATTICES[1]]
    for i, (shape, lo, hi) in enumerate(lats):
        alpha, _ = R.dissipation(dyn, shape, lo, hi)
        X = np.stack(np.meshgrid(*_coords(dyn, shape, lo, hi), indexing='ij'), -1).reshape(-1, len(shape))
        need = np.abs(_corner_rates(dyn, X, np.random.default_rng(6), saturate=False)).max(axis=(0, 1))
        print(f"dyn {dyn} {shape}: alpha {alpha}, max |r'| {need}")
        assert (alpha >= need * (1 - 1e-9)).all(), (alpha, need)
        if dyn == 0 or i == 0:
            np.testing.assert_allclose(alpha, need, rtol=1e-9, atol=0)


# ----------------------------------------------------------------------------------------------------------------------
# 2. Closed-form tubes of rotated slabs
# ----------------------------------------------------------------------------------------------------------------------
SLAB_R, SLAB_T = 0.5, 2.0


def _rotated_slab(shape, phi_deg):
    """l = |s| - r with s = n . p, n = (cos phi, sin phi), its tube max(|s| - [s w < 0] w^2 / (2 A), 0) - r with
    w = n . v and A = |cos phi| + |sin phi| (each axis of the relative acceleration is bounded by 1, so A bounds n . a),
    and the comparison mask: |p_i| <= 3.5 and |v_i| <= 0.8 on every axis, 2 cells off both kinks."""
    phi = math.radians(phi_deg)
    n = np.array([math.cos(phi), math.sin(phi)])
    n[np.abs(n) < 1e-12] = 0.0              # exact axes at 0 and 90 degrees
    A = np.abs(n).sum()
    vecs = _coords(0, shape, DI_LAT[1], DI_LAT[2])
    px, py, vx, vy = np.meshgrid(*vecs, indexing='ij')
    s, w = n[0] * px + n[1] * py, n[0] * vx + n[1] * vy
    l = np.abs(s) - SLAB_R
    exact = np.maximum(np.abs(s) - (s * w < 0) * w ** 2 / (2 * A), 0.0) - SLAB_R
    sp = [v[1] - v[0] for v in vecs]
    ds = abs(n[0]) * sp[0] + abs(n[1]) * sp[1]
    dw = abs(n[0]) * sp[2] + abs(n[1]) * sp[3]
    kink = (np.abs(np.abs(s) - w ** 2 / (2 * A)) < 2 * ds + 2 * dw * np.abs(w) / A) | (np.abs(s) < 2 * ds)
    inside = (np.abs(px) <= 3.5) & (np.abs(py) <= 3.5) & (np.abs(vx) <= 0.8) & (np.abs(vy) <= 0.8)
    return l, exact, inside & ~kink


def _slab_error(V, l, exact, mask, phi):
    assert (V <= l + 4 * np.spacing(np.abs(l))).all()
    if phi == 90:       # a function of (py, vy) alone: bitwise constant along px and vx
        assert np.array_equal(V.view(np.int64), np.broadcast_to(V[:1, :, :1, :], V.shape).view(np.int64))
    return float(np.abs(V - exact)[mask].max())


@pytest.mark.parametrize('phi', [0, 30, 45, 90])
def test_oracle_meets_the_rotated_slab(phi):
    shape = (21, 21, 11, 11)
    l, exact, mask = _rotated_slab(shape, phi)
    V = HO.solve(0, l, DI_LAT[1], DI_LAT[2], [SLAB_T])[0]
    err = _slab_error(V, l, exact, mask, phi)
    print(f"rotated slab phi={phi} {shape}: max |V - V*| = {err * 1e3:.2f} mm over {int(mask.sum())} cells")
    assert err < 0.02


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
def _cuda(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device='cuda')


def _gpu_solve(dyn, lo, hi, horizon):
    return lambda u: R.solve(dyn, _cuda(u), lo, hi, [horizon])[0].cpu().numpy()


@gpu
@pytest.mark.parametrize('seed', [0, 1, 2, 3])
@pytest.mark.parametrize('dyn', [0, 1])
def test_solver_hamiltonian_cell_by_cell(dyn, seed):
    c = _probe_c(dyn, seed)
    for i, (shape, lo, hi) in enumerate(_probe_lattices()[dyn] + [ODD_LATTICES[dyn]]):
        H, r = _check_probe(dyn, shape, lo, hi, c, _gpu_solve(dyn, lo, hi, PROBE_H))
        if dyn == 1 and i == 0:     # the odd lattice's theta nodes need not put every case on the H < 0 side
            _assert_saturation_cases(H, r)


@gpu
def test_solver_meets_the_rotated_slab_and_converges():
    errs = {}
    for shape in (DI_LAT[0], (81, 81, 41, 41)):
        for phi in (0, 30, 45, 90):
            if shape != DI_LAT[0] and phi == 90:
                continue
            l, exact, mask = _rotated_slab(shape, phi)
            V = _gpu_solve(0, DI_LAT[1], DI_LAT[2], SLAB_T)(l)
            errs[shape, phi] = _slab_error(V, l, exact, mask, phi)
            print(f"rotated slab phi={phi} {shape}: max |V - V*| = {errs[shape, phi] * 1e3:.2f} mm "
                  f"over {int(mask.sum())} cells")
    for phi in (0, 30, 45, 90):
        assert errs[DI_LAT[0], phi] < 0.01, phi
    for phi in (0, 30, 45):
        assert errs[DI_LAT[0], phi] >= 1.5 * errs[(81, 81, 41, 41), phi], phi


# ----------------------------------------------------------------------------------------------------------------------
# 3. Computed grids, through SafetyFilter, against trajectories
# ----------------------------------------------------------------------------------------------------------------------
# eps: tolerances fixed before the margins were measured, below one position spacing of the default lattices
# (0.225 m, 0.275 km): the interpolated, first-order-in-time grid against exact (double integrator) or RK4 (airtaxi)
# motion. `spacing`: the default lattice's position spacing.
GAME = {
    0: dict(name='double_integrator', horizon=4.0, switch=0.25, greedy_dt=0.05, sub_dt=0.01, eps=0.05,
            sep=DIC.SEPARATION_DISTANCE, spacing=(DI_LAT[2][0] - DI_LAT[1][0]) / (DI_LAT[0][0] - 1)),
    1: dict(name='airtaxi', horizon=60.0, switch=1.0, greedy_dt=0.5, sub_dt=0.01, eps=0.1,
            sep=ATC.SEPARATION_DISTANCE, spacing=(AT_LAT[2][0] - AT_LAT[1][0]) / (AT_LAT[0][0] - 1)),
}
N_PAIRS = 256
DEV = 'cuda'
_GRIDS = {}


def _filter(dyn):
    from layered_safe_marl_b200 import SafetyFilter
    if dyn not in _GRIDS:
        _GRIDS[dyn] = SafetyFilter(GAME[dyn]['name'], value_grid=R.value_grid(dyn))
    return _GRIDS[dyn]


def _t_corners(dyn, torch):
    """The 16 joint-control corners (16, 4) of the unsaturated box, in the filter's column order."""
    lo = [-DI_A] * 4 if dyn == 0 else [-AT_W, -AT_W, AT_AMIN, AT_AMIN]
    hi = [DI_A] * 4 if dyn == 0 else [AT_W, AT_W, AT_AMAX, AT_AMAX]
    return torch.tensor([[hi[j] if (k >> j) & 1 else lo[j] for j in range(4)] for k in range(16)],
                        dtype=torch.float64, device=DEV)


def _t_advance(dyn, ego, oth, u, dt, torch):
    """Both agents over dt under the constant joint control u (..., 4): exact parabolas (double integrator) or one RK4
    step of the unicycles with the speed clamped to [V_MIN, V_MAX] after it (airtaxi)."""
    if dyn == 0:
        ae, ao = u[..., 0:2], u[..., 2:4]

        def go(s, a):
            p, v = s[..., :2], s[..., 2:]
            return torch.cat([p + v * dt + 0.5 * a * dt * dt, v + a * dt], -1)
        return go(ego, ae), go(oth, ao)

    def rk4(s, w, a):
        def f(z):
            return torch.stack([z[..., 3] * torch.cos(z[..., 2]), z[..., 3] * torch.sin(z[..., 2]),
                                w.expand_as(z[..., 0]), a.expand_as(z[..., 0])], -1)
        k1 = f(s)
        k2 = f(s + 0.5 * dt * k1)
        k3 = f(s + 0.5 * dt * k2)
        k4 = f(s + dt * k3)
        z = s + (dt / 6.0) * (k1 + 2 * k2 + 2 * k3 + k4)
        return torch.cat([z[..., :3], z[..., 3:].clamp(V_MIN, V_MAX)], -1)
    return rk4(ego, u[..., 0], u[..., 2]), rk4(oth, u[..., 1], u[..., 3])


def _t_margin(ego, oth, sep, torch):
    return torch.sqrt((ego[..., 0] - oth[..., 0]) ** 2 + (ego[..., 1] - oth[..., 1]) ** 2) - sep


def _t_in_box(dyn, ego, oth, torch):
    """Whether the pair's relative state lies inside the computed lattice, where the lookup is V itself (outside,
    interpolation clamps to the edge)."""
    lo, hi = (DI_LAT if dyn == 0 else AT_LAT)[1:]
    if dyn == 0:
        r = ego - oth
        dims = range(4)
    else:
        ddx, ddy = oth[..., 0] - ego[..., 0], oth[..., 1] - ego[..., 1]
        ce, se = torch.cos(ego[..., 2]), torch.sin(ego[..., 2])
        r = torch.stack([ddx * ce + ddy * se, ddy * ce - ddx * se], -1)
        dims = range(2)
    ok = torch.ones(r.shape[:-1], dtype=torch.bool, device=r.device)
    for d in dims:
        ok = ok & (r[..., d] >= lo[d]) & (r[..., d] <= hi[d])
    return ok


def _start_pairs(dyn, torch):
    """Seeded absolute pairs whose relative state is well inside the lattice, biased toward conflicts."""
    rng = np.random.default_rng(40 + dyn)
    if dyn == 0:
        r = np.concatenate([rng.uniform(-3.0, 3.0, (N_PAIRS, 2)), rng.uniform(-0.8, 0.8, (N_PAIRS, 2))], -1)
        r[:, 2:] -= 0.5 * r[:, :2] / np.linalg.norm(r[:, :2], axis=1, keepdims=True)  # closing, mostly
        r[:, 2:] = np.clip(r[:, 2:], -0.9, 0.9)
    else:
        r = np.stack([rng.uniform(-4.0, 4.0, N_PAIRS), rng.uniform(-4.0, 4.0, N_PAIRS),
                      rng.uniform(-math.pi, math.pi, N_PAIRS), rng.uniform(V_MIN, V_MAX, N_PAIRS),
                      rng.uniform(V_MIN, V_MAX, N_PAIRS)], -1)
    ego, oth = _abs_pair(dyn, r, rng)
    return torch.as_tensor(ego, device=DEV), torch.as_tensor(oth, device=DEV)


def _rollout(dyn, ego, oth, control, torch):
    """J = min over the horizon of distance - separation, sampled every sub_dt, for control(t) -> (..., 4)."""
    g = GAME[dyn]
    steps = int(round(g['horizon'] / g['sub_dt']))
    J = _t_margin(ego, oth, g['sep'], torch)
    for k in range(steps):
        ego, oth = _t_advance(dyn, ego, oth, control(k * g['sub_dt']), g['sub_dt'], torch)
        J = torch.minimum(J, _t_margin(ego, oth, g['sep'], torch))
    return J


@gpu
@pytest.mark.parametrize('dyn', [0, 1])
def test_no_control_beats_the_computed_value(dyn):
    """(a) The tube is a supremum over controls: J <= V + eps for the 16 constant corners and 16 seeded bang-bang
    sequences that switch every `switch` seconds."""
    import torch
    g = GAME[dyn]
    sf = _filter(dyn)
    ego, oth = _start_pairs(dyn, torch)
    V = sf.values(ego=ego, other=oth)[0]
    assert torch.isfinite(V).all()
    corners = _t_corners(dyn, torch)
    n_seg = int(round(g['horizon'] / g['switch']))
    rng = np.random.default_rng(50 + dyn)
    seqs = torch.as_tensor(rng.integers(0, 16, (16, n_seg)), device=DEV)
    # every pair under every policy at once: (32 policies, N_PAIRS)
    E, O = ego.expand(32, -1, -1).contiguous(), oth.expand(32, -1, -1).contiguous()

    def control(t):
        seg = min(int(t / g['switch'] + 1e-9), n_seg - 1)
        idx = torch.cat([torch.arange(16, device=DEV), seqs[:, seg]])
        return corners[idx].view(32, 1, 4)
    J = _rollout(dyn, E, O, control, torch)
    worst = float((J - V).max())
    print(f"{g['name']}: max over {J.numel()} trajectories of J - V = {worst:+.4f} (eps {g['eps']}); "
          f"V in [{float(V.min()):.3f}, {float(V.max()):.3f}]")
    assert worst <= g['eps']


@gpu
@pytest.mark.parametrize('dyn', [0, 1])
def test_the_computed_value_is_attained(dyn):
    """(b) V is attained: every greedy_dt seconds both agents take the corner that maximises the looked-up V of the
    next state (one batched values call per step), and J >= V - eps. A corner whose next state leaves the lattice is
    not taken while another stays inside.

    Where the best trajectory passes within one position spacing of the other agent, the bound is that spacing
    instead of eps. The target |x[:2]| - sep has its cone vertex at the origin, which the lattice resolves to one
    cell, and the scheme rounds the vertex off, so V over-estimates the deepest closest approaches. Measured on the
    airtaxi default lattice: a head-on pair 0.40 km apart (V = -0.184 km) whose best closest approach is 0.094 km
    (J = -0.363 km; the greedy policy and 8192 random bang-bang sequences agree). The gap is the position
    resolution: 0.179 / 0.130 / 0.103 km with 41 / 61 / 81 position nodes, unchanged with twice the theta or speed
    nodes, any greedy step from 0.1 to 1 s, or without the speed clamp."""
    import torch
    g = GAME[dyn]
    sf = _filter(dyn)
    ego, oth = _start_pairs(dyn, torch)
    V0 = sf.values(ego=ego, other=oth)[0]
    assert torch.isfinite(V0).all()
    corners = _t_corners(dyn, torch)
    n_sub = int(round(g['greedy_dt'] / g['sub_dt']))
    J = _t_margin(ego, oth, g['sep'], torch)
    choice = torch.zeros(N_PAIRS, dtype=torch.long, device=DEV)
    for _ in range(int(round(g['horizon'] / g['greedy_dt']))):
        E, O = ego.expand(16, -1, -1), oth.expand(16, -1, -1)
        Jc = _t_margin(E, O, g['sep'], torch)
        u = corners.view(16, 1, 4)
        for _ in range(n_sub):
            E, O = _t_advance(dyn, E, O, u, g['sub_dt'], torch)
            Jc = torch.minimum(Jc, _t_margin(E, O, g['sep'], torch))
        v = sf.values(ego=E.reshape(-1, 4), other=O.reshape(-1, 4))[0].view(16, N_PAIRS)
        v = torch.where(_t_in_box(dyn, E, O, torch), v, torch.full_like(v, -math.inf))
        stay = torch.isfinite(v).any(0)
        choice = torch.where(stay, v.argmax(0), choice)
        ar = torch.arange(N_PAIRS, device=DEV)
        ego, oth = E[choice, ar], O[choice, ar]
        J = torch.minimum(J, Jc[choice, ar])
    gap = J - V0
    vertex = J + g['sep'] < g['spacing']
    far = float(gap[~vertex].min())
    print(f"{g['name']}: min over {N_PAIRS} greedy trajectories of J - V = {far:+.4f} (eps {g['eps']}) for the "
          f"{int((~vertex).sum())} that stay a position spacing apart"
          + (f", {float(gap[vertex].min()):+.4f} (bound {g['spacing']:.3f}) for the closer ones ({int(vertex.sum())})"
             if vertex.any() else ""))
    assert far >= -g['eps']
    assert (gap[vertex] >= -g['spacing']).all()
