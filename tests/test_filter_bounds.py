"""The safety filter and the airtaxi step at the states random rollouts do not reach.

Parity rollouts are 12 to 25 steps of uniform actions, so no airtaxi reaches V_MAX, the bang-bang box only ever drops
the ego's lower acceleration bound, and the CBF-QP is never infeasible. This file puts the filter on those states:

- `restate` is an independent float64 statement of the filter's resolution (the bang-bang boxes with their jnp.where
  cascade, the CBF-QP with both weightings, the infeasible QP that returns u_ref, the control clips). On CPU it agrees
  with the C oracle bit for bit on crafted rows, and three mutated statements of it do not.
- GPU: the same rows through `SafetyFilter.apply`, HJ lookups on the top and bottom speed nodes, and env rollouts that
  sit at the speed bounds or alias the QP, all against the oracle bit for bit.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))
sys.path.insert(0, os.path.join(REPO, 'tests'))

import _golden as G  # noqa: E402
import oracle_env as O  # noqa: E402
import test_cuda_parity as P  # noqa: E402
import test_safety_filter_op as SF  # noqa: E402
from layered_safe_marl_b200 import config as cfg, hj_grid  # noqa: E402

V_MIN, V_MAX = cfg.AirTaxiConfig.V_MIN, cfg.AirTaxiConfig.V_MAX
AT_AMIN, AT_AMAX, AT_WMAX = cfg.AirTaxiConfig.ACCEL_MIN, cfg.AirTaxiConfig.ACCEL_MAX, cfg.AirTaxiConfig.ANGULAR_RATE_MAX
DI_AMAX = cfg.DoubleIntegratorConfig.ACCELX_MAX
EPS_HJ = 0.4                # least-restrictive switch: bang-bang below this value, CBF-QP above
FILTERED_NORM = 1e-4        # |u - u_ref| above which a row counts as filtered
MUTATIONS = ('first true wins', 'filtered on aliased rows', 'aliased rows not clipped')


def _f32(x):
    return float(np.float32(x))


def _pymin(x, m):
    return np.where(m < x, m, x)         # Python's min(x, m): x unless m is smaller


def _pymax(x, m):
    return np.where(m > x, m, x)


def at_bound_speeds(dt):
    """The airtaxi speeds where the box cascade and the acceleration clip switch, and one double on each side."""
    base = [V_MIN, V_MAX, V_MAX - dt * AT_AMAX, V_MIN - dt * AT_AMIN]
    return np.array(sorted({f(v) for v in base for f in (lambda v: v, lambda v: np.nextafter(v, -1.0),
                                                          lambda v: np.nextafter(v, 1.0))}))


def di_bound_velocities(dt):
    """Double-integrator velocities where the clip switches (relative velocity against an agent at rest), their
    neighbours, the speed limit and rest."""
    thr = DI_AMAX - dt * DI_AMAX
    base = [thr, -thr]
    out = {0.0, 0.5, -0.5}
    for v in base:
        out |= {v, float(np.nextafter(v, -1.0)), float(np.nextafter(v, 1.0))}
    return np.array(sorted(out))


# ----------------------------------------------------------------------------------------------------------------------
# the restatement
# ----------------------------------------------------------------------------------------------------------------------
def relative_state(dyn, ego, other):
    """The relative state in the form the specialised pipeline evaluates (airtaxi: (dx, dy) rotated into the ego frame
    with the shared float64 sin / cos; see oracle/lsm_oracle.c at_relative_state)."""
    if dyn == 0:
        return ego - other
    ddx, ddy = other[:, 0] - ego[:, 0], other[:, 1] - ego[:, 1]
    se, ce = O.math_eval(0, ego[:, 2]), O.math_eval(1, ego[:, 2])
    return np.stack([ddx * ce + ddy * se, ddy * ce - ddx * se, other[:, 2] - ego[:, 2], ego[:, 3], other[:, 3]], -1)


def restate(dyn, params, ego, other, ua, uo, value, grad, mutation=None, nearest=None):
    """The safety handle's apply_safety_filter for rows of one ego against its deconflicting other.

    value: the other's shifted HJ value (+inf out of the grid); grad: the value gradient at the relative state;
    nearest: the distance to the ego's nearest other, which gates the filter (default: the distance to `other`).
    Returns (safe [B, 2], filtered [B], label [B], conds [B, 4], u [B, 4]): label names the branch a row takes; conds
    are the four airtaxi speed tests of the bang-bang box (v_a <= V_MIN, v_a >= V_MAX, v_b <= V_MIN, v_b >= V_MAX) of
    the rows the filter resolves; u is the resolved control vector.

    The control vector is ordered like the control Jacobian's columns (DI [a_x, a_y, -a_x, -a_y] acting on
    [a_ego, a_other]; airtaxi [w_a, w_b, a_a, a_b]) while u_ref is the concatenation of the two raw actions
    ([w_a, a_a, w_b, a_b] for the airtaxi); the safe action is the first two entries. The reference does the same.
    """
    assert mutation in (None,) + MUTATIONS
    B = ego.shape[0]
    dt, cbf = float(params.dt), float(params.cbf_rate)
    rel = relative_state(dyn, ego, other)
    uref = np.concatenate([ua, uo], -1)
    g = grad
    dist = np.sqrt((other[:, 0] - ego[:, 0]) ** 2 + (other[:, 1] - ego[:, 1]) ** 2) if nearest is None else nearest
    act = (dist <= params.coordination_range) & np.isfinite(value)
    v = np.where(act, value, 0.0)
    bang = v < EPS_HJ
    conds = np.zeros((B, 4), bool)
    if dyn == 0:
        a = np.stack([g[:, 2], g[:, 3], -g[:, 2], -g[:, 3]], -1)
        u_bang = np.where(a < 0.0, -DI_AMAX, DI_AMAX)
        b = (g[:, 0] * rel[:, 2] + g[:, 1] * rel[:, 3]) + cbf * v
        pinv = np.ones((B, 4))
    else:
        a = np.stack([(g[:, 0] * rel[:, 1] + g[:, 1] * (-rel[:, 0])) + g[:, 2] * (-1.0), g[:, 2], g[:, 3], g[:, 4]], -1)
        # Air4dCooperativeDynamics.optimal_control_and_disturbance: float32 boxes, then four whole-box jnp.where
        # selections in a row, each against the unmodified box - the LAST true condition decides the box
        lo = np.array([_f32(-AT_WMAX), _f32(-AT_WMAX), _f32(AT_AMIN), _f32(AT_AMIN)])
        hi = np.array([_f32(AT_WMAX), _f32(AT_WMAX), _f32(AT_AMAX), _f32(AT_AMAX)])
        conds = np.stack([rel[:, 3] <= V_MIN, rel[:, 3] >= V_MAX, rel[:, 4] <= V_MIN, rel[:, 4] >= V_MAX], -1)
        cascade = [(0, 'lo', 2), (1, 'hi', 2), (2, 'lo', 3), (3, 'hi', 3)]
        if mutation == 'first true wins':
            cascade = cascade[::-1]
        LO, HI = np.broadcast_to(lo, (B, 4)), np.broadcast_to(hi, (B, 4))
        for c, side, k in cascade:
            lo_c, hi_c = lo.copy(), hi.copy()
            (lo_c if side == 'lo' else hi_c)[k] = 0.0
            LO = np.where(conds[:, c:c + 1], lo_c, LO)
            HI = np.where(conds[:, c:c + 1], hi_c, HI)
        u_bang = np.where(a < 0.0, LO, HI)
        f0 = -rel[:, 3] + rel[:, 4] * O.math_eval(1, rel[:, 2])
        f1 = rel[:, 4] * O.math_eval(0, rel[:, 2])
        b = (g[:, 0] * f0 + g[:, 1] * f1) + cbf * v
        # P^-1 of the QP's weighting: the ego's turn rate is the expensive control when the other is behind it
        pinv = np.where((rel[:, 0] < 0.0)[:, None], np.array([1.0 / 100.0, 1.0 / 10.0, 1.0 / 10.0, 1.0 / 1.0]),
                        np.array([1.0 / 10.0, 1.0 / 1.0, 1.0 / 100.0, 1.0 / 10.0]))
    # min (u - u_ref)' P (u - u_ref) s.t. a.u + b >= 0: u_ref when it is feasible, else the P-weighted projection onto
    # a.u + b = 0; infeasible (a' P^-1 a == 0) returns u_ref itself
    s = (((a[:, 0] * uref[:, 0] + a[:, 1] * uref[:, 1]) + a[:, 2] * uref[:, 2]) + a[:, 3] * uref[:, 3]) + b
    denom = (((a[:, 0] * pinv[:, 0]) * a[:, 0] + (a[:, 1] * pinv[:, 1]) * a[:, 1]) + (a[:, 2] * pinv[:, 2]) * a[:, 2]) \
        + (a[:, 3] * pinv[:, 3]) * a[:, 3]
    inactive = s >= 0.0
    aliased = ~bang & ~inactive & (denom == 0.0)
    with np.errstate(divide='ignore', invalid='ignore'):
        lam = s / denom
        u_proj = uref - lam[:, None] * (pinv * a)
    u_qp = np.where((inactive | aliased)[:, None], uref, u_proj)
    if dyn == 1:        # turn rates of a solved QP back into their box
        solved = ~aliased
        for k in (0, 2):
            u_qp[:, k] = np.where(solved, _pymax(_pymin(u_qp[:, k], AT_WMAX), -AT_WMAX), u_qp[:, k])
    u = np.where(bang[:, None], u_bang, u_qp)
    # clip_ctrl_with_valid_control_bound: no acceleration that would leave the speed box within one step
    clip = ~aliased if mutation == 'aliased rows not clipped' else np.ones(B, bool)
    if dyn == 0:
        for k, r in ((0, rel[:, 2]), (1, rel[:, 3])):
            hi_k = np.where(r < DI_AMAX - dt * DI_AMAX, DI_AMAX, 0.0)
            lo_k = np.where(r > -DI_AMAX - dt * (-DI_AMAX), -DI_AMAX, 0.0)
            u[:, k] = np.where(clip, _pymax(_pymin(u[:, k], hi_k), lo_k), u[:, k])
    else:
        for k, r in ((1, rel[:, 3]), (3, rel[:, 4])):
            hi_k = np.where(r < V_MAX - dt * AT_AMAX, AT_AMAX, 0.0)
            lo_k = np.where(r > V_MIN - dt * AT_AMIN, AT_AMIN, 0.0)
            u[:, k] = np.where(clip, _pymax(_pymin(u[:, k], hi_k), lo_k), u[:, k])
            u[:, k] = np.where(bang, np.float32(u[:, k]).astype(np.float64), u[:, k])     # a float32 array in the reference
    d = u - uref
    nd = np.sqrt(((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) + d[:, 3] * d[:, 3])
    if mutation != 'filtered on aliased rows':
        nd = np.where(aliased, 0.0, nd)
    filtered = act & (nd > FILTERED_NORM)
    safe = np.where(act[:, None], u[:, :2], ua)
    label = np.where(~act, 'pass', np.where(bang, 'bang', np.where(inactive, 'qp_inactive',
                                                                   np.where(aliased, 'qp_infeasible', 'qp_projected'))))
    if dyn == 1:
        winner = np.full(B, 'free', dtype=object)
        for c, name in enumerate(('va<=vmin', 'va>=vmax', 'vb<=vmin', 'vb>=vmax')):
            winner = np.where(conds[:, c], name, winner)
        label = np.where(label == 'bang', np.char.add('bang/', winner.astype(str)), label)
        label = np.where(label == 'qp_projected', np.where(rel[:, 0] < 0.0, 'qp_projected/behind', 'qp_projected/ahead'),
                         label)
    return safe, filtered, label.astype(str), conds & act[:, None], u


# ----------------------------------------------------------------------------------------------------------------------
# grids and crafted rows
# ----------------------------------------------------------------------------------------------------------------------
_GRIDS = {}


def grid(name):
    """'di' / 'at': the synthetic grids. 'di_vfree': a double-integrator value 4 (r - sep) that does not depend on the
    velocity, so the QP's control row is exactly 0. 'at_xonly': an airtaxi value 0.5 + 40 x_r that depends on the
    relative position along the ego's heading only, so the control row is exactly 0 wherever y_r == 0."""
    if name not in _GRIDS:
        if name == 'di':
            g = hj_grid.synthetic_di_grid()
        elif name == 'at':
            g = hj_grid.synthetic_airtaxi_grid()
        elif name == 'di_vfree':
            sep = cfg.DoubleIntegratorConfig.SEPARATION_DISTANCE
            x, y, _, _ = hj_grid._lattice(hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI, hj_grid.DI_GRID_SHAPE, (False,) * 4)
            v = 4.0 * (np.sqrt(x * x + y * y) - sep)
            g = hj_grid.make_hj_handle(-v.astype(np.float32), hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI, (False,) * 4, sep, sep)
        elif name == 'at_xonly':
            sep = cfg.AirTaxiConfig.SEPARATION_DISTANCE
            per = (False, False, True, False, False)
            x = hj_grid._lattice(hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI, hj_grid.AIRTAXI_GRID_SHAPE, per)[0]
            v = 0.5 + 40.0 * x
            g = hj_grid.make_hj_handle(-v.astype(np.float32), hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI, per, sep, sep)
        else:
            raise KeyError(name)
        if name in ('di_vfree', 'at_xonly'):
            first = 2 if name == 'di_vfree' else 1
            assert not g.grads[..., first:].any(), f"{name}: a gradient component the value does not depend on is not 0"
        _GRIDS[name] = g
    return _GRIDS[name]


def params_of(dyn, f32):
    return SF._params(dyn, f32)


def _actions(dyn, rng, B):
    t0, t1 = O.action_tables(dyn)
    return np.stack([rng.choice(t0, B), rng.choice(t1, B)], -1)


def crafted_rows(dyn, gname, seed=0):
    """(ego [B, 4], other [B, 4], ego_action [B, 2], other_action [B, 2]) for one deconflicting other per row."""
    rng = np.random.default_rng(seed)
    params = params_of(dyn, False)
    if dyn == 1:
        S = at_bound_speeds(params.dt)
        va, vb = np.meshgrid(S, S, indexing='ij')
        va, vb = np.tile(va.ravel(), 12), np.tile(vb.ravel(), 12)
        B = va.size
        if gname == 'at_xonly':
            # ego heading 0 and the other on the ego's x axis: y_r == 0 exactly; 0.5 + 40 x_r spans bang and QP
            ego = np.stack([np.zeros(B), rng.uniform(-1, 1, B), np.zeros(B), va], -1)
            dx = rng.choice(np.arange(-24, 17) / 1024.0, B)
            th = rng.choice([0.0, np.pi, 0.5, -2.5, 3.0], B)
            # a third of the others off the axis (y_r != 0): the control row is not 0 there and the QP projects
            dy = np.where(np.arange(B) % 3 == 2, rng.choice([-1 / 64, 1 / 64, 1 / 8], B), 0.0)
            other = np.stack([dx, ego[:, 1] + dy, th, vb], -1)
        else:
            ego = np.stack([rng.uniform(-1, 1, B), rng.uniform(-1, 1, B), rng.uniform(-np.pi, np.pi, B), va], -1)
            d, phi = rng.uniform(0.2, 2.5, B), rng.uniform(-np.pi, np.pi, B)
            other = np.stack([ego[:, 0] + d * np.cos(phi), ego[:, 1] + d * np.sin(phi), rng.uniform(-np.pi, np.pi, B), vb], -1)
    else:
        V = di_bound_velocities(params.dt)
        B = 3000
        ego = np.stack([rng.uniform(-1, 1, B), rng.uniform(-1, 1, B), rng.choice(V, B), rng.choice(V, B)], -1)
        rest = rng.random((B, 2)) < 0.5
        other_v = np.where(rest, 0.0, rng.choice(V, (B, 2)))
        lo, hi = (0.55, 1.1) if gname == 'di_vfree' else (0.1, 2.5)
        d, phi = rng.uniform(lo, hi, B), rng.uniform(-np.pi, np.pi, B)
        # half of the others head straight for the ego at full speed: closing rows with values above EPS_HJ
        toward = np.arange(B) % 2 == 1
        other_v = np.where(toward[:, None], -0.5 * np.stack([np.cos(phi), np.sin(phi)], -1), other_v)
        other = np.stack([ego[:, 0] + d * np.cos(phi), ego[:, 1] + d * np.sin(phi), other_v[:, 0], other_v[:, 1]], -1)
    ua, uo = _actions(dyn, rng, B), _actions(dyn, rng, B)
    return ego, other, ua, uo


def oracle_and_restatement(dyn, gname, f32, rows, mutation=None):
    """The oracle's filter over the rows (rotation form) and the restatement fed with the oracle's value and gradient."""
    params = params_of(dyn, f32)
    g = grid(gname)
    ego, other, ua, uo = rows
    B = ego.shape[0]
    o_safe, o_filt, o_idx, o_val = SF.oracle_rows(params.asdict(), g, ego, other.reshape(B, 1, 4), ua, uo.reshape(B, 1, 2),
                                                  rel_form=1)
    val, grad = SF.oracle_lookup(params.asdict(), g, rel=relative_state(dyn, ego, other))
    assert np.array_equal(val, o_val), "the row's value is not the value of the restated relative state"
    r = restate(dyn, params, ego, other, ua, uo, val, grad, mutation)
    return (o_safe, o_filt, o_idx, o_val), r


def echo_rows(dyn, gname, f32, rows):
    """The rows again with u_ref set to the restated u: the bang-bang rows are then not filtered, so a change of any
    entry of u (the other's half included, which the safe action does not show) flips the filtered flag."""
    _, r = oracle_and_restatement(dyn, gname, f32, rows)
    u = r[4]
    ego, other, _, _ = rows
    return ego, other, u[:, :2].copy(), u[:, 2:].copy()


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the restatement against the oracle
# ----------------------------------------------------------------------------------------------------------------------
ROW_CASES = [(0, 'di'), (0, 'di_vfree'), (1, 'at'), (1, 'at_xonly')]
# the least number of rows of each branch the crafted rows must reach (labels of `restate`)
REQUIRED = {
    'di': {'bang': 100, 'qp_inactive': 100, 'qp_projected': 10},
    'di_vfree': {'bang': 50, 'qp_inactive': 100, 'qp_infeasible': 100},
    'at': {'bang/free': 20, 'bang/va<=vmin': 20, 'bang/va>=vmax': 20, 'bang/vb<=vmin': 20, 'bang/vb>=vmax': 20,
           'qp_inactive': 50, 'qp_projected/ahead': 10},
    'at_xonly': {'bang/vb>=vmax': 10, 'qp_inactive': 100, 'qp_infeasible': 100, 'qp_projected/behind': 20,
                 'qp_projected/ahead': 20},
}


def all_rows(dyn, gname, f32):
    rows = crafted_rows(dyn, gname)
    echo = echo_rows(dyn, gname, f32, rows)
    return [('crafted', rows), ('echo', echo)]


def _check_rows(dyn, gname, f32, rows, what, mutation=None):
    """-> rows where the restatement disagrees with the oracle, and the restatement's result."""
    (o_safe, o_filt, o_idx, _), r = oracle_and_restatement(dyn, gname, f32, rows, mutation)
    safe, filt = r[0], r[1]
    assert (o_idx == 0).all() or not np.isfinite(o_idx).all()
    bad = (safe.view(np.int64) != o_safe.view(np.int64)).any(-1) | (filt != o_filt)
    return bad, r


@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('dyn,gname', ROW_CASES)
def test_restatement_matches_the_oracle_on_crafted_rows(dyn, gname, f32):
    labels, conds = [], []
    for what, rows in all_rows(dyn, gname, f32):
        bad, r = _check_rows(dyn, gname, f32, rows, what)
        if bad.any():
            i = int(np.argmax(bad))
            raise AssertionError(f"{gname} {what}: {int(bad.sum())} rows differ; first {i} ({r[2][i]}): "
                                 f"restated {r[0][i]!r} {r[1][i]}, oracle rows {SF.oracle_rows}")
        labels.append(r[2]); conds.append(r[3])
    labels, conds = np.concatenate(labels), np.concatenate(conds)
    counts = {k: int((labels == k).sum()) for k in np.unique(labels)}
    print(f"{gname} f32={f32}: {counts}")
    for k, n in REQUIRED[gname].items():
        assert counts.get(k, 0) >= n, f"{gname}: {counts.get(k, 0)} rows take '{k}', want >= {n}"
    if dyn == 1 and gname == 'at':
        bang = np.char.startswith(labels, 'bang')
        qp = np.char.startswith(labels, 'qp')
        for mode, m in (('bang', bang), ('qp', qp)):
            for c in range(4):
                assert (conds[m, c]).sum() >= 20, f"{mode} rows: speed test {c} true in too few rows"
            assert (conds[m].sum(-1) >= 2).sum() >= 20, f"{mode} rows: too few rows with two speed tests true"


@pytest.mark.parametrize('mutation', MUTATIONS)
def test_a_mutated_restatement_disagrees_with_the_oracle(mutation):
    failed = 0
    for dyn, gname in ROW_CASES:
        for what, rows in all_rows(dyn, gname, False):
            bad, _ = _check_rows(dyn, gname, False, rows, what, mutation)
            failed += int(bad.sum())
    assert failed > 0, f"the mutation '{mutation}' agrees with the oracle on every crafted row"


def world_labels(params, g, pre, actions):
    """The branch each live agent's filter row takes in one env step, from the oracle's state before it: the oracle's
    rows (World.apply_safety_filter's others, rotation form) pick the deconflicting other, the restatement labels the
    row and must reproduce the oracle's safe action and flag. -> (labels [n * N], conds [n * N, 4])."""
    dyn = int(params.dynamics)
    states = np.asarray(pre['agent_values'], np.float64)
    n, N = states.shape[:2]
    done = np.asarray(pre['done'], bool)
    t0, t1 = O.action_tables(dyn)
    raw = np.stack([t0[actions // 5], t1[actions % 5]], -1).astype(np.float64)
    js = np.array([[j for j in range(N) if j != i] for i in range(N)], dtype=np.int64).reshape(N, N - 1)
    ego, ua = states.reshape(n * N, 4), raw.reshape(n * N, 2)
    others, uos = states[:, js].reshape(n * N, N - 1, 4), raw[:, js].reshape(n * N, N - 1, 2)
    active = (~done[:, js] & ~done[:, :, None]).reshape(n * N, N - 1)
    o_safe, o_filt, o_idx, o_val = SF.oracle_rows(params.asdict(), g, ego, others, ua, uos, active, rel_form=1)
    k = np.maximum(o_idx, 0)
    other, uo = others[np.arange(n * N), k], uos[np.arange(n * N), k]
    _, grad = SF.oracle_lookup(params.asdict(), g, rel=relative_state(dyn, ego, other))
    val = np.where(o_idx >= 0, o_val, np.inf)
    d = np.sqrt((others[..., 0] - ego[:, None, 0]) ** 2 + (others[..., 1] - ego[:, None, 1]) ** 2)
    nearest = np.where(active, d, np.inf).min(-1) if N > 1 else np.full(n * N, np.inf)
    safe, filt, label, conds, _ = restate(dyn, params, ego, other, ua, uo, val, grad, nearest=nearest)
    assert np.array_equal(safe, o_safe) and np.array_equal(filt, o_filt), "restated env rows differ from the oracle"
    return label, conds


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the operator on the crafted rows
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('dyn,gname', ROW_CASES)
def test_operator_matches_oracle_and_restatement_on_crafted_rows(dyn, gname, f32):
    from layered_safe_marl_b200 import SafetyFilter
    params, g = params_of(dyn, f32), grid(gname)
    sf = SafetyFilter('double_integrator' if dyn == 0 else 'airtaxi', value_grid=g, interp_float32=f32)
    for what, rows in all_rows(dyn, gname, f32):
        ego, other, ua, uo = rows
        B = ego.shape[0]
        filt = SF._compare_to_oracle(sf, params, g, ego, other.reshape(B, 1, 4), ua, uo.reshape(B, 1, 2), None, None,
                                     f'{gname} {what}')
        bad, r = _check_rows(dyn, gname, f32, rows, what)
        assert not bad.any() and np.array_equal(filt, r[1]), f"{gname} {what}: the restatement differs"
    # the same rows as one ego against several slots: the crafted other in the middle slot, decoys out of range
    ego, other, ua, uo = all_rows(dyn, gname, f32)[0][1]
    B = ego.shape[0]
    far = other.copy()
    far[:, :2] += 50.0
    oth = np.stack([far, other, far], 1)
    SF._compare_to_oracle(sf, params, g, ego, oth, ua, np.stack([uo, uo, uo], 1), None, None, f'{gname} 3 slots')


# ----------------------------------------------------------------------------------------------------------------------
# GPU: lookups on the first and last speed node
# ----------------------------------------------------------------------------------------------------------------------
LOOKUP_CASES = [(0, 'di'), (0, 'di_vfree'), (1, 'at'), (1, 'at_xonly')]


def bound_node_points(dyn, rng, K=512):
    """Relative states with the speed (airtaxi: both speeds; DI: both relative velocities) on the lattice's first and
    last node and one double outside each."""
    if dyn == 1:
        ends = np.array([V_MIN, V_MAX, np.nextafter(V_MIN, -1.0), np.nextafter(V_MAX, 1.0)])
        pts = np.stack([rng.uniform(-3, 3, K), rng.uniform(-3, 3, K), rng.uniform(-np.pi, np.pi, K),
                        rng.choice(ends, K), rng.choice(ends, K)], -1)
        inner = rng.random(K) < 0.25
        pts[inner, 3 + rng.integers(0, 2, K)[inner]] = rng.uniform(V_MIN, V_MAX, int(inner.sum()))
    else:
        ends = np.array([-1.0, 1.0, np.nextafter(-1.0, -2.0), np.nextafter(1.0, 2.0)])
        pts = np.stack([rng.uniform(-2, 2, K), rng.uniform(-2, 2, K), rng.choice(ends, K), rng.choice(ends, K)], -1)
    return pts


@pytest.mark.gpu
@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('dyn,gname', LOOKUP_CASES)
def test_lookups_on_the_last_speed_node_match_the_oracle(dyn, gname, f32):
    import torch
    from layered_safe_marl_b200 import SafetyFilter
    params, g = params_of(dyn, f32), grid(gname)
    sf = SafetyFilter('double_integrator' if dyn == 0 else 'airtaxi', value_grid=g, interp_float32=f32)
    rel = bound_node_points(dyn, np.random.default_rng(3 + dyn))
    v, gr = sf.values(rel=torch.as_tensor(rel, device=sf.device), gradients=True)
    ov, og = SF.oracle_lookup(params.asdict(), g, rel=rel)
    v, gr = v.cpu().numpy(), gr.cpu().numpy()
    assert np.array_equal(v.view(np.int64), ov.view(np.int64)), f"values differ at {np.argwhere(v != ov)[:5].ravel()}"
    assert np.array_equal(gr.view(np.int64), og.view(np.int64)), \
        f"gradients differ at {np.argwhere((gr != og).any(-1))[:5].ravel()}"
    assert np.isfinite(ov).all()


# ----------------------------------------------------------------------------------------------------------------------
# GPU: env steps at the bounds, against the oracle
# ----------------------------------------------------------------------------------------------------------------------
ENV_SHAPES = {
    'at10': (dict(dynamics_type='airtaxi', num_agents=10, episode_length=350, world_size=6), dict(POTENTIAL_CONFLICT=True)),
    'di8': (dict(num_agents=8, episode_length=250, world_size=4), {}),
    'at10_f32': (dict(dynamics_type='airtaxi', num_agents=10, episode_length=350, world_size=6, interp_float32=True),
                 dict(POTENTIAL_CONFLICT=True)),
    'di8_f32': (dict(num_agents=8, episode_length=250, world_size=4, interp_float32=True), {}),
    # shapes the product library runs on the generic kernel
    'at6_generic': (dict(dynamics_type='airtaxi', num_agents=6, episode_length=350, world_size=6), dict(POTENTIAL_CONFLICT=True)),
    'di5_generic': (dict(num_agents=5, episode_length=250, world_size=4), {}),
}
TUNINGS = [dict(pair_placement=0, packed_grid=1), dict(pair_placement=4, packed_grid=1),
           dict(pair_placement=0, packed_grid=0), dict(pair_placement=4, packed_grid=0)]
ENV_CASES = [(s, k) for s in ('at10', 'di8') for k in range(len(TUNINGS))] + \
    [(s, None) for s in ('at10_f32', 'di8_f32', 'at6_generic', 'di5_generic')]


def place_pairs_at_bounds(dyn, dt, seed):
    """after_reset hook: agents 2k and 2k + 1 of every env a short distance apart, every speed on a bound of the box
    cascade or the acceleration clip (or one double beside it), random headings; both sides get the same state."""
    def hook(ora, cu):
        rng = np.random.default_rng(seed)
        s = ora.get_state()
        av = np.array(s['agent_values'])
        n, N = av.shape[:2]
        P2 = N // 2
        span, (dlo, dhi) = (4.0, (0.3, 2.0)) if dyn == 1 else (2.5, (0.2, 1.5))
        c = rng.uniform(-span, span, (n, P2, 2))
        d, phi = rng.uniform(dlo, dhi, (n, P2)), rng.uniform(-np.pi, np.pi, (n, P2))
        av[:, 0:2 * P2:2, :2] = c
        av[:, 1:2 * P2:2, :2] = c + d[..., None] * np.stack([np.cos(phi), np.sin(phi)], -1)
        if dyn == 1:
            av[..., 2] = rng.uniform(-np.pi, np.pi, (n, N))
            av[..., 3] = rng.choice(at_bound_speeds(dt), (n, N))
        else:
            V = di_bound_velocities(dt)
            av[..., 2] = rng.choice(V, (n, N))
            av[..., 3] = np.where(rng.random((n, N)) < 0.5, 0.0, rng.choice(V, (n, N)))
        s['agent_values'] = av
        ora.set_state(s)
        ora.observe()
        if cu is not None:
            cu.set_state(s)
            cu.observe()
    return hook


def env_case(shape, tuning, n, T, hook_seed=None, grids=None, actions=None, on_step=None, compare=None):
    kw, flags = ENV_SHAPES[shape]
    args = G.default_args(use_safety_filter=True, **kw)
    params = cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags(flags))
    hook = None if hook_seed is None else place_pairs_at_bounds(int(params.dynamics), float(params.dt), hook_seed)
    run = compare or P._compare_with_oracle
    return run(args, G.BinaryFlags(flags), n=n, T=T, episode=6249, seed=29, auto_reset=True, grids=grids,
               tuning=None if tuning is None else TUNINGS[tuning], after_reset=hook, actions=actions, on_step=on_step)


@pytest.mark.gpu
@pytest.mark.parametrize('shape,tuning', ENV_CASES)
def test_env_steps_from_bound_speeds_match_the_oracle(shape, tuning):
    ora, cu = env_case(shape, tuning, n=128, T=4, hook_seed=11)
    li = cu.env.launch_info()
    assert li['specialised'] == (0 if shape.endswith('_generic') else 1)
    if tuning is not None:
        assert li['pair_placement'] == TUNINGS[tuning]['pair_placement']


class MaxSpeedStats:
    """on_step hook of the max-acceleration airtaxi rollout: agent-steps at exactly V_MAX, filter rows with a speed at
    or above V_MAX, and the branches those rows took."""

    def __init__(self, params, g):
        self.params, self.g = params, g
        self.live = self.at_vmax = self.rows_vmax = 0
        self.labels = {}

    def __call__(self, t, a, pre, post):
        done = np.asarray(pre['done'], bool)
        s3 = np.asarray(pre['agent_values'])[..., 3]
        self.live += int((~done).sum())
        self.at_vmax += int(((s3 == V_MAX) & ~done).sum())
        label, conds = world_labels(self.params, self.g, pre, a)
        hit = conds[:, 1] | conds[:, 3]
        self.rows_vmax += int(hit.sum())
        for k in label[hit]:
            self.labels[k] = self.labels.get(k, 0) + 1


def max_accel_actions(N, n):
    """Action indices biased to the last acceleration column (ACCEL_MAX): 90 % of agent-steps."""
    def draw(rng, t):
        turn = rng.integers(0, 5, (n, N))
        acc = np.where(rng.random((n, N)) < 0.9, 4, rng.integers(0, 5, (n, N)))
        return turn * 5 + acc
    return draw


MAX_SPEED_T = 150
MAX_SPEED_N = 32


def max_speed_rollout(tuning, compare=None):
    kw, flags = ENV_SHAPES['at10']
    params = cfg.scenario_params_from_args(G.default_args(use_safety_filter=True, **kw), binary_cfg=G.BinaryFlags(flags))
    stats = MaxSpeedStats(params, G.value_grid_for(params)[0])
    out = env_case('at10', tuning, n=MAX_SPEED_N, T=MAX_SPEED_T, actions=max_accel_actions(10, MAX_SPEED_N),
                   on_step=stats, compare=compare)
    return out, stats


@pytest.mark.gpu
@pytest.mark.parametrize('tuning', range(len(TUNINGS)))
def test_airtaxi_rollout_at_max_speed_matches_the_oracle(tuning):
    _, st = max_speed_rollout(tuning)
    frac = st.at_vmax / st.live
    print(f"tuning {TUNINGS[tuning]}: {frac:.1%} of {st.live} live agent-steps at V_MAX, {st.rows_vmax} filter rows "
          f"with a speed >= V_MAX: {st.labels}")
    # an agent the filter resolves is clipped to zero acceleration from V_MAX - dt * ACCEL_MAX on, so it stays below
    # V_MAX; the agents that reach V_MAX are the ones no other agent is near
    assert frac >= 0.05, f"only {frac:.1%} of the live agent-steps sit at V_MAX"
    assert st.rows_vmax >= 100, f"only {st.rows_vmax} filter rows see a speed >= V_MAX"


class AliasStats:
    def __init__(self, params, g):
        self.params, self.g = params, g
        self.labels = {}

    def __call__(self, t, a, pre, post):
        label, _ = world_labels(self.params, self.g, pre, a)
        for k in label:
            self.labels[k] = self.labels.get(k, 0) + 1


def di_alias_rollout(shape, compare=None):
    kw, flags = ENV_SHAPES[shape]
    args = G.default_args(use_safety_filter=True, **dict(kw, world_size=2))
    params = cfg.scenario_params_from_args(args, binary_cfg=G.BinaryFlags(flags))
    stats = AliasStats(params, grid('di_vfree'))
    run = compare or P._compare_with_oracle
    out = run(args, G.BinaryFlags(flags), n=128, T=25, episode=6249, seed=37, auto_reset=True,
              grids=(grid('di_vfree'), None), on_step=stats)
    return out, stats


@pytest.mark.gpu
@pytest.mark.parametrize('shape', ['di8', 'di8_f32'])
def test_di_rollout_with_aliased_qp_matches_the_oracle(shape):
    _, st = di_alias_rollout(shape)
    print(f"{shape}: {st.labels}")
    assert st.labels.get('qp_infeasible', 0) >= 25
