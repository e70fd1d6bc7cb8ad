"""The airtaxi time-to-reach solve (liblsm_b200_hj.so lsm_hj_ttr_*, reachability.solve_ttr / ttr_grid) against the
numpy restatement of its declared scheme (tests/hj_solve_oracle.py, Lattice kind TTR) and against the game it solves.

CPU: the ctypes mirror of lsm_hj_ttr_problem; the library exports the TTR entry points and holds the TTR kernels; the
dissipation coefficients and time step equal the oracle's bit for bit; every invalid argument is refused with code 2;
the oracle's Hamiltonian equals an independent minimum over the control-box corners of an absolute-frame unicycle seen
from its goal, and mutated oracles (max for min, a flipped sin term, no speed saturation) fail that check.
GPU: the solve equals the oracle bit for bit (times and values; odd shapes, CFLs, horizons that end mid-step; arrays
past 2^31 bytes; a side stream); the game - the straight-line closed form and its refinement, a no-turn lower bound,
greedy and perturbed rollouts, the y / theta mirror symmetry; the default horizon; a computed grid through the env,
bit for bit with the C oracle in both interpolation arithmetics."""
import ctypes
import math
import os
import re
import shutil
import subprocess
import sys
import types

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))
sys.path.insert(0, os.path.join(REPO, 'tests'))

import _golden as G  # noqa: E402
import hj_solve_oracle as HO  # noqa: E402
from layered_safe_marl_b200 import _build, _lib, hj_grid  # noqa: E402
from layered_safe_marl_b200 import reachability as R  # noqa: E402
from layered_safe_marl_b200.config import AirTaxiConfig as ATC  # noqa: E402

gpu = pytest.mark.gpu
TTR_LAT = (hj_grid.TTR_GRID_SHAPE, hj_grid.TTR_GRID_LO, hj_grid.TTR_GRID_HI)
F32 = lambda x: float(np.float32(x))  # noqa: E731
W, AMIN, AMAX = F32(ATC.ANGULAR_RATE_MAX), F32(ATC.ACCEL_MIN), F32(ATC.ACCEL_MAX)
V_MIN, V_MAX = ATC.V_MIN, ATC.V_MAX
GOAL_R = ATC.DISTANCE_TO_GOAL_THRESHOLD
H_THR = 0.5 - 0.5 * math.cos(ATC.GOAL_HEADING_THRESHOLD)


# ----------------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------------
def test_ttr_problem_mirror_matches_the_c_header(tmp_path):
    cls = _lib.LsmHjTtrProblem
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lsm_b200_hj.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(lsm_hj_ttr_problem));']
    lines += [f'  printf("{f} %zu\\n", offsetof(lsm_hj_ttr_problem, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / 'p.c', tmp_path / 'p.exe'
    src.write_text('\n'.join(lines))
    subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), '-o', str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    assert int(got['size']) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def test_ttr_kernels_are_built_for_sm100a_and_exported():
    path = _build.build_hj()
    lib = ctypes.CDLL(path)
    for sym in ('lsm_hj_ttr_work_bytes', 'lsm_hj_ttr_dissipation', 'lsm_hj_ttr_solve'):
        assert sym in _lib.HJ_EXPORTED_SYMBOLS
        getattr(lib, sym)
    hj = _lib.load_hj()
    pr = R._ttr_problem(*TTR_LAT, 0.75)
    shape = TTR_LAT[0]
    assert hj.lsm_hj_ttr_work_bytes(ctypes.byref(pr)) == 8 * (3 * int(np.prod(shape)) + sum(shape) + 2 * shape[2])
    nvcc = shutil.which(os.environ.get('NVCC', 'nvcc'))
    exe = os.path.join(os.path.dirname(nvcc), 'cuobjdump') if nvcc else shutil.which('cuobjdump')
    assert exe and os.path.exists(exe), "cuobjdump (CUDA toolkit) not found next to nvcc"
    sass = subprocess.check_output([exe, '-sass', path], text=True)
    names = set(re.findall(r'Function : \S*?(lsm_hj_ttr_\w+?_kernel)', sass))
    assert names == {'lsm_hj_ttr_stage_kernel', 'lsm_hj_ttr_init_kernel'}, names
    assert 'sm_100a' in subprocess.check_output([exe, '-lelf', path], text=True)


@pytest.mark.parametrize('shape,lo,hi,cfl', [
    TTR_LAT + (0.75,),
    ((9, 11, 7, 5), (-2.0, -3.0, -math.pi, V_MIN), (1.0, 3.5, math.pi, V_MAX), 0.5),
    ((2, 3, 2, 2), TTR_LAT[1], TTR_LAT[2], 1.0),
    ((13, 10, 17, 11), (-8.0, -6.0, 0.0, 0.02), (6.0, 9.0, 2 * math.pi, 0.1), 0.3),
])
def test_ttr_dissipation_equals_the_oracle_bit_for_bit(shape, lo, hi, cfl):
    alpha, dt = R.ttr_dissipation(shape, lo, hi, cfl)
    o_alpha, o_dt = HO.dissipation(HO.Lattice(HO.TTR, shape, lo, hi), cfl)
    assert np.array_equal(alpha, o_alpha) and dt == o_dt, (alpha, o_alpha, dt, o_dt)
    assert alpha[2] == W and alpha[3] == max(abs(AMIN), abs(AMAX))


def test_invalid_ttr_arguments_are_refused_with_code_2():
    """Validation runs on the host before anything is enqueued: code 2 and a message, no device needed."""
    lib = _lib.load_hj()
    fake = ctypes.c_void_p(4096)                   # never dereferenced: every case below fails validation first

    def solve_rc(pr, horizon=1.0, target=fake, ttr=fake, final=fake, work=fake):
        return lib.lsm_hj_ttr_solve(pr, target, horizon, ttr, final, work, None)

    def bad(**kw):
        pr = R._ttr_problem(*TTR_LAT, 0.75)
        for k, v in kw.items():
            if k in ('shape', 'lo', 'hi'):
                d, x = v
                getattr(pr, k)[d] = x
            else:
                setattr(pr, k, v)
        return pr

    cases = [bad(shape=(0, 1)), bad(shape=(3, 0)), bad(shape=(2, -4)), bad(lo=(1, 9.0)), bad(lo=(2, float('nan'))),
             bad(hi=(3, float('inf'))), bad(hi=(0, -8.0)), bad(cfl=0.0), bad(cfl=1.5), bad(cfl=float('nan')),
             bad(cfl=-0.5)]
    for pr in cases:
        assert solve_rc(ctypes.byref(pr)) == 2, lib.lsm_hj_last_error()
        assert lib.lsm_hj_ttr_work_bytes(ctypes.byref(pr)) == 0
        a, dt = (ctypes.c_double * 4)(), ctypes.c_double()
        assert lib.lsm_hj_ttr_dissipation(ctypes.byref(pr), a, ctypes.byref(dt)) == 2
    assert lib.lsm_hj_ttr_work_bytes(None) == 0
    assert lib.lsm_hj_ttr_dissipation(None, None, None) == 2
    pr = ctypes.byref(R._ttr_problem(*TTR_LAT, 0.75))
    assert lib.lsm_hj_ttr_dissipation(pr, None, None) == 2
    assert solve_rc(None) == 2 and b'NULL' in lib.lsm_hj_last_error()
    for h in (-1.0, float('nan'), float('inf'), -float('inf')):
        assert solve_rc(pr, horizon=h) == 2, h
        assert b'horizon' in lib.lsm_hj_last_error()
    assert solve_rc(pr, target=None) == 2
    assert solve_rc(pr, ttr=None) == 2
    assert solve_rc(pr, work=None) == 2
    assert solve_rc(pr, work=ctypes.c_void_p(4097)) == 2 and b'aligned' in lib.lsm_hj_last_error()
    with pytest.raises(RuntimeError, match='cfl'):
        R.ttr_dissipation(*TTR_LAT, cfl=2.0)
    with pytest.raises(ValueError):
        R.ttr_dissipation((5, 5, 5), (0, 0, 0), (1, 1, 1))
    with pytest.raises(TypeError):
        import torch
        R.solve_ttr(torch.zeros(TTR_LAT[0], dtype=torch.float64), *TTR_LAT[1:], 10.0)


# --- the Hamiltonian against an independent game -----------------------------------------------------------------------
# Reference: an absolute-frame unicycle (X, Y, Th, v), X' = v cos Th, Y' = v sin Th, Th' = w, v' = a, and a goal
# (gx, gy, gh); the TTR state is rel_pos_from_reference(X, Y, gx, gy, gh), Th - gh, v (oracle/lsm_oracle.c), its rate
# the central difference of that map along the motion. H_ref = min over the four corners of the control box of c . r'.
# The box: w in +-W, a in [AMIN, AMAX]; v <= V_MIN forbids a < 0 and v >= V_MAX forbids a > 0.
CD_STEP = 1e-4
PROBE_H = 1e-7
EDGE = 3
# 13 speed nodes with node 3 bit-equal to V_MIN and node 9 to V_MAX (the lattice's own lo + k (hi - lo) / (n - 1))
SPEED = (0.0012861100000000002, 0.11960823, 13)
PROBE_LAT = ((9, 9, 16, SPEED[2]), (-0.6, -0.6, -math.pi, SPEED[0]), (0.6, 0.6, math.pi, SPEED[1]))
# probe gradients: drift components of either sign, small theta components (the turn term is -W |c2|), speed components
# of both signs so both saturations matter where H < 0
PROBE_C = [(1.0, -0.6, 0.02, 8.0), (0.0, 1.2, -0.03, -7.0), (-0.9, 0.7, 0.0, 6.0), (0.7, 1.1, 0.01, -9.0)]


def _to_goal_frame(s, g):
    dx, dy = s[..., 0] - g[..., 0], s[..., 1] - g[..., 1]
    c, si = np.cos(g[..., 2]), np.sin(g[..., 2])
    return np.stack([c * dx + si * dy, (-si) * dx + c * dy, s[..., 2] - g[..., 2], s[..., 3]], -1)


def _ref_hamiltonian(r, c, rng):
    """min over the control-box corners of c . r' at goal-frame states r (..., 4), from absolute-frame unicycles."""
    shp = r.shape[:-1]
    g = np.stack([rng.uniform(-3, 3, shp), rng.uniform(-3, 3, shp), rng.uniform(-math.pi, math.pi, shp)], -1)
    cg, sg = np.cos(g[..., 2]), np.sin(g[..., 2])
    s = np.stack([g[..., 0] + cg * r[..., 0] - sg * r[..., 1], g[..., 1] + sg * r[..., 0] + cg * r[..., 1],
                  r[..., 2] + g[..., 2], r[..., 3]], -1)
    a_lo = np.where(r[..., 3] <= V_MIN, 0.0, AMIN)
    a_hi = np.where(r[..., 3] >= V_MAX, 0.0, AMAX)
    best = np.full(shp, np.inf)
    for w in (-W, W):
        for a in (a_lo, a_hi):
            ds = np.stack([s[..., 3] * np.cos(s[..., 2]), s[..., 3] * np.sin(s[..., 2]), np.full(shp, w),
                           np.broadcast_to(a, shp)], -1)
            rate = (_to_goal_frame(s + CD_STEP * ds, g) - _to_goal_frame(s - CD_STEP * ds, g)) / (2 * CD_STEP)
            best = np.minimum(best, rate @ c)
    return best


def _check_probe(oracle, c):
    shape, lo, hi = PROBE_LAT
    lat = oracle.Lattice(oracle.TTR, shape, lo, hi)
    X = np.stack(np.meshgrid(*lat.coords, indexing='ij'), -1)
    u = X @ c + 0.3
    alpha, _ = oracle.dissipation(lat)
    V = oracle.rk3_step(lat, u, alpha, PROBE_H)
    inner = tuple(slice(EDGE, n - EDGE) for n in shape)
    r, ui, Vi = X[inner].reshape(-1, 4), u[inner].ravel(), V[inner].ravel()
    H = _ref_hamiltonian(r, c, np.random.default_rng(5))
    rate = (Vi - ui) / PROBE_H
    scale = np.abs(H).max()
    tol = 64 * np.finfo(np.float64).eps * np.abs(ui).max() / PROBE_H + 1e-6 * scale
    err = np.abs(rate - np.minimum(H, 0.0))
    neg = H < 0
    assert 0.2 < neg.mean() < 0.9, "the probe needs cells on both sides of H = 0"
    for what, m in (('v <= V_MIN', r[:, 3] <= V_MIN), ('v >= V_MAX', r[:, 3] >= V_MAX)):
        assert (m & neg).any(), what
    return err.max(), tol, neg.mean()


@pytest.mark.parametrize('k', range(len(PROBE_C)))
def test_oracle_hamiltonian_is_the_unicycle_game(k):
    """One step of 1e-7 from u = c . x + b: (V - u) / h = min(0, H_ref) at every cell 3 nodes inside the lattice, where
    WENO5 returns the slope exactly and the dissipation vanishes."""
    err, tol, neg = _check_probe(HO, np.array(PROBE_C[k]))
    print(f"c={PROBE_C[k]}: H_ref < 0 at {neg:.0%}, max |(V - u)/h - min(0, H_ref)| = {err:.3e} (tol {tol:.3e})")
    assert err <= tol


MUTATIONS = {
    'max for min': ('np.where(a[k] < 0.0, hi[k], lo[k])', 'np.where(a[k] < 0.0, lo[k], hi[k])'),
    'flipped sin term': ('f1 = v * s', 'f1 = -(v * s)'),
    'no speed saturation': ("for cond, which in ((v <= AT_VMIN, 'lo3'), (v >= AT_VMAX, 'hi3')):",
                            'for cond, which in ():'),
}


@pytest.mark.parametrize('name', list(MUTATIONS))
def test_a_mutated_oracle_fails_the_game_check(name):
    old, new = MUTATIONS[name]
    src = open(HO.__file__).read()
    assert src.count(old) == 1, old
    mod = types.ModuleType('hj_solve_oracle_mutant')
    exec(compile(src.replace(old, new), HO.__file__, 'exec'), mod.__dict__)
    failed = 0
    for c in PROBE_C:
        err, tol, _ = _check_probe(mod, np.array(c))
        failed += err > tol
    assert failed > 0, f"the mutation '{name}' passes the game check"


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
def _cuda(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device='cuda')


def _assert_bits(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, what
    same = got.view(np.int64) == want.view(np.int64)
    if not same.all():
        i = tuple(np.argwhere(~same)[0])
        raise AssertionError(f"{what}: {int((~same).sum())} of {same.size} values differ; first {i}: "
                             f"got {got[i]!r} want {want[i]!r}")


SMALL_LO, SMALL_HI = (-1.5, -1.5, -math.pi, V_MIN), (1.5, 1.5, math.pi, V_MAX)


# 2- and 3-node dims: both extrapolation ghosts fire in the same cell, and on a 2-node theta the periodic wrap adds
# (subtracts) n twice
@gpu
@pytest.mark.parametrize('shape', [(9, 11, 8, 5), (11, 7, 12, 6), (2, 3, 3, 2), (3, 2, 2, 3), (7, 9, 5, 4)])
@pytest.mark.parametrize('cfl', [0.5, 0.75, 1.0])
def test_solve_ttr_equals_the_oracle_bit_for_bit(shape, cfl):
    lo, hi = SMALL_LO, SMALL_HI
    l = R.ttr_target(shape, lo, hi)
    rng = np.random.default_rng(11)
    _, dt = R.ttr_dissipation(shape, lo, hi, cfl)
    arrived = 0
    for init in (l, l + 0.05 * rng.standard_normal(shape)):      # noise: every ghost sign and WENO branch
        for horizon in (0.0, 2.5 * dt, 7.3 * dt, 12.0 * dt):
            ttr, V = R.solve_ttr(_cuda(init), lo, hi, horizon, cfl)
            want_t, want_v = HO.solve_ttr(init, lo, hi, horizon, cfl)
            _assert_bits(ttr.cpu().numpy(), want_t, f'ttr {shape} cfl={cfl} horizon={horizon}')
            _assert_bits(V.cpu().numpy(), want_v, f'V {shape} cfl={cfl} horizon={horizon}')
            if horizon == 0.0:
                _assert_bits(V.cpu().numpy(), init, 'horizon 0')
            arrived += int(((want_t > 0) & np.isfinite(want_t)).sum())
    if min(shape) >= 4:
        assert arrived > 0, "no cell arrived during the solve: the arrival path was not compared"


@gpu
def test_ttr_arrays_past_2_31_bytes_advance_one_step():
    import torch
    shape, lo, hi = (401, 401, 24, 73), TTR_LAT[1], TTR_LAT[2]
    cells = int(np.prod(shape))
    assert cells * 8 > 2 ** 31
    lat = HO.Lattice(HO.TTR, shape, lo, hi)
    x = torch.as_tensor(lat.coords[0], device='cuda').view(-1, 1, 1, 1)
    y = torch.as_tensor(lat.coords[1], device='cuda').view(1, -1, 1, 1)
    th = torch.as_tensor(lat.coords[2], device='cuda').view(1, 1, -1, 1)
    init = (torch.sqrt(x * x + y * y) - GOAL_R + 0.01 * torch.cos(th)).expand(shape).contiguous()
    alpha, dt = R.ttr_dissipation(shape, lo, hi)
    ttr, V = R.solve_ttr(init, lo, hi, dt)
    hit = torch.nonzero((ttr > 0) & torch.isfinite(ttr))
    assert hit.shape[0] > 0
    rng = np.random.default_rng(3)
    samples = [tuple(int(rng.integers(0, n)) for n in shape) for _ in range(4)]
    samples += [tuple(int(v) for v in hit[int(rng.integers(0, hit.shape[0]))].tolist()) for _ in range(4)]
    samples += [(0, 0, 0, 0), tuple(n - 1 for n in shape), (400, 3, 23, 36), (2, 398, 1, 72)]
    for c in samples:
        starts = [max(0, k - 9) for k in c]
        stops = [min(n, k + 10) for k, n in zip(c, shape)]
        starts[2], stops[2] = 0, shape[2]                        # the whole periodic dim
        block = init[tuple(slice(a, b) for a, b in zip(starts, stops))].cpu().numpy()
        u3 = HO.step_at(lat, block, starts, alpha, dt)
        t = np.where(block <= 0.0, 0.0, np.inf)
        HO.arrive(t, block, u3, 0.0, dt)
        at = tuple(k - a for k, a in zip(c, starts))
        for what, got, want in (('V', float(V[c]), u3[at]), ('ttr', float(ttr[c]), t[at])):
            assert np.float64(got).view(np.int64) == np.float64(want).view(np.int64), (what, c, got, want)


@gpu
def test_ttr_side_stream():
    import torch
    l = _cuda(R.ttr_target(*TTR_LAT))
    ref = R.solve_ttr(l, *TTR_LAT[1:], 40.0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = R.solve_ttr(l, *TTR_LAT[1:], 40.0)
        done = torch.cuda.Event()
        done.record(s)
    done.synchronize()
    for a, b in zip(got, ref):
        assert torch.equal(a.view(torch.int64), b.view(torch.int64))


# --- the game ---------------------------------------------------------------------------------------------------------
def _t_star(D, v):
    """Least time to cover distance D >= 0 from speed v along a straight line: full acceleration to V_MAX, then cruise."""
    D, v = np.broadcast_arrays(np.asarray(D, np.float64), np.asarray(v, np.float64))
    t1 = (V_MAX - v) / AMAX
    d1 = 0.5 * (v + V_MAX) * t1
    accel = (-v + np.sqrt(v * v + 2 * AMAX * D)) / AMAX
    return np.where(D <= d1, accel, t1 + (D - d1) / V_MAX)


_SOLVED = {}


def _solved(shape=TTR_LAT[0], horizon=R.DEFAULT_TTR_HORIZON):
    key = (tuple(shape), horizon)
    if key not in _SOLVED:
        l = _cuda(R.ttr_target(shape, *TTR_LAT[1:]))
        _SOLVED[key] = R.solve_ttr(l, *TTR_LAT[1:], horizon)[0].cpu().numpy()
    return _SOLVED[key]


def _row_error(shape):
    """Max |TTR - t*| on the y = 0, theta = 0 row over x in [-6, -0.8] and every speed node."""
    t = _solved(shape)
    lat = HO.Lattice(HO.TTR, shape, *TTR_LAT[1:])
    x, th, v = lat.coords[0], lat.coords[2], lat.coords[3]
    j, k = shape[1] // 2, int(np.argmin(np.abs(th)))
    assert lat.coords[1][j] == 0.0 and abs(th[k]) < 1e-12
    sel = (x >= -6.0 - 1e-9) & (x <= -0.8 + 1e-9)
    want = _t_star(np.abs(x[sel])[:, None] - GOAL_R, v[None, :])
    return np.abs(t[sel, j, k, :] - want).max(), (t[sel, j, k, :] - want)


# first measured on an NVIDIA B200 (1000 W power limit), default lattice; each tolerance is that value with a margin
ROW_TOL = 4.0          # s: straight-line row error 2.90 s (x1.4)
LOWER_TOL = 0.5        # s: smallest TTR - lower bound 0.000 s (at the target), 0.5 s below it
ROLLOUT_TOL = 12.0     # s: greedy and perturbed rollouts beat TTR(x0) by up to 9.06 s (x1.3)
SYM_TOL = 1e-6         # s: mirror deviation 5.8e-8 s (x17)


@gpu
def test_straight_line_closed_form_and_refinement():
    """On y = 0, theta = 0, x < 0 the goal is straight ahead and full acceleration is optimal, so TTR = t*(|x| - r, v)."""
    err, d = _row_error(TTR_LAT[0])
    fine = (2 * TTR_LAT[0][0] - 1, 2 * TTR_LAT[0][1] - 1) + TTR_LAT[0][2:]
    err_fine, _ = _row_error(fine)
    print(f"straight-line row: max |TTR - t*| = {err:.3f} s on {TTR_LAT[0]} (signed {d.min():.3f} .. {d.max():.3f}), "
          f"{err_fine:.3f} s on {fine}")
    assert err <= ROW_TOL
    assert err_fine < err


@gpu
def test_no_cell_beats_the_no_turn_lower_bound():
    """No path to the goal disc is shorter than the straight line at full acceleration: TTR >= t*(max(0, d - r), v)."""
    t = _solved()
    lat = HO.Lattice(HO.TTR, *TTR_LAT)
    x, y, v = lat.coords[0], lat.coords[1], lat.coords[3]
    d = np.sqrt(x[:, None] ** 2 + y[None, :] ** 2)
    lb = _t_star(np.maximum(0.0, d - GOAL_R)[:, :, None, None], v[None, None, None, :])
    fin = np.isfinite(t)
    gap = (t - lb)[fin]
    print(f"TTR - lower bound: min {gap.min():.3f} s over {int(fin.sum())} reached cells")
    assert gap.min() >= -LOWER_TOL


@gpu
def test_mirror_symmetry():
    """(x, y, theta, v) -> (x, -y, -theta, v) is a symmetry of the game and of the target."""
    t = _solved()
    n = TTR_LAT[0][2]
    flip = t[:, ::-1][:, :, (-np.arange(n)) % n]
    fin = np.isfinite(t)
    assert (fin == np.isfinite(flip)).all()
    dev = np.abs(t - flip)[fin].max()
    print(f"mirror symmetry: max |TTR(x, y, th, v) - TTR(x, -y, -th, v)| = {dev:.3e} s")
    assert dev <= SYM_TOL


def _interp(t, lat, s):
    """Multilinear interpolation of the grid t at states s (..., 4), theta wrapped; off-lattice positions clamp."""
    out = 0.0
    idx, frac = [], []
    for d in range(4):
        n, sp, lo = lat.shape[d], lat.spacing[d], lat.coords[d][0]
        z = (s[..., d] - lo) / sp
        if lat.periodic[d]:
            i0 = np.floor(z)
            f = z - i0
            i0 = i0.astype(np.int64) % n
            idx.append((i0, (i0 + 1) % n))
        else:
            z = np.clip(z, 0.0, n - 1.0)
            i0 = np.minimum(np.floor(z).astype(np.int64), n - 2)
            f = z - i0
            idx.append((i0, i0 + 1))
        frac.append(f)
    for corner in range(16):
        b = [(corner >> d) & 1 for d in range(4)]
        w = 1.0
        for d in range(4):
            w = w * (frac[d] if b[d] else 1.0 - frac[d])
        out = out + w * t[idx[0][b[0]], idx[1][b[1]], idx[2][b[2]], idx[3][b[3]]]
    return out


def _in_goal(s):
    d = np.sqrt(s[..., 0] ** 2 + s[..., 1] ** 2)
    return np.maximum(d - GOAL_R, (GOAL_R / H_THR) * ((0.5 - 0.5 * np.cos(s[..., 2])) - H_THR)) <= 0.0


def _advance(s, w, a, h):
    """One RK4 step of the unicycle under constant (w, a), with the speed saturation; speeds clamped to the box."""
    a = np.where((s[..., 3] <= V_MIN) & (a < 0), 0.0, a)
    a = np.where((s[..., 3] >= V_MAX) & (a > 0), 0.0, a)

    def f(z):
        return np.stack([z[..., 3] * np.cos(z[..., 2]), z[..., 3] * np.sin(z[..., 2]), np.broadcast_to(w, z.shape[:-1]),
                         np.broadcast_to(a, z.shape[:-1])], -1)
    k1 = f(s); k2 = f(s + 0.5 * h * k1); k3 = f(s + 0.5 * h * k2); k4 = f(s + h * k3)
    out = s + (h / 6.0) * (k1 + 2 * k2 + 2 * k3 + k4)
    out[..., 3] = np.clip(out[..., 3], V_MIN, V_MAX)
    return out


CONTROLS = [(w, a) for w in (-W, 0.0, W) for a in (AMIN, 0.0, AMAX)]
DECIDE, SUB = 1.0, 4            # a control is held for DECIDE seconds; the goal test runs every DECIDE / SUB


def _rollout(t, lat, s0, eps, rng, t_end):
    """Drive the unicycle from s0 (m, 4): greedy on the interpolated TTR (the control whose state after DECIDE s has the
    least TTR, or that enters the goal set soonest within those DECIDE s), with probability eps a uniformly random
    control instead. -> first time in the goal set (inf: never). The goal set itself is known exactly: near it the
    lattice (0.4 km spacing around a 0.35 km disc) blends cells on the target with cells that need a full turn."""
    s = s0.copy()
    m = s.shape[0]
    reach = np.full(m, np.inf)
    reach[_in_goal(s)] = 0.0
    now = 0.0
    while now < t_end and np.isinf(reach).any():
        cand = []
        for w, a in CONTROLS:
            z = s
            enter = np.full(m, np.inf)
            for k in range(SUB):
                z = _advance(z, w, a, DECIDE / SUB)
                enter = np.where(np.isinf(enter) & _in_goal(z), (k + 1) * DECIDE / SUB - 1e3, enter)
            cand.append(np.minimum(enter, _interp(t, lat, z)))
        pick = np.argmin(np.stack(cand), axis=0)
        rnd = rng.random(m) < eps
        pick = np.where(rnd, rng.integers(0, len(CONTROLS), m), pick)
        w = np.array([CONTROLS[k][0] for k in pick])
        a = np.array([CONTROLS[k][1] for k in pick])
        for _ in range(SUB):
            s = _advance(s, w, a, DECIDE / SUB)
            now += DECIDE / SUB
            new = np.isinf(reach) & _in_goal(s)
            reach[new] = now
    return reach


@gpu
def test_rollouts_attain_and_never_beat_the_ttr():
    """Greedy rollouts on the interpolated TTR reach the goal in TTR(x0) within ROLLOUT_TOL; perturbed rollouts
    (30 % random controls) never beat TTR(x0) by more than ROLLOUT_TOL.

    Measured on the default lattice (96 starts): greedy T - TTR(x0) from -9.06 s to +8.0 s, so ROLLOUT_TOL = 12 s. TTR
    is above the greedy time where the path turns (theta spacing 15 deg). 4 starts pass through the goal disc with the
    heading outside the 45 deg cone, where the 0.4 km lattice cannot resolve the 0.35 km disc, and turn once more
    (+45 to +50 s, one turn being 2 pi / w = 63 s); the test allows that for at most 10 % of the starts."""
    t = _solved()
    lat = HO.Lattice(HO.TTR, *TTR_LAT)
    tt = np.where(np.isinf(t), R.DEFAULT_TTR_HORIZON, t)
    rng = np.random.default_rng(17)
    m = 96
    s0 = np.stack([rng.uniform(-5, 5, m), rng.uniform(-5, 5, m), rng.uniform(-math.pi, math.pi, m),
                   rng.uniform(V_MIN, V_MAX, m)], -1)
    s0 = s0[~_in_goal(s0)]
    v0 = _interp(tt, lat, s0)
    greedy = _rollout(tt, lat, s0, 0.0, rng, 400.0)
    assert np.isfinite(greedy).all(), "a greedy rollout never reached the goal"
    dg = greedy - v0
    loops = dg > ROLLOUT_TOL
    print(f"greedy: T - TTR(x0) in [{dg.min():.2f}, {dg[~loops].max():.2f}] s over {len(s0)} starts "
          f"(TTR(x0) {v0.min():.1f} .. {v0.max():.1f} s); {int(loops.sum())} miss the goal set and turn once more: "
          f"{np.round(np.sort(dg[loops]), 1)} s")
    assert dg.min() >= -ROLLOUT_TOL
    assert loops.mean() <= 0.1 and (dg <= 2 * math.pi / W + ROLLOUT_TOL).all()
    best = np.full(len(s0), np.inf)
    for k in range(4):
        best = np.minimum(best, _rollout(tt, lat, s0, 0.3, np.random.default_rng(100 + k), 400.0))
    dp = (best - v0)[np.isfinite(best)]
    print(f"perturbed: {int(np.isfinite(best).sum())} of {len(s0)} starts reached; min T - TTR(x0) = {dp.min():.2f} s")
    assert dp.min() >= -ROLLOUT_TOL


@gpu
def test_default_horizon_reaches_the_interior():
    """Unreached fractions at H and 2H; no cell more than 2 km inside the x/y boundary (one turning diameter,
    2 V_MAX / W = 1.8 km, plus margin) is unreached at H; cells reached before H's last step have the same bits in the
    H and 2H solves."""
    H = R.DEFAULT_TTR_HORIZON
    t1, t2 = _solved(horizon=H), _solved(horizon=2 * H)
    lat = HO.Lattice(HO.TTR, *TTR_LAT)
    x, y = lat.coords[0], lat.coords[1]
    inner = ((np.abs(x)[:, None] <= 8.0 - 2.0 + 1e-9) & (np.abs(y)[None, :] <= 8.0 - 2.0 + 1e-9))[:, :, None, None]
    inner = np.broadcast_to(inner, t1.shape)
    print(f"unreached at H = {H:.0f} s: {np.isinf(t1).mean():.4%} of cells ({np.isinf(t1[inner]).mean():.4%} of the "
          f"interior); at 2H: {np.isinf(t2).mean():.4%}; max finite TTR {t1[np.isfinite(t1)].max():.2f} s")
    assert not np.isinf(t1[inner]).any()
    _, dt = R.ttr_dissipation(*TTR_LAT)
    tau = 0.0
    while H - tau > dt:
        tau = tau + dt
    before = t1 <= tau                                          # tau: the start of H's last (clipped) step
    _assert_bits(t2[before], t1[before], 'cells reached before the last step of H')
    assert (t2[np.isinf(t1)] > tau).all()


@gpu
@pytest.mark.parametrize('f32', [False, True])
def test_computed_ttr_grid_drives_the_env_bit_for_bit_with_the_oracle(f32):
    import test_cuda_parity as P
    from layered_safe_marl_b200 import config as cfg
    tg = R.ttr_grid()
    assert tg.values.dtype == np.float32 and tg.grads is None and tg.periodic == (False, False, True, False)
    assert tg.ttr_max == R.DEFAULT_TTR_HORIZON and np.isfinite(tg.values).all()
    args = G.default_args(dynamics_type='airtaxi', num_agents=10, use_safety_filter=True, episode_length=350,
                          world_size=6, interp_float32=f32)
    flags = G.BinaryFlags(dict(POTENTIAL_CONFLICT=True))
    vg, synth = G.value_grid_for(cfg.scenario_params_from_args(args, binary_cfg=flags))
    _, cu = P._compare_with_oracle(args, flags, n=256, T=8, episode=6249, seed=5, auto_reset=True, grids=(vg, tg))
    rew = cu.reward.copy()
    _, cu_s = P._compare_with_oracle(args, flags, n=256, T=8, episode=6249, seed=5, auto_reset=True,
                                     grids=(vg, synth))
    differ = (rew != cu_s.reward).mean()
    print(f"interp_float32={f32}: rewards at the last step differ from the synthetic-grid run in {differ:.1%}")
    assert differ > 0
