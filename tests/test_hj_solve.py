"""The HJ reachability solver (liblsm_b200_hj.so, layered_safe_marl_b200.reachability) against the numpy restatement
of its declared scheme (tests/hj_solve_oracle.py).

CPU: the ctypes mirror of lsm_hj_problem; the library builds for sm_100a and exports its symbols; the host-side
dissipation coefficients and time step equal the oracle's bit for bit; every invalid argument is refused with code 2;
the oracle checks itself (WENO5 order, extrapolation ghosts, the analytic slab).
GPU: the CUDA solve equals the oracle bit for bit; the slab's closed form on the default lattice; the tube's
invariants and symmetries; computed grids through the environment and SafetyFilter, bit for bit with the C oracle;
arrays past 2^31 bytes; a side stream."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))
sys.path.insert(0, os.path.join(REPO, 'tests'))

import _golden as G  # noqa: E402
import hj_solve_oracle as HO  # noqa: E402
from layered_safe_marl_b200 import _build, _lib, hj_grid  # noqa: E402
from layered_safe_marl_b200 import reachability as R  # noqa: E402

gpu = pytest.mark.gpu
DI_LAT = (hj_grid.DI_GRID_SHAPE, hj_grid.DI_GRID_LO, hj_grid.DI_GRID_HI)
AT_LAT = (hj_grid.AIRTAXI_GRID_SHAPE, hj_grid.AIRTAXI_GRID_LO, hj_grid.AIRTAXI_GRID_HI)


def _ulps(v, k=4):
    """k units in the last place of v: the RK3 combinations (3/4 u + 1/4 u, 1/3 u + 2/3 u) round, so a cell the tube
    leaves alone can move by an ulp either way."""
    return k * np.spacing(np.abs(v))


def _problem(dyn, shape, lo, hi, cfl=0.75):
    return R._problem(dyn, shape, lo, hi, cfl)


# ----------------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------------
def test_problem_mirror_matches_the_c_header(tmp_path):
    cls = _lib.LsmHjProblem
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lsm_b200_hj.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(lsm_hj_problem));']
    lines += [f'  printf("{f} %zu\\n", offsetof(lsm_hj_problem, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / 'p.c', tmp_path / 'p.exe'
    src.write_text('\n'.join(lines))
    subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), '-o', str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    assert int(got['size']) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def test_hj_library_builds_for_sm100a_and_exports_its_symbols():
    path = _build.build_hj()
    lib = ctypes.CDLL(path)
    declared = set(re.findall(r'\b(lsm_[a-z_]+)\s*\(', open(os.path.join(REPO, 'include', 'lsm_b200_hj.h')).read()))
    assert declared == set(_lib.HJ_EXPORTED_SYMBOLS), declared ^ set(_lib.HJ_EXPORTED_SYMBOLS)
    for sym in declared:
        getattr(lib, sym)
    hj = _lib.load_hj()
    assert hj.lsm_hj_abi_version() == 1
    pr = _problem(0, *DI_LAT)
    assert hj.lsm_hj_work_bytes(ctypes.byref(pr)) == 8 * (3 * int(np.prod(DI_LAT[0])) + sum(DI_LAT[0]))
    pr = _problem(1, *AT_LAT)
    assert hj.lsm_hj_work_bytes(ctypes.byref(pr)) == 8 * (3 * int(np.prod(AT_LAT[0])) + sum(AT_LAT[0]) + 2 * AT_LAT[0][2])
    nvcc = shutil.which(os.environ.get('NVCC', 'nvcc'))
    exe = os.path.join(os.path.dirname(nvcc), 'cuobjdump') if nvcc else shutil.which('cuobjdump')
    assert exe and os.path.exists(exe), "cuobjdump (CUDA toolkit) not found next to nvcc"
    assert 'sm_100a' in subprocess.check_output([exe, '-lelf', path], text=True)
    assert 'lsm_hj_stage_kernel' in subprocess.check_output([exe, '-sass', path], text=True)


@pytest.mark.parametrize('dyn,shape,cfl', [(0, DI_LAT[0], 0.75), (0, (9, 11, 7, 5), 0.5), (1, AT_LAT[0], 0.75),
                                           (1, (9, 9, 8, 5, 5), 0.5), (1, (7, 9, 5, 4, 6), 1.0)])
def test_dissipation_equals_the_oracle_bit_for_bit(dyn, shape, cfl):
    lo, hi = (DI_LAT if dyn == 0 else AT_LAT)[1:]
    alpha, dt = R.dissipation(dyn, shape, lo, hi, cfl)
    o_alpha, o_dt = HO.dissipation(HO.Lattice(dyn, shape, lo, hi), cfl)
    assert np.array_equal(alpha, o_alpha) and dt == o_dt, (alpha, o_alpha, dt, o_dt)
    if dyn == 0:
        assert np.array_equal(alpha, [1.0, 1.0, 1.0, 1.0])


def test_invalid_arguments_are_refused_with_code_2():
    """Validation runs on the host before anything is enqueued: code 2 and a message, no device needed."""
    lib = _lib.load_hj()
    fake = ctypes.c_void_p(4096)                   # never dereferenced: every case below fails validation first
    h_ok = (ctypes.c_double * 2)(0.0, 1.0)

    def solve_rc(pr, horizons=h_ok, K=2, initial=fake, out=fake, work=fake):
        return lib.lsm_hj_solve(pr, initial, horizons, K, out, work, None)

    def bad(**kw):
        pr = _problem(0, *DI_LAT)
        for k, v in kw.items():
            if k in ('shape', 'lo', 'hi'):
                d, x = v
                getattr(pr, k)[d] = x
            else:
                setattr(pr, k, v)
        return pr

    cases = [bad(dynamics=2), bad(dynamics=-1), bad(shape=(0, 1)), bad(shape=(3, 0)), bad(lo=(1, 4.5)),
             bad(lo=(2, float('nan'))), bad(hi=(0, float('inf'))), bad(cfl=0.0), bad(cfl=1.5), bad(cfl=float('nan')),
             bad(cfl=-0.5)]
    for pr in cases:
        assert solve_rc(ctypes.byref(pr)) == 2, lib.lsm_hj_last_error()
        assert lib.lsm_hj_work_bytes(ctypes.byref(pr)) == 0
        a, dt = (ctypes.c_double * 5)(), ctypes.c_double()
        assert lib.lsm_hj_dissipation(ctypes.byref(pr), a, ctypes.byref(dt)) == 2
    assert lib.lsm_hj_dissipation(None, None, None) == 2
    pr = ctypes.byref(_problem(1, *AT_LAT))
    assert solve_rc(None) == 2
    for horizons in ((-1.0, 1.0), (0.0, float('nan')), (0.0, float('inf')), (2.0, 1.0)):
        assert solve_rc(pr, (ctypes.c_double * 2)(*horizons)) == 2, horizons
        assert b'horizons' in lib.lsm_hj_last_error()
    assert solve_rc(pr, K=0) == 2
    assert solve_rc(pr, horizons=None) == 2
    assert solve_rc(pr, initial=None) == 2
    assert solve_rc(pr, out=None) == 2
    assert solve_rc(pr, work=None) == 2
    assert solve_rc(pr, work=ctypes.c_void_p(4097)) == 2 and b'aligned' in lib.lsm_hj_last_error()
    with pytest.raises(RuntimeError, match='cfl'):
        R.dissipation('double_integrator', DI_LAT[0], DI_LAT[1], DI_LAT[2], cfl=2.0)
    with pytest.raises(ValueError):
        R.dissipation('double_integrator', (5, 5, 5), (0, 0, 0), (1, 1, 1))
    with pytest.raises(TypeError):
        import torch
        R.solve('double_integrator', torch.zeros(DI_LAT[0], dtype=torch.float64), *DI_LAT[1:], [1.0])


def test_weno5_order_on_a_smooth_periodic_function():
    """Halving the spacing cuts the derivative error by at least 2^3 (Jiang-Peng weights are third order at critical
    points; fifth order elsewhere)."""
    errs = []
    for n in (32, 64, 128):
        x = 2 * np.pi * np.arange(n) / n
        v = np.sin(x) + 0.5 * np.cos(2 * x)
        exact = np.cos(x) - np.sin(2 * x)
        left, right = HO.derivs(v, 0, 1.0 / (2 * np.pi / n), True)
        errs.append(max(np.abs(left - exact).max(), np.abs(right - exact).max()))
    ratios = [errs[i] / errs[i + 1] for i in range(len(errs) - 1)]
    print(f"WENO5 max error {errs}, ratios per halving {ratios}")
    assert all(r >= 8.0 for r in ratios), ratios


def test_extrapolation_ghosts():
    v = np.array([[-2.0, 3.0], [-1.5, 0.0], [0.5, 0.0], [1.0, 4.0], [3.0, -1.0]])
    p = HO.pad(v, 0, False)
    assert p.shape == (11, 2)
    assert np.array_equal(p[3:8], v)
    # away from zero: v[-j] = v[0] + sign(v[0]) |v[1] - v[0]| j
    assert np.array_equal(p[:3, 0], [-2.0 - 1.5, -2.0 - 1.0, -2.0 - 0.5])
    assert np.array_equal(p[:3, 1], [3.0 + 9.0, 3.0 + 6.0, 3.0 + 3.0])
    assert np.array_equal(p[8:, 0], [3.0 + 2.0, 3.0 + 4.0, 3.0 + 6.0])
    assert np.array_equal(p[8:, 1], [-1.0 - 5.0, -1.0 - 10.0, -1.0 - 15.0])
    z = HO.pad(np.array([0.0, 2.0, 1.0]), 0, False)                 # sign(0) = 0: constant ghosts
    assert np.array_equal(z[:3], [0.0, 0.0, 0.0])
    w = HO.pad(np.arange(4.0), 0, True)
    assert np.array_equal(w, [1.0, 2.0, 3.0, 0.0, 1.0, 2.0, 3.0, 0.0, 1.0, 2.0])


def _slab(shape, r=0.5, lo=DI_LAT[1], hi=DI_LAT[2]):
    """The slab target l = |px| - r, its closed-form tube value max(|px| - [px vx < 0] vx^2 / 2, 0) - r (total
    cooperative deceleration 1) and the comparison mask (|px| <= 3.5, |vx| <= 0.8, 2 cells off the kinks)."""
    lat = HO.Lattice(0, shape, lo, hi)
    px = lat.coords[0][:, None, None, None]
    vx = lat.coords[2][None, None, :, None]
    l = np.broadcast_to(np.abs(px) - r, shape).copy()
    exact = np.broadcast_to(np.maximum(np.abs(px) - (px * vx < 0) * vx ** 2 / 2, 0.0) - r, shape)
    dx0, dx2 = lat.spacing[0], lat.spacing[2]
    kink = (np.abs(np.abs(px) - vx ** 2 / 2) < 2 * dx0 + 2 * dx2 * np.abs(vx)) | (np.abs(px) < 2 * dx0)
    mask = np.broadcast_to((np.abs(px) <= 3.5) & (np.abs(vx) <= 0.8) & ~kink, shape)
    return l, exact, mask


def test_oracle_meets_the_analytic_slab():
    shape = (41, 3, 41, 3)
    l, exact, mask = _slab(shape)
    V = HO.solve(0, l, DI_LAT[1], DI_LAT[2], [2.0])[0]
    err = np.abs(V - exact)[mask].max()
    print(f"slab (41, 3, 41, 3), horizon 2 s: max |V - V*| = {err:.3e} m over {int(mask.sum())} cells")
    assert err < 0.1
    assert (V <= l + _ulps(l)).all()


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


# 2- and 3-node dims: both extrapolation ghosts of derivs fire in the same cell, and on a 2-node theta the periodic wrap
# adds (subtracts) n twice
@gpu
@pytest.mark.parametrize('dyn,shape', [(0, (9, 11, 7, 5)), (0, (6, 6, 6, 6)), (1, (9, 9, 8, 5, 5)), (1, (7, 5, 9, 4, 6)),
                                       (0, (2, 3, 9, 3)), (0, (7, 2, 2, 3)), (1, (3, 2, 2, 3, 5)),
                                       (1, (2, 7, 3, 2, 3))])
@pytest.mark.parametrize('cfl', [0.75, 0.5])
def test_solve_equals_the_oracle_bit_for_bit(dyn, shape, cfl):
    _, lo, hi = DI_LAT if dyn == 0 else AT_LAT
    sep = 0.5 if dyn == 0 else 0.4572
    l = R.target(dyn, shape, lo, hi, sep)
    rng = np.random.default_rng(7 + dyn)
    for init in (l, l + 0.05 * rng.standard_normal(shape)):      # noise: every ghost sign and WENO branch
        _, dt = R.dissipation(dyn, shape, lo, hi, cfl)
        horizons = [0.0, 2.5 * dt, 2.5 * dt, 7.3 * dt, 7.3 * dt + 1e-9, 11.0 * dt]
        got = R.solve(dyn, _cuda(init), lo, hi, horizons, cfl).cpu().numpy()
        want = HO.solve(dyn, init, lo, hi, horizons, cfl)
        _assert_bits(got[0], init, 'horizon 0')
        _assert_bits(got[1], got[2], 'repeated horizon')
        _assert_bits(got, want, f'dyn={dyn} shape={shape} cfl={cfl}')


@gpu
def test_slab_on_the_default_lattice_and_refined():
    errs = []
    for shape in (DI_LAT[0], (81, 5, 41, 3)):
        l, exact, mask = _slab(shape)
        V = R.solve(0, _cuda(l), DI_LAT[1], DI_LAT[2], [2.0])[0].cpu().numpy()
        errs.append(np.abs(V - exact)[mask].max())
        assert (V <= l + _ulps(l)).all()
        # no dependence on py or vy at all: bitwise constant along both
        _assert_bits(V, np.broadcast_to(V[:, :1, :, :1], V.shape), f'{shape}: constant along py and vy')
    print(f"slab max |V - V*|: default lattice {errs[0]:.3e} m, (px, vx) spacing halved {errs[1]:.3e} m")
    assert errs[0] < 0.1 and errs[1] < errs[0]


@gpu
def test_tube_invariants_and_symmetries():
    shape, lo, hi = DI_LAT
    l = R.target(0, shape, lo, hi, 0.5)
    V = R.solve(0, _cuda(l), lo, hi, [0.5, 1.0, 2.0, 4.0]).cpu().numpy()
    assert (V <= l + _ulps(l)).all()
    assert (V[1:] <= V[:-1] + _ulps(V[:-1])).all()
    np.testing.assert_allclose(V[-1], V[-1][::-1, ::-1, ::-1, ::-1], rtol=0, atol=1e-9)     # (x, v) -> (-x, -v)
    np.testing.assert_allclose(V[-1], V[-1].transpose(1, 0, 3, 2), rtol=0, atol=1e-9)        # x <-> y
    shape, lo, hi = AT_LAT
    l = R.target(1, shape, lo, hi, 0.4572)
    V = R.solve(1, _cuda(l), lo, hi, [10.0, 30.0]).cpu().numpy()
    assert (V <= l + _ulps(l)).all()
    assert (V[1] <= V[0] + _ulps(V[0])).all()
    n = shape[2]
    flip = V[-1][:, ::-1][:, :, (-np.arange(n)) % n]                                          # (y, th) -> (-y, -th)
    np.testing.assert_allclose(V[-1], flip, rtol=0, atol=1e-9)


@gpu
def test_default_horizons_have_converged():
    for dyn in (0, 1):
        shape, lo, hi = DI_LAT if dyn == 0 else AT_LAT
        H = R.DEFAULT_HORIZON[dyn]
        sep = 0.5 if dyn == 0 else 0.4572
        V = R.solve(dyn, _cuda(R.target(dyn, shape, lo, hi, sep)), lo, hi, [H / 2, H]).cpu().numpy()
        d = np.abs(V[1] - V[0]).max()
        print(f"dynamics {dyn}: max|V({H}) - V({H / 2})| = {d:.3e}")
        assert d < 1e-3 * (np.abs(V[1]).max())


_COMPUTED = {}


def _computed(dyn):
    if dyn not in _COMPUTED:
        _COMPUTED[dyn] = R.value_grid(dyn)
    return _COMPUTED[dyn]


@gpu
@pytest.mark.parametrize('case', ['cfg2', 'cfg3'])
def test_computed_grid_drives_the_env_bit_for_bit_with_the_oracle(case, monkeypatch):
    import test_cuda_parity as P
    from layered_safe_marl_b200 import vec_env
    dyn = 0 if case == 'cfg2' else 1
    grid = _computed(dyn)
    assert grid.values.dtype == np.float32 and grid.grads.shape == grid.shape + (grid.ndim,)
    ttr = hj_grid.synthetic_ttr_grid() if dyn == 1 else None
    monkeypatch.setattr(G, 'value_grid_for', lambda params: (grid, ttr))
    monkeypatch.setattr(vec_env, 'synthetic_di_grid' if dyn == 0 else 'synthetic_airtaxi_grid', lambda: grid)
    if dyn == 0:
        args = G.default_args(num_agents=8, use_safety_filter=True, episode_length=250, world_size=4)
        flags = G.BinaryFlags({})
    else:
        args = G.default_args(dynamics_type='airtaxi', num_agents=10, use_safety_filter=True, episode_length=350,
                              world_size=6)
        flags = G.BinaryFlags(dict(POTENTIAL_CONFLICT=True))
    ora, cu = P._compare_with_oracle(args, flags, n=256, T=8, episode=6249, seed=4 + dyn, auto_reset=True)
    filtered = int(np.asarray(cu.get_state()['safety_filtered']).sum())
    print(f"{case}: filter activations at the last step with the computed grid: {filtered}")


@gpu
@pytest.mark.parametrize('dyn', [0, 1])
def test_safety_filter_over_a_computed_grid_equals_the_oracle(dyn):
    import test_safety_filter_op as F
    from layered_safe_marl_b200 import SafetyFilter
    grid = _computed(dyn)
    params = F._params(dyn, False)
    sf = SafetyFilter('double_integrator' if dyn == 0 else 'airtaxi', value_grid=grid)
    rng = np.random.default_rng(31 + dyn)
    ego, oth, ua, uo = F._random_rows(dyn, 4096, 7, rng)
    filt = F._compare_to_oracle(sf, params, grid, ego, oth, ua, uo, None, None, 'computed grid')
    assert 0 < filt.sum() < filt.size


@gpu
def test_arrays_past_2_31_bytes_advance_one_step():
    import torch
    shape, lo, hi = (181, 181, 91, 91), DI_LAT[1], DI_LAT[2]
    cells = int(np.prod(shape))
    assert cells * 8 > 2 ** 31
    lat = HO.Lattice(0, shape, lo, hi)
    px = torch.as_tensor(lat.coords[0], device='cuda').view(-1, 1, 1, 1)
    py = torch.as_tensor(lat.coords[1], device='cuda').view(1, -1, 1, 1)
    vx = torch.as_tensor(lat.coords[2], device='cuda').view(1, 1, -1, 1)
    init = (torch.sqrt(px * px + py * py) - 0.5 + 0.3 * vx).expand(shape).contiguous()
    alpha, dt = R.dissipation(0, shape, lo, hi)
    out = R.solve(0, init, lo, hi, [dt])[0]
    rng = np.random.default_rng(3)
    samples = [tuple(int(rng.integers(0, n)) for n in shape) for _ in range(6)]
    samples += [(0, 0, 0, 0), tuple(n - 1 for n in shape), (180, 3, 90, 45), (2, 178, 1, 89)]
    for c in samples:
        starts = [max(0, k - 9) for k in c]
        stops = [min(n, k + 10) for k, n in zip(c, shape)]
        block = init[tuple(slice(a, b) for a, b in zip(starts, stops))].cpu().numpy()
        want = HO.step_at(lat, block, starts, alpha, dt)[tuple(k - a for k, a in zip(c, starts))]
        got = float(out[c])
        assert np.float64(got).view(np.int64) == np.float64(want).view(np.int64), (c, got, want)


@gpu
def test_side_stream():
    import torch
    shape, lo, hi = AT_LAT
    l = _cuda(R.target(1, shape, lo, hi, 0.4572))
    ref = R.solve(1, l, lo, hi, [5.0])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = R.solve(1, l, lo, hi, [5.0])
        done = torch.cuda.Event()
        done.record(s)
    done.synchronize()
    assert torch.equal(got.view(torch.int64), ref.view(torch.int64))
