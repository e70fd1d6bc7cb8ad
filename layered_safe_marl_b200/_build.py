"""Build the sm_100a shared library in-tree (nvcc cross-compiles without a GPU).

    python -m layered_safe_marl_b200._build                      the product library (liblsm_b200.so)
    python -m layered_safe_marl_b200._build --shape airtaxi,6,2,0
                                                                 the library of one specialised shape (build_shape)
    python -m layered_safe_marl_b200._build --ppo                the PPO-input library (liblsm_b200_ppo.so, build_ppo)
    python -m layered_safe_marl_b200._build --hj                 the HJ reachability solver (liblsm_b200_hj.so, build_hj)
"""
from __future__ import annotations

import argparse
import fcntl
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.path.join(HERE, 'liblsm_b200.so')
SHAPES_DIR = os.path.join(HERE, 'shapes')
SOURCES = [os.path.join(CSRC, 'lsm_kernels.cu'), os.path.join(CSRC, 'lsm_capi.cu')]
DEPS = SOURCES + [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(('.cuh', '.h'))] + \
    [os.path.join(os.path.dirname(HERE), 'include', f) for f in ('lsm_b200.h', 'lsm_math.h')]

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              # no FMA contraction: float64 intermediates must round like the reference's numpy arithmetic
              '-fmad=false',
              # host code too (lsm_math.h on the host must round like the device and the oracle build)
              '-Xcompiler', '-ffp-contract=off',
              '-Xcompiler', '-fPIC', '-shared']

# the domain lsm_create accepts (include/lsm_b200.h LSM_MAX_AGENTS / LSM_MAX_LANDMARKS / LSM_MAX_OBSTACLES)
MAX_AGENTS, MAX_LANDMARKS, MAX_OBSTACLES = 32, 128, 32
DYNAMICS_TAG = {0: 'di', 1: 'at'}


def needs_build(path: str = LIB_PATH, deps=DEPS) -> bool:
    if not os.path.exists(path):
        return True
    t = os.path.getmtime(path)
    return any(os.path.getmtime(p) > t for p in deps)


# the PPO-input kernels (returns, advantages, advantage moments): no env handle, so a library of their own
PPO_LIB_PATH = os.path.join(HERE, 'liblsm_b200_ppo.so')
PPO_SOURCES = [os.path.join(CSRC, 'lsm_ppo.cu')]
PPO_DEPS = PPO_SOURCES + [os.path.join(os.path.dirname(HERE), 'include', 'lsm_b200_ppo.h')]


def build_ppo(force: bool = False, verbose: bool = False) -> str:
    """liblsm_b200_ppo.so from csrc/lsm_ppo.cu with the product library's flags; rebuilt when a source is newer."""
    if not force and not needs_build(PPO_LIB_PATH, PPO_DEPS):
        return PPO_LIB_PATH
    _nvcc([], PPO_LIB_PATH, verbose, sources=PPO_SOURCES)
    return PPO_LIB_PATH


# the HJ reachability solver (value functions for the safety filter): no env handle, so a library of its own
HJ_LIB_PATH = os.path.join(HERE, 'liblsm_b200_hj.so')
HJ_SOURCES = [os.path.join(CSRC, 'lsm_hj.cu')]
HJ_DEPS = HJ_SOURCES + [os.path.join(os.path.dirname(HERE), 'include', f) for f in ('lsm_b200_hj.h', 'lsm_math.h')]


def build_hj(force: bool = False, verbose: bool = False) -> str:
    """liblsm_b200_hj.so from csrc/lsm_hj.cu with the product library's flags; rebuilt when a source is newer."""
    if not force and not needs_build(HJ_LIB_PATH, HJ_DEPS):
        return HJ_LIB_PATH
    _nvcc([], HJ_LIB_PATH, verbose, sources=HJ_SOURCES)
    return HJ_LIB_PATH


EXP_LIB_PATH = os.path.join(HERE, 'liblsm_b200_exp.so')


def build_experiments(extra_flags=(), verbose: bool = False) -> str:
    """The lab build of the same sources: -DLSM_EXPERIMENTS compiles the ablation switches (LSM_DEBUG, LSM_WPE, LSM_PAIR,
    LSM_AGENT_MINB, ... read from the environment) and the alternative kernel instantiations that the product library
    does not contain. Tools select it with LSM_LIB=<path>."""
    build(force=True, verbose=verbose, extra_flags=['-DLSM_EXPERIMENTS'] + list(extra_flags), out_path=EXP_LIB_PATH)
    return EXP_LIB_PATH


def _nvcc(extra_flags, out_path: str, verbose: bool = False, sources=SOURCES) -> None:
    nvcc = os.environ.get('NVCC', 'nvcc')
    cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (['-Xptxas', '-v'] if verbose else []) + ['-o', out_path] + list(sources)
    try:
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    except OSError as exc:
        raise RuntimeError(f"nvcc could not be started ({nvcc}): {exc}") from exc
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout[-4000:])
    if verbose:
        print(proc.stdout)


def build(force: bool = False, verbose: bool = False, extra_flags=(), out_path: str = LIB_PATH) -> str:
    """`extra_flags` / `out_path` build an A/B variant (extra -D switches) next to the product library; a variant
    is selected at run time with LSM_LIB=<path> (experiments only)."""
    if not force and not needs_build() and out_path == LIB_PATH:
        return LIB_PATH
    _nvcc(extra_flags, out_path, verbose)
    return out_path


def parse_dynamics(dynamics) -> int:
    if isinstance(dynamics, str):
        key = dynamics.strip().lower()
        names = {'double_integrator': 0, 'di': 0, 'airtaxi': 1, 'at': 1}
        if key not in names and not key.isdigit():
            raise ValueError(f"unknown dynamics {dynamics!r} (double_integrator or airtaxi)")
        dynamics = names[key] if key in names else int(key)
    if int(dynamics) not in DYNAMICS_TAG:
        raise ValueError(f"dynamics must be 0 (double_integrator) or 1 (airtaxi), got {dynamics}")
    return int(dynamics)


def check_shape(dynamics, N: int, L: int, O: int):
    """-> (dynamics, N, L, O) as ints; raises ValueError outside the domain lsm_create accepts."""
    dyn = parse_dynamics(dynamics)
    N, L, O = int(N), int(L), int(O)
    if not 1 <= N <= MAX_AGENTS:
        raise ValueError(f"num_agents must be in [1, {MAX_AGENTS}], got {N}")
    if L < 2 or N * L > MAX_LANDMARKS:
        raise ValueError(f"num_landmarks must be >= 2 with num_agents * num_landmarks <= {MAX_LANDMARKS}, got {N} x {L}")
    if not 0 <= O <= MAX_OBSTACLES:
        raise ValueError(f"num_obstacles must be in [0, {MAX_OBSTACLES}], got {O}")
    return dyn, N, L, O


def shape_lib_path(dynamics, N: int, L: int, O: int) -> str:
    dyn, N, L, O = check_shape(dynamics, N, L, O)
    return os.path.join(SHAPES_DIR, f'liblsm_b200_{DYNAMICS_TAG[dyn]}{N}_l{L}_o{O}.so')


def build_shape(dynamics, N: int, L: int, O: int, force: bool = False, verbose: bool = False) -> str:
    """The library of ONE specialised shape: the product library's sources and flags with -DLSM_SHAPE=<dynamics N L O as digits DNNLLOO>,
    which replaces the compiled shape list by this shape (the generic kernels and the C ABI are unchanged). Rebuilt when
    a source is newer. Safe to call from several processes at once: one of them compiles (under a lock), into a private
    file that is renamed into place, and the others wait for it and return the same path."""
    dyn, N, L, O = check_shape(dynamics, N, L, O)
    path = shape_lib_path(dyn, N, L, O)
    if not force and not needs_build(path):
        return path
    os.makedirs(SHAPES_DIR, exist_ok=True)
    with open(path + '.lock', 'w') as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or needs_build(path):       # another process may have built it while this one waited
                fd, tmp = tempfile.mkstemp(prefix=os.path.basename(path) + '.', suffix='.tmp', dir=SHAPES_DIR)
                os.close(fd)
                try:
                    _nvcc([f'-DLSM_SHAPE={dyn * 1000000 + N * 10000 + L * 100 + O}'], tmp, verbose)
                    os.chmod(tmp, 0o755)
                    os.replace(tmp, path)
                finally:
                    if os.path.exists(tmp):
                        os.unlink(tmp)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return path


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(prog='python -m layered_safe_marl_b200._build', description=__doc__.splitlines()[0])
    ap.add_argument('--shape', action='append', default=[], metavar='DYNAMICS,N,L,O',
                    help='build the library of one specialised shape (repeatable), e.g. airtaxi,6,2,0')
    ap.add_argument('--ppo', action='store_true', help='build the PPO-input library (liblsm_b200_ppo.so)')
    ap.add_argument('--hj', action='store_true', help='build the HJ reachability solver (liblsm_b200_hj.so)')
    ap.add_argument('--force', action='store_true', help='rebuild even when the library is up to date')
    ap.add_argument('--verbose', action='store_true', help='print ptxas resource usage')
    a = ap.parse_args(argv)
    if a.ppo or a.hj:
        if a.ppo:
            print(build_ppo(force=a.force, verbose=a.verbose))
        if a.hj:
            print(build_hj(force=a.force, verbose=a.verbose))
        if not a.shape:
            return
    if not a.shape:
        print(build(force=a.force, verbose=a.verbose))
        return
    for spec in a.shape:
        parts = spec.split(',')
        if len(parts) != 4:
            ap.error(f"--shape wants DYNAMICS,N,L,O, got {spec!r}")
        print(build_shape(parts[0], *parts[1:], force=a.force, verbose=a.verbose))


if __name__ == '__main__':
    main()
