#!/usr/bin/env python3
"""Branch coverage of the C oracle (oracle/lsm_oracle.c) by the parity tests: which branches no test ever takes.

Builds the oracle and tests/filter_rows_oracle.c with gcov instrumentation in a temporary directory, replays the oracle
side of the tests on the CPU and prints every branch of lsm_oracle.c that was never taken:
- every `_compare_with_oracle` configuration of tests/test_cuda_parity.py (oracle steps only, same seeds and actions);
- the CPU tests of test_oracle_golden.py, test_host_logic.py, test_rollout_and_eval.py and test_safety_filter_op.py;
- unless --without-bounds: the CPU tests of test_filter_bounds.py and the oracle side of its GPU tests.

    python tools/oracle_branch_coverage.py [--without-bounds] [--out report.txt]
"""
from __future__ import annotations

import argparse
import gzip
import inspect
import itertools
import json
import os
import shutil
import subprocess
import sys
import tempfile
import types

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'oracle'))
sys.path.insert(0, os.path.join(REPO, 'tests'))

CFLAGS = ['-O0', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math', '--coverage']
CPU_TEST_FILES = ['test_oracle_golden.py', 'test_host_logic.py', 'test_rollout_and_eval.py', 'test_safety_filter_op.py']


def build(tmp):
    """-> (oracle library, filter-rows library), both instrumented; their .gcda files land in `tmp`."""
    gcov_a = subprocess.check_output(['gcc', '-print-file-name=libgcov.a'], text=True).strip()
    libs = []
    for src, name in ((os.path.join(REPO, 'oracle', 'lsm_oracle.c'), 'liblsm_oracle'),
                      (os.path.join(REPO, 'tests', 'filter_rows_oracle.c'), 'libfilter_rows_oracle')):
        obj = os.path.join(tmp, name + '.o')
        subprocess.check_call(['gcc'] + CFLAGS + ['-c', '-o', obj, src])
        so = os.path.join(tmp, name + '.so')
        subprocess.check_call(['gcc', '-shared', '-o', so, obj, gcov_a, '-lm', '-lpthread'])
        libs.append(so)
    return libs


def install(oracle_so, rows_so):
    """Point the tests' oracle front-ends at the instrumented libraries: oracle_env loads `oracle_so`, and the compile
    step of test_safety_filter_op's row oracle is replaced by a copy of `rows_so`."""
    import oracle_env as O
    import test_safety_filter_op as SF
    O.LIB_PATH = oracle_so
    O.build = lambda force=False: oracle_so
    O._lib = None

    def check_call(cmd, *a, **k):
        if any(str(c).endswith('filter_rows_oracle.c') for c in cmd):
            shutil.copy(rows_so, cmd[cmd.index('-o') + 1])
            return 0
        return subprocess.check_call(cmd, *a, **k)
    SF.subprocess = types.SimpleNamespace(check_call=check_call, check_output=subprocess.check_output)
    SF._ROWS_LIB = None


def oracle_only_compare(args, flags, n, T, episode, seed, auto_reset, grids=None, prepare=None, tuning=None,
                        after_reset=None, actions=None, on_step=None):
    """The oracle half of test_cuda_parity._compare_with_oracle: same resets, hooks and actions, no CUDA env."""
    import _golden as G
    import oracle_env as O
    from layered_safe_marl_b200 import config as cfg
    params = cfg.scenario_params_from_args(args, binary_cfg=flags)
    vg, tg = G.value_grid_for(params) if grids is None else grids
    ora = O.OracleEnv(params.asdict(), n, value_grid=vg, ttr_grid=tg, seed=seed, nthreads=8)
    # the relative-state form the CUDA side would take (the specialised airtaxi shapes evaluate the rotation form), as
    # near as the shape tells without a handle; it only decides which arm of at_relative_state runs
    spec = params.dynamics != 0 and params.num_agents in (4, 8, 10, 16) and params.num_landmarks == 2
    prev = O.set_relative_state_form(1 if spec else 0)
    try:
        ora.reset(episode=episode, sample=True)
        if after_reset is not None:
            after_reset(ora, None)
        rng = np.random.default_rng(seed + 7)
        for t in range(T):
            a = (rng.integers(0, 25, (n, params.num_agents)) if actions is None else actions(rng, t)).astype(np.int32)
            pre = ora.get_state() if on_step is not None else None
            ora.step(a, episode=episode, auto_reset=auto_reset)
            if on_step is not None:
                on_step(t, a, pre, ora.get_state())
    finally:
        O.set_relative_state_form(prev)
    return ora, None


def _param_sets(fn):
    """Every parameter combination of a test function's parametrize marks."""
    marks = [m for m in getattr(fn, 'pytestmark', []) if m.name == 'parametrize']
    axes = []
    for m in marks:
        names = [s.strip() for s in m.args[0].split(',')] if isinstance(m.args[0], str) else list(m.args[0])
        vals = [v if len(names) > 1 else (v,) for v in m.args[1]]
        axes.append([dict(zip(names, v)) for v in vals])
    for combo in itertools.product(*axes):
        kw = {}
        for d in combo:
            kw.update(d)
        yield kw


def replay_parity():
    """Every test of test_cuda_parity.py that runs _compare_with_oracle, with the oracle-only stand-in."""
    import test_cuda_parity as P
    P._compare_with_oracle = oracle_only_compare
    for name, fn in sorted(vars(P).items()):
        if not (name.startswith('test_') and callable(fn)) or '_compare_with_oracle(' not in inspect.getsource(fn):
            continue
        for kw in _param_sets(fn):
            try:
                fn(**kw)
            except Exception:       # what follows the oracle run needs the CUDA env
                pass


def replay_bounds():
    """The oracle side of test_filter_bounds.py's GPU tests (its CPU tests run under pytest)."""
    import test_filter_bounds as T
    for dyn, gname in T.LOOKUP_CASES:
        for f32 in (False, True):
            T.SF.oracle_lookup(T.params_of(dyn, f32).asdict(), T.grid(gname),
                               rel=T.bound_node_points(dyn, np.random.default_rng(3 + dyn)))
    for shape, tuning in T.ENV_CASES:
        if tuning in (None, 0):
            T.env_case(shape, tuning, n=128, T=4, hook_seed=11, compare=oracle_only_compare)
    _, st = T.max_speed_rollout(0, compare=oracle_only_compare)
    print(f"max-speed rollout: {st.at_vmax / st.live:.1%} of live agent-steps at V_MAX, {st.rows_vmax} filter rows "
          f"with a speed >= V_MAX: {st.labels}")
    for shape in ('di8', 'di8_f32'):
        _, st = T.di_alias_rollout(shape, compare=oracle_only_compare)
        print(f"{shape} on the velocity-free grid: {st.labels}")


def run_pytest(files):
    import pytest
    rc = pytest.main(['-q', '-m', 'not gpu', '-p', 'no:cacheprovider'] + [os.path.join(REPO, 'tests', f) for f in files])
    if rc != 0:
        raise SystemExit(f"pytest failed ({rc}) on {files}")


def untaken_branches(tmp):
    """Merge the branch counts of both objects for lsm_oracle.c -> (total, [(line, taken, total), ...] untaken)."""
    subprocess.check_call(['gcov', '--json-format', '--branch-probabilities', '--object-directory', tmp,
                           os.path.join(tmp, 'liblsm_oracle.o'), os.path.join(tmp, 'libfilter_rows_oracle.o')],
                          cwd=tmp, stdout=subprocess.DEVNULL)
    counts = {}
    for f in os.listdir(tmp):
        if not f.endswith('.gcov.json.gz'):
            continue
        with gzip.open(os.path.join(tmp, f), 'rt') as fh:
            data = json.load(fh)
        for fi in data['files']:
            if not fi['file'].endswith('lsm_oracle.c'):
                continue
            for ln in fi['lines']:
                for k, br in enumerate(ln.get('branches', [])):
                    key = (ln['line_number'], k)
                    counts[key] = counts.get(key, 0) + br['count']
    by_line = {}
    for (line, k), c in counts.items():
        by_line.setdefault(line, []).append(c)
    untaken = [(line, sum(c > 0 for c in cs), len(cs)) for line, cs in sorted(by_line.items()) if any(c == 0 for c in cs)]
    return len(counts), sum(c > 0 for c in counts.values()), untaken


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--without-bounds', action='store_true', help="leave out test_filter_bounds.py")
    ap.add_argument('--out', help="also write the report to this file")
    ap.add_argument('--replay', metavar='DIR', help=argparse.SUPPRESS)      # child: replay against the libraries in DIR
    a = ap.parse_args()
    if a.replay:
        # the counters reach the .gcda files when this process exits
        install(*(os.path.join(a.replay, n + '.so') for n in ('liblsm_oracle', 'libfilter_rows_oracle')))
        replay_parity()
        run_pytest(CPU_TEST_FILES + ([] if a.without_bounds else ['test_filter_bounds.py']))
        if not a.without_bounds:
            replay_bounds()
        return
    tmp = tempfile.mkdtemp(prefix='lsm_oracle_cov_')
    try:
        build(tmp)
        subprocess.check_call([sys.executable, os.path.abspath(__file__), '--replay', tmp]
                              + (['--without-bounds'] if a.without_bounds else []))
        total, taken, untaken = untaken_branches(tmp)
        src = open(os.path.join(REPO, 'oracle', 'lsm_oracle.c')).read().splitlines()
        lines = [f"oracle/lsm_oracle.c: {taken} of {total} branches taken ({100.0 * taken / total:.1f} %)",
                 f"replayed: test_cuda_parity.py oracle side, CPU tests of {', '.join(CPU_TEST_FILES)}"
                 + ("" if a.without_bounds else ", test_filter_bounds.py (CPU tests and the oracle side of its GPU tests)"),
                 "branches never taken (line: taken / branches | source):"]
        lines += [f"{line:5d}: {t}/{n} | {src[line - 1].strip()[:110]}" for line, t, n in untaken]
        report = '\n'.join(lines)
        print(report)
        if a.out:
            with open(a.out, 'w') as f:
                f.write(report + '\n')
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
    main()
