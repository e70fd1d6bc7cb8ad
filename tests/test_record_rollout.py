"""Rollout storage by emit record (DeviceGraphRolloutBuffer(graph_storage='records'), lsm_copy_records,
lsm_emit_from_records): every re-emitted graph row is bit for bit the row the dense buffer stores.

CPU: the ctypes mirror of lsm_record_emit_io; every kernel the library had before the record emission kernel keeps its
SASS instruction for instruction (tests/golden/sass_kernels_pinned.json: sha256 of each kernel's cuobjdump -sass
listing, as the kernels stand since the shared HJ grid lookup of lsm_grid.cuh), and the only kernels added are the
record emission kernel's instantiations.
GPU: equality with the dense buffer across shapes, feature modes, chunked steps and auto-resets; disconnected entities
with flags fixed and changing inside the step; the item edge cases."""
import ctypes
import hashlib
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import _golden as G

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'tools'))

from layered_safe_marl_b200 import _build, _lib      # noqa: E402

gpu = pytest.mark.gpu
DI, AT = 'double_integrator', 'airtaxi'


# ----------------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------------
def test_record_emit_io_mirror_matches_the_c_header(tmp_path):
    cls = _lib.LsmRecordEmitIo
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lsm_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(lsm_record_emit_io));']
    lines += [f'  printf("{f} %zu\\n", offsetof(lsm_record_emit_io, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / 'io.c', tmp_path / 'io.exe'
    src.write_text('\n'.join(lines))
    subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), '-o', str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    assert int(got['size']) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def _cuobjdump():
    exe = shutil.which('cuobjdump')
    if exe is None:
        nvcc = shutil.which(os.environ.get('NVCC', 'nvcc'))
        if nvcc is not None and os.path.exists(os.path.join(os.path.dirname(nvcc), 'cuobjdump')):
            exe = os.path.join(os.path.dirname(nvcc), 'cuobjdump')
    return exe


def test_pinned_kernels_keep_their_sass():
    exe = _cuobjdump()
    assert exe is not None, "cuobjdump (CUDA toolkit) not found next to nvcc"
    import sass_diff
    now = sass_diff.kernels(_build.build(), exe)
    before = json.load(open(os.path.join(REPO, 'tests', 'golden', 'sass_kernels_pinned.json')))
    digest = {k: hashlib.sha256('\n'.join(v).encode()).hexdigest() for k, v in now.items()}
    changed = sorted(k for k in before if digest.get(k) != before[k])
    assert not changed, f"kernels whose SASS changed or vanished: {changed}"
    added = sorted(set(digest) - set(before))
    assert added and all('lsm_record_emit_kernel' in k for k in added), added


# ----------------------------------------------------------------------------------------------------------------------
# GPU: equality with the dense buffer
# ----------------------------------------------------------------------------------------------------------------------
def _args(dyn=DI, N=8, O=0, **kw):
    d = dict(dynamics_type=dyn, num_agents=N, use_safety_filter=True, episode_length=5, world_size=2)
    if O:
        d.update(num_obstacles=O, obstacle_extension=True)
    d.update(kw)
    return G.default_args(**d)


# name -> (args, num_envs, buffer length T, tuning)
CASES = {
    'cfg2_di8': (dict(), 64, 8, None),
    'at10': (dict(dyn=AT, N=10, world_size=4), 32, 7, None),
    'at10_obst4': (dict(dyn=AT, N=10, O=4, world_size=4), 32, 7, None),    # E = 34: two mask words
    'di8_global': (dict(graph_feat_type='global'), 32, 7, None),
    'di32_small_n': (dict(N=32, world_size=4), 3, 6, None),                  # E = 96: three mask words
    'at4_global': (dict(dyn=AT, N=4, graph_feat_type='global'), 32, 7, None),
    'di6_on_demand': (dict(N=6, specialise_shape=True), 32, 7, None),
    'di12_l3_on_demand': (dict(N=12, num_landmarks=3, specialise_shape=True, world_size=3), 16, 7, None),   # E = 48
    'di8_interp_f32': (dict(interp_float32=True), 32, 7, None),
    'di8_chunks3': (dict(), 256, 6, dict(chunks=3)),
}


def _bits(t):
    import torch
    return t.contiguous().view(torch.int32)


def _run_pair(case):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    kw, n, T, tuning = CASES[case]
    args = _args(**kw)
    envs = [B200GraphVecEnv(args, num_envs=n, seed=11, tuning=tuning) for _ in range(2)]
    li = envs[1].launch_info()
    assert li['specialised'] == 1 and li['chunks'] == (tuning or {}).get('chunks', 1), li
    dense = DeviceGraphRolloutBuffer(envs[0], T, zero_copy=True)
    rec = DeviceGraphRolloutBuffer(envs[1], T, zero_copy=True, graph_storage='records')
    assert rec.node_obs is None and rec.adj is None
    assert rec.records.shape == (T + 1, n, envs[1].launch_info()['emit_record_bytes'])
    return envs, dense, rec


def _check_all_rows(envs, dense, rec):
    import torch
    E, F = envs[0].E, envs[0].F
    T, n, N = dense.episode_length, dense.n_rollout_threads, dense.num_agents
    rows = torch.arange(T * n * N, device=envs[0].device)
    no, ad = rec.graph_batch(rows)
    assert torch.equal(_bits(no), _bits(dense.node_obs[:-1].reshape(-1, E, F)))
    assert torch.equal(_bits(ad), _bits(dense.adj[:-1].reshape(-1, E, E)))
    # the last slot through graph_rows, from host indices
    ti, ei, ai = np.meshgrid([T], np.arange(n), np.arange(N), indexing='ij')
    no, ad = rec.graph_rows(ti.ravel(), ei.ravel(), ai.ravel())
    assert torch.equal(_bits(no), _bits(dense.node_obs[T].reshape(-1, E, F)))
    assert torch.equal(_bits(ad), _bits(dense.adj[T].reshape(-1, E, E)))
    assert torch.equal(_bits(rec.obs), _bits(dense.obs)) and torch.equal(_bits(rec.share_obs), _bits(dense.share_obs))
    assert torch.equal(rec.masks, dense.masks) and torch.equal(rec.rewards, dense.rewards)


@gpu
@pytest.mark.parametrize('case', sorted(CASES))
def test_records_buffer_equals_the_dense_buffer(case):
    import torch
    envs, dense, rec = _run_pair(case)
    n, N = envs[0].n, envs[0].N
    rng = np.random.default_rng(3)
    for b in (dense, rec):
        b.warmup()
    resets = 0
    for rnd in range(2):
        for s in range(dense.episode_length):
            a = torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=envs[0].device)
            outs = [e.step(a, 0) for e in envs]
            resets += int(outs[0][5].all(dim=1).sum())
            # the acting forward's view of the current step: dense from the scratch pair
            dense.insert(outs[0]); rec.insert(outs[1])
            rv = rec.runner_view()
            st = rec.step
            for f in ('node_obs', 'adj'):
                got = np.concatenate(getattr(rv, f)[st])
                want = getattr(dense, f)[s + 1]
                assert torch.equal(_bits(got), _bits(want.reshape(got.shape)))
            with pytest.raises(IndexError):
                rv.node_obs[(st + 1) % dense.episode_length]
        _check_all_rows(envs, dense, rec)
        dense.after_update(); rec.after_update()
    torch.cuda.synchronize()
    assert resets > 0, "the rollout should include auto-resets"
    assert rec.graph_nbytes() < dense.graph_nbytes()


# ----------------------------------------------------------------------------------------------------------------------
# GPU: disconnected entities, flags changing inside the step
# ----------------------------------------------------------------------------------------------------------------------
def _all_items(env, records):
    """Re-emit every (env, observer) of one step's records -> (node_obs, adj) shaped like env.node_obs / env.adj."""
    import torch
    n, N = env.n, env.N
    r = torch.arange(n, device=env.device).repeat_interleave(N)
    o = torch.arange(N, device=env.device, dtype=torch.int32).repeat(n)
    no, ad = env.emit_from_records(records, r, o)
    return no.view(env.node_obs.shape), ad.view(env.adj.shape)


@gpu
@pytest.mark.parametrize('dyn', [DI, AT])
def test_disconnected_entities_and_flags_changing_in_the_step(dyn):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    n = 256
    env = B200GraphVecEnv(_args(dyn, 8 if dyn == DI else 10, episode_length=40, world_size=1), num_envs=n, seed=7)
    R = env.launch_info()['emit_record_bytes']
    records = torch.empty((n, R), dtype=torch.uint8, device=env.device)
    rng = np.random.default_rng(5)
    env.reset(0)
    N, L = env.N, env.L
    st = env.get_state()
    # envs 0..63: some agents done and some goals reached (fixed flags: the same graph for every observer)
    done = st['done'].copy(); reached = st['reached_goal'].copy()
    done[:64] = rng.random((64, N)) < 0.3
    reached[:64] = rng.integers(0, L + 1, (64, N))
    # envs 64..191: agents placed on their current goal with its heading and speed, so that they reach it in the step
    vals = st['agent_values'].copy()
    lp, lh, ls = st['landmark_pos'], st['landmark_heading'], st['landmark_speed']
    for e in range(64, 192):
        for a in range(N):
            if rng.random() < 0.5:
                g = reached[e, a] * N + a if reached[e, a] < L else a
                vals[e, a, 0:2] = lp[e, g]
                if dyn == DI:
                    vals[e, a, 2:4] = (ls[e, g] * np.cos(lh[e, g]), ls[e, g] * np.sin(lh[e, g]))
                else:
                    vals[e, a, 2:4] = (lh[e, g], ls[e, g])
    st.update(done=done, reached_goal=reached, agent_values=vals)
    per_observer = 0
    # reset_from_state starts new episodes from the injected positions (flags cleared); observe then emits the injected
    # flags as they are, and the steps move agents onto / off their goals
    for k, call in enumerate(['reset_from_state', 'observe', 'step', 'step', 'step', 'step']):
        if call == 'step':
            env.step(torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=env.device), 0)
        elif call == 'observe':
            env.set_state(st)
            env.observe()
        else:
            env.set_state(st)
            env.reset_from_state(0)
        env.copy_records(records)
        no, ad = _all_items(env, records)
        assert torch.equal(_bits(no), _bits(env.node_obs)), f"{call} #{k}: node_obs"
        assert torch.equal(_bits(ad), _bits(env.adj)), f"{call} #{k}: adj"
        # envs whose observers see different matrices (a flag changed inside the step)
        per_observer += int((env.adj != env.adj[:, :1]).flatten(1).any(dim=1).sum())
        if call == 'observe':
            assert bool((env.adj[:64] == 0).all(dim=-1).any()), "injected disconnected entities should zero whole rows"
    assert per_observer > 0, "the data should contain envs whose observers' matrices differ"


# ----------------------------------------------------------------------------------------------------------------------
# GPU: items
# ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def stepped():
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    n = 48
    env = B200GraphVecEnv(_args(), num_envs=n, seed=2)
    env.reset(0)
    env.step(torch.randint(0, 25, (n, env.N), dtype=torch.int32, device=env.device), 0)
    R = env.launch_info()['emit_record_bytes']
    records = torch.empty((n, R), dtype=torch.uint8, device=env.device)
    env.copy_records(records)
    return env, records


@gpu
def test_random_items_with_duplicates(stepped):
    import torch
    env, records = stepped
    rng = np.random.default_rng(0)
    B = 1000
    r = rng.integers(0, env.n, B); o = rng.integers(0, env.N, B)
    r[10:20] = r[0]; o[10:20] = o[0]
    no, ad = env.emit_from_records(records, torch.as_tensor(r, device=env.device), torch.as_tensor(o, device=env.device, dtype=torch.int32))
    rt, ot = torch.as_tensor(r, device=env.device), torch.as_tensor(o, device=env.device)
    assert torch.equal(_bits(no), _bits(env.node_obs[rt, ot])) and torch.equal(_bits(ad), _bits(env.adj[rt, ot]))
    # the same items from host indices
    no2, ad2 = env.emit_from_records(records, r, o)
    assert torch.equal(_bits(no2), _bits(no)) and torch.equal(_bits(ad2), _bits(ad))


@gpu
def test_zero_and_one_item_and_null_outputs(stepped):
    import torch
    env, records = stepped
    no, ad = env.emit_from_records(records, [], [])
    assert no.shape == (0, env.E, env.F) and ad.shape == (0, env.E, env.E)
    no, ad = env.emit_from_records(records, [5], [3])
    assert torch.equal(_bits(no[0]), _bits(env.node_obs[5, 3])) and torch.equal(_bits(ad[0]), _bits(env.adj[5, 3]))
    # NULL node_obs / adj through the C ABI: the other output is still written, nothing else
    lib, E, F = env.lib, env.E, env.F
    r = torch.tensor([7, 1], dtype=torch.int64, device=env.device); o = torch.tensor([0, 7], dtype=torch.int32, device=env.device)
    for drop in ('node_obs', 'adj'):
        out_no = torch.full((2, E, F), 7.0, device=env.device); out_ad = torch.full((2, E, E), 7.0, device=env.device)
        io = _lib.LsmRecordEmitIo(2, env.n, records.data_ptr(), r.data_ptr(), o.data_ptr(),
                                  None if drop == 'node_obs' else out_no.data_ptr(), None if drop == 'adj' else out_ad.data_ptr())
        _lib.check(lib.lsm_emit_from_records(env._h, ctypes.byref(io), env._stream()), 'lsm_emit_from_records', lib)
        torch.cuda.synchronize()
        if drop == 'node_obs':
            assert bool((out_no == 7.0).all()) and torch.equal(_bits(out_ad), _bits(env.adj[r, o.long()]))
        else:
            assert bool((out_ad == 7.0).all()) and torch.equal(_bits(out_no), _bits(env.node_obs[r, o.long()]))


@gpu
def test_invalid_device_items_are_zero_filled_and_host_items_raise(stepped):
    import torch
    env, records = stepped
    n, N = env.n, env.N
    r = torch.tensor([0, -1, n, 3, 2, 10 ** 12], dtype=torch.int64, device=env.device)
    o = torch.tensor([1, 0, 0, -1, N, 2], dtype=torch.int32, device=env.device)
    no = torch.full((6, env.E, env.F), 7.0, device=env.device); ad = torch.full((6, env.E, env.E), 7.0, device=env.device)
    env.emit_from_records(records, r, o, no, ad)
    torch.cuda.synchronize()
    assert torch.equal(_bits(no[0]), _bits(env.node_obs[0, 1])) and torch.equal(_bits(ad[0]), _bits(env.adj[0, 1]))
    assert bool((no[1:] == 0).all()) and bool((ad[1:] == 0).all())
    for rr, oo in (([n], [0]), ([-1], [0]), ([0], [N]), ([0], [-1])):
        with pytest.raises(IndexError):
            env.emit_from_records(records, rr, oo)
        with pytest.raises(IndexError):
            env.emit_from_records(records, torch.tensor(rr), torch.tensor(oo))


@gpu
def test_records_mode_requirements():
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    env = B200GraphVecEnv(_args(), num_envs=8, seed=0)
    with pytest.raises(ValueError, match='zero_copy'):
        DeviceGraphRolloutBuffer(env, 4, graph_storage='records')
    with pytest.raises(ValueError):
        DeviceGraphRolloutBuffer(env, 4, zero_copy=True, graph_storage='compressed')
    # a shape the product library runs on the generic kernel (DI 5 agents)
    gen = B200GraphVecEnv(_args(N=5), num_envs=8, seed=0)
    assert gen.launch_info()['specialised'] == 0
    with pytest.raises(ValueError, match='specialised'):
        DeviceGraphRolloutBuffer(gen, 4, zero_copy=True, graph_storage='records')
    import torch
    rec = torch.zeros((8, 64), dtype=torch.uint8, device=gen.device)
    with pytest.raises(RuntimeError):
        gen.emit_from_records(rec, [0], [0])
    assert gen.lib.lsm_copy_records(gen._h, ctypes.c_void_p(rec.data_ptr()), None) == 6
    io = _lib.LsmRecordEmitIo(0, 0, None, None, None, None, None)
    assert gen.lib.lsm_emit_from_records(gen._h, ctypes.byref(io), None) == 6


@gpu
def test_graph_rows_host_indices_are_checked():
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    env = B200GraphVecEnv(_args(), num_envs=8, seed=0)
    buf = DeviceGraphRolloutBuffer(env, 4, zero_copy=True, graph_storage='records')
    buf.warmup()
    for t, e, a in (([5], [0], [0]), ([0], [8], [0]), ([0], [0], [8]), ([-1], [0], [0])):
        with pytest.raises(IndexError):
            buf.graph_rows(t, e, a)
    with pytest.raises(IndexError):
        buf.graph_batch([4 * 8 * 8])
    with pytest.raises(IndexError):
        buf.graph_batch(np.array([-1]))
