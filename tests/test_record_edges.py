"""Edge lists from stored emit records (lsm_edges_from_records, B200GraphVecEnv.edges_from_records,
DeviceGraphRolloutBuffer.graph_batch / graph_rows with edges=True): every list equals the reference's process_adj of the
dense rows, edge_index exactly and edge_attr bit for bit.

CPU: the ctypes mirror of lsm_record_edges_io; the null-argument check.
GPU: equality with process_adj across the shapes and modes of test_record_rollout's CASES, on both storages; equality with
the step's own fused edge list; disconnected entities with flags fixed and changing inside the step; the item edge cases
(zero / one item, duplicates, invalid items, short capacities and stale offsets, more than 2^21 items, more than 2^31
edges); the largest shape through a per-shape library; the error codes."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import _golden as G
from test_record_rollout import AT, CASES, DI, _args, _bits, _run_pair
from test_rollout_and_eval import _process_adj

from layered_safe_marl_b200 import _lib

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------------
def test_record_edges_io_mirror_matches_the_c_header(tmp_path):
    cls = _lib.LsmRecordEdgesIo
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lsm_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(lsm_record_edges_io));']
    lines += [f'  printf("{f} %zu\\n", offsetof(lsm_record_edges_io, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / 'io.c', tmp_path / 'io.exe'
    src.write_text('\n'.join(lines))
    subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), '-o', str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    assert int(got['size']) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def test_null_arguments_are_refused():
    lib = _lib.load()
    io = _lib.LsmRecordEdgesIo(0, 0, None, None, None, None, None, None, None, 0)
    assert lib.lsm_edges_from_records(None, ctypes.byref(io), None) == 1
    assert lib.lsm_edges_from_records(None, None, None) == 1


# ----------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ----------------------------------------------------------------------------------------------------------------------
def _assert_edges_equal(got, want, what):
    import torch
    gi, ga = got
    wi, wa = want
    assert gi.dtype == torch.int64 and ga.dtype == torch.float32 and gi.shape[0] == 2 and ga.shape == (gi.shape[1], 1), what
    assert gi.shape == wi.shape, f"{what}: {gi.shape[1]} edges, process_adj has {wi.shape[1]}"
    assert torch.equal(gi, wi), f"{what}: edge_index"
    assert torch.equal(_bits(ga), _bits(wa)), f"{what}: edge_attr"


def _all_items(env, slots, n):
    """Items (slot s, env, agent) in env-major order of `slots` stored steps: record s * n + env, observer agent."""
    import torch
    N = env.N
    r = (torch.arange(slots, device=env.device).repeat_interleave(n * N) * n
         + torch.arange(n, device=env.device).repeat_interleave(N).repeat(slots))
    o = torch.arange(N, device=env.device, dtype=torch.int32).repeat(slots * n)
    return r, o


# ----------------------------------------------------------------------------------------------------------------------
# GPU: equality with process_adj, both storages
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('case', sorted(CASES))
def test_graph_batch_edges_equal_process_adj(case):
    import torch
    envs, dense, rec = _run_pair(case)
    n, N = envs[0].n, envs[0].N
    T = dense.episode_length
    rng = np.random.default_rng(3)
    for b in (dense, rec):
        b.warmup()
    resets = 0
    for rnd in range(2):
        for s in range(T):
            a = torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device=envs[0].device)
            outs = [e.step(a, 0) for e in envs]
            resets += int(outs[0][5].all(dim=1).sum())
            dense.insert(outs[0]); rec.insert(outs[1])
        # every row of the stored episode, in a shuffled order
        rows = torch.as_tensor(rng.permutation(T * n * N), device=envs[0].device)
        no_ref, ad_ref = rec.graph_batch(rows)
        want = _process_adj(ad_ref)
        no, ei, ea = rec.graph_batch(rows, edges=True)
        assert torch.equal(_bits(no), _bits(no_ref)), case
        _assert_edges_equal((ei, ea), want, f"{case} records")
        dno, dei, dea = dense.graph_batch(rows, edges=True)
        assert torch.equal(_bits(dno), _bits(no)), case
        _assert_edges_equal((dei, dea), (ei, ea), f"{case} dense")
        # the last slot through graph_rows, from host indices
        ti, eidx, ai = np.meshgrid([T], np.arange(n), np.arange(N), indexing='ij')
        no, ei, ea = rec.graph_rows(ti.ravel(), eidx.ravel(), ai.ravel(), edges=True)
        assert torch.equal(_bits(no), _bits(dense.node_obs[T].reshape(no.shape)))
        _assert_edges_equal((ei, ea), _process_adj(dense.adj[T].reshape(-1, envs[0].E, envs[0].E)), f"{case} graph_rows")
        dense.after_update(); rec.after_update()
    torch.cuda.synchronize()
    assert resets > 0, "the rollout should include auto-resets"


@gpu
@pytest.mark.parametrize('kw,n,tuning', [(dict(), 64, None), (dict(dyn=AT, N=10, O=4, world_size=4), 32, None),
                                         (dict(), 256, dict(chunks=3)), (dict(N=12, num_landmarks=3, specialise_shape=True, world_size=3), 16, None)],
                         ids=['cfg2_di8', 'at10_obst4', 'di8_chunks3', 'di12_l3_on_demand'])
def test_edges_equal_the_fused_edge_list_of_the_step(kw, n, tuning):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    env = B200GraphVecEnv(_args(**kw), num_envs=n, seed=5, tuning=tuning)
    env.enable_edge_output()
    R = env.record_bytes()
    steps = 9
    records = torch.empty((steps, n, R), dtype=torch.uint8, device=env.device)
    env.reset(0)
    rng = np.random.default_rng(4)
    for s in range(steps):
        env.step(torch.as_tensor(rng.integers(0, 25, (n, env.N)).astype(np.int32), device=env.device), 0)
        env.copy_records(records[s])
        r, o = _all_items(env, 1, n)
        got = env.edges_from_records(records, r + s * n, o)
        want = tuple(x.clone() for x in env.edges())
        _assert_edges_equal(got, want, f"step {s}")


# ----------------------------------------------------------------------------------------------------------------------
# GPU: disconnected entities, flags changing inside the step
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('dyn', [DI, AT])
def test_masked_entities_and_flags_changing_in_the_step(dyn):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    n = 256
    env = B200GraphVecEnv(_args(dyn, 8 if dyn == DI else 10, episode_length=40, world_size=1), num_envs=n, seed=7)
    R = env.record_bytes()
    records = torch.empty((n, R), dtype=torch.uint8, device=env.device)
    rng = np.random.default_rng(5)
    env.reset(0)
    N, L, E = env.N, env.L, env.E
    st = env.get_state()
    # envs 0..63: some agents done and some goals reached (fixed flags); env 0: every agent done and every goal reached
    done = st['done'].copy(); reached = st['reached_goal'].copy()
    done[:64] = rng.random((64, N)) < 0.3
    reached[:64] = rng.integers(0, L + 1, (64, N))
    done[0] = True; reached[0] = L
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
    r, o = _all_items(env, 1, n)
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
        ei, ea = env.edges_from_records(records, r, o)
        _assert_edges_equal((ei, ea), _process_adj(env.adj.reshape(-1, E, E)), f"{call} #{k}")
        per_observer += int((env.adj != env.adj[:, :1]).flatten(1).any(dim=1).sum())
        if call == 'observe':
            assert int((ei[0] < N * E).sum()) == 0, "env 0 (every entity disconnected) should have no edges"
            assert int(ei.shape[1]) > 0
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
    records = torch.empty((n, env.record_bytes()), dtype=torch.uint8, device=env.device)
    env.copy_records(records)
    return env, records


def _passes(env, records, r, o, counts, offsets, edge_index=None, edge_attr=None, capacity=0):
    """One lsm_edges_from_records call through the C ABI (counting pass when edge_index is None); -> error code."""
    io = _lib.LsmRecordEdgesIo(r.numel(), records.numel() // env.record_bytes(), records.data_ptr(), r.data_ptr(), o.data_ptr(),
                               counts.data_ptr() if counts is not None else None, offsets.data_ptr() if offsets is not None else None,
                               edge_index, edge_attr, capacity)
    return env.lib.lsm_edges_from_records(env._h, ctypes.byref(io), env._stream())


@gpu
def test_zero_one_and_random_items(stepped):
    import torch
    env, records = stepped
    E = env.E
    ei, ea = env.edges_from_records(records, [], [])
    assert ei.shape == (2, 0) and ea.shape == (0, 1)
    ei, ea = env.edges_from_records(records, [5], [3])
    _assert_edges_equal((ei, ea), _process_adj(env.adj[5, 3][None]), "one item")
    rng = np.random.default_rng(0)
    B = 1000
    r = rng.integers(0, env.n, B); o = rng.integers(0, env.N, B)
    r[10:20] = r[0]; o[10:20] = o[0]
    rt, ot = torch.as_tensor(r, device=env.device), torch.as_tensor(o, device=env.device)
    want = _process_adj(env.adj[rt, ot])
    _assert_edges_equal(env.edges_from_records(records, rt, ot.to(torch.int32)), want, "device items")
    _assert_edges_equal(env.edges_from_records(records, r, o), want, "host items")
    assert int(want[0].max()) < B * E


@gpu
def test_invalid_device_items_have_no_edges_and_host_items_raise(stepped):
    import torch
    env, records = stepped
    n, N = env.n, env.N
    r = torch.tensor([0, -1, n, 3, 2, 10 ** 12, 7], dtype=torch.int64, device=env.device)
    o = torch.tensor([1, 0, 0, -1, N, 2, 4], dtype=torch.int32, device=env.device)
    dense = torch.zeros((7, env.E, env.E), device=env.device)
    dense[0], dense[6] = env.adj[0, 1], env.adj[7, 4]
    _assert_edges_equal(env.edges_from_records(records, r, o), _process_adj(dense), "invalid items")
    for rr, oo in (([n], [0]), ([-1], [0]), ([0], [N]), ([0], [-1])):
        with pytest.raises(IndexError):
            env.edges_from_records(records, rr, oo)
        with pytest.raises(IndexError):
            env.edges_from_records(records, torch.tensor(rr), torch.tensor(oo))


@gpu
def test_fill_never_writes_past_capacity_or_from_stale_offsets(stepped):
    import torch
    env, records = stepped
    B = 300
    gen = torch.Generator(device=env.device); gen.manual_seed(1)
    r = torch.randint(0, env.n, (B,), generator=gen, device=env.device)
    o = torch.randint(0, env.N, (B,), generator=gen, device=env.device, dtype=torch.int32)
    want_i, want_a = env.edges_from_records(records, r, o)
    nnz = want_i.shape[1]
    counts = torch.empty(B, dtype=torch.int32, device=env.device)
    offsets = torch.empty(B + 1, dtype=torch.int64, device=env.device)
    assert _passes(env, records, r, o, counts, offsets) == 0
    assert int(offsets[B]) == nnz and torch.equal(offsets[1:] - offsets[:-1], counts.long())
    tail, S = 1000, -7
    for cap in (nnz // 2, 1):
        ei = torch.full((2 * cap + tail,), S, dtype=torch.int64, device=env.device)
        ea = torch.full((cap + tail,), float(S), device=env.device)
        assert _passes(env, records, r, o, counts, offsets, ei.data_ptr(), ea.data_ptr(), cap) == 0
        torch.cuda.synchronize()
        assert torch.equal(ei[:cap], want_i[0, :cap]) and torch.equal(ei[cap:2 * cap], want_i[1, :cap])
        assert torch.equal(_bits(ea[:cap]), _bits(want_a[:cap, 0]))
        assert bool((ei[2 * cap:] == S).all()) and bool((ea[cap:] == S).all()), f"capacity {cap}: written past it"
    # offsets of other items, shifted out of [0, capacity) either way: nothing is written
    for shift in (-(nnz + 10 ** 6), nnz, 1 << 40):
        ei = torch.full((2 * nnz + tail,), S, dtype=torch.int64, device=env.device)
        ea = torch.full((nnz + tail,), float(S), device=env.device)
        assert _passes(env, records, r, o, counts, offsets + shift, ei.data_ptr(), ea.data_ptr(), nnz) == 0
        torch.cuda.synchronize()
        assert bool((ei == S).all()) and bool((ea == S).all()), f"shift {shift}"


@gpu
def test_more_than_2_pow_21_items(stepped):
    import torch
    env, records = stepped
    B = (1 << 21) + 77
    gen = torch.Generator(device=env.device); gen.manual_seed(2)
    r = torch.randint(0, env.n, (B,), generator=gen, device=env.device)
    o = torch.randint(0, env.N, (B,), generator=gen, device=env.device, dtype=torch.int32)
    got = env.edges_from_records(records, r, o)
    _, ad = env.emit_from_records(records, r, o)
    _assert_edges_equal(got, _process_adj(ad), f"{B} items")


@gpu
def test_counting_pass_beyond_2_pow_31_edges():
    """offsets are int64 throughout: ~236 k items that all repeat one complete DI 32 graph (E = 96, 9 120 edges)."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    env = B200GraphVecEnv(_args(N=32, world_size=4), num_envs=2, seed=3)
    env.reset(0)
    N, E = env.N, env.E
    st = env.get_state()
    # every entity on a 10 x 10 grid of 5 mm spacing: all pairs inside the radius, none at distance zero
    g = np.stack(np.meshgrid(np.arange(10), np.arange(10), indexing='ij'), -1).reshape(-1, 2)[:E] * 0.005
    vals = st['agent_values'].copy(); vals[:, :, 0:2] = g[:N]
    lp = st['landmark_pos'].copy(); lp[:] = g[N:E]
    st.update(agent_values=vals, landmark_pos=lp, done=np.zeros_like(st['done']), reached_goal=np.zeros_like(st['reached_goal']))
    env.set_state(st)
    env.observe()
    records = torch.empty((2, env.record_bytes()), dtype=torch.uint8, device=env.device)
    env.copy_records(records)
    c = int((env.adj[1, 3] != 0).sum())
    assert c == E * (E - 1), c
    B = (1 << 31) // c + 1000
    r = torch.ones((B,), dtype=torch.int64, device=env.device)
    o = torch.full((B,), 3, dtype=torch.int32, device=env.device)
    counts = torch.empty(B, dtype=torch.int32, device=env.device)
    offsets = torch.empty(B + 1, dtype=torch.int64, device=env.device)
    assert _passes(env, records, r, o, counts, offsets) == 0
    torch.cuda.synchronize()
    assert bool((counts == c).all())
    assert int(offsets[B]) == B * c and B * c > (1 << 31)
    assert torch.equal(offsets, torch.arange(B + 1, device=env.device, dtype=torch.int64) * c)


@gpu
def test_largest_shape_through_a_shape_library():
    """airtaxi 32 x 4 + 32 obstacles: E = 192, six mask words, on a per-shape library."""
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(dynamics_type=AT, num_agents=32, num_landmarks=4, num_obstacles=32, obstacle_extension=True,
                          use_safety_filter=True, world_size=2, episode_length=12, specialise_shape=True)
    n = 6
    env = B200GraphVecEnv(args, num_envs=n, seed=3)
    assert env.E == 192 and env.launch_info()['specialised'] == 1
    records = torch.empty((n, env.record_bytes()), dtype=torch.uint8, device=env.device)
    env.reset(6249)
    rng = np.random.default_rng(2)
    r, o = _all_items(env, 1, n)
    for t in range(3):
        env.step(torch.as_tensor(rng.integers(0, 25, (n, env.N)).astype(np.int32), device=env.device), 6249)
        env.copy_records(records)
        want = _process_adj(env.adj.reshape(-1, env.E, env.E))
        _assert_edges_equal(env.edges_from_records(records, r, o), want, f"E = 192 step {t}")
        assert want[0].shape[1] > 0


@gpu
def test_error_codes_and_zero_items(stepped):
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv
    env, records = stepped
    dev = env.device
    r = torch.tensor([0, 1], dtype=torch.int64, device=dev); o = torch.tensor([0, 1], dtype=torch.int32, device=dev)
    counts = torch.full((2,), -5, dtype=torch.int32, device=dev)
    offsets = torch.full((3,), -5, dtype=torch.int64, device=dev)
    # zero items: the counting pass writes offsets[0] = 0 and nothing else; the fill pass writes nothing
    io = _lib.LsmRecordEdgesIo(0, env.n, records.data_ptr(), None, None, counts.data_ptr(), offsets.data_ptr(), None, None, 0)
    assert env.lib.lsm_edges_from_records(env._h, ctypes.byref(io), env._stream()) == 0
    torch.cuda.synchronize()
    assert offsets.tolist() == [0, -5, -5] and counts.tolist() == [-5, -5]
    ei = torch.full((4,), -5, dtype=torch.int64, device=dev); ea = torch.full((2,), -5.0, device=dev)
    io = _lib.LsmRecordEdgesIo(0, env.n, records.data_ptr(), None, None, None, offsets.data_ptr(), ei.data_ptr(), ea.data_ptr(), 2)
    assert env.lib.lsm_edges_from_records(env._h, ctypes.byref(io), env._stream()) == 0
    torch.cuda.synchronize()
    assert offsets.tolist() == [0, -5, -5] and bool((ei == -5).all()) and bool((ea == -5).all())
    # negative sizes, missing arrays, misaligned records
    bad = [(-1, env.n, records.data_ptr(), counts.data_ptr(), offsets.data_ptr(), None, None, 0),
           (2, -1, records.data_ptr(), counts.data_ptr(), offsets.data_ptr(), None, None, 0),
           (2, env.n, records.data_ptr(), None, offsets.data_ptr(), None, None, 0),
           (2, env.n, records.data_ptr(), counts.data_ptr(), None, None, None, 0),
           (2, env.n, None, counts.data_ptr(), offsets.data_ptr(), None, None, 0),
           (2, env.n, records.data_ptr() + 4, counts.data_ptr(), offsets.data_ptr(), None, None, 0),
           (2, env.n, records.data_ptr(), counts.data_ptr(), offsets.data_ptr(), offsets.data_ptr(), None, 4),
           (2, env.n, records.data_ptr(), counts.data_ptr(), offsets.data_ptr(), offsets.data_ptr(), counts.data_ptr(), -1)]
    for B, nr, rp, cp, op, eip, eap, cap in bad:
        io = _lib.LsmRecordEdgesIo(B, nr, rp, r.data_ptr(), o.data_ptr(), cp, op, eip, eap, cap)
        assert env.lib.lsm_edges_from_records(env._h, ctypes.byref(io), env._stream()) == 2, (B, nr, rp, cp, op, eip, eap, cap)
    io = _lib.LsmRecordEdgesIo(2, env.n, records.data_ptr(), None, o.data_ptr(), counts.data_ptr(), offsets.data_ptr(), None, None, 0)
    assert env.lib.lsm_edges_from_records(env._h, ctypes.byref(io), env._stream()) == 2
    # a generic-kernel handle (DI 5 agents in the product library)
    gen = B200GraphVecEnv(_args(N=5), num_envs=8, seed=0)
    assert gen.launch_info()['specialised'] == 0
    io = _lib.LsmRecordEdgesIo(0, 0, None, None, None, None, None, None, None, 0)
    assert gen.lib.lsm_edges_from_records(gen._h, ctypes.byref(io), None) == 6
    with pytest.raises(RuntimeError):
        gen.edges_from_records(torch.zeros((8, 64), dtype=torch.uint8, device=dev), [0], [0])


@gpu
def test_two_streams_share_one_handle(stepped):
    import torch
    env, records = stepped
    gen = torch.Generator(device=env.device); gen.manual_seed(9)
    items = [(torch.randint(0, env.n, (4000,), generator=gen, device=env.device),
              torch.randint(0, env.N, (4000,), generator=gen, device=env.device, dtype=torch.int32)) for _ in range(2)]
    want = [env.edges_from_records(records, r, o) for r, o in items]
    streams = [torch.cuda.Stream(device=env.device) for _ in range(2)]
    torch.cuda.synchronize()
    got = [None, None]
    for k in (0, 1):
        with torch.cuda.stream(streams[k]):
            got[k] = env.edges_from_records(records, *items[k])
    torch.cuda.synchronize()
    for k in (0, 1):
        _assert_edges_equal(got[k], want[k], f"stream {k}")


@gpu
def test_edges_keyword_rules():
    import torch
    from layered_safe_marl_b200 import B200GraphVecEnv, DeviceGraphRolloutBuffer
    env = B200GraphVecEnv(_args(), num_envs=8, seed=0)
    buf = DeviceGraphRolloutBuffer(env, 4, zero_copy=True, graph_storage='records')
    buf.warmup()
    adj = torch.empty((1, env.E, env.E), device=env.device)
    with pytest.raises(ValueError):
        buf.graph_batch([0], adj=adj, edges=True)
    with pytest.raises(IndexError):
        buf.graph_batch([4 * 8 * 8], edges=True)
    with pytest.raises(IndexError):
        buf.graph_rows([5], [0], [0], edges=True)
    no, ei, ea = buf.graph_batch([], edges=True)
    assert no.shape == (0, env.E, env.F) and ei.shape == (2, 0) and ea.shape == (0, 1)
