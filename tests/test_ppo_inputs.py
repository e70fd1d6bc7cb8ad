"""PPO inputs on the device: lsm_compute_returns (liblsm_b200_ppo.so) and the minibatch generators of
DeviceGraphRolloutBuffer.

CPU: the ctypes mirror of lsm_returns_io; the library builds for sm_100a and exports its symbols; both generators on a
CPU dense buffer equal a numpy restatement of the reference generators' index arithmetic; compute_advantages equals the
numpy nanmean / nanstd expression.
GPU: the kernel equals the torch loop bit for bit in every mode, writes only the slots the loop writes, reproduces the
reference fixture, and its advantages and float64 moments; no host sync; records and dense buffers serve identical
minibatches; 64-bit indexing."""
import ctypes
import os
import re
import shutil
import subprocess
import types

import numpy as np
import pytest
import torch

import _golden as G

from layered_safe_marl_b200 import _build, _lib
from layered_safe_marl_b200.rollout import DeviceGraphRolloutBuffer, process_adj, returns_kernel, returns_loop
from layered_safe_marl_b200.spaces import Discrete

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLLOUT_GOLDEN = os.path.join(REPO, 'tests', 'golden', 'aux', 'rollout_buffer.npz')
gpu = pytest.mark.gpu
MODES = [(gae, ptl) for gae in (True, False) for ptl in (False, True)]


def _fake_env(n, N, L=1, D=3, F=2, device='cpu'):
    e = types.SimpleNamespace()
    e.num_envs, e.N, e.E, e.D, e.F, e.device = n, N, N * (1 + L), D, F, torch.device(device)
    e.action_space = [Discrete(25) for _ in range(N)]
    e.agent_id = torch.arange(N, dtype=torch.int32).view(1, N, 1).expand(n, N, 1).contiguous()
    return e


def _bits(t):
    return t.contiguous().view(torch.int32)


# ----------------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------------
def test_returns_io_mirror_matches_the_c_header(tmp_path):
    cls = _lib.LsmReturnsIo
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lsm_b200_ppo.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(lsm_returns_io));']
    lines += [f'  printf("{f} %zu\\n", offsetof(lsm_returns_io, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / 'io.c', tmp_path / 'io.exe'
    src.write_text('\n'.join(lines))
    subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), '-o', str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    assert int(got['size']) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def test_ppo_library_builds_for_sm100a_and_exports_its_symbols():
    path = _build.build_ppo()
    lib = ctypes.CDLL(path)
    declared = set(re.findall(r'\b(lsm_[a-z_]+)\s*\(', open(os.path.join(REPO, 'include', 'lsm_b200_ppo.h')).read()))
    assert declared == set(_lib.PPO_EXPORTED_SYMBOLS), declared ^ set(_lib.PPO_EXPORTED_SYMBOLS)
    for sym in declared:
        getattr(lib, sym)
    ppo = _lib.load_ppo()
    assert ppo.lsm_ppo_abi_version() == 1
    assert ppo.lsm_returns_scratch_bytes(32768) >= 24 * (32768 // 128)
    # validation runs on the host: an error code and this library's message, no device needed
    io = _lib.LsmReturnsIo(-1, 4)
    with pytest.raises(RuntimeError, match='T and columns'):
        _lib.check(ppo.lsm_compute_returns(ctypes.byref(io), None), 'lsm_compute_returns', ppo)
    nvcc = shutil.which(os.environ.get('NVCC', 'nvcc'))
    exe = os.path.join(os.path.dirname(nvcc), 'cuobjdump') if nvcc else shutil.which('cuobjdump')
    assert exe and os.path.exists(exe), "cuobjdump (CUDA toolkit) not found next to nvcc"
    listing = subprocess.check_output([exe, '-lelf', path], text=True)
    assert 'sm_100a' in listing, listing
    names = subprocess.check_output([exe, '-sass', path], text=True)
    assert 'lsm_returns_kernel' in names and 'lsm_returns_moments_kernel' in names


def _filled_buffer(n=3, N=2, T=7, device='cpu', seed=0, **kw):
    """A dense buffer with every learner field set to distinct seeded values (adj with zeros, so edge lists are sparse)."""
    g = torch.Generator().manual_seed(seed)
    rb = DeviceGraphRolloutBuffer(_fake_env(n, N, device=device), T, recurrent_N=2, hidden_size=3, **kw)
    for name in ('share_obs', 'obs', 'node_obs', 'rnn_states', 'rnn_states_critic', 'value_preds', 'returns', 'actions',
                 'action_log_probs', 'rewards', 'available_actions'):
        x = getattr(rb, name)
        x.copy_(torch.randn(x.shape, generator=g))
    a = torch.rand(rb.adj.shape, generator=g)
    rb.adj.copy_(torch.where(a < 0.5, torch.zeros_like(a), a))
    for name in ('masks', 'active_masks', 'bad_masks'):
        x = getattr(rb, name)
        x.copy_((torch.rand(x.shape, generator=g) < 0.7).float())
    rb.agent_id.copy_(torch.randint(0, 99, rb.agent_id.shape, generator=g, dtype=torch.int32))
    return rb


_REF_FIELDS = {'share_obs': 'share_obs', 'obs': 'obs', 'node_obs': 'node_obs', 'adj': 'adj', 'agent_id': 'agent_id',
               'share_agent_id': 'share_agent_id', 'rnn_states': 'rnn_states', 'rnn_states_critic': 'rnn_states_critic',
               'actions': 'actions', 'value_preds': 'value_preds', 'returns': 'returns', 'masks': 'masks',
               'active_masks': 'active_masks', 'old_action_log_probs': 'action_log_probs',
               'available_actions': 'available_actions'}


def _np_fields(rb, adv):
    """Every field as the reference's generators slice it: the first T steps (numpy)."""
    T = rb.episode_length
    out = {k: getattr(rb, name).numpy()[:T] for k, name in _REF_FIELDS.items()}
    out['adv_targ'] = adv.numpy()
    return out


def _ref_feed_forward(rb, adv, num_mini_batch, mini_batch_size, perm):
    """graph_buffer.py feed_forward_generator's indexing: x[:-1].reshape(-1, *x.shape[3:])[indices]."""
    T, n, N = rb.episode_length, rb.n_rollout_threads, rb.num_agents
    mbs = T * n * N // num_mini_batch if mini_batch_size is None else mini_batch_size
    f = {k: v.reshape(-1, *v.shape[3:]) for k, v in _np_fields(rb, adv).items()}
    for i in range(num_mini_batch):
        idx = perm[i * mbs:(i + 1) * mbs]
        yield {k: v[idx] for k, v in f.items()}


def _ref_recurrent(rb, adv, num_mini_batch, L, perm):
    """graph_buffer.py recurrent_generator's indexing: x[:-1].transpose(1, 2, 0, ...), chunks of L rows, np.stack(axis=1)
    then _flatten; rnn states at each chunk's first row."""
    T, n, N = rb.episode_length, rb.n_rollout_threads, rb.num_agents
    chunks = T * n * N // L
    mbs = chunks // num_mini_batch
    f = {k: v.transpose(1, 2, 0, *range(3, v.ndim)).reshape(-1, *v.shape[3:]) for k, v in _np_fields(rb, adv).items()}
    for i in range(num_mini_batch):
        idx = perm[i * mbs:(i + 1) * mbs]
        b = {}
        for k, v in f.items():
            if k in ('rnn_states', 'rnn_states_critic'):
                b[k] = np.stack([v[j * L] for j in idx]).reshape(mbs, *v.shape[1:])
            else:
                b[k] = np.stack([v[j * L:(j + 1) * L] for j in idx], axis=1).reshape(L * mbs, *v.shape[1:])
        yield b


def _check_batches(got, want, edges):
    got, want = list(got), list(want)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        keys = set(w) - ({'adj'} if edges else set())
        assert set(g) == keys | ({'edge_index', 'edge_attr'} if edges else set()), set(g) ^ keys
        for k in keys:
            np.testing.assert_array_equal(g[k].cpu().numpy(), w[k], err_msg=k)
        if edges:
            ei, ea = process_adj(torch.from_numpy(w['adj']))
            assert torch.equal(g['edge_index'].cpu(), ei) and torch.equal(_bits(g['edge_attr'].cpu()), _bits(ea))


@pytest.mark.parametrize('edges', [False, True])
@pytest.mark.parametrize('case', ['default', 'remainder', 'mini_batch_size', 'perm'])
def test_feed_forward_batches_follow_the_reference_indexing(case, edges):
    rb = _filled_buffer()                                          # T * n * N = 42 rows
    adv = torch.randn(rb.rewards.shape, generator=torch.Generator().manual_seed(5))
    nmb, mbs = {'default': (3, None), 'remainder': (4, None), 'mini_batch_size': (2, 11), 'perm': (3, None)}[case]
    perm = np.random.default_rng(1).permutation(42)
    kw = dict(perm=torch.from_numpy(perm)) if case == 'perm' else dict(perm=perm)
    got = rb.feed_forward_batches(adv, nmb, mini_batch_size=mbs, edges=edges, **kw)
    _check_batches(got, _ref_feed_forward(rb, adv, nmb, mbs, perm), edges)
    if case == 'default':   # the default permutation takes the generator
        a = list(rb.feed_forward_batches(adv, nmb, generator=torch.Generator().manual_seed(7)))
        b = list(rb.feed_forward_batches(adv, nmb, generator=torch.Generator().manual_seed(7)))
        assert all(torch.equal(x['obs'], y['obs']) for x, y in zip(a, b))


@pytest.mark.parametrize('edges', [False, True])
@pytest.mark.parametrize('L,nmb', [(7, 2), (3, 4), (5, 3)])      # T = 7: L = 3 and 5 make chunks cross columns
def test_recurrent_batches_follow_the_reference_indexing(L, nmb, edges):
    rb = _filled_buffer()
    adv = torch.randn(rb.rewards.shape, generator=torch.Generator().manual_seed(5))
    chunks = 42 // L
    perm = np.random.default_rng(L).permutation(chunks)
    got = rb.recurrent_batches(adv, nmb, L, edges=edges, perm=perm)
    _check_batches(got, _ref_recurrent(rb, adv, nmb, L, perm), edges)


def _np_advantages(rb, scale=None, shift=None):
    ret, vp = rb.returns.numpy()[:-1], rb.value_preds.numpy()[:-1]
    if scale is not None:
        vp = vp * np.float32(scale) + np.float32(shift)
    adv = ret - vp
    a = adv.astype(np.float64)
    a[rb.active_masks.numpy()[:-1] == 0] = np.nan
    mean, std = np.float32(np.nanmean(a)), np.float32(np.nanstd(a))
    return adv, mean, std, (adv - mean) / (std + np.float32(1e-5))


@pytest.mark.parametrize('denorm', [False, True])
def test_compute_advantages_cpu_equals_the_numpy_expression(denorm):
    rb = _filled_buffer()
    kw = dict(value_scale=torch.tensor([1.75]), value_shift=torch.tensor([-0.25])) if denorm else {}
    rb.compute_returns(torch.randn(3, 2, 1), **kw)
    adv, mean, std, norm = _np_advantages(rb, 1.75 if denorm else None, -0.25)
    raw, m, s = rb.compute_advantages(normalize=False, **kw)
    np.testing.assert_array_equal(raw.numpy(), adv)
    assert m.dim() == 0 and s.dim() == 0 and m.dtype == torch.float32
    assert m.item() == mean and s.item() == std
    got, _, _ = rb.compute_advantages(**kw)
    np.testing.assert_array_equal(got.numpy(), norm)
    rb.active_masks.zero_()
    _, m, s = rb.compute_advantages()
    assert np.isnan(m.item()) and np.isnan(s.item())


def test_cpu_denormalisation_is_the_two_op_form():
    """returns_loop with value_scale / value_shift: every value read is v * scale + shift (float32, one rounding each)."""
    rb = _filled_buffer(use_gae=True, use_proper_time_limits=True)
    scale, shift = np.float32(1.5), np.float32(0.125)
    nv = torch.randn(3, 2, 1)
    rb.compute_returns(nv, value_scale=torch.tensor([scale]), value_shift=torch.tensor([shift]))
    r, m, b = rb.rewards.numpy(), rb.masks.numpy(), rb.bad_masks.numpy()
    v = rb.value_preds.numpy() * scale + shift
    g32, gl32 = np.float32(rb.gamma), np.float32(rb.gamma * rb.gae_lambda)
    gae = np.zeros_like(v[0])
    for t in reversed(range(rb.episode_length)):
        delta = r[t] + g32 * v[t + 1] * m[t + 1] - v[t]
        gae = (delta + gl32 * m[t + 1] * gae) * b[t + 1]
        np.testing.assert_array_equal(rb.returns.numpy()[t], gae + v[t])


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the kernel against the torch loop
# ----------------------------------------------------------------------------------------------------------------------
def _inputs(T, C, seed, device='cuda'):
    """Seeded (T[+1], C) inputs with zero masks, non-binary bad_masks, signed zeros and large magnitudes."""
    g = torch.Generator(device=device).manual_seed(seed)
    def rnd(rows):
        x = torch.randn((rows, C), generator=g, device=device)
        mag = torch.pow(10.0, torch.randint(-3, 16, (rows, C), generator=g, device=device).float())
        x = torch.where(torch.rand((rows, C), generator=g, device=device) < 0.1, x * mag, x)
        return torch.where(torch.rand((rows, C), generator=g, device=device) < 0.05, torch.full_like(x, -0.0), x)
    u = lambda rows: torch.rand((rows, C), generator=g, device=device)
    masks = (u(T + 1) < 0.8).float()
    bad = torch.where(u(T + 1) < 0.5, (u(T + 1) < 0.7).float(), u(T + 1))          # binary and fractional
    zero = torch.where(u(T + 1) < 0.5, torch.full_like(masks, -0.0), torch.zeros_like(masks))    # both zeros are inactive
    active = torch.where(u(T + 1) < 0.8, u(T + 1) + 0.5, zero)
    return dict(rewards=rnd(T), value_preds=rnd(T + 1), returns=rnd(T + 1), masks=masks, bad_masks=bad,
                active_masks=active, next_value=rnd(1)[0])


def _run(inp, use_gae, ptl, denorm, kernel, gamma=0.99, lam=0.95, adv=False):
    x = {k: v.clone() for k, v in inp.items()}
    dn = dict(value_scale=torch.tensor([1.375], device='cuda'), value_shift=torch.tensor([-2.5], device='cuda')) if denorm else {}
    args = (x['rewards'], x['value_preds'], x['returns'], x['masks'], x['bad_masks'], x['next_value'], gamma, lam,
            use_gae, ptl)
    if kernel:
        if adv:
            x['adv'] = torch.full_like(x['rewards'], 7.0)
            x['stats'] = torch.empty(2, device='cuda')
            x['stats64'] = torch.empty(3, dtype=torch.float64, device='cuda')
            returns_kernel(*args, advantages=x['adv'], active_masks=x['active_masks'], stats=x['stats'],
                           stats64=x['stats64'], **dn)
        else:
            returns_kernel(*args, **dn)
    else:
        returns_loop(*args, **dn)
    return x


SHAPES = [(1, 1), (6, 15), (250, 32768), (350, 163840), (7, 262149)]


@gpu
@pytest.mark.parametrize('denorm', [False, True])
@pytest.mark.parametrize('use_gae,ptl', MODES)
@pytest.mark.parametrize('T,C', SHAPES)
def test_kernel_equals_the_torch_loop_bit_for_bit(T, C, use_gae, ptl, denorm):
    inp = _inputs(T, C, seed=T * 7 + C)
    want = _run(inp, use_gae, ptl, denorm, kernel=False)
    got = _run(inp, use_gae, ptl, denorm, kernel=True)
    for k in ('returns', 'value_preds'):
        assert torch.equal(_bits(got[k]), _bits(want[k])), k
    # only the slots the loop writes: returns[T] (the input's sentinel) stays in GAE mode, value_preds in discounted mode
    if use_gae:
        assert torch.equal(_bits(got['returns'][T]), _bits(inp['returns'][T]))
    else:
        assert torch.equal(_bits(got['value_preds']), _bits(inp['value_preds']))
    for k in ('rewards', 'masks', 'bad_masks', 'next_value'):
        assert torch.equal(_bits(got[k]), _bits(inp[k])), k


@gpu
def test_only_the_written_slots_change_with_a_sentinel():
    T, C = 9, 100
    inp = _inputs(T, C, seed=4)
    sentinel = torch.tensor([0x7fc12345], dtype=torch.int32, device='cuda').view(torch.float32)
    inp['returns'][T] = sentinel
    got = _run(inp, True, True, True, kernel=True, adv=True)
    assert torch.equal(_bits(got['returns'][T]), _bits(inp['returns'][T]))
    assert torch.equal(_bits(got['value_preds'][:T]), _bits(inp['value_preds'][:T]))
    assert torch.equal(_bits(got['value_preds'][T]), _bits(inp['next_value']))


@gpu
@pytest.mark.parametrize('use_gae,ptl', MODES)
def test_reference_fixture_on_a_cuda_buffer(use_gae, ptl):
    """tests/golden/aux/rollout_buffer.npz (the reference GraphReplayBuffer) through compute_returns on CUDA."""
    z = np.load(ROLLOUT_GOLDEN)
    n, N, L, D, F, T = (int(v) for v in z['meta'])
    rb = DeviceGraphRolloutBuffer(_fake_env(n, N, L, D, F, device='cuda'), episode_length=T, gamma=0.97, gae_lambda=0.9,
                                  use_gae=use_gae, use_proper_time_limits=ptl, hidden_size=8)
    dev = lambda name, k=None: torch.from_numpy(z['in_' + name] if k is None else z['in_' + name][k]).cuda()
    rb.warmup(reset_out=(dev('obs0'), dev('agent_id'), torch.zeros_like(rb.node_obs[0]), torch.zeros_like(rb.adj[0])))
    rb.bad_masks.copy_(dev('bad_masks'))
    tag = f"gae{int(use_gae)}_ptl{int(ptl)}_cv1"
    for p in range(2):
        for t in range(T):
            k = p * T + t
            rb.insert((dev('obs', k), dev('agent_id'), dev('node_obs', k), dev('adj', k), dev('rewards', k)[..., 0],
                       dev('dones', k), None), values=dev('values', k), actions=dev('actions', k),
                      action_log_probs=dev('action_log_probs', k), rnn_states=dev('rnn_states', k),
                      rnn_states_critic=dev('rnn_states_critic', k))
        rb.compute_returns(dev('next_values', p))
        for name in ('returns', 'value_preds'):
            np.testing.assert_allclose(getattr(rb, name).cpu().numpy(), z[f"{tag}_pass{p}_{name}"], rtol=1e-6, atol=1e-6)
        rb.after_update()


# ----------------------------------------------------------------------------------------------------------------------
# GPU: advantages and moments
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('denorm', [False, True])
@pytest.mark.parametrize('use_gae,ptl', MODES)
def test_raw_advantages_and_float64_moments(use_gae, ptl, denorm):
    T, C = 250, 32768
    inp = _inputs(T, C, seed=11)
    # a mean 10^3 standard deviations away from zero
    inp['rewards'] = torch.randn((T, C), device='cuda', generator=torch.Generator(device='cuda').manual_seed(2)) + 1000.0
    inp['value_preds'].normal_(0.0, 0.01)
    inp['masks'].fill_(0.0)
    inp['bad_masks'].fill_(1.0)
    got = _run(inp, use_gae, ptl, denorm, kernel=True, adv=True)
    want = _run(inp, use_gae, ptl, denorm, kernel=False)
    assert torch.equal(_bits(got['returns']), _bits(want['returns']))
    vp = want['value_preds'][:-1]
    if denorm:
        vp = vp * torch.tensor([1.375], device='cuda') + torch.tensor([-2.5], device='cuda')
    assert torch.equal(_bits(got['adv']), _bits(want['returns'][:-1] - vp))
    a = got['adv'].cpu().numpy().astype(np.float64)[inp['active_masks'][:-1].cpu().numpy() != 0]
    mean = a.mean()
    std = np.sqrt(((a - mean) ** 2).mean())
    s64 = got['stats64'].cpu().numpy()
    assert s64[0] == a.size
    assert abs(s64[1] - mean) <= 1e-12 * abs(mean) and abs(s64[2] - std) <= 1e-12 * std, (s64, mean, std)
    assert got['stats'].cpu().numpy().tolist() == [np.float32(s64[1]), np.float32(s64[2])]
    again = _run(inp, use_gae, ptl, denorm, kernel=True, adv=True)
    for k in ('adv', 'stats', 'returns'):
        assert torch.equal(_bits(again[k]), _bits(got[k])), k
    assert torch.equal(again['stats64'].view(torch.int64), got['stats64'].view(torch.int64))


@gpu
def test_all_inactive_gives_nan_and_buffer_normalisation():
    rb = _filled_buffer(n=64, N=8, T=25, device='cuda')
    rb.compute_returns(torch.randn(64, 8, 1, device='cuda'))
    adv, mean, std = rb.compute_advantages(normalize=False)
    raw = rb.returns[:-1] - rb.value_preds[:-1]
    assert torch.equal(_bits(adv), _bits(raw))
    norm, m2, s2 = rb.compute_advantages()
    assert torch.equal(_bits(norm), _bits((raw - mean) / (std + 1e-5)))
    assert mean.dim() == 0 and mean.is_cuda and m2.item() == mean.item() and s2.item() == std.item()
    a = raw.cpu().numpy().astype(np.float64)
    a[rb.active_masks[:-1].cpu().numpy() == 0] = np.nan
    assert abs(mean.item() - np.nanmean(a)) <= 1e-6 * abs(np.nanmean(a)) and abs(std.item() - np.nanstd(a)) <= 1e-6 * np.nanstd(a)
    rb.active_masks.zero_()
    _, m, s = rb.compute_advantages()
    assert np.isnan(m.item()) and np.isnan(s.item())


@gpu
def test_no_host_sync_and_side_stream():
    rb = _filled_buffer(n=128, N=8, T=40, device='cuda', use_proper_time_limits=True)
    nv = torch.randn(128, 8, 1, device='cuda')
    scale, shift = torch.tensor([0.5], device='cuda'), torch.tensor([3.0], device='cuda')
    rb.compute_returns(nv, scale, shift)               # loads the library outside the checked region
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        rb.compute_returns(nv, scale, shift)
        adv, mean, std = rb.compute_advantages(value_scale=scale, value_shift=shift)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ref = (rb.returns.clone(), adv.clone(), mean.clone(), std.clone())
    # clear the slots the side-stream pass must rewrite (GAE leaves returns[T] untouched, so it keeps its value)
    rb.returns[:-1].zero_()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        rb.compute_returns(nv, scale, shift)
        adv2, mean2, std2 = rb.compute_advantages(value_scale=scale, value_shift=shift)
    torch.cuda.current_stream().wait_stream(s)
    for a, b in zip(ref, (rb.returns, adv2, mean2, std2)):
        assert torch.equal(_bits(a), _bits(b))


@gpu
def test_64bit_indexing():
    """T * C > 2^31: tail columns and the last steps equal the loop on that column subset."""
    T, C = 129, (1 << 24) + 3
    inp = _inputs(T, C, seed=9)
    cols = torch.cat([torch.arange(64), torch.arange(C - 4099, C)]).cuda()
    sub = {k: v[..., cols].contiguous() for k, v in inp.items()}
    want = _run(sub, True, True, True, kernel=False)
    x = inp                                             # in place: no second copy of ~60 GB
    x['adv'] = torch.empty_like(x['rewards'])
    stats = torch.empty(2, device='cuda')
    returns_kernel(x['rewards'], x['value_preds'], x['returns'], x['masks'], x['bad_masks'], x['next_value'], 0.99, 0.95,
                   True, True, torch.tensor([1.375], device='cuda'), torch.tensor([-2.5], device='cuda'),
                   advantages=x['adv'], active_masks=x['active_masks'], stats=stats)
    assert torch.equal(_bits(x['returns'][:, cols]), _bits(want['returns']))
    assert torch.equal(_bits(x['value_preds'][T, cols]), _bits(want['value_preds'][T]))
    assert torch.isfinite(stats).all()
    del inp, x, sub
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------------------------------------------------
# GPU: records and dense buffers serve identical minibatches
# ----------------------------------------------------------------------------------------------------------------------
def _collected_pair(dyn, N, n, T):
    from layered_safe_marl_b200 import B200GraphVecEnv
    args = G.default_args(dynamics_type=dyn, num_agents=N, use_safety_filter=True, episode_length=T,
                          world_size=2 if N == 8 else 4)
    envs = [B200GraphVecEnv(args, num_envs=n, seed=21) for _ in range(2)]
    bufs = [DeviceGraphRolloutBuffer(envs[0], T, zero_copy=True),
            DeviceGraphRolloutBuffer(envs[1], T, zero_copy=True, graph_storage='records')]
    rng = np.random.default_rng(8)
    for b in bufs:
        b.warmup()
    for s in range(T):
        a = torch.as_tensor(rng.integers(0, 25, (n, N)).astype(np.int32), device='cuda')
        vals = torch.as_tensor(rng.standard_normal((n, N, 1)).astype(np.float32), device='cuda')
        rnn = torch.as_tensor(rng.standard_normal((n, N, 1, 64)).astype(np.float32), device='cuda')
        outs = [e.step(a, 0) for e in envs]
        for b, o in zip(bufs, outs):
            b.insert(o, values=vals, actions=a[..., None].float(), action_log_probs=vals * 0.5, rnn_states=rnn,
                     rnn_states_critic=rnn * 2)
    nv = torch.as_tensor(rng.standard_normal((n, N, 1)).astype(np.float32), device='cuda')
    for b in bufs:
        b.compute_returns(nv)
    return bufs


@gpu
@pytest.mark.parametrize('dyn,N', [('double_integrator', 8), ('airtaxi', 10)])
def test_records_and_dense_buffers_yield_identical_minibatches(dyn, N):
    n, T = 32, 6
    dense, rec = _collected_pair(dyn, N, n, T)
    advs = [b.compute_advantages()[0] for b in (dense, rec)]
    assert torch.equal(_bits(advs[0]), _bits(advs[1]))
    perm_ff = torch.randperm(T * n * N, device='cuda')
    perm_rc = torch.randperm(T * n * N // 4)
    for edges in (False, True):
        for make in (lambda b, a: b.feed_forward_batches(a, 3, edges=edges, perm=perm_ff),
                     lambda b, a: b.recurrent_batches(a, 2, 4, edges=edges, perm=perm_rc)):
            for bd, br in zip(make(dense, advs[0]), make(rec, advs[1])):
                assert set(bd) == set(br)
                for k in bd:
                    assert bd[k].shape == br[k].shape and bd[k].dtype == br[k].dtype, k
                    assert torch.equal(bd[k].view(torch.int32) if bd[k].dtype == torch.float32 else bd[k],
                                       br[k].view(torch.int32) if br[k].dtype == torch.float32 else br[k]), k
                if edges:
                    rows = bd['node_obs'].shape[0]
                    assert bd['edge_index'].numel() == 0 or int(bd['edge_index'].max()) < rows * dense.env.E
    # edges=True equals process_adj of the dense rows
    b = next(dense.feed_forward_batches(advs[0], 3, perm=perm_ff))
    e = next(rec.feed_forward_batches(advs[1], 3, edges=True, perm=perm_ff))
    ei, ea = process_adj(b['adj'])
    assert torch.equal(e['edge_index'], ei) and torch.equal(_bits(e['edge_attr']), _bits(ea))
