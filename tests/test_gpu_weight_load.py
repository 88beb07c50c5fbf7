"""Loading actor and critic weights from CUDA tensors (actor_load_device / critic_load_device): the pack kernel that
builds the weight images on the device, in stream order and without a host round trip.

An actor or critic loaded from CUDA tensors must compute exactly what one loaded from the same numpy arrays computes
(both go through the same pack kernel; the host path stages the arrays first), for every image layout: tensor-core
teams, the fp32 FFMA kernel, the dense3 head that lives outside the staged part of the blob, and observation widths
past 32 where the tensor-core image is not used at all.  Logits and critic values are also checked against the
float64 oracles.  Every device load below goes into a handle that was created with OTHER weights, so a word the pack
kernel fails to write keeps a stale value and shows up.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import actor_ref

gpu = pytest.mark.gpu
ATOL = 1e-5
B = 4099
P = 211  # distinct observation rows: obs[b] = pool[b % P]

# (N, D, heads, dense3 head)
ACTORS = ([(2, D, A, False) for D in (11, 21) for A in (5, [5, 10], [3, 4], 16)] +
          [(3, 10, 5, False), (3, 10, 8, False), (6, 16, 5, True), (12, 28, 5, True), (5, 14, 5, False)] +
          [(2, 33, 5, False), (2, 33, 5, True), (1, 57, 5, False), (1, 57, 5, True)])
CRITICS = [('spread_n3', 10), ('reference', 21), ('model_n12', 28)]


def _impls(N, D, A):
    width = sum(A) if isinstance(A, list) else A
    tc = D <= 32 and (N in (2, 3) or (N in (4, 6, 8, 9, 12) and width <= 8))
    return ['simt', 'tc'] if tc else ['simt']


def _cuda(sd):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in sd.items()}


def _obs(N, D, seed=1):
    pool = np.random.RandomState(seed).uniform(-2, 2, (P, N, D)).astype(np.float32)
    return pool, torch.from_numpy(pool).cuda()[torch.arange(B, device='cuda') % P].contiguous()


def _actor_out(actor, obs):
    out = actor.forward(obs, step=3, env_id_offset=2 ** 32 - 100, want_logits=True, want_onehot=True,
                        want_next_state=actor.has_model)
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in out.items() if v is not None}


def _same_bits(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, k
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k


def _check_logits(out, sd, pool):
    want = np.concatenate(actor_ref.forward(sd, pool)['logits'], -1)
    got = out['logits'].double().cpu().numpy()
    assert np.abs(got - want[np.arange(B) % P]).max() <= ATOL


def _critic_golden(tag):
    from tests.conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, 'critic_%s.npz' % tag))
    return g, {k[3:]: g[k] for k in g.files if k.startswith('sd/')}


def _perturbed(sd, seed):
    rng = np.random.RandomState(seed)
    return {k: (v + rng.uniform(-0.1, 0.1, v.shape)).astype(np.float32) for k, v in sd.items()}


def _critic_out(critic, g):
    out = critic.forward(torch.from_numpy(g['obs']), torch.from_numpy(g['action']))
    torch.cuda.synchronize()
    return {'q': out[0].clone(), 'r': out[1].clone()} if critic.model else {'q': out.clone()}


@gpu
@pytest.mark.parametrize('N,D,A,model', ACTORS)
def test_actor_device_load_matches_host_load(N, D, A, model):
    """An actor created with weights W0 and reloaded with W1 from CUDA tensors gives logits, one-hot, actions and
    next_state bit-identical to a fresh actor created from W1's numpy arrays, on every implementation that covers
    the shape; its logits are within 1e-5 of the float64 oracle."""
    import multiagent_rl_b200 as m
    w0, w1 = actor_ref.init_state_dict(D, A, 10 + N, model_head=model), actor_ref.init_state_dict(D, A, 20 + N, model_head=model)
    pool, obs = _obs(N, D)
    for impl in _impls(N, D, A):
        dev = m.FusedActor(w0, seed=5, impl=impl)
        dev.load_state_dict(_cuda(w1))
        host = m.FusedActor(w1, seed=5, impl=impl)
        got, want = _actor_out(dev, obs), _actor_out(host, obs)
        _same_bits(got, want)
        _check_logits(got, w1, pool)
        assert ('next_state' in got) == model and ('act_c' in got) == isinstance(A, list)


@gpu
@pytest.mark.parametrize('tag,D', CRITICS)
def test_critic_device_load_matches_host_load(tag, D):
    """A critic created with other weights and reloaded from CUDA tensors gives q (and r) bit-identical to one created
    from the fixture's numpy arrays, and within 1e-5 of the reference network's outputs."""
    import multiagent_rl_b200 as m
    g, sd = _critic_golden(tag)
    dev = m.FusedCritic(_perturbed(sd, 1), obs_dim=D)
    dev.load_state_dict(_cuda(sd))
    host = m.FusedCritic(sd, obs_dim=D)
    got, want = _critic_out(dev, g), _critic_out(host, g)
    _same_bits(got, want)
    assert np.abs(got['q'].cpu().numpy() - g['q']).max() <= ATOL
    if 'r' in g.files:
        assert np.abs(got['r'].cpu().numpy() - g['r']).max() <= ATOL


def _flat_views(sd):
    """Each tensor as a view into one flat CUDA buffer, the first at 4 bytes past a 16-byte boundary and the rest at
    whatever offset their sizes give (4-byte aligned only)."""
    flat = torch.empty(1 + sum(v.size for v in sd.values()), dtype=torch.float32, device='cuda')
    out, off = {}, 1
    for k, v in sd.items():
        out[k] = flat[off:off + v.size].view(v.shape)
        out[k].copy_(torch.from_numpy(v))
        off += v.size
    assert next(iter(out.values())).data_ptr() % 16 == 4
    return out


def _transposed(sd):
    """Non-contiguous tensors with the same values: 2-D tensors as transposes of their transposes, 1-D tensors as
    every other element of a buffer twice as long."""
    out = {}
    for k, v in sd.items():
        t = torch.from_numpy(v).cuda()
        out[k] = t.t().contiguous().t() if t.dim() == 2 else torch.stack([t, t], 1)[:, 0]
        assert not out[k].is_contiguous() or 1 in t.shape  # torch calls a view with a dimension of 1 contiguous
    return out


@gpu
@pytest.mark.parametrize('N,D,A,model', [(2, 21, [5, 10], False), (6, 16, 5, True), (1, 57, 5, True)])
def test_actor_device_load_from_unaligned_and_strided_tensors(N, D, A, model):
    import multiagent_rl_b200 as m
    w0, w1 = actor_ref.init_state_dict(D, A, 1, model_head=model), actor_ref.init_state_dict(D, A, 2, model_head=model)
    _, obs = _obs(N, D)
    want = _actor_out(m.FusedActor(w1, seed=5), obs)
    for make in (_flat_views, _transposed):
        actor = m.FusedActor(w0, seed=5)
        actor.load_state_dict(make(w1))
        _same_bits(_actor_out(actor, obs), want)


@gpu
def test_critic_device_load_from_unaligned_and_strided_tensors():
    import multiagent_rl_b200 as m
    g, sd = _critic_golden('model_n12')
    want = _critic_out(m.FusedCritic(sd, obs_dim=28), g)
    for make in (_flat_views, _transposed):
        critic = m.FusedCritic(_perturbed(sd, 2), obs_dim=28)
        critic.load_state_dict(make(sd))
        _same_bits(_critic_out(critic, g), want)


@gpu
def test_device_load_is_stream_ordered_without_a_host_sync():
    """sleep -> in-place change of the CUDA tensors -> load -> forward, enqueued without a synchronize: the call
    returns while the sleep still runs, and the forward sees the changed weights."""
    import multiagent_rl_b200 as m
    N, D, A = 6, 16, 5
    w0 = actor_ref.init_state_dict(D, A, 3, model_head=True)
    _, obs = _obs(N, D)
    actor = m.FusedActor(w0, seed=5)
    params = _cuda(w0)
    warm = _cuda(w0)  # the first launch of a kernel in the process may load its module and wait for the device
    for v in warm.values():
        v.mul_(1.25).add_(0.01)
    actor.load_state_dict(warm)
    actor.forward(obs, want_logits=True, want_onehot=True, want_next_state=True)
    torch.cuda.synchronize()
    torch.cuda._sleep(1_000_000_000)  # about 0.5 s at the B200's clocks
    for v in params.values():
        v.mul_(1.25).add_(0.01)
    actor.load_state_dict(params)
    ev = torch.cuda.Event()
    ev.record()
    pending = not ev.query()
    out = actor.forward(obs, step=3, env_id_offset=2 ** 32 - 100, want_logits=True, want_onehot=True,
                        want_next_state=True)
    assert pending, 'load_state_dict waited for the GPU'
    torch.cuda.synchronize()
    fresh = m.FusedActor({k: v.cpu().numpy() for k, v in params.items()}, seed=5)
    _same_bits({k: v for k, v in out.items() if v is not None}, _actor_out(fresh, obs))


@gpu
@pytest.mark.parametrize('kind', ['actor', 'critic'])
def test_device_load_captures_in_a_cuda_graph(kind):
    """load_state_dict(cuda state_dict) captured in a graph (the capture fails if the call synchronises or allocates):
    after an in-place change of the tensors, a replay loads the changed weights."""
    import multiagent_rl_b200 as m
    if kind == 'actor':
        N, D, A = 3, 10, 5
        w0 = actor_ref.init_state_dict(D, A, 4, model_head=True)
        _, obs = _obs(N, D)
        make = lambda sd: m.FusedActor(sd, seed=5)  # noqa: E731
        run = lambda h: _actor_out(h, obs)  # noqa: E731
    else:
        g, w0 = _critic_golden('model_n12')
        make = lambda sd: m.FusedCritic(sd, obs_dim=28)  # noqa: E731
        run = lambda h: _critic_out(h, g)  # noqa: E731
    h = make(w0)
    params = _cuda(w0)
    before = run(h)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        h.load_state_dict(params)
    _same_bits(run(h), before)  # capturing runs nothing
    for v in params.values():
        v.mul_(0.75).sub_(0.02)
    graph.replay()
    _same_bits(run(h), run(make({k: v.cpu().numpy() for k, v in params.items()})))


def _bad_shape(v):
    return v[:-1] if v.ndim == 1 else v[:, :-1]


@gpu
def test_wrong_shapes_and_missing_keys_are_refused_before_any_launch():
    import multiagent_rl_b200 as m
    N, D, A = 2, 21, [5, 10]
    w0 = actor_ref.init_state_dict(D, A, 6, model_head=True)
    _, obs = _obs(N, D)
    actor = m.FusedActor(w0, seed=5)
    before = _actor_out(actor, obs)
    w1 = actor_ref.init_state_dict(D, A, 7, model_head=True)
    for key in w1:
        bad = dict(w1, **{key: _bad_shape(w1[key])})
        with pytest.raises(ValueError, match=key.replace('.', r'\.')):
            actor.load_state_dict(bad)
        with pytest.raises(ValueError, match=key.replace('.', r'\.')):
            actor.load_state_dict(_cuda(bad))
        short = {k: v for k, v in w1.items() if k != key}
        with pytest.raises(KeyError):
            actor.load_state_dict(short)
        with pytest.raises(KeyError):
            actor.load_state_dict(_cuda(short))
    _same_bits(_actor_out(actor, obs), before)
    g, sd = _critic_golden('model_n12')
    critic = m.FusedCritic(sd, obs_dim=28)
    cbefore = _critic_out(critic, g)
    for key in sd:
        bad = dict(sd, **{key: _bad_shape(sd[key])})
        for src in (bad, _cuda(bad)):
            with pytest.raises(ValueError, match=key.replace('.', r'\.')):
                critic.load_state_dict(src)
        with pytest.raises(KeyError):
            critic.load_state_dict(_cuda({k: v for k, v in sd.items() if k != key}))
    _same_bits(_critic_out(critic, g), cbefore)


def _struct(cls, fields, ptrs):
    w = cls()
    for f, p in zip(fields, ptrs):
        setattr(w, f, p)
    return w


@gpu
def test_host_pointers_are_refused_by_the_device_entry_points():
    """actor_load_device / critic_load_device called with host memory - pageable numpy, pinned torch - in any one
    field, or with a missing tensor: MPE_EINVAL, and the loaded weights are unchanged."""
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    from multiagent_rl_b200.actor import _KEYS
    lib = _lib.load()
    stream = _lib.current_stream(torch.device('cuda'))
    N, D, A = 3, 10, 5
    w0 = actor_ref.init_state_dict(D, A, 8)
    _, obs = _obs(N, D)
    actor = m.FusedActor(w0, seed=5)
    before = _actor_out(actor, obs)
    names = list(_KEYS) + [('dense2_w', 'dense2.module.weight'), ('dense2_b', 'dense2.module.bias')]
    w1 = actor_ref.init_state_dict(D, A, 9)
    dev = [torch.from_numpy(w1[k]).cuda() for _, k in names]
    host = [np.ascontiguousarray(w1[k]) for _, k in names]
    pinned = torch.from_numpy(host[0]).pin_memory()
    fields = [f for f, _ in names]
    for i in range(len(names)):
        for hp in [host[i].ctypes.data, 0] + ([pinned.data_ptr()] if i == 0 else []):  # 0: NULL
            ptrs = [t.data_ptr() for t in dev]
            ptrs[i] = hp
            w = _struct(_lib.ActorWeights, fields, ptrs)
            assert lib.actor_load_device(actor._h, C.byref(w), stream) == _lib.MPE_EINVAL, (i, hp)
    torch.cuda.synchronize()
    _same_bits(_actor_out(actor, obs), before)
    # the same tensors as device pointers load
    assert lib.actor_load_device(actor._h, C.byref(_struct(_lib.ActorWeights, fields, [t.data_ptr() for t in dev])),
                                 stream) == _lib.MPE_OK
    _same_bits(_actor_out(actor, obs), _actor_out(m.FusedActor(w1, seed=5), obs))

    from multiagent_rl_b200.critic import _KEYS as CKEYS
    g, sd = _critic_golden('spread_n3')
    critic = m.FusedCritic(sd, obs_dim=10)
    cbefore = _critic_out(critic, g)
    cfields = [f for f, _ in CKEYS]
    cdev = [torch.from_numpy(_perturbed(sd, 3)[k]).cuda() for _, k in CKEYS]
    chost = [np.ascontiguousarray(sd[k]) for _, k in CKEYS]
    for i in range(len(CKEYS)):
        for hp in (chost[i].ctypes.data, 0):
            ptrs = [t.data_ptr() for t in cdev]
            ptrs[i] = hp
            w = _struct(_lib.CriticWeights, cfields, ptrs)
            assert lib.critic_load_device(critic._h, C.byref(w), stream) == _lib.MPE_EINVAL, (i, hp)
    torch.cuda.synchronize()
    _same_bits(_critic_out(critic, g), cbefore)


def test_device_loads_reject_null_arguments():
    from multiagent_rl_b200 import _lib
    lib = _lib.load()
    assert lib.actor_load_device(None, None, None) == _lib.MPE_EINVAL
    assert b'null' in lib.mpe_last_error()
    assert lib.actor_load_device(None, C.byref(_lib.ActorWeights()), None) == _lib.MPE_EINVAL
    assert lib.critic_load_device(None, None, None) == _lib.MPE_EINVAL
    assert lib.critic_load_device(None, C.byref(_lib.CriticWeights()), None) == _lib.MPE_EINVAL
