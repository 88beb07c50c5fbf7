"""GPU tests of the actor backward (C ABI actor_backward, FusedActor.backward, FusedActorNetwork) against float64
autograd of the torch restatement tests/_actor_torch.py (itself pinned to the reference by
tests/test_actor_grad_oracle.py), and of the properties that hold exactly.

Tolerance per gradient tensor: max|g - g64| <= TOL * max(1, max|g64|), TOL = 1e-4 for default-init weights and 5e-4
for "sharp" weights (saturating gates).  Samples with a float64 dense1 pre-activation or BiLSTM output within 1e-5 of
zero are dropped from the batch before either side runs (fp32 may sit on the other side of the kink); the tests print
how many."""
import copy
import ctypes as C
import hashlib

import numpy as np
import pytest
import torch

from oracle import actor_ref, build_ref
from tests import _actor_torch as at
from tests import _critic_torch as ct
from tests.test_gpu_reference_loop import _trainer_class, ref  # noqa: F401 - the reference-loop fixture

pytestmark = pytest.mark.gpu


def _sharp_actor(seed, D, heads, model):
    """Default-init weights scaled up: many gates saturate, logits are peaked (trained policies are sharper).  Larger
    LSTM weights push so many output gates to zero that most samples have a BiLSTM output within 1e-5 of the kink."""
    sd = actor_ref.init_state_dict(D, heads, seed, model_head=model)
    for k in sd:
        sd[k] = sd[k] * (2.0 if k.startswith('bilstm') or k.startswith('dense1') else 3.0)
    return sd


def _default_actor(seed, D, heads, model):
    import multiagent_rl_b200 as m
    torch.manual_seed(seed)
    return {k: v.numpy() for k, v in m.FusedActorNetwork(D, heads, model_head=model).state_dict().items()}


def _width(heads):
    return sum(heads) if isinstance(heads, (list, tuple)) else heads


def _case(N, D, heads, model, B, weights, seed):
    rng = np.random.RandomState(seed)
    sd = (_sharp_actor if weights == 'sharp' else _default_actor)(seed, D, heads, model)
    obs = rng.uniform(-2, 2, (B, N, D)).astype(np.float32)
    keep = at.kink_free(sd, obs)
    print('dropped %d of %d samples within 1e-5 of a relu kink' % (B - int(keep.sum()), B))
    assert keep.sum() >= 0.7 * B
    return rng, sd, obs[keep]


def _check(got, want, tol, what):
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(np.asarray(got, np.float64) - want).max())
    assert err <= tol * scale, (what, err, scale)


def _fused(sd):
    import multiagent_rl_b200 as m
    return m.FusedActor(sd, impl='simt')


@pytest.mark.parametrize('N,D,heads,model,B,weights,with_dns', [
    pytest.param(1, 6, 5, False, 7, 'sharp', False, id='n1-7-sharp'),
    pytest.param(2, 21, [5, 10], False, 2048, 'default', False, id='n2-reference-2048'),
    pytest.param(2, 11, 5, False, 300, 'sharp', False, id='n2-speaker-300-sharp'),
    pytest.param(3, 10, 5, False, 4099, 'sharp', False, id='n3-4099-sharp'),
    pytest.param(3, 10, 5, False, 1024, 'default', False, id='n3-1024'),
    pytest.param(4, 18, 5, True, 1025, 'sharp', True, id='n4-model-1025-sharp'),
    pytest.param(6, 16, 5, True, 515, 'default', False, id='n6-model-dns-none'),
    pytest.param(6, 16, 5, True, 777, 'sharp', True, id='n6-model-777-sharp'),
    pytest.param(9, 22, [5, 10], False, 333, 'sharp', False, id='n9-two-heads-sharp'),
    pytest.param(12, 28, 5, True, 1187, 'default', True, id='n12-model-past-one-wave'),
    pytest.param(12, 64, [6, 10], True, 129, 'sharp', True, id='n12-d64-two-heads-model'),
    pytest.param(3, 64, 5, False, 1200, 'default', False, id='n3-d64'),
    pytest.param(3, 10, 5, False, 65539, 'default', False, id='b65539-ragged'),
])
def test_actor_backward_vs_float64_autograd(N, D, heads, model, B, weights, with_dns):
    """Every weight gradient and dobs: 1..12 agents, D up to 64, one head, two heads, the model head with dnext_state
    given and None, batches from 7 to past one wave of warps."""
    rng, sd, obs = _case(N, D, heads, model, B, weights, N * 1000 + D + B)
    B = obs.shape[0]
    dl = rng.randn(B, N, _width(heads)).astype(np.float32)
    dn = rng.randn(B, N, D).astype(np.float32) if with_dns else None
    want = at.grads(sd, obs, dl, dn)
    got = _fused(sd).backward(torch.from_numpy(obs), torch.from_numpy(dl), None if dn is None else torch.from_numpy(dn),
                              want_obs=True)
    tol = 5e-4 if weights == 'sharp' else 1e-4
    _check(got['obs'].cpu().numpy(), want['obs'], tol, 'obs')
    assert sorted(got['weights']) == sorted(sd)
    for k, v in got['weights'].items():
        _check(v.cpu().numpy(), want[k], tol, k)
    w = got['weights']
    for sfx in ('', '_reverse'):
        assert torch.equal(w['bilstm.bias_ih_l0' + sfx], w['bilstm.bias_hh_l0' + sfx])


def test_actor_backward_is_bitwise_reproducible_and_position_independent():
    """Weight gradients are the same bits on every call, on a side stream, from a NaN-filled workspace and replayed
    from a CUDA graph; a sample's dobs is the same bits under permutation and slicing of the batch; nothing is written
    past row B or into outputs that were not asked for; bad arguments are refused."""
    from multiagent_rl_b200 import _lib
    N, D, heads, B, pad = 3, 16, [5, 10], 5003, 16
    rng = np.random.RandomState(23)
    sd = _sharp_actor(23, D, heads, True)
    actor = _fused(sd)
    A = _width(heads)
    obs = torch.from_numpy(rng.uniform(-2, 2, (B, N, D)).astype(np.float32)).cuda()
    dl = torch.from_numpy(rng.randn(B, N, A).astype(np.float32)).cuda()
    dn = torch.from_numpy(rng.randn(B, N, D).astype(np.float32)).cuda()
    g1 = actor.backward(obs, dl, dn, want_obs=True)
    g2 = actor.backward(obs, dl, dn, want_obs=True)
    for k in g1['weights']:
        assert torch.equal(g1['weights'][k], g2['weights'][k]), k
    assert torch.equal(g1['obs'], g2['obs'])
    for sfx in ('', '_reverse'):
        assert torch.equal(g1['weights']['bilstm.bias_ih_l0' + sfx], g1['weights']['bilstm.bias_hh_l0' + sfx])
    perm = torch.from_numpy(rng.permutation(B)).cuda()
    gp = actor.backward(obs[perm], dl[perm], dn[perm], want_obs=True, want_weights=False)
    assert torch.equal(gp['obs'], g1['obs'][perm]) and gp['weights'] == {}
    for s0 in (0, 1, 1183, B - 5):
        for b in (1, 2, 5):
            sl = slice(s0, s0 + b)
            gs = actor.backward(obs[sl], dl[sl], dn[sl], want_obs=True, want_weights=False)
            assert torch.equal(gs['obs'], g1['obs'][sl]), (s0, b)
    # side stream, ordered after the load on the current stream
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        gside = actor.backward(obs, dl, dn, want_obs=True)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(gside['obs'], g1['obs'])
    for k in g1['weights']:
        assert torch.equal(gside['weights'][k], g1['weights'][k]), k
    # raw ABI: a NaN-filled workspace reused, NaN sentinels past row B, outputs passed as NULL not computed
    Bs = 37
    st = _lib.current_stream(actor.device)
    nbytes = actor._lib.actor_backward_workspace(actor._h, B, N)
    ws = torch.full((nbytes // 4,), float('nan'), device='cuda')
    dobs = torch.full((Bs + pad, N, D), float('nan'), device='cuda')
    w2b = torch.full((heads[1], 64), float('nan'), device='cuda')
    w3 = torch.full((D, 64), float('nan'), device='cuda')
    g = _lib.ActorGrads(dense2b_w=w2b.data_ptr(), dense3_w=w3.data_ptr())
    for _ in range(2):
        _lib.check(actor._lib.actor_backward(actor._h, _lib.ptr(obs), Bs, N, _lib.ptr(dl), _lib.ptr(dn), _lib.ptr(dobs),
                                             C.byref(g), _lib.ptr(ws), nbytes, st), 'actor_backward')
    ref = actor.backward(obs[:Bs], dl[:Bs], dn[:Bs], want_obs=True)
    assert torch.equal(dobs[:Bs], ref['obs']) and bool(torch.isnan(dobs[Bs:]).all())
    assert torch.equal(w2b, ref['weights']['dense2_2.module.weight'])
    assert torch.equal(w3, ref['weights']['dense3.module.weight'])
    # CUDA graph replay of the whole call
    gr = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(gr):
        gg = actor.backward(obs, dl, dn, want_obs=True)
    gr.replay()
    torch.cuda.synchronize()
    assert torch.equal(gg['obs'], g1['obs'])
    for k in g1['weights']:
        assert torch.equal(gg['weights'][k], g1['weights'][k]), k
    # refusals: a workspace one byte short, B = 0, N = 13, a host pointer
    small = actor._lib.actor_backward_workspace(actor._h, Bs, N)
    assert actor._lib.actor_backward(actor._h, _lib.ptr(obs), Bs, N, _lib.ptr(dl), None, None, None, _lib.ptr(ws),
                                     small - 1, st) == _lib.MPE_EINVAL
    assert actor._lib.actor_backward_workspace(actor._h, 0, N) == 0
    assert actor._lib.actor_backward(actor._h, _lib.ptr(obs), 0, N, _lib.ptr(dl), None, None, None, _lib.ptr(ws), 0,
                                     st) == _lib.MPE_OK
    assert actor._lib.actor_backward_workspace(actor._h, Bs, 13) == _lib.MPE_EUNSUPPORTED
    assert actor._lib.actor_backward(actor._h, _lib.ptr(obs), Bs, 13, _lib.ptr(dl), None, None, None, _lib.ptr(ws),
                                     nbytes, st) == _lib.MPE_EUNSUPPORTED
    host = torch.zeros(Bs, N, D)
    assert actor._lib.actor_backward(actor._h, _lib.ptr(host), Bs, N, _lib.ptr(dl), None, None, None, _lib.ptr(ws),
                                     nbytes, st) == _lib.MPE_EINVAL
    # dnext_state / dense3 gradients without a model head, dense2_2 gradients on a single-head actor
    single = _fused(_sharp_actor(24, D, 5, False))
    dl5 = dl[..., :5].contiguous()
    assert single._lib.actor_backward(single._h, _lib.ptr(obs), Bs, N, _lib.ptr(dl5), _lib.ptr(dn), None, None,
                                      _lib.ptr(ws), nbytes, st) == _lib.MPE_EINVAL
    for field in ('dense3_w', 'dense2b_w'):
        gbad = _lib.ActorGrads(**{field: w3.data_ptr()})
        assert single._lib.actor_backward(single._h, _lib.ptr(obs), Bs, N, _lib.ptr(dl5), None, None, C.byref(gbad),
                                          _lib.ptr(ws), nbytes, st) == _lib.MPE_EINVAL
    with pytest.raises(ValueError, match='dnext_state'):
        single.backward(obs, dl5, dn)


@pytest.mark.parametrize('N,D,heads,weights', [(1, 64, 5, 'default'), (2, 64, [5, 10], 'sharp'), (7, 64, 5, 'sharp'),
                                               (3, 16, [5, 10], 'default'), (12, 28, 5, 'sharp')])
def test_backward_differentiates_the_forward_relu_masks(N, D, heads, weights):
    """A dlogits one-hot in a single (agent row, entry) of a one-sample batch gives, through that entry's row of the
    heads' weight gradient, the backward's recomputed relu(hcat) of that row.  A "+model" actor whose dense3 selects D
    consecutive units of hcat with zero bias exposes the FFMA forward's relu(hcat) as next_state, window by window:
    the two are the same bits.  (The FFMA forward stages a tile of observations next to the weights, so it does not
    run every (N, D); these shapes are ones it runs.)"""
    sd = (_sharp_actor if weights == 'sharp' else _default_actor)(31 + N, D, heads, True)
    sd['dense3.module.bias'] = np.zeros(D, np.float32)
    actor = _fused(sd)
    rng = np.random.RandomState(N)
    obs = torch.from_numpy(rng.uniform(-2, 2, (1, N, D)).astype(np.float32)).cuda()
    hcat = torch.empty(N, 64, device='cuda')
    for off in sorted({min(o, 64 - D) for o in range(0, 64, D)}):
        sd['dense3.module.weight'] = np.eye(D, 64, off, dtype=np.float32)
        actor.load_state_dict(sd)
        hcat[:, off:off + D] = actor.forward(obs, want_next_state=True)['next_state'][0]
    A, A0 = _width(heads), heads[0] if isinstance(heads, list) else heads
    seen = 0
    for t in range(N):
        for a in sorted({0, A - 1, int(rng.randint(A))}):
            dl = torch.zeros(1, N, A, device='cuda')
            dl[0, t, a] = 1.0
            w = actor.backward(obs, dl)['weights']
            row = w['dense2.module.weight'][a] if not isinstance(heads, list) else \
                (w['dense2_1.module.weight'][a] if a < A0 else w['dense2_2.module.weight'][a - A0])
            assert torch.equal(row, hcat[t]), (t, a)
        seen += int((hcat[t] == 0).sum())
    print('relu(hcat) entries at zero: %d of %d' % (seen, N * 64))


# The critic backward of the parent commit on a fixed case: sha256 of every output's bytes.  The reductions moved
# into grad_reduce.cu unchanged, so these must not move.
_CRITIC_BITS = {
    'action': '4defe0e6a1f28a4a0a3d2c0370f32165fec0e1d3f9e904d1757c106b028e1d4b',
    'dense1.module.bias': '8fb9477a341d66fbf7267e0fc4721b9de7fb86f68a8f98f9e0c7590f116c0abf',
    'dense1.module.weight': 'a40dd7e75b145eb5826e8d83fb3489550b3fec061cdc7e15aa743ab435a8c664',
    'dense2.bias': 'ee55e431d4ca262aa39500c420fead30d8fec5e409f530048c9eb6ae2aaadba5',
    'dense2.weight': 'ae9a75a72a6e0e2311faba4711885ed5da13f29eff5c2f45f511140f2ec3f3cf',
    'lstm.bias_hh_l0': '1800ef36dd6852019fef40f2a780760179ddcef1bb22c57be07324fe54af07fb',
    'lstm.bias_ih_l0': '1800ef36dd6852019fef40f2a780760179ddcef1bb22c57be07324fe54af07fb',
    'lstm.weight_hh_l0': 'e7a7459771d46cd82a3fdbbf5a8f7ab38e74f8b29ef04572fb8cd803bb4dce62',
    'lstm.weight_ih_l0': '24bf0e23de1272260f4fed5a46f3dea724b2f4b468e92696255dbb83443eec4c',
    'obs': 'c2a653dc01bac57527e1386ea42e8faf672395985df10848ebceb4c64a51057a',
}


def _critic_case():
    import multiagent_rl_b200 as m
    torch.manual_seed(21)
    sd = m.FusedCriticNetwork(15, 1).state_dict()
    rng = np.random.RandomState(22)
    B, N = 777, 3
    obs = torch.from_numpy(rng.uniform(-2, 2, (B, N, 10)).astype(np.float32)).cuda()
    act = torch.softmax(torch.from_numpy(rng.randn(B, N, 5).astype(np.float32)).cuda(), -1)
    dq = torch.from_numpy(rng.randn(B, 1).astype(np.float32)).cuda()
    g = m.FusedCritic(sd, obs_dim=10).backward(obs, act, dq, want_obs=True)
    out = {'obs': g['obs'], 'action': g['action']}
    out.update(g['weights'])
    return {k: hashlib.sha256(v.contiguous().cpu().numpy().tobytes()).hexdigest() for k, v in out.items()}


def test_critic_gradients_are_the_parent_commits_bits():
    assert _critic_case() == _CRITIC_BITS


def test_fused_actor_network_is_a_differentiable_drop_in():
    """state_dict round trip with networks.ActorNetwork, a forward bit-identical to FusedActor.forward (FFMA), and
    loss.backward() filling .grad and the obs gradient with the float64 parity, through the list-of-heads and the
    (policy, next_state) call forms; an output the loss does not use gets no gradient."""
    import multiagent_rl_b200 as m
    N, D, heads = 4, 18, [5, 10]
    torch.manual_seed(3)
    refnet = m.ActorNetwork(D, heads, model_head=True)
    net = m.FusedActorNetwork(D, heads, model_head=True).cuda()
    net.load_state_dict(refnet.state_dict())
    back = m.ActorNetwork(D, heads, model_head=True)
    back.load_state_dict({k: v.cpu() for k, v in net.state_dict().items()})
    assert all(torch.equal(back.state_dict()[k], refnet.state_dict()[k]) for k in refnet.state_dict())
    sd = {k: v.numpy() for k, v in refnet.state_dict().items()}
    rng = np.random.RandomState(4)
    obs_np = rng.uniform(-2, 2, (300, N, D)).astype(np.float32)
    obs_np = obs_np[at.kink_free(sd, obs_np)]
    obs = torch.from_numpy(obs_np).cuda().requires_grad_(True)
    (p0, p1), ns = net(obs)
    fa = _fused(sd).forward(obs.detach(), want_logits=True, want_next_state=True)
    assert torch.equal(torch.cat([p0, p1], -1), fa['logits']) and torch.equal(ns, fa['next_state'])
    B = obs.shape[0]
    dl = rng.randn(B, N, 15).astype(np.float32)
    dn = rng.randn(B, N, D).astype(np.float32)
    loss = (p0 * torch.from_numpy(dl[..., :5]).cuda()).sum() + (p1 * torch.from_numpy(dl[..., 5:]).cuda()).sum() + \
        (ns * torch.from_numpy(dn).cuda()).sum()
    loss.backward()
    want = at.grads(sd, obs_np, dl, dn)
    _check(obs.grad.cpu().numpy(), want['obs'], 1e-4, 'obs')
    for k, p in net.named_parameters():
        _check(p.grad.cpu().numpy(), want[k], 1e-4, k)
    net.zero_grad(set_to_none=True)
    (q0, q1), _ = net(obs.detach())
    (q0.sum() + q1.sum()).backward()
    assert net.dense3.module.weight.grad is None and net.dense3.module.bias.grad is None
    want = at.grads(sd, obs_np, np.ones((B, N, 15)), None)
    _check(net.dense2_1.module.weight.grad.cpu().numpy(), want['dense2_1.module.weight'], 1e-4, 'dense2_1 (policy only)')
    net.zero_grad(set_to_none=True)
    net(obs.detach())[1].sum().backward()
    assert net.dense2_1.module.weight.grad is None and net.dense3.module.weight.grad is not None


def test_fused_actor_network_module_behaviour():
    """A soft update through .data is seen by the next forward; deepcopy gives an independent module with its own
    handle; torch.no_grad works; CPU / float64 parameters and 13 agents are refused; FusedActingMixin acts with it."""
    import multiagent_rl_b200 as m
    torch.manual_seed(1)
    net = m.FusedActorNetwork(10, 5).cuda()
    rng = np.random.RandomState(2)
    obs = torch.from_numpy(rng.uniform(-1, 1, (64, 3, 10)).astype(np.float32)).cuda()
    with torch.no_grad():
        l0 = net(obs)
    assert not l0.requires_grad
    tgt = copy.deepcopy(net)
    assert tgt._handle.actor is None and tgt._handle is not net._handle
    with torch.no_grad():
        assert torch.equal(tgt(obs), l0)
    assert tgt._handle.actor is not net._handle.actor
    tau = 0.5
    with torch.no_grad():
        for p in net.parameters():
            p.add_(0.05 * torch.randn_like(p))
    for tp, p in zip(tgt.parameters(), net.parameters()):
        tp.data.copy_(tp.data * (1.0 - tau) + p.data * tau)
    with torch.no_grad():
        l1 = tgt(obs)
        assert torch.equal(l1, _fused(tgt.state_dict()).forward(obs, want_logits=True)['logits'])
        assert not torch.equal(l1, l0)
    del tgt
    with pytest.raises(RuntimeError, match='CUDA'):
        m.FusedActorNetwork(10, 5)(obs.cpu())
    with pytest.raises(RuntimeError, match='float32'):
        copy.deepcopy(net).double()(obs)
    with pytest.raises(ValueError, match='12 agents'):
        net(torch.zeros(2, 13, 10, device='cuda'))
    trainer = m.ActingTrainer(net, action_type='Discrete', sample_seed=5)
    onehot = trainer.get_exploration_action(obs.cpu().numpy())
    assert onehot.shape == (64, 3, 5) and np.all(onehot.sum(-1) == 1)


def test_sgd_actor_training_through_a_fused_critic_matches_float64():
    """20 plain-SGD steps of the actor loss of Trainer.optimize() - -Q(obs, soft Gumbel sample of the logits with
    fixed noise) + 1e-3 * mean(logits^2) - through a fixed FusedCriticNetwork: FusedActorNetwork and the float64
    restatements end within 1e-5 (relative) of each other."""
    import multiagent_rl_b200 as m
    N, D, A, B, K, lr = 3, 10, 5, 1024, 20, 0.05
    torch.manual_seed(7)
    net = m.FusedActorNetwork(D, A).cuda()
    critic = m.FusedCriticNetwork(D + A, 1).cuda()
    for p in critic.parameters():
        p.requires_grad_(False)
    ref = at.Actor64({k: v.cpu() for k, v in net.state_dict().items()})
    crit64 = ct.Critic64({k: v.cpu() for k, v in critic.state_dict().items()})
    for p in crit64.parameters():
        p.requires_grad_(False)
    opt, opt64 = torch.optim.SGD(net.parameters(), lr=lr), torch.optim.SGD(ref.parameters(), lr=lr)
    rng = np.random.RandomState(8)
    for _ in range(K):
        obs = rng.uniform(-1.5, 1.5, (B, N, D)).astype(np.float32)
        u = rng.uniform(1e-6, 1 - 1e-6, (B, N, A))
        gum = -np.log(-np.log(u))
        for mod, q, o, dev, dt in ((net, critic, opt, 'cuda', torch.float32), (ref, crit64, opt64, 'cpu', torch.float64)):
            o.zero_grad()
            x = torch.from_numpy(obs).to(dev, dt)
            logits = mod(x) if mod is net else mod(x)[0]
            soft = torch.softmax(logits + torch.from_numpy(gum).to(dev, dt), -1)
            loss = -q(x, soft).mean() + 1e-3 * (logits ** 2).mean()
            loss.backward()
            o.step()
    sd64 = dict(ref.named_parameters())
    worst = 0.0
    for k, p in net.named_parameters():
        p64 = sd64[k].detach().numpy()
        worst = max(worst, float(np.abs(p.detach().cpu().numpy() - p64).max()) / max(1.0, float(np.abs(p64).max())))
    print('largest parameter difference after %d SGD steps: %.3g' % (K, worst))
    assert worst <= 1e-5


# ---- the reference executed (oracle/_ref, byte-compiled from the reference tree) ----
needs_ref = pytest.mark.skipif(not build_ref.available(), reason='oracle/_ref not built (python -m oracle.build_ref)')


def _ref_actor(model):
    build_ref.add_to_path()
    if model:
        from rls.model.ac_network_model_multi_gumbel import ActorNetwork
    else:
        from rls.model.ac_network_multi_gumbel import ActorNetwork
    return ActorNetwork


@needs_ref
@pytest.mark.parametrize('model', [False, True])
def test_reference_actor_gradients_and_initialisation(model):
    """Under one seed FusedActorNetwork and the reference ActorNetwork start bit-identical, and the reference's
    double-precision autograd has the restatement's gradients (1e-10)."""
    import multiagent_rl_b200 as m
    ActorNetwork = _ref_actor(model)
    torch.manual_seed(11)
    refnet = ActorNetwork(input_dim=10, out_dim=5)
    torch.manual_seed(11)
    net = m.FusedActorNetwork(10, 5, model_head=model)
    a, b = refnet.state_dict(), net.state_dict()
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)
    rng = np.random.RandomState(12)
    obs = rng.uniform(-1, 1, (32, 3, 10))
    dl, dn = rng.randn(32, 3, 5), (rng.randn(32, 3, 10) if model else None)
    refnet = refnet.double()
    o = torch.from_numpy(obs).requires_grad_(True)
    out = refnet.forward(o)
    loss = (out[0] * torch.from_numpy(dl)).sum() + (out[1] * torch.from_numpy(dn)).sum() if model else \
        (out * torch.from_numpy(dl)).sum()
    loss.backward()
    want = at.grads({k: v.detach() for k, v in refnet.state_dict().items()}, obs, dl, dn)
    assert np.abs(o.grad.numpy() - want['obs']).max() <= 1e-10
    for k, p in refnet.named_parameters():
        assert np.abs(p.grad.numpy() - want[k]).max() <= 1e-10, k


@needs_ref
def test_reference_optimize_trains_the_fused_actor():
    """examples/train_batched.train(..., fused_actor=True, fused_critic=True): the reference ddpg_gumbel_fix
    Trainer.optimize(), unchanged, trains FusedActorNetwork; its trained state_dict loaded into the reference
    ActorNetwork gives the same logits."""
    import importlib.util
    import os
    from tests.conftest import ROOT
    spec = importlib.util.spec_from_file_location('train_batched', os.path.join(ROOT, 'examples', 'train_batched.py'))
    tb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tb)
    import multiagent_rl_b200 as m
    torch.manual_seed(12345678)  # train()'s construction order: actor first
    w0 = m.FusedActorNetwork(10, 5).state_dict()
    returns, learner, _ = tb.train(num_envs=256, episodes=3, updates_per_episode=2, batch_size=256,
                                   log=lambda s: None, fused_actor=True, fused_critic=True)
    assert isinstance(learner.actor, m.FusedActorNetwork) and all(np.isfinite(returns))
    sd = learner.actor.state_dict()
    assert all(bool(torch.isfinite(v).all()) for v in sd.values())
    assert any(not torch.equal(sd[k].cpu(), w0[k]) for k in sd)
    s0 = learner.memory.sample_index(torch.arange(0, 512, device='cuda'))[0]
    refnet = _ref_actor(False)(input_dim=10, out_dim=5).cuda()
    refnet.load_state_dict(sd)
    with torch.no_grad():
        want, got = refnet.forward(s0), learner.actor(s0)
    assert float((got - want).abs().max()) <= 1e-4 * max(1.0, float(want.abs().max()))


@needs_ref
def test_reference_model_trainer_optimizes_the_fused_actor(ref):  # noqa: F811 - the fixture
    """main_scalability_1.py:30-65 with FusedActorNetwork(model_head=True) as the actor: experiments/run.py ``run``
    and model_ddpg_gumbel_fix.Trainer.optimize(), unchanged, train it at n = 6; the trained state_dict loaded into the
    reference "+model" ActorNetwork gives the same logits and next state."""
    import multiagent_rl_b200 as m
    from tests import _refloop
    scen, run_mod, arglist = ref
    from rls.agent.multiagent.model_ddpg_gumbel_fix import Trainer as RefTrainer
    env = scen.make_env('simple_spread', n=6, benchmark=False, discrete_action=True, local_observation=True)
    _, critic, action_type = _refloop.main_py_setup(env, 12345678, model=True)
    D = env.observation_space[0].shape[0]
    torch.manual_seed(5)
    fused = m.FusedActorNetwork(D, 5, model_head=True)
    w0 = {k: v.clone() for k, v in fused.state_dict().items()}
    arglist.num_episodes, arglist.warmup_steps, arglist.batch_size, arglist.update_rate = 2, 30, 16, 20
    keep = []
    run_mod.run(env, fused, critic, _trainer_class(RefTrainer, True, keep), 'simple_spread_n_agent_6_', action_type,
                cnt=0)
    assert keep[0].actor is fused
    sd = fused.state_dict()
    assert all(bool(torch.isfinite(v).all()) for v in sd.values())
    assert any(not torch.equal(sd[k].cpu(), w0[k]) for k in sd)
    refnet = _ref_actor(True)(input_dim=D, out_dim=5).cuda()
    refnet.load_state_dict(sd)
    obs = torch.from_numpy(np.random.RandomState(9).uniform(-1, 1, (64, 6, D)).astype(np.float32)).cuda()
    with torch.no_grad():
        (p_ref, n_ref), (p, n) = refnet.forward(obs), fused(obs)
    assert float((p - p_ref).abs().max()) <= 1e-4 * max(1.0, float(p_ref.abs().max()))
    assert float((n - n_ref).abs().max()) <= 1e-4 * max(1.0, float(n_ref.abs().max()))
