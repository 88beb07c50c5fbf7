"""GPU tests of the critic backward (C ABI critic_backward, FusedCritic.backward, FusedCriticNetwork) against float64
autograd of the torch restatement tests/_critic_torch.py (itself pinned to the reference by
tests/test_critic_grad_oracle.py).

Tolerance per gradient tensor: max|g - g64| <= TOL * max(1, max|g64|), TOL = 1e-4 for default-init weights and 5e-4
for the "sharp" weights of tests/test_gpu_critic.py (saturating gates, peaked attention).  Samples with a float64 relu
pre-activation within 1e-5 of zero are dropped from the batch before either side runs (fp32 may sit on the other side
of the kink); the tests print how many."""
import copy
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import build_ref
from tests import _critic_torch as ct
from tests import _refloop
from tests.test_gpu_critic import _actions, _sharp_critic
from tests.test_gpu_reference_loop import _trainer_class, ref  # noqa: F401 - the reference-loop fixture

pytestmark = pytest.mark.gpu


def _default_critic(seed, D, A, model, out):
    import multiagent_rl_b200 as m
    torch.manual_seed(seed)
    return {k: v.numpy() for k, v in m.FusedCriticNetwork(D + A, out, model=model).state_dict().items()}


def _case(N, D, A, model, B, out, action, weights, seed):
    rng = np.random.RandomState(seed)
    sd = _sharp_critic(rng, D, A, model, out) if weights == 'sharp' else _default_critic(seed, D, A, model, out)
    obs = rng.uniform(-2, 2, (B, N, D)).astype(np.float32)
    act = _actions(rng, B, N, A, action)
    keep = ct.kink_free(sd, obs, act)
    print('dropped %d of %d samples within 1e-5 of a relu kink' % (B - int(keep.sum()), B))
    # the sharp weights saturate output gates, so with 64 inputs a quarter of the samples has an attention output unit
    # within 1e-5 of the relu's kink
    assert keep.sum() >= 0.7 * B
    return rng, sd, obs[keep], act[keep]


def _check(got, want, tol, what):
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(np.asarray(got, np.float64) - want).max())
    assert err <= tol * scale, (what, err, scale)


@pytest.mark.parametrize('N,D,A,model,B,out,action,weights,with_dr', [
    pytest.param(3, 10, 5, False, 4099, 1, 'onehot', 'sharp', False, id='n3-4099-sharp'),
    pytest.param(3, 10, 5, False, 1024, 1, 'softmax', 'default', False, id='n3-1024-default-soft'),
    pytest.param(6, 16, 5, True, 1025, 1, 'onehot', 'sharp', True, id='n6-model-1025-sharp'),
    pytest.param(12, 28, 5, True, 333, 1, 'onehot', 'default', True, id='n12-model-333'),
    pytest.param(2, 21, 15, False, 2048, 1, 'onehot', 'default', False, id='n2-din36-2048'),
    pytest.param(1, 6, 5, False, 7, 1, 'onehot', 'sharp', False, id='n1-7'),
    pytest.param(16, 36, 5, False, 65, 1, 'onehot', 'sharp', False, id='n16-65'),
    pytest.param(3, 10, 5, False, 1027, 2, 'softmax', 'default', False, id='out2-relu'),
    pytest.param(3, 10, 5, False, 1030, 4, 'uniform', 'sharp', False, id='out4-relu-uniform'),
    pytest.param(6, 16, 5, True, 515, 2, 'softmax', 'sharp', False, id='out2-model-dr-none'),
    pytest.param(12, 28, 5, True, 333, 4, 'onehot', 'sharp', True, id='out4-model'),
    pytest.param(3, 59, 5, False, 2051, 1, 'onehot', 'sharp', False, id='din64-relu'),
    pytest.param(2, 49, 15, True, 1001, 2, 'softmax', 'default', True, id='din64-model-out2'),
    pytest.param(16, 54, 10, True, 4741, 4, 'uniform', 'sharp', True, id='n16-din64-out4-multipass'),
    pytest.param(3, 10, 5, False, 65539, 1, 'onehot', 'default', False, id='b65539-ragged'),
])
def test_critic_backward_vs_float64_autograd(N, D, A, model, B, out, action, weights, with_dr):
    """Every weight gradient, dobs and daction: both critics, 1..16 agents, inputs up to 64 wide, 1..4 outputs,
    ragged batches from 7 to past one pass of every warp, one-hot / soft / uniform actions, dr given or None."""
    import multiagent_rl_b200 as m
    rng, sd, obs, act = _case(N, D, A, model, B, out, action, weights, N * 1000 + D + B)
    B = obs.shape[0]
    dq = rng.randn(B, out).astype(np.float32)
    dr = rng.randn(B, out).astype(np.float32) if with_dr else None
    want = ct.grads(sd, obs, act, dq, dr)
    critic = m.FusedCritic(sd, obs_dim=D)
    got = critic.backward(torch.from_numpy(obs), torch.from_numpy(act), torch.from_numpy(dq),
                          None if dr is None else torch.from_numpy(dr), want_obs=True)
    tol = 5e-4 if weights == 'sharp' else 1e-4
    _check(got['obs'].cpu().numpy(), want['obs'], tol, 'obs')
    _check(got['action'].cpu().numpy(), want['action'], tol, 'action')
    assert sorted(got['weights']) == sorted(ct.KEYS + (ct.KEYS3 if model else []))
    for k, v in got['weights'].items():
        _check(v.cpu().numpy(), want[k], tol, k)
    assert torch.equal(got['weights']['lstm.bias_ih_l0'], got['weights']['lstm.bias_hh_l0'])


@pytest.mark.parametrize('model', [False, True])
def test_critic_backward_is_bitwise_reproducible_and_position_independent(model):
    """Weight gradients are the same bits on every call; a sample's dobs / daction are the same bits under
    permutation and slicing of the batch; nothing is written past row B or into outputs that were not asked for."""
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    N, D, A, B, out, pad = 3, 10, 5, 5003, 2, 16
    rng = np.random.RandomState(23 + model)
    critic = m.FusedCritic(_sharp_critic(rng, D, A, model, out), obs_dim=D)
    obs = torch.from_numpy(rng.uniform(-2, 2, (B, N, D)).astype(np.float32)).cuda()
    act = torch.from_numpy(_actions(rng, B, N, A, 'softmax')).cuda()
    dq = torch.from_numpy(rng.randn(B, out).astype(np.float32)).cuda()
    dr = torch.from_numpy(rng.randn(B, out).astype(np.float32)).cuda() if model else None
    g1 = critic.backward(obs, act, dq, dr, want_obs=True)
    g2 = critic.backward(obs, act, dq, dr, want_obs=True)
    for k in g1['weights']:
        assert torch.equal(g1['weights'][k], g2['weights'][k]), k
    assert torch.equal(g1['obs'], g2['obs']) and torch.equal(g1['action'], g2['action'])
    perm = torch.from_numpy(rng.permutation(B)).cuda()
    gp = critic.backward(obs[perm], act[perm], dq[perm], None if dr is None else dr[perm], want_obs=True,
                         want_weights=False)
    assert torch.equal(gp['obs'], g1['obs'][perm]) and torch.equal(gp['action'], g1['action'][perm])
    assert gp['weights'] == {}
    for s0 in (0, 1, 4093, B - 5):
        for b in (1, 2, 5):
            sl = slice(s0, s0 + b)
            gs = critic.backward(obs[sl], act[sl], dq[sl], None if dr is None else dr[sl], want_obs=True)
            assert torch.equal(gs['obs'], g1['obs'][sl]) and torch.equal(gs['action'], g1['action'][sl]), (s0, b)
    # raw ABI: NaN sentinels past row B stay, and an output passed as NULL is not computed
    Bs = 37
    dobs = torch.full((Bs + pad, N, D), float('nan'), device='cuda')
    dact = torch.full((Bs + pad, N, A), float('nan'), device='cuda')
    w2 = torch.full((out, 64), float('nan'), device='cuda')
    g = _lib.CriticGrads(dense2_w=w2.data_ptr())
    nbytes = critic._lib.critic_backward_workspace(critic._h, Bs, N)
    ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    st = _lib.current_stream(critic.device)
    _lib.check(critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), Bs, N, _lib.ptr(dq), _lib.ptr(dr),
                                           _lib.ptr(dobs), None, C.byref(g), _lib.ptr(ws), nbytes, st), 'critic_backward')
    ref = critic.backward(obs[:Bs], act[:Bs], dq[:Bs], None if dr is None else dr[:Bs], want_obs=True)
    assert torch.equal(dobs[:Bs], ref['obs']) and bool(torch.isnan(dobs[Bs:]).all())
    assert bool(torch.isnan(dact).all())  # daction was not requested
    assert torch.equal(w2, ref['weights']['dense2.weight'])
    # a workspace one byte short, dr on a critic without a reward head, B = 0
    assert critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), Bs, N, _lib.ptr(dq), None, None, None,
                                       None, _lib.ptr(ws), nbytes - 1, st) == _lib.MPE_EINVAL
    if not model:
        assert critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), Bs, N, _lib.ptr(dq), _lib.ptr(dq),
                                           None, None, None, _lib.ptr(ws), nbytes, st) == _lib.MPE_EINVAL
    assert critic._lib.critic_backward_workspace(critic._h, 0, N) == 0
    assert critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), 0, N, _lib.ptr(dq), None, None, None,
                                       None, _lib.ptr(ws), 0, st) == _lib.MPE_OK
    assert critic._lib.critic_backward_workspace(critic._h, Bs, 17) == _lib.MPE_EUNSUPPORTED
    host = torch.zeros(Bs, N, D)
    assert critic._lib.critic_backward(critic._h, _lib.ptr(host), _lib.ptr(act), Bs, N, _lib.ptr(dq), None, None, None,
                                       None, _lib.ptr(ws), nbytes, st) == _lib.MPE_EINVAL


def _golden(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, 'critic_%s.npz' % tag))
    return g, {k[3:]: g[k] for k in g.files if k.startswith('sd/')}


@pytest.mark.parametrize('tag,D', [('spread_n3', 10), ('reference', 21), ('model_n12', 28)])
def test_fused_critic_network_is_a_differentiable_drop_in(golden_dir, tag, D):
    """state_dict keys / shapes of the reference, a forward bit-identical to FusedCritic.forward, and loss.backward()
    filling .grad (and obs / action gradients, through the list-of-heads call form) with the float64 parity."""
    import multiagent_rl_b200 as m
    g, sd = _golden(golden_dir, tag)
    model = 'r' in g.files
    net = m.FusedCriticNetwork(sd['dense1.module.weight'].shape[1], 1, model=model).cuda()
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: v.shape for k, v in sd.items()}
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    keep = ct.kink_free(sd, g['obs'], g['action'])
    obs_np, act_np = g['obs'][keep], g['action'][keep]
    obs = torch.from_numpy(obs_np).cuda().requires_grad_(True)
    act = torch.from_numpy(act_np).cuda().requires_grad_(True)
    heads = [act[..., :5], act[..., 5:]] if tag == 'reference' else act
    res = net(obs, heads)
    fc = m.FusedCritic(sd, obs_dim=D).forward(obs.detach(), act.detach())
    B = obs.shape[0]
    rng = np.random.RandomState(5)
    dq = rng.randn(B, 1).astype(np.float32)
    dr = rng.randn(B, 1).astype(np.float32) if model else None
    if model:
        assert torch.equal(res[0], fc[0]) and torch.equal(res[1], fc[1])
        loss = (res[0] * torch.from_numpy(dq).cuda()).sum() + (res[1] * torch.from_numpy(dr).cuda()).sum()
    else:
        assert torch.equal(res, fc)
        loss = (res * torch.from_numpy(dq).cuda()).sum()
    loss.backward()
    want = ct.grads(sd, obs_np, act_np, dq, dr)
    _check(obs.grad.cpu().numpy(), want['obs'], 1e-4, 'obs')
    _check(act.grad.cpu().numpy(), want['action'], 1e-4, 'action')
    for k, p in net.named_parameters():
        _check(p.grad.cpu().numpy(), want[k], 1e-4, k)
    # only q in the loss of the model critic: dr is None inside the backward
    if model:
        net.zero_grad()
        net(obs.detach(), act.detach())[0].sum().backward()
        want = ct.grads(sd, obs_np, act_np, np.ones((B, 1)), None)
        assert net.dense3.weight.grad is None and net.dense3.bias.grad is None  # as autograd leaves an unused head
        _check(net.dense2.weight.grad.cpu().numpy(), want['dense2.weight'], 1e-4, 'dense2 (q only)')


def test_fused_critic_network_module_behaviour():
    """A soft update through .data is seen by the next forward; deepcopy gives an independent module with its own
    handle; torch.no_grad works; CPU / float64 parameters, 17 agents and an input 65 wide are refused."""
    import multiagent_rl_b200 as m
    torch.manual_seed(1)
    net = m.FusedCriticNetwork(15, 1).cuda()
    rng = np.random.RandomState(2)
    obs = torch.from_numpy(rng.uniform(-1, 1, (64, 3, 10)).astype(np.float32)).cuda()
    act = torch.from_numpy(_actions(rng, 64, 3, 5, 'onehot')).cuda()
    with torch.no_grad():
        q0 = net(obs, act)
    assert not q0.requires_grad
    tgt = copy.deepcopy(net)
    assert tgt._handle.critic is None and tgt._handle is not net._handle
    with torch.no_grad():
        assert torch.equal(tgt(obs, act), q0)
    assert tgt._handle.critic is not net._handle.critic
    # DDPG soft update (ddpg_gumbel_fix.py:212-213 soft_update): writes through .data do not bump _version
    tau = 0.5
    with torch.no_grad():
        for p in net.parameters():
            p.add_(0.05 * torch.randn_like(p))
    for tp, p in zip(tgt.parameters(), net.parameters()):
        tp.data.copy_(tp.data * (1.0 - tau) + p.data * tau)
    with torch.no_grad():
        q1 = tgt(obs, act)
        want = m.FusedCritic(tgt.state_dict(), obs_dim=10).forward(obs, act)
        assert torch.equal(q1, want) and not torch.equal(q1, q0)
        assert torch.equal(net(obs, act), m.FusedCritic(net.state_dict(), obs_dim=10).forward(obs, act))
    del tgt
    with torch.no_grad():
        net(obs, act)
    with pytest.raises(RuntimeError, match='CUDA'):
        m.FusedCriticNetwork(15, 1)(obs.cpu(), act.cpu())
    with pytest.raises(RuntimeError, match='float32'):
        copy.deepcopy(net).double()(obs, act)
    with pytest.raises(ValueError, match='16 agents'):
        net(torch.zeros(2, 17, 10, device='cuda'), torch.zeros(2, 17, 5, device='cuda'))
    with pytest.raises(ValueError, match='64'):
        m.FusedCriticNetwork(65, 1)


@pytest.mark.parametrize('model', [False, True])
def test_sgd_training_matches_float64(model):
    """20 plain-SGD steps on a SmoothL1 TD loss from the same initial weights and batches: FusedCriticNetwork and the
    float64 restatement end with the same parameters (SGD rather than Adam: Adam's first steps turn the sign of
    near-zero gradients into full-size updates)."""
    import multiagent_rl_b200 as m
    N, D, A, B, K, lr = 3, 10, 5, 1024, 20, 0.05
    torch.manual_seed(7)
    net = m.FusedCriticNetwork(D + A, 1, model=model).cuda()
    ref = ct.Critic64({k: v.cpu() for k, v in net.state_dict().items()})
    opt, opt64 = torch.optim.SGD(net.parameters(), lr=lr), torch.optim.SGD(ref.parameters(), lr=lr)
    rng = np.random.RandomState(8)
    for _ in range(K):
        obs = rng.uniform(-1.5, 1.5, (B, N, D)).astype(np.float32)
        act = _actions(rng, B, N, A, 'softmax')
        y = rng.randn(B, 1).astype(np.float32)
        for mod, o, dev, dt in ((net, opt, 'cuda', torch.float32), (ref, opt64, 'cpu', torch.float64)):
            o.zero_grad()
            out = mod(torch.from_numpy(obs).to(dev, dt), torch.from_numpy(act).to(dev, dt))
            q = out[0] if model else out
            loss = torch.nn.functional.smooth_l1_loss(q, torch.from_numpy(y).to(dev, dt))
            if model:
                loss = loss + out[1].abs().mean()
            loss.backward()
            o.step()
    sd64 = dict(ref.named_parameters())
    worst = 0.0
    for k, p in net.named_parameters():
        p64 = sd64[k].detach().numpy()
        err = float(np.abs(p.detach().cpu().numpy() - p64).max()) / max(1.0, float(np.abs(p64).max()))
        worst = max(worst, err)
    print('largest parameter difference after %d SGD steps: %.3g' % (K, worst))
    assert worst <= 1e-5


# ---- the reference executed (oracle/_ref, byte-compiled from the reference tree) ----
needs_ref = pytest.mark.skipif(not build_ref.available(), reason='oracle/_ref not built (python -m oracle.build_ref)')


def _ref_classes(model):
    build_ref.add_to_path()
    if model:
        from rls.model.ac_network_model_multi_gumbel import CriticNetwork
    else:
        from rls.model.ac_network_multi_gumbel import CriticNetwork
    return CriticNetwork


@needs_ref
@pytest.mark.parametrize('model', [False, True])
def test_reference_critic_gradients_and_initialisation(model):
    """The reference CriticNetwork(...).double() has the restatement's gradients (1e-10), and under one seed
    FusedCriticNetwork(input_dim, out_dim) and the reference CriticNetwork(input_dim, out_dim) start bit-identical."""
    import multiagent_rl_b200 as m
    CriticNetwork = _ref_classes(model)
    torch.manual_seed(11)
    refnet = CriticNetwork(input_dim=15, out_dim=1)
    torch.manual_seed(11)
    net = m.FusedCriticNetwork(15, 1, model=model)
    a, b = refnet.state_dict(), net.state_dict()
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)
    rng = np.random.RandomState(12)
    obs, act = rng.uniform(-1, 1, (32, 3, 10)), _actions(rng, 32, 3, 5, 'softmax').astype(np.float64)
    dq, dr = rng.randn(32, 1), (rng.randn(32, 1) if model else None)
    refnet = refnet.double()
    o, ac = torch.from_numpy(obs).requires_grad_(True), torch.from_numpy(act).requires_grad_(True)
    out = refnet.forward(o, ac)
    loss = (out[0] * torch.from_numpy(dq)).sum() + (out[1] * torch.from_numpy(dr)).sum() if model else \
        (out * torch.from_numpy(dq)).sum()
    loss.backward()
    want = ct.grads({k: v.detach() for k, v in refnet.state_dict().items()}, obs, act, dq, dr)
    assert np.abs(o.grad.numpy() - want['obs']).max() <= 1e-10
    assert np.abs(ac.grad.numpy() - want['action']).max() <= 1e-10
    for k, p in refnet.named_parameters():
        assert np.abs(p.grad.numpy() - want[k]).max() <= 1e-10, k


@needs_ref
def test_reference_optimize_trains_the_fused_critic():
    """examples/train_batched.train(..., fused_critic=True): the reference ddpg_gumbel_fix Trainer.optimize(),
    unchanged, over the device replay with FusedCriticNetwork as its critic.  The critic moved, stays finite, and its
    trained state_dict loaded into the reference CriticNetwork gives the same Q."""
    import importlib.util
    from tests.conftest import ROOT
    spec = importlib.util.spec_from_file_location('train_batched', os.path.join(ROOT, 'examples', 'train_batched.py'))
    tb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tb)
    import multiagent_rl_b200 as m
    build_ref.add_to_path()
    from rls.model.ac_network_multi_gumbel import ActorNetwork
    torch.manual_seed(12345678)  # train()'s construction order: actor, then critic
    ActorNetwork(input_dim=10, out_dim=5)
    w0 = m.FusedCriticNetwork(15, 1).state_dict()
    returns, learner, _ = tb.train(num_envs=256, episodes=3, updates_per_episode=2, batch_size=256,
                                   log=lambda s: None, fused_critic=True)
    assert isinstance(learner.critic, m.FusedCriticNetwork) and all(np.isfinite(returns))
    sd = learner.critic.state_dict()
    assert all(bool(torch.isfinite(v).all()) for v in sd.values())
    assert any(not torch.equal(sd[k].cpu(), w0[k]) for k in sd)
    s0, a0, _, _, _ = learner.memory.sample_index(torch.arange(0, 512, device='cuda'))
    refnet = _ref_classes(False)(input_dim=15, out_dim=1).cuda()
    refnet.load_state_dict(sd)
    with torch.no_grad():
        q_ref = refnet.forward(s0, a0)
        q = learner.critic(s0, a0)
    assert float((q - q_ref).abs().max()) <= 1e-4 * max(1.0, float(q_ref.abs().max()))


@needs_ref
def test_reference_model_trainer_optimizes_the_fused_critic(ref):
    """main_scalability_1.py:30-65 with FusedCriticNetwork(model=True) as the critic: experiments/run.py ``run`` and
    model_ddpg_gumbel_fix.Trainer.optimize(), unchanged, train it; the trained state_dict loaded into the reference
    "+model" CriticNetwork gives the same Q and r."""
    import multiagent_rl_b200 as m
    scen, run_mod, arglist = ref
    from rls.agent.multiagent.model_ddpg_gumbel_fix import Trainer as RefTrainer
    env = scen.make_env('simple_spread', n=6, benchmark=False, discrete_action=True, local_observation=True)
    actor, critic, action_type = _refloop.main_py_setup(env, 12345678, model=True)
    din = critic.dense1.module.in_features
    torch.manual_seed(5)
    fused = m.FusedCriticNetwork(din, 1, model=True)
    w0 = {k: v.clone() for k, v in fused.state_dict().items()}
    arglist.num_episodes, arglist.warmup_steps, arglist.batch_size, arglist.update_rate = 2, 30, 16, 20
    keep = []
    run_mod.run(env, actor, fused, _trainer_class(RefTrainer, True, keep), 'simple_spread_n_agent_6_', action_type,
                cnt=0)
    learner = keep[0]
    assert learner.critic is fused
    sd = fused.state_dict()
    assert all(bool(torch.isfinite(v).all()) for v in sd.values())
    assert any(not torch.equal(sd[k].cpu(), w0[k]) for k in sd)
    refnet = _ref_classes(True)(input_dim=din, out_dim=1).cuda()
    refnet.load_state_dict(sd)
    rng = np.random.RandomState(9)
    D = env.observation_space[0].shape[0]
    obs = torch.from_numpy(rng.uniform(-1, 1, (64, 6, D)).astype(np.float32)).cuda()
    act = torch.from_numpy(_actions(rng, 64, 6, din - D, 'softmax')).cuda()
    with torch.no_grad():
        q_ref, r_ref = refnet.forward(obs, act)
        q, r = fused(obs, act)
    assert float((q - q_ref).abs().max()) <= 1e-4 * max(1.0, float(q_ref.abs().max()))
    assert float((r - r_ref).abs().max()) <= 1e-4 * max(1.0, float(r_ref.abs().max()))
