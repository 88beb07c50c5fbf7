"""CPU checks behind the actor backward's GPU tests: the float64 torch restatement (tests/_actor_torch.py) is the
reference actor - it equals oracle/actor_ref.py, which tests/test_oracle.py pins to the reference's own outputs -
and its autograd gradients are the derivatives of that function (central finite differences).  Also: the new ABI
entry points refuse bad arguments without a GPU, and FusedActorNetwork builds the reference's parameters."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import actor_ref
from tests import _actor_torch as at

TAGS = ['spread_n3', 'reference', 'model_n6', 'spread_n12']


def _golden(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, 'actor_%s.npz' % tag))
    return g, {k[3:]: g[k] for k in g.files if k.startswith('sd/')}


@pytest.mark.parametrize('tag', TAGS)
def test_torch_restatement_equals_the_numpy_oracle(golden_dir, tag):
    g, sd = _golden(golden_dir, tag)
    want = actor_ref.forward(sd, g['obs'])
    A = sum(w.shape[-1] for w in want['logits'])
    obs = g['obs'].astype(np.float32)  # actor_ref.forward casts obs to float32 (process_obs)
    got = at.grads(sd, obs, np.ones(obs.shape[:2] + (A,)),
                   np.ones_like(g['obs']) if 'next_state' in want else None)
    assert np.abs(got['logits'] - np.concatenate(want['logits'], -1)).max() <= 1e-12
    if 'next_state' in want:
        assert np.abs(got['next_state'] - want['next_state']).max() <= 1e-12


def _loss(sd, obs, dl, dn):
    """sum(logits * dl) (+ sum(next_state * dn)) of the float64 numpy forward, with float64 inputs throughout
    (actor_ref.forward casts obs to float32 first)."""
    p = {k: np.asarray(v, np.float64) for k, v in sd.items()}
    h1 = np.maximum(obs @ p['dense1.module.weight'].T + p['dense1.module.bias'], 0.0)
    B, N, _ = obs.shape
    sig = lambda z: 1.0 / (1.0 + np.exp(-z))  # noqa: E731
    outs = []
    for sfx, order in (('', range(N)), ('_reverse', range(N - 1, -1, -1))):
        h, c, out = np.zeros((B, 32)), np.zeros((B, 32)), np.zeros((B, N, 32))
        for t in order:
            gg = (h1[:, t] @ p['bilstm.weight_ih_l0' + sfx].T + p['bilstm.bias_ih_l0' + sfx]
                  + h @ p['bilstm.weight_hh_l0' + sfx].T + p['bilstm.bias_hh_l0' + sfx])
            c = sig(gg[:, 32:64]) * c + sig(gg[:, :32]) * np.tanh(gg[:, 64:96])
            h = sig(gg[:, 96:]) * np.tanh(c)
            out[:, t] = h
        outs.append(out)
    hid = np.maximum(np.concatenate(outs, -1), 0.0)
    if 'dense2.module.weight' in p:
        logits = hid @ p['dense2.module.weight'].T + p['dense2.module.bias']
    else:
        logits = np.concatenate([hid @ p['dense2_1.module.weight'].T + p['dense2_1.module.bias'],
                                 hid @ p['dense2_2.module.weight'].T + p['dense2_2.module.bias']], -1)
    total = float((logits * dl).sum())
    if dn is not None:
        total += float(((hid @ p['dense3.module.weight'].T + p['dense3.module.bias']) * dn).sum())
    return total


@pytest.mark.parametrize('tag', TAGS)
def test_autograd_gradients_match_finite_differences(golden_dir, tag):
    """Central differences of the numpy forward (float64, step 1e-6) at sampled coordinates of every weight tensor
    and of obs, for the loss sum(logits * dlogits) (+ sum(next_state * dnext_state))."""
    g, sd = _golden(golden_dir, tag)
    rng = np.random.RandomState(3)
    B = 5
    obs = g['obs'][:B].astype(np.float64)
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    A = sum(v.shape[0] for k, v in sd.items() if k.startswith('dense2') and k.endswith('weight'))
    dl = rng.randn(B, obs.shape[1], A)
    dn = rng.randn(*obs.shape) if 'dense3.module.weight' in sd else None
    got = at.grads(sd64, obs, dl, dn)
    want_loss = float((got['logits'] * dl).sum() + (0 if dn is None else (got['next_state'] * dn).sum()))
    assert abs(_loss(sd64, obs, dl, dn) - want_loss) < 1e-10
    eps = 1e-6
    for name in list(sd64) + ['obs']:
        base = obs if name == 'obs' else sd64[name]
        for flat in rng.choice(base.size, size=min(5, base.size), replace=False):
            idx = np.unravel_index(flat, base.shape)
            vals = []
            for sgn in (1, -1):
                pert = base.copy()
                pert[idx] += sgn * eps
                vals.append(_loss(sd64, pert, dl, dn) if name == 'obs' else _loss(dict(sd64, **{name: pert}), obs, dl, dn))
            fd = (vals[0] - vals[1]) / (2 * eps)
            assert abs(fd - got[name][idx]) <= 1e-6 * max(1.0, abs(fd)), (name, idx, fd, got[name][idx])


@pytest.mark.parametrize('out_dim,model_head', [(5, False), ([5, 10], False), (5, True), ([3, 4], True)])
def test_fused_actor_network_initialises_like_the_package_actor(out_dim, model_head):
    """networks.ActorNetwork and FusedActorNetwork under one seed: same keys in the same order, same shapes, same
    bits (the reference class itself is compared where it is importable, in tests/test_gpu_actor_grad.py)."""
    import multiagent_rl_b200 as m
    torch.manual_seed(17)
    a = m.ActorNetwork(16, out_dim, model_head=model_head).state_dict()
    torch.manual_seed(17)
    b = m.FusedActorNetwork(16, out_dim, model_head=model_head).state_dict()
    assert list(a) == list(b)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_fused_actor_network_refuses_what_the_kernel_cannot_run():
    import multiagent_rl_b200 as m
    with pytest.raises(ValueError, match='64'):
        m.FusedActorNetwork(65, 5)
    with pytest.raises(ValueError, match='16'):
        m.FusedActorNetwork(10, [8, 9])
    with pytest.raises(ValueError, match='16'):
        m.FusedActorNetwork(10, 17)
    net = m.FusedActorNetwork(10, 5)
    with pytest.raises(RuntimeError, match='CUDA'):
        net(torch.zeros(2, 3, 10))
    with pytest.raises(RuntimeError, match='CUDA'):
        net.double()(torch.zeros(2, 3, 10))


def test_backward_entry_points_refuse_bad_arguments_before_cuda():
    from multiagent_rl_b200 import _lib
    lib = _lib.load()
    assert lib.actor_backward(None, None, 4, 3, None, None, None, None, None, 0, None) == _lib.MPE_EINVAL
    assert b'null' in lib.mpe_last_error()
    assert lib.actor_backward_workspace(None, 4, 3) == _lib.MPE_EINVAL
    assert lib.actor_backward_workspace(None, -1, 13) == _lib.MPE_EINVAL
    assert ctypes.sizeof(_lib.ActorGrads) == 16 * 8
