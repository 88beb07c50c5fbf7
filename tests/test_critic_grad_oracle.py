"""CPU checks behind the critic backward's GPU tests: the float64 torch restatement (tests/_critic_torch.py) is the
reference critic - it equals oracle/critic_ref.py, which tests/test_oracle.py pins to the reference's own outputs -
and its autograd gradients are the derivatives of that function (central finite differences).  Also: the new ABI
entry points refuse bad arguments without a GPU, and FusedCriticNetwork builds the reference's parameters."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import critic_ref
from tests import _critic_torch as ct

TAGS = ['spread_n3', 'reference', 'model_n12']
SEEDS = {'spread_n3': 12345683, 'reference': 12345684, 'model_n12': 12345685}  # oracle/gen_golden.py


def _golden(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, 'critic_%s.npz' % tag))
    return g, {k[3:]: g[k] for k in g.files if k.startswith('sd/')}


@pytest.mark.parametrize('tag', TAGS)
def test_torch_restatement_equals_the_numpy_oracle(golden_dir, tag):
    g, sd = _golden(golden_dir, tag)
    want = critic_ref.forward(sd, g['obs'], g['action'])
    got = ct.grads(sd, g['obs'], g['action'], np.ones_like(g['q']), np.ones_like(g['q']) if 'r' in g.files else None)
    assert np.abs(got['q'] - want['q']).max() <= 1e-12
    if 'r' in g.files:
        assert np.abs(got['r'] - want['r']).max() <= 1e-12


@pytest.mark.parametrize('tag', TAGS)
def test_autograd_gradients_match_finite_differences(golden_dir, tag):
    """Central differences of the numpy forward (float64, step 1e-6) at sampled coordinates of every weight tensor,
    of obs and of action, for the loss sum(q * dq) (+ sum(r * dr))."""
    g, sd = _golden(golden_dir, tag)
    rng = np.random.RandomState(3)
    B = 6
    obs, act = g['obs'][:B].astype(np.float64), g['action'][:B].astype(np.float64)
    dq = rng.randn(B, 1)
    dr = rng.randn(B, 1) if 'r' in g.files else None
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    got = ct.grads(sd64, obs, act, dq, dr)

    def loss(sd_, o, a):
        # critic_ref.forward casts obs / action to float32 first; the restatement's inputs are float64 throughout
        p = {k: np.asarray(v, np.float64) for k, v in sd_.items()}
        x = np.concatenate([o, a], -1)
        h1 = np.maximum(x @ p['dense1.module.weight'].T + p['dense1.module.bias'], 0.0)
        B_, N_, _ = x.shape
        h, c, out = np.zeros((B_, 64)), np.zeros((B_, 64)), np.zeros((B_, N_, 64))
        sig = lambda z: 1.0 / (1.0 + np.exp(-z))  # noqa: E731
        for t in range(N_):
            gg = h1[:, t] @ p['lstm.weight_ih_l0'].T + p['lstm.bias_ih_l0'] + h @ p['lstm.weight_hh_l0'].T + p['lstm.bias_hh_l0']
            c = sig(gg[:, 64:128]) * c + sig(gg[:, :64]) * np.tanh(gg[:, 128:192])
            h = sig(gg[:, 192:]) * np.tanh(c)
            out[:, t] = h
        s = np.einsum('bth,bh->bt', out, h)
        s = np.exp(s - s.max(1, keepdims=True))
        n = np.einsum('bth,bt->bh', out, s / s.sum(1, keepdims=True))
        if dr is None:
            return float(((np.maximum(n, 0) @ p['dense2.weight'].T + p['dense2.bias']) * dq).sum())
        return float(((n @ p['dense2.weight'].T + p['dense2.bias']) * dq).sum()
                     + ((n @ p['dense3.weight'].T + p['dense3.bias']) * dr).sum())

    assert abs(loss(sd64, obs, act) - float((got['q'] * dq).sum() + (0 if dr is None else (got['r'] * dr).sum()))) < 1e-10
    eps = 1e-6
    for name in list(sd64) + ['obs', 'action']:
        base = obs if name == 'obs' else act if name == 'action' else sd64[name]
        for flat in rng.choice(base.size, size=min(6, base.size), replace=False):
            idx = np.unravel_index(flat, base.shape)
            vals = []
            for sgn in (1, -1):
                pert = base.copy()
                pert[idx] += sgn * eps
                if name == 'obs':
                    vals.append(loss(sd64, pert, act))
                elif name == 'action':
                    vals.append(loss(sd64, obs, pert))
                else:
                    vals.append(loss(dict(sd64, **{name: pert}), obs, act))
            fd = (vals[0] - vals[1]) / (2 * eps)
            assert abs(fd - got[name][idx]) <= 1e-6 * max(1.0, abs(fd)), (name, idx, fd, got[name][idx])


@pytest.mark.parametrize('tag', TAGS)
def test_fused_critic_network_initialises_like_the_reference(golden_dir, tag):
    """tests/golden/critic_*.npz hold the reference CriticNetwork's state_dict right after construction under
    torch.manual_seed(seed): FusedCriticNetwork(D + A, 1) under the same seed has the same keys, shapes and bits."""
    import multiagent_rl_b200 as m
    g, sd = _golden(golden_dir, tag)
    torch.manual_seed(SEEDS[tag])
    net = m.FusedCriticNetwork(sd['dense1.module.weight'].shape[1], 1, model='dense3.weight' in sd)
    got = net.state_dict()
    assert list(got) == list(sd)
    for k in sd:
        assert np.array_equal(got[k].numpy(), sd[k]), k


def test_fused_critic_network_refuses_what_the_kernel_cannot_run():
    import multiagent_rl_b200 as m
    with pytest.raises(ValueError, match='64'):
        m.FusedCriticNetwork(65, 1)
    with pytest.raises(ValueError, match='out_dim'):
        m.FusedCriticNetwork(15, 5)
    net = m.FusedCriticNetwork(15, 1)
    with pytest.raises(RuntimeError, match='CUDA'):
        net(torch.zeros(2, 3, 10), torch.zeros(2, 3, 5))
    with pytest.raises(RuntimeError, match='CUDA'):
        net.double()(torch.zeros(2, 3, 10), torch.zeros(2, 3, 5))


def test_backward_entry_points_refuse_bad_arguments_before_cuda():
    from multiagent_rl_b200 import _lib
    lib = _lib.load()
    assert lib.critic_backward(None, None, None, 4, 3, None, None, None, None, None, None, 0, None) == _lib.MPE_EINVAL
    assert b'null' in lib.mpe_last_error()
    assert lib.critic_backward_workspace(None, 4, 3) == _lib.MPE_EINVAL
    assert lib.critic_backward_workspace(None, -1, 17) == _lib.MPE_EINVAL
    assert ctypes.sizeof(_lib.CriticGrads) == 10 * 8
